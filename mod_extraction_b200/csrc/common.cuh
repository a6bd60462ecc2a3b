// Shared host/device helpers for libmodfx (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "modfx.h"

namespace modfx {

// ---- error plumbing ------------------------------------------------------------------
void set_error(const char* fmt, ...);
int fail(modfx_status st, const char* fmt, ...);

#define MODFX_CUDA_OK(expr)                                                              \
    do {                                                                                 \
        cudaError_t _e = (expr);                                                         \
        if (_e != cudaSuccess)                                                           \
            return ::modfx::fail(MODFX_ERR_CUDA, "%s failed: %s", #expr, cudaGetErrorString(_e)); \
    } while (0)

#define MODFX_REQUIRE(cond, ...)                                                         \
    do {                                                                                 \
        if (!(cond)) return ::modfx::fail(MODFX_ERR_INVALID, __VA_ARGS__);               \
    } while (0)

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// kernel<<<grid, block, smem, stream>>>(args...), opting in first when smem exceeds the default 48 KB.  That default
// covers static and dynamic shared memory together, but only the dynamic size is tested here: of the kernels launched
// with dynamic shared memory, only fc_wide_kernel (32 B, dynamic size a power of two, never within 32 B of 48 KB) and
// phaser_fused_kernel (under 100 B, dynamic size under 40 KB) also have static shared memory.  A kernel that gains
// static shared memory must count it.
template <typename... Params, typename... Args>
int launch(void (*kernel)(Params...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args... args) {
    if (smem > 48 * 1024)
        MODFX_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kernel<<<grid, block, smem, stream>>>(args...);
    MODFX_CUDA_OK(cudaGetLastError());
    return MODFX_OK;
}

// Grid of a kernel that strides over the elements of row blockIdx.y in blocks of 256 threads: one block per 256
// elements of a row, at most `cap`.  More rows than grid.y holds are refused.
inline int row_grid(dim3& grid, int64_t per_row, int64_t rows, int cap) {
    MODFX_REQUIRE(rows <= 65535, "%lld rows exceed grid.y", (long long)rows);
    const int64_t gx = (per_row + 255) / 256;
    grid = dim3((unsigned)(gx < cap ? gx : cap), (unsigned)rows);
    return MODFX_OK;
}

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;

// ---- float32 constants exactly as torch materialises the python doubles ---------------
// float(2*pi), float(pi), float(pi/2)
#define MODFX_TWO_PI_F 6.2831854820251465f
#define MODFX_PI_F 3.1415927410125732f
#define MODFX_HALF_PI_F 1.5707963705062866f

// torch.remainder(a, b) for b > 0: fmod (exact) then shift into [0, b).
__device__ __forceinline__ float torch_remainder(float a, float b) {
    float m = fmodf(a, b);
    if (m != 0.0f && m < 0.0f) m = __fadd_rn(m, b);
    return m;
}

// Per-example LFO description (already halved for rect shapes by the host, modulations.py:26-29).
struct LfoDesc {
    float inc;     // f32( f32( f32(2pi) * f32(freq) ) / f32(sr) )   -- true IEEE division
    float phase;
    int shape;
    float exp;     // 1.0 => none
};

__device__ __forceinline__ LfoDesc make_lfo_desc(float freq, float phase, int shape, float exp, float sr) {
    LfoDesc d;
    d.inc = __fdiv_rn(__fmul_rn(MODFX_TWO_PI_F, freq), sr);
    d.phase = phase;
    d.shape = shape;
    d.exp = exp;
    return d;
}

// cos evaluated in double and rounded once: within 1 ulp of any faithful float32 cos
// (the reference's is Sleef's 1-ulp vector cos).  Control-rate only, so the cost is nil.
__device__ __forceinline__ float cos_f32(float a) { return (float)cos((double)a); }

// make_mod_signal element i (0-based): torch.cumsum accumulates float32 in double, so
// arg_i = f32(f64(inc) * (i+1)) + phase (modulations.py:31; SURVEY 8a-L1).
__device__ __forceinline__ float lfo_value(const LfoDesc& d, int64_t i) {
    const float arg = __fadd_rn((float)((double)d.inc * (double)(i + 1)), d.phase);
    float v;
    switch (d.shape) {
        case MODFX_SHAPE_COS:            // (cos(arg + pi) + 1) / 2           modulations.py:35
            v = __fdiv_rn(__fadd_rn(cos_f32(__fadd_rn(arg, MODFX_PI_F)), 1.0f), 2.0f);
            break;
        case MODFX_SHAPE_RECT_COS:       // abs(cos(arg + pi/2))              modulations.py:37
            v = fabsf(cos_f32(__fadd_rn(arg, MODFX_HALF_PI_F)));
            break;
        case MODFX_SHAPE_INV_RECT_COS:   // -abs(cos(arg)) + 1                modulations.py:39
            v = __fadd_rn(-fabsf(cos_f32(arg)), 1.0f);
            break;
        case MODFX_SHAPE_SQR: {          // (sign(cos(arg + pi)) + 1) / 2     modulations.py:41-43
            const float c = cos_f32(__fadd_rn(arg, MODFX_PI_F));
            const float s = (c > 0.0f) ? 1.0f : ((c < 0.0f) ? -1.0f : 0.0f);
            v = __fdiv_rn(__fadd_rn(s, 1.0f), 2.0f);
        } break;
        default: {                       // saw = remainder(arg, 2pi) / 2pi   modulations.py:32
            const float saw = __fdiv_rn(torch_remainder(arg, MODFX_TWO_PI_F), MODFX_TWO_PI_F);
            if (d.shape == MODFX_SHAPE_SAW) v = saw;
            else if (d.shape == MODFX_SHAPE_RSAW) v = __fsub_rn(1.0f, saw);     // :48
            else {                                                              // tri :50-51
                const float tri = __fmul_rn(2.0f, saw);
                v = (tri > 1.0f) ? __fsub_rn(2.0f, tri) : tri;
            }
        } break;
    }
    if (d.exp != 1.0f) {                 // torch.pow(Tensor, Scalar) fast paths, modulations.py:55-56
        if (d.exp == 2.0f) v = __fmul_rn(v, v);
        else if (d.exp == 3.0f) v = __fmul_rn(__fmul_rn(v, v), v);
        else if (d.exp == 0.5f) v = __fsqrt_rn(v);
        else v = (float)pow((double)v, (double)d.exp);
    }
    return v;
}

// The two taps and weights of F.interpolate(mode="linear") at source position src of an I-point row (ATen
// upsample_linear1d, util.py:15-29).  Int is the index type of the row.
template <typename Int>
struct LinearTaps {
    Int i0, i1;
    float l0, l1;
};

template <typename Int>
__device__ __forceinline__ LinearTaps<Int> linear_taps(float src, Int I) {
    LinearTaps<Int> t;
    t.i0 = min((Int)src, I - 1);
    t.i1 = t.i0 + ((t.i0 < I - 1) ? 1 : 0);
    t.l1 = __fsub_rn(src, (float)t.i0);
    t.l0 = __fsub_rn(1.0f, t.l1);
    return t;
}

// align_corners=True: output element i reads source position scale * i, scale = f32(I-1)/f32(O-1).
__device__ __forceinline__ LinearTaps<int> taps_ac(float scale, int i, int I) {
    return linear_taps(__fmul_rn(scale, (float)i), I);
}

// The torch CPU build contracts the blend to fma(l0, x0, l1*x1) -- pinned bitwise by tests/golden/interp.npz.
template <typename Int>
__device__ __forceinline__ float blend(const LinearTaps<Int>& t, float v0, float v1) {
    return __fmaf_rn(t.l0, v0, __fmul_rn(t.l1, v1));
}

// F.interpolate(mode="linear", align_corners=True) element i of an O-point output from an I-point row `lo`.
__device__ __forceinline__ float upsample_ac(const float* __restrict__ lo, int I, float scale, int i) {
    const LinearTaps<int> t = taps_ac(scale, i, I);
    return blend(t, lo[t.i0], lo[t.i1]);
}

__device__ __forceinline__ float upsample_scale_ac_dev(int I, int O) {
    return (O > 1) ? __fdiv_rn((float)(I - 1), (float)(O - 1)) : 0.0f;
}

inline float upsample_scale_ac(int64_t I, int64_t O) {
    return (O > 1) ? (float)(I - 1) / (float)(O - 1) : 0.0f;
}

// find_corners (modulations.py:219-238) at sample i of the n-point row m: bit 0 = top corner, bit 1 = bottom corner,
// 0 outside 1..n-2.  A corner is a sign change of the first difference; the flags are
// -floor(diff_l(+/-) * (diff_r + 1e-16)) compared against 1.
template <typename Int>
__device__ __forceinline__ unsigned corner_flags(const float* m, Int i, Int n) {
    if (i < 1 || i > n - 2) return 0u;
    const float dl = __fsub_rn(m[i], m[i - 1]);
    const float dr = __fadd_rn(__fsub_rn(m[i + 1], m[i]), 1e-16f);
    const float pos = (dl > 0.0f) ? dl : 0.0f;          // (diff_l > 0) * diff_l
    const float neg = (dl < 0.0f) ? dl : 0.0f;
    unsigned f = 0;
    if (-floorf(__fmul_rn(pos, dr)) == 1.0f) f |= 1u;
    if (-floorf(__fmul_rn(neg, dr)) == 1.0f) f |= 2u;
    return f;
}

int num_sms();

}  // namespace modfx
