// Post-processing of extracted LFOs on the eval path of the reference (SURVEY 8f, row N4):
//   smoothen                     modulations.py:358-362
//   stretch_corners              modulations.py:259-307  (_stretch_corners per row)
//   find_valid_mod_sig_indices   modulations.py:311-355  (check_mod_sig per row)
// The reference loops over the batch in python on 345-frame signals; here every row is one warp.
// All float32 arithmetic keeps the reference's operation order (bit-exact against the reference goldens).
#include "common.cuh"

#include <climits>
#include <math_constants.h>

namespace modfx {
namespace {

// torch's CPU mean over the last dim of x.unfold(-1, w, 1) adds float32 in this order: four 8-lane vector
// accumulators over blocks of 32 elements, remaining whole 8-vectors into accumulators 0, 1, 2, the four
// accumulators added left to right, the 8 lanes added left to right, then the scalar tail; a true division
// by w ends it.  (Probed on torch 2.11: bitwise for w < 5 and every multiple of 8, which covers the shipped
// windows 4, 8 and the default 32; other windows agree to 2e-7.)
__global__ void __launch_bounds__(256) smoothen_kernel(const float* __restrict__ in, float* __restrict__ out,
                                                       int64_t n, int64_t n_out, int w) {
    const float* x = in + (int64_t)blockIdx.y * n;
    float* y = out + (int64_t)blockIdx.y * n_out;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_out; i += (int64_t)gridDim.x * blockDim.x) {
        const float* p = x + i;
        float acc[32];
#pragma unroll
        for (int q = 0; q < 32; ++q) acc[q] = 0.0f;
        int k = 0;
        for (; k + 32 <= w; k += 32) {
#pragma unroll
            for (int q = 0; q < 32; ++q) acc[q] = __fadd_rn(acc[q], p[k + q]);
        }
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            if (k + 8 <= w) {
#pragma unroll
                for (int l = 0; l < 8; ++l) acc[8 * j + l] = __fadd_rn(acc[8 * j + l], p[k + l]);
                k += 8;
            }
        }
        float s = 0.0f;
#pragma unroll
        for (int l = 0; l < 8; ++l) {
            const float v = __fadd_rn(__fadd_rn(__fadd_rn(acc[l], acc[8 + l]), acc[16 + l]), acc[24 + l]);
            s = (l == 0) ? v : __fadd_rn(s, v);
        }
        for (; k < w; ++k) s = __fadd_rn(s, p[k]);
        y[i] = __fdiv_rn(s, (float)w);
    }
}

constexpr int kMaxAnchors = 64;     // corners + the final sample; rows with more corners are left unchanged anyway
constexpr int kRowsPerBlock = 4;    // warps per CTA, one row each

// stretch_corners after the smoothing: one warp per row.  The anchors (corners in index order, then the
// last sample) cut the row into disjoint segments; a segment whose end points are to move is shifted to
// start at 0, scaled by (target range / current range) and shifted so that it ends on its target
// (top corners 1.0, bottom corners 0.0, last sample itself).  Segments are independent, lanes stride a segment.
__global__ void __launch_bounds__(32 * kRowsPerBlock) stretch_corners_kernel(const float* __restrict__ in,
                                                                              float* __restrict__ out, int rows,
                                                                              int n, int max_n_corners) {
    __shared__ int a_idx[kRowsPerBlock][kMaxAnchors];
    __shared__ float a_val[kRowsPerBlock][kMaxAnchors];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row = blockIdx.x * kRowsPerBlock + warp;
    if (row >= rows) return;
    const float* m = in + (int64_t)row * n;
    float* o = out + (int64_t)row * n;

    // corners in index order
    int n_anchor = 0;
    for (int base = 0; base < n; base += 32) {
        const int i = base + lane;
        const unsigned f = (i < n) ? corner_flags(m, i, n) : 0u;
        const unsigned mask = __ballot_sync(kFull, f != 0u);
        if (f != 0u) {
            const int pos = n_anchor + __popc(mask & ((1u << lane) - 1u));
            if (pos < kMaxAnchors - 1) {
                a_idx[warp][pos] = i;
                a_val[warp][pos] = (f & 1u) ? 1.0f : 0.0f;
            }
        }
        n_anchor += __popc(mask);
    }
    for (int i = lane; i < n; i += 32) o[i] = m[i];
    if (n_anchor > max_n_corners || n_anchor > kMaxAnchors - 1) return;       // modulations.py:300-302
    if (lane == 0) {
        a_idx[warp][n_anchor] = n - 1;
        a_val[warp][n_anchor] = m[n - 1];
    }
    __syncwarp();
    int prev_idx = 0;
    float prev_anchor = m[0];
    for (int s = 0; s <= n_anchor; ++s) {
        const int idx = a_idx[warp][s];
        const float target = a_val[warp][s];
        if (prev_anchor != target && idx > prev_idx) {
            const float curr_range = fabsf(__fsub_rn(m[prev_idx], m[idx]));
            const float target_range = fabsf(__fsub_rn(prev_anchor, target));
            const float scale = __fdiv_rn(target_range, curr_range);
            float mn = CUDART_INF_F;
            bool has_nan = false;
            for (int i = prev_idx + 1 + lane; i <= idx; i += 32) {
                const float v = m[i];
                has_nan |= (v != v);
                mn = fminf(mn, v);
            }
#pragma unroll
            for (int d = 16; d >= 1; d >>= 1) mn = fminf(mn, __shfl_xor_sync(kFull, mn, d));
            if (__any_sync(kFull, has_nan)) mn = CUDART_NAN_F;                 // torch.min propagates NaN
            const float last = __fmul_rn(__fsub_rn(m[idx], mn), scale);
            const float shift = __fsub_rn(target, last);
            for (int i = prev_idx + 1 + lane; i <= idx; i += 32)
                o[i] = __fadd_rn(__fmul_rn(__fsub_rn(m[i], mn), scale), shift);
        }
        prev_idx = idx;
        prev_anchor = target;
    }
}

// check_mod_sig: 1..max corners of each kind and at least `min_frames` between neighbouring corners of a kind
__global__ void __launch_bounds__(32 * kRowsPerBlock) check_mod_sig_kernel(const float* __restrict__ in,
                                                                            uint8_t* __restrict__ valid, int rows,
                                                                            int n, int min_top, int max_top,
                                                                            int min_bottom, int max_bottom,
                                                                            int min_frames) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row = blockIdx.x * kRowsPerBlock + warp;
    if (row >= rows) return;
    const float* m = in + (int64_t)row * n;
    int cnt[2] = {0, 0}, last[2] = {-1, -1}, min_d[2] = {INT_MAX, INT_MAX};
    for (int base = 0; base < n; base += 32) {
        const int i = base + lane;
        const unsigned f = (i < n) ? corner_flags(m, i, n) : 0u;
#pragma unroll
        for (int kind = 0; kind < 2; ++kind) {
            const unsigned mask = __ballot_sync(kFull, (f >> kind) & 1u);
            if (mask == 0u) continue;
            // distances between neighbouring set bits inside the mask, and to the last corner of earlier chunks
            unsigned rest = mask;
            int prev = last[kind];
            while (rest) {
                const int b = __ffs(rest) - 1;
                rest &= rest - 1;
                const int pos = base + b;
                if (prev >= 0) min_d[kind] = min(min_d[kind], pos - prev);
                prev = pos;
            }
            last[kind] = prev;
            cnt[kind] += __popc(mask);
        }
    }
    if (lane == 0) {
        bool ok = cnt[0] >= min_top && cnt[1] >= min_bottom && cnt[0] <= max_top && cnt[1] <= max_bottom;
        if (ok && cnt[0] > 1 && min_d[0] < min_frames) ok = false;
        if (ok && cnt[1] > 1 && min_d[1] < min_frames) ok = false;
        valid[row] = ok ? 1 : 0;
    }
}

}  // namespace
}  // namespace modfx

using namespace modfx;

extern "C" int modfx_smoothen_f32(const float* in, float* out, int64_t rows, int64_t n, int32_t window, void* stream) {
    MODFX_REQUIRE(rows >= 0 && n >= 1 && window >= 1 && window <= n, "bad arguments rows=%lld n=%lld window=%d",
                  (long long)rows, (long long)n, window);
    if (rows == 0) return MODFX_OK;
    MODFX_REQUIRE(in && out, "NULL pointer");
    const int64_t n_out = n - window + 1;
    dim3 grid;
    if (const int st = row_grid(grid, n_out, rows, 1024)) return st;
    return launch(smoothen_kernel, grid, 256, 0, as_stream(stream), in, out, n, n_out, window);
}

extern "C" int modfx_stretch_corners_f32(const float* in, float* out, int64_t rows, int64_t n, int32_t max_n_corners,
                                         void* stream) {
    MODFX_REQUIRE(rows >= 0 && n >= 1 && n < (1ll << 30) && max_n_corners >= 0, "bad arguments rows=%lld n=%lld",
                  (long long)rows, (long long)n);
    if (max_n_corners > kMaxAnchors - 2)
        return fail(MODFX_ERR_UNSUPPORTED, "max_n_corners=%d (at most %d are built)", max_n_corners, kMaxAnchors - 2);
    if (rows == 0) return MODFX_OK;
    MODFX_REQUIRE(in && out && in != out, "NULL or aliased pointer");
    MODFX_REQUIRE(rows < (1ll << 31), "too many rows");
    const unsigned grid = (unsigned)((rows + kRowsPerBlock - 1) / kRowsPerBlock);
    return launch(stretch_corners_kernel, grid, 32 * kRowsPerBlock, 0, as_stream(stream), in, out, (int)rows, (int)n,
                  max_n_corners);
}

extern "C" int modfx_check_mod_sig_f32(const float* in, uint8_t* valid, int64_t rows, int64_t n, int32_t min_top,
                                       int32_t max_top, int32_t min_bottom, int32_t max_bottom, int32_t min_frames,
                                       void* stream) {
    MODFX_REQUIRE(rows >= 0 && n >= 1 && n < (1ll << 30), "bad arguments rows=%lld n=%lld", (long long)rows, (long long)n);
    if (rows == 0) return MODFX_OK;
    MODFX_REQUIRE(in && valid, "NULL pointer");
    MODFX_REQUIRE(rows < (1ll << 31), "too many rows");
    const unsigned grid = (unsigned)((rows + kRowsPerBlock - 1) / kRowsPerBlock);
    return launch(check_mod_sig_kernel, grid, 32 * kRowsPerBlock, 0, as_stream(stream), in, valid, (int)rows, (int)n,
                  min_top, max_top, min_bottom, max_bottom, min_frames);
}
