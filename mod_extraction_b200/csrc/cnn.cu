// LFO-net body behind the log-mel front end (SURVEY 8f, row N3), float32 pieces:
//   layer norm over (mel bins, frames) per (example, channel)     nn.LayerNorm(..., elementwise_affine=False)
//   5x13 convolution (time-dilated) + 2x1 max-pool + PReLU        Conv2d -> MaxPool2d -> PReLU
//   mean over mel bins + 1x1 convolution + sigmoid                tr.mean / Conv1d / tr.sigmoid
// Reference: Spectral2DCNN.__init__ / forward, mod_extraction/models.py:183-195,209-214.
//
// Activations are channels-last (B, H, W, C): the 64 channels of a pixel are one 256-byte line, which is the
// K-contiguous operand layout of the tensor-core convolution (cnn_tc.cu) and gives float4 traffic here.
// The CUDA-core convolution in this file is the exact-float32 path (and the only one for the 2-channel first
// layer, 3 % of the network's flops); layers 2..6 normally run on tcgen05 (MODFX_CNN_TF32).
#include "common.cuh"

#include <cuda_fp16.h>

#include <algorithm>

namespace modfx {

int cnn_conv_tf32(const void* x, const void* x_lo, float* y, int B, int H, int W, int dil_w, const void* weight,
                  const void* w_lo, const float* bias, const float* prelu, bool half, cudaStream_t stream);   // cnn_tc.cu
int cnn_conv1_tf32(const float* x, float* y, int B, int H, int W, const float* weight, const float* bias,
                   const float* prelu, cudaStream_t stream);     // cnn_tc.cu (2 input channels, dilation 1)

namespace {

constexpr int kLnThreads = 256;
constexpr int kLnChunkElems = 64 * 1024;      // elements of one example reduced by one CTA

__device__ __forceinline__ float round_tf32(float v) {
    unsigned u;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(v));
    return __uint_as_float(u);
}

// ---- layer norm, pass 1: per-chunk sums -------------------------------------------------------------
// Rows: channels-last input -> one row per example with C interleaved channels (row length P * C);
// NCHW input -> one row per (example, channel) with C == 1.  kLnThreads is a multiple of C, so a thread
// always meets the same channel and keeps its sums in registers (double: the variance is E[x^2] - mean^2).
__global__ void __launch_bounds__(kLnThreads) ln_stats_kernel(const float* __restrict__ x, double* __restrict__ part,
                                                              int64_t row_len, int C, int chunks) {
    __shared__ double s_sum[kLnThreads], s_sq[kLnThreads];
    const int tid = threadIdx.x;
    const int64_t row = blockIdx.y;
    const int64_t e0 = (int64_t)blockIdx.x * kLnChunkElems;
    const int64_t e1 = min(e0 + kLnChunkElems, row_len);
    const float* xr = x + row * row_len;
    double s = 0.0, q = 0.0;
    for (int64_t e = e0 + tid; e < e1; e += kLnThreads) {
        const double v = (double)xr[e];
        s += v;
        q += v * v;
    }
    s_sum[tid] = s;
    s_sq[tid] = q;
    __syncthreads();
    if (tid < C) {
        double ts = 0.0, tq = 0.0;
        for (int t = tid; t < kLnThreads; t += C) {       // fixed order: deterministic
            ts += s_sum[t];
            tq += s_sq[t];
        }
        double* p = part + ((row * chunks + blockIdx.x) * C + tid) * 2;
        p[0] = ts;
        p[1] = tq;
    }
}

// ---- layer norm, pass 2: normalise (and transpose NCHW -> NHWC for the first layer) ---------------------
template <bool kNchw>
__global__ void __launch_bounds__(kLnThreads) ln_apply_kernel(const float* __restrict__ x, float* __restrict__ y,
                                                              const double* __restrict__ part, int64_t P, int C,
                                                              int chunks, float eps, int round, int64_t lo_plane) {
    extern __shared__ float s_stat[];       // [C] mean, [C] rstd
    const int tid = threadIdx.x;
    const int64_t b = blockIdx.y;
    for (int c = tid; c < C; c += kLnThreads) {
        double ts = 0.0, tq = 0.0;
        if (kNchw) {
            const double* p = part + ((b * C + c) * chunks) * 2;
            for (int k = 0; k < chunks; ++k) { ts += p[2 * k]; tq += p[2 * k + 1]; }
        } else {
            const double* p = part + (b * chunks * C + c) * 2;
            for (int k = 0; k < chunks; ++k) { ts += p[(int64_t)k * C * 2]; tq += p[(int64_t)k * C * 2 + 1]; }
        }
        const double mean = ts / (double)P;
        const double var = fmax(tq / (double)P - mean * mean, 0.0);
        s_stat[c] = (float)mean;
        s_stat[C + c] = (float)(1.0 / sqrt(var + (double)eps));
    }
    __syncthreads();
    const int64_t n = P * C;
    const int64_t e0 = (int64_t)blockIdx.x * kLnChunkElems;
    const int64_t e1 = min(e0 + kLnChunkElems, n);
    const float* xb = x + b * n;
    float* yb = y + b * n;
    if (kNchw && C == 2) {
        // the log-mel tensor of the front end: a thread takes one pixel, reads it from both planes (coalesced) and writes
        // the interleaved pair
        const float m0 = s_stat[0], r0 = s_stat[2], m1 = s_stat[1], r1 = s_stat[3];
        for (int64_t p = e0 / 2 + tid; p < e1 / 2; p += kLnThreads) {
            float a = (xb[p] - m0) * r0, c = (xb[P + p] - m1) * r1;
            if (round) { a = round_tf32(a); c = round_tf32(c); }
            *reinterpret_cast<float2*>(yb + 2 * p) = make_float2(a, c);
        }
    } else if (kNchw) {
        // output element e = p * C + c reads x[c * P + p]
        for (int64_t e = e0 + tid; e < e1; e += kLnThreads) {
            const int64_t p = e / C;
            const int c = (int)(e - p * C);
            float v = (xb[(int64_t)c * P + p] - s_stat[c]) * s_stat[C + c];
            yb[e] = round ? round_tf32(v) : v;
        }
    } else if ((C & 3) == 0) {
        for (int64_t e = e0 + 4 * tid; e < e1; e += 4 * kLnThreads) {
            const int c = (int)(e % C);
            float4 v = *reinterpret_cast<const float4*>(xb + e);
            v.x = (v.x - s_stat[c]) * s_stat[C + c];
            v.y = (v.y - s_stat[c + 1]) * s_stat[C + c + 1];
            v.z = (v.z - s_stat[c + 2]) * s_stat[C + c + 2];
            v.w = (v.w - s_stat[c + 3]) * s_stat[C + c + 3];
            if (round == 3) {       // float16 operands of the tensor-core convolution (round-to-nearest)
                __half2* yh = reinterpret_cast<__half2*>(reinterpret_cast<__half*>(y) + b * n + e);
                yh[0] = __floats2half2_rn(v.x, v.y);
                yh[1] = __floats2half2_rn(v.z, v.w);
                continue;
            }
            if (round == 2) {       // error-compensated TF32: hi plane here, lo = tf32(v - hi) one plane further
                const float4 h = make_float4(round_tf32(v.x), round_tf32(v.y), round_tf32(v.z), round_tf32(v.w));
                *reinterpret_cast<float4*>(yb + e) = h;
                *reinterpret_cast<float4*>(yb + lo_plane + e) =
                    make_float4(round_tf32(v.x - h.x), round_tf32(v.y - h.y), round_tf32(v.z - h.z), round_tf32(v.w - h.w));
                continue;
            }
            if (round) v = make_float4(round_tf32(v.x), round_tf32(v.y), round_tf32(v.z), round_tf32(v.w));
            *reinterpret_cast<float4*>(yb + e) = v;
        }
    } else {
        for (int64_t e = e0 + tid; e < e1; e += kLnThreads) {
            const int c = (int)(e % C);
            float v = (xb[e] - s_stat[c]) * s_stat[C + c];
            yb[e] = round ? round_tf32(v) : v;
        }
    }
}

// ---- 5x13 convolution + 2x1 max-pool + PReLU on the CUDA cores ------------------------------------------
// A CTA owns one pooled output row (conv rows h0 = 2 hp and h0 + 1), 64 frames and all 64 output channels;
// a thread owns 4 frames x 4 channels x the 2 conv rows = 32 accumulators.  The 6 input rows h0-2 .. h0+3 are
// walked one at a time, channels in slabs of kCk: the slab of the input row (with its 6*dil halo, zero padded
// like padding="same") and the weights of the two kernel rows that meet it (kh = r for the upper conv row,
// kh = r - 1 for the lower) are staged in shared memory.
constexpr int kCo = 64, kKH = 5, kKW = 13;
constexpr int kTw = 64;                       // frames per CTA
constexpr int kConvThreads = 256;
constexpr int kMaxDil = 16;
constexpr int kXw = kTw + (kKW - 1) * kMaxDil;        // 256: widest staged input row

constexpr int kXPad = 4, kWPad = 4;             // row paddings that make the transposing stores conflict-free

template <int kCk>
struct ConvSmem {
    float xs[kCk][kXw + kXPad];               // input slab, [channel][frame]
    float ws[2][kKW][kCk][kCo + kWPad];       // weights, [conv row][kw][channel][out channel]
};

template <int kCin, int kCk>
__global__ void __launch_bounds__(kConvThreads) conv_fp32_kernel(const float* __restrict__ x, float* __restrict__ y,
                                                                 int H, int W, int dil,
                                                                 const float* __restrict__ weight,
                                                                 const float* __restrict__ bias,
                                                                 const float* __restrict__ prelu) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    ConvSmem<kCk>& sm = *reinterpret_cast<ConvSmem<kCk>*>(smem_raw);
    const int tid = threadIdx.x;
    const int tw = tid & 15, tc = tid >> 4;           // frames tw + 16 i (i < 4), channels 4 tc .. 4 tc + 3
    const int w0 = blockIdx.x * kTw;
    const int hp = blockIdx.y;
    const int64_t b = blockIdx.z;
    const int h0 = 2 * hp;
    const int xw = kTw + (kKW - 1) * dil;             // staged frames: w0 - 6 dil .. w0 + 63 + 6 dil
    const int wl = w0 - (kKW / 2) * dil;

    float acc[2][4][4];
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[r][i][j] = 0.0f;

    for (int r = 0; r < kKH + 1; ++r) {
        const int hi = h0 - kKH / 2 + r;
        if (hi < 0 || hi >= H) continue;              // zero padding: contributes nothing (CTA-uniform)
        const float* xrow = x + ((b * H + hi) * (int64_t)W) * kCin;
        for (int c0 = 0; c0 < kCin; c0 += kCk) {
            __syncthreads();                          // previous slab fully consumed
            for (int i = tid; i < xw * kCk; i += kConvThreads) {
                const int j = i / kCk, c = i - j * kCk;
                const int w = wl + j;
                sm.xs[c][j] = (w >= 0 && w < W) ? xrow[(int64_t)w * kCin + c0 + c] : 0.0f;
            }
            // weight (KH, KW, Cout, Cin): slot 0 = kernel row r (upper conv row), slot 1 = r - 1 (lower)
            for (int sk = 0; sk < 2 * kKW; ++sk) {
                const int slot = sk / kKW, kw = sk - slot * kKW;
                const int kh = r - slot;
                const bool live = kh >= 0 && kh < kKH;
                const float* wsrc = weight + ((int64_t)(live ? kh : 0) * kKW + kw) * kCo * kCin + c0;
                for (int e = tid; e < kCo * kCk; e += kConvThreads) {
                    const int co = e / kCk, c = e % kCk;
                    sm.ws[slot][kw][c][co] = live ? wsrc[co * kCin + c] : 0.0f;
                }
            }
            __syncthreads();
#pragma unroll 1
            for (int kw = 0; kw < kKW; ++kw) {
#pragma unroll
                for (int c = 0; c < kCk; ++c) {
                    const float* xp = &sm.xs[c][tw + kw * dil];
                    const float xv[4] = {xp[0], xp[16], xp[32], xp[48]};
                    const float4 wa = *reinterpret_cast<const float4*>(&sm.ws[0][kw][c][4 * tc]);
                    const float4 wb = *reinterpret_cast<const float4*>(&sm.ws[1][kw][c][4 * tc]);
                    const float w0v[4] = {wa.x, wa.y, wa.z, wa.w};
                    const float w1v[4] = {wb.x, wb.y, wb.z, wb.w};
#pragma unroll
                    for (int i = 0; i < 4; ++i)
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            acc[0][i][j] = fmaf(xv[i], w0v[j], acc[0][i][j]);
                            acc[1][i][j] = fmaf(xv[i], w1v[j], acc[1][i][j]);
                        }
                }
            }
        }
    }
    // bias is common to both conv rows: max first, then bias, then PReLU (MaxPool2d before PReLU, models.py:188-189)
    const float4 bv = *reinterpret_cast<const float4*>(bias + 4 * tc);
    const float4 pv = *reinterpret_cast<const float4*>(prelu + 4 * tc);
    const float bb[4] = {bv.x, bv.y, bv.z, bv.w};
    const float pp[4] = {pv.x, pv.y, pv.z, pv.w};
    float* yrow = y + ((b * (H / 2) + hp) * (int64_t)W) * kCo;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int w = w0 + tw + 16 * i;
        if (w >= W) continue;
        float o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float v = fmaxf(acc[0][i][j], acc[1][i][j]) + bb[j];
            o[j] = v > 0.0f ? v : pp[j] * v;
        }
        *reinterpret_cast<float4*>(yrow + (int64_t)w * kCo + 4 * tc) = make_float4(o[0], o[1], o[2], o[3]);
    }
}

// ---- head: mean over mel bins, 1x1 convolution, sigmoid ---------------------------------------------------
constexpr int kHeadW = 32;      // frames per CTA
__global__ void __launch_bounds__(256) head_kernel(const float* __restrict__ x, float* __restrict__ latent,
                                                   float* __restrict__ out, int H, int W, int C, int L,
                                                   const float* __restrict__ weight, const float* __restrict__ bias) {
    extern __shared__ float s_lat[];        // [C][kHeadW + 1]
    const int tid = threadIdx.x;
    const int w0 = blockIdx.x * kHeadW;
    const int64_t b = blockIdx.y;
    const int nw = min(kHeadW, W - w0);
    const float inv = 1.0f / (float)H;
    for (int i = tid; i < nw * C; i += blockDim.x) {
        const int j = i / C, c = i - j * C;
        float s = 0.0f;
        for (int h = 0; h < H; ++h) s += x[((b * H + h) * (int64_t)W + w0 + j) * C + c];
        s_lat[c * (kHeadW + 1) + j] = s * inv;
    }
    __syncthreads();
    for (int i = tid; i < nw * C; i += blockDim.x) {
        const int c = i / nw, j = i - c * nw;
        latent[(b * C + c) * (int64_t)W + w0 + j] = s_lat[c * (kHeadW + 1) + j];
    }
    for (int i = tid; i < nw * L; i += blockDim.x) {
        const int l = i / nw, j = i - l * nw;
        float s = bias[l];
        for (int c = 0; c < C; ++c) s = fmaf(weight[l * C + c], s_lat[c * (kHeadW + 1) + j], s);
        out[(b * L + l) * (int64_t)W + w0 + j] = 1.0f / (1.0f + expf(-s));
    }
}

int ln_chunks(int64_t row_len) { return (int)((row_len + kLnChunkElems - 1) / kLnChunkElems); }

}  // namespace
}  // namespace modfx

using namespace modfx;

extern "C" int64_t modfx_cnn_layernorm_workspace_bytes(int32_t B, int32_t C, int32_t H, int32_t W) {
    if (B < 0 || C < 1 || H < 1 || W < 1) return -1;
    // channels-last: B rows of chunks(P*C) * C pairs; NCHW: B*C rows of chunks(P) pairs -- take the larger
    const int64_t P = (int64_t)H * W;
    const int64_t a = (int64_t)B * ln_chunks(P * C) * C;
    const int64_t b = (int64_t)B * C * ln_chunks(P);
    return std::max(a, b) * 2 * (int64_t)sizeof(double) + 16;
}

extern "C" int modfx_cnn_layernorm_f32(const float* x, float* y, int32_t B, int32_t C, int32_t H, int32_t W,
                                       int32_t x_is_nchw, float eps, int32_t round_tf32, void* workspace,
                                       void* stream) {
    MODFX_REQUIRE(x && y && workspace, "NULL pointer");
    MODFX_REQUIRE(B >= 0 && C >= 1 && H >= 1 && W >= 1, "bad shape B=%d C=%d H=%d W=%d", B, C, H, W);
    MODFX_REQUIRE(!(x_is_nchw && x == y), "in-place needs a channels-last input");
    MODFX_REQUIRE(round_tf32 >= 0 && round_tf32 <= 3, "round_tf32=%d", round_tf32);
    if (round_tf32 >= 2 && (x_is_nchw || (C & 3) || x == y))
        return fail(MODFX_ERR_UNSUPPORTED, "the hi/lo split and the float16 output need a channels-last input, C %% 4 == 0 and y != x");
    if (kLnThreads % C != 0 && !x_is_nchw)
        return fail(MODFX_ERR_UNSUPPORTED, "C=%d: the channel count must divide %d", C, kLnThreads);
    if (C > 1024) return fail(MODFX_ERR_UNSUPPORTED, "C=%d too large", C);
    if (B == 0) return MODFX_OK;
    MODFX_REQUIRE(B <= 65535, "B=%d: at most 65535 examples per call", B);
    const int64_t P = (int64_t)H * W;
    double* part = reinterpret_cast<double*>((reinterpret_cast<uintptr_t>(workspace) + 15) & ~(uintptr_t)15);
    cudaStream_t st = as_stream(stream);
    const size_t smem = 2 * (size_t)C * sizeof(float);
    if (x_is_nchw) {
        MODFX_REQUIRE((int64_t)B * C <= 65535, "B*C too large for one call");
        const int chunks = ln_chunks(P);
        ln_stats_kernel<<<dim3(chunks, B * C), kLnThreads, 0, st>>>(x, part, P, 1, chunks);
        ln_apply_kernel<true><<<dim3(ln_chunks(P * C), B), kLnThreads, smem, st>>>(x, y, part, P, C, chunks, eps,
                                                                                   round_tf32, 0);
    } else {
        const int chunks = ln_chunks(P * C);
        ln_stats_kernel<<<dim3(chunks, B), kLnThreads, 0, st>>>(x, part, P * C, C, chunks);
        ln_apply_kernel<false><<<dim3(chunks, B), kLnThreads, smem, st>>>(x, y, part, P, C, chunks, eps, round_tf32,
                                                                          (int64_t)B * P * C);
    }
    MODFX_CUDA_OK(cudaGetLastError());
    return MODFX_OK;
}

template <int kCin, int kCk>
static int launch_conv_fp32(const float* x, float* y, int B, int H, int W, int dil, const float* weight,
                            const float* bias, const float* prelu, cudaStream_t st) {
    return launch(conv_fp32_kernel<kCin, kCk>, dim3((W + kTw - 1) / kTw, H / 2, B), kConvThreads, sizeof(ConvSmem<kCk>), st,
                  x, y, H, W, dil, weight, bias, prelu);
}

// The limits every convolution entry point shares.  An empty batch passes them: the caller returns before launching.
static int check_conv_shape(int B, int H, int dil_w) {
    if ((H & 1) || dil_w < 1 || dil_w > kMaxDil)
        return fail(MODFX_ERR_UNSUPPORTED, "H=%d must be even and the time dilation %d in [1, %d]", H, dil_w, kMaxDil);
    if (B > 0) MODFX_REQUIRE(B <= 65535 && H / 2 <= 65535, "grid too large");
    return MODFX_OK;
}

extern "C" int modfx_cnn_conv_pool_prelu_f32(const float* x, float* y, int32_t B, int32_t H, int32_t W, int32_t Cin,
                                             int32_t Cout, int32_t KH, int32_t KW, int32_t dil_w,
                                             const float* weight, const float* bias, const float* prelu,
                                             int32_t precision, void* stream) {
    MODFX_REQUIRE(x && y && weight && bias && prelu, "NULL pointer");
    MODFX_REQUIRE(B >= 0 && H >= 2 && W >= 1 && Cin >= 1, "bad shape B=%d H=%d W=%d Cin=%d", B, H, W, Cin);
    MODFX_REQUIRE(x != y, "x and y must not alias");
    if (KH != kKH || KW != kKW || Cout != kCo)
        return fail(MODFX_ERR_UNSUPPORTED, "only 5x13 kernels with 64 output channels are built (got %dx%d, %d)", KH, KW,
                    Cout);
    if (const int st = check_conv_shape(B, H, dil_w); st != MODFX_OK || B == 0) return st;
    cudaStream_t st = as_stream(stream);
    if (precision == MODFX_CNN_TF32) {
        if (Cin == 2 && dil_w == 1) return cnn_conv1_tf32(x, y, B, H, W, weight, bias, prelu, st);
        if (Cin != 64)
            return fail(MODFX_ERR_UNSUPPORTED, "the tensor-core convolution is built for Cin=64, and Cin=2 with dilation 1 (got %d, %d)",
                        Cin, dil_w);
        return cnn_conv_tf32(x, nullptr, y, B, H, W, dil_w, weight, nullptr, bias, prelu, false, st);
    }
    if (precision != MODFX_CNN_FP32) return fail(MODFX_ERR_INVALID, "precision=%d", precision);
    if (Cin == 2) return launch_conv_fp32<2, 2>(x, y, B, H, W, dil_w, weight, bias, prelu, st);
    if (Cin == 64) return launch_conv_fp32<64, 8>(x, y, B, H, W, dil_w, weight, bias, prelu, st);
    return fail(MODFX_ERR_UNSUPPORTED, "Cin=%d (2 and 64 are built)", Cin);
}

extern "C" int modfx_cnn_conv_pool_prelu_tf32x3_f32(const float* x_hi, const float* x_lo, float* y, int32_t B, int32_t H,
                                                    int32_t W, int32_t dil_w, const float* w_hi, const float* w_lo,
                                                    const float* bias, const float* prelu, void* stream) {
    MODFX_REQUIRE(x_hi && x_lo && y && w_hi && w_lo && bias && prelu, "NULL pointer");
    MODFX_REQUIRE(B >= 0 && H >= 2 && W >= 1, "bad shape B=%d H=%d W=%d", B, H, W);
    MODFX_REQUIRE(x_hi != y && x_lo != y, "x and y must not alias");
    if (const int st = check_conv_shape(B, H, dil_w); st != MODFX_OK || B == 0) return st;
    return cnn_conv_tf32(x_hi, x_lo, y, B, H, W, dil_w, w_hi, w_lo, bias, prelu, false, as_stream(stream));
}

extern "C" int modfx_cnn_conv_pool_prelu_f16_f32(const void* x_f16, float* y, int32_t B, int32_t H, int32_t W,
                                                 int32_t dil_w, const void* w_f16, const float* bias, const float* prelu,
                                                 void* stream) {
    MODFX_REQUIRE(x_f16 && y && w_f16 && bias && prelu, "NULL pointer");
    MODFX_REQUIRE(B >= 0 && H >= 2 && W >= 1, "bad shape B=%d H=%d W=%d", B, H, W);
    MODFX_REQUIRE(x_f16 != (const void*)y, "x and y must not alias");
    if (const int st = check_conv_shape(B, H, dil_w); st != MODFX_OK || B == 0) return st;
    return cnn_conv_tf32(x_f16, nullptr, y, B, H, W, dil_w, w_f16, nullptr, bias, prelu, true, as_stream(stream));
}

extern "C" int modfx_cnn_head_f32(const float* x, float* latent, float* out, int32_t B, int32_t H, int32_t W,
                                  int32_t C, int32_t L, const float* weight, const float* bias, void* stream) {
    MODFX_REQUIRE(x && latent && out && weight && bias, "NULL pointer");
    MODFX_REQUIRE(B >= 0 && H >= 1 && W >= 1 && C >= 1 && L >= 1, "bad shape");
    if (C > 1024) return fail(MODFX_ERR_UNSUPPORTED, "C=%d too large", C);
    if (B == 0) return MODFX_OK;
    MODFX_REQUIRE(B <= 65535, "B too large");
    return launch(head_kernel, dim3((W + kHeadW - 1) / kHeadW, B), 256, (size_t)C * (kHeadW + 1) * sizeof(float),
                  as_stream(stream), x, latent, out, H, W, C, L, weight, bias);
}
