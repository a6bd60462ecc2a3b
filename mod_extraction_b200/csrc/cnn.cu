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
int cnn_conv_tf32_grad(const float* x, float* y, float* z, uint8_t* am, int B, int H, int W, int dil, const float* weight,
                       const float* bias, const float* prelu, cudaStream_t stream);            // cnn_tc.cu
int cnn_conv1_tf32_train(const float* x, float* y, float* z, uint8_t* am, int B, int H, int W, const float* weight,
                         const float* bias, const float* prelu, cudaStream_t stream);          // cnn_tc.cu
int cnn_conv_wgrad_tf32(const float* x, const float* dconv, float* part, int B, int H, int W, int dil,
                        cudaStream_t stream);                                                  // cnn_tc.cu
int cnn_wgrad_splits();

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

// ==== backward pass of the body (training, TF32 semantics: operand rounding is a straight-through step) ==========
// Every reduction writes one partial per CTA; sum_parts_kernel adds them in a fixed order, so gradients are
// bit-reproducible run to run.

// out[i] = sum_k part[k * n + i] (k ascending); i < n0 goes to out0, the rest to out1
__global__ void __launch_bounds__(256) sum_parts_kernel(const float* __restrict__ part, int n_parts, int64_t n, int64_t n0,
                                                        float* __restrict__ out0, float* __restrict__ out1) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    float s = 0.0f;
    for (int k = 0; k < n_parts; ++k) s += part[(int64_t)k * n + i];
    if (i < n0) out0[i] = s;
    else out1[i - n0] = s;
}

// ---- max-pool (2x1) + PReLU backward: dA (B, H/2, W, 64) -> dConv (B, H, W, 64) rounded to TF32 (the operand of both
// gradient GEMMs); the pool routes dz = dA * PReLU'(z) to the conv row its argmax names.  Partials per CTA:
// [0, 64) dbias = sum dz, [64, 128) dslope = sum dA * z * [z <= 0].
constexpr int kBwdChunk = 64 * 1024;          // pooled elements per CTA
__global__ void __launch_bounds__(256) pool_prelu_bwd_kernel(const float* __restrict__ dA, const float* __restrict__ z,
                                                             const uint8_t* __restrict__ am,
                                                             const float* __restrict__ slope, float* __restrict__ dconv,
                                                             float* __restrict__ part, int64_t n, int W) {
    __shared__ float s_b[256], s_s[256];
    const int tid = threadIdx.x, c = tid & 63;
    const float a = slope[c];
    const int64_t e0 = (int64_t)blockIdx.x * kBwdChunk, e1 = min(e0 + kBwdChunk, n);
    float sb = 0.0f, ss = 0.0f;
    for (int64_t e = e0 + tid; e < e1; e += 256) {
        const int64_t pix = e >> 6, bp = pix / W, w = pix - bp * W;
        const float g = dA[e], zv = z[e];
        const float dz = zv > 0.0f ? g : a * g;
        sb += dz;
        if (zv <= 0.0f) ss += g * zv;
        const int64_t up = ((2 * bp * W + w) << 6) + c, lo = up + ((int64_t)W << 6);
        const float r = round_tf32(dz);
        dconv[up] = am[e] ? 0.0f : r;
        dconv[lo] = am[e] ? r : 0.0f;
    }
    s_b[tid] = sb;
    s_s[tid] = ss;
    __syncthreads();
    if (tid < 64) {
        float tb = 0.0f, ts = 0.0f;
        for (int t = tid; t < 256; t += 64) {
            tb += s_b[t];
            ts += s_s[t];
        }
        part[(int64_t)blockIdx.x * 128 + tid] = tb;
        part[(int64_t)blockIdx.x * 128 + 64 + tid] = ts;
    }
}

// mean / rstd of (b, c) from the partial sums of the forward's ln_stats_kernel, exactly as ln_apply_kernel<false> forms them
__device__ __forceinline__ float2 ln_stat(const double* __restrict__ part, int64_t b, int c, int C, int chunks, int64_t P,
                                          float eps) {
    double ts = 0.0, tq = 0.0;
    const double* p = part + (b * chunks * C + c) * 2;
    for (int k = 0; k < chunks; ++k) { ts += p[(int64_t)k * C * 2]; tq += p[(int64_t)k * C * 2 + 1]; }
    const double mean = ts / (double)P;
    const double var = fmax(tq / (double)P - mean * mean, 0.0);
    return make_float2((float)mean, (float)(1.0 / sqrt(var + (double)eps)));
}

// ---- layer norm backward, pass 1: per-chunk sums of g and g * xhat per (b, c), xhat = (x - mean) * rstd unrounded
__global__ void __launch_bounds__(kLnThreads) ln_bwd_stats_kernel(const float* __restrict__ g, const float* __restrict__ x,
                                                                  const double* __restrict__ fwd, double* __restrict__ part,
                                                                  int64_t P, int C, int chunks, float eps) {
    __shared__ double s_sum[kLnThreads], s_gx[kLnThreads];
    __shared__ float s_stat[2 * kLnThreads];
    const int tid = threadIdx.x;
    const int64_t b = blockIdx.y, n = P * C;
    for (int c = tid; c < C; c += kLnThreads) {
        const float2 mr = ln_stat(fwd, b, c, C, chunks, P, eps);
        s_stat[c] = mr.x;
        s_stat[C + c] = mr.y;
    }
    __syncthreads();
    const int64_t e0 = (int64_t)blockIdx.x * kLnChunkElems, e1 = min(e0 + kLnChunkElems, n);
    const int c = tid % C;
    const float m = s_stat[c], r = s_stat[C + c];
    double s = 0.0, q = 0.0;
    for (int64_t e = e0 + tid; e < e1; e += kLnThreads) {
        const float gv = g[b * n + e];
        const float xh = (x[b * n + e] - m) * r;
        s += (double)gv;
        q += (double)gv * (double)xh;
    }
    s_sum[tid] = s;
    s_gx[tid] = q;
    __syncthreads();
    if (tid < C) {
        double ts = 0.0, tq = 0.0;
        for (int t = tid; t < kLnThreads; t += C) {
            ts += s_sum[t];
            tq += s_gx[t];
        }
        double* p = part + ((b * chunks + blockIdx.x) * C + tid) * 2;
        p[0] = ts;
        p[1] = tq;
    }
}

// ---- layer norm backward, pass 2: dx = rstd * (g - mean(g) - xhat * mean(g * xhat))
__global__ void __launch_bounds__(kLnThreads) ln_bwd_apply_kernel(const float* __restrict__ g, const float* __restrict__ x,
                                                                  const double* __restrict__ fwd,
                                                                  const double* __restrict__ part, float* __restrict__ dx,
                                                                  int64_t P, int C, int chunks, float eps) {
    __shared__ float s_stat[4 * kLnThreads];    // mean, rstd, mean(g), mean(g * xhat)
    const int tid = threadIdx.x;
    const int64_t b = blockIdx.y, n = P * C;
    for (int c = tid; c < C; c += kLnThreads) {
        const float2 mr = ln_stat(fwd, b, c, C, chunks, P, eps);
        s_stat[c] = mr.x;
        s_stat[C + c] = mr.y;
    }
    for (int c = tid; c < C; c += kLnThreads) {
        double ts = 0.0, tq = 0.0;
        const double* p = part + (b * chunks * C + c) * 2;
        for (int k = 0; k < chunks; ++k) { ts += p[(int64_t)k * C * 2]; tq += p[(int64_t)k * C * 2 + 1]; }
        const double inv = 1.0 / (double)P;
        s_stat[2 * C + c] = (float)(ts * inv);
        s_stat[3 * C + c] = (float)(tq * inv);
    }
    __syncthreads();
    const int64_t e0 = (int64_t)blockIdx.x * kLnChunkElems, e1 = min(e0 + kLnChunkElems, n);
    const int c = tid % C;
    const float m = s_stat[c], r = s_stat[C + c], mg = s_stat[2 * C + c], mgx = s_stat[3 * C + c];
    for (int64_t e = e0 + tid; e < e1; e += kLnThreads) {
        const float xh = (x[b * n + e] - m) * r;
        dx[b * n + e] = r * (g[b * n + e] - mg - xh * mgx);
    }
}

// ---- weight gradient of the 2-channel first layer on the CUDA cores (3 % of the backward's flops).  A CTA walks a fixed
// range of (example, conv row, 64-frame) tiles; thread (co, g) keeps the 17 taps t = g + 4 j of output channel co for
// both input channels.  Partial per CTA in the parameter's layout (64, 2, 5, 13).
constexpr int kW1Tw = 64, kW1Parts = 296;
__global__ void __launch_bounds__(256) wgrad1_kernel(const float* __restrict__ x, const float* __restrict__ dconv,
                                                     float* __restrict__ part, int B, int H, int W) {
    __shared__ float s_d[kW1Tw][kCo];
    __shared__ float2 s_x[kKH][kW1Tw + kKW - 1];
    const int tid = threadIdx.x, co = tid & 63, g = __shfl_sync(kFull, tid >> 6, 0);
    const int ntw = (W + kW1Tw - 1) / kW1Tw;
    const int64_t tiles = (int64_t)B * H * ntw;
    const int64_t k0 = tiles * blockIdx.x / gridDim.x, k1 = tiles * (blockIdx.x + 1) / gridDim.x;
    constexpr int kJ = (kKH * kKW + 3) / 4;     // 17
    float acc[kJ][2];
    int off[kJ];
#pragma unroll
    for (int j = 0; j < kJ; ++j) {
        const int t = min(g + 4 * j, kKH * kKW - 1);
        off[j] = (t / kKW) * (kW1Tw + kKW - 1) + t % kKW;
        acc[j][0] = acc[j][1] = 0.0f;
    }
    for (int64_t k = k0; k < k1; ++k) {
        const int tw = (int)(k % ntw);
        const int64_t bh = k / ntw;
        const int h = (int)(bh % H);
        const int64_t b = bh / H;
        const int w0 = tw * kW1Tw;
        __syncthreads();
        for (int i = tid; i < kW1Tw * kCo; i += 256) {
            const int w = w0 + (i >> 6);
            s_d[i >> 6][i & 63] = w < W ? dconv[((b * H + h) * W + w) * kCo + (i & 63)] : 0.0f;
        }
        for (int i = tid; i < kKH * (kW1Tw + kKW - 1); i += 256) {
            const int r = i / (kW1Tw + kKW - 1), j = i - r * (kW1Tw + kKW - 1);
            const int hr = h + r - kKH / 2, w = w0 + j - kKW / 2;
            s_x[r][j] = (hr >= 0 && hr < H && w >= 0 && w < W)
                            ? *reinterpret_cast<const float2*>(x + ((b * H + hr) * W + w) * 2)
                            : make_float2(0.0f, 0.0f);
        }
        __syncthreads();
        const float2* xs = &s_x[0][0];
#pragma unroll 4
        for (int w = 0; w < kW1Tw; ++w) {
            const float d = s_d[w][co];
#pragma unroll
            for (int j = 0; j < kJ; ++j) {
                const float2 v = xs[off[j] + w];
                acc[j][0] = fmaf(d, v.x, acc[j][0]);
                acc[j][1] = fmaf(d, v.y, acc[j][1]);
            }
        }
    }
#pragma unroll
    for (int j = 0; j < kJ; ++j) {
        const int t = g + 4 * j;
        if (t < kKH * kKW) {
            part[(int64_t)blockIdx.x * kCo * 2 * kKH * kKW + (co * 2 + 0) * kKH * kKW + t] = acc[j][0];
            part[(int64_t)blockIdx.x * kCo * 2 * kKH * kKW + (co * 2 + 1) * kKH * kKW + t] = acc[j][1];
        }
    }
}

// ---- head backward: out = sigmoid(W latent + b), latent = mean_H(x).  dx (B, H, W, C) = (W^T dlogit + dlatent) / H
// on every row; partials per CTA: [0, L C) dW_out, [L C, L C + L) db_out.
__global__ void __launch_bounds__(256) head_bwd_kernel(const float* __restrict__ latent, const float* __restrict__ out,
                                                       const float* __restrict__ dout, const float* __restrict__ dlatent,
                                                       float* __restrict__ dx, float* __restrict__ part, int H, int W,
                                                       int C, int L, const float* __restrict__ weight) {
    extern __shared__ float s_h[];              // [L][kHeadW + 1] dlogit, [C][kHeadW + 1] d(latent) / H
    float* s_dl = s_h;
    float* s_dt = s_h + L * (kHeadW + 1);
    const int tid = threadIdx.x;
    const int w0 = blockIdx.x * kHeadW;
    const int64_t b = blockIdx.y;
    const int nw = min(kHeadW, W - w0);
    const float inv = 1.0f / (float)H;
    for (int i = tid; i < L * nw; i += blockDim.x) {
        const int l = i / nw, j = i - l * nw;
        const int64_t o = (b * L + l) * (int64_t)W + w0 + j;
        s_dl[l * (kHeadW + 1) + j] = dout[o] * out[o] * (1.0f - out[o]);
    }
    __syncthreads();
    for (int i = tid; i < C * nw; i += blockDim.x) {
        const int c = i / nw, j = i - c * nw;
        float s = dlatent[(b * C + c) * (int64_t)W + w0 + j];
        for (int l = 0; l < L; ++l) s = fmaf(weight[l * C + c], s_dl[l * (kHeadW + 1) + j], s);
        s_dt[c * (kHeadW + 1) + j] = s * inv;
    }
    __syncthreads();
    for (int64_t i = tid; i < (int64_t)H * nw * C; i += blockDim.x) {
        const int c = (int)(i % C);
        const int64_t hj = i / C;
        const int j = (int)(hj % nw), h = (int)(hj / nw);
        dx[((b * H + h) * (int64_t)W + w0 + j) * C + c] = s_dt[c * (kHeadW + 1) + j];
    }
    float* pp = part + (b * gridDim.x + blockIdx.x) * (int64_t)(L * C + L);
    for (int i = tid; i < L * C + L; i += blockDim.x) {
        const int l = i < L * C ? i / C : i - L * C, c = i < L * C ? i - l * C : -1;
        float s = 0.0f;
        for (int j = 0; j < nw; ++j)
            s = fmaf(s_dl[l * (kHeadW + 1) + j], c >= 0 ? latent[(b * C + c) * (int64_t)W + w0 + j] : 1.0f, s);
        pp[i] = s;
    }
}

int sum_parts(const float* part, int n_parts, int64_t n, int64_t n0, float* out0, float* out1, cudaStream_t s) {
    return launch(sum_parts_kernel, dim3((unsigned)((n + 255) / 256)), 256, 0, s, part, n_parts, n, n0, out0, out1);
}

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
    cudaStream_t s = as_stream(stream);
    const size_t smem = 2 * (size_t)C * sizeof(float);
    int st;
    if (x_is_nchw) {
        MODFX_REQUIRE((int64_t)B * C <= 65535, "B*C too large for one call");
        const int chunks = ln_chunks(P);
        st = launch(ln_stats_kernel, dim3(chunks, B * C), kLnThreads, 0, s, x, part, P, 1, chunks);
        if (st == MODFX_OK)
            st = launch(ln_apply_kernel<true>, dim3(ln_chunks(P * C), B), kLnThreads, smem, s, x, y, part, P, C, chunks,
                        eps, round_tf32, 0);
    } else {
        const int chunks = ln_chunks(P * C);
        st = launch(ln_stats_kernel, dim3(chunks, B), kLnThreads, 0, s, x, part, P * C, C, chunks);
        if (st == MODFX_OK)
            st = launch(ln_apply_kernel<false>, dim3(chunks, B), kLnThreads, smem, s, x, y, part, P, C, chunks, eps,
                        round_tf32, (int64_t)B * P * C);
    }
    return st;
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

// ==== training: forward with saves, and the backward pass (TF32, the shipped 5x13 / 64-channel shape) ================

extern "C" int64_t modfx_cnn_train_workspace_bytes(int32_t B, int32_t H, int32_t W, int32_t L) {
    if (B < 0 || H < 2 || W < 1 || L < 1) return -1;
    const int64_t wg = (int64_t)cnn_wgrad_splits() * kCo * kCo * kKH * kKW;
    const int64_t wg1 = (int64_t)kW1Parts * kCo * 2 * kKH * kKW;
    const int64_t pool = ((int64_t)B * (H / 2) * W * kCo + kBwdChunk - 1) / kBwdChunk * 128;
    const int64_t ln = (int64_t)B * ln_chunks((int64_t)H * W * kCo) * kCo * 2 * 2;     // doubles, as floats
    const int64_t head = (int64_t)B * ((W + kHeadW - 1) / kHeadW) * ((int64_t)L * kCo + L);
    return std::max(std::max(std::max(wg, wg1), std::max(pool, ln)), head) * (int64_t)sizeof(float) + 16;
}

static float* ws_align(void* workspace) {
    return reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(workspace) + 15) & ~(uintptr_t)15);
}

extern "C" int modfx_cnn_conv_pool_prelu_train_f32(const float* x, float* y, float* z, uint8_t* argmax, int32_t B,
                                                   int32_t H, int32_t W, int32_t Cin, int32_t dil_w, const float* weight,
                                                   const float* bias, const float* prelu, void* stream) {
    MODFX_REQUIRE(x && y && z && argmax && weight && bias && prelu, "NULL pointer");
    MODFX_REQUIRE(B >= 0 && H >= 2 && W >= 1, "bad shape B=%d H=%d W=%d", B, H, W);
    MODFX_REQUIRE(x != y && x != z && y != z, "x, y and z must not alias");
    if (const int st = check_conv_shape(B, H, dil_w); st != MODFX_OK || B == 0) return st;
    cudaStream_t st = as_stream(stream);
    if (Cin == 2 && dil_w == 1) return cnn_conv1_tf32_train(x, y, z, argmax, B, H, W, weight, bias, prelu, st);
    if (Cin != 64)
        return fail(MODFX_ERR_UNSUPPORTED, "the training forward is built for Cin=64, and Cin=2 with dilation 1 (got %d, %d)",
                    Cin, dil_w);
    return cnn_conv_tf32_grad(x, y, z, argmax, B, H, W, dil_w, weight, bias, prelu, st);
}

extern "C" int modfx_cnn_conv_dgrad_tf32_f32(const float* dconv, float* dx, int32_t B, int32_t H, int32_t W, int32_t dil_w,
                                             const float* weight_t, void* stream) {
    MODFX_REQUIRE(dconv && dx && weight_t, "NULL pointer");
    MODFX_REQUIRE(B >= 0 && H >= 2 && W >= 1, "bad shape B=%d H=%d W=%d", B, H, W);
    MODFX_REQUIRE(dconv != dx, "dconv and dx must not alias");
    if (const int st = check_conv_shape(B, H, dil_w); st != MODFX_OK || B == 0) return st;
    return cnn_conv_tf32_grad(dconv, dx, nullptr, nullptr, B, H, W, dil_w, weight_t, nullptr, nullptr, as_stream(stream));
}

extern "C" int modfx_cnn_conv_wgrad_tf32_f32(const float* x, const float* dconv, float* dweight, int32_t B, int32_t H,
                                             int32_t W, int32_t Cin, int32_t dil_w, void* workspace, void* stream) {
    MODFX_REQUIRE(x && dconv && dweight && workspace, "NULL pointer");
    MODFX_REQUIRE(B >= 1 && H >= 2 && W >= 1, "bad shape B=%d H=%d W=%d (an empty batch has no gradient)", B, H, W);
    if (const int st = check_conv_shape(B, H, dil_w); st != MODFX_OK) return st;
    if (!(Cin == 64 || (Cin == 2 && dil_w == 1)))
        return fail(MODFX_ERR_UNSUPPORTED, "the weight gradient is built for Cin=64, and Cin=2 with dilation 1 (got %d, %d)",
                    Cin, dil_w);
    float* part = ws_align(workspace);
    cudaStream_t s = as_stream(stream);
    const int64_t n = (int64_t)kCo * Cin * kKH * kKW;
    int st;
    int n_parts;
    if (Cin == 2) {
        const int64_t tiles = (int64_t)B * H * ((W + kW1Tw - 1) / kW1Tw);
        n_parts = (int)std::min<int64_t>(tiles, kW1Parts);
        st = launch(wgrad1_kernel, dim3(n_parts), 256, 0, s, x, dconv, part, B, H, W);
    } else {
        n_parts = cnn_wgrad_splits();
        st = cnn_conv_wgrad_tf32(x, dconv, part, B, H, W, dil_w, s);
    }
    if (st != MODFX_OK) return st;
    return sum_parts(part, n_parts, n, n, dweight, nullptr, s);
}

extern "C" int modfx_cnn_pool_prelu_bwd_f32(const float* dy, const float* z, const uint8_t* argmax, const float* prelu,
                                            float* dconv, float* dbias, float* dprelu, int32_t B, int32_t H, int32_t W,
                                            void* workspace, void* stream) {
    MODFX_REQUIRE(dy && z && argmax && prelu && dconv && dbias && dprelu && workspace, "NULL pointer");
    MODFX_REQUIRE(B >= 1 && H >= 2 && W >= 1 && !(H & 1), "bad shape B=%d H=%d W=%d (H even, an empty batch has no gradient)",
                  B, H, W);
    const int64_t n = (int64_t)B * (H / 2) * W * kCo;
    const int64_t ctas = (n + kBwdChunk - 1) / kBwdChunk;
    MODFX_REQUIRE(ctas <= 0x7fffffff, "too many elements");
    float* part = ws_align(workspace);
    cudaStream_t s = as_stream(stream);
    const int st = launch(pool_prelu_bwd_kernel, dim3((unsigned)ctas), 256, 0, s, dy, z, argmax, prelu, dconv, part, n, W);
    if (st != MODFX_OK) return st;
    return sum_parts(part, (int)ctas, 2 * kCo, kCo, dbias, dprelu, s);
}

extern "C" int modfx_cnn_layernorm_bwd_f32(const float* g, const float* x, const void* stats, float* dx, int32_t B,
                                           int32_t C, int32_t H, int32_t W, float eps, void* workspace, void* stream) {
    MODFX_REQUIRE(g && x && stats && dx && workspace, "NULL pointer");
    MODFX_REQUIRE(B >= 0 && C >= 1 && H >= 1 && W >= 1, "bad shape B=%d C=%d H=%d W=%d", B, C, H, W);
    if (kLnThreads % C != 0) return fail(MODFX_ERR_UNSUPPORTED, "C=%d: the channel count must divide %d", C, kLnThreads);
    if (B == 0) return MODFX_OK;
    MODFX_REQUIRE(B <= 65535, "B=%d: at most 65535 examples per call", B);
    const int64_t P = (int64_t)H * W;
    const int chunks = ln_chunks(P * C);
    const double* fwd = reinterpret_cast<const double*>((reinterpret_cast<uintptr_t>(stats) + 15) & ~(uintptr_t)15);
    double* part = reinterpret_cast<double*>(ws_align(workspace));
    cudaStream_t s = as_stream(stream);
    const int st = launch(ln_bwd_stats_kernel, dim3(chunks, B), kLnThreads, 0, s, g, x, fwd, part, P, C, chunks, eps);
    if (st != MODFX_OK) return st;
    return launch(ln_bwd_apply_kernel, dim3(chunks, B), kLnThreads, 0, s, g, x, fwd, (const double*)part, dx, P, C, chunks,
                  eps);
}

extern "C" int modfx_cnn_head_bwd_f32(const float* latent, const float* out, const float* dout, const float* dlatent,
                                      float* dx, float* dweight, float* dbias, int32_t B, int32_t H, int32_t W, int32_t C,
                                      int32_t L, const float* weight, void* workspace, void* stream) {
    MODFX_REQUIRE(latent && out && dout && dlatent && dx && dweight && dbias && weight && workspace, "NULL pointer");
    MODFX_REQUIRE(B >= 1 && H >= 1 && W >= 1 && C >= 1 && L >= 1, "bad shape (an empty batch has no gradient)");
    if (C > 1024 || L > 1024) return fail(MODFX_ERR_UNSUPPORTED, "C=%d / L=%d too large", C, L);
    MODFX_REQUIRE(B <= 65535, "B too large");
    const int ntw = (W + kHeadW - 1) / kHeadW;
    float* part = ws_align(workspace);
    cudaStream_t s = as_stream(stream);
    const int st = launch(head_bwd_kernel, dim3(ntw, B), 256, (size_t)(C + L) * (kHeadW + 1) * sizeof(float), s, latent, out,
                          dout, dlatent, dx, part, H, W, C, L, weight);
    if (st != MODFX_OK) return st;
    return sum_parts(part, B * ntw, (int64_t)L * C + L, (int64_t)L * C, dweight, dbias, s);
}
