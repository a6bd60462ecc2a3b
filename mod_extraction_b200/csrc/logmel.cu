// Log-mel front end of the lfo_2dcnn extractor, fused into one kernel:
//   reflect-pad -> frame -> periodic Hann -> 1024-point real FFT -> |.|^2 -> banded mel -> clip -> log
// Replaces Spectral2DCNN.spectrogram (torchaudio MelSpectrogram) + tr.clip + tr.log, reference
// mod_extraction/models.py:170-175,199,207-208.
//
// Why no tensor cores (DESIGN.md "M1"): a dense DFT is 17x the flops of the FFT and needs 3xTF32 or
// 6xBF16 error compensation to hold the 1e-4 log-mel tolerance; the mel matrix is 0.77 % dense.
// Both are not "genuine dense contractions", so the FFT runs in registers on the FP32 pipes
// (fft_core.h) and the mel projection is a <=14-tap banded sum.
//
// Work split: a work item is (row, group of 8 consecutive frames); a CTA of 4 warps walks a list of items.
// Large batches (>= 16 rows per SM) launch one CTA per row and let the hardware place CTAs as others retire;
// smaller ones launch 4 persistent CTAs per SM that stride over all items, so even a handful of rows fills
// the chip (all items cost the same; the tables are set up once per CTA either way).
// Per item: the audio span of the 8 frames is brought into shared memory by ONE bulk copy (TMA engine +
// mbarrier) issued while the previous item is still being transformed, every warp transforms two adjacent
// frames (sharing the window, the twiddles and 12 of 16 sample reads between them), the 8 power spectra
// meet in shared memory and the mel/log stage writes 8 consecutive frames of every mel row (32 B segments
// of the (R, n_mels, n_frames) output).
//
// Shared memory per CTA (bytes): pass-1 twiddles 4096 | exchange 4 x 8448 | span 11264 | mel table ~5100.
// The power spectra and the staged outputs live inside the exchange regions (each is dead while the other
// is live) and the window is read through L1, which is what lets 4 CTAs share an SM.  The kernel is bound
// by the shared-memory data pipe (~70 % of its wavefront rate, ncu) with the FP32 pipe at ~45 %.
#include "common.cuh"
#include "fft_core.h"

#include <algorithm>

namespace modfx {
namespace {

constexpr int kNfft = 1024;
constexpr int kBins = kNfft / 2 + 1;     // 513
constexpr int kWarps = 4;
constexpr int kThreads = kWarps * kWarp;
constexpr int kCtasPerSm = 4;            // 128 registers, ~54 KB of shared memory each
constexpr int kFB = 2 * kWarps;          // frames per work item
constexpr int kEStride = 33;             // padded row of the pass-1 -> pass-2 exchange buffer
constexpr int kRegion = 2 * 32 * kEStride;            // floats per warp region: float2 Ew[32][33] = 8448 B
// inside a region, once pass 2 has pulled the exchange data into registers:
//   floats [0, 1026)      power spectra of the warp's two frames, Pw[bin][2]
//   floats [1088, 2112)   staged outputs of 128 mel bands x 8 frames (band m lives in region m >> 7)
constexpr int kStageOff = 1088;
constexpr int kStageBands = (kRegion - kStageOff) / kFB;       // 128
static_assert(kBins * 2 <= kStageOff && (kStageOff % 4) == 0 && (kRegion % 4) == 0, "region layout");

struct LogMelArgs {
    const float* x;
    float* out;
    int64_t R, T;
    int hop, n_mels, n_frames;
    const float* window;
    const int32_t* fb_start;
    const int32_t* fb_count;
    const float* fb_weight;
    int fb_stride;
    int fb_taps;         // capacity of the compact in-smem weight table (>= sum of fb_count)
    float eps;
    int apply_log;
    int64_t x_row_stride, out_row_stride;
    const int32_t* row_index;
    int iters;           // work items (groups of kFB frames) per row
    int n_items;         // R * iters
    int by_row;          // 1: CTA c walks the items of row c (large batches); 0: items c, c + grid, ... (persistent)
    int n_rounds;        // ceil(n_mels / kThreads): rounds of the mel stage
};

__device__ __forceinline__ int reflect_index(int i, int T) {
    // torch.nn.functional.pad(mode="reflect"): -1 -> 1, T -> T-2
    if (i < 0) i = -i;
    if (i >= T) i = 2 * (T - 1) - i;
    return max(0, min(i, T - 1));      // frames past the end of a short clip are computed but never stored
}

// log(x) for x >= eps > 0 (never denormal after the clip): one MUFU.LG2 and one multiply, <= 3 ulp
__device__ __forceinline__ float fast_log(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y * 0.69314718055994530942f;
}

__device__ __forceinline__ unsigned smem_addr(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_addr(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
    unsigned done;
    do {
        asm volatile(
            "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
            : "=r"(done)
            : "r"(smem_addr(bar)), "r"(parity)
            : "memory");
    } while (!done);
}

// Stage samples [s0, s0 + span) of one row (center=True: reflect-padded at both ends) into sbuf.  The part
// that exists in the row goes as ONE bulk copy (TMA engine, completion on `bar`), so the staging costs the
// LSU / shared-memory pipe nothing; only the reflected ends of a row (first and last item of 44) and rows
// that are not 16-byte aligned take scalar loads.  Returns whether a bulk copy was issued (CTA-uniform).
__device__ __forceinline__ bool stage_span(float* sbuf, const float* xr, int s0, int T, int span, int tid,
                                           unsigned long long* bar) {
    const bool aligned = ((reinterpret_cast<uintptr_t>(xr) & 15) == 0) && ((s0 & 3) == 0);
    int lo = s0 + span, hi = s0 + span;          // [lo, hi): samples that go by bulk copy
    if (aligned) {
        lo = max(s0, 0);
        hi = s0 + ((min(s0 + span, T) - s0) & ~3);
        if (hi <= lo) lo = hi = s0 + span;
    }
    const bool bulk = hi > lo;
    if (bulk && tid == 0) {
        const unsigned bytes = (unsigned)(hi - lo) * 4u;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_addr(bar)), "r"(bytes)
                     : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                         smem_addr(sbuf + (lo - s0))),
                     "l"(xr + lo), "r"(bytes), "r"(smem_addr(bar))
                     : "memory");
    }
    for (int i = tid; i < lo - s0; i += kThreads) sbuf[i] = xr[reflect_index(s0 + i, T)];
    for (int i = hi - s0 + tid; i < span; i += kThreads) sbuf[i] = xr[reflect_index(s0 + i, T)];
    return bulk;
}

__global__ void __launch_bounds__(kThreads, kCtasPerSm) logmel_kernel(const LogMelArgs a) {
    extern __shared__ __align__(16) float smem[];
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    const int T = (int)a.T;
    const int span = (kFB - 1) * a.hop + kNfft;      // samples staged per item

    unsigned long long* bar = reinterpret_cast<unsigned long long*>(smem);         // completion of the bulk copy
    float2* tw1 = reinterpret_cast<float2*>(smem + 4);          // [16][32]  exp(-2 pi i n2 k1 / 512) as (cos, sin)
    float* E = smem + 4 + 2 * 512;                              // kWarps regions, see kRegion
    float2* Ew = reinterpret_cast<float2*>(E + warp * kRegion);
    float* sbuf = E + kWarps * kRegion;                         // [span rounded up to 4]
    float* melw = sbuf + ((span + 3) & ~3);                     // [fb_taps] band weights, bands back to back
    unsigned short* moff = reinterpret_cast<unsigned short*>(melw + a.fb_taps);    // [n_mels + 1] first weight of band m
    unsigned short* mstart = moff + a.n_mels + 2;                                  // [n_mels] first FFT bin of band m

    if (tid == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    const float* win = a.window;        // 4 KB read by every CTA: stays in L1, costs no shared memory
    for (int i = tid; i < 512; i += kThreads) {
        const int k1 = i >> 5, n2 = i & 31;
        float s, c;
        sincospif(-(float)(n2 * k1) / 256.0f, &s, &c);
        tw1[i] = make_float2(c, s);
    }
    // compact copy of the banded mel table (<= 14 taps per band for the reference configuration):
    // counts -> exclusive prefix (every thread sums the counts below its band from shared memory)
    for (int m = tid; m < a.n_mels; m += kThreads) mstart[m] = (unsigned short)min(a.fb_count[m], 65535);
    __syncthreads();
    for (int m = tid; m <= a.n_mels; m += kThreads) {
        int off = 0;
        for (int i = 0; i < m; ++i) off += mstart[i];
        moff[m] = (unsigned short)min(off, a.fb_taps);
    }
    __syncthreads();
    for (int m = tid; m < a.n_mels; m += kThreads) {
        mstart[m] = (unsigned short)a.fb_start[m];
        const int o = moff[m], c = moff[m + 1] - o;
        for (int j = 0; j < c; ++j) melw[o + j] = a.fb_weight[(int64_t)m * a.fb_stride + j];
    }
    // split twiddle of this lane's bins k = k1 + 16 k2: w_k = w_{k1} * w_{16 k2}
    float c1, s1;
    sincospif((float)(lane & 15) / 512.0f, &s1, &c1);

    const int w_step = a.by_row ? 1 : (int)gridDim.x;
    int w = a.by_row ? (int)blockIdx.x * a.iters : (int)blockIdx.x;
    const int w_end = a.by_row ? min(w + a.iters, a.n_items) : a.n_items;
    if (w >= w_end) return;
    int item = w / a.iters;
    int it = w - item * a.iters;
    int64_t row = a.row_index ? a.row_index[item] : item;
    // (the two __syncthreads of the table set-up above order the barrier init before its first use)
    bool bulk = stage_span(sbuf, a.x + row * a.x_row_stride, it * kFB * a.hop - kNfft / 2, T, span, tid, bar);
    unsigned parity = 0;

    while (true) {
        const int t0 = it * kFB;
        float* orow = a.out + row * a.out_row_stride;
        // ---- the audio span of frames t0 .. t0+7 was staged while the previous item was in flight
        __syncthreads();                // scalar part of the staging
        if (bulk) {
            mbar_wait(bar, parity);     // bulk part
            parity ^= 1;
        }

        const int lf = 2 * warp;                        // local index of this warp's first frame
        const bool active = t0 + lf < a.n_frames;
        float2 v[32];
        if (active) {
            // ---- pass 1: lane = n2; 16-point FFT over n1 of z[32 n1 + n2], both frames at once so that the
            // window and twiddle reads are shared; with the reference hop of 256 = 4 * 64 the second frame's
            // samples for n1 are the first frame's for n1 + 4, so only 20 of the 32 sample reads remain
            float2 u0[16], u1[16];
            {
                const float* fr = sbuf + lf * a.hop + 2 * lane;
#pragma unroll
                for (int n1 = 0; n1 < 16; ++n1) u0[n1] = *reinterpret_cast<const float2*>(fr + 64 * n1);
                if (a.hop == 256) {
#pragma unroll
                    for (int n1 = 0; n1 < 12; ++n1) u1[n1] = u0[n1 + 4];
#pragma unroll
                    for (int n1 = 12; n1 < 16; ++n1) u1[n1] = *reinterpret_cast<const float2*>(fr + 256 + 64 * n1);
                } else {
#pragma unroll
                    for (int n1 = 0; n1 < 16; ++n1) u1[n1] = *reinterpret_cast<const float2*>(fr + a.hop + 64 * n1);
                }
#pragma unroll
                for (int n1 = 0; n1 < 16; ++n1) {
                    const float2 w2 = __ldg(reinterpret_cast<const float2*>(win + 64 * n1 + 2 * lane));
                    u0[n1] = c_mul2(u0[n1], w2);
                    u1[n1] = c_mul2(u1[n1], w2);
                }
            }
            fft_dif<16>(u0);
            fft_dif<16>(u1);
#pragma unroll
            for (int k1 = 0; k1 < 16; ++k1) {
                const float2 t = tw1[k1 * 32 + lane];
                Ew[k1 * kEStride + lane] = c_mul_tw(u0[BitRev<16>::of(k1)], t.x, t.y);
                Ew[(16 + k1) * kEStride + lane] = c_mul_tw(u1[BitRev<16>::of(k1)], t.x, t.y);
            }
        }
        __syncthreads();        // every warp is done with sbuf: the next item's span may land in it
        // ---- next item of this CTA; its span is fetched behind pass 2 and the mel stage
        w += w_step;
        const bool more = w < w_end;
        int64_t row_n = 0;
        int it_n = 0;
        if (more) {
            if (a.by_row) {                         // same row, next group of frames
                it_n = it + 1;
                row_n = row;
            } else {
                const int item_n = w / a.iters;
                it_n = w - item_n * a.iters;
                row_n = a.row_index ? a.row_index[item_n] : item_n;
            }
            bulk = stage_span(sbuf, a.x + row_n * a.x_row_stride, it_n * kFB * a.hop - kNfft / 2, T, span, tid, bar);
        }
        if (active) {
            // ---- pass 2: lane = (frame f, k1); 32-point FFT over n2
#pragma unroll
            for (int n2 = 0; n2 < 32; ++n2) v[n2] = Ew[lane * kEStride + n2];
            __syncwarp();       // the power spectra below overwrite this warp's exchange rows
            fft_dif<32>(v);
            // ---- real-FFT split + power.  Bins k and 512-k share all their intermediate terms
            // (X[512-k] uses the same sums / differences with two signs flipped), so each pair is
            // computed once: this lane handles its own bins k = k1 + 16 k2 for k2 < 16 together with the
            // mirror bins 512-k, which belong to the partner lane (f, 16-k1) at k2' = 31-k2.
            constexpr float C64[32] = MODFX_C64;
            constexpr float S64[32] = MODFX_S64;
            const int f = lane >> 4, k1 = lane & 15;
            const int partner = (lane & 16) | ((16 - k1) & 15);
            const int k1m = (16 - k1) & 15;                 // k1 of the mirror bins
            // Pw[bin][2]: the 32 lanes of a store hit 32 different banks for the own and the mirror bins alike
            float* Pown = reinterpret_cast<float*>(Ew) + 2 * k1 + f;
            // mirror bins: 512 - k = k1m + 16 (31 - k2) for k1 != 0 and 16 (32 - k2) for k1 == 0, i.e. one base
            // pointer minus k2 * 16 rows in both cases
            float* Pmir = reinterpret_cast<float*>(Ew) + 2 * ((k1 == 0) ? 512 : (k1m + 496)) + f;
#pragma unroll
            for (int k2 = 0; k2 < 16; ++k2) {
                const int own = BitRev<32>::of(k2);
                const int src_other = BitRev<32>::of(31 - k2);          // Z[512-k] lives in the partner lane
                const int src_self = BitRev<32>::of((32 - k2) & 31);    // ... or in this lane when k1 == 0
                float2 p = make_float2(__shfl_sync(kFull, v[src_other].x, partner),
                                       __shfl_sync(kFull, v[src_other].y, partner));
                if (k1 == 0) p = v[src_self];
                // split twiddle (cos, sin)(2 pi k / 1024) = (c1 + i s1) * (C + i S), k = k1 + 16 k2
                const float2 cs = c_mul_tw(make_float2(c1, s1), C64[k2], S64[k2]);
                const float2 pw = rfft_split_power_pair(v[own], p, cs.x, cs.y);
                Pown[32 * k2] = pw.x;
                if (!(k1 == 0 && k2 == 0)) Pmir[-32 * k2] = pw.y;
            }
            if (k1 == 0) {
                // k = 0 was written above (X[0] = Re Z[0] + Im Z[0]); Nyquist and the self-paired k = 256
                const float d = v[0].x - v[0].y;                        // X[512] = Re Z[0] - Im Z[0]
                Pown[2 * 512] = d * d;
                const float2 zq = v[BitRev<32>::of(16)];                // Z[256]: its own mirror, X[256] = conj Z[256]
                Pown[2 * 256] = zq.x * zq.x + zq.y * zq.y;
            }
        }
        __syncthreads();

        // ---- banded mel projection + clip + log.  A thread owns a whole mel band per round (bands in
        // ascending order in even rounds, descending in odd ones, so that the 1..14 taps of a thread's low and
        // high band balance) and all 8 frames of the item: per tap one weight, one 8-byte read of the power
        // row of every warp, eight FMAs.  (A schedule that gives every half-warp 16 different bank pairs was
        // measured: no bank conflicts, but 64 instead of 40 tap iterations per item and 5 % slower overall.)
        {
            for (int k = 0; k < a.n_rounds; ++k) {
                const int m = k * kThreads + ((k & 1) ? (kThreads - 1 - tid) : tid);
                if (m >= a.n_mels) continue;
                const int o = moff[m], cnt = moff[m + 1] - o;
                const float* wt = melw + o;
                float acc[kFB];
#pragma unroll
                for (int t = 0; t < kFB; ++t) acc[t] = 0.0f;
                const float2* pr = reinterpret_cast<const float2*>(E) + (int)mstart[m];
#pragma unroll 2
                for (int j = 0; j < cnt; ++j) {
                    const float wj = wt[j];
#pragma unroll
                    for (int g = 0; g < kWarps; ++g) {
                        const float2 p = pr[g * (kRegion / 2) + j];
                        acc[2 * g] = fmaf(wj, p.x, acc[2 * g]);
                        acc[2 * g + 1] = fmaf(wj, p.y, acc[2 * g + 1]);
                    }
                }
                // results go through shared memory (the free tail of the exchange regions) so that the
                // global stores below are 32-byte segments instead of 4-byte scatters
                float4 o0, o1;
                if (a.apply_log) {
                    o0 = make_float4(fast_log(fmaxf(acc[0], a.eps)), fast_log(fmaxf(acc[1], a.eps)),
                                     fast_log(fmaxf(acc[2], a.eps)), fast_log(fmaxf(acc[3], a.eps)));
                    o1 = make_float4(fast_log(fmaxf(acc[4], a.eps)), fast_log(fmaxf(acc[5], a.eps)),
                                     fast_log(fmaxf(acc[6], a.eps)), fast_log(fmaxf(acc[7], a.eps)));
                } else {
                    o0 = make_float4(acc[0], acc[1], acc[2], acc[3]);
                    o1 = make_float4(acc[4], acc[5], acc[6], acc[7]);
                }
                // the 16-byte halves are swapped on every other group of 4 bands: conflict-free 16-byte stores
                float4* st = reinterpret_cast<float4*>(E + (m / kStageBands) * kRegion + kStageOff +
                                                       (m % kStageBands) * kFB);
                const int sw = (m >> 2) & 1;
                st[sw] = o0;
                st[sw ^ 1] = o1;
            }
            __syncthreads();
            // 8 consecutive lanes write the 8 frames of one band: one 32-byte segment per band row
            const int live = min(kFB, a.n_frames - t0);
            const int t = tid & (kFB - 1);
            if (t < live) {
                // band m = mb + 16 i lives in region m >> 7 at row m & 127; bit 2 of m (the half swap) is bit 2 of mb
                const int mb = tid >> 3;
                const float* ep = E + kStageOff + mb * kFB + (t ^ (mb & 4));
                float* op = orow + (int64_t)mb * a.n_frames + t0 + t;
                const int64_t ostep = (int64_t)(kThreads / kFB) * a.n_frames;
                static_assert(kStageBands == 128 && kThreads / kFB == 16, "store loop layout");
#pragma unroll 8
                for (int m = mb, i = 0; m < a.n_mels; m += kThreads / kFB, ++i) {
                    *op = *ep;
                    op += ostep;
                    ep += ((i & 7) == 7) ? (kRegion - 7 * 16 * kFB) : 16 * kFB;
                }
            }
        }
        // no barrier here: the next item's first barrier orders these reads of the exchange regions before
        // pass 1 writes them again
        if (!more) break;
        row = row_n;
        it = it_n;
    }
}

// SpecAugment of the reference's training forward (models.py:201-205): torchaudio FrequencyMasking /
// TimeMasking zero one band of mel bins and one band of frames of EVERY row between the mel power and
// clip + log, so in the fused output the masked cells hold log(max(0, eps)).
__global__ void specaugment_fill_kernel(float* __restrict__ out, int64_t n, int n_mels, int n_frames, int f0, int f1,
                                        int t0, int t1, float fill) {
    const int64_t per_row = (int64_t)n_mels * n_frames;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t e = i % per_row;
        const int m = (int)(e / n_frames), t = (int)(e - (int64_t)m * n_frames);
        if ((m >= f0 && m < f1) || (t >= t0 && t < t1)) out[i] = fill;
    }
}

}  // namespace
}  // namespace modfx

using namespace modfx;

extern "C" int modfx_specaugment_fill_f32(float* out, int64_t R, int32_t n_mels, int32_t n_frames, int32_t f0,
                                          int32_t f1, int32_t t0, int32_t t1, float eps, int32_t is_log, void* stream) {
    MODFX_REQUIRE(out, "NULL pointer");
    MODFX_REQUIRE(R >= 0 && n_mels >= 1 && n_frames >= 1, "bad shape");
    MODFX_REQUIRE(0 <= f0 && f0 <= f1 && f1 <= n_mels && 0 <= t0 && t0 <= t1 && t1 <= n_frames, "bad mask bounds");
    MODFX_REQUIRE(eps > 0.0f, "eps must be positive");
    const int64_t n = R * n_mels * (int64_t)n_frames;
    if (n == 0 || (f0 == f1 && t0 == t1)) return MODFX_OK;
    // same arithmetic as the kernel's own log of a clipped zero: lg2.approx(eps) * ln 2
    const float fill = is_log ? log2f(eps) * 0.69314718055994530942f : 0.0f;
    const int grid = (int)std::min<int64_t>((n + 255) / 256, (int64_t)num_sms() * 16);
    return launch(specaugment_fill_kernel, grid, 256, 0, as_stream(stream), out, n, n_mels, n_frames, f0, f1, t0, t1,
                  fill);
}

extern "C" int modfx_logmel_f32(const float* x, float* out, int64_t R, int64_t T, int32_t n_fft, int32_t hop,
                                int32_t n_mels, const float* window, const int32_t* fb_start,
                                const int32_t* fb_count, const float* fb_weight, int32_t fb_stride, int32_t fb_taps,
                                float eps, int32_t apply_log, int64_t x_row_stride, int64_t out_row_stride,
                                const int32_t* row_index, int32_t n_index, void* stream) {
    MODFX_REQUIRE(x && out && window && fb_start && fb_count && fb_weight, "NULL pointer");
    MODFX_REQUIRE(R >= 0 && T >= 1, "bad shape R=%lld T=%lld", (long long)R, (long long)T);
    if (n_fft != kNfft) return fail(MODFX_ERR_UNSUPPORTED, "n_fft=%d (only 1024 is built)", n_fft);
    if (hop < 2 || hop > 512 || (hop & 1))
        return fail(MODFX_ERR_UNSUPPORTED, "hop=%d (even hops in [2, 512] are built)", hop);
    MODFX_REQUIRE(T > n_fft / 2, "reflect padding needs T > n_fft/2 (T=%lld)", (long long)T);   // torch raises too
    MODFX_REQUIRE(T < (1ll << 30), "T too long");
    MODFX_REQUIRE(n_mels >= 1 && fb_stride >= 1 && fb_taps >= 1, "bad mel table");
    if (n_mels > kWarps * kStageBands || fb_taps > 8192)
        return fail(MODFX_ERR_UNSUPPORTED, "mel table too large for shared memory (n_mels=%d taps=%d)", n_mels, fb_taps);
    if (row_index) R = n_index;
    if (R <= 0) return MODFX_OK;
    LogMelArgs a{};
    a.x = x; a.out = out; a.R = R; a.T = T; a.hop = hop; a.n_mels = n_mels;
    a.n_frames = (int)(T / hop) + 1;
    a.window = window; a.fb_start = fb_start; a.fb_count = fb_count; a.fb_weight = fb_weight;
    a.fb_stride = fb_stride; a.eps = eps; a.apply_log = apply_log;
    a.fb_taps = fb_taps;
    a.x_row_stride = x_row_stride > 0 ? x_row_stride : T;
    a.out_row_stride = out_row_stride > 0 ? out_row_stride : (int64_t)n_mels * a.n_frames;
    a.row_index = row_index;
    a.iters = (a.n_frames + kFB - 1) / kFB;
    MODFX_REQUIRE(R * a.iters < (1ll << 31), "too many frames in one call");
    a.n_items = (int)(R * a.iters);
    a.n_rounds = (n_mels + kThreads - 1) / kThreads;
    // Large batches: one CTA per row, placed by the hardware scheduler as CTAs retire (measured 3-4 % faster
    // than the static stride once there are >= 16 rows per SM).  Otherwise persistent CTAs over all items,
    // which fills the chip however few rows there are.
    a.by_row = R >= 16ll * num_sms() ? 1 : 0;
    const int64_t grid = a.by_row ? R : std::min<int64_t>(a.n_items, (int64_t)kCtasPerSm * num_sms());
    const int span = (kFB - 1) * hop + kNfft;
    const size_t smem = sizeof(float) * (size_t)(4 + 2 * 512 + kWarps * kRegion + ((span + 3) & ~3) + fb_taps) +
                        sizeof(unsigned short) * (size_t)(2 * n_mels + 4) + 16;
    MODFX_CUDA_OK(cudaFuncSetAttribute(logmel_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                       cudaSharedmemCarveoutMaxShared));
    return launch(logmel_kernel, (unsigned)grid, kThreads, smem, as_stream(stream), a);
}
