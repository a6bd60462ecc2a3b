// Phaser: 6 first-order TPT all-pass stages sharing one swept cutoff + feedback, as rendered by
// pedalboard.Phaser (juce::dsp::Phaser) at reference mod_extraction/datasets.py:455-482.
// PARITY UNPINNED: pedalboard==0.7.3 / JUCE are not available offline; the arithmetic follows this
// repo's own scalar CPU restatement of the JUCE algorithm (test infrastructure) and is checked against it.
//
// The filter is a 7-state linear time-varying recurrence (6 all-pass states + the fed-back output),
// strictly serial per example: ~100 dependent cycles per sample.  It is parallelised over time with
// a chunked affine scan (DESIGN.md "P1"): phaser_phase_kernel accumulates the oscillator phase in float32
// exactly like the reference (sequentially inside each host block), and phaser_fused_kernel renders one
// 4096-sample segment per CTA out of shared memory -- coefficients, per-sub-chunk affine maps, their chain
// (with the segment's entry state taken from the previous segment's CTA), the re-run, mix and clip.
#include "common.cuh"

namespace modfx {
namespace {

constexpr int kStagesAP = 6;     // all-pass stages (juce::dsp::Phaser numStages)
constexpr int kUpd = 4;          // cutoff update period in samples (maxUpdateCounter)
constexpr int kChunk = 128;      // samples per scan chunk
constexpr int kCtl = kChunk / kUpd;
constexpr int kState = 7;        // s1..s6, lastOutput
constexpr int kMapFloats = 8 * kState;   // 7 columns of Phi + zero-state response
constexpr int kSFloats = 8;      // padded state record

struct PhaserArgs {
    const float* x;
    float* y;
    int N;
    float sr;
    const float *rate, *depth, *centre, *feedback, *mix;
    int block;
    const int32_t* index;
    int n_items;
    int n_ctl;                  // control points per example = ceil(N / 4)
    int n_chunks;               // ceil(N / kChunk)
    const int32_t* start;       // (B,) first delivered sample of each row, or nullptr (0)
    int n_out;                  // delivered samples per row
    float* dry_out;             // (B, n_out) window of the dry input, or nullptr
    int x_compact;              // 1: row `item` of x (a compact (n_items, N) array), 0: row b like every other array
    const int64_t* x_offset;    // (n_items,) or nullptr: x is a packed ragged array, row `item` starts at x + x_offset[item]
                                // and holds start + n_out samples (the prefix that determines the delivered window)
    int n_seg;
    int* ticket;                // 1 int, zero at launch
    int* flags;                 // (n_items, n_seg), zero at launch
    float* rec;                 // (n_items, n_seg, kRec)
    float2* ph;                 // (n_items, n_chunks): phase at the chunk's first control point, phase of the one before
    float* phc;                 // (n_items, n_ctl): phase of every control point; used instead of ph (then nullptr) when
                                // the host block is not a multiple of kChunk samples
};

__device__ __forceinline__ int example_of(const PhaserArgs& a, int item) { return a.index ? a.index[item] : item; }

// One sample of the cascade.  With c = 2G-1 the TPT all-pass (v = G(in-s); y = v+s; s' = y+v; out = 2y-in)
// is out = c*in + (1-c)*s, s' = (1+c)*in - c*s.  Carrying w = (1-c)*s instead of s turns every stage into
// the transposed direct form II of a first-order all-pass -- two dependent FMAs:  out = c*in + w,
// w' = in - c*out  -- at the price of rescaling w by (1-c_new)/(1-c_old) when the coefficient moves (every
// 4th sample).  All kernels keep the states in this form, scaled for the coefficient of the last sample done.
__device__ __forceinline__ float cascade_step(float in, float (&w)[kStagesAP], float c) {
    float v = in;
#pragma unroll
    for (int k = 0; k < kStagesAP; ++k) {
        const float y = fmaf(c, v, w[k]);
        w[k] = fmaf(-c, y, v);
        v = y;
    }
    return v;
}

__device__ __forceinline__ void cascade_retune(float (&w)[kStagesAP], float c_old, float c_new) {
    const float r = __fdividef(1.0f - c_new, 1.0f - c_old);     // 1 - c = 2 (1 - G) in (0.06, 2]: well conditioned
#pragma unroll
    for (int k = 0; k < kStagesAP; ++k) w[k] *= r;
}

// Two runs of the cascade at once, one per half of a float2 (same coefficient): Blackwell's packed FFMA2 does the
// work of two FFMAs in one issue slot, and the map stage is bound by instruction issue.
__device__ __forceinline__ float2 cascade_step2(float2 in, float2 (&w)[kStagesAP], float c) {
    const float2 c2 = make_float2(c, c), nc2 = make_float2(-c, -c);
    float2 v = in;
#pragma unroll
    for (int k = 0; k < kStagesAP; ++k) {
        const float2 y = __ffma2_rn(c2, v, w[k]);
        w[k] = __ffma2_rn(nc2, y, v);
        v = y;
    }
    return v;
}

__device__ __forceinline__ void cascade_retune2(float2 (&w)[kStagesAP], float c_old, float c_new) {
    const float r = __fdividef(1.0f - c_new, 1.0f - c_old);
    const float2 r2 = make_float2(r, r);
#pragma unroll
    for (int k = 0; k < kStagesAP; ++k) w[k] = __fmul2_rn(w[k], r2);
}

// =====================================================================================================================
// Single-pass fused phaser: one kernel reads the audio once and writes the result once.
//
// A CTA owns one SEGMENT of 4096 samples of one example and does everything for it out of shared memory (a pipeline
// of separate kernels, with the audio read twice and the coefficients and per-chunk maps round-tripping HBM, moved 2.3x
// the algorithmic bytes):
//   A  the segment's audio lands in shared memory (one coalesced pass); the float32 oscillator phases of its 1024
//      control points are walked chunk by chunk from chunk-start phases (phaser_phase_kernel below: a few bytes per
//      128 samples, the only thing that is precomputed) -- sequential adds with the wrap at 2 pi, like the restatement.
//      With a host block that is not a multiple of 128 samples a block boundary can fall inside a chunk, and the phase
//      of every control point is precomputed and copied instead;
//   B  the transcendental map phase -> all-pass coefficient c = 2G - 1, all threads;
//   C  per 64-sample sub-chunk the 7 unit-state runs + the zero-state run (two runs per thread, packed FFMA2) give its
//      affine map; lanes = sub-chunks, so a warp's 32 lanes walk 32 different sub-chunks (padded rows: no conflicts);
//   D  the state at the segment start comes from the CTA of the previous segment of the same example through global
//      memory (decoupled look-back: CTAs take their (segment, example) from an atomic ticket in segment-major order, so a
//      predecessor always holds an earlier ticket and is running or done: no deadlock); 8 lanes chain the 64 maps, the
//      exit state is published for the next segment at once;
//   E  64 threads re-run their sub-chunk from its true entry state, mix, clip;
//   F  coalesced store -- optionally only the window [start[b], start[b] + n_out) of the row, together with the same
//      window of the dry input: the random crop of PedalboardPhaserDataset.__getitem__ (datasets.py:445-447).
// Segments past the last needed sample are never touched; a segment wholly before the window ends once its exit state
// is published (no E, no stores).  HBM traffic: 4 B in + 4 B out per sample + 64 B per segment.
// Shared memory is kept under 37.8 KB so that 6 CTAs fit an SM, which the 40 registers of a thread also allow.
constexpr int kSegChunks = 32;                       // 128-sample chunks per segment
constexpr int kSeg = kSegChunks * kChunk;            // 4096 samples
constexpr int kSub = 64;                             // samples per scan sub-chunk
constexpr int kSubs = kSeg / kSub;                   // 64 sub-chunks per segment
constexpr int kSubCtl = kSub / kUpd;                 // 16 control points per sub-chunk
constexpr int kSegCtl = kSeg / kUpd;                 // 1024
constexpr int kFusedThreads = 256;
constexpr int kFusedCtasPerSM = 6;
constexpr int kRec = 8;                              // published state record: w1..w6, lastOutput, c the states are scaled for
constexpr int kFusedSmemFloats = kSubs * (kSub + 1) + kSubs * (kSubCtl + 1) + kSubs * (kMapFloats + 1) + kSubs * kSFloats;
// (+ 1 KB per CTA reserved by the runtime, + the few static bytes, within the 228 KB of an SM)
static_assert(kFusedCtasPerSM * (kFusedSmemFloats * 4 + 128 + 1024) <= 228 * 1024, "phaser_fused_kernel: 6 CTAs per SM");

// Oscillator phases: one thread per (example, host block), juce::dsp::Oscillator semantics.  Control points sit at
// global multiples of 4 samples; inside a host block the phase advances by `inc` per control point with a wrap at 2 pi
// (sequential float32 adds, reproduced exactly); a block starts from the previous block's start phase advanced by
// inc * (control points in that block) in one step.
// The float32 phase is a chain of sequential additions with the wrap at 2 pi, so a host block of 8192 samples is 2048
// dependent steps whatever is done -- what can be kept short is the step: when the increment is below 2 pi (always, for
// an LFO) the wrap is ONE conditional subtraction (p + inc < 4 pi), computed branch-free (add, subtract, select: 12 cycles
// instead of a data-dependent loop), and every block is walked exactly once: the phase of a block's last control point,
// which the next block's first chunk needs as its "control point before", is written there by the thread that walks it.
__device__ __forceinline__ float phase_advance(float p, float inc, float two_pi) {
    const float next = p + inc;
    const float wrapped = next - two_pi;
    return (next >= two_pi) ? wrapped : next;
}

__global__ void __launch_bounds__(128) phaser_phase_kernel(const PhaserArgs a, int n_blocks) {
    const int pair = blockIdx.x * blockDim.x + threadIdx.x;
    if (pair >= a.n_items * n_blocks) return;
    const int item = pair / n_blocks, blk = pair - item * n_blocks;
    const int b = example_of(a, item);
    const int need = a.start ? min(a.N, a.start[b] + a.n_out) : a.N;
    // (a block past the window still has to hand its last phase to nobody: nothing after `need` is rendered)
    if ((int64_t)blk * a.block >= need) return;
    const float two_pi = MODFX_TWO_PI_F;
    const float sr_down = (float)((double)a.sr / (double)kUpd);
    const float inc = a.rate[b] * (two_pi / sr_down);
    float p = 0.0f;
    for (int i = 0; i < blk; ++i) {                  // whole blocks before this one: phase.advance(freq * n_down)
        // a rounded product, like the reference: contracted into an FMA it drifts from it whenever inc * n_down is inexact
        const int n_down = ((i + 1) * a.block + kUpd - 1) / kUpd - (i * a.block + kUpd - 1) / kUpd;
        float next = __fadd_rn(p, __fmul_rn(inc, (float)n_down));
        while (next >= two_pi) next -= two_pi;
        p = next;
    }
    const int s0 = blk * a.block, s1 = min(s0 + a.block, a.N);
    if (a.phc) {                                     // the phase of every control point of the block
        float* out = a.phc + (int64_t)item * a.n_ctl;
        for (int j = (s0 + kUpd - 1) / kUpd; j < (s1 + kUpd - 1) / kUpd; ++j) {
            out[j] = p;
            float next = p + inc;
            while (next >= two_pi) next -= two_pi;
            p = next;
        }
        return;
    }
    const int c0 = s0 / kChunk, c1 = (s1 + kChunk - 1) / kChunk;
    float2* out = a.ph + (int64_t)item * a.n_chunks;
    // a clip's very first control point has no predecessor and the value is unused (all filter states are zero there)
    float prev = 0.0f;
    const bool small = inc < two_pi;
    for (int c = c0; c < c1; ++c) {
        out[c].x = p;
        if (c > c0 || blk == 0) out[c].y = prev;     // the first chunk of a later block: written by the previous block's thread
        if (small) {
#pragma unroll 8
            for (int j = 0; j < kCtl; ++j) {
                prev = p;
                p = phase_advance(p, inc, two_pi);
            }
        } else {
            for (int j = 0; j < kCtl; ++j) {
                prev = p;
                float next = p + inc;
                while (next >= two_pi) next -= two_pi;
                p = next;
            }
        }
    }
    // this block's last control point is the one before the next block's first (only a full block has a successor)
    if (s1 - s0 == a.block && c1 < a.n_chunks) out[c1].y = prev;
}

__device__ __forceinline__ float phaser_coef(float phase, float vol, float ctr, float log_span, float log_min, float w0) {
    float lfo = sinf(phase - MODFX_PI_F) * vol + ctr;
    lfo = fminf(fmaxf(lfo, 0.0f), 1.0f);
    const float fc = exp10f(lfo * log_span + log_min);                   // mapToLog10
    const float g = tanf(w0 * fc);                                       // TPT prewarp
    return 2.0f * (g / (1.0f + g)) - 1.0f;
}

// Stores samples [lo, hi) of a segment (sample n in xs at n - n_base) to row[n - start]: float4 stores where row + (n - start)
// is 16-byte aligned, scalar stores for the at most 3 + 3 samples at the ends (with start % 4 != 0 a float4 there would
// straddle the neighbouring segment, which another CTA stores).
__device__ __forceinline__ void store_window(float* row, const float (*xs)[kSub + 1], int n_base, int start, int lo, int hi,
                                             int tid) {
    const auto at = [&](int n) { const unsigned i = n - n_base; return xs[i / kSub][i % kSub]; };
    if ((reinterpret_cast<uintptr_t>(row) & 15) != 0) {
        for (int n = lo + tid; n < hi; n += kFusedThreads) row[n - start] = at(n);
        return;
    }
    const int v0 = min(lo + ((start - lo) & 3), hi), v1 = max(hi - ((hi - start) & 3), v0);
    for (int n = v0 + 4 * tid; n < v1; n += 4 * kFusedThreads)
        *reinterpret_cast<float4*>(row + (n - start)) = make_float4(at(n), at(n + 1), at(n + 2), at(n + 3));
    if (tid < v0 - lo) row[lo + tid - start] = at(lo + tid);
    if (tid < hi - v1) row[v1 + tid - start] = at(v1 + tid);
}

__global__ void __launch_bounds__(kFusedThreads, kFusedCtasPerSM) phaser_fused_kernel(const PhaserArgs a) {
    extern __shared__ __align__(16) float sm[];
    float(*xs)[kSub + 1] = reinterpret_cast<float(*)[kSub + 1]>(sm);                        // [64][65] audio, then output
    float(*cs)[kSubCtl + 1] = reinterpret_cast<float(*)[kSubCtl + 1]>(sm + kSubs * (kSub + 1));   // [64][17] col 0: coefficient before
    float(*Ms)[kMapFloats + 1] = reinterpret_cast<float(*)[kMapFloats + 1]>(sm + kSubs * (kSub + 1) + kSubs * (kSubCtl + 1));   // [64][57]
    float(*Ss)[kSFloats] = reinterpret_cast<float(*)[kSFloats]>(sm + kSubs * (kSub + 1) + kSubs * (kSubCtl + 1) + kSubs * (kMapFloats + 1));
    float* phs = reinterpret_cast<float*>(Ms);                           // [1024 + 1] phases (dead before the maps are written)
    __shared__ int tile_s;
    __shared__ float entry[kRec];
    __shared__ float coef_k[5];                                          // log_min, log_span, w0, vol, ctr of phaser_coef
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) tile_s = atomicAdd(a.ticket, 1);
    __syncthreads();
    const int tile = tile_s;
    const int seg = tile / a.n_items, item = tile - seg * a.n_items;     // segment-major: predecessors hold earlier tickets
    const int b = example_of(a, item);
    const int start = a.start ? a.start[b] : 0;
    const int need = min(a.N, start + a.n_out);
    const int n_base = seg * kSeg;
    if (n_base >= need) return;
    const float* xr = a.x_offset ? a.x + a.x_offset[item] : a.x + (int64_t)(a.x_compact ? item : b) * a.N;
    const int row_len = a.x_offset ? need : a.N;                          // samples that exist in this row

    // ---- A: audio + oscillator phases
    const bool vec = ((reinterpret_cast<uintptr_t>(xr) & 15) == 0) && (n_base + kSeg <= row_len);
    if (vec) {                                                            // 16-byte loads, 4 per thread
#pragma unroll
        for (int k = 0; k < kSeg / 4 / kFusedThreads; ++k) {
            const int i4 = tid + k * kFusedThreads;
            const float4 v = __ldg(reinterpret_cast<const float4*>(xr + n_base) + i4);
            float* d = &xs[i4 >> 4][(i4 & 15) << 2];
            d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
        }
    } else {
        for (int i = tid; i < kSeg; i += kFusedThreads) {
            const int n = n_base + i;
            xs[i / kSub][i % kSub] = (n < row_len) ? __ldg(xr + n) : 0.0f;
        }
    }
    if (tid == kFusedThreads - 1) {                                       // the per-example constants of B, once per CTA
        const float f_lo = 20.0f;
        const double f_hi_d = (0.49 * (double)a.sr < 20000.0) ? 0.49 * (double)a.sr : 20000.0;
        const float log_min = log10f(f_lo), log_span = log10f((float)f_hi_d) - log_min;
        coef_k[0] = log_min;
        coef_k[1] = log_span;
        coef_k[2] = MODFX_PI_F / a.sr;
        coef_k[3] = a.depth[b] * 0.5f;
        coef_k[4] = (log10f(a.centre[b]) - log_min) / log_span;
    }
    const float two_pi = MODFX_TWO_PI_F;
    if (a.phc) {                                                          // precomputed: copy them
        const float* pr = a.phc + (int64_t)item * a.n_ctl;
        for (int i = tid; i <= kSegCtl; i += kFusedThreads) {
            const int j = seg * kSegCtl - 1 + i;                          // i = 0: the control point before the segment
            phs[i] = (j >= 0 && j < a.n_ctl) ? pr[j] : 0.0f;
        }
    } else if (tid < kSegChunks) {
        const int chunk = seg * kSegChunks + tid;
        const float sr_down = (float)((double)a.sr / (double)kUpd);
        const float inc = a.rate[b] * (two_pi / sr_down);
        float2 pp = (chunk < a.n_chunks) ? a.ph[(int64_t)item * a.n_chunks + chunk] : make_float2(0.0f, 0.0f);
        if (tid == 0) phs[0] = pp.y;                                      // control point before the segment
        float p = pp.x;
        if (inc < two_pi) {
#pragma unroll 8
            for (int q = 0; q < kCtl; ++q) {
                phs[1 + tid * kCtl + q] = p;
                p = phase_advance(p, inc, two_pi);
            }
        } else {
            for (int q = 0; q < kCtl; ++q) {
                phs[1 + tid * kCtl + q] = p;
                float next = p + inc;
                while (next >= two_pi) next -= two_pi;
                p = next;
            }
        }
    }
    __syncthreads();
    // ---- B: phase -> all-pass coefficient
    {
        const float log_min = coef_k[0], log_span = coef_k[1], w0 = coef_k[2], vol = coef_k[3], ctr = coef_k[4];
        float cv[(kSegCtl + 1 + kFusedThreads - 1) / kFusedThreads];
#pragma unroll
        for (int k = 0; k < (kSegCtl + 1 + kFusedThreads - 1) / kFusedThreads; ++k) {
            const int j = tid + k * kFusedThreads;                        // j = 0: the control point before the segment
            cv[k] = (j <= kSegCtl) ? phaser_coef(phs[j], vol, ctr, log_span, log_min, w0) : 0.0f;
        }
        __syncthreads();                                                  // phs aliases Ms: all reads done before cs / Ms are written
#pragma unroll
        for (int k = 0; k < (kSegCtl + 1 + kFusedThreads - 1) / kFusedThreads; ++k) {
            const int j = tid + k * kFusedThreads;
            if (j <= kSegCtl) {
                if (j >= 1) cs[(j - 1) / kSubCtl][1 + (j - 1) % kSubCtl] = cv[k];
                if (j % kSubCtl == 0 && j < kSegCtl) cs[j / kSubCtl][0] = cv[k];     // coefficient before sub-chunk j / 16
            }
        }
    }
    __syncthreads();
    const float fbk = a.feedback[b];
    // ---- C: affine map of every sub-chunk (runs 2p, 2p+1 per thread; run 6 = unit lastOutput, run 7 = zero state + audio)
    {
        const int pair = warp >> 1, sc = ((warp & 1) << 5) | lane;
        float2 s[kStagesAP];
#pragma unroll
        for (int k = 0; k < kStagesAP; ++k) s[k] = make_float2((2 * pair == k) ? 1.0f : 0.0f, (2 * pair + 1 == k) ? 1.0f : 0.0f);
        float2 out_prev = make_float2(0.0f, 0.0f);
        const float2 nfb = make_float2(-fbk, -fbk);
        float c_cur = cs[sc][0];
        int g0 = 0;
        if (pair == 3) {
            // unit lastOutput = out_prev of 1 / feedback: fed as u = -1 by hand for the first sample (finite for feedback 0);
            // both runs start with zero all-pass states, so nothing to retune before the first control group
            const float c0 = cs[sc][1];
            out_prev = cascade_step2(make_float2(-1.0f, xs[sc][0]), s, c0);
#pragma unroll
            for (int q = 1; q < kUpd; ++q)
                out_prev = cascade_step2(__ffma2_rn(nfb, out_prev, make_float2(0.0f, xs[sc][q])), s, c0);
            c_cur = c0;
            g0 = 1;
        }
#pragma unroll 2
        for (int g = g0; g < kSubCtl; ++g) {
            const float c = cs[sc][1 + g];
            cascade_retune2(s, c_cur, c);
            c_cur = c;
#pragma unroll
            for (int q = 0; q < kUpd; ++q) {
                const float2 u = (pair == 3) ? __ffma2_rn(nfb, out_prev, make_float2(0.0f, xs[sc][g * kUpd + q]))
                                             : __fmul2_rn(nfb, out_prev);
                out_prev = cascade_step2(u, s, c);
            }
        }
        float* m = &Ms[sc][2 * pair * kState];
#pragma unroll
        for (int k = 0; k < kStagesAP; ++k) {
            m[k] = s[k].x;
            m[kState + k] = s[k].y;
        }
        m[6] = out_prev.x * fbk;
        m[kState + 6] = out_prev.y * fbk;
    }
    __syncthreads();
    // ---- D: entry state of the segment (look-back), entry state of every sub-chunk, exit state published.
    // Three short passes instead of one chain of 64 dependent steps: (1) every warp composes the 8 maps of its group
    // into one, all groups at once; (2) warp 0 takes the segment's entry state from the previous segment's CTA and
    // chains the 8 group maps; (3) every warp chains its 8 sub-chunks from its group's entry state.
    // Pass 3 never reads the last map of a group (it would give the next group's entry), so pass 1 leaves the group map
    // in that row, and pass 2 leaves a group's entry state in the state row of its first sub-chunk.
    {
        // (1) lane = (row i = lane >> 3 and i + 4, column r = lane & 7) of the running product [Phi | z], in registers;
        // element (j, r) is in lane ((j & 3) << 3) | r
        const int r = lane & 7, i0 = lane >> 3, i1 = i0 + 4;
        float g0, g1;
        {
            const float* m = Ms[warp * 8];
            g0 = m[r * kState + i0];
            g1 = (i1 < kState) ? m[r * kState + i1] : 0.0f;
        }
#pragma unroll 1
        for (int k = 1; k < 8; ++k) {
            const float* m = Ms[warp * 8 + k];
            float a0 = (r == 7) ? m[7 * kState + i0] : 0.0f;
            float a1 = (r == 7 && i1 < kState) ? m[7 * kState + i1] : 0.0f;
#pragma unroll
            for (int j = 0; j < kState; ++j) {
                const float cj = __shfl_sync(0xffffffffu, (j < 4) ? g0 : g1, ((j & 3) << 3) | r);
                a0 = fmaf(m[j * kState + i0], cj, a0);
                if (i1 < kState) a1 = fmaf(m[j * kState + i1], cj, a1);
            }
            g0 = a0;
            g1 = a1;
        }
        __syncwarp();                                                     // every lane is done with the group's last map
        float* g = Ms[warp * 8 + 7];
        g[r * kState + i0] = g0;
        if (i1 < kState) g[r * kState + i1] = g1;
    }
    __syncthreads();
    if (warp == 0) {
        float* rec = a.rec + ((int64_t)item * a.n_seg + seg) * kRec;
        if (seg > 0) {
            const int* flag = a.flags + (int64_t)item * a.n_seg + seg - 1;
            if (lane == 0) {
                while (atomicAdd(const_cast<int*>(flag), 0) == 0) __nanosleep(64);
                __threadfence();
            }
            __syncwarp();
            if (lane < kRec) entry[lane] = __ldcg(rec - kRec + lane);
        } else if (lane < kRec) {
            entry[lane] = 0.0f;
        }
        __syncwarp();
        // (2) the predecessor left its all-pass states scaled for ITS last coefficient, which is this segment's cs[0][0]
        const int i = lane & 7, ii = (i < kState) ? i : 0;
        float sv = (i < kState) ? entry[i] : 0.0f;
        if (lane < 8) {
#pragma unroll 1
            for (int gq = 0; gq < 8; ++gq) {
                Ss[gq * 8][i] = sv;
                const float* m = Ms[gq * 8 + 7];
                float acc = m[7 * kState + ii];
#pragma unroll
                for (int r = 0; r < kState; ++r) acc = fmaf(m[r * kState + ii], __shfl_sync(0xffu, sv, r, 8), acc);
                sv = (i < kState) ? acc : 0.0f;
            }
            if (i < kState) rec[i] = sv;
            else rec[7] = cs[kSubs - 1][kSubCtl];
            __threadfence();
        }
        __syncwarp();
        if (lane == 0) atomicExch(a.flags + (int64_t)item * a.n_seg + seg, 1);
    }
    // a segment wholly before the window owed its successor the exit state, nothing else (CTA-uniform)
    if (n_base + kSeg <= start) return;
    // delivered samples of this segment: [lo, hi)
    const int lo = max(n_base, start), hi = min(n_base + kSeg, need);
    // the window of the dry input goes out while warp 0 chains (xs still holds the audio)
    if (a.dry_out) store_window(a.dry_out + (int64_t)b * a.n_out, xs, n_base, start, lo, hi, tid);
    __syncthreads();
    // (3) entry state of every sub-chunk: each warp chains its group (8 lanes, lane i < 7 owns state component i)
    if (lane < 8) {
        const int i = lane, ii = (i < kState) ? i : 0;
        float sv = (i < kState) ? Ss[warp * 8][i] : 0.0f;
#pragma unroll 1
        for (int k = 0; k < 7; ++k) {
            const int sc = warp * 8 + k;
            const float* m = Ms[sc];
            float acc = m[7 * kState + ii];
#pragma unroll
            for (int r = 0; r < kState; ++r) acc = fmaf(m[r * kState + ii], __shfl_sync(0xffu, sv, r, 8), acc);
            sv = (i < kState) ? acc : 0.0f;
            Ss[sc + 1][i] = sv;
        }
    }
    __syncthreads();
    // ---- E: re-run every sub-chunk from its true entry state, mix and clip (datasets.py:472)
    if (tid < kSubs) {
        const int sc = tid;
        float s[kStagesAP];
#pragma unroll
        for (int k = 0; k < kStagesAP; ++k) s[k] = Ss[sc][k];
        float last = Ss[sc][6];
        const float wet = a.mix[b], dry = 1.0f - a.mix[b];
        float c_cur = cs[sc][0];
#pragma unroll 2
        for (int g = 0; g < kSubCtl; ++g) {
            const float c = cs[sc][1 + g];
            cascade_retune(s, c_cur, c);
            c_cur = c;
#pragma unroll
            for (int q = 0; q < kUpd; ++q) {
                const float in = xs[sc][g * kUpd + q];
                const float out = cascade_step(in - last, s, c);
                last = out * fbk;
                xs[sc][g * kUpd + q] = fminf(fmaxf(fmaf(wet, out, dry * in), -1.0f), 1.0f);
            }
        }
    }
    __syncthreads();
    // ---- F: coalesced store of the delivered window
    float* yr = a.y + (int64_t)b * a.n_out;
    if (start == 0 && n_base + kSeg <= a.n_out && ((reinterpret_cast<uintptr_t>(yr) & 15) == 0)) {
#pragma unroll
        for (int k = 0; k < kSeg / 4 / kFusedThreads; ++k) {
            const int i4 = tid + k * kFusedThreads;
            const float* d = &xs[i4 >> 4][(i4 & 15) << 2];
            reinterpret_cast<float4*>(yr + n_base)[i4] = make_float4(d[0], d[1], d[2], d[3]);
        }
    } else {
        store_window(yr, xs, n_base, start, lo, hi, tid);
    }
}

int64_t align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

}  // namespace
}  // namespace modfx

using namespace modfx;

extern "C" int64_t modfx_phaser_workspace_bytes(int32_t B, int64_t N) {
    if (B <= 0 || N <= 0) return 0;
    const int64_t n_ctl = (N + kUpd - 1) / kUpd, n_chunks = (N + kChunk - 1) / kChunk;
    const int64_t n_seg = (N + kSeg - 1) / kSeg;
    const int64_t phase_bytes = (n_ctl * 4 > n_chunks * 8) ? n_ctl * 4 : n_chunks * 8;     // phc or ph, per row
    return 256 + align_up((int64_t)B * n_seg * 4, 256) + align_up((int64_t)B * n_seg * kRec * 4, 256) +
           align_up((int64_t)B * phase_bytes, 256) + 256;
}

namespace {

// The entry points fill in the pointers, sr, block, index, n_items and what a cropped call adds; the rest is set here.
int phaser_launch(PhaserArgs a, int32_t B, int64_t N, int64_t n_out, void* workspace, void* stream) {
    MODFX_REQUIRE(a.x && a.y && a.rate && a.depth && a.centre && a.feedback && a.mix, "NULL pointer");
    MODFX_REQUIRE(B >= 0 && N >= 1 && N < (1ll << 30), "bad shape B=%d N=%lld", B, (long long)N);
    MODFX_REQUIRE(n_out >= 1 && n_out <= N, "bad output window n_out=%lld (row length %lld)", (long long)n_out, (long long)N);
    MODFX_REQUIRE(a.sr > 0.0f, "sample rate must be positive");
    if (a.block <= 0) a.block = 8192;       // pedalboard's default buffer_size
    a.N = (int)N;
    a.n_out = (int)n_out;
    if (!a.index) a.n_items = B;
    if (a.n_items == 0) return MODFX_OK;
    MODFX_REQUIRE(a.n_items > 0 && workspace, "workspace is NULL or n_items=%d", a.n_items);
    a.n_ctl = (int)((N + kUpd - 1) / kUpd);
    a.n_chunks = (int)((N + kChunk - 1) / kChunk);
    cudaStream_t s = as_stream(stream);
    char* w = static_cast<char*>(workspace);
    const int n_blocks = (int)((N + a.block - 1) / a.block);

    a.n_seg = (int)((N + kSeg - 1) / kSeg);
    a.ticket = reinterpret_cast<int*>(w);                                     w += 256;
    a.flags = reinterpret_cast<int*>(w);
    const int64_t flag_bytes = align_up((int64_t)a.n_items * a.n_seg * 4, 256);  w += flag_bytes;
    a.rec = reinterpret_cast<float*>(w);                                      w += align_up((int64_t)a.n_items * a.n_seg * kRec * 4, 256);
    if (a.block % kChunk == 0) a.ph = reinterpret_cast<float2*>(w);
    else a.phc = reinterpret_cast<float*>(w);
    MODFX_CUDA_OK(cudaMemsetAsync(workspace, 0, (size_t)(256 + flag_bytes), s));
    const int pairs = a.n_items * n_blocks;
    phaser_phase_kernel<<<(pairs + 127) / 128, 128, 0, s>>>(a, n_blocks);
    const int64_t tiles = (int64_t)a.n_items * a.n_seg;
    MODFX_REQUIRE(tiles < (1ll << 31), "too many segments in one call");
    MODFX_CUDA_OK(cudaFuncSetAttribute(phaser_fused_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                       cudaSharedmemCarveoutMaxShared));
    phaser_fused_kernel<<<(unsigned)tiles, kFusedThreads, sizeof(float) * kFusedSmemFloats, s>>>(a);
    MODFX_CUDA_OK(cudaGetLastError());
    return MODFX_OK;
}

}  // namespace

extern "C" int modfx_phaser_f32(const float* x, float* y, int32_t B, int64_t N, float sr, const float* rate_hz,
                                const float* depth, const float* centre_hz, const float* feedback,
                                const float* mix, int32_t block, const int32_t* example_index, int32_t n_items,
                                void* workspace, void* stream) {
    PhaserArgs a{};
    a.x = x; a.y = y; a.sr = sr;
    a.rate = rate_hz; a.depth = depth; a.centre = centre_hz; a.feedback = feedback; a.mix = mix;
    a.block = block; a.index = example_index; a.n_items = n_items;
    return phaser_launch(a, B, N, N, workspace, stream);
}

extern "C" int modfx_phaser_crop_f32(const float* x, int32_t x_compact, float* y, float* dry_out, int32_t B, int64_t N,
                                     int64_t n_out, const int32_t* start, float sr, const float* rate_hz, const float* depth,
                                     const float* centre_hz, const float* feedback, const float* mix, int32_t block,
                                     const int32_t* example_index, int32_t n_items, void* workspace, void* stream) {
    MODFX_REQUIRE(start, "start is NULL");
    MODFX_REQUIRE(!x_compact || example_index, "x_compact needs an example_index list");
    PhaserArgs a{};
    a.x = x; a.y = y; a.sr = sr;
    a.rate = rate_hz; a.depth = depth; a.centre = centre_hz; a.feedback = feedback; a.mix = mix;
    a.block = block; a.index = example_index; a.n_items = n_items;
    a.start = start; a.dry_out = dry_out; a.x_compact = x_compact ? 1 : 0;
    return phaser_launch(a, B, N, n_out, workspace, stream);
}

extern "C" int modfx_phaser_crop_packed_f32(const float* x, const int64_t* x_offset, float* y, float* dry_out, int32_t B,
                                            int64_t N_max, int64_t n_out, const int32_t* start, float sr, const float* rate_hz,
                                            const float* depth, const float* centre_hz, const float* feedback, const float* mix,
                                            int32_t block, const int32_t* example_index, int32_t n_items, void* workspace,
                                            void* stream) {
    MODFX_REQUIRE(start && x_offset, "start or x_offset is NULL");
    MODFX_REQUIRE(example_index, "a packed x needs an example_index list (row i belongs to example example_index[i])");
    PhaserArgs a{};
    a.x = x; a.y = y; a.sr = sr;
    a.rate = rate_hz; a.depth = depth; a.centre = centre_hz; a.feedback = feedback; a.mix = mix;
    a.block = block; a.index = example_index; a.n_items = n_items;
    a.start = start; a.dry_out = dry_out; a.x_compact = 1; a.x_offset = x_offset;
    return phaser_launch(a, B, N_max, n_out, workspace, stream);
}
