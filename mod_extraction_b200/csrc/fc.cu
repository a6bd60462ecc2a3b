// Flanger / chorus modulated fractional-delay line with feedback (and tremolo).
//
// Replaces MonoFlangerChorusModule.apply_effect (reference mod_extraction/fx.py:72-119), whose
// python loop costs ~105 us per time step.  Bit-exact with it: every float32 operation of the
// reference is one IEEE-RN operation here (explicit __f*_rn intrinsics, never contracted).
//
// Two kernels share the per-sample arithmetic (=> the same bits): fc_cta_kernel (default: a CTA of three producer
// warps + one consumer warp per delay line, for every modulation source) and fc_wide_kernel (a CTA per delay line
// whose every tap lies more than 384 samples back: the chorus); fc_allpass_kernel is the all-pass interpolation mode.
//
// Parallelisation (DESIGN.md "E1"): the recurrence v[n] = x[n] + fb*interp(v[n-kp], v[n-kq]) is
// sequential in time per delay line, but a sample only depends on samples at least
// `near = min(kp,kq)` steps back.  The written values v live in a shared-memory ring indexed by time.
// A tile of 128 samples is rendered in one shot when every dependency falls before the tile (always
// true for chorus, true for flanger while the delay exceeds 128 samples); otherwise 32-sample blocks
// are resolved as "waves" of independent prefixes, and stretches with a delay of a few samples fall
// back to a lock-step serial loop with register forwarding.  Only the schedule changes, never the
// arithmetic of a sample, so the result is identical in all modes.
#include "common.cuh"

namespace modfx {
namespace {

constexpr int kTile = 128;          // samples per tile (4 sub-steps x 32 lanes)
constexpr int kSub = kTile / kWarp; // 4
constexpr int kPollNs = 128;        // producers polling for the consumer: 32 / 100 / 300 ns measured within noise of each other (1.17-1.26 ms), longer leaves more issue slots

struct FcArgs {
    const float* x;
    float* y;
    int B, C, N;
    int Mmin, Mlfo, M;
    int ring_mask;                  // ring size - 1 (power of two >= M + kTile)
    // modulation source
    const float* mod;
    int mod_has_ch;
    int n_lo;
    float up_scale;
    float sr_lo;
    const float* lfo_freq;
    const float* lfo_phase;
    const int32_t* lfo_shape;
    const float* lfo_exp;
    // effect parameters: device array or pre-rounded scalar
    const float* fb_p;    float fb_s;
    const float* mdw_p;   float min_delay_s;   // scalar: f32(mdw * Mmin) computed in double
    const float* width_p; float lfo_delay_s;   // scalar: f32(Mlfo * width) computed in double
    const float* depth_p; float depth_s;
    const float* mix_p;   float mix_s; float omm_s;   // scalar: f32(1.0 - mix) computed in double
    const int32_t* index;
    int n_items;
    int wide;                       // 1: examples that qualify for fc_wide_kernel are rendered there and skipped here
};

enum ModMode { kAudioRate = 0, kControlRate = 1, kDirectLfo = 2 };

struct Coef {
    float A, D0, fb, depth, mix, omm, Mf;
    int M, mask;
};

struct Samp {       // per-sample, per-lane state of the current tile
    float x, fr, omfr;
    int kp;         // distance (in samples, 1..M) to the write that filled tap p
};

__device__ __forceinline__ int kq_of(int kp, int M) { return kp > 1 ? kp - 1 : M; }

// Index arithmetic of fx.py:95-102 for sample n (w = n mod M), in the reference's op order.
__device__ __forceinline__ void fc_index(float m, int w, const Coef& c, float& fr, float& omfr, int& kp) {
    const float d = __fadd_rn(__fmul_rn(c.A, m), c.D0);                 // fx.py:98
    const float t = __fadd_rn(__fsub_rn((float)w, d), c.Mf);            // fx.py:99 (before %)
    float r;
    if (t >= 0.0f && t < c.Mf) r = t;                                   // fmod is exact here
    else if (t >= c.Mf && t < __fadd_rn(c.Mf, c.Mf)) r = __fsub_rn(t, c.Mf);   // Sterbenz: exact
    else r = torch_remainder(t, c.Mf);
    const float pf = floorf(r);
    fr = __fsub_rn(r, pf);                                              // fx.py:100
    int p = (int)pf;                                                    // fx.py:101
    p = max(0, min(p, c.M - 1));
    omfr = __fsub_rn(1.0f, fr);                                         // (1.0 - fraction), fx.py:113
    kp = w - p;
    if (kp <= 0) kp += c.M;     // read-before-write: a tap at the write slot is M samples old
}

// One sample of fx.py:111-118 given the two taps.
__device__ __forceinline__ void fc_sample(const Samp& s, float vp, float vq, const Coef& c, float& v, float& out) {
    const float it = __fadd_rn(__fmul_rn(s.fr, vq), __fmul_rn(s.omfr, vp));   // fx.py:113
    v = __fadd_rn(s.x, __fmul_rn(c.fb, it));                                    // fx.py:114
    const float o = __fadd_rn(s.x, __fmul_rn(c.depth, it));                     // fx.py:115
    float r = __fadd_rn(__fmul_rn(c.omm, s.x), __fmul_rn(c.mix, o));            // fx.py:117
    out = fminf(fmaxf(r, -1.0f), 1.0f);                                         // fx.py:118
}

// ---- cp.async staging of the dry audio (and the audio-rate mod_sig) ---------------------
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void cp_async_4(void* dst, const void* src, int src_bytes) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(smem_u32(dst)), "l"(src), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

// ---- wide path: delay lines whose every tap lies more than a tile back (chorus) ------------------------------
// With a minimum delay of D0 = min_delay_width * Mmin samples (485 for the reference's chorus) a sample never depends on
// the previous kWideTile samples, so a whole CTA can render 384 samples of ONE delay line at a time, with one barrier
// per tile and no producer / consumer hand-off.  Same per-sample arithmetic (the branch-free form of fx.py:95-118 used
// by fc_cta_kernel's producers), so the bits are identical.
// Whether an example qualifies is decided from its parameters and the extremes of its control-rate row by
// wide_pred(), evaluated identically by both kernels: the wide kernel renders the example iff it holds, fc_cta_kernel
// iff it does not.
constexpr int kWideThreads = 128;
constexpr int kWideSub = 3;
constexpr int kWideTile = kWideThreads * kWideSub;      // 384
constexpr int kWideMargin = 4;                          // samples of slack on the delay bound (tap = ceil(delay) +- 1)

__device__ __forceinline__ bool wide_pred(const Coef& c, float m_min, float m_max) {
    const bool coef_ok = (c.A >= 0.0f) && (c.D0 >= 0.0f) && (__fadd_rn(c.A, c.D0) <= c.Mf);
    const float d_min = __fadd_rn(__fmul_rn(c.A, m_min), c.D0);         // the delay is monotone in the modulation
    return coef_ok && (m_min >= 0.0f) && (m_max <= 1.0f) && (d_min >= (float)(kWideTile + kWideMargin));
}

__device__ __forceinline__ void warp_minmax(float& mn, float& mx) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mn = fminf(mn, __shfl_xor_sync(kFull, mn, o));
        mx = fmaxf(mx, __shfl_xor_sync(kFull, mx, o));
    }
}

__device__ __forceinline__ Coef make_coef(const FcArgs& a, int b) {
    Coef c;
    c.M = a.M;
    c.Mf = (float)a.M;
    c.mask = a.ring_mask;
    c.A = a.width_p ? __fmul_rn((float)a.Mlfo, a.width_p[b]) : a.lfo_delay_s;      // fx.py:98
    c.D0 = a.mdw_p ? __fmul_rn(a.mdw_p[b], (float)a.Mmin) : a.min_delay_s;          // fx.py:97
    c.fb = a.fb_p ? a.fb_p[b] : a.fb_s;
    c.depth = a.depth_p ? a.depth_p[b] : a.depth_s;
    c.mix = a.mix_p ? a.mix_p[b] : a.mix_s;
    c.omm = a.mix_p ? __fsub_rn(1.0f, c.mix) : a.omm_s;                             // fx.py:117
    return c;
}

__global__ void __launch_bounds__(kWideThreads) fc_wide_kernel(const FcArgs a, int wide_mask) {
    extern __shared__ __align__(16) float ring[];           // written samples, indexed by time & wide_mask
    __shared__ float red[2][kWideThreads / kWarp];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int item = blockIdx.x / a.C;
    const int ch = blockIdx.x - item * a.C;
    const int b = a.index ? a.index[item] : item;
    const int N = a.N;
    Coef c = make_coef(a, b);
    const float* lo = a.mod + (int64_t)b * a.n_lo;

    // extremes of the control-rate row -> does this example belong to the wide path?
    float mn = INFINITY, mx = -INFINITY;
    for (int i = tid; i < a.n_lo; i += kWideThreads) {
        const float v = __ldg(lo + i);
        mn = fminf(mn, v);
        mx = fmaxf(mx, v);
        if (!(v == v)) mx = INFINITY;                       // NaN: never eligible
    }
    warp_minmax(mn, mx);
    if (lane == 0) { red[0][warp] = mn; red[1][warp] = mx; }
    __syncthreads();
    mn = red[0][0]; mx = red[1][0];
#pragma unroll
    for (int w = 1; w < kWideThreads / kWarp; ++w) { mn = fminf(mn, red[0][w]); mx = fmaxf(mx, red[1][w]); }
    if (!wide_pred(c, mn, mx)) return;                      // left to fc_cta_kernel (CTA-uniform)

    const float* xs = a.x + ((int64_t)b * a.C + ch) * (int64_t)N;
    float* ys = a.y + ((int64_t)b * a.C + ch) * (int64_t)N;
    for (int i = tid; i <= wide_mask; i += kWideThreads) ring[i] = 0.0f;            // fx.py:92
    int wk[kWideSub];
    float xv[kWideSub];
#pragma unroll
    for (int k = 0; k < kWideSub; ++k) {
        const int n = k * kWideThreads + tid;
        wk[k] = n % c.M;
        xv[k] = (n < N) ? __ldg(xs + n) : 0.0f;
    }
    const int last_lo = a.n_lo - 1;
    __syncthreads();
    for (int n0 = 0; n0 < N; n0 += kWideTile) {
        float v[kWideSub], out[kWideSub];
#pragma unroll
        for (int k = 0; k < kWideSub; ++k) {
            const int n = n0 + k * kWideThreads + tid;
            // x100 upsample (util.py:15-29) and index arithmetic (fx.py:95-102), branch-free: 0 <= mod <= 1 and the
            // parameter bounds keep (w - d) + M inside [0, 2M)
            const float src = __fmul_rn(a.up_scale, (float)min(n, N - 1));
            const int i0 = min((int)src, last_lo);
            const float l1 = __fsub_rn(src, (float)i0);
            const float l0 = __fsub_rn(1.0f, l1);
            const float m = __fmaf_rn(l0, __ldg(lo + i0), __fmul_rn(l1, __ldg(lo + min(i0 + 1, last_lo))));
            const float d = __fadd_rn(__fmul_rn(c.A, m), c.D0);                     // fx.py:98
            const float t = __fadd_rn(__fsub_rn((float)wk[k], d), c.Mf);            // fx.py:99
            const float r = (t >= c.Mf) ? __fsub_rn(t, c.Mf) : t;                   // % M
            const float pf = floorf(r);
            Samp sm;
            sm.x = xv[k];
            sm.fr = __fsub_rn(r, pf);                                                // fx.py:100
            sm.omfr = __fsub_rn(1.0f, sm.fr);
            int kp = wk[k] - (int)pf;                                                // fx.py:101
            if (kp <= 0) kp += c.M;
            sm.kp = kp;
            const float vp = ring[(n - kp) & wide_mask];
            const float vq = ring[(n - kq_of(kp, c.M)) & wide_mask];
            fc_sample(sm, vp, vq, c, v[k], out[k]);
        }
#pragma unroll
        for (int k = 0; k < kWideSub; ++k) {
            const int n = n0 + k * kWideThreads + tid;
            if (n < N) {
                ring[n & wide_mask] = v[k];
                ys[n] = out[k];
            }
            const int nn = n + kWideTile;                   // next tile's dry sample
            xv[k] = (nn < N) ? __ldg(xs + nn) : 0.0f;
            wk[k] += kWideTile;
            if (wk[k] >= c.M) wk[k] -= c.M;
            if (wk[k] >= c.M) wk[k] %= c.M;
        }
        __syncthreads();        // this tile's samples are in the ring before the next tile reads its taps
    }
}

// ---- CTA per delay line, warp-specialised: the latency-oriented schedule (DESIGN.md "E1") ------------------
// A single warp per delay line spends ~1400 cycles per 128-sample tile because it does everything in turn: index
// arithmetic, x100 upsample, taps, the recurrence, the mix.  Only the recurrence v[n] = x[n] + fb * it[n] is
// sequential; everything else is a function of n alone.  Here a CTA of 4 warps owns one delay line:
//   * 3 PRODUCER warps run ahead, a 128-sample tile each in turn: they fill a ring of tile slots with
//     {x, fraction, 1 - fraction, shared-memory indices of the two taps} per sample (fx.py:95-102 + the upsample of
//     util.py:15-29) and a dependency summary {min / max tap distance, slack} per 32-sample block; the same warp later
//     takes the interpolated values the consumer left in the slot and does fx.py:115-118 + the store;
//   * 1 CONSUMER warp only resolves the recurrence -- a single warp issues at most one instruction per cycle, so what it
//     executes per sample is kept to the loads of the two taps, the five float operations of fx.py:113-114 and two
//     stores: 128 samples in one shot when no tap falls inside the tile, four one-wave blocks when no tap falls inside
//     its own block, else per block one wave / waves / a register-history serial run.
// Hand-off through two kinds of shared-memory counters (tiles filled per producer, tiles done by the consumer) written
// with st.release and polled with ld.acquire; both sides cache what they last read, so in steady state a tile costs
// no synchronisation at all (an mbarrier try_wait costs ~90 cycles even when the phase is already complete).
// A slot is refilled by the warp that drained it.  The consumer role rotates over the warp index with the CTA index
// (warp w runs on scheduler w % 4: otherwise every consumer of an SM would share one scheduler).
// Same per-sample arithmetic => same bits.
constexpr int kCtaProd = 3;
constexpr int kCtaThreads = (kCtaProd + 1) * kWarp;     // 128
constexpr int kNT = 2 * kCtaProd;                       // tile slots in flight (two per producer)
constexpr int kXDepth = 4;                              // dry-audio tiles in flight per producer warp (cp.async)
constexpr int kLoSmemMax = 2048;                        // in-kernel synthesised control rows staged in shared memory up to this many points
constexpr int kSlotFloats = 4 * kTile + kTile + 8;      // float4 coef[128] | it[128] | slack of the four blocks, schedule codes
constexpr int kSerialK = 8;                             // register-history serial runs cover tap distances up to this (+1)

__device__ __forceinline__ void st_release(int* p, int v) {
    asm volatile("st.release.cta.shared::cta.u32 [%0], %1;\n" ::"r"(smem_u32(p)), "r"(v) : "memory");
}
__device__ __forceinline__ int ld_acquire(const int* p) {
    int v;
    asm volatile("ld.acquire.cta.shared::cta.u32 %0, [%1];\n" : "=r"(v) : "r"(smem_u32(p)) : "memory");
    return v;
}

// Lock-step serial run over `ngroups` groups of 4 consecutive samples (whole 32-sample blocks) whose tap distances are
// all K or K+1.  A pre-pass (one sample per lane, see serial_records) has turned the per-sample records into
// {x, cA, cB, cC}: it = cA * v[n-K+1] + (cB * v[n-K] + cC * v[n-K-1]) with (cA, cB, cC) = (fraction, 1 - fraction, 0)
// for a tap distance of K and (0, fraction, 1 - fraction) for K+1 -- the product with the zero coefficient adds an
// exact zero, so the sum has the bits of fx.py:113 -- and for K = 1, where the far tap of a sub-sample delay is the
// stale sample M back, {x, cA, cB, S}: it = cA * v[n-1] + (cB * v[n-2] + S), S = fraction * stale or 0.  No select is
// left in the loop: the previous sample enters through one multiply, so a sample costs the four dependent float
// operations of fx.py:113-114.  A real loop (the body stays in the instruction cache); the records of the next group
// are pulled into registers ahead of the dependent chain, the taps come from history REGISTERS, results leave as two
// 16-byte stores per group from one lane.

template <int K>
__device__ __noinline__ void serial_run(float* __restrict__ ring, int mask, int nb, const float4* __restrict__ coef,
                                        float fb, float* __restrict__ it_out, int lane, int ngroups) {
    // Four groups of 4 samples per loop iteration over ONE register window w[]: for a group with base `o`,
    // w[o + 3 - u] is sample u of the group and w[o + 3 + j] the sample j before the group, so the tap of sample u at
    // distance d is w[o + 3 - u + d] whether it lies before the group or inside it.  The groups work at o = 12, 8, 4, 0
    // (each one's history starts with its predecessor's outputs, no copy), the window slides by 16 once per iteration and
    // the coefficient records of consecutive groups live in two register sets that swap roles -- the moves that a one-group loop spends on shifting the
    // window and on "current = next" every 4 samples sat right behind the dependent chain, where nothing hides them.
    float w[K + 17];
#pragma unroll
    for (int j = 1; j <= K + 1; ++j) w[15 + j] = ring[(nb - j) & mask];
    float4* dst = reinterpret_cast<float4*>(ring + (nb & mask));    // tiles are 128-aligned, the ring a multiple of 128
    float4* ito = reinterpret_cast<float4*>(it_out);
    float4 ca[4], cb[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) ca[u] = coef[u];
#define MODFX_SERIAL_GROUP(O, CF, ITS)                                                                              \
    _Pragma("unroll") for (int u = 0; u < 4; ++u) {                                                                 \
        const float4 cf = CF[u];                                                                                    \
        const float far = (K == 1) ? cf.w : __fmul_rn(cf.w, w[(O) + 3 - u + K + 1]);                                \
        const float it = __fadd_rn(__fmul_rn(cf.y, w[(O) + 3 - u + (K == 1 ? 1 : K - 1)]),                          \
                                   __fadd_rn(__fmul_rn(cf.z, w[(O) + 3 - u + (K == 1 ? 2 : K)]), far)); /* fx.py:113 */ \
        ITS[u] = it;                                                                                                \
        w[(O) + 3 - u] = __fadd_rn(cf.x, __fmul_rn(fb, it));                                            /* fx.py:114 */ \
    }
    // one group: prefetch the records of group G + 1 into NEXT, resolve group G from CUR at window base O, store
#define MODFX_SERIAL_STEP(G, O, CUR, NEXT)                                                                          \
    {                                                                                                               \
        const int gn = min((G) + 1, last);                                                                          \
        _Pragma("unroll") for (int u = 0; u < 4; ++u) NEXT[u] = coef[4 * gn + u];                                   \
        float its[4];                                                                                               \
        MODFX_SERIAL_GROUP(O, CUR, its)                                                                             \
        if (lane == 0) {            /* every lane holds the same values: one lane stores */                         \
            dst[G] = make_float4(w[(O) + 3], w[(O) + 2], w[(O) + 1], w[(O)]);                                       \
            ito[G] = make_float4(its[0], its[1], its[2], its[3]);                                                   \
        }                                                                                                           \
    }
    const int last = ngroups - 1;
    int g = 0;
#pragma unroll 1
    for (; g + 4 <= ngroups; g += 4) {
        MODFX_SERIAL_STEP(g, 12, ca, cb)
        MODFX_SERIAL_STEP(g + 1, 8, cb, ca)
        MODFX_SERIAL_STEP(g + 2, 4, ca, cb)
        MODFX_SERIAL_STEP(g + 3, 0, cb, ca)
#pragma unroll
        for (int k = K + 16; k >= 16; --k) w[k] = w[k - 16];
    }
    // (the callers hand over whole 32-sample blocks, 8 groups each, so nothing is left; kept for other group counts)
#pragma unroll 1
    for (; g < ngroups; ++g) {
        MODFX_SERIAL_STEP(g, 12, ca, cb)
#pragma unroll
        for (int u = 0; u < 4; ++u) ca[u] = cb[u];
#pragma unroll
        for (int k = K + 16; k >= 16; --k) w[k] = w[k - 4];
    }
#undef MODFX_SERIAL_STEP
#undef MODFX_SERIAL_GROUP
}

// Where fc_cta_kernel's producers take the modulation from: memory (an audio-rate or control-rate mod_sig), or the LFO
// parameters -- synthesised into shared memory first (control rows up to kLoSmemMax points) or evaluated where it is
// needed (every sample of kDirectLfo, the two taps of every sample of a longer control row).
enum Synth { kRead = 0, kStaged = 1, kAtTap = 2 };

// lfo_value out of line, for the two taps of kAtTap control rows: inlined twice into the producer loop, its
// double-precision cos makes ptxas spill
__device__ __noinline__ float lfo_at(LfoDesc d, int i) { return lfo_value(d, i); }

template <int MODE, int SYNTH>
__global__ void __launch_bounds__(kCtaThreads) fc_cta_kernel(const FcArgs a, int lo_smem) {
    extern __shared__ __align__(16) float smem[];
    int* filled = reinterpret_cast<int*>(smem);                            // [kCtaProd] tiles filled by producer p
    int* done = filled + 4;                                                // tiles resolved by the consumer
    float* red = smem + 8;                                                 // [8]
    float* slots = smem + 16;                                              // [kNT][kSlotFloats]
    float* xstage = slots + kNT * kSlotFloats;                             // [kCtaProd][kXDepth][128] dry audio in flight
    float* mstage = xstage + kCtaProd * kXDepth * kTile;                   // same for an audio-rate mod_sig
    float* lo_s = mstage + ((MODE == kAudioRate) ? kCtaProd * kXDepth * kTile : 0);   // [lo_smem] synthesised control row (or none)
    float* ring = lo_s + lo_smem;                                          // written samples, indexed by time & mask
    const int ring_w = (int)(ring - smem);                                 // word index of the ring inside smem[]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int item = blockIdx.x / a.C;
    const int ch = blockIdx.x - item * a.C;
    const int b = a.index ? a.index[item] : item;
    const int N = a.N;
    const Coef c = make_coef(a, b);
    const int mask = c.mask;
    const float* lo = (MODE == kControlRate) ? (SYNTH == kStaged ? lo_s : a.mod + (int64_t)b * a.n_lo) : nullptr;

    if (MODE == kControlRate && SYNTH == kRead && a.wide) {
        // examples whose every tap lies more than a wide tile back were rendered by fc_wide_kernel (same predicate)
        float mn = INFINITY, mx = -INFINITY;
        for (int i = tid; i < a.n_lo; i += kCtaThreads) {
            const float v = __ldg(lo + i);
            mn = fminf(mn, v);
            mx = fmaxf(mx, v);
            if (!(v == v)) mx = INFINITY;
        }
        warp_minmax(mn, mx);
        if (lane == 0) { red[warp] = mn; red[4 + warp] = mx; }
        __syncthreads();
        mn = fminf(fminf(red[0], red[1]), fminf(red[2], red[3]));
        mx = fmaxf(fmaxf(red[4], red[5]), fmaxf(red[6], red[7]));
        if (wide_pred(c, mn, mx)) return;                  // CTA-uniform
    }
    if (tid < 8) filled[tid] = 0;
    for (int i = tid; i <= mask; i += kCtaThreads) ring[i] = 0.0f;                   // fx.py:92
    LfoDesc lfo{};
    if (SYNTH != kRead) lfo = make_lfo_desc(a.lfo_freq[b], a.lfo_phase[b], a.lfo_shape[b], a.lfo_exp ? a.lfo_exp[b] : 1.0f, a.sr_lo);
    if (SYNTH == kStaged)
        for (int i = tid; i < a.n_lo; i += kCtaThreads) lo_s[i] = lfo_value(lfo, i);
    __syncthreads();

    const int ntiles = (N + kTile - 1) / kTile;
    const float* xs = a.x + ((int64_t)b * a.C + ch) * (int64_t)N;
    float* ys = a.y + ((int64_t)b * a.C + ch) * (int64_t)N;
    const int cw = blockIdx.x & 3;                          // the consumer's warp index rotates with the CTA index

    if (warp != cw) {
        // ================================ producers ================================
        const int p = (warp - cw - 1) & 3;                  // 0 .. 2
        const float* ms = nullptr;
        if (MODE == kAudioRate) ms = a.mod + (a.mod_has_ch ? ((int64_t)b * a.C + ch) : (int64_t)b) * (int64_t)N;
        float* xq = xstage + p * kXDepth * kTile;
        float* mq = mstage + p * kXDepth * kTile;
        const bool coef_ok = (c.A >= 0.0f) && (c.D0 >= 0.0f) && (__fadd_rn(c.A, c.D0) <= c.Mf);
        const int last_lo = a.n_lo - 1;
        // dry audio (and the audio-rate mod_sig) of this warp's next kXDepth tiles travels through cp.async
#pragma unroll
        for (int d = 0; d < kXDepth - 1; ++d) {
#pragma unroll
            for (int k = 0; k < kSub; ++k) {
                const int n = (p + d * kCtaProd) * kTile + k * kWarp + lane;
                if (n < N) {
                    cp_async_4(xq + d * kTile + k * kWarp + lane, xs + n, 4);
                    if (MODE == kAudioRate) cp_async_4(mq + d * kTile + k * kWarp + lane, ms + n, 4);
                }
            }
            cp_async_commit();
        }
        int wk[kSub];
#pragma unroll
        for (int k = 0; k < kSub; ++k) wk[k] = (p * kTile + k * kWarp + lane) % c.M;
        const int wstep = (kCtaProd * kTile) % c.M;
        int q = 0;                                          // stage of this warp's current tile
        int done_seen = 0;
        for (int t = p; t < ntiles + kNT; t += kCtaProd) {
            float* slot = slots + (t % kNT) * kSlotFloats;
            float4* cs = reinterpret_cast<float4*>(slot);
            float* itb = slot + 4 * kTile;
            int* meta = reinterpret_cast<int*>(slot + 5 * kTile);
            if (t >= kNT) {
                // ---- epilogue of tile t - kNT, which lived in this slot: fx.py:115-118 ----
                const int td = t - kNT;
                while (done_seen <= td) {
                    done_seen = ld_acquire(done);
                    if (done_seen <= td) __nanosleep(kPollNs);   // leave the issue slots to the warps that have work
                }
#pragma unroll
                for (int k = 0; k < kSub; ++k) {
                    const float x = cs[k * kWarp + lane].x;
                    const float it = itb[k * kWarp + lane];
                    const float o = __fadd_rn(x, __fmul_rn(c.depth, it));                       // fx.py:115
                    const float r = __fadd_rn(__fmul_rn(c.omm, x), __fmul_rn(c.mix, o));        // fx.py:117
                    const int nj = td * kTile + k * kWarp + lane;
                    if (nj < N) ys[nj] = fminf(fmaxf(r, -1.0f), 1.0f);                          // fx.py:118
                }
                __syncwarp();
            }
            if (t < ntiles) {
                {   // keep kXDepth - 1 tiles in flight
                    int qs = q + kXDepth - 1;
                    if (qs >= kXDepth) qs -= kXDepth;
#pragma unroll
                    for (int k = 0; k < kSub; ++k) {
                        const int n = (t + (kXDepth - 1) * kCtaProd) * kTile + k * kWarp + lane;
                        if (n < N) {
                            cp_async_4(xq + qs * kTile + k * kWarp + lane, xs + n, 4);
                            if (MODE == kAudioRate) cp_async_4(mq + qs * kTile + k * kWarp + lane, ms + n, 4);
                        }
                    }
                    cp_async_commit();
                }
                cp_async_wait<kXDepth - 1>();               // every lane reads back only what it copied itself
                // straight-line arithmetic for the four 32-sample blocks of the tile (independent chains interleave);
                // the exact-remainder path of fc_index is taken afterwards for the whole tile if any sample needs it
                float xv[kSub], mv[kSub], frv[kSub], omv[kSub];
                int kpv[kSub];
                bool bad = !coef_ok;
#pragma unroll
                for (int k = 0; k < kSub; ++k) {
                    const int n = t * kTile + k * kWarp + lane;
                    const bool mine = n < N;
                    xv[k] = mine ? xq[q * kTile + k * kWarp + lane] : 0.0f;
                    float m;
                    if (MODE == kAudioRate) {
                        m = mine ? mq[q * kTile + k * kWarp + lane] : 0.0f;
                    } else if (MODE == kDirectLfo) {
                        m = lfo_value(lfo, min(n, N - 1));
                    } else {
                        const float src = __fmul_rn(a.up_scale, (float)min(n, N - 1));          // util.py:15-29
                        const int i0 = min((int)src, last_lo);
                        const int i1 = min(i0 + 1, last_lo);
                        const float l1 = __fsub_rn(src, (float)i0);
                        const float l0 = __fsub_rn(1.0f, l1);
                        float m0, m1;
                        if (SYNTH == kRead) { m0 = __ldg(lo + i0); m1 = __ldg(lo + i1); }
                        else if (SYNTH == kStaged) { m0 = lo[i0]; m1 = lo[i1]; }
                        else { m0 = lfo_at(lfo, i0); m1 = lfo_at(lfo, i1); }
                        m = __fmaf_rn(l0, m0, __fmul_rn(l1, m1));
                    }
                    mv[k] = m;
                    bad = bad || !(m >= 0.0f && m <= 1.0f);
                    // 0 <= d <= M, so (w - d) + M lies in [0, 2M): the remainder is one conditional subtraction
                    const float d = __fadd_rn(__fmul_rn(c.A, m), c.D0);                         // fx.py:98
                    const float tt = __fadd_rn(__fsub_rn((float)wk[k], d), c.Mf);               // fx.py:99
                    const float r = (tt >= c.Mf) ? __fsub_rn(tt, c.Mf) : tt;                    // % M
                    const float pf = floorf(r);
                    frv[k] = __fsub_rn(r, pf);                                                   // fx.py:100
                    omv[k] = __fsub_rn(1.0f, frv[k]);
                    int kp = wk[k] - min((int)pf, c.M - 1);                                      // fx.py:101
                    if (kp <= 0) kp += c.M;
                    kpv[k] = kp;
                }
                if (__any_sync(kFull, bad)) {
#pragma unroll
                    for (int k = 0; k < kSub; ++k) fc_index(mv[k], wk[k], c, frv[k], omv[k], kpv[k]);
                }
                int slk[kSub];
#pragma unroll
                for (int k = 0; k < kSub; ++k) {
                    const int n = t * kTile + k * kWarp + lane;
                    const int kp = kpv[k];
                    // where the two taps live: word indices into smem[] (the consumer loads smem[ip], smem[iq])
                    const int ip = ring_w + ((n - kp) & mask);
                    const int iq = ring_w + ((n - kq_of(kp, c.M)) & mask);
                    cs[k * kWarp + lane] = make_float4(xv[k], frv[k], omv[k], __int_as_float((ip << 16) | iq));
                    // slack > 0: no sample of the block has a tap inside the block (near = min(kp, kq))
                    slk[k] = __reduce_min_sync(kFull, (n < N) ? (max(kp - 1, 1) - lane) : 0x7fffffff);
                    wk[k] += wstep;
                    if (wk[k] >= c.M) wk[k] -= c.M;
                }
                // Blocks with a tap inside themselves (rare outside the low-delay stretches, where the producers idle
                // anyway) are classified here, off the consumer's critical path: 1..kSerialK = every tap distance is
                // K or K+1 (register-history serial run; the records are rewritten to the select-free form
                // {x, cA, cB, cC} of serial_run), 14 = waves, 15 = generic serial run; 0 = no tap inside the block.
                unsigned codes = 0;
                if (min(min(slk[0], slk[1]), min(slk[2], slk[3])) <= 0) {
#pragma unroll
                    for (int k = 0; k < kSub; ++k) {
                        if (slk[k] <= 0) {                  // warp-uniform
                            const int nb = t * kTile + k * kWarp;
                            const bool mine = nb + lane < N;
                            const int kp = kpv[k];
                            const int kmin = __reduce_min_sync(kFull, mine ? kp : 0x7fffffff);
                            const int kmax = __reduce_max_sync(kFull, mine ? kp : 0);
                            unsigned code;
                            // (M >= a tile: a K = 1 run takes the stale sample M back of each of its samples before it
                            // starts, so that sample must precede the run, and a run covers up to a whole tile)
                            if (nb + kWarp <= N && kmax - kmin <= 1 && kmin <= kSerialK && c.M >= kTile) {
                                code = (unsigned)kmin;
                                const bool sel = kp == kmin;        // tap distance K (else K + 1)
                                float4 o;
                                o.x = xv[k];
                                if (kmin == 1) {    // taps (previous, stale M back) or (2 back, previous); the consumer
                                    o.y = sel ? omv[k] : frv[k];    // multiplies .w by the stale sample before the run
                                    o.z = sel ? 0.0f : omv[k];
                                    o.w = sel ? frv[k] : 0.0f;
                                } else {
                                    o.y = sel ? frv[k] : 0.0f;
                                    o.z = sel ? omv[k] : frv[k];
                                    o.w = sel ? 0.0f : omv[k];
                                }
                                cs[k * kWarp + lane] = o;
                            } else {
                                code = (kmin >= 3) ? 14u : 15u;
                            }
                            codes |= code << (4 * k);
                        }
                    }
                }
                if (lane == 0) {
                    reinterpret_cast<int4*>(meta)[0] = make_int4(slk[0], slk[1], slk[2], slk[3]);
                    meta[4] = (int)codes;
                }
                __syncwarp();
                if (lane == 0) st_release(filled + p, t / kCtaProd + 1);
                if (++q == kXDepth) q = 0;
            }
        }
        cp_async_wait<0>();
        return;
    }

    // ================================ consumer ================================
    int avail = 0;                                          // tiles [0, avail) are known to be filled
    int sl = 0;
    for (int t = 0; t < ntiles; ++t) {
        while (t >= avail) {
            const int f0 = ld_acquire(filled), f1 = ld_acquire(filled + 1), f2 = ld_acquire(filled + 2);
            avail = min(min(kCtaProd * f0, kCtaProd * f1 + 1), kCtaProd * f2 + 2);
        }
        float* slot = slots + sl * kSlotFloats;
        float4* cs = reinterpret_cast<float4*>(slot);
        float* itb = slot + 4 * kTile;
        const int4 sk4 = *reinterpret_cast<const int4*>(slot + 5 * kTile);
        const int sk[kSub] = {sk4.x, sk4.y, sk4.z, sk4.w};
        const int n0 = t * kTile;
        const bool whole = n0 + kTile <= N;
        bool shot = whole, waves1 = whole;                  // no tap inside the tile / inside its own block
#pragma unroll
        for (int j = 0; j < kSub; ++j) {
            shot = shot && (sk[j] - j * kWarp > 0);
            waves1 = waves1 && (sk[j] > 0);
        }
        if (waves1) {
            float4 r[kSub];
#pragma unroll
            for (int j = 0; j < kSub; ++j) r[j] = cs[j * kWarp + lane];
            float* wr = ring + ((n0 + lane) & mask);        // tiles are 128-aligned, the ring a multiple of 128
            if (shot) {
                // ---- no tap of these 128 samples falls inside them: one shot ----
                float vp[kSub], vq[kSub];
#pragma unroll
                for (int j = 0; j < kSub; ++j) {
                    const unsigned pk = __float_as_uint(r[j].w);
                    vp[j] = smem[pk >> 16];
                    vq[j] = smem[pk & 0xffffu];
                }
#pragma unroll
                for (int j = 0; j < kSub; ++j) {
                    const float it = __fadd_rn(__fmul_rn(r[j].y, vq[j]), __fmul_rn(r[j].z, vp[j]));    // fx.py:113
                    wr[j * kWarp] = __fadd_rn(r[j].x, __fmul_rn(c.fb, it));                             // fx.py:114
                    itb[j * kWarp + lane] = it;
                }
            } else if (sk[1] > kWarp && sk[3] > kWarp) {
                // ---- every tap lies more than 64 samples back within a pair of blocks (delays of 64 .. 128 samples): two
                // waves of 64 samples, half the dependent steps of the four-wave path below ----
#pragma unroll
                for (int h = 0; h < kSub; h += 2) {
                    float vp[2], vq[2];
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        const unsigned pk = __float_as_uint(r[h + j].w);
                        vp[j] = smem[pk >> 16];
                        vq[j] = smem[pk & 0xffffu];
                    }
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        const float it = __fadd_rn(__fmul_rn(r[h + j].y, vq[j]), __fmul_rn(r[h + j].z, vp[j]));    // fx.py:113
                        wr[(h + j) * kWarp] = __fadd_rn(r[h + j].x, __fmul_rn(c.fb, it));                           // fx.py:114
                        itb[(h + j) * kWarp + lane] = it;
                    }
                    __syncwarp();
                }
            } else {
                // ---- no tap of a block falls inside that block: four waves, nothing but the taps in between ----
#pragma unroll
                for (int j = 0; j < kSub; ++j) {
                    const unsigned pk = __float_as_uint(r[j].w);
                    const float vp = smem[pk >> 16];
                    const float vq = smem[pk & 0xffffu];
                    const float it = __fadd_rn(__fmul_rn(r[j].y, vq), __fmul_rn(r[j].z, vp));           // fx.py:113
                    wr[j * kWarp] = __fadd_rn(r[j].x, __fmul_rn(c.fb, it));                             // fx.py:114
                    itb[j * kWarp + lane] = it;
                    __syncwarp();
                }
            }
        } else {
            // ---- some block has a tap inside itself: the producer left a schedule code per block
            const unsigned codes = (unsigned)reinterpret_cast<const int*>(slot + 5 * kTile)[4];
            // (a rolled loop on purpose: four unrolled copies of the schedules below do not fit the instruction cache)
            int j = 0;
#pragma unroll 1
            while (j < kSub) {
                const unsigned code = (codes >> (4 * j)) & 15u;
                const int nb = n0 + j * kWarp;
                const int cnt = min(kWarp, N - nb);
                if (cnt <= 0) break;
                const int n = nb + lane;
                const bool mine = lane < cnt;
                if (code >= 1 && code <= (unsigned)kSerialK) {
                    // ---- delays of K..K+1 samples: register-history serial run over this block and the blocks of the tile
                    // that follow with the same K (records already in serial form) ----
                    int L = 1;
                    while (j + L < kSub && ((codes >> (4 * (j + L))) & 15u) == code) ++L;
                    float4* cb = cs + j * kWarp;
                    if (code == 1) {
                        // far tap of a sub-sample delay: the stale sample M back, S = fraction * stale (fx.py:113)
                        for (int l = 0; l < L; ++l) {
                            float* wp = &cb[l * kWarp + lane].w;
                            *wp = __fmul_rn(*wp, ring[(n + l * kWarp - c.M) & mask]);
                        }
                    }
                    __syncwarp();
                    float* ito = itb + j * kWarp;
                    switch (code) {
                        case 1: serial_run<1>(ring, mask, nb, cb, c.fb, ito, lane, 8 * L); break;
                        case 2: serial_run<2>(ring, mask, nb, cb, c.fb, ito, lane, 8 * L); break;
                        case 3: serial_run<3>(ring, mask, nb, cb, c.fb, ito, lane, 8 * L); break;
                        case 4: serial_run<4>(ring, mask, nb, cb, c.fb, ito, lane, 8 * L); break;
                        case 5: serial_run<5>(ring, mask, nb, cb, c.fb, ito, lane, 8 * L); break;
                        case 6: serial_run<6>(ring, mask, nb, cb, c.fb, ito, lane, 8 * L); break;
                        case 7: serial_run<7>(ring, mask, nb, cb, c.fb, ito, lane, 8 * L); break;
                        default: serial_run<8>(ring, mask, nb, cb, c.fb, ito, lane, 8 * L); break;
                    }
                    __syncwarp();
                    j += L;
                    continue;
                }
                const float4 r = cs[j * kWarp + lane];
                const unsigned pk = __float_as_uint(r.w);
                const int ip = pk >> 16, iq = pk & 0xffffu;
                float my_it = 0.0f;
                if (code == 0) {
                    // every sample depends only on samples before the block: one wave
                    my_it = __fadd_rn(__fmul_rn(r.y, smem[iq]), __fmul_rn(r.z, smem[ip]));
                    if (mine) ring[n & mask] = __fadd_rn(r.x, __fmul_rn(c.fb, my_it));
                    itb[j * kWarp + lane] = my_it;
                    __syncwarp();
                } else if (code == 14) {
                    // waves of kmin - 1 consecutive samples: sample i depends on samples <= i - (kmin - 1).  Every lane
                    // computes in every wave (no divergence); only the lanes of the wave keep and store their result.
                    const int kp = (n - (ip - ring_w)) & mask;
                    const int mn = __reduce_min_sync(kFull, mine ? kp : 0x7fffffff) - 1;
                    for (int dn = 0; dn < cnt; dn += mn) {
                        const float it = __fadd_rn(__fmul_rn(r.y, smem[iq]), __fmul_rn(r.z, smem[ip]));
                        const float v = __fadd_rn(r.x, __fmul_rn(c.fb, it));
                        if (lane >= dn && lane < dn + mn && mine) {
                            ring[n & mask] = v;
                            my_it = it;
                        }
                        __syncwarp();
                    }
                    itb[j * kWarp + lane] = my_it;
                } else {
                    // ---- anything else with a 1-2 sample delay in it: generic lock-step serial run; taps at
                    // distance 1 and 2 come from registers, older taps are loaded two samples ahead ----
                    const int kp = (n - (ip - ring_w)) & mask;
                    float p1 = ring[(nb - 1) & mask];
                    float p2 = ring[(nb - 2) & mask];
                    int kpa = __shfl_sync(kFull, kp, 0);
                    int kpb = __shfl_sync(kFull, kp, 1);
                    float lpa = ring[(nb - kpa) & mask];
                    float lqa = ring[(nb - kq_of(kpa, c.M)) & mask];
                    float lpb = ring[(nb + 1 - kpb) & mask];
                    float lqb = ring[(nb + 1 - kq_of(kpb, c.M)) & mask];
#pragma unroll 1
                    for (int i = 0; i < cnt; ++i) {
                        const int kpc = __shfl_sync(kFull, kp, (i + 2) & 31);
                        const float lpc = ring[(nb + i + 2 - kpc) & mask];
                        const float lqc = ring[(nb + i + 2 - kq_of(kpc, c.M)) & mask];
                        const float xi = __shfl_sync(kFull, r.x, i);
                        const float fri = __shfl_sync(kFull, r.y, i);
                        const float omi = __shfl_sync(kFull, r.z, i);
                        const int kqa = kq_of(kpa, c.M);
                        const float vp = (kpa == 1) ? p1 : ((kpa == 2) ? p2 : lpa);
                        const float vq = (kqa == 1) ? p1 : ((kqa == 2) ? p2 : lqa);
                        const float it = __fadd_rn(__fmul_rn(fri, vq), __fmul_rn(omi, vp));     // fx.py:113
                        const float v = __fadd_rn(xi, __fmul_rn(c.fb, it));                      // fx.py:114
                        if (lane == 0) ring[(nb + i) & mask] = v;    // every lane holds the same value: one lane stores
                        __syncwarp();
                        if (lane == i) my_it = it;
                        p2 = p1; p1 = v;
                        kpa = kpb; lpa = lpb; lqa = lqb;
                        kpb = kpc; lpb = lpc; lqb = lqc;
                    }
                    itb[j * kWarp + lane] = my_it;
                    __syncwarp();
                }
                ++j;
            }
        }
        __syncwarp();
        if (lane == 0) st_release(done, t + 1);
        if (++sl == kNT) sl = 0;
    }
}

// ---- all-pass fractional-delay interpolation (north_star: "per-sample linear or all-pass interpolation") -----------
// The reference only has the linear blend of fx.py:113 (SURVEY F2); this mode is this repository's OWN definition,
// stated in include/modfx.h: the read position lies delta = 1 - fraction samples behind the newer tap q, and
//   it[n] = eta * (buf[q] - it[n-1]) + buf[p],   eta = (1 - delta) / (1 + delta) = fraction / (2 - fraction)
// replaces the blend; index arithmetic, feedback, mix and clip stay those of fx.py:95-118.  The interpolator carries
// a state from sample to sample, so a delay line is serial whatever its delay: one LANE per delay line, up to 32 lines
// per one-warp CTA, the written samples in a shared-memory ring laid out [time][line] (conflict-free), audio moved
// through 32 x 32 transposing tiles so that global traffic stays coalesced.  A mode behind a flag, not the hot path.
__global__ void __launch_bounds__(kWarp) fc_allpass_kernel(const FcArgs a, int L, int ring_mask, int n_lines) {
    extern __shared__ __align__(16) float smem[];
    float(*xt)[kWarp + 1] = reinterpret_cast<float(*)[kWarp + 1]>(smem);
    float(*mt)[kWarp + 1] = reinterpret_cast<float(*)[kWarp + 1]>(smem + kWarp * (kWarp + 1));
    float* ring = smem + 2 * kWarp * (kWarp + 1);           // [(ring_mask + 1)][L]
    const int lane = threadIdx.x;
    const int line = blockIdx.x * L + lane;                 // (item, channel)
    const bool live = lane < L && line < n_lines;
    const int item = live ? line / a.C : 0;
    const int ch = live ? line - item * a.C : 0;
    const int b = a.index ? a.index[item] : item;
    const int N = a.N;
    const Coef c = make_coef(a, b);
    const float* xs = a.x + ((int64_t)b * a.C + ch) * (int64_t)N;
    float* ys = a.y + ((int64_t)b * a.C + ch) * (int64_t)N;
    const bool audio = a.n_lo == 0;
    const float* ms = audio ? a.mod + (a.mod_has_ch ? ((int64_t)b * a.C + ch) : (int64_t)b) * (int64_t)N
                            : a.mod + (int64_t)b * a.n_lo;
    for (int i = lane; i < (ring_mask + 1) * L; i += kWarp) ring[i] = 0.0f;             // fx.py:92
    __syncwarp();
    float it_prev = 0.0f;
    int wk = 0;
    for (int n0 = 0; n0 < N; n0 += kWarp) {
        for (int l = 0; l < L; ++l) {                       // line l's next 32 samples: one 128-byte request
            const float* xr = reinterpret_cast<const float*>(__shfl_sync(kFull, reinterpret_cast<unsigned long long>(xs), l));
            const float* mr = reinterpret_cast<const float*>(__shfl_sync(kFull, reinterpret_cast<unsigned long long>(ms), l));
            const bool ok = __shfl_sync(kFull, (int)live, l) && (n0 + lane < N);
            xt[l][lane] = ok ? xr[n0 + lane] : 0.0f;
            if (audio) mt[l][lane] = ok ? mr[n0 + lane] : 0.0f;
        }
        __syncwarp();
        if (live) {
            const int cnt = min(kWarp, N - n0);
            for (int i = 0; i < cnt; ++i) {
                const int n = n0 + i;
                const float m = audio ? mt[lane][i] : upsample_ac(ms, a.n_lo, a.up_scale, n);
                float fr, omfr;
                int kp;
                fc_index(m, wk, c, fr, omfr, kp);                                       // fx.py:95-102
                const float vp = ring[((n - kp) & ring_mask) * L + lane];
                const float vq = ring[((n - kq_of(kp, c.M)) & ring_mask) * L + lane];
                const float eta = __fdiv_rn(fr, __fsub_rn(2.0f, fr));
                const float it = __fadd_rn(__fmul_rn(eta, __fsub_rn(vq, it_prev)), vp);
                it_prev = it;
                const float x = xt[lane][i];
                ring[(n & ring_mask) * L + lane] = __fadd_rn(x, __fmul_rn(c.fb, it));   // fx.py:114
                const float o = __fadd_rn(x, __fmul_rn(c.depth, it));                   // fx.py:115
                const float r = __fadd_rn(__fmul_rn(c.omm, x), __fmul_rn(c.mix, o));    // fx.py:117
                xt[lane][i] = fminf(fmaxf(r, -1.0f), 1.0f);                             // fx.py:118
                if (++wk == c.M) wk = 0;
            }
        }
        __syncwarp();
        for (int l = 0; l < L; ++l) {
            float* yr = reinterpret_cast<float*>(__shfl_sync(kFull, reinterpret_cast<unsigned long long>(ys), l));
            const bool ok = __shfl_sync(kFull, (int)live, l) && (n0 + lane < N);
            if (ok) yr[n0 + lane] = xt[l][lane];
        }
        __syncwarp();
    }
}

// apply_tremolo, fx.py:13-22: ((1 - mix) * x) + ((mix * mod) * x); one block per (example, channel).
template <int MODE>
__global__ void __launch_bounds__(256) tremolo_kernel(const FcArgs a) {
    extern __shared__ float smem[];
    const int b = blockIdx.x / a.C;
    const int ch = blockIdx.x - b * a.C;
    const int N = a.N;
    const float* lo = smem;
    LfoDesc lfo;
    if (MODE == kDirectLfo || (MODE == kControlRate && a.lfo_freq))
        lfo = make_lfo_desc(a.lfo_freq[b], a.lfo_phase[b], a.lfo_shape[b], a.lfo_exp ? a.lfo_exp[b] : 1.0f, a.sr_lo);
    if (MODE == kControlRate) {
        if (a.lfo_freq) {       // synthesise the control-rate row once per block
            for (int i = threadIdx.x; i < a.n_lo; i += blockDim.x) smem[i] = lfo_value(lfo, i);
            __syncthreads();
        } else {
            lo = a.mod + (int64_t)b * a.n_lo;   // elementwise op: the two taps stay in L1
        }
    }
    const float mix = a.mix_p ? a.mix_p[b] : a.mix_s;
    const float omm = a.mix_p ? __fsub_rn(1.0f, mix) : a.omm_s;
    const float* xs = a.x + ((int64_t)b * a.C + ch) * (int64_t)N;
    float* ys = a.y + ((int64_t)b * a.C + ch) * (int64_t)N;
    const float* ms = nullptr;
    if (MODE == kAudioRate) ms = a.mod + (a.mod_has_ch ? ((int64_t)b * a.C + ch) : (int64_t)b) * (int64_t)N;
    for (int n = blockIdx.y * blockDim.x + threadIdx.x; n < N; n += gridDim.y * blockDim.x) {
        float m;
        if (MODE == kAudioRate) m = ms[n];
        else if (MODE == kControlRate) m = upsample_ac(lo, a.n_lo, a.up_scale, n);
        else m = lfo_value(lfo, n);
        const float xv = xs[n];
        ys[n] = __fadd_rn(__fmul_rn(omm, xv), __fmul_rn(__fmul_rn(mix, m), xv));
    }
}

int next_pow2(int v) {
    int p = 1;
    while (p < v) p <<= 1;
    return p;
}

constexpr size_t kMaxSmem = 200 * 1024;    // dynamic shared memory an effect kernel may take; larger requests are refused

int fill_mod(FcArgs& a, const modfx_mod_source* mod, int64_t N, int& mode) {
    MODFX_REQUIRE(mod != nullptr, "mod source is NULL");
    a.mod = mod->mod;
    a.mod_has_ch = mod->mod_has_ch;
    a.n_lo = 0;
    a.up_scale = 0.0f;
    a.sr_lo = mod->sr_lo;
    a.lfo_freq = nullptr;
    a.lfo_phase = nullptr;
    a.lfo_shape = nullptr;
    a.lfo_exp = nullptr;
    switch (mod->kind) {
        case MODFX_MOD_AUDIO_RATE:
            MODFX_REQUIRE(mod->mod != nullptr, "audio-rate mod pointer is NULL");
            mode = kAudioRate;
            break;
        case MODFX_MOD_CONTROL_RATE:
            MODFX_REQUIRE(mod->mod != nullptr, "control-rate mod pointer is NULL");
            MODFX_REQUIRE(mod->n_lo >= 1 && mod->n_lo <= N, "control-rate n_lo=%lld must be in [1, N]",
                          (long long)mod->n_lo);
            a.n_lo = (int)mod->n_lo;
            a.up_scale = upsample_scale_ac(mod->n_lo, N);
            mode = kControlRate;
            if (mod->n_lo == N) mode = kAudioRate, a.mod_has_ch = 0;   // util.py:18-19: same length => untouched
            break;
        case MODFX_MOD_LFO:
            MODFX_REQUIRE(mod->lfo_freq && mod->lfo_phase && mod->lfo_shape, "LFO parameter pointer is NULL");
            MODFX_REQUIRE(mod->sr_lo > 0.0f, "LFO sample rate must be positive");
            MODFX_REQUIRE(mod->n_lo >= 1, "LFO n_lo must be >= 1");
            a.lfo_freq = mod->lfo_freq;
            a.lfo_phase = mod->lfo_phase;
            a.lfo_shape = mod->lfo_shape;
            a.lfo_exp = mod->lfo_exp;
            if (mod->n_lo == N) mode = kDirectLfo;
            else {
                MODFX_REQUIRE(mod->n_lo <= N, "LFO n_lo=%lld must be <= N", (long long)mod->n_lo);
                a.n_lo = (int)mod->n_lo;
                a.up_scale = upsample_scale_ac(mod->n_lo, N);
                mode = kControlRate;
            }
            break;
        default:
            return fail(MODFX_ERR_INVALID, "unknown mod kind %d", mod->kind);
    }
    return MODFX_OK;
}

int check_scalar(const modfx_param& p, const char* name, bool can_be_one) {
    if (p.dev) return MODFX_OK;     // device arrays are range-checked by the caller (fx.py:52-57 needs a sync)
    // fx.py:65-69
    MODFX_REQUIRE(p.value >= 0.0, "%s=%g must be >= 0", name, p.value);
    if (can_be_one) MODFX_REQUIRE(p.value <= 1.0, "%s=%g must be <= 1", name, p.value);
    else MODFX_REQUIRE(p.value < 1.0, "%s=%g must be < 1", name, p.value);
    return MODFX_OK;
}

enum FcEffect { kLinearDelay, kAllpassDelay, kTremolo };

struct FcParams { modfx_param feedback, min_delay_width, width, depth, mix; };    // tremolo takes mix alone

// Validates the arguments of one entry point, in an order that gives every refusal its status and message, and fills
// `a` and the modulation mode.  a.n_items == 0 on success: nothing to render.
int fc_setup(FcArgs& a, int& mode, FcEffect fx, const float* x, float* y, int32_t B, int32_t C, int64_t N, int32_t Mmin,
             int32_t Mlfo, const modfx_mod_source* mod, const FcParams& p, const int32_t* example_index, int32_t n_items) {
    a = FcArgs{};
    MODFX_REQUIRE(x && y, "x / y is NULL");
    // the linear delay line names an over-long N on its own; the other two count it as a bad shape
    MODFX_REQUIRE(B >= 0 && C >= 1 && N >= 1 && (fx == kLinearDelay || N < (1ll << 30)), "bad shape B=%d C=%d N=%lld", B,
                  C, (long long)N);
    MODFX_REQUIRE(N < (1ll << 30), "N=%lld too long (max 2^30-1 samples)", (long long)N);
    int st;
    if (fx != kTremolo) {
        MODFX_REQUIRE(Mmin >= 0 && Mlfo >= 0 && Mmin + Mlfo >= 1, "bad delay line Mmin=%d Mlfo=%d", Mmin, Mlfo);
        if ((st = check_scalar(p.feedback, "feedback", false)) != MODFX_OK) return st;          // fx.py:86
        if ((st = check_scalar(p.min_delay_width, "min_delay_width", true)) != MODFX_OK) return st;
        if ((st = check_scalar(p.width, "width", true)) != MODFX_OK) return st;
        if ((st = check_scalar(p.depth, "depth", true)) != MODFX_OK) return st;
    }
    if ((st = check_scalar(p.mix, "mix", true)) != MODFX_OK) return st;                          // fx.py:21
    a.x = x; a.y = y; a.B = B; a.C = C; a.N = (int)N;
    a.Mmin = Mmin; a.Mlfo = Mlfo; a.M = Mmin + Mlfo;
    if ((st = fill_mod(a, mod, N, mode)) != MODFX_OK) return st;
    if (fx == kAllpassDelay) {
        if (mode == kDirectLfo || a.lfo_freq)
            return fail(MODFX_ERR_UNSUPPORTED, "all-pass interpolation takes the modulation signal from memory (audio or control rate)");
        if (mode == kAudioRate) a.n_lo = 0;
    }
    a.fb_p = p.feedback.dev;         a.fb_s = (float)p.feedback.value;
    a.mdw_p = p.min_delay_width.dev; a.min_delay_s = (float)(p.min_delay_width.value * (double)Mmin);
    a.width_p = p.width.dev;         a.lfo_delay_s = (float)((double)Mlfo * p.width.value);
    a.depth_p = p.depth.dev;         a.depth_s = (float)p.depth.value;
    a.mix_p = p.mix.dev;             a.mix_s = (float)p.mix.value; a.omm_s = (float)(1.0 - p.mix.value);
    a.index = example_index;
    a.n_items = example_index ? n_items : B;
    MODFX_REQUIRE(a.n_items >= 0, "n_items=%d", a.n_items);
    return MODFX_OK;
}

}  // namespace
}  // namespace modfx

using namespace modfx;

extern "C" int modfx_flanger_chorus_f32(const float* x, float* y, int32_t B, int32_t C, int64_t N,
                                        int32_t Mmin, int32_t Mlfo, const modfx_mod_source* mod,
                                        modfx_param feedback, modfx_param min_delay_width, modfx_param width,
                                        modfx_param depth, modfx_param mix, const int32_t* example_index,
                                        int32_t n_items, void* stream) {
    FcArgs a;
    int mode = 0, st;
    if ((st = fc_setup(a, mode, kLinearDelay, x, y, B, C, N, Mmin, Mlfo, mod,
                       {feedback, min_delay_width, width, depth, mix}, example_index, n_items)) != MODFX_OK ||
        a.n_items == 0)
        return st;
    const int ring = next_pow2(a.M + kTile);
    a.ring_mask = ring - 1;

    // The CTA-per-delay-line kernel renders every modulation source; a control row synthesised in-kernel is staged in
    // shared memory up to kLoSmemMax points and evaluated at the taps beyond that.
    const bool synth = a.lfo_freq != nullptr;
    const int lo_smem = (mode == kControlRate && synth && a.n_lo <= kLoSmemMax) ? ((a.n_lo + 3) & ~3) : 0;
    const size_t csmem = sizeof(float) * (16 + (size_t)kNT * kSlotFloats +
                                          (size_t)kCtaProd * kXDepth * kTile * (mode == kAudioRate ? 2 : 1) +
                                          (size_t)lo_smem + (size_t)ring);
    if (csmem > kMaxSmem)
        return fail(MODFX_ERR_UNSUPPORTED, "delay line of %d samples needs %zu B of shared memory", a.M, csmem);
    const dim3 grid((unsigned)((int64_t)a.n_items * C));
    cudaStream_t s = as_stream(stream);
    // Delay lines that can never reach back less than a wide tile (min_delay_width * Mmin >= 388 samples: the chorus) go
    // through the CTA-per-example kernel first; fc_cta_kernel then skips exactly those examples.
    a.wide = 0;
    if (mode == kControlRate && !synth && Mmin >= kWideTile + kWideMargin) {
        const int wring = next_pow2(a.M + kWideTile);
        const size_t wsmem = sizeof(float) * (size_t)wring;
        if (wsmem <= kMaxSmem) {
            a.wide = 1;
            if ((st = launch(fc_wide_kernel, grid, kWideThreads, wsmem, s, a, wring - 1)) != MODFX_OK) return st;
        }
    }
    void (*cta)(FcArgs, int);
    if (mode == kAudioRate) cta = fc_cta_kernel<kAudioRate, kRead>;
    else if (mode == kDirectLfo) cta = fc_cta_kernel<kDirectLfo, kAtTap>;
    else if (!synth) cta = fc_cta_kernel<kControlRate, kRead>;
    else if (lo_smem > 0) cta = fc_cta_kernel<kControlRate, kStaged>;
    else cta = fc_cta_kernel<kControlRate, kAtTap>;
    return launch(cta, grid, kCtaThreads, csmem, s, a, lo_smem);
}

extern "C" int modfx_flanger_chorus_allpass_f32(const float* x, float* y, int32_t B, int32_t C, int64_t N,
                                                int32_t Mmin, int32_t Mlfo, const modfx_mod_source* mod,
                                                modfx_param feedback, modfx_param min_delay_width, modfx_param width,
                                                modfx_param depth, modfx_param mix, const int32_t* example_index,
                                                int32_t n_items, void* stream) {
    FcArgs a;
    int mode = 0, st;
    if ((st = fc_setup(a, mode, kAllpassDelay, x, y, B, C, N, Mmin, Mlfo, mod,
                       {feedback, min_delay_width, width, depth, mix}, example_index, n_items)) != MODFX_OK ||
        a.n_items == 0)
        return st;
    const int ring = next_pow2(a.M + 1);
    a.ring_mask = ring - 1;
    int L = kWarp;
    while (L > 1 && (size_t)ring * L * sizeof(float) > 160 * 1024) L >>= 1;
    const size_t smem = sizeof(float) * ((size_t)ring * L + 2 * kWarp * (kWarp + 1));
    if (smem > kMaxSmem) return fail(MODFX_ERR_UNSUPPORTED, "delay line of %d samples exceeds shared memory", a.M);
    const int n_lines = a.n_items * C;
    return launch(fc_allpass_kernel, (unsigned)((n_lines + L - 1) / L), kWarp, smem, as_stream(stream), a, L, ring - 1,
                  n_lines);
}

extern "C" int modfx_tremolo_f32(const float* x, float* y, int32_t B, int32_t C, int64_t N,
                                 const modfx_mod_source* mod, modfx_param mix, void* stream) {
    FcArgs a;
    FcParams p{};
    p.mix = mix;
    int mode = 0, st;
    if ((st = fc_setup(a, mode, kTremolo, x, y, B, C, N, 0, 0, mod, p, nullptr, 0)) != MODFX_OK || a.n_items == 0)
        return st;
    const size_t smem = sizeof(float) * ((mode == kControlRate && a.lfo_freq) ? (size_t)a.n_lo : 0);
    if (smem > kMaxSmem)
        return fail(MODFX_ERR_UNSUPPORTED, "tremolo with an in-kernel control-rate LFO of %d points exceeds shared memory", a.n_lo);
    int ny = (int)((N + 256 * 8 - 1) / (256 * 8));
    if (ny < 1) ny = 1;
    if (ny > 65535) ny = 65535;
    const dim3 grid((unsigned)(B * C), (unsigned)ny);
    void (*kernel)(FcArgs);
    if (mode == kAudioRate) kernel = tremolo_kernel<kAudioRate>;
    else if (mode == kControlRate) kernel = tremolo_kernel<kControlRate>;
    else kernel = tremolo_kernel<kDirectLfo>;
    return launch(kernel, grid, 256, smem, as_stream(stream), a);
}
