// 5x13 time-dilated convolution (64 -> 64 channels) + 2x1 max-pool + PReLU of the LFO-net on the 5th-generation
// tensor cores: tcgen05.mma kind::tf32, operands staged by TMA, accumulators in tensor memory.
// Reference: nn.Conv2d(64, 64, (5, 13), dilation=(1, d), padding="same") -> nn.MaxPool2d((2, 1)) -> nn.PReLU(64),
// mod_extraction/models.py:187-190 (layers 2..6 of configs/models/spectral_2dcnn.yml, 97 % of the network's flops).
//
// Implicit GEMM, no im2col buffer.  Activations are channels-last (B, H, W, 64), so for one kernel tap (kh, kw)
// the A operand of a tile of 128 consecutive frames is the box  x[b, h + kh - 2, w0 + (kw - 6) d : +128, 0:64]:
// a plain 4-D TMA tile whose out-of-range rows / frames are zero-filled by the TMA unit -- that IS
// padding="same".  The B operand is the 64 x 64 weight slice of the tap.  K = 64 channels per tap, 65 taps.
//
// A CTA owns 8 conv rows (4 pooled output rows) x 128 frames: 8 accumulators of 64 columns fill the 512 columns of
// tensor memory (lane = frame).  Loop order: kw outermost; for one kw the 5 weight slices (kh = 4 .. 0, 80 KB) stay in
// shared memory while the 12 input rows h0-2 .. h0+9 stream through a 4-deep ring of 32 KB A tiles.  Input row r
// feeds conv rows a = r - kh: those accumulators are neighbours in tensor memory and (with kh stored in descending
// order) their weight slices are neighbours in shared memory, so one tcgen05.mma with N = 64 * (number of kernel
// rows) <= 256 serves them all -- the A tile is read once per 5 taps instead of once per tap, which keeps the
// shared-memory read rate (A 4 KB + B 2 KB per N = 64 step would be 192 B/cycle) and the L2 -> SM traffic
// (45 B/cycle/SM at full MMA rate) inside what an SM can take.  The max-pool is a per-thread max of two TMEM reads.
//
// Warp roles (256 threads): warp 0 = A producer, warp 2 = B producer, warps 1 and 3 = MMA issuers for accumulators
// 0..3 and 4..7 (one lane each), warps 4..7 = epilogue (tcgen05.ld -> max -> bias -> PReLU -> 128-byte stores of the channels-last output).  SWIZZLE_128B in both
// the tensor maps and the UMMA descriptors.
#include "common.cuh"

#include <cuda.h>

namespace modfx {
namespace {

constexpr int kC = 64;                    // channels in = channels out = K per tap
constexpr int kKH = 5, kKW = 13;
constexpr int kTileW = 128;               // frames per CTA = UMMA M
constexpr int kRows = 8;                  // conv rows per CTA = accumulators in tensor memory (8 x 64 = 512 columns)
constexpr int kInRows = kRows + kKH - 1;  // input rows a CTA walks
constexpr int kPanelA = kTileW * 128;     // bytes: 128 frames x one 128-byte swizzle row (32 float32 / 64 float16 channels)
constexpr int kTileB = kC * 128;          // bytes: 64 output channels x one 128-byte row of input channels of a kernel tap
constexpr int kPanelB = kKH * kTileB;     // 40 KB: the 5 kernel rows of one kw, kh = 4 first

// Operand format of the 64 -> 64 convolution.  float32 storage read as TF32 (two 128-byte panels of 32 channels per tap,
// K = 8 per MMA) or float16 storage (one panel of 64 channels, K = 16 per MMA): float16 has TF32's 11 significant bits,
// and normalised activations / weights sit well inside its range, so the parity bars are the same -- at twice the MMA
// rate and half the operand traffic.
template <bool kHalf>
struct Fmt {
    static constexpr int kPanels = kHalf ? 1 : 2;
    static constexpr int kChanPerPanel = kC / kPanels;
    static constexpr int kRowBytes = kPanels * kPanelA;         // one input row of the tile: 32 KB / 16 KB
    // input rows per pipeline stage.  With float16 operands a row is only ~210 cycles of tensor-pipe time per issuer,
    // less than the issuer's own per-stage work (barrier waits, election, commits): two rows share one stage
    // (a CTA's live input rows always come in an even number: 8 conv rows + 4 halo rows - 0 / 2 / 4 outside the image)
    static constexpr int kRowsPerStage = kHalf ? 2 : 1;
    static constexpr int kStageA = kRowsPerStage * kRowBytes;   // 32 KB either way
    static constexpr int kBytesB = kPanels * kPanelB;           // 80 KB / 40 KB
    static constexpr int kAStages = 4;                          // power of two; 128 KB of A in flight
    static constexpr int kNumBars = 2 * kAStages + 2 * kKH + 1;
    static constexpr int kSmemBytes = kAStages * kStageA + kBytesB + 1024 /* alignment slack */ + 8 * kNumBars + 16;
    static constexpr uint32_t kFormat = kHalf ? 0u : 2u;        // instruction descriptor: F16 = 0, TF32 = 2
};
constexpr int kThreads = 8 * 32;
constexpr int kTmemCols = kRows * kC;     // 512: all of tensor memory

// kind::tf32 instruction descriptor: D = F32 (bits 4-5 = 1), A = B = TF32 (bits 7-9, 10-12 = 2), both K-major,
// N >> 3 at bits 17-22, M >> 4 at bits 24-28
__device__ __forceinline__ uint32_t idesc_fmt(int n, uint32_t fmt) {
    return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kTileW >> 4) << 24);
}
__device__ __forceinline__ uint32_t idesc_tf32(int n) { return idesc_fmt(n, 2u); }

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
// Bounded spin: a broken pipeline traps (the launch fails with an error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    for (uint32_t spin = 0; !done; ++spin) {
        asm volatile(
            "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (spin > (1u << 26)) __trap();
    }
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2,
                                            int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
// K-major, SWIZZLE_128B shared-memory matrix descriptor: rows of 128 bytes, 8-row groups 1024 bytes apart.
// Low word: start address >> 4 (bits 0-13) and the (unused) leading byte offset (bits 16-29); advancing the
// operand by n bytes inside the tile is `lo + (n >> 4)`.  High word (constant): stride byte offset 1024 >> 4,
// descriptor version 1 (bit 46), SWIZZLE_128B (bits 61-63).
__device__ __forceinline__ uint32_t umma_desc_lo(uint32_t addr) { return ((addr & 0x3FFFFu) >> 4) | (1u << 16); }
constexpr uint32_t kDescHi = (1024u >> 4) | (1u << 14) | (2u << 29);
__device__ __forceinline__ uint64_t umma_desc(uint32_t lo) { return ((uint64_t)kDescHi << 32) | lo; }
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n"
        " tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}\n"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// One lane of a converged warp.  tcgen05.mma / commit / TMA are warp-level instructions in SASS fed from uniform
// registers: issued from `if (lane == 0)` code the compiler wraps each one in an elect / waterfall loop (~10 extra
// issue slots, and a lone thread issues only every ~4.4 cycles: 56 cycles per MMA measured, the price of an N = 112
// MMA); under elect.sync on a converged warp with warp-uniform operands they come out back to back.
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n .reg .pred P;\n elect.sync _|P, 0xffffffff;\n selp.u32 %0, 1, 0, P;\n}\n" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         uint32_t accumulate) {
    asm volatile(
        "{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n"
        " tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}\n"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}

// Which input rows / kernel rows a CTA touches.  Input row r (0 .. kInRows-1) is image row h0 - 2 + r; it feeds conv
// row a = r - kh through kernel row kh.  Rows outside the image are zero (padding="same") and are skipped by every
// role alike; `nrows` < 8 only at the bottom of an image whose height is not a multiple of 8.
struct RowPlan {
    int h0, H, nrows;
    __device__ __forceinline__ bool row_live(int r) const {
        const int hi = h0 - kKH / 2 + r;
        return hi >= 0 && hi < H && r <= nrows - 1 + kKH - 1;
    }
    __device__ __forceinline__ int kh_lo(int r) const { return max(0, r - (nrows - 1)); }
    __device__ __forceinline__ int kh_hi(int r) const { return min(kKH - 1, r); }
    // first / last live input row that uses kernel row kh (first > last: the CTA never uses it)
    __device__ __forceinline__ int first_use(int kh) const {
        for (int r = kh; r <= kh + nrows - 1; ++r)
            if (row_live(r)) return r;
        return kInRows;
    }
    __device__ __forceinline__ int last_use(int kh) const {
        for (int r = kh + nrows - 1; r >= kh; --r)
            if (row_live(r)) return r;
        return -1;
    }
};

// n_pass = 1: plain TF32.  n_pass = 3: error-compensated TF32 ("3xTF32"): activations and weights arrive split as
// hi + lo (hi = the value rounded to TF32, lo = the rounded remainder) and the tap loop runs three times into the same
// accumulators -- hi*hi, hi*lo, lo*hi (lo*lo is below float32 resolution) -- at a third of the TF32 rate.  That removes
// the operand rounding; the residual (2e-4 per layer against 1e-3 for plain TF32) is the tensor pipe's accumulator, which
// truncates rather than rounds.  Through the whole network the mode meets the float32 parity bars.
struct ConvMaps {
    CUtensorMap x[2];       // activations: hi, lo
    CUtensorMap w[2];       // weights: hi, lo
};

template <bool kHalf>
__global__ void __launch_bounds__(kThreads, 1) conv_tf32_kernel(const __grid_constant__ ConvMaps tm, int n_pass,
                                                                float* __restrict__ y, int H, int W, int dil,
                                                                const float* __restrict__ bias,
                                                                const float* __restrict__ prelu) {
    using F = Fmt<kHalf>;
    constexpr int kAStages = F::kAStages, kStageA = F::kStageA, kBytesB = F::kBytesB, kNumBars = F::kNumBars;
    extern __shared__ unsigned char smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;                   // SWIZZLE_128B wants 1024-byte aligned tiles
    const uint32_t a_base = base;                                   // kAStages x 32 KB
    const uint32_t b_base = base + kAStages * kStageA;              // 2 panels x 5 tiles x 8 KB
    const uint32_t bar0 = b_base + kBytesB;
    // barriers: A full[s], A empty[s], B full[j], B empty[j] (j = 4 - kh), accumulators ready
    const uint32_t bar_afull = bar0, bar_aempty = bar0 + 8 * kAStages;
    const uint32_t bar_bfull = bar0 + 16 * kAStages, bar_bempty = bar_bfull + 8 * kKH;
    const uint32_t bar_acc = bar_bempty + 8 * kKH;
    volatile uint32_t* tmem_slot =
        reinterpret_cast<volatile uint32_t*>(smem_raw + (bar_acc + 8 - raw));

    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(kFull, tid >> 5, 0);               // warp-uniform as far as the compiler can see
    const int w0 = blockIdx.x * kTileW;
    const int b = blockIdx.z;
    RowPlan plan;
    plan.h0 = blockIdx.y * kRows;
    plan.H = H;
    plan.nrows = min(kRows, H - plan.h0);

    if (tid == 0) {
        // "full" barriers: one producer arrival (+ its bytes); "empty" / "accumulators ready": one commit per MMA issuer
        for (int i = 0; i < kAStages; ++i) {
            mbar_init(bar_afull + 8 * i, 1);
            mbar_init(bar_aempty + 8 * i, 2);
        }
        for (int i = 0; i < kKH; ++i) {
            mbar_init(bar_bfull + 8 * i, 1);
            mbar_init(bar_bempty + 8 * i, 2);
        }
        mbar_init(bar_acc, 2);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 4) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(bar_acc + 8), "n"(kTmemCols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = __shfl_sync(kFull, *tmem_slot, 0);

    if (warp == 0) {
        // ===== A producer (whole warp walks the loop, one elected lane issues): a 128-frame x 64-channel box per
        // (kw, live input row) =====
        int it = 0, sub = 0;                                        // stage counter, row inside the stage
        for (int v = 0; v < n_pass * kKW; ++v) {                     // v = pass * 13 + kw
            const int pass = v / kKW, kw = v - pass * kKW;
            const CUtensorMap* tmx = &tm.x[pass == 2 ? 1 : 0];      // passes: hi*hi, hi*lo, lo*hi
            const int wx = w0 + (kw - kKW / 2) * dil;
            for (int r = 0; r < kInRows; ++r) {
                if (!plan.row_live(r)) continue;
                const int s = it % kAStages;
                if (sub == 0) mbar_wait(bar_aempty + 8 * s, (((uint32_t)(it / kAStages)) & 1u) ^ 1u);
                if (elect_one()) {
                    const uint32_t full = bar_afull + 8 * s;
                    const uint32_t st = a_base + s * kStageA + sub * F::kRowBytes;
                    if (sub == 0) mbar_expect_tx(full, kStageA);
#pragma unroll
                    for (int p = 0; p < F::kPanels; ++p)
                        tma_load_4d(st + p * kPanelA, tmx, full, p * F::kChanPerPanel, wx, plan.h0 - kKH / 2 + r, b);
                }
                __syncwarp();
                if (++sub == F::kRowsPerStage) {
                    sub = 0;
                    ++it;
                }
            }
        }
    } else if (warp == 2) {
        // ===== B producer: the 5 kernel rows of one kw, slot j = 4 - kh, refilled as soon as the MMAs release it =====
        for (int v = 0; v < n_pass * kKW; ++v) {
            const int pass = v / kKW, kw = v - pass * kKW;
            const CUtensorMap* tmw = &tm.w[pass == 1 ? 1 : 0];
            for (int kh = 0; kh < kKH; ++kh) {
                if (plan.first_use(kh) > plan.last_use(kh)) continue;
                const int j = kKH - 1 - kh;
                mbar_wait(bar_bempty + 8 * j, ((uint32_t)v & 1u) ^ 1u);
                if (elect_one()) {
                    const uint32_t full = bar_bfull + 8 * j;
                    mbar_expect_tx(full, F::kPanels * kTileB);
#pragma unroll
                    for (int p = 0; p < F::kPanels; ++p)
                        tma_load_3d(b_base + p * kPanelB + j * kTileB, tmw, full, p * F::kChanPerPanel, 0, kh * kKW + kw);
                }
                __syncwarp();
            }
        }
    } else if (warp == 1 || warp == 3) {
        // ===== MMA issuers: warp 1 owns accumulators 0..3, warp 3 accumulators 4..7 (an accumulator belongs to one
        // issuer, so the summation order -- and the result -- stays fixed).  The whole warp walks the loops with
        // warp-uniform state; the tcgen05 instructions are issued by one elected lane.
        // Input row r feeds accumulators r - kh_hi .. r - kh_lo through kernel rows kh_hi .. kh_lo.  Neighbouring
        // accumulators are neighbours in tensor memory and (kernel rows stored in descending order) their weight
        // slices neighbours in shared memory: ONE MMA of N = 64 n serves the n <= 4 of them this issuer owns. =====
        const int own_lo = (warp == 1) ? 0 : kRows / 2, own_hi = own_lo + kRows / 2 - 1;
        // per input row (registers, the r loops below are fully unrolled): first own accumulator, how many, and which
        // weight slots must have landed before / may be released after the row
        int run_a[kInRows], run_n[kInRows];
        uint32_t wait_b[kInRows], free_b[kInRows];
        bool live[kInRows];
#pragma unroll
        for (int r = 0; r < kInRows; ++r) {
            live[r] = plan.row_live(r);
            const int a0 = max(r - plan.kh_hi(r), own_lo), a1 = min(r - plan.kh_lo(r), own_hi);
            run_a[r] = a0;
            run_n[r] = live[r] ? max(a1 - a0 + 1, 0) : 0;
            wait_b[r] = free_b[r] = 0;
        }
#pragma unroll
        for (int kh = 0; kh < kKH; ++kh) {
            const int f = plan.first_use(kh), l = plan.last_use(kh);
#pragma unroll
            for (int r = 0; r < kInRows; ++r) {
                if (f <= l && f == r) wait_b[r] |= 1u << kh;
                if (f <= l && l == r) free_b[r] |= 1u << kh;
            }
        }
        int it = 0, sub = 0;                                        // stage counter, row inside the stage
        uint32_t free_pending = 0;                                  // weight slots to release at the end of the stage
#pragma unroll 1
        for (int v = 0; v < n_pass * kKW; ++v) {                     // v = pass * 13 + kw: the weight ring turns once per v
            const uint32_t b_par = (uint32_t)v & 1u;
            uint32_t started = (v == 0) ? 0u : 0xFFu;              // accumulators that hold a partial sum
#pragma unroll
            for (int r = 0; r < kInRows; ++r) {
                if (!live[r]) continue;
                const int s = it & (kAStages - 1);
#pragma unroll
                for (int kh = 0; kh < kKH; ++kh)
                    if ((wait_b[r] >> kh) & 1u) mbar_wait(bar_bfull + 8 * (kKH - 1 - kh), b_par);
                // (waited for even when this issuer has no accumulator under the row: it keeps the two issuers within
                // one ring revolution of each other, which the two-arrival "empty" barriers rely on)
                if (sub == 0) mbar_wait(bar_afull + 8 * s, ((uint32_t)(it / kAStages)) & 1u);
                if (run_n[r] > 0) {
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t a_lo = umma_desc_lo(a_base) + s * (kStageA >> 4) + sub * (F::kRowBytes >> 4);
                    // at the very first tap a fresh accumulator overwrites while its neighbours already add: split the run there
                    int a = run_a[r];
                    int left = run_n[r];
                    while (left > 0) {
                        const uint32_t flag = (started >> a) & 1u;
                        int n = 1;
                        while (n < left && ((started >> (a + n)) & 1u) == flag) ++n;
                        const uint32_t b_lo = umma_desc_lo(b_base) + (kKH - 1 - (r - a)) * (kTileB >> 4);
                        const uint32_t idesc = idesc_fmt(n * kC, F::kFormat);
                        const uint32_t d = tmem + a * kC;
                        if (elect_one()) {
#pragma unroll
                            for (int pk = 0; pk < 4 * F::kPanels; ++pk) {        // 32 bytes of K per instruction
                                const int p = pk >> 2, k = pk & 3;
                                const uint64_t ad = umma_desc(a_lo + ((p * kPanelA + k * 32) >> 4));
                                const uint64_t bd = umma_desc(b_lo + ((p * kPanelB + k * 32) >> 4));
                                if (kHalf) umma_f16(d, ad, bd, idesc, flag | (pk > 0));
                                else umma_tf32(d, ad, bd, idesc, flag | (pk > 0));
                            }
                        }
                        __syncwarp();
                        a += n;
                        left -= n;
                    }
                }
                // accumulators r - kh_hi .. r - kh_lo (either issuer's) have been written once this row is through
                started |= ((2u << (r - plan.kh_lo(r))) - 1u) & ~((1u << (r - plan.kh_hi(r))) - 1u);
                free_pending |= free_b[r];
                if (++sub == F::kRowsPerStage) {
                    // end of the stage: its A slot, and the weight slots whose last reader was in it, go back to the
                    // producers once this issuer's MMAs have read them
                    if (elect_one()) {
                        umma_commit(bar_aempty + 8 * s);
#pragma unroll
                        for (int kh = 0; kh < kKH; ++kh)
                            if ((free_pending >> kh) & 1u) umma_commit(bar_bempty + 8 * (kKH - 1 - kh));
                    }
                    __syncwarp();
                    free_pending = 0;
                    sub = 0;
                    ++it;
                }
            }
        }
        if (elect_one()) umma_commit(bar_acc);                      // this issuer's accumulators are complete
        __syncwarp();
    } else {
        // ===== epilogue: lane = frame, column = output channel; conv rows 2 p and 2 p + 1 pool into output row p =====
        mbar_wait(bar_acc, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int q = warp & 3;                                     // the TMEM lane quadrant this warp may read
        const int w = w0 + 32 * q + lane;
        for (int pr = 0; pr < plan.nrows / 2; ++pr) {
            float* yp = y + (((int64_t)b * (H / 2) + plan.h0 / 2 + pr) * W + w) * kC;
#pragma unroll 1
            for (int half = 0; half < 2; ++half) {
                uint32_t up[32], lo[32];
                const uint32_t taddr = tmem + ((uint32_t)(32 * q) << 16) + 2 * pr * kC + 32 * half;
                tmem_ld32(taddr, up);
                tmem_ld32(taddr + kC, lo);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (w < W) {
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        float o[4];
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const int c = 32 * half + j + i;
                            const float v =
                                fmaxf(__uint_as_float(up[j + i]), __uint_as_float(lo[j + i])) + __ldg(bias + c);
                            o[i] = v > 0.0f ? v : __ldg(prelu + c) * v;
                        }
                        *reinterpret_cast<float4*>(yp + 32 * half + j) = make_float4(o[0], o[1], o[2], o[3]);
                    }
                }
            }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    }
    __syncthreads();
    if (warp == 4) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(kTmemCols) : "memory");
    }
}

// ---------------------------------------------------------------------------------------------------------------
// First layer (2 -> 64 channels, dilation 1) on the tensor cores.  With 2 input channels a kernel tap is only K = 2,
// so the 13 taps of a kernel row are folded into K: for kernel row kh
//   A[frame][2 kw + c] = x[b, h + kh - 2, frame + kw - 6, c]     (26 columns, zero padded to 32 = one 128-byte row)
//   B[co][2 kw + c]    = weight[kh][kw][co][c]
// A is a Toeplitz matrix -- row `frame` is the 26 consecutive floats of the channels-last input starting 6 frames to
// the left -- with a row pitch of 8 bytes, which no tensor map can describe (strides are multiples of 16 bytes), so four
// builder warps write the SWIZZLE_128B tiles themselves (one frame row per thread, 16-byte chunk c lands at chunk
// c ^ (row & 7)) and hand them to the MMA warp through fence.proxy.async + an mbarrier; the same warps build the five
// B tiles once per CTA and run the epilogue at the end.  A CTA owns 4 conv rows (2 pooled) x 128 frames = 4 accumulators
// = 256 TMEM columns, two CTAs per SM, so one CTA's build / epilogue overlaps the other's MMAs.
constexpr int kRows1 = 4;
constexpr int kInRows1 = kRows1 + kKH - 1;
constexpr int kStages1 = 4;
constexpr int kTileA1 = kTileW * 128;     // 16 KB
constexpr int kTileB1 = kC * 128;         // 8 KB
constexpr int kThreads1 = 5 * 32;
constexpr int kTmemCols1 = kRows1 * kC;   // 256
constexpr int kSmemBytes1 = kStages1 * kTileA1 + kKH * kTileB1 + 1024 + 8 * (2 * kStages1 + 2) + 16;

__global__ void __launch_bounds__(kThreads1, 2) conv1_tf32_kernel(const float* __restrict__ x, float* __restrict__ y,
                                                                  int H, int W, const float* __restrict__ weight,
                                                                  const float* __restrict__ bias,
                                                                  const float* __restrict__ prelu) {
    extern __shared__ unsigned char smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    const uint32_t a_base = base, b_base = base + kStages1 * kTileA1;
    const uint32_t bar_full = b_base + kKH * kTileB1, bar_empty = bar_full + 8 * kStages1;
    const uint32_t bar_b = bar_empty + 8 * kStages1, bar_acc = bar_b + 8;
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem_raw + (bar_acc + 8 - raw));
    unsigned char* gen = smem_raw + (base - raw);                   // generic pointer to the aligned area

    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(kFull, tid >> 5, 0);
    const int w0 = blockIdx.x * kTileW;
    const int b = blockIdx.z;
    const int h0 = blockIdx.y * kRows1;
    const int nrows = min(kRows1, H - h0);

    if (tid == 0) {
        for (int i = 0; i < kStages1; ++i) {
            mbar_init(bar_full + 8 * i, 128);
            mbar_init(bar_empty + 8 * i, 1);
        }
        mbar_init(bar_b, 128);
        mbar_init(bar_acc, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 4) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(bar_acc + 8), "n"(kTmemCols1)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = __shfl_sync(kFull, *tmem_slot, 0);

    auto row_live = [&](int r) {
        const int hi = h0 - kKH / 2 + r;
        return hi >= 0 && hi < H && r <= nrows - 1 + kKH - 1;
    };

    if (warp < 4) {
        // ===== builders: B tiles (slot j = 4 - kh, like the 64-channel kernel), then one A tile per live input row =====
        {
            const int co = tid & 63, half = tid >> 6;               // this thread's B row and which 4 of its 8 chunks
            for (int kh = 0; kh < kKH; ++kh) {
                unsigned char* tile = gen + kStages1 * kTileA1 + (kKH - 1 - kh) * kTileB1 + co * 128;
#pragma unroll
                for (int cc = 0; cc < 4; ++cc) {
                    const int c = 4 * half + cc;                    // chunk: taps kw = 2 c, 2 c + 1
                    float2 t0 = make_float2(0.0f, 0.0f), t1 = t0;
                    if (2 * c < kKW) t0 = *reinterpret_cast<const float2*>(weight + (((int64_t)kh * kKW + 2 * c) * kC + co) * 2);
                    if (2 * c + 1 < kKW)
                        t1 = *reinterpret_cast<const float2*>(weight + (((int64_t)kh * kKW + 2 * c + 1) * kC + co) * 2);
                    *reinterpret_cast<float4*>(tile + ((c ^ (co & 7)) << 4)) = make_float4(t0.x, t0.y, t1.x, t1.y);
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar_b) : "memory");
        }
        // live rows are one contiguous range (dead rows lie above / below the image); the window of the NEXT row is
        // fetched into registers before this row's tile is written, so the global-load latency hides behind the stores
        int r_lo = 0, r_hi = -1;
        for (int r = 0; r < kInRows1; ++r)
            if (row_live(r)) { if (r_hi < 0) r_lo = r; r_hi = r; }
        const int wl = w0 + tid - kKW / 2;                          // leftmost frame under this row's window
        auto fetch = [&](int r, float2 (&v)[14]) {
            const float* xrow = x + (((int64_t)b * H + (h0 - kKH / 2 + r)) * W) * 2;
#pragma unroll
            for (int kw = 0; kw < 14; ++kw) {
                const int w = wl + kw;
                v[kw] = (kw < kKW && w >= 0 && w < W) ? *reinterpret_cast<const float2*>(xrow + 2 * (int64_t)w)
                                                       : make_float2(0.0f, 0.0f);
            }
        };
        float2 v[14], vn[14];
        if (r_hi >= r_lo) fetch(r_lo, v);
        int it = 0;
        for (int r = r_lo; r <= r_hi; ++r) {
            const int s = it & (kStages1 - 1);
            if (r < r_hi) fetch(r + 1, vn);
            mbar_wait(bar_empty + 8 * s, (((uint32_t)it >> 2) & 1u) ^ 1u);
            unsigned char* row = gen + s * kTileA1 + tid * 128;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const float4 q = (c < 7) ? make_float4(v[2 * c].x, v[2 * c].y, v[2 * c + 1].x, v[2 * c + 1].y)
                                         : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                *reinterpret_cast<float4*>(row + ((c ^ (tid & 7)) << 4)) = q;
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar_full + 8 * s) : "memory");
#pragma unroll
            for (int kw = 0; kw < 14; ++kw) v[kw] = vn[kw];
            ++it;
        }
        // ===== epilogue =====
        mbar_wait(bar_acc, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int w = w0 + tid;                                     // warp q reads TMEM lanes 32 q .. 32 q + 31
        for (int pr = 0; pr < nrows / 2; ++pr) {
            float* yp = y + (((int64_t)b * (H / 2) + h0 / 2 + pr) * W + w) * kC;
#pragma unroll 1
            for (int half = 0; half < 2; ++half) {
                uint32_t up[32], lo[32];
                const uint32_t taddr = tmem + ((uint32_t)(32 * warp) << 16) + 2 * pr * kC + 32 * half;
                tmem_ld32(taddr, up);
                tmem_ld32(taddr + kC, lo);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (w < W) {
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        float o[4];
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const int c = 32 * half + j + i;
                            const float v2 =
                                fmaxf(__uint_as_float(up[j + i]), __uint_as_float(lo[j + i])) + __ldg(bias + c);
                            o[i] = v2 > 0.0f ? v2 : __ldg(prelu + c) * v2;
                        }
                        *reinterpret_cast<float4*>(yp + 32 * half + j) = make_float4(o[0], o[1], o[2], o[3]);
                    }
                }
            }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    } else {
        // ===== MMA issuer (converged warp, elected lane): input row r feeds accumulators r - kh, K = 32 per kernel row =====
        mbar_wait(bar_b, 0);
        int it = 0;
        uint32_t started = 0;
#pragma unroll
        for (int r = 0; r < kInRows1; ++r) {
            if (!row_live(r)) continue;
            const int s = it & (kStages1 - 1);
            mbar_wait(bar_full + 8 * s, ((uint32_t)it >> 2) & 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t a_lo = umma_desc_lo(a_base) + s * (kTileA1 >> 4);
            const int kh_lo = max(0, r - (nrows - 1)), kh_hi = min(kKH - 1, r);
            int a = r - kh_hi, left = kh_hi - kh_lo + 1;
            while (left > 0) {
                const uint32_t flag = (started >> a) & 1u;
                int n = 1;
                while (n < left && ((started >> (a + n)) & 1u) == flag) ++n;
                const uint32_t b_lo = umma_desc_lo(b_base) + (kKH - 1 - (r - a)) * (kTileB1 >> 4);
                const uint32_t idesc = idesc_tf32(n * kC);
                const uint32_t d = tmem + a * kC;
                if (elect_one()) {
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        umma_tf32(d, umma_desc(a_lo + 2 * k), umma_desc(b_lo + 2 * k), idesc, flag | (k > 0));
                }
                __syncwarp();
                started |= ((1u << n) - 1u) << a;
                a += n;
                left -= n;
            }
            if (elect_one()) umma_commit(bar_empty + 8 * s);
            __syncwarp();
            ++it;
        }
        if (elect_one()) umma_commit(bar_acc);
        __syncwarp();
    }
    __syncthreads();
    if (warp == 4) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(kTmemCols1) : "memory");
    }
}


typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

}  // namespace

static int make_maps(EncodeTiledFn enc, CUtensorMap* tm_x, CUtensorMap* tm_w, const void* x, const void* weight, int B,
                     int H, int W, bool half) {
    const cuuint64_t eb = half ? 2 : 4;                          // bytes per element
    const cuuint32_t row = (cuuint32_t)(128 / eb);               // channels in one 128-byte swizzle row
    const CUtensorMapDataType dt = half ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
    {
        // channels-last activations (B, H, W, 64): box = one 128-byte row of channels x 128 frames of one image row
        const cuuint64_t dims[4] = {(cuuint64_t)kC, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
        const cuuint64_t strides[3] = {(cuuint64_t)kC * eb, (cuuint64_t)W * kC * eb, (cuuint64_t)H * W * kC * eb};
        const cuuint32_t box[4] = {row, (cuuint32_t)kTileW, 1, 1};
        const cuuint32_t es[4] = {1, 1, 1, 1};
        const CUresult r = enc(tm_x, dt, 4, const_cast<void*>(x), dims, strides, box, es,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return fail(MODFX_ERR_CUDA, "cuTensorMapEncodeTiled(activations) failed: %d", (int)r);
    }
    {
        // weights (KH, KW, Cout, Cin) = (tap, out channel, in channel): box = one row of in x 64 out channels of one tap
        const cuuint64_t dims[3] = {(cuuint64_t)kC, (cuuint64_t)kC, (cuuint64_t)(kKH * kKW)};
        const cuuint64_t strides[2] = {(cuuint64_t)kC * eb, (cuuint64_t)kC * kC * eb};
        const cuuint32_t box[3] = {row, (cuuint32_t)kC, 1};
        const cuuint32_t es[3] = {1, 1, 1};
        const CUresult r = enc(tm_w, dt, 3, const_cast<void*>(weight), dims, strides, box, es,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return fail(MODFX_ERR_CUDA, "cuTensorMapEncodeTiled(weights) failed: %d", (int)r);
    }
    return MODFX_OK;
}

// x_lo / w_lo == nullptr: one pass (TF32 on float32 storage, or float16 storage when `half`); otherwise the
// error-compensated three-pass TF32 form
int cnn_conv_tf32(const void* x, const void* x_lo, float* y, int B, int H, int W, int dil, const void* weight,
                  const void* w_lo, const float* bias, const float* prelu, bool half, cudaStream_t stream) {
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return fail(MODFX_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
    MODFX_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(weight) & 15) == 0 &&
                      (reinterpret_cast<uintptr_t>(y) & 15) == 0 && (reinterpret_cast<uintptr_t>(x_lo) & 15) == 0 &&
                      (reinterpret_cast<uintptr_t>(w_lo) & 15) == 0,
                  "x, y and weight must be 16-byte aligned");
    MODFX_REQUIRE((x_lo == nullptr) == (w_lo == nullptr), "x_lo and w_lo go together");
    const bool split = x_lo != nullptr;
    MODFX_REQUIRE(!(split && half), "the three-pass form is TF32 only");
    ConvMaps tm;
    int st = make_maps(enc, &tm.x[0], &tm.w[0], x, weight, B, H, W, half);
    if (st != MODFX_OK) return st;
    st = make_maps(enc, &tm.x[1], &tm.w[1], split ? x_lo : x, split ? w_lo : weight, B, H, W, half);
    if (st != MODFX_OK) return st;
    const dim3 grid((W + kTileW - 1) / kTileW, (H + kRows - 1) / kRows, B);
    if (half)
        return launch(conv_tf32_kernel<true>, grid, kThreads, Fmt<true>::kSmemBytes, stream, tm, 1, y, H, W, dil, bias, prelu);
    return launch(conv_tf32_kernel<false>, grid, kThreads, Fmt<false>::kSmemBytes, stream, tm, split ? 3 : 1, y, H, W, dil,
                  bias, prelu);
}

int cnn_conv1_tf32(const float* x, float* y, int B, int H, int W, const float* weight, const float* bias,
                   const float* prelu, cudaStream_t stream) {
    MODFX_REQUIRE((reinterpret_cast<uintptr_t>(x) & 7) == 0 && (reinterpret_cast<uintptr_t>(weight) & 7) == 0 &&
                      (reinterpret_cast<uintptr_t>(y) & 15) == 0,
                  "x and weight must be 8-byte, y 16-byte aligned");
    MODFX_CUDA_OK(cudaFuncSetAttribute(conv1_tf32_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                       cudaSharedmemCarveoutMaxShared));
    return launch(conv1_tf32_kernel, dim3((W + kTileW - 1) / kTileW, (H + kRows1 - 1) / kRows1, B), kThreads1, kSmemBytes1,
                  stream, x, y, H, W, weight, bias, prelu);
}

}  // namespace modfx
