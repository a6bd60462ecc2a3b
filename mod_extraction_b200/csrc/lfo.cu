// LFO synthesis (make_mod_signal, reference mod_extraction/modulations.py:16-57) and
// linear resampling (util.linear_interpolate_last_dim, reference mod_extraction/util.py:15-29)
// as stand-alone batched kernels.  In the render path both are fused into the effect kernels
// (fc.cu); these entry points serve callers that want the signals themselves
// (make_rand_mod_signal, the phaser ground-truth LFO of datasets.py:442-450, targets at 345 frames).
#include "common.cuh"

namespace modfx {
namespace {

// modulations.py:26-29: make_mod_signal halves frequency and phase for the rectified shapes (exact in float32)
__device__ __forceinline__ bool is_rect(int shape) {
    return shape == MODFX_SHAPE_RECT_COS || shape == MODFX_SHAPE_INV_RECT_COS;
}

// make_mod_signal(len, len, 1.0, 0.0, shape) of one section of make_combined_mod_sig, modulations.py:208
__device__ __forceinline__ LfoDesc section_lfo(int shape, float len) {
    return make_lfo_desc(is_rect(shape) ? 0.5f : 1.0f, 0.0f, shape, 1.0f, len);
}

__global__ void __launch_bounds__(256) lfo_kernel(float* __restrict__ out, int64_t n, float sr,
                                                  const float* __restrict__ freq, const float* __restrict__ phase,
                                                  const int32_t* __restrict__ shape, const float* __restrict__ exp_) {
    const int b = blockIdx.y;
    const LfoDesc d = make_lfo_desc(freq[b], phase[b], shape[b], exp_ ? exp_[b] : 1.0f, sr);
    float* o = out + (int64_t)b * n;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        o[i] = lfo_value(d, i);
}

// ATen upsample_linear1d: align_corners=True reads source position scale * i with scale = (I - 1) / (O - 1),
// align_corners=False src = max(fma(scale, i + 0.5, -0.5), 0) with scale = I / O.
__global__ void __launch_bounds__(256) interp_kernel(const float* __restrict__ in, float* __restrict__ out,
                                                     int64_t I, int64_t O, float scale, int align_corners) {
    const float* xi = in + (int64_t)blockIdx.y * I;
    float* yo = out + (int64_t)blockIdx.y * O;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < O; i += (int64_t)gridDim.x * blockDim.x) {
        float src;
        if (align_corners) src = __fmul_rn(scale, (float)i);
        else src = fmaxf(__fmaf_rn(scale, __fadd_rn((float)i, 0.5f), -0.5f), 0.0f);
        const LinearTaps<int64_t> t = linear_taps(src, I);
        yo[i] = blend(t, xi[t.i0], xi[t.i1]);
    }
}

}  // namespace
}  // namespace modfx

using namespace modfx;

extern "C" int modfx_lfo_f32(float* out, int32_t B, int64_t n, float sr, const float* freq, const float* phase,
                             const int32_t* shape, const float* exp_or_null, void* stream) {
    MODFX_REQUIRE(out && freq && phase && shape, "NULL pointer");
    MODFX_REQUIRE(B >= 0 && n >= 1 && sr > 0.0f, "bad arguments B=%d n=%lld sr=%g", B, (long long)n, sr);
    if (B == 0) return MODFX_OK;
    dim3 grid;
    if (const int st = row_grid(grid, n, B, 1024)) return st;
    return launch(lfo_kernel, grid, 256, 0, as_stream(stream), out, n, sr, freq, phase, shape, exp_or_null);
}

extern "C" int modfx_interp_linear_f32(const float* in, float* out, int64_t rows, int64_t I, int64_t O,
                                       int32_t align_corners, void* stream) {
    MODFX_REQUIRE(in && out, "NULL pointer");
    MODFX_REQUIRE(rows >= 0 && I >= 1 && O >= 1, "bad shape rows=%lld I=%lld O=%lld", (long long)rows, (long long)I, (long long)O);
    if (rows == 0) return MODFX_OK;
    dim3 grid;
    if (const int st = row_grid(grid, O, rows, 2048)) return st;
    float scale;
    if (align_corners) scale = upsample_scale_ac(I, O);
    else scale = (float)I / (float)O;
    return launch(interp_kernel, grid, 256, 0, as_stream(stream), in, out, I, O, scale, align_corners);
}

// ---------------------------------------------------------------------------------------------
// Control-rate helpers of the RNG-driven LFO variants (quasi-periodic, combined).  The random
// draws and the integer bookkeeping stay on the host (torch global CPU generator, SURVEY H6);
// every float32 operation of the reference happens here.
namespace modfx {
namespace {

// find_corners, reference modulations.py:219-238, as two flag rows
__global__ void __launch_bounds__(256) corners_kernel(const float* __restrict__ mod, uint8_t* __restrict__ top,
                                                      uint8_t* __restrict__ bottom, int64_t n) {
    const float* m = mod + (int64_t)blockIdx.y * n;
    uint8_t* t = top + (int64_t)blockIdx.y * n;
    uint8_t* bt = bottom + (int64_t)blockIdx.y * n;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const unsigned f = corner_flags(m, i, n);
        t[i] = f & 1u;
        bt[i] = f >> 1;
    }
}

// make_combined_mod_sig's overwrite loop, reference modulations.py:203-209: section s of example b
// covers out[start, start+len) with make_mod_signal(len, len, 1.0, 0.0, shape); later sections win
// at the shared end point, which is what "largest start <= i" selects.
__global__ void __launch_bounds__(256) lfo_sections_kernel(float* __restrict__ out, int64_t n,
                                                           const int32_t* __restrict__ sec_off,
                                                           const int32_t* __restrict__ sec_start,
                                                           const int32_t* __restrict__ sec_len,
                                                           const int32_t* __restrict__ sec_shape) {
    const int b = blockIdx.y;
    const int s0 = sec_off[b], s1 = sec_off[b + 1];
    if (s0 == s1) return;
    float* o = out + (int64_t)b * n;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        int sec = -1;
        for (int s = s0; s < s1; ++s)
            if (sec_start[s] <= i && i < sec_start[s] + sec_len[s]) sec = s;
        if (sec < 0) continue;
        o[i] = lfo_value(section_lfo(sec_shape[sec], (float)sec_len[sec]), i - sec_start[sec]);
    }
}

// make_quasi_periodic's concatenation, reference modulations.py:139-159: output positions
// [out_start, out_start + out_len) of example b hold the first out_len points of section
// in[in_start, in_start + in_len) resampled to new_len points (align_corners=True).
__global__ void __launch_bounds__(256) stretch_sections_kernel(const float* __restrict__ in, float* __restrict__ out,
                                                               int64_t n, const int32_t* __restrict__ sec_off,
                                                               const int32_t* __restrict__ in_start,
                                                               const int32_t* __restrict__ in_len,
                                                               const int32_t* __restrict__ new_len,
                                                               const int32_t* __restrict__ out_start) {
    const int b = blockIdx.y;
    const int s0 = sec_off[b], s1 = sec_off[b + 1];
    const float* x = in + (int64_t)b * n;
    float* o = out + (int64_t)b * n;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        if (s0 == s1) {         // fewer than two corners: signal returned unchanged (modulations.py:136-137)
            o[i] = x[i];
            continue;
        }
        int sec = s0;
        for (int s = s0; s < s1; ++s)
            if (out_start[s] <= i) sec = s;
        const int j = (int)i - out_start[sec];
        const int I = in_len[sec], O = new_len[sec];
        const float* xs = x + in_start[sec];
        o[i] = (I == O) ? xs[j] : upsample_ac(xs, I, upsample_scale_ac_dev(I, O), j);
    }
}

}  // namespace
}  // namespace modfx

extern "C" int modfx_find_corners_f32(const float* mod, uint8_t* top, uint8_t* bottom, int64_t rows, int64_t n,
                                      void* stream) {
    MODFX_REQUIRE(mod && top && bottom, "NULL pointer");
    MODFX_REQUIRE(rows >= 0 && n >= 1, "bad shape");
    if (rows == 0) return MODFX_OK;
    dim3 grid;
    if (const int st = row_grid(grid, n, rows, 256)) return st;
    return launch(corners_kernel, grid, 256, 0, as_stream(stream), mod, top, bottom, n);
}

extern "C" int modfx_lfo_sections_f32(float* out, int32_t B, int64_t n, const int32_t* sec_off,
                                      const int32_t* sec_start, const int32_t* sec_len, const int32_t* sec_shape,
                                      void* stream) {
    MODFX_REQUIRE(out && sec_off && sec_start && sec_len && sec_shape, "NULL pointer");
    MODFX_REQUIRE(B >= 0 && n >= 1, "bad shape");
    if (B == 0) return MODFX_OK;
    dim3 grid;
    if (const int st = row_grid(grid, n, B, 256)) return st;
    return launch(lfo_sections_kernel, grid, 256, 0, as_stream(stream), out, n, sec_off, sec_start, sec_len, sec_shape);
}

extern "C" int modfx_stretch_sections_f32(const float* in, float* out, int32_t B, int64_t n, const int32_t* sec_off,
                                          const int32_t* in_start, const int32_t* in_len, const int32_t* new_len,
                                          const int32_t* out_start, void* stream) {
    MODFX_REQUIRE(in && out && sec_off && in_start && in_len && new_len && out_start, "NULL pointer");
    MODFX_REQUIRE(B >= 0 && n >= 1, "bad shape");
    if (B == 0) return MODFX_OK;
    dim3 grid;
    if (const int st = row_grid(grid, n, B, 256)) return st;
    return launch(stretch_sections_kernel, grid, 256, 0, as_stream(stream), in, out, n, sec_off, in_start, in_len,
                  new_len, out_start);
}

// ---------------------------------------------------------------------------------------------
// make_combined_mod_sig for a whole batch without a host round trip (reference modulations.py:191-210, called per
// example at datasets.py:375-380).  The reference draws, per example, one base shape and then one shape per span
// between consecutive bottom corners of the base signal -- a data-dependent number of draws from the torch global
// CPU generator.  The caller hands over the generator's next raw 32-bit words (mod_extraction_b200/_rng.py: one
// word per util.choice); the device replays the draw order:
//   1. every candidate base shape of every example is rendered (combined_cand_kernel);
//   2. the bottom corners of every candidate are listed (corner_list_kernel, one warp per row);
//   3. ONE thread walks the examples in order: base = shapes[word % S], sections = corners - 1, next example starts
//      1 + sections words later (combined_scan_kernel) -- integer work only, fed from shared memory;
//   4. every example takes its base candidate and overwrites the spans with make_mod_signal(len, len, 1.0, 0.0, shape)
//      (combined_fill_kernel; later spans win at shared end points like the reference's in-order slice assignment).
// The number of words consumed comes back so the host can advance the generator by exactly that much.
namespace modfx {
namespace {

constexpr int kMaxCorners = 64;     // bottom corners listed per candidate row (a 2 s control-rate LFO below 30 Hz has fewer)

__global__ void __launch_bounds__(256) combined_cand_kernel(float* __restrict__ cand, int n, float sr,
                                                            const float* __restrict__ freq, const float* __restrict__ phase,
                                                            const int32_t* __restrict__ shapes, int S) {
    const int row = blockIdx.y;                 // b * S + k
    const int b = row / S, k = row - b * S;
    const int shape = shapes[k];
    const bool rect = is_rect(shape);
    const LfoDesc d = make_lfo_desc(rect ? freq[b] * 0.5f : freq[b], rect ? phase[b] * 0.5f : phase[b], shape, 1.0f, sr);
    float* o = cand + (int64_t)row * n;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) o[i] = lfo_value(d, i);
}

// bottom corners of find_corners (modulations.py:219-238), as an index list per row
__global__ void __launch_bounds__(128) corner_list_kernel(const float* __restrict__ mod, int rows, int n,
                                                          int16_t* __restrict__ idx, int32_t* __restrict__ cnt) {
    const int row = blockIdx.x * (blockDim.x / kWarp) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows) return;
    const float* m = mod + (int64_t)row * n;
    int16_t* out = idx + (int64_t)row * kMaxCorners;
    int c = 0;
    for (int i0 = 0; i0 < n; i0 += kWarp) {
        const int i = i0 + lane;
        const bool fb = corner_flags(m, i, n) & 2u;
        const unsigned bal = __ballot_sync(kFull, fb);
        if (fb) {
            const int pos = c + __popc(bal & ((1u << lane) - 1u));
            if (pos < kMaxCorners) out[pos] = (int16_t)i;
        }
        c += __popc(bal);
    }
    if (lane == 0) cnt[row] = c;
}

// Step 3: the chain  off(b+1) = off(b) + 1 + sections(b, words[off(b)] % S)  is serial by construction.  One CTA stages
// what the chain touches in shared memory -- the corner counts of a tile of examples (all S candidates) and a window of
// generator words starting at the current offset -- and thread 0 walks the tile at shared-memory latency (two dependent
// byte loads per example -- the choice `word mod S` and the number of words each candidate would consume are computed by
// all threads while staging -- instead of two dependent L2 round trips: 2 ms -> 0.1 ms for 4096 examples).
constexpr int kScanThreads = 256;
constexpr int kScanWords = 16384;           // words staged per window, reduced to (word mod S) bytes
constexpr int kScanCnt = 16384;             // word increments staged per tile (one byte per example and candidate)

__global__ void __launch_bounds__(kScanThreads) combined_scan_kernel(const uint32_t* __restrict__ words, int64_t n_words,
                                                                     const int32_t* __restrict__ cnt, int B, int S,
                                                                     int32_t* __restrict__ base, int32_t* __restrict__ woff,
                                                                     int32_t* __restrict__ consumed) {
    __shared__ uint8_t sk[kScanWords];      // util.choice of every word of the window: word mod S (modulations.py:196)
    __shared__ uint8_t sinc[kScanCnt];      // words example b consumes if it draws candidate k: 1 + sections (:203-204)
    __shared__ long long s_off;
    __shared__ int s_b, s_err;
    const int tid = threadIdx.x;
    const int tile = max(1, kScanCnt / S);                              // examples per tile
    if (tid == 0) { s_off = 0; s_b = 0; s_err = 0; }
    __syncthreads();
    int tile_lo = -1;
    while (true) {
        const int b0 = s_b;
        const long long off0 = s_off;
        if (b0 >= B) break;
        const int t_lo = b0 / tile * tile, t_hi = min(t_lo + tile, B);
        if (t_lo != tile_lo) {
            for (int i = tid; i < (t_hi - t_lo) * S; i += kScanThreads) {
                const int c = cnt[(int64_t)t_lo * S + i];               // 255: more corners than the list holds -- an error
                sinc[i] = (uint8_t)(c > kMaxCorners ? 255 : 1 + ((c > 1) ? c - 1 : 0));      // only if that candidate is drawn
            }
            tile_lo = t_lo;
        }
        const int n_win = (int)min((long long)kScanWords, (long long)n_words - off0);
        for (int i = tid; i < n_win; i += kScanThreads) sk[i] = (uint8_t)(words[off0 + i] % (uint32_t)S);
        __syncthreads();
        if (tid == 0) {
            long long off = off0;
            int b = b0, err = s_err;
            for (; b < t_hi; ++b) {
                if (off >= n_words) {                                   // out of words: flag it, the rest gets base 0
                    err = err ? err : 1;
                    woff[b] = (int32_t)off;
                    base[b] = 0;
                    continue;
                }
                const int rel = (int)(off - off0);
                if (rel >= n_win) break;                                // next window
                woff[b] = (int32_t)off;
                const int k = sk[rel];
                base[b] = k;
                const int inc = sinc[(b - t_lo) * S + k];
                if (inc == 255) err = 2;                                // more corners than the list holds
                off += inc;
            }
            s_off = off; s_b = b; s_err = err;
        }
        __syncthreads();
    }
    if (tid == 0) {
        const long long off = s_off;
        woff[B] = (int32_t)off;
        consumed[0] = (int32_t)off;
        consumed[1] = (off > n_words && s_err == 0) ? 1 : s_err;
    }
}

__global__ void __launch_bounds__(256) combined_fill_kernel(float* __restrict__ out, int n, const float* __restrict__ cand,
                                                            const int16_t* __restrict__ idx, const int32_t* __restrict__ cnt,
                                                            const int32_t* __restrict__ base, const int32_t* __restrict__ woff,
                                                            const uint32_t* __restrict__ words,
                                                            const int32_t* __restrict__ shapes, int S) {
    __shared__ int16_t cs[kMaxCorners];
    const int b = blockIdx.y;
    const int row = b * S + base[b];
    const int c = min(cnt[row], kMaxCorners);
    for (int i = threadIdx.x; i < c; i += blockDim.x) cs[i] = idx[(int64_t)row * kMaxCorners + i];
    __syncthreads();
    const float* src = cand + (int64_t)row * n;
    float* o = out + (int64_t)b * n;
    const int64_t w0 = woff[b] + 1;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float v = src[i];
        if (c > 1 && i >= cs[0] && i <= cs[c - 1]) {
            // span s covers [corner s, corner s + 1]; spans are assigned in order, so a shared end point keeps the later one
            int s = 0;
            for (int j = 1; j <= c - 2; ++j)
                if (cs[j] <= i) s = j;
            const int start = cs[s];
            const float len = (float)(cs[s + 1] - start + 1);
            const int shape = shapes[words[w0 + s] % (uint32_t)S];      // util.choice(shapes), modulations.py:207
            v = lfo_value(section_lfo(shape, len), i - start);
        }
        o[i] = v;
    }
}

int64_t align256(int64_t v) { return (v + 255) / 256 * 256; }

}  // namespace
}  // namespace modfx

extern "C" int64_t modfx_combined_lfo_workspace_bytes(int32_t B, int64_t n, int32_t n_shapes) {
    if (B <= 0 || n <= 0 || n_shapes <= 0) return 0;
    const int64_t rows = (int64_t)B * n_shapes;
    return align256(rows * n * 4) + align256(rows * kMaxCorners * 2) + align256(rows * 4) + align256(((int64_t)B + 1) * 4);
}

extern "C" int modfx_combined_lfo_f32(float* out, int32_t B, int64_t n, float sr, const float* freq, const float* phase,
                                      const int32_t* shapes, int32_t n_shapes, const uint32_t* words, int64_t n_words,
                                      int32_t* base_out, int32_t* consumed_out, void* workspace, void* stream) {
    MODFX_REQUIRE(out && freq && phase && shapes && words && base_out && consumed_out && workspace, "NULL pointer");
    MODFX_REQUIRE(B >= 0 && n >= 3 && n <= 32767 && sr > 0.0f, "bad arguments B=%d n=%lld sr=%g", B, (long long)n, sr);
    MODFX_REQUIRE(n_shapes >= 1 && n_shapes <= 64 && n_words >= 0, "bad shape list / word count");
    if (B == 0) return MODFX_OK;
    const int64_t rows = (int64_t)B * n_shapes;
    dim3 cand_grid, fill_grid;
    if (const int st = row_grid(cand_grid, n, rows, 64)) return st;
    if (const int st = row_grid(fill_grid, n, B, 64)) return st;
    char* w = static_cast<char*>(workspace);
    float* cand = reinterpret_cast<float*>(w);          w += align256(rows * n * 4);
    int16_t* idx = reinterpret_cast<int16_t*>(w);       w += align256(rows * kMaxCorners * 2);
    int32_t* cnt = reinterpret_cast<int32_t*>(w);       w += align256(rows * 4);
    int32_t* woff = reinterpret_cast<int32_t*>(w);
    cudaStream_t s = as_stream(stream);
    int st = launch(combined_cand_kernel, cand_grid, 256, 0, s, cand, (int)n, sr, freq, phase, shapes, n_shapes);
    if (st == MODFX_OK)
        st = launch(corner_list_kernel, (unsigned)((rows + 3) / 4), 128, 0, s, cand, (int)rows, (int)n, idx, cnt);
    if (st == MODFX_OK)
        st = launch(combined_scan_kernel, 1, kScanThreads, 0, s, words, n_words, cnt, B, n_shapes, base_out, woff,
                    consumed_out);
    if (st == MODFX_OK)
        st = launch(combined_fill_kernel, fill_grid, 256, 0, s, out, (int)n, cand, idx, cnt, base_out, woff, words, shapes,
                    n_shapes);
    return st;
}

// ---------------------------------------------------------------------------------------------
// Ground-truth LFO of PedalboardPhaserDataset.__getitem__ (datasets.py:442-450) without the audio-rate signal:
//   mod = make_mod_signal(proc_n, sr, rate, phase, shape)[start : start + n_window]      (datasets.py:442, 448)
//   out = linear_interpolate_last_dim(mod, n_out, align_corners=True)                    (datasets.py:450)
// Element i of out only needs the two LFO values around scale * i inside the window, and make_mod_signal has a closed
// form per element (lfo_value), so each output is two evaluations and the blend of util.py:15-29.
namespace modfx {
namespace {
__global__ void __launch_bounds__(256) lfo_window_kernel(float* __restrict__ out, int n_out, int n_window, float sr,
                                                         const float* __restrict__ freq, const float* __restrict__ phase,
                                                         const int32_t* __restrict__ shape, const float* __restrict__ exp_,
                                                         const int32_t* __restrict__ start) {
    const int b = blockIdx.y;
    const LfoDesc d = make_lfo_desc(freq[b], phase[b], shape[b], exp_ ? exp_[b] : 1.0f, sr);
    const int s0 = start ? start[b] : 0;
    const float scale = upsample_scale_ac_dev(n_window, n_out);
    float* o = out + (int64_t)b * n_out;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_out; i += gridDim.x * blockDim.x) {
        if (n_out == n_window) {                            // util.py:18-19: same length => untouched
            o[i] = lfo_value(d, s0 + i);
            continue;
        }
        const LinearTaps<int> t = taps_ac(scale, i, n_window);
        o[i] = blend(t, lfo_value(d, s0 + t.i0), lfo_value(d, s0 + t.i1));
    }
}
}  // namespace
}  // namespace modfx

extern "C" int modfx_lfo_window_f32(float* out, int32_t B, int64_t n_out, int64_t n_window, float sr, const float* freq,
                                    const float* phase, const int32_t* shape, const float* exp_or_null,
                                    const int32_t* start_or_null, void* stream) {
    MODFX_REQUIRE(out && freq && phase && shape, "NULL pointer");
    MODFX_REQUIRE(B >= 0 && n_out >= 1 && n_window >= 1 && n_window < (1ll << 30) && n_out <= n_window && sr > 0.0f,
                  "bad arguments B=%d n_out=%lld n_window=%lld", B, (long long)n_out, (long long)n_window);
    if (B == 0) return MODFX_OK;
    dim3 grid;
    if (const int st = row_grid(grid, n_out, B, 256)) return st;
    return launch(lfo_window_kernel, grid, 256, 0, as_stream(stream), out, (int)n_out, (int)n_window, sr, freq, phase,
                  shape, exp_or_null, start_or_null);
}
