/*
 * modfx.h -- C ABI of libmodfx.so: B200 (sm_100a) renderer for the effect hot path of
 * christhetree/mod_extraction.
 *
 * The reference has no FFI layer; its boundary for this path is a set of Python
 * signatures (SURVEY.md section 8b).  Each entry point below names the reference
 * interface it replaces (file:line relative to the reference root).  All pointers
 * named *_dev / x / y / mod are DEVICE pointers unless the function name ends in
 * _host; everything is float32, contiguous, row-major.  `stream` is a cudaStream_t
 * passed as void* (0 = legacy default stream).  Calls are asynchronous on `stream`
 * (the _host variants synchronise before returning).  No hidden state is kept
 * between calls; calls on different streams may run concurrently.
 *
 * Every function returns MODFX_OK (0) or a negative modfx_status; on failure
 * modfx_last_error() returns a thread-local message.  There is no CPU fallback:
 * without a CUDA device every compute entry point returns MODFX_ERR_CUDA.
 */
#ifndef MODFX_H_
#define MODFX_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MODFX_ABI_VERSION 1

typedef enum {
    MODFX_OK = 0,
    MODFX_ERR_INVALID = -1,      /* bad shape / null pointer / out-of-range scalar */
    MODFX_ERR_UNSUPPORTED = -2,  /* valid request the kernels do not cover (e.g. delay line > smem) */
    MODFX_ERR_CUDA = -3          /* CUDA runtime error (message holds cudaGetErrorString) */
} modfx_status;

/* LFO shapes of make_mod_signal, mod_extraction/modulations.py:25 */
typedef enum {
    MODFX_SHAPE_COS = 0,
    MODFX_SHAPE_RECT_COS = 1,
    MODFX_SHAPE_INV_RECT_COS = 2,
    MODFX_SHAPE_TRI = 3,
    MODFX_SHAPE_SAW = 4,
    MODFX_SHAPE_RSAW = 5,
    MODFX_SHAPE_SQR = 6
} modfx_shape;

/*
 * A per-example effect parameter: the reference accepts `Union[float, Tensor(B,)]`
 * (fx.py:75-79).  dev != NULL  -> (B,) float32 device array (torch-tensor semantics:
 * float32 arithmetic); dev == NULL -> python-float semantics: `value` is combined with
 * other python numbers in double and rounded to float32 where it meets a tensor.
 */
typedef struct {
    const float* dev;
    double value;
} modfx_param;

/* Where the modulation signal comes from. */
typedef enum {
    MODFX_MOD_AUDIO_RATE = 0,   /* mod (B,N) or (B,C,N) float32: the literal forward(x, mod_sig) */
    MODFX_MOD_CONTROL_RATE = 1, /* mod (B,n_lo): upsampled in-kernel exactly like
                                   util.linear_interpolate_last_dim(mod, N) (util.py:15-29,
                                   called at data_modules.py:454-455) */
    MODFX_MOD_LFO = 2           /* synthesised in-kernel from per-example LFO parameters like
                                   make_mod_signal(n_lo, sr_lo, freq, phase, shape, exp)
                                   (modulations.py:16-57; datasets.py:382), then upsampled
                                   to N as above when n_lo != N */
} modfx_mod_kind;

typedef struct {
    int32_t kind;            /* modfx_mod_kind */
    const float* mod;        /* AUDIO_RATE / CONTROL_RATE */
    int32_t mod_has_ch;      /* AUDIO_RATE: 1 if mod is (B,C,N), 0 if (B,N) */
    int64_t n_lo;            /* CONTROL_RATE / LFO: points per example */
    float sr_lo;             /* LFO: sample rate the LFO is generated at */
    const float* lfo_freq;   /* LFO: (B,) Hz  (already halved for rect shapes, modulations.py:26-29) */
    const float* lfo_phase;  /* LFO: (B,) rad (already halved for rect shapes) */
    const int32_t* lfo_shape;/* LFO: (B,) modfx_shape */
    const float* lfo_exp;    /* LFO: (B,) exponent, or NULL for 1.0 */
} modfx_mod_source;

int modfx_abi_version(void);
const char* modfx_last_error(void);
/* Number of CUDA devices visible to the library (0 if none / no driver). */
int modfx_device_count(void);

/*
 * Replaces MonoFlangerChorusModule.forward / apply_effect, mod_extraction/fx.py:72-130
 * (ctor arithmetic fx.py:40-42 gives Mmin, Mlfo).  Bit-exact with the reference for
 * identical x / mod / parameters (IEEE round-to-nearest, no FMA contraction).
 *   x, y          (B, C, N)
 *   example_index optional (n_items,) int32: render only these examples (rows of x / y /
 *                 mod / parameter arrays are still indexed by the example id); NULL = all B.
 */
int modfx_flanger_chorus_f32(const float* x, float* y, int32_t B, int32_t C, int64_t N,
                             int32_t max_min_delay_samples, int32_t max_lfo_delay_samples,
                             const modfx_mod_source* mod,
                             modfx_param feedback, modfx_param min_delay_width, modfx_param width,
                             modfx_param depth, modfx_param mix,
                             const int32_t* example_index, int32_t n_items, void* stream);

/*
 * The same delay line with first-order ALL-PASS instead of linear fractional-delay interpolation (north_star names
 * "linear or all-pass"; the reference, fx.py:113, only has the linear blend -- this mode is this library's own
 * definition, restated in oracle/modfx_oracle.c: it[n] = eta * (buf[q] - it[n-1]) + buf[p], eta = fr / (2 - fr)).
 * Same arguments as modfx_flanger_chorus_f32; the modulation signal must come from memory (AUDIO_RATE / CONTROL_RATE).
 */
int modfx_flanger_chorus_allpass_f32(const float* x, float* y, int32_t B, int32_t C, int64_t N,
                                     int32_t max_min_delay_samples, int32_t max_lfo_delay_samples,
                                     const modfx_mod_source* mod,
                                     modfx_param feedback, modfx_param min_delay_width, modfx_param width,
                                     modfx_param depth, modfx_param mix,
                                     const int32_t* example_index, int32_t n_items, void* stream);

/* Replaces apply_tremolo, mod_extraction/fx.py:13-22. */
int modfx_tremolo_f32(const float* x, float* y, int32_t B, int32_t C, int64_t N,
                      const modfx_mod_source* mod, modfx_param mix, void* stream);

/*
 * Replaces make_mod_signal / make_rand_mod_signal's inner call, modulations.py:16-57,98:
 * out (B, n) = LFO per example.  freq/phase already halved for rect shapes.
 */
int modfx_lfo_f32(float* out, int32_t B, int64_t n, float sr, const float* freq, const float* phase,
                  const int32_t* shape, const float* exp_or_null, void* stream);

/*
 * Ground-truth LFO of PedalboardPhaserDataset.__getitem__, mod_extraction/datasets.py:442-450, without materialising
 * the audio-rate signal: out (B, n_out) = linear_interpolate_last_dim(make_mod_signal(..)[start[b] : start[b] + n_window],
 * n_out, align_corners=True).  freq / phase already halved for rect shapes; start may be NULL (0).
 */
int modfx_lfo_window_f32(float* out, int32_t B, int64_t n_out, int64_t n_window, float sr, const float* freq,
                         const float* phase, const int32_t* shape, const float* exp_or_null,
                         const int32_t* start_or_null, void* stream);

/* Replaces util.linear_interpolate_last_dim, mod_extraction/util.py:15-29 (F.interpolate
 * mode="linear").  in (rows, I) -> out (rows, O). */
int modfx_interp_linear_f32(const float* in, float* out, int64_t rows, int64_t I, int64_t O,
                            int32_t align_corners, void* stream);

/*
 * Control-rate pieces of the RNG-driven LFO variants.  The random draws and the integer section
 * bookkeeping stay with the caller (torch global CPU generator, reference util.py:32-49); the
 * float32 arithmetic of the reference runs here.
 *
 * modfx_find_corners_f32      replaces find_corners, modulations.py:219-238:
 *                             mod (rows, n) -> top / bottom (rows, n) uint8 flags.
 * modfx_lfo_sections_f32      replaces the overwrite loop of make_combined_mod_sig,
 *                             modulations.py:203-209: sections [sec_off[b], sec_off[b+1]) of example b
 *                             overwrite out[b, start : start+len) with
 *                             make_mod_signal(len, len, 1.0, 0.0, shape); later sections win.
 * modfx_stretch_sections_f32  replaces the section stretching + concatenation of make_quasi_periodic,
 *                             modulations.py:139-159: out[b, out_start[s] ...) = first points of
 *                             linear_interpolate_last_dim(in[b, in_start : in_start+in_len], new_len);
 *                             an example without sections is copied unchanged.
 */
int modfx_find_corners_f32(const float* mod, uint8_t* top, uint8_t* bottom, int64_t rows, int64_t n,
                           void* stream);
int modfx_lfo_sections_f32(float* out, int32_t B, int64_t n, const int32_t* sec_off,
                           const int32_t* sec_start, const int32_t* sec_len, const int32_t* sec_shape,
                           void* stream);
int modfx_stretch_sections_f32(const float* in, float* out, int32_t B, int64_t n, const int32_t* sec_off,
                               const int32_t* in_start, const int32_t* in_len, const int32_t* new_len,
                               const int32_t* out_start, void* stream);

/*
 * Replaces make_combined_mod_sig, mod_extraction/modulations.py:191-210, for a batch of (freq, phase) pairs as
 * datasets.py:375-380 calls it per example, WITHOUT a host round trip: the caller passes the next raw 32-bit
 * outputs of the torch global CPU generator (mt19937; one word per util.choice, util.py:32-42) and the device
 * replays the reference's draw order -- per example one base shape, then one shape per span between consecutive
 * bottom corners of the base signal.
 *   out        (B, n) float32
 *   freq/phase (B,) as make_mod_signal receives them (NOT halved for the rectified shapes; done here)
 *   shapes     (n_shapes,) modfx_shape ids of the candidate list
 *   words      (n_words,) uint32 raw generator outputs, device
 *   base_out   (B,) int32: index into shapes of the base shape each example drew
 *   consumed_out (2,) int32 device: [0] words consumed (advance the generator by this many), [1] error flag
 *              (1: n_words too small, 2: more than 64 bottom corners in a base signal) -- on error `out` is invalid
 *   workspace  modfx_combined_lfo_workspace_bytes(B, n, n_shapes) bytes
 */
int64_t modfx_combined_lfo_workspace_bytes(int32_t B, int64_t n, int32_t n_shapes);
int modfx_combined_lfo_f32(float* out, int32_t B, int64_t n, float sr, const float* freq, const float* phase,
                           const int32_t* shapes, int32_t n_shapes, const uint32_t* words, int64_t n_words,
                           int32_t* base_out, int32_t* consumed_out, void* workspace, void* stream);

/*
 * Post-processing of extracted LFOs (eval path), mod_extraction/modulations.py:259-362.  Rows are
 * independent (n frames each, 345 for 2 s of audio); all float32 arithmetic in the reference's order.
 *   modfx_smoothen_f32         replaces smoothen, modulations.py:358-362: out (rows, n - window + 1) =
 *                              moving average of in (rows, n) over `window` frames, no padding.
 *   modfx_stretch_corners_f32  replaces find_corners + _stretch_corners of stretch_corners,
 *                              modulations.py:259-307, applied to an already smoothed signal: every
 *                              stretch between neighbouring corners is rescaled so that top corners reach
 *                              1.0 and bottom corners 0.0; rows with more than max_n_corners corners
 *                              are copied unchanged.  in and out must not alias.
 *   modfx_check_mod_sig_f32    replaces check_mod_sig / find_valid_mod_sig_indices, modulations.py:311-355:
 *                              valid[r] = 1 when row r has min..max top and bottom corners and neighbouring
 *                              corners of a kind are at least min_frames apart.
 */
int modfx_smoothen_f32(const float* in, float* out, int64_t rows, int64_t n, int32_t window, void* stream);
int modfx_stretch_corners_f32(const float* in, float* out, int64_t rows, int64_t n, int32_t max_n_corners,
                              void* stream);
int modfx_check_mod_sig_f32(const float* in, uint8_t* valid, int64_t rows, int64_t n, int32_t min_top,
                            int32_t max_top, int32_t min_bottom, int32_t max_bottom, int32_t min_frames,
                            void* stream);

/*
 * Replaces Spectral2DCNN.spectrogram + clip + log, mod_extraction/models.py:170-175,199,207-208
 * (torchaudio MelSpectrogram n_fft=1024, hop 256, center/reflect, periodic Hann, power 2).
 *   x         (R, T) rows = batch*channels
 *   out       (R, n_mels, T/hop + 1)
 *   window    (n_fft,) device
 *   fb_start, fb_count (n_mels,) int32 device: first FFT bin and number of taps of each mel band
 *   fb_weight (n_mels, fb_stride) float32 device: tap weights, zero padded
 *   fb_taps   sum of fb_count (the kernel keeps a compact copy of the table in shared memory)
 *   x_row_stride / out_row_stride: distance in floats between consecutive rows of x / out (0 = dense:
 *             T and n_mels*n_frames); row_index: optional (n_index,) int32 list of the rows to process
 *             (NULL = all R).  Together they let dry and wet audio live in separate buffers while the
 *             result lands in the (B, 2, n_mels, n_frames) tensor the extractor consumes, and let the
 *             dry half start before the effects have finished.
 *   apply_log 1: out = log(max(mel, eps)) (models.py:207-208); 0: out = mel power, which is what
 *             the `spectrogram` attribute itself returns (SpecAugment sits between the two in
 *             training, models.py:201-205)
 * Supported: n_fft == 1024, even hop in [2, 512].
 */
int modfx_logmel_f32(const float* x, float* out, int64_t R, int64_t T, int32_t n_fft, int32_t hop,
                     int32_t n_mels, const float* window, const int32_t* fb_start,
                     const int32_t* fb_count, const float* fb_weight, int32_t fb_stride, int32_t fb_taps,
                     float eps, int32_t apply_log, int64_t x_row_stride, int64_t out_row_stride,
                     const int32_t* row_index, int32_t n_index, void* stream);

/*
 * SpecAugment of the training forward, models.py:201-205 (torchaudio FrequencyMasking / TimeMasking with
 * iid_masks=False: one band of mel bins [f0, f1) and one band of frames [t0, t1), the same for every row).
 * The reference zeroes the mel power before clip + log; on the fused log-mel output (R, n_mels, n_frames)
 * the masked cells are therefore set to log(eps) (is_log = 1) or to 0 (is_log = 0, mel power).  The two
 * random draws per mask stay with the caller (torch global CPU generator).
 */
int modfx_specaugment_fill_f32(float* out, int64_t R, int32_t n_mels, int32_t n_frames, int32_t f0, int32_t f1,
                               int32_t t0, int32_t t1, float eps, int32_t is_log, void* stream);

/*
 * Replaces PedalboardPhaserDataset.apply_pedalboard_phaser's DSP, mod_extraction/datasets.py:455-482
 * (pedalboard.Phaser -> juce::dsp::Phaser, 6 TPT all-pass stages + feedback, cutoff updated every
 * 4th sample).  PARITY UNPINNED: checked only against this repo's own CPU restatement.
 *   x, y (B, N); per-example (B,) device arrays; `block` = host block size of pedalboard (8192).
 *   workspace: device scratch of modfx_phaser_workspace_bytes(B, N) bytes.
 */
int64_t modfx_phaser_workspace_bytes(int32_t B, int64_t N);
int modfx_phaser_f32(const float* x, float* y, int32_t B, int64_t N, float sr, const float* rate_hz,
                     const float* depth, const float* centre_hz, const float* feedback,
                     const float* mix, int32_t block, const int32_t* example_index, int32_t n_items,
                     void* workspace, void* stream);

/*
 * The DSP of one batch of PedalboardPhaserDataset.__getitem__, mod_extraction/datasets.py:428-453: row b of x holds
 * proc_n = n_out + round(sr / rate_hz[b]) samples ("one extra LFO period", rows padded to the common pitch N); the
 * phaser runs over the row from its first sample and the window [start[b], start[b] + n_out) of the wet signal AND of
 * the dry input is delivered (datasets.py:445-447): y (B, n_out), dry_out (B, n_out) or NULL.  Samples past the window
 * are never processed (the effect is causal).
 * With an example_index list and x_compact = 1, x is a compact (n_items, N) array whose row i belongs to example
 * example_index[i] (every other array stays indexed by the example id): an interleaved batch keeps the long phaser
 * rows apart from its (B, n_out) dry / wet tensors, into which y / dry_out may point.
 */
int modfx_phaser_crop_f32(const float* x, int32_t x_compact, float* y, float* dry_out, int32_t B, int64_t N, int64_t n_out,
                          const int32_t* start, float sr, const float* rate_hz, const float* depth,
                          const float* centre_hz, const float* feedback, const float* mix, int32_t block,
                          const int32_t* example_index, int32_t n_items, void* workspace, void* stream);

/*
 * The same step over a PACKED ragged input, the layout a collate function produces from the variable-length chunks
 * PedalboardPhaserDataset reads (proc_n differs per example, mod_extraction/datasets.py:433-436): row i of x starts at
 * x + x_offset[i] (float index, device array of n_items) and holds at least start[b] + n_out samples, b =
 * example_index[i] -- the causal prefix that determines the delivered window; nothing past it is read.  N_max bounds
 * start[b] + n_out over the call and sizes the workspace (modfx_phaser_workspace_bytes(n_items, N_max)).  Rows whose
 * address is 16-byte aligned take the vector loads.
 */
int modfx_phaser_crop_packed_f32(const float* x, const int64_t* x_offset, float* y, float* dry_out, int32_t B, int64_t N_max,
                                 int64_t n_out, const int32_t* start, float sr, const float* rate_hz, const float* depth,
                                 const float* centre_hz, const float* feedback, const float* mix, int32_t block,
                                 const int32_t* example_index, int32_t n_items, void* workspace, void* stream);

/*
 * LFO-net body behind the log-mel front end (SURVEY section 8f, row N3): Spectral2DCNN.cnn, the mean over
 * mel bins, the 1x1 output convolution and the sigmoid, mod_extraction/models.py:183-195,209-214.
 * Activations between layers are channels-last float32: (B, H, W, C) with H = mel bins, W = frames.
 *
 *   modfx_cnn_layernorm_f32   replaces nn.LayerNorm([n_bins, n_frames], elementwise_affine=False),
 *                             models.py:186: y = (x - mean) / sqrt(var + eps) per (b, c) over H x W
 *                             (biased variance).  x is (B, C, H, W) when x_is_nchw (the log-mel tensor
 *                             the front end writes) else (B, H, W, C); y is always (B, H, W, C) and may
 *                             alias x when both are channels-last.  round_tf32 = 1 rounds y to TF32
 *                             (round-to-nearest), the operand format of the tensor-core convolution;
 *                             round_tf32 = 2 writes the error-compensated split instead: y holds TWO planes of
 *                             B*H*W*C floats, hi = tf32(v) and lo = tf32(v - hi) (channels-last input, y != x);
 *                             round_tf32 = 3 writes y as (B, H, W, C) IEEE float16 (round-to-nearest), the
 *                             operand format of modfx_cnn_conv_pool_prelu_f16_f32.
 *                             workspace: modfx_cnn_layernorm_workspace_bytes(B, C, H, W) bytes.
 *   modfx_cnn_conv_pool_prelu_f32
 *                             replaces Conv2d(Cin, Cout, (KH, KW), dilation=(1, dil_w), padding="same")
 *                             -> MaxPool2d((2, 1)) -> PReLU(Cout), models.py:187-190.
 *                             x (B, H, W, Cin) -> y (B, H/2, W, Cout).
 *                             weight (KH, KW, Cout, Cin) float32 (the reference's (Cout, Cin, KH, KW)
 *                             permuted), bias (Cout,), prelu (Cout,).
 *                             precision MODFX_CNN_FP32: float32 FMAs on the CUDA cores (any Cin that
 *                             is 2 or a multiple of 8); MODFX_CNN_TF32: tcgen05 tensor cores, TF32
 *                             operands / float32 accumulation (Cin == 64; what cuDNN does for the
 *                             reference on a GPU, torch.backends.cudnn.allow_tf32 defaults to True).
 *                             Built: KH = 5, KW = 13, Cout = 64, H even.
 *   modfx_cnn_conv_pool_prelu_tf32x3_f32
 *                             the same layer (Cin = Cout = 64) in error-compensated TF32 on the tensor cores:
 *                             operands split as hi + lo (modfx_cnn_layernorm_f32 with round_tf32 = 2 for the
 *                             activations; the caller splits the weights the same way), three MMA passes
 *                             hi*hi + hi*lo + lo*hi into one accumulator, a third of the TF32 rate.  The operand
 *                             rounding error is gone (the dropped lo*lo term is ~2^-22 relative); what remains is
 *                             the tensor pipe's truncating accumulator: 2e-4 per layer where plain TF32 has
 *                             1e-3, and float32-grade results through the whole network.
 *   modfx_cnn_conv_pool_prelu_f16_f32
 *                             the same layer (Cin = Cout = 64) with float16 operands (x (B, H, W, 64) and weight
 *                             (5, 13, 64, 64) as IEEE half) and float32 accumulation / output on the tensor cores.
 *                             float16 has TF32's 11 significant bits and normalised activations / weights sit
 *                             inside its range, so the parity bars are those of MODFX_CNN_TF32 -- at twice the
 *                             MMA rate and half the operand traffic.
 *   modfx_cnn_head_f32        replaces tr.mean(x, dim=-2), Conv1d(C, L, 1) and tr.sigmoid,
 *                             models.py:210-214: x (B, H, W, C) -> latent (B, C, W), out (B, L, W).
 *                             weight (L, C), bias (L,).
 *
 * Training (parameter gradients only, TF32, the shipped 5x13 / 64-channel shape).  Gradient semantics are those of
 * cuDNN TF32 training: operand rounding is a straight-through step, the max-pool routes to the upper row of a tied
 * pair, the layer-norm backward uses the unrounded normalised value.  Every reduction is a fixed-order sum of per-CTA
 * partials: results are bit-reproducible.  `workspace`: modfx_cnn_train_workspace_bytes(B, H, W, L) bytes, H = the
 * largest conv-input height of the call (the network's n_mels covers every layer).
 *   modfx_cnn_conv_pool_prelu_train_f32
 *                             forward of Conv2d -> MaxPool2d((2, 1)) -> PReLU (models.py:187-190) that also keeps what
 *                             its backward needs: y as modfx_cnn_conv_pool_prelu_f32 (MODFX_CNN_TF32, bit for bit),
 *                             z (B, H/2, W, 64) = maxpool(conv) + bias and argmax (B, H/2, W, 64) bytes, 1 where the
 *                             lower conv row of the pair won.  Cin = 64, or Cin = 2 with dil_w = 1.
 *   modfx_cnn_conv_dgrad_tf32_f32
 *                             input gradient of Conv2d(64, 64, (5, 13), dilation=(1, dil_w), padding="same"):
 *                             dconv (B, H, W, 64) -> dx (B, H, W, 64), the same tensor-core convolution with
 *                             weight_t[kh][kw][ci][co] = weight[4 - kh][12 - kw][co][ci] (TF32-rounded).
 *   modfx_cnn_conv_wgrad_tf32_f32
 *                             weight gradient of that Conv2d: x (B, H, W, Cin) (the TF32 conv input), dconv
 *                             (B, H, W, 64) -> dweight (64, Cin, 5, 13), the parameter's own layout.  Cin = 64 on
 *                             the tensor cores; Cin = 2 (dil_w = 1) on the CUDA cores.
 *   modfx_cnn_pool_prelu_bwd_f32
 *                             backward of MaxPool2d((2, 1)) -> PReLU: dy (B, H/2, W, 64), z, argmax, prelu ->
 *                             dconv (B, H, W, 64) rounded to TF32, dbias (64,) and dprelu (64,).
 *   modfx_cnn_layernorm_bwd_f32
 *                             input gradient of nn.LayerNorm(elementwise_affine=False) (models.py:186): g and x
 *                             (B, H, W, C) channels-last, stats = the workspace modfx_cnn_layernorm_f32 filled in the
 *                             forward of x (left untouched since) -> dx = rstd (g - mean(g) - xhat mean(g xhat)).
 *   modfx_cnn_head_bwd_f32    backward of tr.mean(x, dim=-2), Conv1d(C, L, 1) and tr.sigmoid (models.py:210-214):
 *                             latent (B, C, W), out (B, L, W), dout, dlatent -> dx (B, H, W, C), dweight (L, C),
 *                             dbias (L,).
 */
typedef enum {
    MODFX_CNN_FP32 = 0,
    MODFX_CNN_TF32 = 1
} modfx_cnn_precision;

int64_t modfx_cnn_layernorm_workspace_bytes(int32_t B, int32_t C, int32_t H, int32_t W);
int modfx_cnn_layernorm_f32(const float* x, float* y, int32_t B, int32_t C, int32_t H, int32_t W,
                            int32_t x_is_nchw, float eps, int32_t round_tf32, void* workspace, void* stream);
int modfx_cnn_conv_pool_prelu_f32(const float* x, float* y, int32_t B, int32_t H, int32_t W, int32_t Cin,
                                  int32_t Cout, int32_t KH, int32_t KW, int32_t dil_w,
                                  const float* weight, const float* bias, const float* prelu,
                                  int32_t precision, void* stream);
int modfx_cnn_conv_pool_prelu_tf32x3_f32(const float* x_hi, const float* x_lo, float* y, int32_t B, int32_t H,
                                         int32_t W, int32_t dil_w, const float* w_hi, const float* w_lo,
                                         const float* bias, const float* prelu, void* stream);
int modfx_cnn_conv_pool_prelu_f16_f32(const void* x_f16, float* y, int32_t B, int32_t H, int32_t W, int32_t dil_w,
                                      const void* w_f16, const float* bias, const float* prelu, void* stream);
int modfx_cnn_head_f32(const float* x, float* latent, float* out, int32_t B, int32_t H, int32_t W, int32_t C,
                       int32_t L, const float* weight, const float* bias, void* stream);

int64_t modfx_cnn_train_workspace_bytes(int32_t B, int32_t H, int32_t W, int32_t L);
int modfx_cnn_conv_pool_prelu_train_f32(const float* x, float* y, float* z, uint8_t* argmax, int32_t B, int32_t H,
                                        int32_t W, int32_t Cin, int32_t dil_w, const float* weight, const float* bias,
                                        const float* prelu, void* stream);
int modfx_cnn_conv_dgrad_tf32_f32(const float* dconv, float* dx, int32_t B, int32_t H, int32_t W, int32_t dil_w,
                                  const float* weight_t, void* stream);
int modfx_cnn_conv_wgrad_tf32_f32(const float* x, const float* dconv, float* dweight, int32_t B, int32_t H, int32_t W,
                                  int32_t Cin, int32_t dil_w, void* workspace, void* stream);
int modfx_cnn_pool_prelu_bwd_f32(const float* dy, const float* z, const uint8_t* argmax, const float* prelu, float* dconv,
                                 float* dbias, float* dprelu, int32_t B, int32_t H, int32_t W, void* workspace,
                                 void* stream);
int modfx_cnn_layernorm_bwd_f32(const float* g, const float* x, const void* stats, float* dx, int32_t B, int32_t C,
                                int32_t H, int32_t W, float eps, void* workspace, void* stream);
int modfx_cnn_head_bwd_f32(const float* latent, const float* out, const float* dout, const float* dlatent, float* dx,
                           float* dweight, float* dbias, int32_t B, int32_t H, int32_t W, int32_t C, int32_t L,
                           const float* weight, void* workspace, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MODFX_H_ */
