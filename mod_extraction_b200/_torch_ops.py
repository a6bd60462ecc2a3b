"""Registers the render ops with PyTorch as ``torch.ops.modfx.*`` -- CUDA dispatch key only.

There is deliberately no CPU (or any other backend) registration: calling an op with CPU tensors
fails in the dispatcher ("could not run 'modfx::...' with arguments from the 'CPU' backend"), which is the
"no CPU fallback" rule enforced at the framework level.  The implementations are the ctypes calls into
libmodfx.so of ``_ops.py``; registering them costs nothing when the ops are not used.

    torch.ops.modfx.flanger_chorus(x, mod_lo, feedback, min_delay_width, width, depth, mix, m_min, m_lfo)
    torch.ops.modfx.interp_linear(x, n, align_corners)
    torch.ops.modfx.lfo(freq, phase, shape, exp, n, sr)
    torch.ops.modfx.phaser(x, rate_hz, depth, centre_hz, feedback, mix, sr, block)
    torch.ops.modfx.tremolo(x, mod, mix)                                       # fx.py:13-22
    torch.ops.modfx.mel_power(x, window, fb_start, fb_count, fb_weight, fb_taps, hop, eps)     # the `spectrogram` attribute
    torch.ops.modfx.logmel(x, window, fb_start, fb_count, fb_weight, fb_taps, hop, eps)        # + clip + log, models.py:199-208
    torch.ops.modfx.find_corners(mod_sig) -> (top, bottom)                     # modulations.py:219-238
    torch.ops.modfx.lfo_sections(out, sec_off, sec_start, sec_len, sec_shape)  # make_combined_mod_sig's overwrite loop
    torch.ops.modfx.stretch_sections(x, sec_off, in_start, in_len, new_len, out_start)         # make_quasi_periodic
    torch.ops.modfx.combined_lfo(freq, phase, shapes, words, n, sr) -> (out, base, consumed)   # modulations.py:191-210
    torch.ops.modfx.smoothen(x, window)                                        # modulations.py:358-362
    torch.ops.modfx.stretch_corners(x, max_n_corners)                          # modulations.py:259-307
    torch.ops.modfx.check_mod_sig(x, min_top, max_top, min_bottom, max_bottom, min_frames)     # modulations.py:311-355
    torch.ops.modfx.cnn_layernorm(x, x_is_nchw, eps, round_tf32)               # -> channels-last (B, H, W, C)
    torch.ops.modfx.cnn_conv_pool_prelu(x, weight, bias, slope, dil_w, tf32)    # tcgen05 when tf32
    torch.ops.modfx.cnn_head(x, weight, bias)                                   # -> (output, latent)
    torch.ops.modfx.cnn_conv_pool_prelu_train(x, weight, bias, slope, dil_w)    # -> (y, z, argmax), TF32
    torch.ops.modfx.cnn_conv_dgrad(dconv, weight_t, dil_w)                      # TF32 training backward ...
    torch.ops.modfx.cnn_conv_wgrad(x, dconv, dil_w)
    torch.ops.modfx.cnn_pool_prelu_bwd(dy, z, argmax, slope)                    # -> (dconv, dbias, dslope)
    torch.ops.modfx.cnn_layernorm_bwd(g, x, eps)
    torch.ops.modfx.cnn_head_bwd(latent, out, dout, dlatent, weight, H)         # -> (dx, dweight, dbias)
"""
from __future__ import annotations

import torch
from torch import Tensor

from . import _ops
from ._ops import ModSource

_lib = torch.library.Library("modfx", "DEF")
_lib.define("flanger_chorus(Tensor x, Tensor mod, Tensor feedback, Tensor min_delay_width, Tensor width, "
            "Tensor depth, Tensor mix, int m_min, int m_lfo) -> Tensor")
_lib.define("interp_linear(Tensor x, int n, bool align_corners) -> Tensor")
_lib.define("lfo(Tensor freq, Tensor phase, Tensor shape, Tensor exp, int n, float sr) -> Tensor")
_lib.define("phaser(Tensor x, Tensor rate_hz, Tensor depth, Tensor centre_hz, Tensor feedback, Tensor mix, "
            "float sr, int block) -> Tensor")
_lib.define("tremolo(Tensor x, Tensor mod, Tensor mix) -> Tensor")
_lib.define("mel_power(Tensor x, Tensor window, Tensor fb_start, Tensor fb_count, Tensor fb_weight, int fb_taps, int hop, "
            "float eps) -> Tensor")
_lib.define("logmel(Tensor x, Tensor window, Tensor fb_start, Tensor fb_count, Tensor fb_weight, int fb_taps, int hop, "
            "float eps) -> Tensor")
_lib.define("find_corners(Tensor mod_sig) -> (Tensor, Tensor)")
_lib.define("lfo_sections(Tensor(a!) out, Tensor sec_off, Tensor sec_start, Tensor sec_len, Tensor sec_shape) -> Tensor(a!)")
_lib.define("stretch_sections(Tensor x, Tensor sec_off, Tensor in_start, Tensor in_len, Tensor new_len, Tensor out_start) -> Tensor")
_lib.define("combined_lfo(Tensor freq, Tensor phase, Tensor shapes, Tensor words, int n, float sr) -> (Tensor, Tensor, Tensor)")
_lib.define("smoothen(Tensor x, int window) -> Tensor")
_lib.define("stretch_corners(Tensor x, int max_n_corners) -> Tensor")
_lib.define("check_mod_sig(Tensor x, int min_top, int max_top, int min_bottom, int max_bottom, int min_frames) -> Tensor")
_lib.define("cnn_layernorm(Tensor x, bool x_is_nchw, float eps, bool round_tf32) -> Tensor")
_lib.define("cnn_conv_pool_prelu(Tensor x, Tensor weight, Tensor bias, Tensor slope, int dil_w, bool tf32) -> Tensor")
_lib.define("cnn_head(Tensor x, Tensor weight, Tensor bias) -> (Tensor, Tensor)")
_lib.define("cnn_conv_pool_prelu_train(Tensor x, Tensor weight, Tensor bias, Tensor slope, int dil_w) -> (Tensor, Tensor, Tensor)")
_lib.define("cnn_conv_dgrad(Tensor dconv, Tensor weight_t, int dil_w) -> Tensor")
_lib.define("cnn_conv_wgrad(Tensor x, Tensor dconv, int dil_w) -> Tensor")
_lib.define("cnn_pool_prelu_bwd(Tensor dy, Tensor z, Tensor argmax, Tensor slope) -> (Tensor, Tensor, Tensor)")
_lib.define("cnn_layernorm_bwd(Tensor g, Tensor x, float eps) -> Tensor")
_lib.define("cnn_head_bwd(Tensor latent, Tensor out, Tensor dout, Tensor dlatent, Tensor weight, int H) -> (Tensor, Tensor, Tensor)")


def _flanger_chorus(x: Tensor, mod: Tensor, feedback: Tensor, min_delay_width: Tensor, width: Tensor, depth: Tensor,
                    mix: Tensor, m_min: int, m_lfo: int) -> Tensor:
    src = ModSource.audio_rate(mod) if mod.size(-1) == x.size(-1) else ModSource.control_rate(mod)
    return _ops.flanger_chorus(x, src, m_min, m_lfo, feedback, min_delay_width, width, depth, mix)


def _interp_linear(x: Tensor, n: int, align_corners: bool) -> Tensor:
    return _ops.interp_linear(x, n, align_corners)


def _lfo(freq: Tensor, phase: Tensor, shape: Tensor, exp: Tensor, n: int, sr: float) -> Tensor:
    return _ops.lfo(n, sr, freq, phase, shape, exp)


def _phaser(x: Tensor, rate_hz: Tensor, depth: Tensor, centre_hz: Tensor, feedback: Tensor, mix: Tensor, sr: float,
            block: int) -> Tensor:
    return _ops.phaser(x, sr, rate_hz, depth, centre_hz, feedback, mix, block)


def _tremolo(x: Tensor, mod: Tensor, mix: Tensor) -> Tensor:
    src = ModSource.audio_rate(mod) if mod.size(-1) == x.size(-1) else ModSource.control_rate(mod)
    return _ops.tremolo(x, src, mix)


def _mel(apply_log: bool):
    def run(x: Tensor, window: Tensor, fb_start: Tensor, fb_count: Tensor, fb_weight: Tensor, fb_taps: int, hop: int,
            eps: float) -> Tensor:
        return _ops.logmel(x, window, fb_start, fb_count, fb_weight, fb_taps, hop, eps, apply_log)
    return run


def _sections_args(*ts: Tensor):
    return [t.to(torch.int32) for t in ts]


_impl = torch.library.Library("modfx", "IMPL", "CUDA")
_impl.impl("tremolo", _tremolo)
_impl.impl("mel_power", _mel(False))
_impl.impl("logmel", _mel(True))
_impl.impl("find_corners", lambda mod_sig: _ops.find_corners(mod_sig))
_impl.impl("lfo_sections", lambda out, a, b, c, d: _ops.lfo_sections_(out, *_sections_args(a, b, c, d)))
_impl.impl("stretch_sections", lambda x, a, b, c, d, e: _ops.stretch_sections(x, *_sections_args(a, b, c, d, e)))
_impl.impl("combined_lfo", lambda freq, phase, shapes, words, n, sr: _ops.combined_lfo(n, sr, freq, phase, shapes, words))
_impl.impl("smoothen", lambda x, window: _ops.smoothen(x, window))
_impl.impl("stretch_corners", lambda x, max_n_corners: _ops.stretch_corners(x, max_n_corners))
_impl.impl("check_mod_sig", lambda x, a, b, c, d, e: _ops.check_mod_sig(x, a, b, c, d, e))
_impl.impl("flanger_chorus", _flanger_chorus)
_impl.impl("interp_linear", _interp_linear)
_impl.impl("lfo", _lfo)
_impl.impl("phaser", _phaser)
_impl.impl("cnn_layernorm", lambda x, x_is_nchw, eps, round_tf32: _ops.cnn_layernorm(x, x_is_nchw, eps, round_tf32))
_impl.impl("cnn_conv_pool_prelu", lambda x, weight, bias, slope, dil_w, tf32: _ops.cnn_conv_pool_prelu(x, weight, bias, slope,
                                                                                                      dil_w, tf32))
_impl.impl("cnn_head", lambda x, weight, bias: _ops.cnn_head(x, weight, bias))
_impl.impl("cnn_conv_pool_prelu_train", lambda x, w, b, s, d: _ops.cnn_conv_pool_prelu_train(x, w, b, s, d))
_impl.impl("cnn_conv_dgrad", lambda dconv, weight_t, dil_w: _ops.cnn_conv_dgrad(dconv, weight_t, dil_w))
_impl.impl("cnn_conv_wgrad", lambda x, dconv, dil_w: _ops.cnn_conv_wgrad(x, dconv, dil_w))
_impl.impl("cnn_pool_prelu_bwd", lambda dy, z, am, slope: _ops.cnn_pool_prelu_bwd(dy, z, am, slope))
_impl.impl("cnn_layernorm_bwd", lambda g, x, eps: _ops.cnn_layernorm_bwd(g, x, eps))
_impl.impl("cnn_head_bwd", lambda latent, out, dout, dlatent, weight, H: _ops.cnn_head_bwd(latent, out, dout, dlatent, weight, H))
