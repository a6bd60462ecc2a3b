"""Log-mel front end and CNN body of the reference's LFO extractor (lfo_2dcnn), on the GPU.

Reference: ``Spectral2DCNN`` builds ``self.spectrogram = MelSpectrogram(sample_rate=int(sr), n_fft,
hop_length, normalized=False, n_mels, center=True)`` (models.py:170-175) and its ``forward`` does
``spectrogram(x)`` -> [SpecAugment when training] -> ``clip(min=eps)`` -> ``log`` (models.py:199-208).
``LogMelLoss`` (losses.py:105-130) uses the same front end.

``MelSpectrogram`` here is a drop-in for that ``spectrogram`` attribute (same constructor keywords,
returns mel *power*, (..., T) -> (..., n_mels, T // hop + 1)); ``LogMelSpectrogram`` fuses the clip
and log into the same kernel for inference, where no masking sits in between.

``Spectral2DCNN`` (SURVEY 8f, row N3) is the whole extractor with the reference's constructor, ``forward(x) ->
(sigmoid output, latent)`` and state-dict keys (models.py:127-215): log-mel kernel -> [SpecAugment fill when
training] -> 6 x {layer norm, 5x13 dilated conv + 2x1 max-pool + PReLU} -> mean over mel -> 1x1 conv -> sigmoid,
activations channels-last, the 64->64 convolutions on tcgen05 tensor cores (TF32, like cuDNN's default for the
reference on a GPU) or, with ``precision="fp32"``, on the CUDA cores.  With ``precision="tf32"`` the body and head are
trainable: parameter gradients (cuDNN TF32 training semantics) come from libmodfx's backward kernels.
"""
from __future__ import annotations

import ctypes
import math
from typing import Dict, List, Optional, Tuple

import numpy as np
import torch
from torch import Tensor, nn

from . import _lib

__all__ = ["MelSpectrogram", "LogMelSpectrogram", "Spectral2DCNN", "RandomLFO", "mel_filterbank", "banded"]


def _hz_to_mel(f: float) -> float:
    return 2595.0 * math.log10(1.0 + f / 700.0)


def mel_filterbank(sr: int, n_fft: int, n_mels: int, f_min: float = 0.0, f_max: Optional[float] = None) -> Tensor:
    """HTK triangular filterbank, norm=None: (n_fft//2+1, n_mels) float32.

    torchaudio builds this table in float32, where the triangle edges are ill-conditioned (one ulp
    of a band edge near 20 kHz moves a weight by ~3e-5, i.e. ~3e-4 in log-mel).  To be a bit-level
    drop-in we use torchaudio's own generator when it is importable and fall back to a float64
    evaluation (closer to the mathematical filterbank, up to ~3e-5 away from torchaudio's)."""
    f_max = float(sr // 2) if f_max is None else f_max
    n_freqs = n_fft // 2 + 1
    try:
        from torchaudio.functional import melscale_fbanks
        return melscale_fbanks(n_freqs, f_min, f_max, n_mels, sr, norm=None, mel_scale="htk").float()
    except Exception:       # torchaudio missing: mathematically exact table
        all_freqs = np.linspace(0.0, sr // 2, n_freqs)
        m_pts = np.linspace(_hz_to_mel(f_min), _hz_to_mel(f_max), n_mels + 2)
        f_pts = 700.0 * (10.0 ** (m_pts / 2595.0) - 1.0)
        f_diff = f_pts[1:] - f_pts[:-1]
        slopes = f_pts[None, :] - all_freqs[:, None]
        down = -slopes[:, :-2] / f_diff[:-1]
        up = slopes[:, 2:] / f_diff[1:]
        return torch.from_numpy(np.maximum(0.0, np.minimum(down, up)).astype(np.float32))


def banded(fb: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    """(n_freqs, n_mels) filterbank -> (start (n_mels,), count (n_mels,), weights (n_mels, stride)).
    The table is 0.77 % dense (<= 14 taps per band for the reference configuration)."""
    fbn = fb.detach().cpu().numpy()
    n_freqs, n_mels = fbn.shape
    start = np.zeros(n_mels, dtype=np.int32)
    count = np.zeros(n_mels, dtype=np.int32)
    for m in range(n_mels):
        nz = np.nonzero(fbn[:, m])[0]
        if nz.size:
            start[m] = nz[0]
            count[m] = nz[-1] - nz[0] + 1
    stride = max(4, int(-(-int(count.max()) // 4) * 4))
    w = np.zeros((n_mels, stride), dtype=np.float32)
    for m in range(n_mels):
        w[m, :count[m]] = fbn[start[m]:start[m] + count[m], m]
    return torch.from_numpy(start), torch.from_numpy(count), torch.from_numpy(w)


class MelSpectrogram(nn.Module):
    """GPU replacement for the ``spectrogram`` attribute of Spectral2DCNN / LogMelLoss."""

    apply_log = False

    def __init__(self, sample_rate: int = 44100, n_fft: int = 1024, hop_length: int = 256, n_mels: int = 256,
                 normalized: bool = False, center: bool = True, eps: float = 1e-7,
                 fb: Optional[Tensor] = None, window: Optional[Tensor] = None) -> None:
        super().__init__()
        assert not normalized and center, "only the reference configuration (normalized=False, center=True)"
        self.sample_rate, self.n_fft, self.hop_length, self.n_mels, self.eps = sample_rate, n_fft, hop_length, n_mels, eps
        fb = mel_filterbank(sample_rate, n_fft, n_mels) if fb is None else fb.detach().float().cpu()
        assert fb.shape == (n_fft // 2 + 1, n_mels)
        window = torch.hann_window(n_fft, periodic=True) if window is None else window.detach().float().cpu()
        start, count, weight = banded(fb)
        self.fb_taps = max(1, int(count.sum()))
        self.register_buffer("fb", fb, persistent=False)
        self.register_buffer("window", window, persistent=False)
        self.register_buffer("fb_start", start, persistent=False)
        self.register_buffer("fb_count", count, persistent=False)
        self.register_buffer("fb_weight", weight, persistent=False)

    @classmethod
    def from_torchaudio(cls, mel, eps: float = 1e-7):
        """Build from an existing torchaudio.transforms.MelSpectrogram (e.g. ``net.spectrogram``):
        reuses its very filterbank and window buffers."""
        return cls(sample_rate=mel.sample_rate, n_fft=mel.n_fft, hop_length=mel.hop_length, n_mels=mel.n_mels,
                   eps=eps, fb=mel.mel_scale.fb, window=mel.spectrogram.window)

    def n_frames(self, n_samples: int) -> int:
        return n_samples // self.hop_length + 1

    @torch.no_grad()
    def forward_rows(self, x: Tensor, T: int, n_rows: int, out: Tensor, x_row_stride: int, out_row_stride: int,
                     row_index: Optional[Tensor] = None) -> None:
        """Strided / indexed variant used by the batch renderer: row r of the input starts at
        ``x.data_ptr() + 4*r*x_row_stride`` and its (n_mels, n_frames) result is written at
        ``out.data_ptr() + 4*r*out_row_stride``; ``row_index`` (int32, CUDA) selects rows."""
        if self.fb_weight.device != x.device:
            self.to(x.device)
        vp = lambda t: ctypes.c_void_p(0 if t is None else t.data_ptr())
        with torch.cuda.device(x.device):
            _lib.check(_lib.lib().modfx_logmel_f32(
                vp(x), vp(out), n_rows, T, self.n_fft, self.hop_length, self.n_mels, vp(self.window), vp(self.fb_start),
                vp(self.fb_count), vp(self.fb_weight), self.fb_weight.size(1), self.fb_taps, float(self.eps),
                1 if self.apply_log else 0, x_row_stride, out_row_stride, vp(row_index),
                0 if row_index is None else row_index.numel(),
                ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))

    @torch.no_grad()
    def forward(self, x: Tensor, out: Optional[Tensor] = None) -> Tensor:
        if not x.is_cuda:
            raise RuntimeError("modfx: the log-mel front end needs a CUDA tensor (no CPU kernel)")
        if self.fb_weight.device != x.device:
            self.to(x.device)
        x = x.detach().float().contiguous()
        T = x.size(-1)
        lead = x.shape[:-1]
        R = x.numel() // T
        nf = self.n_frames(T)
        if out is None:
            out = torch.empty(lead + (self.n_mels, nf), device=x.device, dtype=torch.float32)
        assert out.is_contiguous() and out.numel() == R * self.n_mels * nf
        if R == 0:                      # empty batch: nothing to launch (and no device pointer to pass)
            return out
        vp = lambda t: ctypes.c_void_p(t.data_ptr())
        with torch.cuda.device(x.device):
            _lib.check(_lib.lib().modfx_logmel_f32(
                vp(x), vp(out), R, T, self.n_fft, self.hop_length, self.n_mels, vp(self.window), vp(self.fb_start),
                vp(self.fb_count), vp(self.fb_weight), self.fb_weight.size(1), self.fb_taps, float(self.eps),
                1 if self.apply_log else 0, 0, 0, None, 0,
                ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
        return out


class LogMelSpectrogram(MelSpectrogram):
    """``log(clip(MelSpectrogram(x), min=eps))`` in one kernel (models.py:199,207-208)."""

    apply_log = True


def _vp(t: Optional[Tensor]) -> ctypes.c_void_p:
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


def _stream() -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def round_to_tf32(w: Tensor) -> Tensor:
    """Round float32 to the nearest TF32 value (10-bit mantissa, ties away from zero like cvt.rna.tf32.f32):
    the tensor cores ignore the low 13 mantissa bits of their operands, i.e. they would truncate."""
    bits = w.contiguous().view(torch.int32)
    return ((bits + 0x1000) & ~0x1FFF).view(torch.float32)


def specaugment_bounds(size: int, mask_param: int) -> Tuple[int, int]:
    """The two draws of torchaudio.functional.mask_along_axis (torch global CPU generator, this order):
    ``value = rand(1) * mask_param; min_value = rand(1) * (size - value)`` -> [start, end)."""
    if mask_param < 1:
        return 0, 0
    value = torch.rand(1) * mask_param
    min_value = torch.rand(1) * (size - value)
    start = int(min_value.long())
    end = start + int(value.long())
    return start, end


class Spectral2DCNN(nn.Module):
    """GPU drop-in for ``mod_extraction.models.Spectral2DCNN`` (models.py:127-215).

    Same constructor arguments, same ``forward(x) -> (x, latent)`` with x (B, in_ch, n_samples) ->
    (B, latent_dim, n_frames) and latent (B, out_channels[-1], n_frames), and the same parameter names, so
    ``load_state_dict`` takes a reference checkpoint unchanged (the torch sub-modules below only hold the
    parameters; the arithmetic runs in libmodfx).  ``precision``: "tf32" (tcgen05, default), "fp16" (tcgen05 with
    float16 operand storage for the 64-channel layers: TF32's 11 significant bits at twice the rate), "tf32x3" (tcgen05 with
    error-compensated operands: meets the float32 parity bars of the network at a third of the TF32 rate, 6x faster than
    the CUDA-core path) or "fp32" (CUDA cores, exact float32 FMAs).
    Built: kernel_size (5, 13), pool_size (2, 1), 64 channels per layer, bin dilation 1, use_ln=True.

    Training: in train mode, with grad enabled and a parameter that requires grad, ``forward`` / ``forward_features``
    return outputs attached to the autograd graph (bitwise the no-grad numbers) and ``backward`` fills ``.grad`` of
    every parameter -- ``precision="tf32"`` only: the other precisions run their forward-only path, whose outputs carry
    no graph.  No gradient flows to the log-mel or the audio (an input that requires grad raises NotImplementedError).
    """

    def __init__(self, in_ch: int = 1, n_samples: int = 88200, sr: float = 44100, n_fft: int = 1024,
                 hop_len: int = 256, n_mels: int = 256, kernel_size: Tuple[int, int] = (5, 13),
                 out_channels: Optional[List[int]] = None, bin_dilations: Optional[List[int]] = None,
                 temp_dilations: Optional[List[int]] = None, pool_size: Tuple[int, int] = (3, 1),
                 latent_dim: int = 1, freq_mask_amount: float = 0.0, time_mask_amount: float = 0.0,
                 use_ln: bool = True, eps: float = 1e-7, precision: str = "tf32", max_chunk: int = 256) -> None:
        super().__init__()
        assert pool_size[1] == 1
        if out_channels is None:
            out_channels = [64] * 5
        if bin_dilations is None:
            bin_dilations = [1] * len(out_channels)
        if temp_dilations is None:
            temp_dilations = [2 ** idx for idx in range(len(out_channels))]
        assert len(out_channels) == len(bin_dilations) == len(temp_dilations)
        if tuple(kernel_size) != (5, 13) or tuple(pool_size) != (2, 1) or any(c != 64 for c in out_channels) \
                or any(d != 1 for d in bin_dilations) or not use_ln or in_ch != 2:
            raise NotImplementedError(
                "modfx builds the shipped lfo_2dcnn (configs/models/spectral_2dcnn.yml): in_ch 2, kernel (5, 13), "
                "pool (2, 1), 64 channels per layer, bin dilation 1, use_ln")
        assert n_mels % (2 ** len(out_channels)) == 0, "n_mels must survive the 2x1 pools"
        assert precision in ("fp16", "tf32", "tf32x3", "fp32")
        self.in_ch, self.n_samples, self.sr, self.n_fft, self.hop_len, self.n_mels = in_ch, n_samples, sr, n_fft, hop_len, n_mels
        self.kernel_size, self.pool_size, self.latent_dim = tuple(kernel_size), tuple(pool_size), latent_dim
        self.freq_mask_amount, self.time_mask_amount, self.use_ln, self.eps = freq_mask_amount, time_mask_amount, use_ln, eps
        self.out_channels, self.bin_dilations, self.temp_dilations = list(out_channels), list(bin_dilations), list(temp_dilations)
        self.precision = precision
        self.max_chunk = max_chunk                # examples per pass: the first layer's output is 11.3 MB per example
        self.ln_eps = 1e-5                        # nn.LayerNorm default (models.py:186)

        self.spectrogram = LogMelSpectrogram(sample_rate=int(sr), n_fft=n_fft, hop_length=hop_len, n_mels=n_mels, eps=eps)
        n_frames = n_samples // hop_len + 1
        self.freq_mask_param = int(freq_mask_amount * n_mels)          # models.py:180
        self.time_mask_param = int(time_mask_amount * n_frames)        # models.py:181
        # parameter containers with the reference's module indices (LayerNorm, Conv2d, MaxPool2d, PReLU per layer)
        layers: List[nn.Module] = []
        n_bins, c_in = n_mels, in_ch
        for out_ch, t_dil in zip(out_channels, temp_dilations):
            layers.append(nn.LayerNorm([n_bins, n_frames], elementwise_affine=False))
            layers.append(nn.Conv2d(c_in, out_ch, kernel_size, stride=(1, 1), dilation=(1, t_dil), padding="same"))
            layers.append(nn.MaxPool2d(kernel_size=pool_size))
            layers.append(nn.PReLU(num_parameters=out_ch))
            c_in = out_ch
            n_bins //= pool_size[0]
        self.cnn = nn.Sequential(*layers)
        self.output = nn.Conv1d(out_channels[-1], latent_dim, kernel_size=(1,))
        self._packed = None
        self._packed_key = None

    def load_state_dict(self, state_dict, strict: bool = True, **kw):
        """Accepts a reference checkpoint as is: its ``spectrogram.*`` buffers (torchaudio's window and mel table,
        models.py:170-175) are not parameters here -- they rebuild the front end instead."""
        sd = dict(state_dict)
        fb = sd.pop("spectrogram.mel_scale.fb", None)
        window = sd.pop("spectrogram.spectrogram.window", None)
        if fb is not None or window is not None:
            self.spectrogram = LogMelSpectrogram(sample_rate=int(self.sr), n_fft=self.n_fft, hop_length=self.hop_len,
                                                 n_mels=self.n_mels, eps=self.eps, fb=fb, window=window)
        return super().load_state_dict(sd, strict=strict, **kw)

    # ---- weights in the layout the kernels read: (KH, KW, Cout, Cin), TF32-rounded for the tensor-core layers
    def _pack(self, device) -> list:
        params = list(self.parameters())
        key = (str(device), self.precision) + tuple((p.data_ptr(), p._version) for p in params)
        if self._packed is None or self._packed_key != key:
            packed = []
            for i in range(len(self.out_channels)):
                conv, act = self.cnn[4 * i + 1], self.cnn[4 * i + 3]
                w = conv.weight.detach().to(device=device, dtype=torch.float32).permute(2, 3, 0, 1).contiguous()
                # tensor-core layers: 64 input channels, or the 2-channel first layer when it is not dilated
                tc = self.precision in ("tf32", "fp16") and (w.size(3) == 64 or (w.size(3) == 2 and self.temp_dilations[i] == 1))
                x3 = self.precision == "tf32x3" and w.size(3) == 64
                mode = _lib.CNN_TF32 if tc else (_lib.CNN_TF32X3 if x3 else _lib.CNN_FP32)
                if self.precision == "fp16" and w.size(3) == 64:
                    mode, tc = _lib.CNN_FP16, False
                    w = w.to(torch.float16)            # round-to-nearest: the 11 significant bits TF32 keeps
                if tc:
                    w = round_to_tf32(w)
                elif x3:                                   # w = hi + lo, both exactly representable in TF32
                    hi = round_to_tf32(w)
                    w = torch.stack([hi, round_to_tf32(w - hi)])
                packed.append((w, conv.bias.detach().to(device=device, dtype=torch.float32).contiguous(),
                               act.weight.detach().to(device=device, dtype=torch.float32).contiguous(), mode))
            # data-gradient weights of the tensor-core layers: w_t[kh][kw][ci][co] = w[4 - kh][12 - kw][co][ci]
            self._packed_t = [w.flip(0, 1).transpose(2, 3).contiguous() if mode == _lib.CNN_TF32 and w.size(3) == 64 else None
                              for (w, _, _, mode) in packed]
            w_out = self.output.weight.detach().to(device=device, dtype=torch.float32).reshape(self.latent_dim, -1).contiguous()
            b_out = self.output.bias.detach().to(device=device, dtype=torch.float32).contiguous()
            self._packed, self._packed_key = (packed, w_out, b_out), key
        return self._packed

    def _builds_graph(self, x: Tensor) -> bool:
        # the backward pass is TF32; other precisions keep their forward-only path, whose outputs carry no graph
        if not (torch.is_grad_enabled() and self.training and self.precision == "tf32"
                and any(p.requires_grad for p in self.parameters())):
            return False
        if x.requires_grad:
            raise NotImplementedError("modfx: Spectral2DCNN has no gradient to its input (log-mel / audio)")
        return True

    def forward_features(self, logmel: Tensor) -> Tuple[Tensor, Tensor]:
        """(B, in_ch, n_mels, n_frames) log-mel (clip + log already applied) -> (output, latent)."""
        if self._builds_graph(logmel):
            if not logmel.is_cuda:
                raise RuntimeError("modfx: Spectral2DCNN needs CUDA tensors (no CPU kernel)")
            outs = [_BodyFunction.apply(self, logmel[i:i + self.max_chunk], *self._grad_params())
                    for i in range(0, logmel.size(0), self.max_chunk)]
            if len(outs) == 1:
                return outs[0]
            return torch.cat([o[0] for o in outs], 0), torch.cat([o[1] for o in outs], 0)
        return self._forward_features(logmel)

    def _grad_params(self) -> List[Tensor]:
        ps = []
        for i in range(len(self.out_channels)):
            ps += [self.cnn[4 * i + 1].weight, self.cnn[4 * i + 1].bias, self.cnn[4 * i + 3].weight]
        return ps + [self.output.weight, self.output.bias]

    @torch.no_grad()
    def _forward_features(self, logmel: Tensor) -> Tuple[Tensor, Tensor]:
        if not logmel.is_cuda:
            raise RuntimeError("modfx: Spectral2DCNN needs CUDA tensors (no CPU kernel)")
        L = _lib.lib()
        dev = logmel.device
        logmel = logmel.detach().float().contiguous()
        B, C, H, W = logmel.shape
        assert C == self.in_ch and H == self.n_mels
        if B == 0:
            return (torch.empty((0, self.latent_dim, W), dtype=torch.float32, device=dev),
                    torch.empty((0, self.out_channels[-1], W), dtype=torch.float32, device=dev))
        if B > self.max_chunk:                    # examples are independent: bound the activation memory
            outs = [self._forward_features(logmel[i:i + self.max_chunk]) for i in range(0, B, self.max_chunk)]
            return torch.cat([o[0] for o in outs], 0), torch.cat([o[1] for o in outs], 0)
        packed, w_out, b_out = self._pack(dev)
        with torch.cuda.device(dev):
            ws_bytes = max(L.modfx_cnn_layernorm_workspace_bytes(B, C, H, W), L.modfx_cnn_layernorm_workspace_bytes(B, 64, H // 2, W))
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            x = torch.empty((B, H, W, C), dtype=torch.float32, device=dev)
            _lib.check(L.modfx_cnn_layernorm_f32(_vp(logmel), _vp(x), B, C, H, W, 1, self.ln_eps,
                                                 1 if packed[0][3] == _lib.CNN_TF32 else 0, _vp(ws), _stream()))
            for i, (w, bias, slope, prec) in enumerate(packed):
                y = torch.empty((B, H // 2, W, 64), dtype=torch.float32, device=dev)
                if prec == _lib.CNN_FP16:                  # x and w are float16
                    _lib.check(L.modfx_cnn_conv_pool_prelu_f16_f32(_vp(x), _vp(y), B, H, W, self.temp_dilations[i], _vp(w),
                                                                  _vp(bias), _vp(slope), _stream()))
                elif prec == _lib.CNN_TF32X3:              # x holds the hi and lo planes, w likewise
                    _lib.check(L.modfx_cnn_conv_pool_prelu_tf32x3_f32(_vp(x[0]), _vp(x[1]), _vp(y), B, H, W, self.temp_dilations[i],
                                                                     _vp(w[0]), _vp(w[1]), _vp(bias), _vp(slope), _stream()))
                else:
                    _lib.check(L.modfx_cnn_conv_pool_prelu_f32(_vp(x), _vp(y), B, H, W, C, 64, 5, 13, self.temp_dilations[i],
                                                              _vp(w), _vp(bias), _vp(slope), prec, _stream()))
                H, C, x = H // 2, 64, y
                if i + 1 < len(packed):
                    nxt = packed[i + 1][3]
                    if nxt == _lib.CNN_FP16:               # normalise into float16
                        x = torch.empty((B, H, W, C), dtype=torch.float16, device=dev)
                        _lib.check(L.modfx_cnn_layernorm_f32(_vp(y), _vp(x), B, C, H, W, 0, self.ln_eps, 3, _vp(ws), _stream()))
                    elif nxt == _lib.CNN_TF32X3:           # normalise into the two-plane hi / lo split
                        x = torch.empty((2, B, H, W, C), dtype=torch.float32, device=dev)
                        _lib.check(L.modfx_cnn_layernorm_f32(_vp(y), _vp(x), B, C, H, W, 0, self.ln_eps, 2, _vp(ws), _stream()))
                    else:
                        _lib.check(L.modfx_cnn_layernorm_f32(_vp(x), _vp(x), B, C, H, W, 0, self.ln_eps,
                                                            1 if nxt == _lib.CNN_TF32 else 0, _vp(ws), _stream()))
            latent = torch.empty((B, C, W), dtype=torch.float32, device=dev)
            out = torch.empty((B, self.latent_dim, W), dtype=torch.float32, device=dev)
            _lib.check(L.modfx_cnn_head_f32(_vp(x), _vp(latent), _vp(out), B, H, W, C, self.latent_dim, _vp(w_out), _vp(b_out),
                                           _stream()))
        return out, latent

    @torch.no_grad()
    def _train_forward(self, logmel: Tensor):
        """The TF32 forward of one chunk that keeps what the backward needs: per layer the layer-norm input and its
        statistics, the conv input, z = maxpool(conv) + bias and the pool's argmax."""
        L = _lib.lib()
        dev = logmel.device
        logmel = logmel.detach().float().contiguous()
        B, C, H, W = logmel.shape
        assert C == self.in_ch and H == self.n_mels
        packed, w_out, b_out = self._pack(dev)
        saves = []
        with torch.cuda.device(dev):
            ws = torch.empty(L.modfx_cnn_layernorm_workspace_bytes(B, C, H, W), dtype=torch.uint8, device=dev)
            x = torch.empty((B, H, W, C), dtype=torch.float32, device=dev)
            _lib.check(L.modfx_cnn_layernorm_f32(_vp(logmel), _vp(x), B, C, H, W, 1, self.ln_eps, 1, _vp(ws), _stream()))
            ln_in = stats = None
            for i, (w, bias, slope, prec) in enumerate(packed):
                y = torch.empty((B, H // 2, W, 64), dtype=torch.float32, device=dev)
                z = torch.empty_like(y)
                am = torch.empty((B, H // 2, W, 64), dtype=torch.uint8, device=dev)
                _lib.check(L.modfx_cnn_conv_pool_prelu_train_f32(_vp(x), _vp(y), _vp(z), _vp(am), B, H, W, C,
                                                                 self.temp_dilations[i], _vp(w), _vp(bias), _vp(slope),
                                                                 _stream()))
                saves.append((ln_in, stats, x, z, am))
                H, C = H // 2, 64
                if i + 1 < len(packed):
                    ln_in = y
                    stats = torch.empty(L.modfx_cnn_layernorm_workspace_bytes(B, C, H, W), dtype=torch.uint8, device=dev)
                    x = torch.empty_like(y)
                    _lib.check(L.modfx_cnn_layernorm_f32(_vp(y), _vp(x), B, C, H, W, 0, self.ln_eps, 1, _vp(stats),
                                                        _stream()))
            latent = torch.empty((B, C, W), dtype=torch.float32, device=dev)
            out = torch.empty((B, self.latent_dim, W), dtype=torch.float32, device=dev)
            _lib.check(L.modfx_cnn_head_f32(_vp(y), _vp(latent), _vp(out), B, H, W, C, self.latent_dim, _vp(w_out), _vp(b_out),
                                           _stream()))
        return out, latent, saves

    @torch.no_grad()
    def _backward(self, saves, out: Tensor, latent: Tensor, dout: Tensor, dlatent: Tensor) -> List[Tensor]:
        """Parameter gradients of one chunk, in the order of ``_grad_params``."""
        L = _lib.lib()
        dev = out.device
        packed, w_out, _ = self._pack(dev)
        B, C, W = latent.shape
        n = len(packed)
        H = self.n_mels >> n
        grads: List[Optional[Tensor]] = [None] * (3 * n + 2)
        with torch.cuda.device(dev):
            ws = torch.empty(L.modfx_cnn_train_workspace_bytes(B, self.n_mels, W, self.latent_dim), dtype=torch.uint8,
                             device=dev)
            dy = torch.empty((B, H, W, C), dtype=torch.float32, device=dev)
            dw_out = torch.empty((self.latent_dim, C), dtype=torch.float32, device=dev)
            db_out = torch.empty((self.latent_dim,), dtype=torch.float32, device=dev)
            _lib.check(L.modfx_cnn_head_bwd_f32(_vp(latent), _vp(out), _vp(dout), _vp(dlatent), _vp(dy), _vp(dw_out),
                                               _vp(db_out), B, H, W, C, self.latent_dim, _vp(w_out), _vp(ws), _stream()))
            grads[3 * n] = dw_out.view_as(self.output.weight)
            grads[3 * n + 1] = db_out
            for i in range(n - 1, -1, -1):
                ln_in, stats, x, z, am = saves[i]
                slope = packed[i][2]
                H *= 2
                cin = x.size(3)
                dconv = torch.empty((B, H, W, 64), dtype=torch.float32, device=dev)
                dbias = torch.empty(64, dtype=torch.float32, device=dev)
                dslope = torch.empty(64, dtype=torch.float32, device=dev)
                _lib.check(L.modfx_cnn_pool_prelu_bwd_f32(_vp(dy), _vp(z), _vp(am), _vp(slope), _vp(dconv), _vp(dbias),
                                                         _vp(dslope), B, H, W, _vp(ws), _stream()))
                dw = torch.empty((64, cin, 5, 13), dtype=torch.float32, device=dev)
                _lib.check(L.modfx_cnn_conv_wgrad_tf32_f32(_vp(x), _vp(dconv), _vp(dw), B, H, W, cin, self.temp_dilations[i],
                                                          _vp(ws), _stream()))
                grads[3 * i:3 * i + 3] = [dw, dbias, dslope]
                if i > 0:
                    g = torch.empty((B, H, W, 64), dtype=torch.float32, device=dev)
                    _lib.check(L.modfx_cnn_conv_dgrad_tf32_f32(_vp(dconv), _vp(g), B, H, W, self.temp_dilations[i],
                                                              _vp(self._packed_t[i]), _stream()))
                    dy = torch.empty_like(ln_in)
                    _lib.check(L.modfx_cnn_layernorm_bwd_f32(_vp(g), _vp(ln_in), _vp(stats), _vp(dy), B, 64, H, W,
                                                            self.ln_eps, _vp(ws), _stream()))
        return grads

    def forward(self, x: Tensor) -> Tuple[Tensor, Tensor]:
        assert x.ndim == 3
        if x.requires_grad and self._builds_graph(x):
            raise NotImplementedError("modfx: Spectral2DCNN has no gradient to its input (log-mel / audio)")
        logmel = self.spectrogram(x)                               # models.py:199,207-208 fused
        if self.training:                                          # models.py:201-205
            f0 = f1 = t0 = t1 = 0
            if self.freq_mask_amount > 0:
                f0, f1 = specaugment_bounds(logmel.size(-2), self.freq_mask_param)
            if self.time_mask_amount > 0:
                t0, t1 = specaugment_bounds(logmel.size(-1), self.time_mask_param)
            with torch.cuda.device(logmel.device):
                _lib.check(_lib.lib().modfx_specaugment_fill_f32(
                    _vp(logmel), logmel.size(0) * logmel.size(1), logmel.size(-2), logmel.size(-1), f0, f1, t0, t1,
                    float(self.eps), 1, _stream()))
        return self.forward_features(logmel)


class _BodyFunction(torch.autograd.Function):
    """Body + head of Spectral2DCNN for one chunk of examples: the forward keeps its saves, the backward returns the
    parameter gradients (none to the log-mel, which is data)."""

    @staticmethod
    def forward(ctx, net: "Spectral2DCNN", logmel: Tensor, *params: Tensor):
        out, latent, saves = net._train_forward(logmel)
        ctx.net, ctx.saves = net, saves
        ctx.save_for_backward(out, latent)
        return out, latent

    @staticmethod
    def backward(ctx, dout: Tensor, dlatent: Tensor):
        out, latent = ctx.saved_tensors
        grads = ctx.net._backward(ctx.saves, out, latent, dout.float().contiguous(), dlatent.float().contiguous())
        ctx.saves = None
        return (None, None) + tuple(grads)


class RandomLFO(nn.Module):
    """Drop-in for ``mod_extraction.models.RandomLFO`` (models.py:19-69, configs/models/baseline_rand_lfo.yml): the
    random-LFO baseline "model".  Same constructor and ``forward(batch_size, fx_params) -> (B, 1, n_samples)``; the
    draws come from the torch global CPU generator in the reference's order (phase, frequency, shape per example),
    the batch of LFOs is one launch (``modulations.make_rand_mod_signal``)."""

    def __init__(self, n_samples: int, sr: float, use_shape_gt: bool = False, use_phase_gt: bool = False,
                 use_freq_gt: bool = False, shapes: Optional[List[str]] = None, freq_min: float = 0.5,
                 freq_max: float = 3.0, phase_error: float = 0.0, freq_error: float = 0.0) -> None:
        super().__init__()
        self.n_samples, self.sr = n_samples, sr
        self.use_shape_gt, self.use_phase_gt, self.use_freq_gt = use_shape_gt, use_phase_gt, use_freq_gt
        self.shapes, self.freq_min, self.freq_max = shapes, freq_min, freq_max
        self.phase_error, self.freq_error = phase_error, freq_error

    def forward(self, batch_size: int, fx_params: Optional[Dict[str, Tensor]] = None) -> Tensor:
        from .modulations import make_rand_mod_signal
        shapes_gt = phase_gt = freq_gt = None
        if self.use_shape_gt:
            assert fx_params is not None and "shape" in fx_params          # models.py:49
            shapes_gt = fx_params["shape"]
        if self.use_phase_gt:
            assert fx_params is not None and "phase" in fx_params          # models.py:52
            phase_gt = fx_params["phase"]
        if self.use_freq_gt:
            assert fx_params is not None and "rate_hz" in fx_params        # models.py:55
            freq_gt = fx_params["rate_hz"]
        return make_rand_mod_signal(batch_size, self.n_samples, self.sr, self.freq_min, self.freq_max, shapes_gt,
                                    self.shapes, phase_gt, self.phase_error, freq_gt, self.freq_error).unsqueeze(1)
