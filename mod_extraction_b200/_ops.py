"""Thin tensor-level wrappers over the libmodfx C ABI (one function per entry point).

These take CUDA float32 tensors, launch on the current torch stream and return new tensors;
they are what ``torch.ops.modfx.*`` dispatches to (CUDA key only -- see ``_torch_ops.py``) and what
the reference-signature shims in ``fx.py`` / ``modulations.py`` / ``util.py`` / ``models.py`` call.
"""
from __future__ import annotations

import ctypes
from typing import Optional, Sequence, Union

import torch
from torch import Tensor

from . import _lib
from ._lib import ModfxModSource, ModfxParam

Param = Union[float, Tensor]


def _require_cuda(t: Tensor, name: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(f"modfx: `{name}` must be a CUDA tensor (got {t.device}); there is no CPU kernel")
    if t.dtype != torch.float32:
        raise RuntimeError(f"modfx: `{name}` must be float32 (got {t.dtype})")


def _stream() -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t: Optional[Tensor]) -> ctypes.c_void_p:
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


class _Keep:
    """Holds temporaries alive until the call has been enqueued."""

    def __init__(self):
        self.items = []

    def __call__(self, t):
        self.items.append(t)
        return t


def as_param(p: Param, B: int, device, keep: _Keep, name: str) -> ModfxParam:
    """float -> python-scalar semantics; (B,) tensor -> float32 device array (fx.py:46-70)."""
    if isinstance(p, Tensor):
        if p.shape != (B,):
            raise AssertionError(f"{name}: expected shape ({B},), got {tuple(p.shape)}")
        t = keep(p.detach().to(device=device, dtype=torch.float32, non_blocking=True).contiguous())
        return ModfxParam(t.data_ptr(), 0.0)
    return ModfxParam(None, float(p))


class ModSource:
    """Python-side description of where the modulation signal comes from (modfx_mod_source)."""

    def __init__(self, kind: int, mod: Optional[Tensor] = None, n_lo: int = 0, sr_lo: float = 0.0,
                 freq: Optional[Tensor] = None, phase: Optional[Tensor] = None, shape: Optional[Tensor] = None,
                 exp: Optional[Tensor] = None):
        self.kind, self.mod, self.n_lo, self.sr_lo = kind, mod, n_lo, sr_lo
        self.freq, self.phase, self.shape, self.exp = freq, phase, shape, exp

    @staticmethod
    def audio_rate(mod_sig: Tensor) -> "ModSource":
        return ModSource(_lib.MOD_AUDIO_RATE, mod=mod_sig)

    @staticmethod
    def control_rate(mod_lo: Tensor) -> "ModSource":
        return ModSource(_lib.MOD_CONTROL_RATE, mod=mod_lo, n_lo=mod_lo.size(-1))

    @staticmethod
    def lfo(n_lo: int, sr_lo: float, freq: Tensor, phase: Tensor, shape: Tensor, exp: Optional[Tensor] = None):
        return ModSource(_lib.MOD_LFO, n_lo=n_lo, sr_lo=sr_lo, freq=freq, phase=phase, shape=shape, exp=exp)

    def to_c(self, B: int, C: int, N: int, device, keep: _Keep) -> ModfxModSource:
        s = ModfxModSource()
        s.kind = self.kind
        if self.kind in (_lib.MOD_AUDIO_RATE, _lib.MOD_CONTROL_RATE):
            m = self.mod
            _require_cuda(m, "mod_sig")
            m = keep(m.contiguous())
            has_ch = 0
            if self.kind == _lib.MOD_AUDIO_RATE:
                if m.ndim == 3:
                    if m.size(1) == C and C > 1:
                        has_ch = 1
                    elif m.size(1) == 1 or C == 1:
                        m = keep(m.reshape(m.size(0), m.size(-1)))      # (B,1,N): broadcast over channels
                    else:
                        raise AssertionError("mod_sig channel dim must be 1 or n_ch")
                assert m.size(0) == B and m.size(-1) == N
            else:
                assert m.ndim == 2 and m.size(0) == B
            s.mod = m.data_ptr()
            s.mod_has_ch = has_ch
            s.n_lo = m.size(-1)
        else:
            f = keep(self.freq.to(device=device, dtype=torch.float32).contiguous())
            p = keep(self.phase.to(device=device, dtype=torch.float32).contiguous())
            sh = keep(self.shape.to(device=device, dtype=torch.int32).contiguous())
            assert f.shape == (B,) and p.shape == (B,) and sh.shape == (B,)
            s.lfo_freq, s.lfo_phase, s.lfo_shape = f.data_ptr(), p.data_ptr(), sh.data_ptr()
            if self.exp is not None:
                e = keep(self.exp.to(device=device, dtype=torch.float32).contiguous())
                assert e.shape == (B,)
                s.lfo_exp = e.data_ptr()
            s.n_lo = int(self.n_lo)
            s.sr_lo = float(self.sr_lo)
        return s


def flanger_chorus(x: Tensor, mod: ModSource, m_min: int, m_lfo: int, feedback: Param, min_delay_width: Param,
                   width: Param, depth: Param, mix: Param, example_index: Optional[Tensor] = None,
                   out: Optional[Tensor] = None, interpolation: str = "linear") -> Tensor:
    """interpolation: "linear" (the reference, fx.py:113) or "allpass" (own definition, include/modfx.h)."""
    _require_cuda(x, "x")
    assert x.ndim == 3 and interpolation in ("linear", "allpass")
    x = x.contiguous()
    B, C, N = x.shape
    y = torch.empty_like(x) if out is None else out
    assert y.is_cuda and y.is_contiguous() and y.shape == x.shape and y.dtype == torch.float32
    keep = _Keep()
    with torch.cuda.device(x.device):
        src = mod.to_c(B, C, N, x.device, keep)
        args = [as_param(p, B, x.device, keep, n) for p, n in
                ((feedback, "feedback"), (min_delay_width, "min_delay_width"), (width, "width"),
                 (depth, "depth"), (mix, "mix"))]
        idx_ptr, n_items = ctypes.c_void_p(0), 0
        if example_index is not None:
            idx = keep(example_index.to(device=x.device, dtype=torch.int32).contiguous())
            idx_ptr, n_items = ctypes.c_void_p(idx.data_ptr()), idx.numel()
            if n_items == 0:
                return y
        L = _lib.lib()
        fn = L.modfx_flanger_chorus_f32 if interpolation == "linear" else L.modfx_flanger_chorus_allpass_f32
        _lib.check(fn(_ptr(x), _ptr(y), B, C, N, m_min, m_lfo, ctypes.byref(src), *args, idx_ptr, n_items, _stream()))
    return y


def tremolo(x: Tensor, mod: ModSource, mix: Param) -> Tensor:
    _require_cuda(x, "x")
    assert x.ndim == 3
    x = x.contiguous()
    B, C, N = x.shape
    y = torch.empty_like(x)
    keep = _Keep()
    with torch.cuda.device(x.device):
        src = mod.to_c(B, C, N, x.device, keep)
        _lib.check(_lib.lib().modfx_tremolo_f32(_ptr(x), _ptr(y), B, C, N, ctypes.byref(src),
                                                as_param(mix, B, x.device, keep, "mix"), _stream()))
    return y


def lfo(n: int, sr: float, freq: Tensor, phase: Tensor, shape: Tensor, exp: Optional[Tensor] = None) -> Tensor:
    _require_cuda(freq, "freq")
    B = freq.numel()
    out = torch.empty((B, n), device=freq.device, dtype=torch.float32)
    keep = _Keep()
    with torch.cuda.device(freq.device):
        f = keep(freq.contiguous())
        p = keep(phase.to(device=freq.device, dtype=torch.float32).contiguous())
        s = keep(shape.to(device=freq.device, dtype=torch.int32).contiguous())
        e = None if exp is None else keep(exp.to(device=freq.device, dtype=torch.float32).contiguous())
        _lib.check(_lib.lib().modfx_lfo_f32(_ptr(out), B, n, float(sr), _ptr(f), _ptr(p), _ptr(s), _ptr(e), _stream()))
    return out


def lfo_window(n_out: int, n_window: int, sr: float, freq: Tensor, phase: Tensor, shape: Tensor,
               start: Optional[Tensor] = None, exp: Optional[Tensor] = None) -> Tensor:
    """(B, n_out) = linear_interpolate_last_dim(make_mod_signal(...)[start : start + n_window], n_out) per example
    (datasets.py:442-450), computed from the LFO's closed form."""
    _require_cuda(freq, "freq")
    B, dev = freq.numel(), freq.device
    out = torch.empty((B, n_out), device=dev, dtype=torch.float32)
    keep = _Keep()
    with torch.cuda.device(dev):
        f = keep(freq.contiguous())
        p = keep(phase.to(device=dev, dtype=torch.float32).contiguous())
        s = keep(shape.to(device=dev, dtype=torch.int32).contiguous())
        e = None if exp is None else keep(exp.to(device=dev, dtype=torch.float32).contiguous())
        st = None if start is None else keep(start.to(device=dev, dtype=torch.int32).contiguous())
        _lib.check(_lib.lib().modfx_lfo_window_f32(_ptr(out), B, n_out, n_window, float(sr), _ptr(f), _ptr(p), _ptr(s),
                                                   _ptr(e), _ptr(st), _stream()))
    return out


def interp_linear(x: Tensor, n: int, align_corners: bool = True) -> Tensor:
    _require_cuda(x, "x")
    x = x.contiguous()
    I = x.size(-1)
    rows = x.numel() // I
    out = torch.empty(x.shape[:-1] + (n,), device=x.device, dtype=torch.float32)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().modfx_interp_linear_f32(_ptr(x), _ptr(out), rows, I, n, 1 if align_corners else 0,
                                                      _stream()))
    return out


def phaser(x: Tensor, sr: float, rate_hz: Tensor, depth: Tensor, centre_hz: Tensor, feedback: Tensor, mix: Tensor,
           block: int = 8192, example_index: Optional[Tensor] = None, out: Optional[Tensor] = None) -> Tensor:
    """x: (B, N) CUDA float32; per-example (B,) parameters."""
    _require_cuda(x, "x")
    assert x.ndim == 2
    x = x.contiguous()
    B, N = x.shape
    y = torch.empty_like(x) if out is None else out
    assert y.is_cuda and y.is_contiguous() and y.shape == x.shape and y.dtype == torch.float32
    keep = _Keep()
    with torch.cuda.device(x.device):
        ps = []
        for p, name in ((rate_hz, "rate_hz"), (depth, "depth"), (centre_hz, "centre_frequency_hz"),
                        (feedback, "feedback"), (mix, "mix")):
            t = keep(torch.as_tensor(p).detach().to(device=x.device, dtype=torch.float32).reshape(-1).contiguous())
            if t.numel() == 1 and B != 1:
                t = keep(t.expand(B).contiguous())
            assert t.shape == (B,), f"{name}: expected ({B},)"
            ps.append(t)
        idx_ptr, n_items = ctypes.c_void_p(0), 0
        n_work = B
        if example_index is not None:
            idx = keep(example_index.to(device=x.device, dtype=torch.int32).contiguous())
            idx_ptr, n_items = ctypes.c_void_p(idx.data_ptr()), idx.numel()
            n_work = n_items
            if n_items == 0:
                return y
        L = _lib.lib()
        ws = keep(torch.empty((max(1, int(L.modfx_phaser_workspace_bytes(n_work, N))),), device=x.device,
                              dtype=torch.uint8))
        _lib.check(L.modfx_phaser_f32(_ptr(x), _ptr(y), B, N, float(sr), *[_ptr(t) for t in ps], int(block),
                                      idx_ptr, n_items, _ptr(ws), _stream()))
    return y


def phaser_crop(x: Tensor, n_out: int, start: Tensor, sr: float, rate_hz: Tensor, depth: Tensor, centre_hz: Tensor,
                feedback: Tensor, mix: Tensor, block: int = 8192, want_dry: bool = True,
                example_index: Optional[Tensor] = None, out: Optional[Tensor] = None, dry_out: Optional[Tensor] = None,
                row_offsets: Optional[Tensor] = None, max_len: Optional[int] = None):
    """x: (rows, L) CUDA float32 rows of (at least) start + n_out samples.  Returns (wet (B, n_out), dry (B, n_out) or
    None): the phaser over each row from its first sample, delivered on the window [start, start + n_out)
    (PedalboardPhaserDataset.__getitem__, datasets.py:436-447).
    Without `example_index`: rows = B examples.  With it: x is COMPACT -- row i belongs to example example_index[i] --
    while start, the parameters and the (B, n_out) outputs `out` / `dry_out` stay indexed by the example id.
    With `row_offsets` (int64, one per row of `example_index`) x is a PACKED 1-D array: row i starts at x[row_offsets[i]]
    and holds start + n_out samples of example example_index[i]; `max_len` bounds start + n_out."""
    _require_cuda(x, "x")
    if row_offsets is not None:
        assert x.ndim == 1 and example_index is not None and max_len is not None and max_len >= n_out
        x = x.contiguous()
        rows, L_ = example_index.numel(), int(max_len)
        assert row_offsets.numel() == rows
    else:
        assert x.ndim == 2
        x = x.contiguous()
        rows, L_ = x.shape
    keep = _Keep()
    with torch.cuda.device(x.device):
        ps = [keep(torch.as_tensor(p).detach().to(device=x.device, dtype=torch.float32).reshape(-1).contiguous())
              for p in (rate_hz, depth, centre_hz, feedback, mix)]
        B = ps[0].numel()
        assert all(t.shape == (B,) for t in ps)
        st = keep(torch.as_tensor(start).to(device=x.device, dtype=torch.int32).reshape(-1).contiguous())
        assert st.shape == (B,)
        idx_ptr, n_items, compact = ctypes.c_void_p(0), 0, 0
        if example_index is not None:
            idx = keep(example_index.to(device=x.device, dtype=torch.int32).contiguous())
            assert idx.numel() == rows
            idx_ptr, n_items, compact = ctypes.c_void_p(idx.data_ptr()), idx.numel(), 1
        else:
            assert rows == B
        y = torch.empty((B, n_out), device=x.device, dtype=torch.float32) if out is None else out
        dry = dry_out if dry_out is not None else (torch.empty((B, n_out), device=x.device, dtype=torch.float32) if want_dry else None)
        assert y.is_contiguous() and y.numel() == B * n_out and (dry is None or (dry.is_contiguous() and dry.numel() == B * n_out))
        if example_index is not None and n_items == 0:
            return y, dry
        L = _lib.lib()
        ws = keep(torch.empty((max(1, int(L.modfx_phaser_workspace_bytes(max(rows, 1), L_))),), device=x.device, dtype=torch.uint8))
        if row_offsets is not None:
            offs = keep(row_offsets.to(device=x.device, dtype=torch.int64).contiguous())
            _lib.check(L.modfx_phaser_crop_packed_f32(_ptr(x), _ptr(offs), _ptr(y), _ptr(dry), B, L_, n_out, _ptr(st), float(sr),
                                                      *[_ptr(t) for t in ps], int(block), idx_ptr, n_items, _ptr(ws), _stream()))
        else:
            _lib.check(L.modfx_phaser_crop_f32(_ptr(x), compact, _ptr(y), _ptr(dry), B, L_, n_out, _ptr(st), float(sr),
                                               *[_ptr(t) for t in ps], int(block), idx_ptr, n_items, _ptr(ws), _stream()))
        ws.record_stream(torch.cuda.current_stream(x.device))
    return y, dry


def find_corners(mod_sig: Tensor):
    """(rows, n) CUDA float32 -> (top, bottom) uint8 flags (modulations.py:219-238)."""
    _require_cuda(mod_sig, "mod_sig")
    assert mod_sig.ndim == 2
    m = mod_sig.contiguous()
    top = torch.empty(m.shape, device=m.device, dtype=torch.uint8)
    bottom = torch.empty(m.shape, device=m.device, dtype=torch.uint8)
    with torch.cuda.device(m.device):
        _lib.check(_lib.lib().modfx_find_corners_f32(_ptr(m), _ptr(top), _ptr(bottom), m.size(0), m.size(1), _stream()))
    return top, bottom


def smoothen(x: Tensor, window: int) -> Tensor:
    """(rows, n) CUDA float32 -> (rows, n - window + 1) moving average (modulations.py:358-362)."""
    _require_cuda(x, "x")
    assert x.ndim == 2 and 1 <= window <= x.size(1)
    m = x.contiguous()
    out = torch.empty((m.size(0), m.size(1) - window + 1), device=m.device, dtype=torch.float32)
    with torch.cuda.device(m.device):
        _lib.check(_lib.lib().modfx_smoothen_f32(_ptr(m), _ptr(out), m.size(0), m.size(1), int(window), _stream()))
    return out


def stretch_corners(x: Tensor, max_n_corners: int) -> Tensor:
    """find_corners + _stretch_corners on an already smoothed (rows, n) CUDA float32 signal
    (modulations.py:259-307)."""
    _require_cuda(x, "x")
    assert x.ndim == 2
    m = x.contiguous()
    out = torch.empty_like(m)
    with torch.cuda.device(m.device):
        _lib.check(_lib.lib().modfx_stretch_corners_f32(_ptr(m), _ptr(out), m.size(0), m.size(1), int(max_n_corners),
                                                        _stream()))
    return out


def check_mod_sig(x: Tensor, min_top: int, max_top: int, min_bottom: int, max_bottom: int, min_frames: int) -> Tensor:
    """(rows, n) CUDA float32 -> (rows,) uint8 validity flags (modulations.py:311-345)."""
    _require_cuda(x, "x")
    assert x.ndim == 2
    m = x.contiguous()
    valid = torch.empty((m.size(0),), device=m.device, dtype=torch.uint8)
    with torch.cuda.device(m.device):
        _lib.check(_lib.lib().modfx_check_mod_sig_f32(_ptr(m), _ptr(valid), m.size(0), m.size(1), int(min_top),
                                                      int(max_top), int(min_bottom), int(max_bottom), int(min_frames),
                                                      _stream()))
    return valid


def _i32(values, device) -> Tensor:
    if isinstance(values, Tensor):
        return values.to(device=device, dtype=torch.int32, non_blocking=True).contiguous()
    return torch.tensor(values, dtype=torch.int32).to(device, non_blocking=True)


def logmel(x: Tensor, window: Tensor, fb_start: Tensor, fb_count: Tensor, fb_weight: Tensor, fb_taps: int, hop: int = 256,
           eps: float = 1e-7, apply_log: bool = True) -> Tensor:
    """(..., T) CUDA float32 -> (..., n_mels, T // hop + 1): MelSpectrogram [-> clip -> log] of models.py:170-175,199,207-208
    with the banded mel table of models.banded() (n_fft = len(window) = 1024)."""
    _require_cuda(x, "x")
    x = x.detach().float().contiguous()
    T, lead = x.size(-1), x.shape[:-1]
    R = x.numel() // T
    n_mels, nf = fb_start.numel(), T // hop + 1
    out = torch.empty(lead + (n_mels, nf), device=x.device, dtype=torch.float32)
    if R == 0:
        return out
    keep = _Keep()
    w = keep(window.to(device=x.device, dtype=torch.float32).contiguous())
    s = keep(fb_start.to(device=x.device, dtype=torch.int32).contiguous())
    c = keep(fb_count.to(device=x.device, dtype=torch.int32).contiguous())
    fw = keep(fb_weight.to(device=x.device, dtype=torch.float32).contiguous())
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().modfx_logmel_f32(_ptr(x), _ptr(out), R, T, w.numel(), hop, n_mels, _ptr(w), _ptr(s), _ptr(c),
                                               _ptr(fw), fw.size(1), int(fb_taps), float(eps), 1 if apply_log else 0, 0, 0,
                                               ctypes.c_void_p(0), 0, _stream()))
    return out


def lfo_sections_(out: Tensor, sec_off, sec_start, sec_len, sec_shape) -> Tensor:
    """In place: overwrite sections of `out` (B, n) with one-period LFOs (modulations.py:203-209)."""
    _require_cuda(out, "out")
    assert out.ndim == 2 and out.is_contiguous()
    dev = out.device
    ts = [_i32(v, dev) for v in (sec_off, sec_start, sec_len, sec_shape)]
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().modfx_lfo_sections_f32(_ptr(out), out.size(0), out.size(1), *[_ptr(t) for t in ts],
                                                     _stream()))
    return out


def stretch_sections(x: Tensor, sec_off, in_start, in_len, new_len, out_start) -> Tensor:
    """(B, n) -> (B, n): resampled sections concatenated (modulations.py:139-159)."""
    _require_cuda(x, "mod_sig")
    assert x.ndim == 2
    x = x.contiguous()
    out = torch.empty_like(x)
    ts = [_i32(v, x.device) for v in (sec_off, in_start, in_len, new_len, out_start)]
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().modfx_stretch_sections_f32(_ptr(x), _ptr(out), x.size(0), x.size(1),
                                                         *[_ptr(t) for t in ts], _stream()))
    return out


def combined_lfo(n: int, sr: float, freq: Tensor, phase: Tensor, shapes: Tensor, words: Tensor):
    """Batched make_combined_mod_sig with the reference's draw order replayed on the device (modulations.py:191-210).
    freq / phase (B,) float32 CUDA, shapes (S,) int32 CUDA, words (K,) raw generator outputs as int32 / uint32 CUDA.
    Returns (out (B, n), base (B,) int32 index into shapes, consumed (2,) int32 = [words used, error flag])."""
    _require_cuda(freq, "freq")
    dev = freq.device
    B, S = freq.numel(), shapes.numel()
    out = torch.empty((B, n), device=dev, dtype=torch.float32)
    base = torch.empty((B,), device=dev, dtype=torch.int32)
    consumed = torch.zeros((2,), device=dev, dtype=torch.int32)
    L = _lib.lib()
    ws = torch.empty((max(1, int(L.modfx_combined_lfo_workspace_bytes(B, n, S))),), device=dev, dtype=torch.uint8)
    with torch.cuda.device(dev):
        _lib.check(L.modfx_combined_lfo_f32(_ptr(out), B, n, float(sr), _ptr(freq), _ptr(phase), _ptr(shapes), S,
                                            _ptr(words), words.numel(), _ptr(base), _ptr(consumed), _ptr(ws), _stream()))
    ws.record_stream(torch.cuda.current_stream(dev))
    return out, base, consumed


# ---- LFO-net body (SURVEY 8f N3), channels-last activations -----------------------------------------------
def cnn_layernorm(x: Tensor, x_is_nchw: bool = False, eps: float = 1e-5, round_tf32: bool = False,
                  out: Optional[Tensor] = None) -> Tensor:
    """nn.LayerNorm([H, W], elementwise_affine=False) per (b, c) (models.py:186).  x (B, C, H, W) when
    `x_is_nchw` else (B, H, W, C); returns (B, H, W, C) (in place when `out is x` and x is channels-last)."""
    _require_cuda(x, "x")
    assert x.ndim == 4
    x = x.contiguous()
    B, C, H, W = x.shape if x_is_nchw else (x.size(0), x.size(3), x.size(1), x.size(2))
    if out is None:
        out = torch.empty((B, H, W, C), device=x.device, dtype=torch.float32)
    L = _lib.lib()
    ws = torch.empty(max(int(L.modfx_cnn_layernorm_workspace_bytes(B, C, H, W)), 16), dtype=torch.uint8, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(L.modfx_cnn_layernorm_f32(_ptr(x), _ptr(out), B, C, H, W, 1 if x_is_nchw else 0, float(eps),
                                             1 if round_tf32 else 0, _ptr(ws), _stream()))
        ws.record_stream(torch.cuda.current_stream())
    return out


def cnn_conv_pool_prelu(x: Tensor, weight: Tensor, bias: Tensor, slope: Tensor, dil_w: int = 1, tf32: bool = True) -> Tensor:
    """Conv2d(Cin, 64, (5, 13), dilation=(1, dil_w), padding="same") -> MaxPool2d((2, 1)) -> PReLU (models.py:187-189).
    x (B, H, W, Cin) channels-last; weight (5, 13, 64, Cin); returns (B, H/2, W, 64).  tf32: tcgen05 tensor cores."""
    for t, n in ((x, "x"), (weight, "weight"), (bias, "bias"), (slope, "slope")):
        _require_cuda(t, n)
    assert x.ndim == 4 and weight.ndim == 4 and weight.size(3) == x.size(3)
    x, weight, bias, slope = x.contiguous(), weight.contiguous(), bias.contiguous(), slope.contiguous()
    B, H, W, Cin = x.shape
    KH, KW, Cout, _ = weight.shape
    y = torch.empty((B, H // 2, W, Cout), device=x.device, dtype=torch.float32)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().modfx_cnn_conv_pool_prelu_f32(
            _ptr(x), _ptr(y), B, H, W, Cin, Cout, KH, KW, int(dil_w), _ptr(weight), _ptr(bias), _ptr(slope),
            _lib.CNN_TF32 if tf32 else _lib.CNN_FP32, _stream()))
    return y


def cnn_head(x: Tensor, weight: Tensor, bias: Tensor):
    """tr.mean(x, dim=-2) -> Conv1d(C, L, 1) -> sigmoid (models.py:210-214).  x (B, H, W, C) channels-last,
    weight (L, C); returns (output (B, L, W), latent (B, C, W))."""
    for t, n in ((x, "x"), (weight, "weight"), (bias, "bias")):
        _require_cuda(t, n)
    x, weight, bias = x.contiguous(), weight.contiguous(), bias.contiguous()
    B, H, W, C = x.shape
    Ld = weight.size(0)
    latent = torch.empty((B, C, W), device=x.device, dtype=torch.float32)
    out = torch.empty((B, Ld, W), device=x.device, dtype=torch.float32)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().modfx_cnn_head_f32(_ptr(x), _ptr(latent), _ptr(out), B, H, W, C, Ld, _ptr(weight), _ptr(bias),
                                                 _stream()))
    return out, latent


# ---- training (TF32 parameter gradients of the body, models.Spectral2DCNN) ----------------------------------------

def _train_ws(B: int, H: int, W: int, L: int, device) -> Tensor:
    return torch.empty(int(_lib.lib().modfx_cnn_train_workspace_bytes(B, H, W, L)), dtype=torch.uint8, device=device)


def cnn_conv_pool_prelu_train(x: Tensor, weight: Tensor, bias: Tensor, slope: Tensor, dil_w: int = 1):
    """cnn_conv_pool_prelu (TF32) that also returns what its backward needs: (y, z = maxpool(conv) + bias, argmax uint8,
    1 where the lower conv row of a pooled pair won)."""
    for t, n in ((x, "x"), (weight, "weight"), (bias, "bias"), (slope, "slope")):
        _require_cuda(t, n)
    x, weight, bias, slope = x.contiguous(), weight.contiguous(), bias.contiguous(), slope.contiguous()
    B, H, W, Cin = x.shape
    y = torch.empty((B, H // 2, W, 64), device=x.device, dtype=torch.float32)
    z = torch.empty_like(y)
    am = torch.empty((B, H // 2, W, 64), device=x.device, dtype=torch.uint8)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().modfx_cnn_conv_pool_prelu_train_f32(_ptr(x), _ptr(y), _ptr(z), _ptr(am), B, H, W, Cin, int(dil_w),
                                                                  _ptr(weight), _ptr(bias), _ptr(slope), _stream()))
    return y, z, am


def cnn_conv_dgrad(dconv: Tensor, weight_t: Tensor, dil_w: int = 1) -> Tensor:
    """Input gradient of the 64 -> 64 convolution: dconv (B, H, W, 64), weight_t[kh][kw][ci][co] = weight[4-kh][12-kw][co][ci]."""
    _require_cuda(dconv, "dconv")
    _require_cuda(weight_t, "weight_t")
    dconv, weight_t = dconv.contiguous(), weight_t.contiguous()
    B, H, W, _ = dconv.shape
    dx = torch.empty_like(dconv)
    with torch.cuda.device(dconv.device):
        _lib.check(_lib.lib().modfx_cnn_conv_dgrad_tf32_f32(_ptr(dconv), _ptr(dx), B, H, W, int(dil_w), _ptr(weight_t), _stream()))
    return dx


def cnn_conv_wgrad(x: Tensor, dconv: Tensor, dil_w: int = 1) -> Tensor:
    """Weight gradient (64, Cin, 5, 13) of the convolution: x (B, H, W, Cin) its TF32 input, dconv (B, H, W, 64)."""
    _require_cuda(x, "x")
    _require_cuda(dconv, "dconv")
    x, dconv = x.contiguous(), dconv.contiguous()
    B, H, W, Cin = x.shape
    dw = torch.empty((64, Cin, 5, 13), device=x.device, dtype=torch.float32)
    ws = _train_ws(B, H, W, 1, x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().modfx_cnn_conv_wgrad_tf32_f32(_ptr(x), _ptr(dconv), _ptr(dw), B, H, W, Cin, int(dil_w), _ptr(ws),
                                                            _stream()))
        ws.record_stream(torch.cuda.current_stream())
    return dw


def cnn_pool_prelu_bwd(dy: Tensor, z: Tensor, argmax: Tensor, slope: Tensor):
    """Backward of MaxPool2d((2, 1)) -> PReLU: (dconv (B, H, W, 64) rounded to TF32, dbias (64,), dslope (64,))."""
    for t, n in ((dy, "dy"), (z, "z"), (argmax, "argmax"), (slope, "slope")):
        _require_cuda(t, n)
    dy, z, argmax, slope = dy.contiguous(), z.contiguous(), argmax.contiguous(), slope.contiguous()
    B, Hp, W, C = dy.shape
    dconv = torch.empty((B, 2 * Hp, W, C), device=dy.device, dtype=torch.float32)
    db = torch.empty(C, device=dy.device, dtype=torch.float32)
    ds = torch.empty(C, device=dy.device, dtype=torch.float32)
    ws = _train_ws(B, 2 * Hp, W, 1, dy.device)
    with torch.cuda.device(dy.device):
        _lib.check(_lib.lib().modfx_cnn_pool_prelu_bwd_f32(_ptr(dy), _ptr(z), _ptr(argmax), _ptr(slope), _ptr(dconv), _ptr(db),
                                                           _ptr(ds), B, 2 * Hp, W, _ptr(ws), _stream()))
        ws.record_stream(torch.cuda.current_stream())
    return dconv, db, ds


def cnn_layernorm_bwd(g: Tensor, x: Tensor, eps: float = 1e-5) -> Tensor:
    """Input gradient of cnn_layernorm on a channels-last x (B, H, W, C), given the output gradient g."""
    _require_cuda(g, "g")
    _require_cuda(x, "x")
    g, x = g.contiguous(), x.contiguous()
    B, H, W, C = x.shape
    L = _lib.lib()
    stats = torch.empty(max(int(L.modfx_cnn_layernorm_workspace_bytes(B, C, H, W)), 16), dtype=torch.uint8, device=x.device)
    ws = _train_ws(B, H, W, 1, x.device)
    dx = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.check(L.modfx_cnn_layernorm_f32(_ptr(x), _ptr(dx), B, C, H, W, 0, float(eps), 0, _ptr(stats), _stream()))   # statistics
        _lib.check(L.modfx_cnn_layernorm_bwd_f32(_ptr(g), _ptr(x), _ptr(stats), _ptr(dx), B, C, H, W, float(eps), _ptr(ws),
                                                 _stream()))
        ws.record_stream(torch.cuda.current_stream())
        stats.record_stream(torch.cuda.current_stream())
    return dx


def cnn_head_bwd(latent: Tensor, out: Tensor, dout: Tensor, dlatent: Tensor, weight: Tensor, H: int):
    """Backward of cnn_head: (dx (B, H, W, C), dweight (L, C), dbias (L,))."""
    for t, n in ((latent, "latent"), (out, "out"), (dout, "dout"), (dlatent, "dlatent"), (weight, "weight")):
        _require_cuda(t, n)
    latent, out, dout, dlatent, weight = (t.contiguous() for t in (latent, out, dout, dlatent, weight))
    B, C, W = latent.shape
    Ld = out.size(1)
    dx = torch.empty((B, H, W, C), device=latent.device, dtype=torch.float32)
    dw = torch.empty((Ld, C), device=latent.device, dtype=torch.float32)
    db = torch.empty(Ld, device=latent.device, dtype=torch.float32)
    ws = _train_ws(B, 2, W, Ld, latent.device)
    with torch.cuda.device(latent.device):
        _lib.check(_lib.lib().modfx_cnn_head_bwd_f32(_ptr(latent), _ptr(out), _ptr(dout), _ptr(dlatent), _ptr(dx), _ptr(dw),
                                                     _ptr(db), B, int(H), W, C, Ld, _ptr(weight), _ptr(ws), _stream()))
        ws.record_stream(torch.cuda.current_stream())
    return dx, dw, db
