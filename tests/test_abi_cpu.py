"""CPU tests: the C-ABI library loads and exports every symbol include/modfx.h declares."""
import os
import re

import pytest

from mod_extraction_b200 import _build, _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    txt = open(os.path.join(ROOT, "include", "modfx.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(modfx_[a-z0-9_]+)\s*\(", txt)))


def test_library_builds_and_exports_header_symbols():
    _build.build()
    L = _lib.lib()
    names = header_symbols()
    assert "modfx_flanger_chorus_f32" in names and "modfx_logmel_f32" in names
    for n in names:
        assert hasattr(L, n), f"libmodfx.so does not export {n}"
    assert sorted(_lib.exported_symbols()) == names, "ctypes signature table and header disagree"
    assert L.modfx_abi_version() == 1


def test_no_cpu_fallback():
    """Without a GPU the product must fail loudly, never compute on the host."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from mod_extraction_b200 import fx, modulations, util
    m = fx.MonoFlangerChorusModule(1, 1, 64, 44100, 1.0, 10.0)
    with pytest.raises(RuntimeError):
        m(torch.zeros(1, 1, 64), torch.zeros(1, 64))
    with pytest.raises(RuntimeError):
        modulations.make_mod_signal(10, 441, 2.0)
    with pytest.raises(RuntimeError):
        util.linear_interpolate_last_dim(torch.zeros(2, 8), 16)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "mod_extraction_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("no oracle", ""), f"{f} mentions the oracle"


def test_reference_asserts_are_kept():
    import torch
    from mod_extraction_b200 import fx
    m = fx.MonoFlangerChorusModule(2, 1, 64, 44100, 1.0, 10.0)
    x = torch.zeros(2, 1, 64)
    with pytest.raises(AssertionError):
        m(x, torch.zeros(2, 63))                       # fx.py:83
    with pytest.raises(AssertionError):
        m(x, torch.zeros(2, 64), feedback=1.0)         # fx.py:69 (feedback < 1 strictly)
    with pytest.raises(AssertionError):
        m(x, torch.zeros(2, 64), mix=torch.tensor([0.5, 1.5]))     # fx.py:55
    with pytest.raises(AssertionError):
        m(x[:, 0], torch.zeros(2, 64))                 # fx.py:80
    with pytest.raises(AssertionError):
        fx.apply_tremolo(x, torch.zeros(2, 64), mix=1.5)           # fx.py:21


def test_torch_ops_registered_cuda_only():
    """torch.ops.modfx.* exist and have no CPU kernel: the dispatcher itself refuses CPU tensors."""
    import torch
    import mod_extraction_b200._torch_ops  # noqa: F401
    assert hasattr(torch.ops.modfx, "flanger_chorus") and hasattr(torch.ops.modfx, "phaser")
    assert hasattr(torch.ops.modfx, "cnn_conv_pool_prelu") and hasattr(torch.ops.modfx, "cnn_head")
    for name in ("tremolo", "mel_power", "logmel", "find_corners", "lfo_sections", "stretch_sections", "combined_lfo",
                 "smoothen", "stretch_corners", "check_mod_sig", "lfo", "interp_linear"):      # SURVEY 8b: every op of the path
        assert hasattr(torch.ops.modfx, name), name
    with pytest.raises((NotImplementedError, RuntimeError)):
        torch.ops.modfx.smoothen(torch.zeros(2, 40), 4)
    with pytest.raises((NotImplementedError, RuntimeError)):
        torch.ops.modfx.cnn_layernorm(torch.zeros(1, 2, 4, 4), True, 1e-5, False)
    with pytest.raises((NotImplementedError, RuntimeError)):
        torch.ops.modfx.interp_linear(torch.zeros(2, 8), 16, True)


def test_cnn_entry_points_validate_before_touching_the_gpu():
    """Argument checks of the N3 entry points run on the host: status codes without a device."""
    import ctypes
    L = _lib.lib()
    buf = (ctypes.c_float * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    nul = ctypes.c_void_p(0)
    assert L.modfx_cnn_conv_pool_prelu_f32(nul, p, 1, 2, 4, 64, 64, 5, 13, 1, p, p, p, 1, nul) == -1          # NULL x
    assert L.modfx_cnn_conv_pool_prelu_f32(p, p, 1, 2, 4, 64, 64, 5, 13, 1, p, p, p, 1, nul) == -1            # x aliases y
    assert L.modfx_cnn_conv_pool_prelu_f32(p, nul, 1, 2, 4, 64, 64, 5, 13, 1, p, p, p, 1, nul) == -1
    q = ctypes.cast(ctypes.addressof(buf) + 64, ctypes.c_void_p)
    assert L.modfx_cnn_conv_pool_prelu_f32(p, q, 1, 2, 4, 64, 64, 3, 3, 1, p, p, p, 0, nul) == -2             # 3x3 kernel
    assert L.modfx_cnn_conv_pool_prelu_f32(p, q, 1, 3, 4, 64, 64, 5, 13, 1, p, p, p, 0, nul) == -2            # odd H
    assert L.modfx_cnn_conv_pool_prelu_f32(p, q, 1, 2, 4, 64, 64, 5, 13, 32, p, p, p, 0, nul) == -2           # dilation 32
    assert L.modfx_cnn_conv_pool_prelu_f32(p, q, 0, 2, 4, 64, 64, 5, 13, 1, p, p, p, 1, nul) == 0             # empty batch
    assert L.modfx_cnn_conv_pool_prelu_tf32x3_f32(p, nul, q, 1, 2, 4, 1, p, p, p, p, nul) == -1
    assert L.modfx_cnn_layernorm_f32(p, p, 1, 2, 4, 4, 1, 1e-5, 0, p, nul) == -1                               # NCHW in place
    assert L.modfx_cnn_layernorm_f32(p, q, 1, 3, 4, 4, 0, 1e-5, 0, p, nul) == -2                               # 3 does not divide 256
    assert L.modfx_cnn_layernorm_f32(p, q, 0, 2, 4, 4, 0, 1e-5, 0, p, nul) == 0
    assert L.modfx_cnn_layernorm_workspace_bytes(4, 64, 128, 345) > 0 and L.modfx_cnn_layernorm_workspace_bytes(1, 0, 1, 1) == -1
    assert L.modfx_cnn_head_f32(p, p, nul, 1, 1, 1, 1, 1, p, p, nul) == -1
    assert L.modfx_specaugment_fill_f32(p, 1, 4, 4, 3, 2, 0, 0, 1e-7, 1, nul) == -1                            # f0 > f1
    assert L.modfx_specaugment_fill_f32(p, 1, 4, 4, 0, 0, 0, 0, 1e-7, 1, nul) == 0                             # nothing to mask


def test_effect_entry_points_validate_before_touching_the_gpu():
    """Argument checks of the flanger / chorus, tremolo and phaser entry points run on the host: status codes without a
    device, and a call with nothing to render returns MODFX_OK before any shared-memory refusal."""
    import ctypes
    L = _lib.lib()
    buf = (ctypes.c_float * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    nul = ctypes.c_void_p(0)
    P = _lib.ModfxParam
    Mod = _lib.ModfxModSource
    audio = Mod(kind=_lib.MOD_AUDIO_RATE, mod=p)
    lfo = Mod(kind=_lib.MOD_LFO, n_lo=64, sr_lo=100.0, lfo_freq=p, lfo_phase=p, lfo_shape=p)

    def fc(x=p, B=1, N=64, M=(10, 10), mod=audio, feedback=0.5, index=nul, n_items=0, allpass=False):
        f = L.modfx_flanger_chorus_allpass_f32 if allpass else L.modfx_flanger_chorus_f32
        half = P(None, 0.5)
        return f(x, p, B, 1, N, M[0], M[1], ctypes.byref(mod), P(None, feedback), half, half, half, half, index,
                 n_items, nul)

    long_line = (20000, 20441)                                                  # 40 441 samples
    assert fc(x=nul) == -1
    assert fc(feedback=1.0) == -1                                               # fx.py:69 (feedback < 1 strictly)
    assert fc(B=0, M=long_line) == 0
    assert fc(index=p, n_items=0, M=long_line) == 0                             # empty example_index
    assert fc(M=long_line) == -2 and b"shared memory" in L.modfx_last_error()
    assert fc(M=long_line, allpass=True) == -2 and b"shared memory" in L.modfx_last_error()
    assert fc(mod=lfo, allpass=True) == -2                                      # all-pass reads mod from memory
    assert fc(mod=Mod(kind=_lib.MOD_CONTROL_RATE, mod=p, n_lo=65)) == -1       # n_lo > N
    assert fc(mod=Mod(kind=7, mod=p)) == -1                                     # unknown modulation kind

    def tremolo(B, mod=audio, N=64):
        return L.modfx_tremolo_f32(p, p, B, 1, N, ctypes.byref(mod), P(None, 0.5), nul)

    big_lfo = Mod(kind=_lib.MOD_LFO, n_lo=60000, sr_lo=100.0, lfo_freq=p, lfo_phase=p, lfo_shape=p)
    assert tremolo(0) == 0
    assert tremolo(0, big_lfo, N=100000) == 0
    assert tremolo(1, big_lfo, N=100000) == -2 and b"shared memory" in L.modfx_last_error()

    sr = ctypes.c_float(44100.0)
    assert L.modfx_phaser_f32(nul, p, 1, 64, sr, p, p, p, p, p, 0, nul, 0, p, nul) == -1
    assert L.modfx_phaser_f32(p, p, 1, 64, sr, p, p, p, p, p, 0, p, 0, nul, nul) == 0       # empty example_index
    assert L.modfx_phaser_crop_f32(p, 0, p, nul, 1, 64, 64, nul, sr, p, p, p, p, p, 0, nul, 0, p, nul) == -1   # NULL start
    assert L.modfx_phaser_crop_f32(p, 0, p, nul, 1, 64, 65, p, sr, p, p, p, p, p, 0, nul, 0, p, nul) == -1     # n_out > N
    assert L.modfx_phaser_crop_f32(p, 1, p, nul, 1, 64, 64, p, sr, p, p, p, p, p, 0, nul, 0, p, nul) == -1     # x_compact
    assert L.modfx_phaser_crop_packed_f32(p, p, p, nul, 1, 64, 64, p, sr, p, p, p, p, p, 0, nul, 0, p, nul) == -1


def test_build_is_keyed_by_source_content():
    """_build.build() must not reuse a library built from other sources: the hash of csrc/ + include/ + flags is stored
    beside the library and compared, whatever the file times say."""
    from mod_extraction_b200 import _build
    path = _build.build()
    assert os.path.exists(path)
    stamp = open(_build.STAMP_PATH).read().strip()
    assert stamp == _build.source_hash()
    assert _build.is_current()
    # a library with a foreign stamp is stale
    try:
        open(_build.STAMP_PATH, "w").write("0" * 64)
        assert not _build.is_current()
    finally:
        open(_build.STAMP_PATH, "w").write(stamp)
