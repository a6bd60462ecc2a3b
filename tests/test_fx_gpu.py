"""GPU parity: flanger/chorus, tremolo, LFO synthesis and resampling through the C ABI
(mod_extraction_b200 shims -> libmodfx.so) against the CPU oracle and the reference goldens."""
import math

import numpy as np
import pytest
import torch

from oracle import oracle
from tests.helpers import SHAPES6, SR, fc_params_from_golden, golden, guitar, snr_db, white

pytestmark = pytest.mark.gpu


def dev():
    return torch.device("cuda", 0)


def to_t(p):
    return torch.from_numpy(p).to(dev()) if isinstance(p, np.ndarray) else p


# --------------------------------------------------------------------------- E1 goldens (bit-exact)

def test_flanger_chorus_bit_exact_vs_reference_goldens():
    from mod_extraction_b200.fx import MonoFlangerChorusModule
    g = golden("flanger_chorus")
    for k in range(int(g["n"])):
        x = g[f"x{k}"]
        B, C, N = x.shape
        mmd, mld = (float(v) for v in g[f"delays{k}"])
        m = MonoFlangerChorusModule(B, C, N, SR, mmd, mld)
        params = [to_t(p) for p in fc_params_from_golden(g, k)]
        y = m(torch.from_numpy(x).to(dev()), torch.from_numpy(g[f"mod{k}"]).to(dev()), *params)
        assert y.is_cuda and y.shape == x.shape
        assert np.array_equal(y.cpu().numpy(), g[f"y{k}"]), str(g[f"name{k}"])


def test_flanger_cpu_tensors_in_cpu_out():
    """The reference call site hands CPU tensors (data_modules.py:457)."""
    from mod_extraction_b200.fx import MonoFlangerChorusModule
    g = golden("flanger_chorus")
    k = 1
    x = g[f"x{k}"]
    B, C, N = x.shape
    m = MonoFlangerChorusModule(B, C, N, SR, *[float(v) for v in g[f"delays{k}"]])
    params = [torch.from_numpy(p) if isinstance(p, np.ndarray) else p for p in fc_params_from_golden(g, k)]
    y = m(torch.from_numpy(x), torch.from_numpy(g[f"mod{k}"]), *params)
    assert not y.is_cuda
    assert np.array_equal(y.numpy(), g[f"y{k}"])


# --------------------------------------------------------------------------- E1 vs oracle, seeded

def _rand_params(B, rng, mdw_lo=0.0, fb_hi=0.7):
    U = lambda lo, hi: rng.uniform(lo, hi, B).astype(np.float32)
    return [U(0.0, fb_hi), U(mdw_lo, 1.0), U(0.25, 1.0), U(0.25, 1.0), U(0.25, 1.0)]


def _lfo_lo(B, rng, n_lo=882, sr_lo=441.0, rate=(0.5, 3.0), exp=1.0):
    rows = []
    for b in range(B):
        f = float(np.exp(rng.uniform(np.log(rate[0]), np.log(rate[1]))))
        rows.append(oracle.make_mod_signal(n_lo, sr_lo, f, float(rng.uniform(0, 2 * math.pi)), SHAPES6[b % 6], exp))
    return np.stack(rows)


@pytest.mark.parametrize("name,mmd,mld,mdw_lo", [("flanger", 1.0, 10.0, 0.0), ("chorus", 30.0, 10.0, 0.367),
                                                 ("flanger_eval", 1.0, 4.0, 0.0)])
@pytest.mark.parametrize("family", ["white", "guitar"])
def test_flanger_chorus_bit_exact_vs_oracle_2s(name, mmd, mld, mdw_lo, family):
    from mod_extraction_b200.fx import MonoFlangerChorusModule
    rng = np.random.RandomState(hash((name, family)) % 2 ** 31)
    B, N = 12, 88200
    x = white((B, 1, N), 5) if family == "white" else guitar(B, N, 6)
    lo = _lfo_lo(B, rng)
    mod = oracle.linear_interpolate_last_dim(lo, N)
    params = _rand_params(B, rng, mdw_lo)
    ref = oracle.flanger_chorus(x, mod, *params, max_min_delay_ms=mmd, max_lfo_delay_ms=mld)
    m = MonoFlangerChorusModule(B, 1, N, SR, mmd, mld)
    xd = torch.from_numpy(x).to(dev())
    tp = [to_t(p) for p in params]
    # (a) literal signature: audio-rate mod_sig
    y = m(xd, torch.from_numpy(mod).to(dev()), *tp).cpu().numpy()
    assert np.array_equal(y, ref)
    # (b) fused x100 upsample of the control-rate LFO (data_modules.py:454-455)
    y2 = m.forward_control_rate(xd, torch.from_numpy(lo).to(dev()), *tp).cpu().numpy()
    assert np.array_equal(y2, ref)


def test_flanger_worst_case_serial_delays():
    """Delay pinned at 0..2 samples (strictly serial recurrence) and random jumps of the
    modulation: every schedule of the kernel must give the reference's bits."""
    from mod_extraction_b200.fx import MonoFlangerChorusModule
    rng = np.random.RandomState(17)
    B, N = 6, 20000
    x = white((B, 1, N), 9)
    mod = np.zeros((B, N), dtype=np.float32)
    mod[0] = 0.0                                            # d = mdw*44 exactly
    mod[1] = rng.uniform(0, 0.004, N)                       # sub-sample .. 2 samples
    mod[2] = rng.uniform(0, 1, N)                           # white modulation: all schedules mixed
    mod[3] = (np.arange(N) % 700) / 700.0 * 0.2             # ramps through the 32 / 128 thresholds
    mod[4] = np.clip(np.sin(np.arange(N) * 0.01) * 0.05 + 0.04, 0, 1)
    mod[5] = 1.0
    fb = np.array([0.69, 0.6, 0.5, 0.69, 0.3, 0.0], dtype=np.float32)
    mdw = np.array([0.0, 0.0, 0.0, 0.01, 0.2, 1.0], dtype=np.float32)
    ones = np.ones(B, dtype=np.float32)
    params = [fb, mdw, ones, ones * 0.9, ones * 0.8]
    ref = oracle.flanger_chorus(x, mod, *params, max_min_delay_ms=1.0, max_lfo_delay_ms=10.0)
    m = MonoFlangerChorusModule(B, 1, N, SR, 1.0, 10.0)
    y = m(torch.from_numpy(x).to(dev()), torch.from_numpy(mod).to(dev()), *[to_t(p) for p in params])
    assert np.array_equal(y.cpu().numpy(), ref)


def test_flanger_every_schedule_of_the_kernel():
    """Constant delays of 0.5 .. 9.5, 31.5, 32.5, 64 .. 128.5 samples and slow ramps across those
    boundaries: exercises the register-history serial run for every tap distance K, the wave
    schedule, the one-wave block, the two-wave and the one-shot 128-sample tile, plus the transitions between
    them."""
    from mod_extraction_b200.fx import MonoFlangerChorusModule
    N = 12000
    delays = [0.0, 0.5, 1.0, 1.5, 2.5, 3.5, 4.5, 5.5, 6.5, 7.5, 8.5, 9.5, 15.25, 31.5, 32.5, 64.0, 65.5, 96.5, 127.5, 128.5,
              300.0]
    ramps = [(0.0, 12.0), (12.0, 0.0), (6.0, 40.0), (140.0, 20.0), (0.0, 484.0), (60.0, 135.0)]
    B = len(delays) + len(ramps)
    x = white((B, 1, N), 77)
    mod = np.zeros((B, N), dtype=np.float32)
    for i, d in enumerate(delays):
        mod[i] = d / 441.0
    t = np.linspace(0.0, 1.0, N)
    for i, (d0, d1) in enumerate(ramps):
        mod[len(delays) + i] = (d0 + (d1 - d0) * t) / 441.0
    rng = np.random.RandomState(5)
    fb = rng.uniform(0.3, 0.69, B).astype(np.float32)
    zeros, ones = np.zeros(B, dtype=np.float32), np.ones(B, dtype=np.float32)
    params = [fb, zeros, ones, ones * 0.8, ones * 0.9]          # min_delay_width = 0: delay = 441 * mod
    ref = oracle.flanger_chorus(x, mod, *params, max_min_delay_ms=1.0, max_lfo_delay_ms=10.0)
    m = MonoFlangerChorusModule(B, 1, N, SR, 1.0, 10.0)
    y = m(torch.from_numpy(x).to(dev()), torch.from_numpy(mod).to(dev()), *[to_t(p) for p in params]).cpu().numpy()
    for i in range(B):
        assert np.array_equal(y[i], ref[i]), (i, (delays + ramps)[i])
    # same through the control-rate path (delays now follow the x100 upsample of 120 control points)
    lo = mod[:, ::100].copy()
    ref2 = oracle.flanger_chorus(x, oracle.linear_interpolate_last_dim(lo, N), *params, max_min_delay_ms=1.0,
                                 max_lfo_delay_ms=10.0)
    y2 = m.forward_control_rate(torch.from_numpy(x).to(dev()), torch.from_numpy(lo).to(dev()),
                                *[to_t(p) for p in params]).cpu().numpy()
    assert np.array_equal(y2, ref2)


@pytest.mark.parametrize("N", [1, 31, 32, 33, 127, 128, 129, 485, 1000])
def test_flanger_ragged_lengths(N):
    from mod_extraction_b200.fx import MonoFlangerChorusModule
    rng = np.random.RandomState(N)
    B, C = 3, 2
    x = white((B, C, N), N)
    mod = rng.uniform(0, 1, (B, C, N)).astype(np.float32)
    params = _rand_params(B, rng)
    for mmd, mld in [(1.0, 10.0), (30.0, 10.0), (0.05, 0.05)]:
        ref = oracle.flanger_chorus(x, mod, *params, max_min_delay_ms=mmd, max_lfo_delay_ms=mld)
        m = MonoFlangerChorusModule(B, C, N, SR, mmd, mld)
        y = m(torch.from_numpy(x).to(dev()), torch.from_numpy(mod).to(dev()), *[to_t(p) for p in params])
        assert np.array_equal(y.cpu().numpy(), ref), (N, mmd)


def test_flanger_example_index_and_out():
    from mod_extraction_b200.fx import MonoFlangerChorusModule
    rng = np.random.RandomState(3)
    B, N = 9, 5000
    x = white((B, 1, N), 1)
    lo = _lfo_lo(B, rng, n_lo=50, sr_lo=441.0)
    params = _rand_params(B, rng)
    ref = oracle.flanger_chorus(x, oracle.linear_interpolate_last_dim(lo, N), *params, max_min_delay_ms=1.0,
                                max_lfo_delay_ms=10.0)
    m = MonoFlangerChorusModule(B, 1, N, SR, 1.0, 10.0)
    out = torch.full((B, 1, N), 7.0, device=dev())
    idx = torch.tensor([0, 3, 4, 8], dtype=torch.int32)
    m.forward_control_rate(torch.from_numpy(x).to(dev()), torch.from_numpy(lo).to(dev()), *[to_t(p) for p in params],
                           example_index=idx, out=out)
    got = out.cpu().numpy()
    for b in range(B):
        if b in (0, 3, 4, 8):
            assert np.array_equal(got[b], ref[b])
        else:
            assert (got[b] == 7.0).all()


# (max_min_delay_ms, max_lfo_delay_ms, lowest min_delay_width) of the fused-LFO tests: the flanger, and the chorus with
# min_delay_width in [0, 1] -- a synthesised LFO never takes fc_wide_kernel, so chorus-length lines go through
# fc_cta_kernel in each of its in-kernel LFO modes
_FUSED_LFO_LINES = [(1.0, 10.0, 0.0), (30.0, 10.0, 0.0)]


def test_flanger_fused_lfo_synthesis():
    """LFO params in, audio out: the LFO itself is within 1e-6 of the reference arithmetic
    (cos is not bit-identical across libms), so the audio is compared per shape family:
    bit-exact for the cos-free shapes, SNR-bounded for the cos shapes (SURVEY F3)."""
    for line in _FUSED_LFO_LINES:
        _check_fused_lfo(882, 441.0, *line)     # the control row of the reference pipeline, staged in shared memory


def test_flanger_fused_lfo_long_row():
    """Same comparison for a synthesised control row longer than the kernel stages: evaluated at the taps."""
    for line in _FUSED_LFO_LINES:
        _check_fused_lfo(8820, 4410.0, *line)


def test_flanger_fused_lfo_direct():
    """Same comparison with one LFO value per sample (n_lo = N): no upsample."""
    for line in _FUSED_LFO_LINES:
        _check_fused_lfo(88200, float(SR), *line)


def _check_fused_lfo(n_lo, sr_lo, mmd, mld, mdw_lo):
    from mod_extraction_b200.fx import MonoFlangerChorusModule
    from mod_extraction_b200.modulations import SHAPE_ID
    rng = np.random.RandomState(23)
    B, N = 12, 88200
    x = guitar(B, N, 2)
    shapes = [["tri", "saw", "rsaw", "cos", "rect_cos", "inv_rect_cos"][b % 6] for b in range(B)]
    rate = np.exp(rng.uniform(np.log(0.5), np.log(3.0), B))
    phase = rng.uniform(0, 2 * math.pi, B)
    lo = np.stack([oracle.make_mod_signal(n_lo, sr_lo, rate[b], phase[b], shapes[b], 2.0) for b in range(B)])
    params = _rand_params(B, rng, mdw_lo)
    ref = oracle.flanger_chorus(x, oracle.linear_interpolate_last_dim(lo, N), *params, max_min_delay_ms=mmd,
                                max_lfo_delay_ms=mld)
    m = MonoFlangerChorusModule(B, 1, N, SR, mmd, mld)
    y = m.forward_lfo(torch.from_numpy(x).to(dev()), torch.from_numpy(rate), torch.from_numpy(phase),
                      torch.tensor([SHAPE_ID[s] for s in shapes]), exp=torch.full((B,), 2.0), n_lo=n_lo, sr_lo=sr_lo,
                      feedback=to_t(params[0]), min_delay_width=to_t(params[1]), width=to_t(params[2]),
                      depth=to_t(params[3]), mix=to_t(params[4])).cpu().numpy()
    for b in range(B):
        if shapes[b] in ("tri", "saw", "rsaw"):
            assert np.array_equal(y[b], ref[b]), (mmd, shapes[b])
        else:
            assert np.abs(y[b] - ref[b]).max() <= 1e-4 and snr_db(ref[b], y[b]) >= 80.0, (mmd, shapes[b])


# --------------------------------------------------------------------------- E2, L1, L2, U1

def test_tremolo_bit_exact():
    from mod_extraction_b200.fx import apply_tremolo
    g = golden("tremolo")
    for i in range(2):
        y = apply_tremolo(torch.from_numpy(g["x"]).to(dev()), torch.from_numpy(g["mod"]).to(dev()), float(g[f"mix{i}"]))
        assert np.array_equal(y.cpu().numpy(), g[f"y{i}"])
    mix = np.array([0.1, 0.5, 1.0], dtype=np.float32)
    ref = oracle.tremolo(g["x"], g["mod"], mix)
    y = apply_tremolo(torch.from_numpy(g["x"]).to(dev()), torch.from_numpy(g["mod"]).to(dev()), to_t(mix))
    assert np.array_equal(y.cpu().numpy(), ref)


def test_lfo_vs_reference_goldens():
    from mod_extraction_b200.modulations import make_mod_signal
    g = golden("lfo")
    for i, c in enumerate(g["cases"]):
        n, sr, f, ph, sid, e = c
        out = make_mod_signal(int(n), sr, f, ph, oracle.SHAPES[int(sid)], e)
        assert out.is_cuda and out.shape == (int(n),)
        tol = 1e-6 if e >= 1.0 else 5e-5            # north_star: LFO within 1e-6 (see DESIGN.md for exp<1)
        assert np.abs(out.cpu().numpy() - g[f"out{i}"]).max() <= tol, (i, c)


def test_lfo_cos_free_shapes_bit_exact_vs_oracle():
    from mod_extraction_b200.modulations import make_mod_signal_batch
    rng = np.random.RandomState(4)
    B = 64
    shapes = [["tri", "saw", "rsaw"][b % 3] for b in range(B)]
    f = np.exp(rng.uniform(np.log(0.5), np.log(3.0), B))
    ph = rng.uniform(-2 * math.pi, 2 * math.pi, B)
    for n, sr in [(882, 441.0), (26460, 441.0), (176400, 44100.0)]:
        out = make_mod_signal_batch(n, sr, f, ph, shapes, np.full(B, 2.0)).cpu().numpy()
        for b in range(0, B, 7):
            ref = oracle.make_mod_signal(n, sr, f[b], ph[b], shapes[b], 2.0)
            assert np.array_equal(out[b], ref), (n, b)


def test_lfo_all_shapes_within_tolerance_long():
    """60 s at control rate and the 4 s audio-rate phaser ground truth (datasets.py:442)."""
    from mod_extraction_b200.modulations import make_mod_signal_batch
    rng = np.random.RandomState(5)
    shapes = oracle.SHAPES
    B = len(shapes)
    f = np.exp(rng.uniform(np.log(0.5), np.log(3.0), B))
    ph = rng.uniform(0, 2 * math.pi, B)
    for n, sr in [(26460, 441.0), (176400, 44100.0)]:
        out = make_mod_signal_batch(n, sr, f, ph, shapes).cpu().numpy()
        for b in range(B):
            ref = oracle.make_mod_signal(n, sr, f[b], ph[b], shapes[b])
            err = np.abs(out[b] - ref)
            if shapes[b] == "sqr":      # a sign flip at a zero crossing is a whole step: count, don't bound
                assert (err > 1e-6).sum() <= 2
            else:
                assert err.max() <= 1e-6, (shapes[b], n)


def test_make_rand_mod_signal_same_draws_as_reference_order():
    from mod_extraction_b200.modulations import make_rand_mod_signal
    torch.manual_seed(123)
    out = make_rand_mod_signal(5, 345, 172.5, 0.5, 3.0).cpu().numpy()
    torch.manual_seed(123)
    shapes = ["cos", "tri", "rect_cos", "inv_rect_cos", "saw", "rsaw"]
    for b in range(5):          # modulations.py:74-99: phase, freq, shape per example
        ph = (torch.rand(1) * (2 * math.pi - 0.0) + 0.0).item()
        f = (torch.rand(1) * (3.0 - 0.5) + 0.5).item()
        s = shapes[torch.randint(0, 6, (1,)).item()]
        ref = oracle.make_mod_signal(345, 172.5, f, ph, s)
        assert np.abs(out[b] - ref).max() <= 1e-6


def test_random_lfo_baseline_model_wrapper():
    """models.RandomLFO (models.py:19-69, baseline_rand_lfo.yml: 345 frames at 172.5 Hz): same draws as a direct call."""
    from mod_extraction_b200.models import RandomLFO
    from mod_extraction_b200.modulations import make_rand_mod_signal
    m = RandomLFO(n_samples=345, sr=172.5)
    torch.manual_seed(7)
    a = m(6)
    torch.manual_seed(7)
    b = make_rand_mod_signal(6, 345, 172.5, 0.5, 3.0, None, None, None, 0.0, None, 0.0)
    assert a.shape == (6, 1, 345) and torch.equal(a.squeeze(1), b)
    g = RandomLFO(n_samples=345, sr=172.5, use_freq_gt=True, use_phase_gt=True, use_shape_gt=True)
    with pytest.raises(AssertionError):
        g(2)                                                      # models.py:49: ground truth requested, none given
    out = g(2, {"shape": ["tri", "cos"], "phase": torch.tensor([0.0, 1.0]), "rate_hz": torch.tensor([2.0, 1.0])})
    ref = oracle.make_mod_signal(345, 172.5, 2.0, 0.0, "tri")
    assert np.abs(out[0, 0].cpu().numpy() - ref).max() <= 1e-6


def test_interp_bit_exact_vs_reference_goldens():
    from mod_extraction_b200.util import linear_interpolate_last_dim
    g = golden("interp")
    for i in range(int(g["n"])):
        rows, I, O, ac = g[f"cfg{i}"]
        y = linear_interpolate_last_dim(torch.from_numpy(g[f"x{i}"]).to(dev()), int(O), bool(ac))
        assert np.array_equal(y.cpu().numpy(), g[f"y{i}"]), i
    x = torch.rand(4, 3, 100, device=dev())
    assert linear_interpolate_last_dim(x, 100) is x            # util.py:18-19
    y = linear_interpolate_last_dim(x, 1234)
    ref = oracle.linear_interpolate_last_dim(x.cpu().numpy(), 1234)
    assert np.array_equal(y.cpu().numpy(), ref)
    y1 = linear_interpolate_last_dim(x[0, 0], 77)
    assert y1.shape == (77,)


# --------------------------------------------------------------------------- BASELINE-size properties

def test_full_size_properties_config3():
    """B=1024 x 88200 (BASELINE config 3): size-independent properties + sampled oracle check."""
    from mod_extraction_b200.fx import MonoFlangerChorusModule
    rng = np.random.RandomState(44)
    B, N = 1024, 88200
    g = torch.Generator(device="cpu").manual_seed(44)
    x = ((torch.rand((B, 1, N), generator=g) * 2 - 1) * 0.5)
    lo = torch.from_numpy(_lfo_lo(B, rng, exp=2.0))
    params = _rand_params(B, rng, 0.0)
    xd, lod = x.to(dev()), lo.to(dev())
    tp = [to_t(p) for p in params]
    fl = MonoFlangerChorusModule(B, 1, N, SR, 1.0, 10.0)
    y = fl.forward_control_rate(xd, lod, *tp)
    assert float(y.abs().max()) <= 1.0                                  # clip, fx.py:118
    # (1) determinism / idempotence of the schedule: a second run gives the same bits
    assert torch.equal(y, fl.forward_control_rate(xd, lod, *tp))
    # (2) mix = 0 returns the dry signal exactly: (1-0)*x + 0*o
    y0 = fl.forward_control_rate(xd, lod, tp[0], tp[1], tp[2], tp[3], 0.0)
    assert torch.equal(y0, xd.clamp(-1, 1))
    # (3) batch independence: rendering a subset equals the rows of the full render
    sub = torch.arange(0, B, 97)
    fs = MonoFlangerChorusModule(len(sub), 1, N, SR, 1.0, 10.0)
    ys = fs.forward_control_rate(xd[sub.to(dev())], lod[sub.to(dev())], *[p[sub.to(dev())] for p in tp])
    assert torch.equal(ys, y[sub.to(dev())])
    # (4) sampled rows against the oracle, bit-exact
    rows = [0, 511, 1023]
    ref = oracle.flanger_chorus(x[rows].numpy(), oracle.linear_interpolate_last_dim(lo[rows].numpy(), N),
                                *[p[rows] for p in params], max_min_delay_ms=1.0, max_lfo_delay_ms=10.0)
    assert np.array_equal(y[rows].cpu().numpy(), ref)


def test_torch_ops_dispatch_on_cuda():
    import mod_extraction_b200._torch_ops  # noqa: F401
    x = torch.rand(3, 50, device=dev())
    y = torch.ops.modfx.interp_linear(x, 120, True)
    assert np.array_equal(y.cpu().numpy(), oracle.linear_interpolate_last_dim(x.cpu().numpy(), 120))


def test_torch_ops_of_the_whole_path_dispatch_on_cuda():
    """SURVEY 8b: every op of the path is reachable as torch.ops.modfx.* (CUDA key only)."""
    import mod_extraction_b200._torch_ops  # noqa: F401
    from mod_extraction_b200.models import LogMelSpectrogram
    d = dev()
    x = torch.from_numpy(white((2, 1, 4096), 9)).to(d)
    mod = torch.rand(2, 4096, device=d)
    y = torch.ops.modfx.tremolo(x, mod, torch.tensor([0.3, 0.9], device=d))
    assert np.array_equal(y.cpu().numpy(), oracle.tremolo(x.cpu().numpy(), mod.cpu().numpy(), np.array([0.3, 0.9], np.float32)))
    m = LogMelSpectrogram().to(d)
    lm = torch.ops.modfx.logmel(x, m.window, m.fb_start, m.fb_count, m.fb_weight, m.fb_taps, 256, 1e-7)
    assert torch.equal(lm, m(x))
    mp = torch.ops.modfx.mel_power(x, m.window, m.fb_start, m.fb_count, m.fb_weight, m.fb_taps, 256, 1e-7)
    assert float((torch.log(torch.clip(mp, min=1e-7)) - lm).abs().max()) <= 1e-5
    sig = torch.from_numpy(np.stack([oracle.make_mod_signal(345, 172.5, 1.3, 0.4, "tri"),
                                     oracle.make_mod_signal(345, 172.5, 2.1, 1.0, "cos")])).to(d)
    top, bottom = torch.ops.modfx.find_corners(sig)
    rt, rb = oracle.find_corners(sig.cpu().numpy())
    assert np.array_equal(top.cpu().numpy(), rt) and np.array_equal(bottom.cpu().numpy(), rb)
    sm = torch.ops.modfx.smoothen(sig, 8)
    assert np.array_equal(sm.cpu().numpy(), oracle.smoothen(sig.cpu().numpy(), 8))
    st = torch.ops.modfx.stretch_corners(sm, 10)
    assert st.shape == sm.shape and torch.isfinite(st).all()
    valid = torch.ops.modfx.check_mod_sig(sig, 1, 6, 1, 6, 34)
    assert valid.shape == (2,)


@pytest.mark.parametrize("mmd,mld", [(1.0, 10.0), (30.0, 10.0)])
def test_allpass_interpolation_mode_matches_own_restatement(mmd, mld):
    """north_star names "linear or all-pass" interpolation; the reference only has linear (SURVEY F2), so this mode is
    checked against this repository's OWN restatements: bit-exact against the float32 one (same operation order), and
    against the float64 python loop on a short clip within 1e-4 on >= 99 % of the samples with an SNR >= 40 dB (where
    the delay passes an integer number of samples, float32 and float64 index arithmetic pick different taps for a
    sample -- the same input sensitivity as SURVEY F3 -- and the interpolator's state carries the difference on)."""
    from tests.helpers import snr_db
    from mod_extraction_b200.fx import MonoFlangerChorusModule
    rng = np.random.RandomState(17)
    B, C, N = 5, 2, 6000
    x = white((B, C, N), 18) * np.float32(0.4)
    lo = _lfo_lo(B, rng, n_lo=N // 100, sr_lo=441.0)
    params = _rand_params(B, rng)
    mod = oracle.linear_interpolate_last_dim(lo, N)
    ref = oracle.flanger_chorus(x, mod, *params, max_min_delay_ms=mmd, max_lfo_delay_ms=mld, interpolation="allpass")
    m = MonoFlangerChorusModule(B, C, N, SR, mmd, mld, interpolation="allpass")
    xd = torch.from_numpy(x).to(dev())
    y_audio = m(xd, torch.from_numpy(mod).to(dev()), *[to_t(p) for p in params]).cpu().numpy()
    y_ctrl = m.forward_control_rate(xd, torch.from_numpy(lo).to(dev()), *[to_t(p) for p in params]).cpu().numpy()
    assert np.array_equal(y_audio, ref) and np.array_equal(y_ctrl, ref)
    f64 = oracle.flanger_chorus_allpass_f64(x[0, 0, :3000], mod[0, :3000], *[float(p[0]) for p in params],
                                            max_min_delay_ms=mmd, max_lfo_delay_ms=mld)
    e64 = np.abs(y_audio[0, 0, :3000] - f64)
    assert (e64 <= 1e-4).mean() >= 0.99 and snr_db(f64, y_audio[0, 0, :3000]) >= 40.0, (e64.max(), (e64 <= 1e-4).mean())
    # it is a different interpolator, not a different effect: close to the linear rendering, not equal to it
    lin = oracle.flanger_chorus(x, mod, *params, max_min_delay_ms=mmd, max_lfo_delay_ms=mld)
    assert not np.array_equal(lin, ref) and np.corrcoef(lin.ravel(), ref.ravel())[0, 1] > 0.9
    # subsets and many lines (more than one CTA of 32 delay lines)
    B2 = 40
    x2 = white((B2, 1, 2000), 19)
    mod2 = rng.uniform(0, 1, (B2, 2000)).astype(np.float32)
    p2 = _rand_params(B2, rng)
    ref2 = oracle.flanger_chorus(x2, mod2, *p2, max_min_delay_ms=mmd, max_lfo_delay_ms=mld, interpolation="allpass")
    m2 = MonoFlangerChorusModule(B2, 1, 2000, SR, mmd, mld, interpolation="allpass")
    y2 = m2(torch.from_numpy(x2).to(dev()), torch.from_numpy(mod2).to(dev()), *[to_t(p) for p in p2]).cpu().numpy()
    assert np.array_equal(y2, ref2)
