"""Flanger / chorus delay lines at the edges of their schedules, bit for bit against the CPU oracle.

modfx_flanger_chorus_f32 (csrc/fc.cu) renders a control-rate example in one of two kernels: fc_wide_kernel takes it when
its shortest delay is at least a wide tile plus a margin, fc_cta_kernel takes everything else.  Both kernels evaluate the
same predicate, and each must render exactly the rows the other skips.  These tests cover:
  * that split, with rows on both sides of it;
  * chorus-length lines in every modulation source and at other sample rates;
  * the longest lines shared memory holds, and the refusal one sample past them (also for the all-pass kernel, at each
    of its lines-per-CTA steps);
  * lines of a few samples.

Every output is compared with oracle.flanger_chorus (which test_oracle_cpu.py pins bitwise to the reference's goldens)
with np.array_equal.  Outputs are rendered into an `out` filled with NaN: a row the kernels should have written but did
not stays NaN, and a row left out of example_index must still be NaN afterwards.
"""
import math

import numpy as np
import pytest
import torch

from oracle import oracle
from tests.helpers import SR, white

pytestmark = pytest.mark.gpu

F32 = np.float32

# ---- limits, as fc.cu derives them.  The refusal tests pin the observable ones, so moving a constant in fc.cu fails
# ---- here instead of quietly testing another boundary.
# fc_wide_kernel renders 3 samples per thread of a 128-thread CTA per tile; it takes a row iff
# A * min(mod_lo) + D0 >= kWideTile + kWideMargin.
WIDE_TILE = 128 * 3                                 # kWideTile = 384
WIDE_MIN_DELAY = WIDE_TILE + 4                      # kWideTile + kWideMargin = 388
SMEM_FLOATS = 200 * 1024 // 4                       # dynamic shared memory either launcher allows itself, in floats
# fc_wide_kernel's ring is next_pow2(M + kWideTile) floats: <= SMEM_FLOATS -> <= 32768 -> M <= 32768 - 384.
# Longer lines skip the wide kernel, and fc_cta_kernel must render their wide-eligible rows too.
WIDE_MAX_M = 32768 - WIDE_TILE                      # 32384
# fc_cta_kernel: 16 + kNT * kSlotFloats (6 * 648) + kCtaProd * kXDepth * kTile (3 * 4 * 128; twice that with an
# audio-rate mod) + a staged LFO row (<= 2048) + a ring of next_pow2(M + kTile) floats must stay <= SMEM_FLOATS: at most
# 7 024 + ring, so the ring can be 32768 floats but not 65536 -> M <= 32768 - 128.  Longer lines are refused.
CTA_MAX_M = 32768 - 128                             # 32640
# fc_allpass_kernel: L lines per one-warp CTA, L halved from 32 while next_pow2(M + 1) * L > 160 KiB / 4; at L = 1 it
# needs next_pow2(M + 1) + 2 * 32 * 33 <= SMEM_FLOATS floats -> next_pow2(M + 1) <= 32768 -> M <= 32767.
ALLPASS_MAX_M = 32768 - 1                           # 32767; refused at 32768


def _next_pow2(v):
    p = 1
    while p < v:
        p <<= 1
    return p


def _allpass_lines_per_cta(M):
    ring, L = _next_pow2(M + 1), 32
    while L > 1 and ring * L > 160 * 1024 // 4:
        L //= 2
    return L


def dev():
    return torch.device("cuda", 0)


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev())


def _module(B, C, N, Mmin, Mlfo, sr=SR, interpolation="linear"):
    """A module whose delay line is exactly Mmin + Mlfo samples (fx.py:40-41 rounds ms * sr / 1000 to the nearest)."""
    from mod_extraction_b200.fx import MonoFlangerChorusModule
    mmd, mld = Mmin * 1000.0 / sr, Mlfo * 1000.0 / sr
    m = MonoFlangerChorusModule(B, C, N, sr, mmd, mld, interpolation=interpolation)
    assert (m.max_min_delay_samples, m.max_lfo_delay_samples) == (Mmin, Mlfo)
    assert oracle.delay_samples(sr, mmd, mld) == (Mmin, Mlfo)
    return m


def _oracle(m, x, mod, params):
    return oracle.flanger_chorus(x, mod, *params, sr=m.sr, max_min_delay_ms=m.max_min_delay_ms,
                                 max_lfo_delay_ms=m.max_lfo_delay_ms, interpolation=m.interpolation)


def _render(m, x, src, params, idx=None):
    """The module's render call into a NaN-filled out; returns it on the host."""
    from mod_extraction_b200 import _ops
    out = torch.full(tuple(x.shape), float("nan"), device=dev())
    y = _ops.flanger_chorus(_t(x), src, m.max_min_delay_samples, m.max_lfo_delay_samples,
                            *[_t(p) if isinstance(p, np.ndarray) else p for p in params],
                            example_index=None if idx is None else torch.tensor(idx, dtype=torch.int32),
                            out=out, interpolation=m.interpolation)
    assert y.data_ptr() == out.data_ptr()
    return out.cpu().numpy()


def _assert_rows(got, ref, rows=None, what=""):
    """Rows `rows` (all by default) equal the oracle bit for bit; every other row is still all NaN."""
    rows = range(got.shape[0]) if rows is None else rows
    for b in range(got.shape[0]):
        if b in rows:
            assert np.array_equal(got[b], ref[b]), (what, "row", b, "samples off", int((got[b] != ref[b]).sum()),
                                                    "of which NaN", int(np.isnan(got[b]).sum()))
        else:
            assert np.isnan(got[b]).all(), (what, "row", b, "written but not in example_index")


def _audio(mod):
    from mod_extraction_b200._ops import ModSource
    return ModSource.audio_rate(_t(mod))


def _control(lo):
    from mod_extraction_b200._ops import ModSource
    return ModSource.control_rate(_t(lo))


def _lfo(n_lo, sr_lo, rate, phase, shapes, exp):
    from mod_extraction_b200._ops import ModSource
    from mod_extraction_b200.modulations import lfo_kernel_params
    return ModSource.lfo(n_lo, sr_lo, *lfo_kernel_params(rate, phase, shapes, exp, sr_lo, dev()))


def _lfo_rows(n_lo, sr_lo, rate, phase, shapes, exp):
    return np.stack([oracle.make_mod_signal(n_lo, sr_lo, rate[b], phase[b], shapes[b], exp[b])
                     for b in range(len(shapes))])


# --------------------------------------------------------------------------- 1. the wide / CTA split

CHORUS = (1323, 441)                # 30 ms / 10 ms at 44.1 kHz
N_SPLIT = 88200


def _mdw_for(d0, mmin, exact=True):
    """The float32 min_delay_width whose product with mmin, rounded once to float32 as make_coef does, is nearest to d0
    (`exact`: and equal to it)."""
    lo = hi = F32(float(d0) / mmin)
    cands = [lo]
    for _ in range(64):
        lo, hi = np.nextafter(lo, F32(0)), np.nextafter(hi, F32(2))
        cands += [lo, hi]
    best = min(cands, key=lambda c: abs(float(F32(c * F32(mmin))) - float(d0)))
    assert not exact or F32(best * F32(mmin)) == F32(d0), f"no float32 min_delay_width gives D0 = {d0!r}"
    return best


def _d_min(A, D0, m_min):
    return F32(F32(A * F32(m_min)) + D0)                # wide_pred: the delay at the row's minimum


def _crossing(A, D0):
    """Consecutive float32 row minima m_lo < m_hi with A * m_lo + D0 < 388 <= A * m_hi + D0 in float32."""
    edge = F32(WIDE_MIN_DELAY)
    m = F32((float(edge) - float(D0)) / float(A))
    while _d_min(A, D0, m) >= edge:
        m = np.nextafter(m, F32(-1))
    while _d_min(A, D0, np.nextafter(m, F32(2))) < edge:
        m = np.nextafter(m, F32(2))
    return m, np.nextafter(m, F32(2))


def _coef(mdw, width, Mmin, Mlfo):
    """make_coef's A = Mlfo * width and D0 = min_delay_width * Mmin for per-example (float32 array) parameters."""
    return F32(F32(Mlfo) * F32(width)), F32(F32(mdw) * F32(Mmin))


def _is_wide(A, D0, m_min, m_max, M):
    """wide_pred of fc.cu, in float32."""
    coef_ok = A >= 0 and D0 >= 0 and F32(A + D0) <= F32(M)
    return bool(coef_ok and m_min >= 0 and m_max <= 1 and _d_min(A, D0, m_min) >= WIDE_MIN_DELAY)


def _valley(n_lo, pos, lo, hi):
    """A control row with its one minimum `lo` at `pos` and its maximum `hi` at the far end.  Near the minimum the row is
    flat to ~1e-4 for a few control points (hundreds of samples at N = 88 200): there the delay stays at its minimum over
    more than a wide tile, so a row rendered by the wide kernel with its taps inside the tile cannot go unnoticed."""
    k = np.abs(np.arange(n_lo) - pos) / max(pos, n_lo - 1 - pos)
    row = (float(lo) + (float(hi) - float(lo)) * 0.5 * (1.0 - np.cos(np.pi * k))).astype(F32)
    assert row[pos] == F32(lo) and (row == F32(lo)).sum() == 1 and row.min() == F32(lo) and row.max() == F32(hi)
    return row


def _split_rows():
    """(min_delay_width, width, row minimum, row maximum) of each example."""
    below, above = np.nextafter(F32(388), F32(0)), np.nextafter(F32(388), F32(1000))
    rows = []
    # D0 = fl32(mdw) * 1323 on each side of 388, at row minimum 0: d_min = D0.  (No float32 mdw gives D0 = 388 itself --
    # the products step by 3.9e-5 there, the float32 grid by 3.05e-5 -- so test_wide_split_at_exactly_388 takes it.  Nor
    # 485, the reference chorus' shortest delay: that row takes the nearest product, 2e-5 away.)
    for i, d0 in enumerate((380, 384, 385, 386, 387, below, above, 392, 485)):
        rows.append((_mdw_for(d0, CHORUS[0], exact=d0 != 485), (0.6, 0.3, 1.0)[i % 3], 0.0, 0.9))
    # D0 < 388 with the row minimum lifting d_min across 388, both sides (width 1: A = 441)
    for mdw in (F32(0.2267574), F32(0.0)):
        m_lo, m_hi = _crossing(F32(441), F32(mdw * F32(CHORUS[0])))
        rows += [(mdw, 1.0, m_lo, 1.0), (mdw, 1.0, m_hi, 1.0)]
    rows += [(_mdw_for(384, CHORUS[0]), 0.0, 0.0, 0.9),         # width 0: the delay is D0 everywhere
             (_mdw_for(below, CHORUS[0]), 0.0, 0.0, 0.9),
             (_mdw_for(above, CHORUS[0]), 0.0, 0.0, 0.9),
             (_mdw_for(485, CHORUS[0], exact=False), 0.8, 0.0, 1.0),     # row maximum exactly 1
             (F32(1.0), 1.0, 0.0, 1.0)]                          # mdw = 1: A + D0 = M
    return rows


def _effect_params(B, rng):
    """feedback, depth, mix: feedback >= 0.3 so that a wrong sample also reaches later ones."""
    return rng.uniform(0.3, 0.69, B).astype(F32), rng.uniform(0.5, 1.0, B).astype(F32), rng.uniform(0.5, 1.0, B).astype(F32)


SPLIT_N_LO = [129, 882, 883]


def _split_case(n_lo, C, rows, seed):
    B = len(rows)
    rng = np.random.RandomState(seed)
    x = white((B, C, N_SPLIT), seed)
    mid = n_lo // 2 + 7
    # each row's minimum at index 0, the last index or mid-row, rotating with n_lo: the strided min/max reductions of
    # both kernels (thread i % 128 reads index i) must find it wherever it sits
    shift = SPLIT_N_LO.index(n_lo)
    positions = [(0, n_lo - 1, mid)[(b + shift) % 3] for b in range(B)]
    lo = np.stack([_valley(n_lo, positions[b], rows[b][2], rows[b][3]) for b in range(B)])
    fb, depth, mix = _effect_params(B, rng)
    return x, lo, fb, depth, mix


@pytest.mark.parametrize("C", [1, 2])
@pytest.mark.parametrize("n_lo", SPLIT_N_LO)
def test_wide_split_chorus_rows(n_lo, C):
    """Control-rate chorus rows whose shortest delay lies on either side of 388 samples, rendered all at once and as an
    example_index subset that interleaves rows of the two kernels."""
    rows = _split_rows()
    B = len(rows)
    x, lo, fb, depth, mix = _split_case(n_lo, C, rows, seed=n_lo + C)
    mdw = np.array([r[0] for r in rows], dtype=F32)
    width = np.array([r[1] for r in rows], dtype=F32)
    wide = [_is_wide(*_coef(mdw[b], width[b], *CHORUS), lo[b].min(), lo[b].max(), sum(CHORUS)) for b in range(B)]
    assert wide == [False] * 6 + [True] * 3 + [False, True, False, True] + [False, False, True, True, True]
    params = [fb, mdw, width, depth, mix]
    m = _module(B, C, N_SPLIT, *CHORUS)
    ref = _oracle(m, x, oracle.linear_interpolate_last_dim(lo, N_SPLIT), params)
    _assert_rows(_render(m, x, _control(lo), params), ref)
    w_rows = [b for b in range(B) if wide[b]]
    c_rows = [b for b in range(B) if not wide[b]]
    idx = [r for pair in zip(w_rows[::-2], c_rows[::2]) for r in pair]      # wide, CTA, wide, ... out of order
    _assert_rows(_render(m, x, _control(lo), params, idx), ref, idx)


@pytest.mark.parametrize("n_lo", [129, 883])
def test_wide_split_at_exactly_388(n_lo):
    """D0 = 388 exactly, through a scalar min_delay_width (rounded once from double), at row minimum 0: every row goes
    to the wide kernel with its shortest delay on the predicate's edge; width 0 keeps it there for the whole clip."""
    Mmin, Mlfo = CHORUS
    mdw = WIDE_MIN_DELAY / Mmin
    D0 = F32(mdw * Mmin)
    assert D0 == F32(WIDE_MIN_DELAY)
    widths = [0.0, 0.25, 1.0, 0.0, 0.5, 1.0]
    rows = [(mdw, w, 0.0, 0.9) for w in widths]
    B, C = len(rows), 2
    x, lo, fb, depth, mix = _split_case(n_lo, C, rows, seed=7 * n_lo)
    assert all(_is_wide(F32(F32(Mlfo) * F32(w)), D0, lo[b].min(), lo[b].max(), Mmin + Mlfo) for b, w in enumerate(widths))
    params = [fb, mdw, np.array(widths, dtype=F32), depth, mix]
    m = _module(B, C, N_SPLIT, Mmin, Mlfo)
    ref = _oracle(m, x, oracle.linear_interpolate_last_dim(lo, N_SPLIT), params)
    _assert_rows(_render(m, x, _control(lo), params), ref)
    _assert_rows(_render(m, x, _control(lo), params, [4, 0, 3]), ref, [4, 0, 3])


# --------------------------------------------------------------------------- 2. chorus-length lines at other sample rates

def _lfo_params(B, rng, shapes=("cos", "tri", "rect_cos", "inv_rect_cos", "saw", "rsaw")):
    rate = np.exp(rng.uniform(np.log(0.5), np.log(3.0), B))
    phase = rng.uniform(0, 2 * math.pi, B)
    return rate, phase, [shapes[b % len(shapes)] for b in range(B)]


def _rand_params(B, rng, fb_hi=0.69):
    """feedback, min_delay_width in [0, 1], width, depth, mix."""
    U = lambda lo, hi: rng.uniform(lo, hi, B).astype(F32)
    return [U(0.0, fb_hi), U(0.0, 1.0), U(0.25, 1.0), U(0.25, 1.0), U(0.25, 1.0)]


@pytest.mark.parametrize("sr", [48000, 96000, 192000])
def test_chorus_and_flanger_at_other_sample_rates(sr):
    """2 s at 48, 96 and 192 kHz: delay lines of (sr / 1000 + sr / 100) and (30 sr / 1000 + sr / 100) samples -- at
    192 kHz the chorus is 7680 samples in an 8192-float ring -- with min_delay_width in [0, 1], so that control-rate
    chorus rows go to both kernels."""
    rng = np.random.RandomState(sr // 1000)
    B, C, N = 6, 2, 2 * sr
    x = white((B, C, N), sr // 1000)
    rate, phase, shapes = _lfo_params(B, rng)
    lo = _lfo_rows(N // 100, sr / 100.0, rate, phase, shapes, [1.0] * B)
    mod = oracle.linear_interpolate_last_dim(lo, N)
    for mmin, mlfo in ((sr // 1000, sr // 100), (30 * sr // 1000, sr // 100)):
        params = _rand_params(B, rng)
        params[1][0], params[1][1] = 0.0, 1.0
        m = _module(B, C, N, mmin, mlfo, sr=sr)
        ref = _oracle(m, x, mod, params)
        _assert_rows(_render(m, x, _audio(mod), params), ref, what=(mmin, mlfo, "audio rate"))
        _assert_rows(_render(m, x, _control(lo), params), ref, what=(mmin, mlfo, "control rate"))


# --------------------------------------------------------------------------- 3. the longest lines

LONG_MLFO = 441
COS_FREE = ("tri", "saw", "rsaw")       # LFO shapes the kernels synthesise bit for bit like the oracle


def _long_case(M):
    B, N = 4, 3 * M + 77                # the ring wraps; N is not a multiple of 128 or 384
    rng = np.random.RandomState(M)
    x = white((B, 1, N), M)
    rate, phase, shapes = _lfo_params(B, rng, COS_FREE)
    exp = [2.0, 1.0, 2.0, 1.0]
    params = _rand_params(B, rng)
    params[1][:] = [0.0, 0.006, 0.4, 1.0]   # D0 from 0 to M - 441: rows on both sides of the wide split
    return x, rate, phase, shapes, exp, params


def _long_sources(N,rate, phase, shapes, exp):
    """(name, source, audio-rate modulation the oracle sees) for every modulation source of fc_cta_kernel."""
    out = []
    lo = _lfo_rows(N // 100, 441.0, rate, phase, shapes, exp)
    mod = oracle.linear_interpolate_last_dim(lo, N)
    out.append(("control-rate read", _control(lo), mod))
    out.append(("audio-rate", _audio(mod), mod))
    assert N // 100 <= 2048
    out.append(("staged LFO", _lfo(N // 100, 441.0, rate, phase, shapes, exp), mod))
    assert N // 10 > 2048
    lo10 = _lfo_rows(N // 10, 4410.0, rate, phase, shapes, exp)
    out.append(("at-tap LFO", _lfo(N // 10, 4410.0, rate, phase, shapes, exp),
                oracle.linear_interpolate_last_dim(lo10, N)))
    out.append(("direct LFO", _lfo(N, float(SR), rate, phase, shapes, exp),
                _lfo_rows(N, float(SR), rate, phase, shapes, exp)))
    return out, lo


@pytest.mark.parametrize("M", [WIDE_MAX_M, WIDE_MAX_M + 1, CTA_MAX_M])
def test_longest_lines_every_source(M):
    """The longest line the wide kernel holds, one sample longer (the wide kernel is skipped: fc_cta_kernel renders the
    wide-eligible rows too), and the longest line fc_cta_kernel holds, in every modulation source."""
    x, rate, phase, shapes, exp, params = _long_case(M)
    B, _, N = x.shape
    m = _module(B, 1, N, M - LONG_MLFO, LONG_MLFO)
    sources, lo = _long_sources(N,rate, phase, shapes, exp)
    wide = [_is_wide(*_coef(params[1][b], params[2][b], M - LONG_MLFO, LONG_MLFO), lo[b].min(), lo[b].max(), M)
            for b in range(B)]
    assert wide == [False, False, True, True]
    for name, src, mod in sources:
        _assert_rows(_render(m, x, src, params), _oracle(m, x, mod, params), what=name)


def test_line_past_shared_memory_is_refused():
    """One sample past CTA_MAX_M the ring needs 65536 floats: every source is refused before anything is written."""
    M = CTA_MAX_M + 1
    x, rate, phase, shapes, exp, params = _long_case(M)
    B, _, N = x.shape
    m = _module(B, 1, N, M - LONG_MLFO, LONG_MLFO)
    sources, _ = _long_sources(N,rate, phase, shapes, exp)
    from mod_extraction_b200 import _ops
    for name, src, _ in sources:
        out = torch.full((B, 1, N), float("nan"), device=dev())
        with pytest.raises(RuntimeError, match="shared memory"):
            _ops.flanger_chorus(_t(x), src, M - LONG_MLFO, LONG_MLFO, *[_t(p) for p in params], out=out)
        assert torch.isnan(out).all(), name


@pytest.mark.parametrize("M", [1023, 1024, 4095, 8191, 16383, ALLPASS_MAX_M])
def test_allpass_lines_per_cta(M):
    """The all-pass kernel at each lines-per-CTA step L = 32 .. 1, with L + 3 lines: several CTAs, the last one partial."""
    L = _allpass_lines_per_cta(M)
    assert L == {1023: 32, 1024: 16, 4095: 8, 8191: 4, 16383: 2, ALLPASS_MAX_M: 1}[M]
    B, N = L + 3, 3 * M + 77
    rng = np.random.RandomState(M)
    x = white((B, 1, N), M)
    rate, phase, shapes = _lfo_params(B, rng)
    lo = _lfo_rows(N // 100, 441.0, rate, phase, shapes, [1.0] * B)
    mod = oracle.linear_interpolate_last_dim(lo, N)
    params = _rand_params(B, rng)
    m = _module(B, 1, N, M - LONG_MLFO, LONG_MLFO, interpolation="allpass")
    ref = _oracle(m, x, mod, params)
    _assert_rows(_render(m, x, _audio(mod), params), ref, what="audio rate")
    _assert_rows(_render(m, x, _control(lo), params), ref, what="control rate")


def test_allpass_line_past_shared_memory_is_refused():
    M = ALLPASS_MAX_M + 1
    B, N = 2, 3 * M + 77
    m = _module(B, 1, N, M - LONG_MLFO, LONG_MLFO, interpolation="allpass")
    from mod_extraction_b200 import _ops
    x = torch.zeros((B, 1, N), device=dev())
    out = torch.full((B, 1, N), float("nan"), device=dev())
    for src in (_audio(np.zeros((B, N), F32)), _control(np.zeros((B, N // 100), F32))):
        with pytest.raises(RuntimeError, match="shared memory"):
            _ops.flanger_chorus(x, src, M - LONG_MLFO, LONG_MLFO, 0.5, 0.5, 0.5, 0.5, 0.5, out=out,
                                interpolation="allpass")
        assert torch.isnan(out).all()


# --------------------------------------------------------------------------- 4. lines of a few samples

N_TINY = 20000
N_LO_TINY = 200


def _tiny_mods(n, rng):
    """Constant 0, constant 1, uniform noise, a 0 -> 1 ramp."""
    return np.stack([np.zeros(n), np.ones(n), rng.uniform(0, 1, n), np.linspace(0.0, 1.0, n)]).astype(F32)


def _tiny_params(Mmin, Mlfo, rng):
    """Rows 0-3: random parameters.  Rows 4-7: delays of at most ~1.3 samples (D0 = 0.37, A <= 0.9), so that whole tiles
    take the taps one sample back and, for a delay below one sample, M back (read-before-write)."""
    B = 8
    U = lambda lo, hi, n: rng.uniform(lo, hi, n).astype(F32)
    fb = np.concatenate([U(0.0, 0.69, 3), [0.69], [0.69, 0.5, 0.69, 0.3]]).astype(F32)
    mdw = np.concatenate([U(0.0, 1.0, 4), np.full(4, min(1.0, 0.37 / Mmin) if Mmin else 0.0)]).astype(F32)
    width = np.concatenate([U(0.0, 1.0, 4), np.full(4, min(1.0, 0.9 / Mlfo) if Mlfo else 0.0)]).astype(F32)
    return [fb, mdw, width, U(0.25, 1.0, B), U(0.25, 1.0, B)]


@pytest.mark.parametrize("C", [1, 2])
@pytest.mark.parametrize("Mmin,Mlfo", [(0, 1), (1, 0), (1, 1), (0, 2), (2, 1), (31, 32), (32, 32), (33, 32), (64, 63),
                                       (64, 64), (65, 64)])
def test_tiny_lines(Mmin, Mlfo, C):
    """Lines of 1 to 129 samples (the register-history serial runs start at 64): constant, noise and ramp modulation,
    linear interpolation from an audio-rate (one row per channel when C = 2) and a control-rate modulation, and the
    all-pass kernel."""
    M = Mmin + Mlfo
    rng = np.random.RandomState(100 * M + C)
    B = 8
    x = white((B, C, N_TINY), M + 1000 * C)
    params = _tiny_params(Mmin, Mlfo, rng)
    mod = np.concatenate([_tiny_mods(N_TINY, rng)] * 2)
    if C == 2:
        mod = np.stack([mod, np.concatenate([_tiny_mods(N_TINY, rng)] * 2)], axis=1)
    lo = np.concatenate([_tiny_mods(N_LO_TINY, rng)] * 2)
    mod_lo = oracle.linear_interpolate_last_dim(lo, N_TINY)
    for interpolation in ("linear", "allpass"):
        m = _module(B, C, N_TINY, Mmin, Mlfo, interpolation=interpolation)
        _assert_rows(_render(m, x, _audio(mod), params), _oracle(m, x, mod, params), what=(interpolation, "audio rate"))
        _assert_rows(_render(m, x, _control(lo), params), _oracle(m, x, mod_lo, params),
                     what=(interpolation, "control rate"))
