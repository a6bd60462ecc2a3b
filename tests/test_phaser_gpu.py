"""GPU phaser vs this repo's own CPU restatement of pedalboard/JUCE (PARITY UNPINNED, SURVEY F1):
the chunked affine scan re-associates the recurrence, so the bar is the north_star tolerance
(1e-4 max-abs, SNR >= 80 dB), not bit-exactness."""
import numpy as np
import pytest
import torch

from oracle import oracle
from tests.helpers import guitar, snr_db, white

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _params(B, seed):
    rng = np.random.RandomState(seed)
    logu = lambda lo, hi: np.exp(rng.uniform(np.log(lo), np.log(hi), B)).astype(np.float32)
    U = lambda lo, hi: rng.uniform(lo, hi, B).astype(np.float32)
    # configs/train_lfo_phaser.yml:33-48
    return logu(0.5, 3.0), U(0.2, 1.0), logu(70.0, 18000.0), U(0.0, 0.7), U(0.2, 1.0)


@pytest.mark.parametrize("family", ["white", "guitar"])
@pytest.mark.parametrize("N", [88200, 88200 + 14700, 5000, 127, 129])
def test_phaser_vs_own_oracle(family, N):
    from mod_extraction_b200.phaser import Phaser
    B = 16
    x = white((B, N), 3) if family == "white" else guitar(B, N, 4)[:, 0]
    ps = _params(B, N)
    ref = oracle.phaser(x, 44100.0, *ps)
    y = Phaser(44100.0)(torch.from_numpy(x).to(DEV), *[torch.from_numpy(p) for p in ps]).cpu().numpy()
    err = np.abs(y - ref).max()
    assert err <= 1e-4 and snr_db(ref, y) >= 80.0, (family, N, float(err), snr_db(ref, y))


@pytest.mark.parametrize("block", [1000, 130, 100, 384])
def test_phaser_host_block_sizes(block):
    """Host blocks other than pedalboard's 8192: 1000 is not a multiple of the 4-sample update period, 130 puts one block
    boundary inside a 128-sample chunk, 100 several, 384 is a multiple of 128 whose boundaries fall inside segments."""
    from mod_extraction_b200.phaser import Phaser
    B, N = 32, 88200
    x = white((B, N), 6)
    ps = _params(B, block)
    ref = oracle.phaser(x, 44100.0, *ps, block=block)
    y = Phaser(44100.0, buffer_size=block)(torch.from_numpy(x).to(DEV), *[torch.from_numpy(p) for p in ps]).cpu().numpy()
    err = np.abs(y - ref).max()
    assert err <= 1e-4 and snr_db(ref, y) >= 80.0, (block, float(err), snr_db(ref, y))


def test_phaser_extreme_parameters():
    from mod_extraction_b200.phaser import Phaser
    N = 30000
    x = white((6, N), 9)
    rate = np.array([0.5, 3.0, 3.0, 0.5, 1.0, 2.0], dtype=np.float32)
    depth = np.array([1.0, 1.0, 0.2, 0.2, 1.0, 0.0], dtype=np.float32)
    centre = np.array([70.0, 18000.0, 20.0, 1000.0, 300.0, 5000.0], dtype=np.float32)
    fb = np.array([0.7, 0.7, 0.0, 0.69, 0.7, 0.3], dtype=np.float32)
    mix = np.array([1.0, 0.2, 1.0, 0.5, 0.0, 1.0], dtype=np.float32)
    ref = oracle.phaser(x, 44100.0, rate, depth, centre, fb, mix)
    y = Phaser(44100.0)(torch.from_numpy(x).to(DEV), rate, depth, centre, fb, mix).cpu().numpy()
    assert np.abs(y - ref).max() <= 1e-4
    assert np.array_equal(y[4], np.clip(x[4], -1, 1))       # mix = 0 -> dry, exactly


def test_phaser_subset_and_shapes():
    from mod_extraction_b200.phaser import Phaser
    B, N = 8, 20000
    x = torch.from_numpy(white((B, 1, N), 5)).to(DEV)
    ps = [torch.from_numpy(p) for p in _params(B, 1)]
    ph = Phaser(44100.0)
    y = ph(x, *ps)
    assert y.shape == (B, 1, N)
    out = torch.zeros_like(x)
    ph(x, *ps, example_index=torch.tensor([1, 6]), out=out)
    assert torch.equal(out[1], y[1]) and torch.equal(out[6], y[6]) and float(out[0].abs().max()) == 0.0
    ycpu = ph(x.cpu(), *ps)
    assert not ycpu.is_cuda and torch.equal(ycpu, y.cpu())


def test_apply_pedalboard_phaser_draw_order():
    """Same host RNG draws, in the order of datasets.py:461-465."""
    from mod_extraction_b200.phaser import apply_pedalboard_phaser
    ranges = {"depth": {"min": 0.2, "max": 1.0}, "centre_frequency_hz": {"min": 70.0, "max": 18000.0},
              "feedback": {"min": 0.0, "max": 0.7}, "mix": {"min": 0.2, "max": 1.0}}
    x = torch.from_numpy(white((1, 30000), 8))
    torch.manual_seed(5)
    np.random.seed(5)
    y, p = apply_pedalboard_phaser(x, 44100.0, 1.7, ranges)
    torch.manual_seed(5)
    np.random.seed(5)
    depth = (torch.rand(1) * (1.0 - 0.2) + 0.2).item()
    from scipy.stats import loguniform
    centre = float(loguniform.rvs(70.0, 18000.0, size=1)[0])
    feedback = (torch.rand(1) * (0.7 - 0.0) + 0.0).item()
    mix = (torch.rand(1) * (1.0 - 0.2) + 0.2).item()
    assert p == {"depth": depth, "feedback": feedback, "mix": mix, "rate_hz": 1.7, "shape": "cos"}
    ref = oracle.phaser(x.numpy(), 44100.0, 1.7, depth, centre, feedback, mix)
    assert np.abs(y.numpy() - ref).max() <= 1e-4


def test_phaser_render_step_follows_getitem_example_by_example():
    """Batched PedalboardPhaserDataset.__getitem__ (datasets.py:428-453): per-example draw order on both RNG streams,
    one extra LFO period rendered, random crop of dry / wet, ground-truth LFO cropped and resampled to n // 100 points.
    The restatement below walks the examples with the reference's scalar draws; the DSP is this repo's own phaser
    restatement (PARITY UNPINNED)."""
    _check_render_step(8192)


def test_phaser_render_step_odd_host_block():
    """The same cropped render with a host block that is not a multiple of the 4-sample update period."""
    _check_render_step(1000)


def _check_render_step(buffer_size):
    from scipy.stats import loguniform
    from mod_extraction_b200.phaser import PhaserRenderStep
    cfg = {"pedalboard_phaser": {"rate_hz": {"min": 0.5, "max": 3.0}, "depth": {"min": 0.2, "max": 1.0},
                                 "centre_frequency_hz": {"min": 70.0, "max": 18000.0},
                                 "feedback": {"min": 0.0, "max": 0.7}, "mix": {"min": 0.2, "max": 1.0}}}
    sr, n, B = 44100.0, 22050, 7
    step = PhaserRenderStep(cfg, n, sr, buffer_size=buffer_size)
    L = step.max_proc_n_samples
    assert L == n + 88200
    audio = white((B, 1, L), 31)
    torch.manual_seed(12)
    np.random.seed(12)
    dry, wet, mod_sig, fx = step(torch.from_numpy(audio).to(DEV))
    tail_t, tail_n = torch.rand(2), np.random.uniform(size=2)
    assert dry.shape == (B, 1, n) and wet.shape == (B, 1, n) and mod_sig.shape == (B, n // 100)
    torch.manual_seed(12)
    np.random.seed(12)
    c = cfg["pedalboard_phaser"]
    for b in range(B):
        rate = float(loguniform.rvs(c["rate_hz"]["min"], c["rate_hz"]["max"], size=1)[0])          # datasets.py:429-432
        proc_n = n + int((sr / rate) + 0.5)
        chunk = audio[b, :, :proc_n]
        depth = (torch.rand(1) * (c["depth"]["max"] - c["depth"]["min"]) + c["depth"]["min"]).item()
        centre = float(loguniform.rvs(c["centre_frequency_hz"]["min"], c["centre_frequency_hz"]["max"], size=1)[0])
        feedback = (torch.rand(1) * (c["feedback"]["max"] - c["feedback"]["min"]) + c["feedback"]["min"]).item()
        mix = (torch.rand(1) * (c["mix"]["max"] - c["mix"]["min"]) + c["mix"]["min"]).item()
        proc = oracle.phaser(chunk, sr, rate, depth, centre, feedback, mix, block=buffer_size)
        gt = oracle.make_mod_signal(proc_n, sr, rate, np.pi / 2, "cos")                              # datasets.py:442
        start = torch.randint(low=0, high=proc_n - n + 1, size=(1,)).item()                         # datasets.py:445
        assert fx["rate_hz"][b].item() == rate and fx["depth"][b].item() == depth
        assert fx["feedback"][b].item() == feedback and fx["mix"][b].item() == mix and fx["shape"][b] == "cos"
        assert np.array_equal(dry[b].cpu().numpy(), chunk[:, start:start + n])
        assert np.abs(wet[b].cpu().numpy() - proc[:, start:start + n]).max() <= 1e-4
        ref_mod = oracle.linear_interpolate_last_dim(gt[None, start:start + n], n // 100)[0]       # datasets.py:448-450
        # 60-second-deep float32 LFO arguments: the reference's own closed form (SURVEY F3a), cos within 1 ulp
        assert np.abs(mod_sig[b].cpu().numpy() - ref_mod).max() <= 1e-6
    assert torch.equal(tail_t, torch.rand(2)) and np.array_equal(tail_n, np.random.uniform(size=2))
    # CPU tensors in -> CPU tensors out, same numbers
    torch.manual_seed(12)
    np.random.seed(12)
    d2, w2, m2, _ = step(torch.from_numpy(audio))
    assert not w2.is_cuda and torch.equal(w2, wet.cpu()) and torch.equal(d2, dry.cpu()) and torch.equal(m2, mod_sig.cpu())
