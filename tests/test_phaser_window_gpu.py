"""The phaser's cropped windows, bit for bit: a row rendered over [0, start + n_out) and delivered on [start, start + n_out)
runs its 4096-sample segments at the same sample offsets as the plain render of the whole row, so the delivered window
must equal the plain render's samples there exactly, and the dry window the input's.  Starts on both sides of the segment
edges (4096, 8192, 12288) and of every float4 phase (start % 4) cover the segments that are skipped before the window,
the vector stores and their scalar edges; an n_out that is not a multiple of 4 leaves the output rows unaligned."""
import numpy as np
import pytest
import torch

from tests.helpers import white

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SR = 44100.0
L = 88200 + 14700
STARTS = [0, 1, 2, 3, 4095, 4096, 4097, 8191, 8192, 12289]
SUBSET = [10, 0, 3, 7, 1, 5, 9, 2]          # examples 4, 6 and 8 are left out


def _case(n_out, block):
    from mod_extraction_b200 import _ops
    starts = np.array(STARTS + [L - n_out], dtype=np.int32)
    B = len(starts)
    rng = np.random.RandomState(n_out + block)
    logu = lambda lo, hi: torch.from_numpy(np.exp(rng.uniform(np.log(lo), np.log(hi), B)).astype(np.float32)).to(DEV)
    U = lambda lo, hi: torch.from_numpy(rng.uniform(lo, hi, B).astype(np.float32)).to(DEV)
    ps = [logu(0.5, 3.0), U(0.2, 1.0), logu(70.0, 18000.0), U(0.0, 0.7), U(0.2, 1.0)]
    x = torch.from_numpy(white((B, L), 21)).to(DEV)
    plain = _ops.phaser(x, SR, *ps, block=block).cpu().numpy()
    return x, starts, ps, plain


def _nan_outputs(B, n_out):
    return (torch.full((B, n_out), float("nan"), device=DEV), torch.full((B, n_out), float("nan"), device=DEV))


def _check(wet, dry, x, starts, plain, n_out, rows):
    wet, dry, xn = wet.cpu().numpy(), dry.cpu().numpy(), x.cpu().numpy()
    for b in range(len(starts)):
        s = int(starts[b])
        if b in rows:
            assert np.array_equal(wet[b], plain[b, s:s + n_out]), (b, s)
            assert np.array_equal(dry[b], xn[b, s:s + n_out]), (b, s)
        else:
            assert np.isnan(wet[b]).all() and np.isnan(dry[b]).all(), b


@pytest.mark.parametrize("block", [8192, 1000])
@pytest.mark.parametrize("n_out", [88200, 88201])
@pytest.mark.parametrize("layout", ["rows", "compact", "packed"])
def test_phaser_window_equals_plain_render(layout, n_out, block):
    from mod_extraction_b200 import _ops
    x, starts, ps, plain = _case(n_out, block)
    B = len(starts)
    wet, dry = _nan_outputs(B, n_out)
    st = torch.from_numpy(starts).to(DEV)
    if layout == "rows":
        _ops.phaser_crop(x, n_out, st, SR, *ps, block, out=wet, dry_out=dry)
        rows = range(B)
    else:
        idx = torch.tensor(SUBSET, dtype=torch.int32, device=DEV)
        if layout == "compact":
            _ops.phaser_crop(x[idx.long()].contiguous(), n_out, st, SR, *ps, block, example_index=idx, out=wet, dry_out=dry)
        else:                               # rows of start + n_out samples back to back (unaligned starts included)
            lens = [int(starts[e]) + n_out for e in SUBSET]
            offs = torch.tensor(np.concatenate([[0], np.cumsum(lens)[:-1]]), dtype=torch.int64, device=DEV)
            packed = torch.cat([x[e, :n] for e, n in zip(SUBSET, lens)])
            _ops.phaser_crop(packed, n_out, st, SR, *ps, block, example_index=idx, out=wet, dry_out=dry,
                             row_offsets=offs, max_len=L)
        rows = set(SUBSET)
    torch.cuda.synchronize()
    _check(wet, dry, x, starts, plain, n_out, rows)
