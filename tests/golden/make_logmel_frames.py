"""Generate logmel_frames.npz: the reference's own log-mel front end on the inputs of tests/test_logmel_gpu.py that
have no other golden.

    python tests/golden/make_logmel_frames.py

The reference computes its log-mel with torchaudio (MelSpectrogram -> clip -> log, models.py:170-175,199,207-208;
tests/helpers.torchaudio_reference).  Its full outputs are megabytes, so each case stores
  <case>_frames, <case>_ref  every batch row, channel and mel band of a seeded sample of frames (~16k values), and
  <case>_ref_err             the maximum and 99.99th percentile of |reference - exact| over EVERY element, exact being
                             oracle.log_mel with a float64 FFT and the golden mel table, as the tests compute it,
which is all tests.helpers.check_logmel_case needs of the reference.  The tests then compare without importing
torchaudio, and a different torchaudio release cannot move what they compare against.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import oracle  # noqa: E402
from tests.helpers import golden, guitar, torchaudio_reference, white  # noqa: E402

VALUES_PER_CASE = 16384


def config4_rows():
    """test_logmel_full_size_properties: rows 0 and 300 of its (512, 2, 88200) batch."""
    gen = torch.Generator().manual_seed(1)
    return ((torch.rand((512, 2, 88200), generator=gen) * 2 - 1) * 0.5)[[0, 300]].numpy()


CASES = {
    # test_logmel_vs_float64_oracle_and_live_reference
    "white": lambda: white((3, 2, 30000), 7),
    "guitar": lambda: np.concatenate([guitar(2, 30000, 8)] * 2, axis=1),
    # test_logmel_ragged_lengths_and_floor, the lengths compared with the reference
    "white_T88200": lambda: white((2, 1, 88200), 88200),
    "white_T100000": lambda: white((2, 1, 100000), 100000),
    "config4_rows": config4_rows,
}


def main():
    live = torchaudio_reference()
    assert live is not None, "torchaudio is needed to generate these goldens"
    fb = golden("logmel")["fb"]
    d = {}
    for name, make in CASES.items():
        x = make()
        y = live(x)
        e_rt = np.abs(y.astype(np.float64) - oracle.log_mel(x, fb=fb, fft_dtype=np.float64))
        per_frame = y.size // y.shape[-1]
        k = -(-VALUES_PER_CASE // per_frame)
        frames = np.sort(np.random.RandomState(0).choice(y.shape[-1], k, replace=False))
        d[name + "_frames"] = frames
        d[name + "_ref"] = np.ascontiguousarray(y[..., frames])
        d[name + "_ref_err"] = np.array([e_rt.max(), np.quantile(e_rt, 0.9999)])
        print(f"{name}: {y.shape}, |reference - exact| max {e_rt.max():.3e}, 99.99th percentile "
              f"{np.quantile(e_rt, 0.9999):.3e}, frames {frames.tolist()}")
    path = os.path.join(HERE, "logmel_frames.npz")
    np.savez_compressed(path, **d)
    print(f"{path}: {os.path.getsize(path) / 1024:.0f} KiB")


if __name__ == "__main__":
    main()
