"""CPU: bench.py --dump-outputs writes the same fixed rows of every output, as float32 .npy files."""
import numpy as np
import torch

import bench


def test_dump_outputs_samples_the_same_rows_of_every_output(tmp_path, monkeypatch):
    outputs = {"wet": torch.arange(8 * 6, dtype=torch.float32).view(8, 1, 6),
               "logmel": torch.arange(8 * 4, dtype=torch.float64).view(8, 4)}
    bench.dump_outputs(str(tmp_path / "all"), outputs)
    for name, t in outputs.items():
        got = np.load(tmp_path / "all" / f"{name}.npy")
        assert got.dtype == np.float32 and np.array_equal(got, t.float().numpy())
    monkeypatch.setattr(bench, "DUMP_BYTES", 3 * (6 + 4) * 4)      # room for three rows of both
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), outputs)
    wet, logmel = np.load(tmp_path / "a" / "wet.npy"), np.load(tmp_path / "a" / "logmel.npy")
    assert wet.shape == (3, 1, 6) and logmel.shape == (3, 4)
    rows = wet[:, 0, 0].astype(np.int64) // 6
    assert np.all(np.diff(rows) > 0) and np.array_equal(logmel[:, 0].astype(np.int64) // 4, rows)
    for name in outputs:
        assert np.array_equal(np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy"))
