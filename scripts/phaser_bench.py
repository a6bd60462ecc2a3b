"""Device-time probe of one phaser launch (memset of the look-back flags + phaser_phase_kernel + phaser_fused_kernel) on
the shapes bench.py renders, with a digest of every output so that two builds (MODFX_LIB=...) can be compared bit for bit.

    python scripts/phaser_bench.py [c4] [c2] [c5] [--reps R]

  c4  config 4's phaser group: 1365 compact rows of N + 88 200 samples (N + one period of the slowest LFO), cropped at
      the starts of bench.host_params(4096, 43), wet and dry windows written into the (4096, N) outputs
  c2  config 2's PhaserRenderStep: 256 rows of N + 88 200, cropped at the starts its sample_params draws, wet + dry
  c5  config 5's plain render: 512 x 60 s
Inputs are white noise from fixed seeds; every input and output exceeds the 126 MB L2.
"""
import hashlib
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import bench
from mod_extraction_b200 import _ops

dev = torch.device("cuda", 0)
SR, N = bench.SR, bench.N
args = sys.argv[1:]
REPS = int(args[args.index("--reps") + 1]) if "--reps" in args else 20
which = [a for a in args if a in ("c4", "c2", "c5")] or ["c4", "c2", "c5"]
PH_CFG = {"rate_hz": {"min": 0.5, "max": 3.0}, "depth": {"min": 0.2, "max": 1.0},
          "centre_frequency_hz": {"min": 70.0, "max": 18000.0}, "feedback": {"min": 0.0, "max": 0.7},
          "mix": {"min": 0.2, "max": 1.0}}                                 # configs/train_lfo_phaser.yml:33-48


def timed(fn, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), float(np.min(ts)), float(np.max(ts)), reps


def white(B, L, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    return (torch.rand((B, L), device=dev, generator=g) * 2 - 1) * 0.5


def digest(*ts):
    h = hashlib.sha256()
    for t in ts:
        h.update(t.cpu().numpy().tobytes())
    return h.hexdigest()[:16]


def report(name, t, out_samples, outs, note=""):
    med, lo, hi, reps = t
    print(f"{name:44s} {med:8.3f} ms (min {lo:.3f}, max {hi:.3f}, {reps} reps)  "
          f"{out_samples / SR / (med * 1e-3) / 1e6:6.3f} M audio-s/s  digest {digest(*outs)}{note}", flush=True)


def dev32(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)


if "c4" in which:
    B = 4096
    effect, _, ph, _, _ = bench.host_params(B, 43)
    i_ph = np.nonzero(effect == 2)[0]
    L = N + int(SR / 0.5 + 0.5)
    x = white(len(i_ph), L, 50)
    idx = torch.from_numpy(i_ph.astype(np.int32)).to(dev)
    start = torch.from_numpy(ph["start_idx"]).to(dev)
    prm = [dev32(ph[k]) for k in bench.PH_KEYS]
    wet, dry = torch.zeros((B, N), device=dev), torch.zeros((B, N), device=dev)
    fn = lambda: _ops.phaser_crop(x, N, start, float(SR), *prm, example_index=idx, out=wet, dry_out=dry)
    st = ph["start_idx"][i_ph].astype(np.int64)
    seg = 4096
    before, touched = int((st // seg).sum()), int(((st + N + seg - 1) // seg).sum())
    report("config 4 phaser group, cropped (1365 rows)", timed(fn, REPS), len(i_ph) * N, (wet, dry),
           f"  segments before the window {before} of {touched}")
    del x, wet, dry
if "c2" in which:
    from mod_extraction_b200.phaser import PhaserRenderStep
    B = 256
    prs = PhaserRenderStep(PH_CFG, N, float(SR))
    np.random.seed(43)
    torch.manual_seed(43)
    p = prs.sample_params(B)
    x = white(B, prs.max_proc_n_samples, 51)
    start = torch.from_numpy(p["start_idx"].astype(np.int32)).to(dev)
    prm = [dev32(p[k]) for k in bench.PH_KEYS]
    wet, dry = torch.zeros((B, N), device=dev), torch.zeros((B, N), device=dev)
    fn = lambda: _ops.phaser_crop(x, N, start, float(SR), *prm, out=wet, dry_out=dry)
    report("config 2 PhaserRenderStep (256 rows)", timed(fn, REPS), B * N, (wet, dry))
    del x, wet, dry
if "c5" in which:
    B, n = 512, bench.N_LONG
    rng = np.random.RandomState(46)
    prm = [dev32(np.exp(rng.uniform(np.log(0.5), np.log(3.0), B))), dev32(rng.uniform(0.2, 1.0, B)),
           dev32(np.exp(rng.uniform(np.log(70.0), np.log(18000.0), B))), dev32(rng.uniform(0.0, 0.7, B)),
           dev32(rng.uniform(0.2, 1.0, B))]
    x = white(B, n, 52)
    y = torch.zeros_like(x)
    fn = lambda: _ops.phaser(x, float(SR), *prm, out=y)
    report("config 5 plain 512 x 60 s", timed(fn, max(3, REPS // 4)), B * n, (y,))
