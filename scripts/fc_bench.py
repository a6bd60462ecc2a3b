"""Device-time probe of the flanger / chorus kernels on the BASELINE shapes and on the in-kernel LFO sources (one value
per sample, n_lo = N; a synthesised control row too long to stage in shared memory), with a digest of every output so
that two builds (MODFX_LIB=...) can be compared bit for bit.

    python scripts/fc_bench.py [c4] [c4s] [c3] [c5] [c1] [lfo]
"""
import hashlib
import math
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from mod_extraction_b200.fx import MonoFlangerChorusModule
from mod_extraction_b200.modulations import SHAPE_ID, make_combined_mod_sig_batch, make_mod_signal_batch

dev = torch.device("cuda", 0)
SR = 44100
SHAPES6 = ["cos", "tri", "rect_cos", "inv_rect_cos", "saw", "rsaw"]
which = sys.argv[1:] or ["c1", "c4", "c4s", "c3", "c5", "lfo"]


def timed(fn, reps):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts))


def white(B, N, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    return (torch.rand((B, 1, N), device=dev, generator=g) * 2 - 1) * 0.5


def run(name, B, N, lo=None, mmd=1.0, mld=10.0, mdw_lo=0.0, reps=10, seed=0, lfo=None):
    """lo: (B, n_lo) control-rate row, or lfo: (n_lo, sr_lo) to synthesise the LFO in-kernel (forward_lfo)."""
    rng = np.random.RandomState(seed)
    x = white(B, N, seed + 1)
    U = lambda a, b: torch.from_numpy(rng.uniform(a, b, B).astype(np.float32)).to(dev)
    p = [U(0, 0.7), U(mdw_lo, 1.0), U(0.25, 1), U(0.25, 1), U(0.25, 1)]
    m = MonoFlangerChorusModule(B, 1, N, SR, mmd, mld, check_ranges=False)
    out = torch.empty_like(x)
    if lfo is None:
        fn = lambda: m.forward_control_rate(x, lo, *p, out=out)
    else:
        n_lo, sr_lo = lfo
        rate = torch.from_numpy(np.exp(rng.uniform(math.log(0.5), math.log(3.0), B)))
        phase = torch.from_numpy(rng.uniform(0, 2 * math.pi, B))
        shape = torch.tensor([SHAPE_ID[SHAPES6[b % 6]] for b in range(B)])
        fn = lambda: m.forward_lfo(x, rate, phase, shape, n_lo=n_lo, sr_lo=sr_lo, feedback=p[0], min_delay_width=p[1],
                                   width=p[2], depth=p[3], mix=p[4], out=out)
    t = timed(fn, reps)
    gbs = B * N * 8 / (t * 1e-3) / 1e9
    digest = hashlib.sha256(out.cpu().numpy().tobytes()).hexdigest()[:16]
    print(f"{name:38s} B={B:5d} N={N:8d} {t:8.3f} ms  {B * N / SR / (t * 1e-3) / 1e6:7.3f} M audio-s/s  "
          f"{gbs:7.1f} GB/s ({gbs / 6547.8 * 100:5.1f} %)  output sha256 {digest}", flush=True)


def plain_lfo(B, n_lo, rate_lo, rate_hi, exp, seed):
    rng = np.random.RandomState(seed)
    f = np.exp(rng.uniform(math.log(rate_lo), math.log(rate_hi), B))
    ph = rng.uniform(0, 2 * math.pi, B)
    return make_mod_signal_batch(n_lo, 441.0, f, ph, [SHAPES6[b % 6] for b in range(B)], None if exp == 1.0 else np.full(B, exp))


if "c1" in which:
    run("config 1: one 2 s clip, tri 2 Hz", 1, 88200, make_mod_signal_batch(882, 441.0, [2.0], [0.0], ["tri"]))
if "c4" in which:
    B = 1366
    rng = np.random.RandomState(43)
    torch.manual_seed(43)
    lo = make_combined_mod_sig_batch(882, 441, np.exp(rng.uniform(0.0, math.log(3.0), B)), rng.uniform(0, 2 * math.pi, B), SHAPES6, dev)
    run("config 4 flanger group (1366)", B, 88200, lo)
if "c4s" in which:
    B = 171
    rng = np.random.RandomState(44)
    torch.manual_seed(44)
    lo = make_combined_mod_sig_batch(882, 441, np.exp(rng.uniform(0.0, math.log(3.0), B)), rng.uniform(0, 2 * math.pi, B), SHAPES6, dev)
    run("config 4 strong, 512/GPU (171)", B, 88200, lo)
if "c3" in which:
    run("config 3 flanger half, exp=2 (512)", 512, 88200, plain_lfo(512, 882, 0.5, 3.0, 2.0, 45))
    run("config 3 chorus half (512)", 512, 88200, plain_lfo(512, 882, 0.5, 3.0, 2.0, 45), mmd=30.0, mdw_lo=0.367)
if "c5" in which:
    run("config 5 flanger 60 s x 512", 512, 2646000, plain_lfo(512, 26460, 0.5, 3.0, 1.0, 46), reps=3)
    run("config 5 flanger 60 s x 64 (8 GPUs)", 64, 2646000, plain_lfo(64, 26460, 0.5, 3.0, 1.0, 47), reps=3)
if "lfo" in which:
    run("in-kernel LFO, n_lo = N (512)", 512, 88200, lfo=(88200, float(SR)))
    run("in-kernel LFO 60 s, 26 460-point row (512)", 512, 2646000, lfo=(26460, 441.0), reps=3)
