#!/usr/bin/env python
"""Benchmark of the render hot path (BASELINE.json metric: audio-seconds rendered per second).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config {1,2,3,4,5}] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workloads = BASELINE.json `configs` with the shapes and ranges of SURVEY 8(d):
  1  flanger, one 2 s clip, 2 Hz triangle LFO (the reference's own CPU-runnable case)
  2  phaser 256 x 88200 with its audio-rate ground-truth cosine LFO (datasets.py:428-453)
  3  chorus + flanger 1024 x 88200, quasi-periodic and distorted control-rate LFOs
  4  (default, the configuration the metric is quoted on) `train_lfo_interwoven_all` data path: examples interleaved
     flanger / chorus / phaser (datasets.py:79-83), combined-shape control-rate LFOs for flanger and chorus (upsampled
     x100 inside the effect kernel), log-mel front end of cat[dry, wet] -> (B, 2, 256, 345)
  5  long-form: 60 s clips x 512, each of the three effects in turn
One step = one pass of the hot path over one batch of synthetic mono 44.1 kHz audio.  Examples are independent, so
ranks render disjoint batch shards with no collective.  Config 4 reports the weak-scaling figure (4096 examples per
GPU) as `value` and, for N > 1, the strong-scaling one north_star names (global batch 4096 cut by
sharding.shard_range, parameters drawn once from one seed, result checked against the single-GPU render) under
`strong`; configs 2, 3 and 5 always cut their fixed global batch (strong scaling).

Prints ONE JSON line on rank 0.  `--impl reference` times the CPU restatement of the reference algorithm (oracle/,
kind "port": the reference itself is python and cannot travel to the GPU box) on the host cores.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SR = 44100
N = 88200
N_LONG = 2646000
N_MELS = 256
SHAPES6 = ["cos", "tri", "rect_cos", "inv_rect_cos", "saw", "rsaw"]
FC_KEYS = ("feedback", "min_delay_width", "width", "depth", "mix")
PH_KEYS = ("rate_hz", "depth", "centre_frequency_hz", "feedback", "mix")
WORKLOADS = {
    1: "config1: flanger, one 2 s clip, 2 Hz triangle control-rate LFO",
    2: "config2: phaser 256 x 88200 + audio-rate ground-truth cosine LFO",
    3: "config3: chorus + flanger 1024 x 88200, quasi-periodic and distorted control-rate LFOs",
    4: "config4: interwoven flanger/chorus/phaser + combined control-rate LFO + log-mel (B,2,256,345)",
    5: "config5: long-form 60 s x 512, flanger + chorus + phaser in turn",
}
# the python reference itself, measured once in the build container (SURVEY 6; it cannot travel to the GPU box)
PY_REFERENCE = {"what": "unmodified reference MonoFlangerChorusModule.forward, config 1 (one 2 s clip), torch CPU, 8 threads",
                "seconds_per_call": 9.32, "audio_s_per_s": 0.215, "source": "SURVEY.md section 6, measured in the build container"}


def env_int(name, default):
    return int(os.environ.get(name, default))


def n_frames(n):
    return n // 256 + 1


# --------------------------------------------------------------------------------------------- inputs

def host_params(B, seed):
    """Per-example parameters with the reference's ranges (configs/data/gen_idmt_{fl,ch}.yml:34-51,
    configs/data/interwoven_idmt_all.yml:24-40, configs/eval_lfo_combined.yml:35-49)."""
    rng = np.random.RandomState(seed)
    effect = np.arange(B) % 3                                   # flanger, chorus, phaser (datasets.py:79-83)
    U = lambda lo, hi: rng.uniform(lo, hi, B).astype(np.float32)
    logU = lambda lo, hi: np.exp(rng.uniform(math.log(lo), math.log(hi), B))
    mdw = U(0.0, 1.0)
    mdw_ch = U(0.367, 1.0)
    fc = {"feedback": U(0.0, 0.7), "min_delay_width": np.where(effect == 1, mdw_ch, mdw).astype(np.float32),
          "width": U(0.25, 1.0), "depth": U(0.25, 1.0), "mix": U(0.25, 1.0)}
    ph = {"rate_hz": logU(0.5, 3.0).astype(np.float32), "depth": U(0.2, 1.0),
          "centre_frequency_hz": logU(70.0, 18000.0).astype(np.float32), "feedback": U(0.0, 0.7), "mix": U(0.2, 1.0)}
    lfo_rate = logU(1.0, 3.0)
    lfo_phase = rng.uniform(0.0, 2 * math.pi, B)
    # phaser examples are rendered over one extra LFO period and cropped at a random start (datasets.py:433-447)
    extra = (SR / ph["rate_hz"].astype(np.float64) + 0.5).astype(np.int64)
    ph["start_idx"] = (rng.randint(0, 1 << 30, B) % (extra + 1)).astype(np.int32)
    return effect, fc, ph, lfo_rate, lfo_phase


# --------------------------------------------------------------------------------------------- clocks

class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = [s for s in sm if s > 0.5 * max(sm)] or sm
        return {"sm_mhz": statistics.median(busy), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------------------------- CPU arm (oracle/)

def _blas_single_threaded():
    """One BLAS thread per worker: the log-mel restatement runs one python thread per core, and each of them calls a
    matmul -- a multi-threaded BLAS underneath oversubscribes the cores several times over."""
    try:
        from threadpoolctl import threadpool_limits
        return threadpool_limits(limits=1)
    except Exception:                                           # pragma: no cover
        import contextlib
        return contextlib.nullcontext()


def _oracle_logmel_rows(both, threads, fb=None):
    from concurrent.futures import ThreadPoolExecutor
    from oracle import oracle
    fb = oracle.mel_filterbank() if fb is None else fb
    with _blas_single_threaded(), ThreadPoolExecutor(max_workers=threads) as ex:
        rows = list(ex.map(lambda b: oracle.log_mel(both[b], fb=fb), range(both.shape[0])))
    return np.stack(rows)


def oracle_step(dry, effect, mod_lo, fc, ph, threads, fb=None):
    """Config 4 through the CPU restatement (oracle/): returns (wet, logmel).  `fb`: mel table to use (parity checks
    pass the product's, which is torchaudio's own: a from-scratch float32 table differs by ~3e-5 in a few weights)."""
    from oracle import oracle
    n = dry.shape[-1]
    wet = np.empty_like(dry)
    for k, (mmd, mld) in ((0, (1.0, 10.0)), (1, (30.0, 10.0))):
        idx = np.nonzero(effect == k)[0]
        if idx.size:
            mod = oracle.linear_interpolate_last_dim(mod_lo[idx], n)
            wet[idx] = oracle.flanger_chorus(dry[idx], mod, *[fc[kk][idx] for kk in FC_KEYS],
                                             sr=SR, max_min_delay_ms=mmd, max_lfo_delay_ms=mld)
    idx = np.nonzero(effect == 2)[0]
    if idx.size:
        wet[idx, 0] = oracle.phaser(dry[idx, 0], float(SR), *[ph[kk][idx] for kk in PH_KEYS])    # (no extra period here)
    both = np.concatenate([dry, wet], axis=1)                    # lightning.py:106
    return wet, _oracle_logmel_rows(both, threads, fb)


def oracle_inputs(B, seed, n=N):
    from oracle import oracle
    effect, fc, ph, rate, phase = host_params(B, seed)
    rng = np.random.RandomState(seed + 1)
    dry = ((rng.random_sample((B, 1, n)) * 2 - 1) * 0.5).astype(np.float32)
    draws = oracle.ReplayDraws(choices=rng.randint(0, 6, 64 * B))
    mod_lo = np.stack([oracle.make_combined_mod_sig(n // 100, SR // 100, rate[b], phase[b], SHAPES6, rng=draws)
                       for b in range(B)])
    return dry, effect, mod_lo, fc, ph


def oracle_workload(config, sample_B):
    """(callable doing one bounded CPU pass of `config`, audio seconds it renders, description)."""
    from oracle import oracle
    oracle.build()
    threads = oracle.num_threads()
    if config == 4:
        dry, effect, mod_lo, fc, ph = oracle_inputs(sample_B, 1234)
        fn = lambda: oracle_step(dry, effect, mod_lo, fc, ph, threads)
        return fn, sample_B * N / SR, f"{sample_B} examples x 2 s of the same workload", threads
    rng = np.random.RandomState(7)
    U = lambda lo, hi, B: rng.uniform(lo, hi, B).astype(np.float32)
    if config == 1:
        x = ((rng.random_sample((1, 1, N)) * 2 - 1) * 0.5).astype(np.float32)
        mod = oracle.linear_interpolate_last_dim(oracle.make_mod_signal(882, 441.0, 2.0, 0.0, "tri")[None], N)
        fn = lambda: oracle.flanger_chorus(x, mod, *[np.full(1, v, np.float32) for v in (0.5, 1.0, 1.0, 1.0, 1.0)],
                                           sr=SR, max_min_delay_ms=1.0, max_lfo_delay_ms=10.0)
        return fn, N / SR, "the whole workload (one 2 s clip)", 1
    if config == 2:
        B = sample_B
        x = ((rng.random_sample((B, N)) * 2 - 1) * 0.5).astype(np.float32)
        p = [np.exp(U(math.log(0.5), math.log(3.0), B)), U(0.2, 1, B), np.exp(U(math.log(70), math.log(18000), B)),
             U(0, 0.7, B), U(0.2, 1, B)]
        fn = lambda: oracle.phaser(x, float(SR), *p)
        return fn, B * N / SR, f"{B} of the 256 clips", threads
    n = N if config == 3 else N_LONG
    B = sample_B if config == 3 else max(2, sample_B // 16)
    x = ((rng.random_sample((B, 1, n)) * 2 - 1) * 0.5).astype(np.float32)
    lo = np.stack([oracle.make_mod_signal(n // 100, 441.0, float(np.exp(rng.uniform(math.log(0.5), math.log(3.0)))),
                                          float(rng.uniform(0, 2 * math.pi)), SHAPES6[b % 6],
                                          2.0 if (config == 3 and b % 2) else 1.0) for b in range(B)])
    mod = oracle.linear_interpolate_last_dim(lo, n)
    p = [U(0, 0.7, B), U(0.367, 1, B), U(0.25, 1, B), U(0.25, 1, B), U(0.25, 1, B)]
    ph = [np.exp(U(math.log(0.5), math.log(3.0), B)), U(0.2, 1, B), np.exp(U(math.log(70), math.log(18000), B)),
          U(0, 0.7, B), U(0.2, 1, B)]

    def fn():
        oracle.flanger_chorus(x, mod, *p, sr=SR, max_min_delay_ms=30.0, max_lfo_delay_ms=10.0)
        if config == 5:
            oracle.flanger_chorus(x, mod, *p, sr=SR, max_min_delay_ms=1.0, max_lfo_delay_ms=10.0)
            oracle.phaser(x[:, 0], float(SR), *ph)
    if config == 3:
        return fn, B * n / SR, f"{B} of the 1024 clips (chorus delay line; LFOs given)", threads
    return fn, 3 * B * n / SR, f"{B} of the 512 60 s clips through all three effects", threads


def time_oracle(config, sample_B, reps):
    fn, audio_s, sample, threads = oracle_workload(config, sample_B)
    fn()                                                        # warm caches / lazy init
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    t = statistics.median(ts)
    return audio_s / t, t, threads, sample


def cpu_baseline_block(value, threads, sample):
    return {"value": value, "unit": "audio-s/s", "cores": threads, "kind": "port", "host_cpus": os.cpu_count(),
            "threads": f"{threads} worker threads (pthreads in the C restatement, one python thread per core for the log-mel "
                       "rows), BLAS / OpenMP pinned to 1 thread per worker",
            "sample": sample, "python_reference": PY_REFERENCE}


def run_reference_arm(args, rank):
    if rank != 0:
        return
    fn, audio_s, sample, threads = oracle_workload(args.config, args.cpu_sample)
    ts = []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        fn()
        if i >= args.warmup:
            ts.append(time.perf_counter() - t0)
    total = sum(ts)
    value = audio_s * len(ts) / total
    line = {
        "impl": "reference", "metric": "audio_seconds_rendered_per_second", "value": value, "unit": "audio-s/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(ts),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOADS[args.config], "n_samples": N_LONG if args.config == 5 else N, "sr": SR,
                   "sample": sample},
        "cpu_baseline": cpu_baseline_block(value, threads, f"{sample} per step, {args.steps} steps"),
        "e2e": {"value": value, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------- GPU arm helpers

class Ctx:
    """torch / distributed handles shared by the workloads."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.args = torch, dist, args
        self.rank, self.world, self.local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
        from mod_extraction_b200.sharding import bind_to_gpu_numa_node
        self.numa_cpus = None if args.no_numa_bind else bind_to_gpu_numa_node(self.local_rank)   # before pinned allocations
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, v):
        if self.world == 1:
            return v
        t = self.torch.tensor([v], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def timed(self, step, steps, warmup, sampler=None):
        """W warm-ups, then exactly K steps between CUDA events, barrier + synchronize on both sides, max over ranks."""
        torch = self.torch
        for _ in range(warmup):
            step()
        self.barrier()
        if sampler:
            sampler.start()
            time.sleep(0.25)
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        self.barrier()
        ms = e0.elapsed_time(e1)
        clocks = sampler.stop() if sampler else None
        return self.max_over_ranks(ms) / steps, clocks

    def kernel_ms(self, fn, reps):
        torch = self.torch
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record(); torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return statistics.median(ts)

    def white(self, B, n, seed, lo=0, hi=None):
        """Family W (SURVEY H4): U(-0.5, 0.5) rows [lo, hi) of a (B, 1, n) batch that is the same on every rank."""
        torch = self.torch
        hi = B if hi is None else hi
        gen = torch.Generator(device=self.dev).manual_seed(seed)
        out = torch.empty((hi - lo, 1, n), device=self.dev)
        step = max(1, (1 << 27) // n)
        for c0 in range(0, B, step):
            c1 = min(B, c0 + step)
            x = (torch.rand((c1 - c0, 1, n), device=self.dev, generator=gen) * 2 - 1) * 0.5
            a, b = max(c0, lo), min(c1, hi)
            if a < b:
                out[a - lo:b - lo] = x[a - c0:b - c0]
        return out


def load_peaks():
    peaks, traffic = {}, {}
    for name, dst in (("MEASURED_PEAKS.json", peaks), (os.path.join("profiles", "traffic.json"), traffic)):
        try:
            dst.update(json.load(open(os.path.join(ROOT, name))))
        except Exception:
            pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    src = "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    return peaks, traffic, peak, src


def roofline_block(kernels, dom, names, peak, peak_src, pipeline=None):
    r = {"bound": "hbm", "kernel": names[dom], "achieved": kernels[dom]["gbs"], "peak": peak, "unit": "GB/s",
         "frac": kernels[dom]["gbs"] / peak, "traffic": kernels[dom].get("dram_traffic_bytes"), "peak_source": peak_src,
         "traffic_source": "ncu dram__bytes_read+write per unit of work (profiles/traffic.json), scaled to this launch",
         "how": "algorithmic bytes of the launch / median CUDA-event duration, launches serialised on one stream after the "
                "timed region (inside the timed region the streams overlap)",
         "kernels": kernels}
    if pipeline:
        r["pipeline"] = pipeline
    return r


KERNEL_NAMES = {"logmel": "logmel_kernel (one launch over B dry rows; the wet half is a second identical launch)",
                "flanger": "fc_cta_kernel<control-rate> (flanger group, one CTA of 3 producer warps + 1 consumer warp per delay line)",
                "chorus": "fc_wide_kernel (chorus group)",
                "phaser": "phaser_fused_kernel (+ phaser_phase_kernel), phaser rows rendered over N + one LFO period and cropped"}


def bit_checksum(torch, t):
    """Order-independent exact checksum of a float32 tensor: the sum of its bit patterns."""
    return int(t.contiguous().view(torch.int32).to(torch.int64).sum().item())


DUMP_BYTES = 32 << 20       # --dump-outputs: above this, a sample of rows (a config-4 step returns 4.3 GB)


def dump_outputs(path, outputs):
    """--dump-outputs: each batch-first tensor of `outputs` as <path>/<name>.npy in float32.  All rows when the outputs
    fit in DUMP_BYTES together, else the same rows of each: sorted(RandomState(0).choice(B, k, replace=False))."""
    import torch
    os.makedirs(path, exist_ok=True)
    B = len(next(iter(outputs.values())))
    row_bytes = sum(t[0].numel() * 4 for t in outputs.values())
    k = min(B, max(1, DUMP_BYTES // row_bytes))
    rows = np.sort(np.random.RandomState(0).choice(B, k, replace=False))
    for name, t in outputs.items():
        sample = t.index_select(0, torch.from_numpy(rows).to(t.device))
        np.save(os.path.join(path, name + ".npy"), sample.float().cpu().numpy())


# --------------------------------------------------------------------------------------------- config 4

def make_batch4(cx, R, Bg, seed, lo, hi):
    """Rows [lo, hi) of the global batch of Bg examples drawn from `seed` (the same on every rank)."""
    torch, dev = cx.torch, cx.dev
    from mod_extraction_b200.modulations import make_combined_mod_sig_batch
    n_lo, L_PH = N // 100, N + int(SR / 0.5 + 0.5)      # N + one period of the slowest phaser LFO (0.5 Hz)
    effect, fc_np, ph_np, rate, phase = host_params(Bg, seed)
    torch.manual_seed(seed)
    t0 = time.perf_counter()
    mod_all = make_combined_mod_sig_batch(n_lo, SR // 100, rate, phase, SHAPES6, device=dev)
    torch.cuda.synchronize()
    lfo_s = time.perf_counter() - t0
    # the longer chunks of this shard's phaser examples (N + one period of the slowest LFO, rows in batch order)
    n_ph = int((effect[lo:hi] == 2).sum())
    ph_before = int((effect[:lo] == 2).sum())
    n_ph_all = int((effect == 2).sum())
    b = {"dry": cx.white(Bg, N, seed, lo, hi), "effect": torch.from_numpy(effect[lo:hi].copy()),
         "ph_long": cx.white(n_ph_all, L_PH, seed + 7, ph_before, ph_before + n_ph).view(n_ph, L_PH),
         "ph_start": torch.from_numpy(ph_np["start_idx"][lo:hi].copy()).to(dev),
         "read_samples": int(np.where(effect[lo:hi] == 2, ph_np["start_idx"][lo:hi].astype(np.int64) + N, N).sum()),
         "mod_lo": mod_all[lo:hi].contiguous(), "rate": rate[lo:hi], "phase": phase[lo:hi],
         "fc": {k: torch.from_numpy(v[lo:hi].copy()).to(dev) for k, v in fc_np.items()},
         "ph": {k: torch.from_numpy(v[lo:hi].copy()).to(dev) for k, v in ph_np.items() if k != "start_idx"},
         "lfo_s": lfo_s}
    b["wet"], b["logmel"] = R.alloc_outputs(hi - lo)
    return b


def make_e2e_step(cx, R, wb, chunk):
    """The host-buffer step behind `e2e`: returns (step(logmel_h=None), {"h2d": bytes, "d2h": bytes}).
    Pinned host buffers in the per-effect layout the reference's three datasets produce: the dry audio of the flanger /
    chorus examples as one compact array, the longer chunks of the phaser examples as another, parameters; wet audio
    (+ the dry windows of the phaser examples + per-example log-mel mean) come back into pinned host buffers."""
    torch, dev, rank = cx.torch, cx.dev, cx.rank
    from mod_extraction_b200.modulations import make_combined_mod_sig_batch
    B = wb["dry"].size(0)
    n_lo = N // 100
    dry, wet, logmel = wb["dry"], wb["wet"], wb["logmel"]
    i_fc = R._groups(wb["effect"])[3]
    n_phx = int((wb["effect"] == 2).sum())
    pin = lambda t: t.cpu().pin_memory()
    dry_h = torch.empty((B, 1, N), dtype=torch.float32, device="meta")        # shape only: see dry_fc_h
    dry_fc_h = pin(dry.view(B, N).index_select(0, i_fc))                        # dry audio of the flanger / chorus examples
    fc_h = {k: pin(v) for k, v in wb["fc"].items()}
    ph_h = {k: pin(v) for k, v in wb["ph"].items()}
    # two sets of pinned output buffers: consecutive steps alternate between them when they are pipelined
    wet_hs = [torch.empty((B, 1, N), dtype=torch.float32).pin_memory() for _ in range(2)]
    stat_hs = [torch.empty((B, 2), dtype=torch.float32).pin_memory() for _ in range(2)]
    wet_h, stat_h = wet_hs[0], stat_hs[0]
    dry_d = torch.empty_like(dry)
    # the phaser chunks as a collate function would hand them over: variable-length rows back to back (16-byte aligned
    # starts), each cut to the prefix that determines its window (start + N samples; the effect is causal)
    ph_start_h = pin(wb["ph_start"])
    rows = np.nonzero(wb["effect"].numpy() == 2)[0]
    lens = (ph_start_h.numpy()[rows].astype(np.int64) + N + 3) // 4 * 4
    offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    ph_packed_h = torch.empty((int(offs[-1]),), dtype=torch.float32).pin_memory()
    ph_long_c = wb["ph_long"].cpu()
    for i in range(n_phx):
        ph_packed_h[offs[i]:offs[i + 1]] = ph_long_c[i, :lens[i]]
    del ph_long_c
    words_bytes = B * 17 * 4 + 2 * B * 4                       # generator words + (rate, phase) of the LFO synthesis
    h2d = dry_fc_h.numel() * 4 + ph_packed_h.numel() * 4 + ph_start_h.numel() * 4 + n_phx * 8 + words_bytes + \
        sum(v.numel() * 4 for v in fc_h.values()) + sum(v.numel() * 4 for v in ph_h.values())
    d2h = wet_h.numel() * 4 + stat_h.numel() * 4 + 8

    def lfos(blocking=False):
        torch.manual_seed(43 + rank)
        return make_combined_mod_sig_batch(n_lo, SR // 100, wb["rate"], wb["phase"], SHAPES6, device=dev, deferred=not blocking)

    def e2e_step(logmel_h=None, wait=True, alt=0, duplex=True):
        # host (rate, phase) + generator state in, pinned dry audio in; wet audio (+ log-mel) out to pinned host
        return R.render_host(dry_h, wb["effect"], lfos, fc_h, ph_h, wet_hs[alt], logmel, stat_hs[alt], chunk=chunk,
                             dry_d=dry_d, wet_d=wet, logmel_h=logmel_h, ph_packed_h=ph_packed_h, ph_offsets=offs,
                             ph_start_h=ph_start_h, dry_fc_h=dry_fc_h, wait=wait, duplex=duplex)
    return e2e_step, {"h2d": h2d, "d2h": d2h}


def run_config4(cx, args):
    torch, dev, rank, world = cx.torch, cx.dev, cx.rank, cx.world
    from mod_extraction_b200 import _ops
    from mod_extraction_b200._ops import ModSource
    from mod_extraction_b200.modulations import make_combined_mod_sig_batch
    from mod_extraction_b200.render import InterwovenRenderer
    from mod_extraction_b200.sharding import shard_range
    n_lo = N // 100
    nm = N_MELS * n_frames(N)
    L_PH = N + int(SR / 0.5 + 0.5)                                  # N + one period of the slowest phaser LFO (0.5 Hz)
    R = InterwovenRenderer(N, float(SR), dev)

    make_batch = lambda Bg, seed, lo, hi: make_batch4(cx, R, Bg, seed, lo, hi)

    def step_of(b):
        return lambda: R.render(b["dry"], b["effect"], b["mod_lo"], b["fc"], b["ph"], wet=b["wet"], logmel=b["logmel"],
                                ph_long=b["ph_long"], ph_start=b["ph_start"])

    # ---------------- weak scaling: `value` (every rank its own batch, as in round 1)
    B = args.batch_per_gpu
    wb = make_batch(B, 43 + rank, 0, B)                             # configs/train_lfo_interwoven_all.yml:1
    lfo_gen_s = wb["lfo_s"]                                         # first call: includes lazy allocations
    step = step_of(wb)
    sampler = ClockSampler(cx.local_rank) if rank == 0 else None
    ms_per_step, clocks = cx.timed(step, args.steps, args.warmup, sampler)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"wet": wb["wet"], "logmel": wb["logmel"]})
    value = world * B * (N / SR) / (ms_per_step * 1e-3)
    checksum = float(wb["wet"].double().abs().mean().item())
    # algorithmic bytes of the step: dry audio read once (a phaser example up to the end of its window: start + N
    # samples of its longer chunk, plus the dry window written back), wet written, log-mel written
    n_phx = int((wb["effect"] == 2).sum())
    step_bytes = wb["read_samples"] * 4 + n_phx * N * 4 + B * N * 4 + B * 2 * nm * 4
    bytes_per_example = step_bytes / B

    # ---------------- the same step with the LFO synthesis inside it (north_star puts it on the hot path)
    def step_with_lfo():
        torch.manual_seed(43 + rank)
        wb["mod_lo"], finish = make_combined_mod_sig_batch(n_lo, SR // 100, wb["rate"], wb["phase"], SHAPES6, device=dev,
                                                           deferred=True)
        step()
        assert finish()             # waits for the LFO kernels only: the next step's host work overlaps this render
    ms_lfo, _ = cx.timed(step_with_lfo, args.steps, 3)
    with_lfo = {"value": world * B * (N / SR) / (ms_lfo * 1e-3), "ms_per_step": ms_lfo,
                "lfo_ms": max(0.0, ms_lfo - ms_per_step),
                "note": "combined-shape control-rate LFOs regenerated every step from (rate, phase) and the torch global "
                        "generator: candidates + corner search + draw-order replay + span synthesis on the device, one "
                        "8-byte read-back taken after the render has been queued (make_combined_mod_sig_batch(deferred=True))"}

    # ---------------- per-kernel durations, serialised (same launches, one stream) for the roofline
    Rs = InterwovenRenderer(N, float(SR), dev, concurrent=False)
    i_fl, i_ch, i_ph, i_fc = Rs._groups(wb["effect"])
    fc_args = [wb["fc"][k] for k in FC_KEYS]
    ph_args = [wb["ph"][k] for k in PH_KEYS]
    dry, wet, logmel, mod_lo = wb["dry"], wb["wet"], wb["logmel"], wb["mod_lo"]
    dry2, wet2 = dry.view(B, N), wet.view(B, N)
    launches = {
        "flanger": (lambda: _ops.flanger_chorus(dry, ModSource.control_rate(mod_lo), Rs.fl[0], Rs.fl[1], *fc_args,
                                                example_index=i_fl, out=wet), i_fl.numel() * N * 8, 1),
        "chorus": (lambda: _ops.flanger_chorus(dry, ModSource.control_rate(mod_lo), Rs.ch[0], Rs.ch[1], *fc_args,
                                               example_index=i_ch, out=wet), i_ch.numel() * N * 8, 2),
        "phaser": (lambda: _ops.phaser_crop(wb["ph_long"], N, wb["ph_start"], float(SR), *ph_args, example_index=i_ph,
                                            out=wet2, dry_out=dry2),
                   (wb["read_samples"] - (B - n_phx) * N) * 4 + 2 * n_phx * N * 4, PHASER_LAUNCHES),
        "logmel": (lambda: Rs.front.forward_rows(dry2, N, B, logmel.view(-1), N, 2 * nm, None),
                   B * (N * 4 + nm * 4), 1),
    }
    peaks, traffic_tab, peak, peak_src = load_peaks()
    kernels = {}
    for name, (fn, nbytes, n_launch) in launches.items():
        ms = cx.kernel_ms(fn, max(3, min(10, args.steps)))
        kernels[name] = {"ms": ms, "algorithmic_bytes": nbytes, "gbs": nbytes / (ms * 1e-3) / 1e9, "launches": n_launch}
    step()                                                      # leave wet / log-mel consistent again
    units = {"logmel": ("bytes_per_row", B), "flanger": ("bytes_per_example", i_fl.numel()),
             "chorus": ("bytes_per_example", i_ch.numel()), "phaser": ("bytes_per_example", i_ph.numel())}
    for name, (key, n_units) in units.items():
        ratio = traffic_tab.get(name, {}).get("per_algorithmic_byte")      # ncu DRAM bytes per algorithmic byte of the capture
        t = traffic_tab.get(name, {}).get(key)
        kernels[name]["dram_traffic_bytes"] = (ratio * kernels[name]["algorithmic_bytes"] if ratio is not None else
                                               (None if t is None else t * n_units))
    dom = max(kernels, key=lambda k: kernels[k]["ms"] * (2 if k == "logmel" else 1))
    gbs_pipe = step_bytes / (ms_per_step * 1e-3) / 1e9
    roofline = roofline_block(kernels, dom, KERNEL_NAMES, peak, peak_src,
                              {"achieved": gbs_pipe, "frac": gbs_pipe / peak, "bytes_per_example": bytes_per_example,
                               "bytes_per_step": step_bytes})

    # ---------------- end to end through the public API with host buffers (`e2e`), LFO synthesis included
    e2e = e2e_full = None
    if not args.no_e2e:
        e2e_step, io = make_e2e_step(cx, R, wb, args.e2e_chunk)
        h2d, d2h = io["h2d"], io["d2h"]

        def host_timed(fn, n_rep):
            for _ in range(2):
                fn()
            cx.barrier()
            t0 = time.perf_counter()
            for _ in range(n_rep):
                fn()
            cx.barrier()
            return cx.max_over_ranks((time.perf_counter() - t0) / n_rep)

        def host_timed_pipelined(n_rep):
            """Steady-state step time with consecutive steps overlapped: step i+1 is queued (its input copies start)
            while the last output copies of step i drain; every step's copies, kernels and read-back are inside the
            timed region, which ends when the last byte of the last step has landed."""
            def burst(n):
                h = None
                for i in range(n):
                    nxt = e2e_step(wait=False, alt=i & 1)
                    if h is not None:
                        h.wait()
                    h = nxt
                h.wait()
            burst(2)
            cx.barrier()
            t0 = time.perf_counter()
            burst(n_rep)
            cx.barrier()
            return cx.max_over_ranks((time.perf_counter() - t0) / n_rep)

        n_e2e = max(3, min(args.steps, 10))
        dt_serial = host_timed(e2e_step, n_e2e)
        dt_pipe = host_timed_pipelined(n_e2e)
        dt_half = host_timed(lambda: e2e_step(duplex=False), n_e2e) if world > 1 else float("inf")
        # Three schedules of the same public call.  Steps pipelined (wait=False) keep both copy directions busy all the
        # time: fastest on a host that sustains full duplex (one rank: 34 vs 38 ms), slower where several ranks share a
        # host whose duplex rate collapses (two ranks on these boxes: 65 vs 52 ms); there, holding the output copies back
        # until the inputs are in (duplex=False) can win.  The headline is the fastest schedule; all are shown.
        dt, schedule = min((dt_pipe, "steps pipelined (render_host(wait=False))"),
                           (dt_serial, "one step at a time (render_host(wait=True))"),
                           (dt_half, "one step at a time, one copy direction at a time (render_host(duplex=False))"))
        e2e = {"value": world * B * (N / SR) / dt, "unit": "audio-s/s", "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "ms_per_step": dt * 1e3, "steps": n_e2e, "chunk": args.e2e_chunk,
               "schedule": schedule,
               "steps_pipelined": {"ms": dt_pipe * 1e3, "value": world * B * (N / SR) / dt_pipe},
               "half_duplex": None if world == 1 else {"ms": dt_half * 1e3, "value": world * B * (N / SR) / dt_half},
               "one_step_alone": {"ms": dt_serial * 1e3, "value": world * B * (N / SR) / dt_serial,
                                  "note": "the same call with every step synchronised before the next one starts (latency of "
                                          "one step: first input byte to last output byte)"},
               "note": "per step, InterwovenRenderer.render_host: pinned host dry audio of the flanger / chorus examples + the "
                       "variable-length chunks of the phaser examples (packed back to back, each cut to the start + N samples "
                       "that determine its window) + parameters in, LFO synthesis on the device from host (rate, phase) + "
                       "generator words behind the first copies, wet audio + per-example log-mel mean out (the dry windows of "
                       "the phaser examples are slices of host data and are not copied back), chunks pipelined over "
                       "copy/compute/copy streams; measured one step at a time and with consecutive steps pipelined the same way "
                       "(render_host(wait=False): step i+1 is queued while the last output copies of step i drain, two "
                       "alternating sets of pinned output buffers; timed from the first call to the last byte of the last "
                       "step), the faster schedule is the headline (`schedule`); the (B,2,256,345) log-mel "
                       "tensor stays in HBM where the extractor consumes it (e2e_full delivers it to the host too)"}
        if not args.no_e2e_full:
            try:
                logmel_h = torch.empty(tuple(logmel.shape), dtype=torch.float32).pin_memory()
                dt2 = host_timed(lambda: e2e_step(logmel_h), max(3, n_e2e // 2))
                e2e_full = {"value": world * B * (N / SR) / dt2, "unit": "audio-s/s", "ms_per_step": dt2 * 1e3,
                            "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h + logmel_h.numel() * 4,
                            "note": "as e2e, with the log-mel tensor copied to pinned host memory as well"}
                del logmel_h
            except Exception as exc:                            # a side measurement must not take the headline down
                e2e_full = {"error": f"{type(exc).__name__}: {exc}"[:200]}

    # ---------------- strong scaling: the global batch of config 4 cut over the ranks (SURVEY 8e)
    strong = None
    if world > 1 or args.scaling == "strong":
        Bg = args.global_batch
        lo, hi = shard_range(Bg, rank, world)
        sb = make_batch(Bg, 43, lo, hi)
        ms_s, _ = cx.timed(step_of(sb), args.steps, args.warmup)
        torch.cuda.synchronize()
        mine = torch.tensor([bit_checksum(torch, sb["wet"]), bit_checksum(torch, sb["logmel"])], dtype=torch.int64, device=dev)
        sums = [mine]
        if world > 1:
            sums = [torch.zeros_like(mine) for _ in range(world)]
            cx.dist.all_gather(sums, mine)
        ok = None
        if rank == 0:
            # what one GPU renders for the same global batch: every shard must reproduce its rows bit for bit
            full = make_batch(Bg, 43, 0, Bg)
            step_of(full)()
            torch.cuda.synchronize()
            ok = True
            for r in range(world):
                a, b = shard_range(Bg, r, world)
                ok = ok and int(sums[r][0]) == bit_checksum(torch, full["wet"][a:b]) and \
                    int(sums[r][1]) == bit_checksum(torch, full["logmel"][a:b])
            del full
        strong = {"global_batch": Bg, "per_gpu": hi - lo, "ms_per_step": ms_s, "value": Bg * (N / SR) / (ms_s * 1e-3),
                  "unit": "audio-s/s", "scaling": "strong", "shards_equal_single_gpu_render": ok,
                  "note": "parameters and audio drawn once from seed 43 for the global batch, rank r renders "
                          "sharding.shard_range(global_batch, r, N); bit-pattern checksums of every shard's wet audio and "
                          "log-mel compared with the same rows of a single-GPU render of the whole batch"}
    gather_ms = None
    if world > 1:
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        cs = torch.tensor([checksum], dtype=torch.float64, device=dev)
        out = torch.empty((world,), dtype=torch.float64, device=dev)
        g0.record()
        cx.dist.all_gather_into_tensor(out, cs)
        g1.record()
        torch.cuda.synchronize()
        gather_ms = g0.elapsed_time(g1)
        checksum = float(out.mean().item())
    line = {
        "value": value, "ms_per_step": ms_per_step, "scaling": "weak",
        "config": {"workload": WORKLOADS[4], "batch_per_gpu": B, "global_batch": world * B, "n_samples": N, "sr": SR,
                   "audio": "white noise U(-0.5,0.5)", "lfo": "combined shapes, 882-pt control rate; x100 upsample fused in the "
                   "effect kernel; `value` takes the LFOs as given, `with_lfo` and `e2e` regenerate them every step",
                   "l2": "inputs (1.4 GB dry + 1.4 GB wet + 2.9 GB log-mel per step) far exceed the 126 MB L2",
                   "parallelism": f"batch-sharded x{world}, no collective while rendering"},
        "clocks": clocks, "e2e": e2e, "e2e_full": e2e_full, "with_lfo": with_lfo, "strong": strong,
        # per step (ncu launch list, profiles/r02_launches_all.txt): flanger 1 (fc_cta_kernel) + chorus 2 (fc_wide_kernel, then
        # fc_cta_kernel for the rest, which finds nothing left) + phaser 2 (phaser_phase_kernel, phaser_fused_kernel; the
        # memset of the look-back flags is the driver's) + log-mel 6 (wet rows of the three groups, dry rows of the three groups)
        "gpu_launches": args.steps * (1 + 2 + 2 + 6),
        "roofline": roofline, "lfo_generation_s": lfo_gen_s, "metrics_gather_ms": gather_ms,
        "wet_abs_mean": checksum,
    }
    return line


PHASER_LAUNCHES = 3     # memset of the look-back flags, phase kernel, fused kernel


# --------------------------------------------------------------------------------------------- configs 1, 2, 3, 5

def run_small_configs(cx, args):
    torch, dev, rank, world = cx.torch, cx.dev, cx.rank, cx.world
    from mod_extraction_b200 import modulations as M
    from mod_extraction_b200.fx import MonoFlangerChorusModule
    from mod_extraction_b200.phaser import Phaser
    from mod_extraction_b200.sharding import shard_range
    cfg = args.config
    peaks, traffic_tab, peak, peak_src = load_peaks()
    rng = np.random.RandomState(43)
    extra = {}
    if cfg == 1:
        Bg, n = 1, N
    elif cfg == 2:
        Bg, n = 256, N
    elif cfg == 3:
        Bg, n = 1024, N
    else:
        Bg, n = 512, N_LONG
    lo, hi = shard_range(Bg, rank, world) if cfg != 1 else (0, 1)
    B = hi - lo
    U = lambda a, b: rng.uniform(a, b, Bg).astype(np.float32)
    LU = lambda a, b: np.exp(rng.uniform(math.log(a), math.log(b), Bg)).astype(np.float32)
    dv = lambda a: torch.from_numpy(np.ascontiguousarray(a[lo:hi])).to(dev)
    x = cx.white(Bg, n, 42 + cfg, lo, hi)
    out = torch.empty_like(x)
    kernels, names = {}, dict(KERNEL_NAMES)
    e2e = None
    if cfg == 1:
        fl = MonoFlangerChorusModule(1, 1, n, SR, 1.0, 10.0, check_ranges=False)
        lo_sig = M.make_mod_signal_batch(882, 441.0, [2.0], [0.0], ["tri"])
        step = lambda: fl.forward_control_rate(x, lo_sig, 0.5, 1.0, 1.0, 1.0, 1.0, out=out)
        audio_s, launches, step_bytes = n / SR, 1, n * 8
        dominant = ("flanger", step, n * 8)
        x_cpu, lo_cpu = x.cpu(), lo_sig.cpu()
        fl.forward_control_rate(x_cpu, lo_cpu, 0.5, 1.0, 1.0, 1.0, 1.0)
        t0 = time.perf_counter()
        reps = 20
        for _ in range(reps):
            y_cpu = fl.forward_control_rate(x_cpu, lo_cpu, 0.5, 1.0, 1.0, 1.0, 1.0)
        dt = (time.perf_counter() - t0) / reps
        e2e = {"value": audio_s / dt, "unit": "audio-s/s", "ms_per_step": dt * 1e3, "h2d_bytes_per_step": n * 4 + 882 * 4,
               "d2h_bytes_per_step": n * 4, "steps": reps,
               "note": "the reference's call site: CPU tensors in, CPU tensor out through MonoFlangerChorusModule "
                       "(H2D + kernel + D2H + sync per call)"}
    elif cfg == 2:
        # the online phaser of train_lfo_phaser: one batch of PedalboardPhaserDataset.__getitem__ (datasets.py:428-453):
        # chunks of N + one LFO period, phaser from the first sample, random window of N, ground-truth LFO
        from mod_extraction_b200.phaser import PhaserRenderStep
        pcfg = {"rate_hz": {"min": 0.5, "max": 3.0}, "depth": {"min": 0.2, "max": 1.0},
                "centre_frequency_hz": {"min": 70.0, "max": 18000.0}, "feedback": {"min": 0.0, "max": 0.7},
                "mix": {"min": 0.2, "max": 1.0}}                          # configs/train_lfo_phaser.yml:33-48
        prs = PhaserRenderStep(pcfg, n, float(SR))
        np.random.seed(43)
        torch.manual_seed(43)
        allp = prs.sample_params(Bg)
        params = {k: v[lo:hi] for k, v in allp.items()}
        audio = cx.white(Bg, prs.max_proc_n_samples, 42 + cfg, lo, hi)
        del x, out
        holder = {}

        def step():
            holder["out"] = prs(audio, params)
        step()
        out = holder["out"][1]
        read = int((params["start_idx"] + n).sum())
        audio_s, launches, step_bytes = Bg * n / SR, PHASER_LAUNCHES + 1, read * 4 + B * n * 8 + B * (n // 100) * 4
        rate_d, start_d = holder["out"][3]["rate_hz"].float().to(dev), torch.from_numpy(params["start_idx"].astype(np.int32)).to(dev)
        prm = [torch.from_numpy(params[k].astype(np.float32)).to(dev) for k in ("rate_hz", "depth", "centre_frequency_hz", "feedback", "mix")]
        from mod_extraction_b200 import _ops
        a2 = audio.view(B, -1)
        dominant = ("phaser", lambda: _ops.phaser_crop(a2, n, start_d, float(SR), *prm), read * 4 + B * n * 8)
    elif cfg == 3:
        half = Bg // 2
        rates_q, ph_q = LU(0.5, 2.0)[:half], U(0, 2 * math.pi)[:half]
        rates_d, ph_d = LU(0.5, 3.0)[:half], U(0, 2 * math.pi)[:half]
        shp = [SHAPES6[i % 6] for i in range(half)]

        def gen_lfos():
            torch.manual_seed(44)
            base = M.make_mod_signal_batch(882, 441.0, rates_q, ph_q, shp)
            quasi = M.make_quasi_periodic_batch(base, 0.10, 0.3333, 0.10, 0.3333, 0.5)      # configs/eval_lfo_quasi.yml:49-54
            dist_ = M.make_mod_signal_batch(882, 441.0, rates_d, ph_d, shp, np.full(half, 2.0))   # eval_lfo_distorted.yml:48
            return torch.cat([quasi, dist_], 0)
        t0 = time.perf_counter()
        mod_all = gen_lfos()
        torch.cuda.synchronize()
        extra["lfo_generation_ms_global_batch"] = (time.perf_counter() - t0) * 1e3
        mod_lo = mod_all[lo:hi].contiguous()
        p_ch = [dv(a) for a in (U(0, 0.7), U(0.367, 1), U(0.25, 1), U(0.25, 1), U(0.25, 1))]
        p_fl = [dv(a) for a in (U(0, 0.7), U(0.0, 1), U(0.25, 1), U(0.25, 1), U(0.25, 1))]
        g = np.arange(lo, hi)
        idx_ch = torch.from_numpy(np.nonzero(g % 2 == 0)[0].astype(np.int32)).to(dev)      # chorus = even examples
        idx_fl = torch.from_numpy(np.nonzero(g % 2 == 1)[0].astype(np.int32)).to(dev)
        ch = MonoFlangerChorusModule(B, 1, n, SR, 30.0, 10.0, check_ranges=False)
        fl = MonoFlangerChorusModule(B, 1, n, SR, 1.0, 10.0, check_ranges=False)
        s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()

        def step():
            cur = torch.cuda.current_stream()
            ev = torch.cuda.Event(); ev.record(cur)
            for s, m, pp, idx in ((s1, ch, p_ch, idx_ch), (s2, fl, p_fl, idx_fl)):
                s.wait_event(ev)
                with torch.cuda.stream(s):
                    m.forward_control_rate(x, mod_lo, *pp, example_index=idx, out=out)
                    e = torch.cuda.Event(); e.record(s)
                cur.wait_event(e)
        audio_s, launches, step_bytes = Bg * n / SR, 3, B * n * 8
        kernels["chorus"] = {"ms": cx.kernel_ms(lambda: ch.forward_control_rate(x, mod_lo, *p_ch, example_index=idx_ch, out=out), 5),
                             "algorithmic_bytes": idx_ch.numel() * n * 8}
        dominant = ("flanger", lambda: fl.forward_control_rate(x, mod_lo, *p_fl, example_index=idx_fl, out=out),
                    idx_fl.numel() * n * 8)
    else:
        n_lo = n // 100
        mod_all = M.make_mod_signal_batch(n_lo, 441.0, LU(0.5, 3.0), U(0, 2 * math.pi), [SHAPES6[i % 6] for i in range(Bg)])
        mod_lo = mod_all[lo:hi].contiguous()
        p_ch = [dv(a) for a in (U(0, 0.7), U(0.367, 1), U(0.25, 1), U(0.25, 1), U(0.25, 1))]
        p_fl = [p_ch[0], dv(U(0.0, 1)), *p_ch[2:]]
        prm = [dv(a) for a in (LU(0.5, 3), U(0.2, 1), LU(70, 18000), U(0, 0.7), U(0.2, 1))]
        ch = MonoFlangerChorusModule(B, 1, n, SR, 30.0, 10.0, check_ranges=False)
        fl = MonoFlangerChorusModule(B, 1, n, SR, 1.0, 10.0, check_ranges=False)
        ph = Phaser(SR)
        x2, o2 = x.view(B, n), out.view(B, n)
        f_ch = lambda: ch.forward_control_rate(x, mod_lo, *p_ch, out=out)
        f_fl = lambda: fl.forward_control_rate(x, mod_lo, *p_fl, out=out)
        f_ph = lambda: ph(x2, *prm, out=o2)

        def step():
            f_ch(); f_fl(); f_ph()
        audio_s, launches, step_bytes = 3 * Bg * n / SR, 2 + 1 + PHASER_LAUNCHES + 2, 3 * B * n * 8
        for name, fn in (("chorus", f_ch), ("phaser", f_ph)):
            kernels[name] = {"ms": cx.kernel_ms(fn, 3), "algorithmic_bytes": B * n * 8}
        dominant = ("flanger", f_fl, B * n * 8)
    sampler = ClockSampler(cx.local_rank) if rank == 0 else None
    ms_per_step, clocks = cx.timed(step, args.steps, args.warmup, sampler)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dict(zip(("dry", "wet", "mod_sig"), holder["out"][:3])) if cfg == 2 else
                     {"wet": out})
    value = audio_s / (ms_per_step * 1e-3)
    dname, dfn, dbytes = dominant
    kernels[dname] = {"ms": cx.kernel_ms(dfn, 3 if cfg == 5 else 10), "algorithmic_bytes": dbytes}
    for k in kernels.values():
        k["gbs"] = k["algorithmic_bytes"] / (k["ms"] * 1e-3) / 1e9
    dom = max(kernels, key=lambda k: kernels[k]["ms"])
    t = traffic_tab.get(dom, {}).get("bytes_per_example")
    kernels[dom]["dram_traffic_bytes"] = None if (t is None or n != N) else t * kernels[dom]["algorithmic_bytes"] / (n * 8)
    gbs_pipe = step_bytes / (ms_per_step * 1e-3) / 1e9
    roofline = roofline_block(kernels, dom, names, peak, peak_src,
                              {"achieved": gbs_pipe, "frac": gbs_pipe / peak, "bytes_per_step_per_gpu": step_bytes})
    line = {
        "value": value, "ms_per_step": ms_per_step, "scaling": "strong" if cfg != 1 else "weak",
        "config": {"workload": WORKLOADS[cfg], "global_batch": Bg, "batch_per_gpu": B, "n_samples": n, "sr": SR,
                   "audio": "white noise U(-0.5,0.5)",
                   "l2": ("one 353 KB clip: L2-resident by nature (the reference's own CPU case)" if cfg == 1 else
                          "inputs + outputs per step exceed the 126 MB L2"),
                   "parallelism": f"global batch cut over {world} ranks (sharding.shard_range), no collective"},
        "clocks": clocks, "e2e": e2e, "gpu_launches": args.steps * launches, "roofline": roofline,
        "wet_abs_mean": float(out.double().abs().mean().item()), **extra,
    }
    return line


# --------------------------------------------------------------------------------------------- main

def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="modfx", choices=["modfx", "reference"])
    ap.add_argument("--config", type=int, default=4, choices=[1, 2, 3, 4, 5],
                    help="BASELINE.json configuration (4 = the one the metric is quoted on)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="config 4: also measure the strong-scaling split at N = 1 (always measured for N > 1)")
    ap.add_argument("--batch-per-gpu", type=int, default=4096,
                    help="config 4, weak scaling: examples per GPU per step (BASELINE config 4 names 4096)")
    ap.add_argument("--global-batch", type=int, default=4096, help="config 4, strong scaling: examples over all GPUs")
    ap.add_argument("--cpu-sample", type=int, default=96, help="examples in the bounded CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-e2e-full", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true", help="do not pin the process to the GPU-local CPUs")
    ap.add_argument("--e2e-chunk", type=int, default=512, help="examples per pipelined chunk of the host-buffer path")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned as DIR/<name>.npy (float32; a fixed sample of rows when "
                         "the outputs exceed 32 MiB), rank 0's rows, to compare two builds on the same inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; --impl reference has none")
    args.warmup = max(args.warmup, 3)

    rank = env_int("RANK", 0)
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    cx = Ctx(args)
    from mod_extraction_b200 import _lib
    _lib.lib()                                                  # fail loudly if the extension is missing
    body = run_config4(cx, args) if args.config == 4 else run_small_configs(cx, args)

    cpu_baseline = None
    if cx.rank == 0 and cx.world == 1 and not args.no_cpu_baseline:
        v, t, threads, sample = time_oracle(args.config, args.cpu_sample, reps=2)
        cpu_baseline = cpu_baseline_block(v, threads, f"{sample}, median of 2 runs ({t:.2f} s each)")
    if cx.rank == 0:
        line = {"metric": "audio_seconds_rendered_per_second", "unit": "audio-s/s", "n_gpus": cx.world, "steps": args.steps,
                "warmup": args.warmup, "higher_is_better": True, "vs_baseline": None, "dtype": "f32", "data": "synthetic"}
        line.update(body)
        line["cpu_baseline"] = cpu_baseline
        line["host_binding"] = (None if cx.numa_cpus is None else
                                f"rank 0 pinned to {len(cx.numa_cpus)} GPU-local CPUs (NVML affinity)")
        print(json.dumps(line), flush=True)
    if cx.world > 1:
        cx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
