"""Training-step benchmark of Spectral2DCNN (precision "tf32"): forward with saves + backward of the LFO-net body and
head at B = 100 and 128 (n_mels 256, 345 frames), per-kernel times of the gradient kernels, the same step done by
torch / cuDNN TF32 on the module's own containers, and peak memory.  Prints the card's name and power limit beside the
numbers; writes nothing.

    python scripts/train_step_bench.py [--steps 10]
"""
import argparse
import ctypes
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from mod_extraction_b200 import _lib
from mod_extraction_b200.models import Spectral2DCNN, round_to_tf32

N_MELS, W = 256, 345
DILS = [1, 1, 2, 4, 8, 16]


def timed(fn, steps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("train_step_bench: no CUDA device")
    info = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    print("device:", info)
    torch.manual_seed(0)
    vp = lambda t: ctypes.c_void_p(t.data_ptr())
    st = lambda: ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    L = _lib.lib()
    for B in (100, 128):
        net = Spectral2DCNN(in_ch=2, n_samples=(W - 1) * 256, n_mels=N_MELS, out_channels=[64] * 6, temp_dilations=DILS,
                            pool_size=(2, 1), precision="tf32").cuda().train()
        logmel = torch.randn(B, 2, N_MELS, W, device="cuda")

        def step():
            out, latent = net.forward_features(logmel)
            (out.sum() + latent.sum()).backward()

        torch.cuda.reset_peak_memory_stats()
        t_lib = timed(step, args.steps)
        peak = torch.cuda.max_memory_allocated() / 2 ** 30

        ref = torch.nn.ModuleDict({"cnn": net.cnn, "output": net.output})
        torch.backends.cudnn.allow_tf32 = True
        torch.backends.cudnn.benchmark = True

        def step_ref():
            h = ref["cnn"](logmel)
            latent = h.mean(dim=-2)
            out = torch.sigmoid(ref["output"](latent))
            (out.sum() + latent.sum()).backward()

        torch.cuda.reset_peak_memory_stats()
        t_ref = timed(step_ref, args.steps)
        peak_ref = torch.cuda.max_memory_allocated() / 2 ** 30
        fwd_gf = sum(2 * B * (N_MELS >> i) * W * 64 * (2 if i == 0 else 64) * 65 for i in range(6)) / 1e9
        print(f"B={B}: modfx step {t_lib:.2f} ms ({3 * fwd_gf / t_lib:.0f} TFLOP/s over fwd+bwd conv flops), "
              f"peak {peak:.1f} GiB | cuDNN TF32 step {t_ref:.2f} ms, peak {peak_ref:.1f} GiB")

        # per kernel, layer 1 (64 ch, H = 128) and layer 0 (2 ch, H = 256)
        H = N_MELS // 2
        x = round_to_tf32(torch.randn(B, H, W, 64, device="cuda"))
        d = round_to_tf32(torch.randn(B, H, W, 64, device="cuda"))
        wt = round_to_tf32(torch.randn(5, 13, 64, 64, device="cuda"))
        dx = torch.empty_like(x)
        ws = torch.empty(L.modfx_cnn_train_workspace_bytes(B, N_MELS, W, 1), dtype=torch.uint8, device="cuda")
        dw = torch.empty(64, 64, 5, 13, device="cuda")
        gf = 2 * B * H * W * 64 * 64 * 65 / 1e9
        t_d = timed(lambda: _lib.check(L.modfx_cnn_conv_dgrad_tf32_f32(vp(d), vp(dx), B, H, W, 2, vp(wt), st())), args.steps)
        t_w = timed(lambda: _lib.check(L.modfx_cnn_conv_wgrad_tf32_f32(vp(x), vp(d), vp(dw), B, H, W, 64, 2, vp(ws), st())),
                    args.steps)
        x0 = round_to_tf32(torch.randn(B, N_MELS, W, 2, device="cuda"))
        d0 = round_to_tf32(torch.randn(B, N_MELS, W, 64, device="cuda"))
        dw0 = torch.empty(64, 2, 5, 13, device="cuda")
        t_0 = timed(lambda: _lib.check(L.modfx_cnn_conv_wgrad_tf32_f32(vp(x0), vp(d0), vp(dw0), B, N_MELS, W, 2, 1, vp(ws),
                                                                      st())), args.steps)
        gf0 = 2 * B * N_MELS * W * 64 * 2 * 65 / 1e9
        print(f"B={B} layer 1 (H={H}): dgrad {t_d:.3f} ms {gf / t_d:.0f} TFLOP/s, wgrad {t_w:.3f} ms {gf / t_w:.0f} TFLOP/s; "
              f"layer 0 wgrad (CUDA cores) {t_0:.3f} ms {gf0 / t_0:.1f} TFLOP/s")
        del net, ref, x, d, dx, x0, d0, ws
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
