"""GPU tests of the Spectral2DCNN backward pass (TF32, parameter gradients): the gradient kernels against float64
references, and the trainable module against torch float64 autograd and cuDNN TF32 training of its own containers.

Bounds (relative L2 error per tensor) were set from a B200 run with about 2x head-room, see each test's docstring; the
elementwise bounds of check_conv_grads with about 4x."""
import copy
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from mod_extraction_b200 import _lib
from mod_extraction_b200.models import Spectral2DCNN, round_to_tf32

from .helpers import CNN_DILATIONS, cnn_weights, guitar, white

pytestmark = pytest.mark.gpu

N_SAMPLES, N_MELS = 8192, 64


def _vp(t):
    return ctypes.c_void_p(t.data_ptr())


def _s():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / b.norm().clamp_min(1e-300))


def bounded(name, lib, ref, mag, c):
    """Asserts |lib - ref| <= c * mag elementwise (ref, mag float64; an unwritten NaN fails) and prints the worst
    |lib - ref| / mag."""
    err = (lib.double() - ref).abs()
    assert bool(torch.isfinite(err).all()), (name, "non-finite output")
    worst = float((err / mag.clamp_min(1e-300)).max())
    print(f"{name}: max |lib - ref| / M = {worst:.2e} (bound {c:.1e})")
    assert bool((err <= c * mag).all()), (name, worst, c)


# Elementwise bounds of the tensor-core convolution gradients, in units of the float64 magnitude (the same operation
# on |operands|), about 4x the worst |lib - ref| / M measured on a B200 over test_cnn_backward_gpu.py and
# test_cnn_backward_stages_gpu.py (2^-24 = 6.0e-8).
C_DGRAD = 1e-5      # measured max 2.3e-6 (38 x 2^-24: K = 4160 products, tensor-core accumulation)
C_WGRAD = 1.6e-6    # measured max 4.1e-7
C_WGRAD1 = 5e-7     # layer 0 (CUDA cores); measured max 1.1e-7


def check_conv_grads(x, dconv, w, dil, dx, dw):
    """dgrad `dx` (None: not checked) and wgrad `dw` (co, ci, kh, kw) of the 'same' convolution of channels-last x
    (B, H, W, Cin) with w (co, ci, kh, kw) against float64 autograd of the same TF32 operands, elementwise.  Without
    dx, only the weight gradient is formed, and w (which it does not depend on) may be None."""
    if w is None:
        w = torch.zeros(64, x.size(3), 5, 13, device=x.device)

    def grads(xx, dd, ww):
        x64 = xx.permute(0, 3, 1, 2).double().requires_grad_(dx is not None)
        w64 = ww.double().requires_grad_(True)
        (F.conv2d(x64, w64, dilation=(1, dil), padding="same") * dd.permute(0, 3, 1, 2).double()).sum().backward()
        return x64.grad, w64.grad
    rx, rw = grads(x, dconv, w)
    mx, mw = grads(x.abs(), dconv.abs(), w.abs())
    if dx is not None:
        bounded(f"dgrad dil {dil}", dx, rx.permute(0, 2, 3, 1), mx.permute(0, 2, 3, 1), C_DGRAD)
    bounded(f"wgrad Cin {x.size(3)} dil {dil}", dw, rw, mw, C_WGRAD if x.size(3) == 64 else C_WGRAD1)


def make_net(seed=3, max_chunk=256, n_mels=N_MELS, n_samples=N_SAMPLES):
    net = Spectral2DCNN(in_ch=2, n_samples=n_samples, n_mels=n_mels, out_channels=[64] * 6, temp_dilations=CNN_DILATIONS,
                        pool_size=(2, 1), precision="tf32", max_chunk=max_chunk)
    net.load_state_dict({k: torch.from_numpy(v) for k, v in cnn_weights(seed).items()}, strict=False)
    return net.cuda().train()


def audio(kind, B, seed=0):
    x = white((B, 2, N_SAMPLES), seed) if kind == "white" else np.repeat(guitar(B, N_SAMPLES, seed), 2, axis=1)
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def loss_of(out, latent, seed=11):
    g = torch.Generator(device="cpu").manual_seed(seed)
    r1 = torch.randn(out.shape, generator=g, dtype=torch.float64).to(out.device, out.dtype)
    r2 = torch.randn(latent.shape, generator=g, dtype=torch.float64).to(out.device, out.dtype)
    return (out * r1).sum() + 0.1 * (latent * r2).sum()


def torch_grads(net, logmel, dtype, tf32):
    ref = torch.nn.ModuleDict({"cnn": copy.deepcopy(net.cnn), "output": copy.deepcopy(net.output)}).to(dtype)
    old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = tf32
    try:
        h = ref["cnn"](logmel.to(dtype))
        latent = h.mean(dim=-2)
        out = torch.sigmoid(ref["output"](latent))
        loss_of(out, latent).backward()
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
    return {n: p.grad for n, p in ref.named_parameters()}


def lib_grads(net, x):
    net.zero_grad(set_to_none=True)
    out, latent = net(x)
    loss_of(out, latent).backward()
    return {n: p.grad.clone() for n, p in net.named_parameters()}


@pytest.mark.parametrize("kind", ["white", "guitar"])
def test_gradient_parity_against_float64_and_cudnn_tf32(kind):
    """Every parameter gradient of a loss on out and latent, against torch float64 autograd of the module's own
    containers.  Bounds, from a B200 run: relative L2 <= 2e-1 per tensor (measured maximum 1.1e-1, cnn.1.bias on white
    noise, where cuDNN TF32 has 5.6e-2), and, for layers 0-3 and the head, within 3x (+ 2e-3) of cuDNN TF32's own error
    (measured ratios 0.9-2.0x).  Layers 4 and 5 see 4 and 2 mel rows here, a few hundred pooled cells per channel: their
    gradients are decided by a handful of PReLU-sign / pool-argmax flips of the TF32 forward, and both TF32 paths land
    0.3x-20x apart on them (1e-3 to 5e-2 either way), so only the absolute bound applies there."""
    torch.manual_seed(0)
    net = make_net()
    x = audio(kind, 3)
    g = lib_grads(net, x)
    with torch.no_grad():
        logmel = net.spectrogram(x)
    g64 = torch_grads(net, logmel, torch.float64, False)
    g32 = torch_grads(net, logmel, torch.float32, True)
    assert set(g) == set(g64)
    errs = {}
    for n in g64:
        assert g[n].shape == g64[n].shape, n
        errs[n] = (rel(g[n], g64[n]), rel(g32[n], g64[n]))
    print(kind, "rel-L2 (modfx, cuDNN TF32) vs float64:", {n: ("%.1e" % a, "%.1e" % b) for n, (a, b) in errs.items()})
    deep = {f"cnn.{4 * i + k}.{p}" for i in (4, 5) for k in (1, 3) for p in ("weight", "bias")}
    for n, (e_lib, e_cud) in errs.items():
        assert e_lib <= 2e-1, (n, e_lib, e_cud)
        if n not in deep:
            assert e_lib <= 3.0 * e_cud + 2e-3, (n, e_lib, e_cud)


def test_forward_with_graph_is_bitwise_the_no_grad_forward():
    net = make_net()
    x = audio("white", 2, seed=5)
    out, latent = net(x)
    assert out.requires_grad and latent.requires_grad
    with torch.no_grad():
        out0, latent0 = net(x)
    assert torch.equal(out.detach(), out0) and torch.equal(latent.detach(), latent0)


def test_deterministic_and_chunked():
    """Two backward passes are bit-identical; B > max_chunk gives the one-pass gradients up to summation order."""
    net = make_net()
    x = audio("guitar", 3, seed=2)
    g1, g2 = lib_grads(net, x), lib_grads(net, x)
    for n in g1:
        assert torch.equal(g1[n], g2[n]), n
    net.max_chunk = 2
    g3 = lib_grads(net, x)
    for n in g1:
        assert rel(g3[n], g1[n]) <= 1e-5, (n, rel(g3[n], g1[n]))


def test_unsupported_requests_raise():
    net = make_net()
    x = audio("white", 1)
    with pytest.raises(NotImplementedError):
        net(x.clone().requires_grad_(True))
    net32 = make_net()
    net32.precision = "fp32"
    net32._packed = None
    out, latent = net32(x)                  # the forward-only path: no graph
    assert not out.requires_grad and not latent.requires_grad
    with torch.no_grad():
        out, _ = net(x)
    assert not out.requires_grad
    net.eval()
    out, _ = net(x)
    assert not out.requires_grad


def test_it_trains():
    """20 Adam steps on a fixed batch lower the reference loss (l1 + 5 fdl1 + 10 sdl1 against a target LFO)."""
    torch.manual_seed(0)
    net = make_net()
    x = audio("guitar", 3, seed=7)
    n_frames = N_SAMPLES // 256 + 1
    t = torch.linspace(0, 1, n_frames, device="cuda")
    target = (0.5 + 0.4 * torch.sin(2 * np.pi * 2.0 * t))[None, None].expand(3, 1, n_frames)

    def ref_loss(out):
        d1 = lambda v: v[..., 1:] - v[..., :-1]
        return (F.l1_loss(out, target) + 5 * F.l1_loss(d1(out), d1(target)) + 10 * F.l1_loss(d1(d1(out)), d1(d1(target))))

    opt = torch.optim.Adam(net.parameters(), lr=1e-3)
    losses = []
    for _ in range(20):
        opt.zero_grad()
        out, _ = net(x)
        loss = ref_loss(out)
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert losses[-1] < 0.9 * losses[0], losses


@pytest.mark.parametrize("dil", [1, 2, 4, 8, 16])
@pytest.mark.parametrize("B,H,W", [(1, 2, 200), (2, 8, 130), (3, 16, 345), (1, 6, 1), (1, 12, 127), (1, 20, 128),
                                   (17, 6, 1), (3, 12, 129), (2, 20, 257)])
def test_dgrad_and_wgrad_kernels_against_float64(dil, B, H, W):
    """dgrad (tensor-core conv with flipped weights) and wgrad (tcgen05, MN-major operands) against float64
    transposed convolution / correlation of the same TF32 operands.  Bounds: relative L2 <= 1e-5 (the operands are
    exact in TF32, only the float32 accumulation differs), and elementwise check_conv_grads.
    Heights 6, 12 and 20 end in a partial 8-row tile of 6 or 4 rows.  The wgrad K steps B * H * ceil(W / 128) are 6 and
    12 (fewer than the 17 K slices: empty slices), 102 = 6 * 17, and 20, 72, 120 (uneven slices); H is even, so exactly
    17 cannot occur."""
    L = _lib.lib()
    g = torch.Generator(device="cpu").manual_seed(B * 100 + H + dil)
    x = round_to_tf32(torch.randn(B, H, W, 64, generator=g)).cuda()
    d = round_to_tf32(torch.randn(B, H, W, 64, generator=g)).cuda()
    w = round_to_tf32(torch.randn(64, 64, 5, 13, generator=g) * 0.05).cuda()            # (co, ci, kh, kw)
    wt = w.permute(2, 3, 0, 1).flip(0, 1).transpose(2, 3).contiguous()                  # [kh][kw][ci][co] flipped
    dx = torch.full_like(x, float("nan"))
    _lib.check(L.modfx_cnn_conv_dgrad_tf32_f32(_vp(d), _vp(dx), B, H, W, dil, _vp(wt), _s()))
    ws = torch.empty(L.modfx_cnn_train_workspace_bytes(B, H, W, 1), dtype=torch.uint8, device="cuda")
    dw = torch.full((64, 64, 5, 13), float("nan"), device="cuda")
    _lib.check(L.modfx_cnn_conv_wgrad_tf32_f32(_vp(x), _vp(d), _vp(dw), B, H, W, 64, dil, _vp(ws), _s()))
    x64, d64, w64 = (t.double() for t in (x.permute(0, 3, 1, 2), d.permute(0, 3, 1, 2), w))
    x64.requires_grad_(True)
    w64.requires_grad_(True)
    y = F.conv2d(x64, w64, dilation=(1, dil), padding="same")
    (y * d64).sum().backward()
    assert rel(dx.permute(0, 3, 1, 2), x64.grad) <= 1e-5
    assert rel(dw, w64.grad) <= 1e-5
    check_conv_grads(x, d, w, dil, dx, dw)


def test_wgrad_first_layer_and_pool_prelu_ties():
    """Layer 0's CUDA-core weight gradient against float64; exact pool ties route to the upper row."""
    L = _lib.lib()
    B, H, W = 2, 16, 150
    g = torch.Generator(device="cpu").manual_seed(4)
    x = round_to_tf32(torch.randn(B, H, W, 2, generator=g)).cuda()
    d = round_to_tf32(torch.randn(B, H, W, 64, generator=g)).cuda()
    ws = torch.empty(L.modfx_cnn_train_workspace_bytes(B, H, W, 1), dtype=torch.uint8, device="cuda")
    dw = torch.empty(64, 2, 5, 13, device="cuda")
    _lib.check(L.modfx_cnn_conv_wgrad_tf32_f32(_vp(x), _vp(d), _vp(dw), B, H, W, 2, 1, _vp(ws), _s()))
    w64 = torch.zeros(64, 2, 5, 13, dtype=torch.float64, device="cuda", requires_grad=True)
    (F.conv2d(x.permute(0, 3, 1, 2).double(), w64, padding="same") * d.permute(0, 3, 1, 2).double()).sum().backward()
    assert rel(dw, w64.grad) <= 1e-5

    # training forward on a constant input, both kernels (64 channels; 2 channels at dilation 1): every pooled pair is an
    # exact tie -> argmax 0 (upper row), and the backward puts the whole gradient on the upper row
    for cin in (64, 2):
        xin = torch.zeros(1, 4, 8, cin, device="cuda")
        w = torch.full((5, 13, 64, cin), 0.0, device="cuda")
        bias = torch.linspace(-1, 1, 64, device="cuda")
        slope = torch.full((64,), 0.25, device="cuda")
        y, z = torch.empty(1, 2, 8, 64, device="cuda"), torch.empty(1, 2, 8, 64, device="cuda")
        am = torch.full((1, 2, 8, 64), 255, dtype=torch.uint8, device="cuda")
        _lib.check(L.modfx_cnn_conv_pool_prelu_train_f32(_vp(xin), _vp(y), _vp(z), _vp(am), 1, 4, 8, cin, 1, _vp(w),
                                                         _vp(bias), _vp(slope), _s()))
        assert int(am.sum()) == 0 and torch.equal(z, bias.expand_as(z)), cin
        dy = torch.ones_like(y)
        dconv = torch.empty(1, 4, 8, 64, device="cuda")
        db, ds = torch.empty(64, device="cuda"), torch.empty(64, device="cuda")
        _lib.check(L.modfx_cnn_pool_prelu_bwd_f32(_vp(dy), _vp(z), _vp(am), _vp(slope), _vp(dconv), _vp(db), _vp(ds), 1, 4,
                                                  8, _vp(ws), _s()))
        assert torch.all(dconv[:, 1::2] == 0) and torch.all(dconv[:, 0::2] != 0)
        zz = bias.double()
        assert torch.allclose(db.double(), torch.where(zz > 0, 1.0, 0.25).double() * 16, rtol=1e-6)
        assert torch.allclose(ds.double(), torch.where(zz > 0, 0.0, zz) * 16, rtol=1e-5, atol=1e-6)


def test_layernorm_and_head_backward_against_float64():
    """The torch ops of the layer-norm and head backward against float64 autograd.  Bound: relative L2 <= 1e-5."""
    import mod_extraction_b200._torch_ops  # noqa: F401
    g = torch.Generator(device="cpu").manual_seed(9)
    x = (torch.randn(2, 8, 37, 64, generator=g) * 3 + 1).cuda()
    gy = torch.randn(2, 8, 37, 64, generator=g).cuda()
    dx = torch.ops.modfx.cnn_layernorm_bwd(gy, x, 1e-5)
    x64 = x.double().permute(0, 3, 1, 2).requires_grad_(True)
    (F.layer_norm(x64, (8, 37), eps=1e-5) * gy.double().permute(0, 3, 1, 2)).sum().backward()
    assert rel(dx.permute(0, 3, 1, 2), x64.grad) <= 1e-5

    y = torch.randn(2, 4, 37, 64, generator=g).cuda()
    w = (torch.randn(1, 64, generator=g) * 0.3).cuda()
    b = torch.randn(1, generator=g).cuda()
    out, latent = torch.ops.modfx.cnn_head(y, w, b)
    dout, dlat = torch.randn(out.shape, generator=g).cuda(), torch.randn(latent.shape, generator=g).cuda()
    dy, dw, db = torch.ops.modfx.cnn_head_bwd(latent, out, dout, dlat, w, 4)
    y64, w64, b64 = (t.double().requires_grad_(True) for t in (y, w, b))
    lat64 = y64.mean(dim=1).permute(0, 2, 1)
    o64 = torch.sigmoid(torch.einsum("lc,bcw->blw", w64, lat64) + b64[None, :, None])
    ((o64 * dout.double()).sum() + (lat64 * dlat.double()).sum()).backward()
    assert rel(dy, y64.grad) <= 1e-5 and rel(dw, w64.grad) <= 1e-5 and rel(db, b64.grad) <= 1e-5
