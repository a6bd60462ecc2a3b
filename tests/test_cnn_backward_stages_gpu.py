"""GPU tests of the Spectral2DCNN training path (TF32) stage by stage: the forward with saves and every backward kernel
against float64 arithmetic on exactly the operands the kernel saw, at the tile edges of each kernel and at the shipped
shape; and the module's gradients against the test's own chain of entry points, bit for bit.

Each float64 reference comes with a magnitude M, the same float64 operation on absolute values (conv(|x|, |w|) + |bias|,
wgrad(|x|, |dconv|), ...).  The operands are exact in TF32, so the kernels differ from float64 only by float32
accumulation, and every element must satisfy |lib - ref| <= c * M.  c was set from a B200 run with about 4x head-room;
the measured maximum of |lib - ref| / M stands beside each c.  Outputs are NaN-prefilled (argmax 255), so an element
that is never written fails."""
import numpy as np
import pytest
import torch

from mod_extraction_b200 import _lib
from mod_extraction_b200.models import round_to_tf32

from .helpers import CNN_DILATIONS, white
from .test_cnn_backward_gpu import _s, _vp, bounded, check_conv_grads, make_net

pytestmark = pytest.mark.gpu

# c, and the worst |lib - ref| / M measured on a B200 over this file (2^-24 = 6.0e-8)
C_FWD = 5e-6        # z of the training forward: measured max 1.2e-6 (64 input channels), 5.0e-7 (2)
C_POOL = 3e-7       # dbias / dslope of the pool + PReLU backward, per Σ|terms|: measured max 7.3e-8
C_LN = 6e-7         # layer-norm backward: measured max 1.5e-7 (1.3e-7 with a common offset of 300)
C_HEAD = 7e-7       # head backward (dx, dweight, dbias): measured max 1.8e-7
NAN = float("nan")


def nans(*shape):
    return torch.full(shape, NAN, device="cuda")


def tf32_randn(g, *shape, scale=1.0):
    return round_to_tf32(torch.randn(*shape, generator=g) * scale).cuda()


def train_ws(B, H, W, L=1):
    return torch.empty(_lib.lib().modfx_cnn_train_workspace_bytes(B, H, W, L), dtype=torch.uint8, device="cuda")


# ---- float64 checks of one stage, shared by the kernel tests and the module walk ------------------------------------

def check_train_forward(x, w, bias, slope, dil, y, z, am):
    """Training forward of one layer: x (B, H, W, Cin) its TF32 input, w (KH, KW, Cout, Cin) the TF32 packed weights;
    y / z / am (B, H/2, W, 64) its outputs (y None: not available).  z = max(up, lo) + bias within C_FWD of float64;
    argmax = the float64 winner wherever the float64 margin exceeds twice that bound; y = PReLU(z) bitwise."""
    def conv(xx, ww):
        c = torch.nn.functional.conv2d(xx.permute(0, 3, 1, 2).double(), ww.permute(2, 3, 0, 1).double(),
                                       dilation=(1, dil), padding="same")
        return c.permute(0, 2, 3, 1)                                        # (B, H, W, 64)
    ref, mag = conv(x, w), conv(x.abs(), w.abs())
    up, lo = ref[:, 0::2], ref[:, 1::2]
    mz = torch.maximum(mag[:, 0::2], mag[:, 1::2]) + bias.double().abs()
    bounded(f"z Cin {x.size(3)} dil {dil}", z, torch.maximum(up, lo) + bias.double(), mz, C_FWD)
    assert int(am.max()) <= 1
    decided = (lo - up).abs() > 2 * C_FWD * mz
    assert torch.equal(am.bool()[decided], (lo > up)[decided])
    assert int(decided.sum()) >= decided.numel() // 2
    if y is not None:
        assert torch.equal(y, torch.where(z > 0, z, slope * z))


def check_pool_prelu_bwd(dy, z, am, slope, dconv, db, ds):
    """dconv = round_tf32(dz) on the argmax row and 0 on the other, bitwise (dz = dy where z > 0, slope * dy elsewhere,
    in float32 as the kernel forms it); dbias = Σ dz and dslope = Σ dy z [z <= 0] within C_POOL of Σ|terms|."""
    B, Hp, W, C = dy.shape
    r = round_to_tf32(torch.where(z > 0, dy, slope * dy))
    low = am.bool()
    want = torch.stack([torch.where(low, 0.0, r), torch.where(low, r, 0.0)], 2).reshape(B, 2 * Hp, W, C)
    assert torch.equal(dconv, want)
    dy64, z64 = dy.double(), z.double()
    dz = torch.where(z64 > 0, dy64, slope.double() * dy64)
    tz = torch.where(z64 <= 0, dy64 * z64, 0.0)
    bounded("dbias", db, dz.sum((0, 1, 2)), dz.abs().sum((0, 1, 2)), C_POOL)
    bounded("dslope", ds, tz.sum((0, 1, 2)), tz.abs().sum((0, 1, 2)), C_POOL)


def check_layernorm_bwd(g, x, dx, name="layernorm dx", eps=1e-5):
    """Layer-norm backward over (H, W) per (example, channel) of channels-last x: dx = r (g - mean g - xh mean(g xh)).
    The magnitude is the same formula on absolute values, plus the one error that grows with a common offset: the
    kernel's xh = (x - mean) r uses the float32 mean, which shifts xh of a whole (example, channel) by up to
    d = r |mean| 2^-24, and that moves dx by r d (mean(g xh) + xh mean(g)), linear in d and in the signed means."""
    x64, g64 = x.double(), g.double()
    mean = lambda t: t.mean((1, 2), keepdim=True)
    mu = mean(x64)
    r = (x64.var((1, 2), correction=0, keepdim=True) + eps).rsqrt()
    xh = (x64 - mu) * r
    mg, mgx = mean(g64), mean(g64 * xh)
    ref = r * (g64 - mg - xh * mgx)
    mag = r * (g64.abs() + mean(g64.abs()) + xh.abs() * mean((g64 * xh).abs())) \
        + r * (r * mu.abs()) * (mgx.abs() + xh.abs() * mg.abs())
    bounded(name, dx, ref, mag, C_LN)


def check_head_bwd(latent, out, dout, dlat, w, H, dx, dw, db):
    """Head backward from the forward's own latent (B, C, W) and out (B, L, W): dlogit = dout out (1 - out),
    dx (B, H, W, C) = (w^T dlogit + dlatent) / H on every row, dweight = Σ dlogit latent, dbias = Σ dlogit."""
    dl = dout.double() * out.double() * (1 - out.double())
    w64, lat = w.double(), latent.double()
    ref = ((torch.einsum("lc,blw->bcw", w64, dl) + dlat.double()) / H).permute(0, 2, 1)[:, None].expand(-1, H, -1, -1)
    mag = ((torch.einsum("lc,blw->bcw", w64.abs(), dl.abs()) + dlat.double().abs()) / H).permute(0, 2, 1)[:, None]
    bounded("head dx", dx, ref, mag.expand_as(ref), C_HEAD)
    bounded("head dweight", dw, torch.einsum("blw,bcw->lc", dl, lat), torch.einsum("blw,bcw->lc", dl.abs(), lat.abs()),
            C_HEAD)
    bounded("head dbias", db, dl.sum((0, 2)), dl.abs().sum((0, 2)), C_HEAD)


# ---- the entry points, NaN-prefilled -------------------------------------------------------------------------------

def train_forward(x, w, bias, slope, dil):
    B, H, W, cin = x.shape
    y, z = nans(B, H // 2, W, 64), nans(B, H // 2, W, 64)
    am = torch.full((B, H // 2, W, 64), 255, dtype=torch.uint8, device="cuda")
    _lib.check(_lib.lib().modfx_cnn_conv_pool_prelu_train_f32(_vp(x), _vp(y), _vp(z), _vp(am), B, H, W, cin, dil, _vp(w),
                                                              _vp(bias), _vp(slope), _s()))
    return y, z, am


def pool_prelu_bwd(dy, z, am, slope):
    B, Hp, W, _ = dy.shape
    dconv, db, ds = nans(B, 2 * Hp, W, 64), nans(64), nans(64)
    _lib.check(_lib.lib().modfx_cnn_pool_prelu_bwd_f32(_vp(dy), _vp(z), _vp(am), _vp(slope), _vp(dconv), _vp(db), _vp(ds),
                                                       B, 2 * Hp, W, _vp(train_ws(B, 2 * Hp, W)), _s()))
    return dconv, db, ds


def wgrad(x, dconv, dil):
    B, H, W, cin = x.shape
    dw = nans(64, cin, 5, 13)
    _lib.check(_lib.lib().modfx_cnn_conv_wgrad_tf32_f32(_vp(x), _vp(dconv), _vp(dw), B, H, W, cin, dil,
                                                        _vp(train_ws(B, H, W)), _s()))
    return dw


def dgrad(dconv, w_t, dil):
    B, H, W, _ = dconv.shape
    dx = nans(B, H, W, 64)
    _lib.check(_lib.lib().modfx_cnn_conv_dgrad_tf32_f32(_vp(dconv), _vp(dx), B, H, W, dil, _vp(w_t), _s()))
    return dx


def layernorm_bwd(g, x, stats, eps=1e-5):
    B, H, W, C = x.shape
    dx = nans(B, H, W, C)
    _lib.check(_lib.lib().modfx_cnn_layernorm_bwd_f32(_vp(g), _vp(x), _vp(stats), _vp(dx), B, C, H, W, eps,
                                                      _vp(train_ws(B, H, W)), _s()))
    return dx


def head_bwd(latent, out, dout, dlat, w, H):
    B, C, W = latent.shape
    L = out.size(1)
    dx, dw, db = nans(B, H, W, C), nans(L, C), nans(L)
    _lib.check(_lib.lib().modfx_cnn_head_bwd_f32(_vp(latent), _vp(out), _vp(dout), _vp(dlat), _vp(dx), _vp(dw), _vp(db),
                                                 B, H, W, C, L, _vp(w), _vp(train_ws(B, 2, W, L)), _s()))
    return dx, dw, db


# ---- A. training forward ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("cin,dil", [(64, 1), (64, 2), (64, 4), (64, 8), (64, 16), (2, 1)])
@pytest.mark.parametrize("B,H,W", [(1, 8, 1), (2, 10, 127), (1, 12, 128), (1, 14, 129), (1, 20, 345)])
def test_train_forward_against_float64(cin, dil, B, H, W):
    """Both training-forward kernels (64 channels: 8-row tiles; 2 channels: 4-row tiles) at heights whose last tile has
    8, 2, 4, 6 and 4 conv rows (2 or 4 for the 2-channel kernel), and at 1, 127, 128, 129 and 345 frames (W = 1 lies
    inside every dilation's reach).  y is also bitwise the inference TF32 kernel's."""
    g = torch.Generator(device="cpu").manual_seed(1000 * cin + 100 * dil + H + W)
    x = tf32_randn(g, B, H, W, cin)
    w = tf32_randn(g, 5, 13, 64, cin, scale=1.7 / np.sqrt(65 * cin))
    bias = (torch.randn(64, generator=g) * 0.1).cuda()
    slope = (torch.rand(64, generator=g) * 0.35 + 0.05).cuda()
    y, z, am = train_forward(x, w, bias, slope, dil)
    check_train_forward(x, w, bias, slope, dil, y, z, am)
    y_inf = nans(B, H // 2, W, 64)
    _lib.check(_lib.lib().modfx_cnn_conv_pool_prelu_f32(_vp(x), _vp(y_inf), B, H, W, cin, 64, 5, 13, dil, _vp(w), _vp(bias),
                                                        _vp(slope), _lib.CNN_TF32, _s()))
    assert torch.equal(y, y_inf)


# ---- C. layer-0 weight gradient (2 input channels, CUDA cores) --------------------------------------------------------

@pytest.mark.parametrize("B,H,W", [(21, 14, 63), (37, 8, 1), (1, 148, 65), (149, 2, 64), (1, 256, 345)])
def test_wgrad_first_layer_against_float64(B, H, W):
    """The kernel splits B * H * ceil(W / 64) tiles over at most 296 CTAs: 294 and 296 tiles (one per CTA), 298 (two CTAs
    loop over a second tile) and the shipped 1 x 256 x 345 = 1536 (every CTA loops); H is even, so 295 and 297 cannot
    occur."""
    g = torch.Generator(device="cpu").manual_seed(B * H + W)
    x = tf32_randn(g, B, H, W, 2)
    d = tf32_randn(g, B, H, W, 64)
    dw = wgrad(x, d, 1)
    check_conv_grads(x, d, None, 1, None, dw)


# ---- D. pool + PReLU backward -------------------------------------------------------------------------------------------

@pytest.mark.parametrize("B,H,W", [(1, 2, 1), (1, 2, 1024), (1, 2, 1025), (2, 6, 257), (3, 10, 345)])
def test_pool_prelu_bwd_against_float64(B, H, W):
    """Pooled element counts 64, exactly one 65 536-element CTA chunk, one chunk + 64, and 2 and 6 CTAs with W not
    dividing the chunk; random dy and argmax, z with negatives and exact zeros."""
    g = torch.Generator(device="cpu").manual_seed(B * H * W)
    dy = torch.randn(B, H // 2, W, 64, generator=g).cuda()
    z = torch.randn(B, H // 2, W, 64, generator=g)
    z[torch.rand(z.shape, generator=g) < 0.1] = 0.0
    z = z.cuda()
    am = torch.randint(0, 2, (B, H // 2, W, 64), generator=g, dtype=torch.uint8).cuda()
    slope = (torch.rand(64, generator=g) * 0.35 + 0.05).cuda()
    check_pool_prelu_bwd(dy, z, am, slope, *pool_prelu_bwd(dy, z, am, slope))


# ---- E. layer-norm backward -----------------------------------------------------------------------------------------

@pytest.mark.parametrize("offset", [0.0, 300.0])
@pytest.mark.parametrize("B,H,W", [(1, 3, 341), (3, 8, 128), (3, 5, 205), (1, 128, 345)])
def test_layernorm_bwd_against_float64(B, H, W, offset):
    """P * C = 65 472, 65 536 (one 65 536-element chunk), 65 600 (a second chunk of one pixel) and the shipped layer-1
    input 128 x 345 x 64 (44 chunks); with a common offset of 300 the mean cancels in xh = (x - mean) * rstd."""
    L = _lib.lib()
    g = torch.Generator(device="cpu").manual_seed(B * H * W + int(offset))
    x = (offset + torch.randn(B, H, W, 64, generator=g) * (0.5 + torch.rand(64, generator=g))).cuda()
    gy = torch.randn(B, H, W, 64, generator=g).cuda()
    stats = torch.empty(L.modfx_cnn_layernorm_workspace_bytes(B, 64, H, W), dtype=torch.uint8, device="cuda")
    xn = torch.empty_like(x)
    _lib.check(L.modfx_cnn_layernorm_f32(_vp(x), _vp(xn), B, 64, H, W, 0, 1e-5, 1, _vp(stats), _s()))
    check_layernorm_bwd(gy, x, layernorm_bwd(gy, x, stats), f"layernorm dx, offset {offset:g}")


# ---- F. head backward -------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("B,H", [(1, 16), (5, 1), (5, 2)])
@pytest.mark.parametrize("L", [1, 3])
@pytest.mark.parametrize("W", [1, 31, 32, 33, 345])
def test_head_bwd_against_float64(W, L, B, H):
    """Frame counts around the 32-frame CTA tile, 1 and 3 outputs, 1, 2 and 16 mel rows."""
    Lb = _lib.lib()
    g = torch.Generator(device="cpu").manual_seed(W * 100 + L * 10 + B * H)
    y = torch.randn(B, H, W, 64, generator=g).cuda()
    w = (torch.randn(L, 64, generator=g) * 0.3).cuda()
    b = torch.randn(L, generator=g).cuda()
    latent, out = nans(B, 64, W), nans(B, L, W)
    _lib.check(Lb.modfx_cnn_head_f32(_vp(y), _vp(latent), _vp(out), B, H, W, 64, L, _vp(w), _vp(b), _s()))
    dout, dlat = torch.randn(B, L, W, generator=g).cuda(), torch.randn(B, 64, W, generator=g).cuda()
    check_head_bwd(latent, out, dout, dlat, w, H, *head_bwd(latent, out, dout, dlat, w, H))


# ---- G. the module, stage by stage ----------------------------------------------------------------------------------

def chain(net, logmel, dout, dlat):
    """The training step of one chunk through the entry points, every stage checked against float64 on the library's
    own inputs to it; returns the parameter gradients by name."""
    out, latent, saves = net._train_forward(logmel)
    n = len(CNN_DILATIONS)
    layers = []
    for i in range(n):
        conv, act = net.cnn[4 * i + 1], net.cnn[4 * i + 3]
        w = round_to_tf32(conv.weight.detach().permute(2, 3, 0, 1).contiguous())          # (KH, KW, Cout, Cin)
        layers.append((w, conv.bias.detach(), act.weight.detach()))
    for i, (w, bias, slope) in enumerate(layers):
        _, _, x, z, am = saves[i]
        y = saves[i + 1][0] if i + 1 < n else None
        check_train_forward(x, w, bias, slope, CNN_DILATIONS[i], y, z, am)

    grads = {}
    w_out = net.output.weight.detach().reshape(net.latent_dim, -1)
    H = net.n_mels >> n
    dy, dw_out, db_out = head_bwd(latent, out, dout, dlat, w_out, H)
    check_head_bwd(latent, out, dout, dlat, w_out, H, dy, dw_out, db_out)
    grads["output.weight"], grads["output.bias"] = dw_out.view_as(net.output.weight), db_out
    for i in range(n - 1, -1, -1):
        ln_in, stats, x, z, am = saves[i]
        w, _, slope = layers[i]
        dil = CNN_DILATIONS[i]
        dconv, db, ds = pool_prelu_bwd(dy, z, am, slope)
        check_pool_prelu_bwd(dy, z, am, slope, dconv, db, ds)
        dw = wgrad(x, dconv, dil)
        dx = dgrad(dconv, w.flip(0, 1).transpose(2, 3).contiguous(), dil) if i > 0 else None
        check_conv_grads(x, dconv, w.permute(2, 3, 0, 1), dil, dx, dw)
        grads[f"cnn.{4 * i + 1}.weight"], grads[f"cnn.{4 * i + 1}.bias"], grads[f"cnn.{4 * i + 3}.weight"] = dw, db, ds
        if i > 0:
            dy = layernorm_bwd(dx, ln_in, stats)
            check_layernorm_bwd(dx, ln_in, dy)
    return out, latent, grads


@pytest.mark.parametrize("n_mels,n_samples,B,max_chunk", [(256, 88200, 2, 256), (192, 44100, 2, 256), (64, 8192, 3, 2)])
def test_module_backward_stage_by_stage(n_mels, n_samples, B, max_chunk):
    """The shipped shape (256 mels, 345 frames, dilations 1 1 2 4 8 16), 192 mels (layers 4 and 5 at 12 and 6 rows:
    partial tiles) at 173 frames, and 64 mels at 33 frames in chunks of 2 examples.  Every stage of every layer is
    checked against float64; then forward_features + backward must leave every .grad bitwise equal to the chain's
    (the chunks' gradients summed), which pins the wiring of Spectral2DCNN._backward."""
    torch.manual_seed(0)
    net = make_net(seed=5, max_chunk=max_chunk, n_mels=n_mels, n_samples=n_samples)
    x = torch.from_numpy(white((B, 2, n_samples), 21)).cuda()
    with torch.no_grad():
        logmel = net.spectrogram(x)
    g = torch.Generator(device="cpu").manual_seed(8)
    W = logmel.size(-1)
    dout = torch.randn(B, 1, W, generator=g).cuda()
    dlat = (torch.randn(B, 64, W, generator=g) * 0.1).cuda()
    outs, want = [], {}
    for i in range(0, B, max_chunk):
        out, latent, grads = chain(net, logmel[i:i + max_chunk], dout[i:i + max_chunk], dlat[i:i + max_chunk])
        outs.append((out, latent))
        for k, v in grads.items():
            want[k] = v if k not in want else want[k] + v

    net.zero_grad(set_to_none=True)
    out, latent = net.forward_features(logmel)
    assert torch.equal(out.detach(), torch.cat([o for o, _ in outs]))
    assert torch.equal(latent.detach(), torch.cat([lat for _, lat in outs]))
    torch.autograd.backward([out, latent], [dout, dlat])
    got = {k: p.grad for k, p in net.named_parameters()}
    assert set(got) == set(want)
    for k in want:
        assert torch.equal(got[k], want[k]), k
