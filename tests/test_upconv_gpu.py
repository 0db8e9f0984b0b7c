"""The generator's up-convolution (b3d.conv.upconv_banked: conv3x3(up2(x)) as four 2x2 parity-class convolutions of x, class
taps from the weight bank) and the half-resolution skip of the fused CBN kernel, on the GPU.  Forward, input gradient and
weight gradient (through the bank, back to the 3x3 weight) against fp64 torch on the upsampled tensor, at the generator's
geometries with B = 32; tolerance 4e-3 of the largest magnitude, as the other tf32 convolution tests."""
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 4e-3


def _close(a, b, what):
    err, scale = float((a.double() - b.double()).abs().max()), float(b.abs().max())
    assert err <= TOL * scale, (what, err, scale)


def _ref_upconv(xp, w):
    """fp64 conv3x3(up2(x)), zero padding in y; xp = x replicate-padded by one column (NCHW)."""
    up = F.interpolate(xp[..., 1:-1], scale_factor=2, mode='nearest')
    return F.conv2d(F.pad(up, (1, 1, 0, 0), mode='replicate'), w, padding=(1, 0))


# (input H, W, Cin, Cout): blk2, blk3a, blk4, blk5, blk6, blk3_mesh conv1 of the 256^2 generator
@pytest.mark.parametrize("H,W,Cin,Cout", [(8, 4, 512, 256), (16, 8, 256, 256), (32, 16, 256, 128), (64, 32, 128, 128),
                                          (128, 64, 128, 64), (16, 8, 256, 64)])
def test_upconv_matches_conv_of_upsample(H, W, Cin, Cout):
    from b3d.bank import WeightBank
    from b3d.conv import upconv_banked
    from models.gan import TCConv2d
    torch.manual_seed(H + Cout)
    conv = nn.utils.spectral_norm(TCConv2d(Cin, Cout, 3, padding=(1, 0), bias=False)).to(DEV)
    bank = WeightBank({"c": conv}, up2=["c"])
    B = 32
    x = torch.randn(B, Cin, H, W, device=DEV, dtype=torch.float64)
    xp = F.pad(x, (1, 1, 0, 0), mode='replicate')
    xp32 = xp.float().contiguous(memory_format=torch.channels_last).requires_grad_(True)
    lw = bank.forward(training=False)["c"]
    stats = torch.zeros(2 * Cout, device=DEV, dtype=torch.float64)
    y = upconv_banked(xp32, lw, stats=stats)
    gy = torch.randn(y.shape, device=DEV, dtype=torch.float64)
    (y * gy.float()).sum().backward()

    # eval mode: sigma = u . (W v) with the stored u, v
    u, v = conv.weight_u.double(), conv.weight_v.double()
    sigma = float(u @ (conv.weight_orig.detach().double().reshape(Cout, -1) @ v))
    w = (conv.weight_orig.detach().double() / sigma).requires_grad_(True)
    xr = xp.clone().requires_grad_(True)
    ref = _ref_upconv(xr, w)
    _close(y, ref, "forward")
    r_sum, r_sq = ref.sum(dim=(0, 2, 3)), (ref * ref).sum(dim=(0, 2, 3))
    _close(stats[:Cout], r_sum, "epilogue sum")
    _close(stats[Cout:], r_sq, "epilogue sum of squares")
    gx_ref, gw_ref = torch.autograd.grad(ref, (xr, w), gy)
    gx = xp32.grad.double()
    # the pad columns' gradient is the producer's to fold back: compare after folding, as the producer does
    gx[..., 1] += gx[..., 0]
    gx[..., W] += gx[..., W + 1]
    _close(gx[..., 1:W + 1], gx_ref[..., 1:W + 1], "input gradient")
    # weight_orig's gradient through d(W / sigma) with u, v constants: project the reference the same way
    g = gw_ref.reshape(Cout, -1)
    wm = w.detach().reshape(Cout, -1)
    ref_orig = (g - (g * wm).sum() * torch.outer(u, v)) / sigma
    _close(conv.weight_orig.grad.reshape(Cout, -1), ref_orig, "weight gradient")


@pytest.mark.parametrize("identity", [True, False])
def test_half_resolution_skip_matches_upsampled_skip(identity):
    """cbn_act_pad(y, skip at half resolution, skip_half) == cbn_act_pad(y, up2(skip)) forward and backward (the skip
    gradient comes back as the 2x2 sums)."""
    from argparse import Namespace
    from b3d.ew import cbn_act_pad
    from models.gan import ConditionalBatchNorm2d
    torch.manual_seed(5)
    N, C, H, W = 32, 64, 32, 16
    cbn = ConditionalBatchNorm2d(Namespace(norm_g='batch'), C, 16).to(DEV)
    z = torch.randn(N, 16, device=DEV)
    y = torch.randn(N, C, H, W, device=DEV).contiguous(memory_format=torch.channels_last)
    lo = torch.randn(N, C, H // 2, W // 2, device=DEV)
    off = 1 if identity else 0
    skip_lo = (F.pad(lo, (1, 1, 0, 0), mode='replicate') if identity else lo).contiguous(memory_format=torch.channels_last)
    skip_hi = F.interpolate(lo, scale_factor=2, mode='nearest')
    skip_hi = (F.pad(skip_hi, (1, 1, 0, 0), mode='replicate') if identity else skip_hi).contiguous(memory_format=torch.channels_last)
    outs, grads = [], []
    for sk, half in ((skip_lo, True), (skip_hi, False)):
        yy, ss = y.clone().requires_grad_(True), sk.clone().requires_grad_(True)
        o = cbn_act_pad(yy, cbn, z, skip_nchw=ss, skip_off=off, up=1, pad=1, post_leaky=True, skip_half=half)
        go = torch.randn(o.shape, device=DEV, generator=torch.Generator(DEV).manual_seed(9))
        o.backward(go)
        outs.append(o.detach())
        grads.append((yy.grad, ss.grad))
    torch.testing.assert_close(outs[0], outs[1], rtol=0, atol=0)
    torch.testing.assert_close(grads[0][0], grads[1][0], rtol=1e-5, atol=1e-6)      # per-sample sums: atomics order
    g_hi = grads[1][1][..., off:off + W]
    g_lo = grads[0][1][..., off:off + W // 2]
    torch.testing.assert_close(g_lo, F.avg_pool2d(g_hi, 2) * 4, rtol=1e-5, atol=1e-5)
