"""Host-side index logic of the up-convolution (CPU, no kernel launches): conv3x3(up2(x)) as four 2x2 parity-class
convolutions of x.  The class taps (csrc/sn_kernels.cu up2_taps), the tap / offset lists b3d.conv.upconv_taps hands the
kernels for the forward, input gradient and weight gradient, and the adjoint b3d_bank_up2_grad applies are emulated in
float64 torch and compared with the convolution of the upsampled tensor and with autograd."""
import pytest
import torch
import torch.nn.functional as F

A = [torch.tensor([[1., 0., 0.], [0., 1., 1.]], dtype=torch.float64), torch.tensor([[1., 1., 0.], [0., 0., 1.]], dtype=torch.float64)]


def class_taps(w):
    """[Cout,Cin,3,3] -> [16,Cout,Cin], tap ((a*2 + b)*2 + u)*2 + v = (A_a W A_b^T)[u][v] (the bank's UF layout)."""
    k = [torch.einsum('ur,oirs,vs->uvoi', A[a], w, A[b]) for a in range(2) for b in range(2)]
    return torch.stack(k).reshape(16, *w.shape[:2])


def class_adjoint(dk):
    """[16 (R*4 + S)][Cin][Cout] (the swapped weight gradient, tap-major) -> dW [Cout,Cin,3,3] (b3d_bank_up2_grad)."""
    g = dk.reshape(4, 4, *dk.shape[1:])
    dw = torch.zeros(dk.shape[2], dk.shape[1], 3, 3, dtype=dk.dtype)
    for r in range(3):
        for s in range(3):
            dw[:, :, r, s] = g[2 - r:4 - r, 2 - s:4 - s].sum(dim=(0, 1)).t()      # R in {3-r, 2-r}, S in {3-s, 2-s}
    return dw


def reference(xp, w):
    """conv3x3(up2(x)) with zero padding in y; xp = x replicate-padded by one column."""
    x = xp[..., 1:-1]
    up = F.interpolate(x, scale_factor=2, mode='nearest')
    return F.conv2d(F.pad(up, (1, 1, 0, 0), mode='replicate'), w, padding=(1, 0))


def emulate_fwd(xp, k):
    from b3d.conv import upconv_taps
    classes, fdy, fdx, _, _ = upconv_taps()
    N, Cin, H, Wp = xp.shape
    W = Wp - 2
    out = torch.zeros(N, k.shape[1], 2 * H, 2 * W, dtype=xp.dtype)
    xz = F.pad(xp, (0, 0, 4, 4))                                    # zero rows: the kernel's out-of-bounds fill
    for t in range(16):
        a, b = classes[t // 4]
        dy, dx = fdy[t], fdx[t]
        assert 0 <= dx and dx + W <= Wp                                # the forward never leaves the padded columns
        src = xz[:, :, 4 + dy:4 + dy + H, dx:dx + W]
        out[:, :, a::2, b::2] += torch.einsum('oi,nihw->nohw', k[t], src)
    return out


def emulate_dgrad(gy, k, H, Wp):
    from b3d.conv import upconv_taps
    _, _, _, ddy, ddx = upconv_taps()
    N, Cout = gy.shape[:2]
    gx = torch.zeros(N, k.shape[2], H, Wp, dtype=gy.dtype)
    for t in range(16):
        for i in range(H):
            for j in range(Wp):
                yy, xx = 2 * i + ddy[t], 2 * j + ddx[t]
                if 0 <= yy < gy.shape[2] and 0 <= xx < gy.shape[3]:
                    gx[:, :, i, j] += gy[:, :, yy, xx] @ k[t]
    return gx


def emulate_wgrad(xp, gy):
    """b3d_conv2d_wgrad_tf32(dy = xp, x = gy, kh = kw = 4, pad_y = 1, stride = 2, x_off = -3, tap major): [16][Cin][Cout]."""
    N, Cin, H, Wp = xp.shape
    gz = F.pad(gy, (4, 4, 4, 4))
    dk = torch.zeros(16, Cin, gy.shape[1], dtype=xp.dtype)
    for R in range(4):
        for S in range(4):
            ys = [2 * i + R - 1 + 4 for i in range(H)]
            xs = [2 * j + S - 3 + 4 for j in range(Wp)]
            sl = gz[:, :, ys][:, :, :, xs]
            dk[R * 4 + S] = torch.einsum('nihw,nohw->io', xp, sl)
    return dk


GEOMS = [(8, 4, 512, 256), (16, 8, 256, 256), (32, 16, 256, 128), (64, 32, 128, 128), (128, 64, 128, 64), (16, 8, 256, 64)]


@pytest.mark.parametrize("H,W,Cin,Cout", GEOMS)
def test_class_convolutions_equal_conv_of_upsample(H, W, Cin, Cout):
    g = torch.Generator().manual_seed(H + Cout)
    N = 1
    ci, co = min(Cin, 8), min(Cout, 4)                             # channel counts do not enter the index logic
    x = torch.randn(N, ci, H, W, generator=g, dtype=torch.float64)
    xp = F.pad(x, (1, 1, 0, 0), mode='replicate')
    w = torch.randn(co, ci, 3, 3, generator=g, dtype=torch.float64)
    torch.testing.assert_close(emulate_fwd(xp, class_taps(w)), reference(xp, w), rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("H,W", [(8, 4), (6, 10), (16, 8)])
def test_input_and_weight_gradient_maps(H, W):
    g = torch.Generator().manual_seed(H * W)
    ci, co = 3, 5
    xp = F.pad(torch.randn(2, ci, H, W, generator=g, dtype=torch.float64), (1, 1, 0, 0), mode='replicate').requires_grad_(True)
    w = torch.randn(co, ci, 3, 3, generator=g, dtype=torch.float64, requires_grad=True)
    y = reference(xp, w)
    gy = torch.randn(y.shape, generator=g, dtype=torch.float64)
    rgx, rgw = torch.autograd.grad(y, (xp, w), gy)
    k = class_taps(w.detach())
    dgx = emulate_dgrad(gy, k, H, W + 2)
    # the up-convolution's input gradient covers the pad columns; their adjoint (added to the edge columns) is the producer's
    dgx[..., 1] += dgx[..., 0]
    dgx[..., W] += dgx[..., W + 1]
    dgx[..., 0] = dgx[..., W + 1] = 0
    torch.testing.assert_close(dgx, rgx, rtol=1e-10, atol=1e-10)
    torch.testing.assert_close(class_adjoint(emulate_wgrad(xp.detach(), gy)), rgw, rtol=1e-10, atol=1e-10)


def test_adjoint_of_the_class_tap_map():
    """<K(W), dK> = <W, K^T(dK)> with K^T in the swapped weight gradient's tap order."""
    g = torch.Generator().manual_seed(3)
    w = torch.randn(4, 6, 3, 3, generator=g, dtype=torch.float64)
    dk = torch.randn(16, 6, 4, generator=g, dtype=torch.float64)    # [R*4 + S][Cin][Cout]
    k = class_taps(w)                                               # [((a*2 + b)*2 + u)*2 + v][Cout][Cin]
    lhs = 0.0
    for a in range(2):
        for b in range(2):
            for u in range(2):
                for v in range(2):
                    R, S = 3 - a - 2 * u, 3 - b - 2 * v
                    lhs += (k[((a * 2 + b) * 2 + u) * 2 + v] * dk[R * 4 + S].t()).sum()
    assert abs(lhs - (w * class_adjoint(dk)).sum()) < 1e-10


def test_tap_lists():
    from b3d.conv import upconv_taps
    classes, fdy, fdx, ddy, ddx = upconv_taps()
    assert classes == [(0, 0), (0, 1), (1, 0), (1, 1)]
    assert fdy == [-1, -1, 0, 0, -1, -1, 0, 0, 0, 0, 1, 1, 0, 0, 1, 1]
    assert fdx == [0, 1, 0, 1, 1, 2, 1, 2, 0, 1, 0, 1, 1, 2, 1, 2]
    assert ddy == [2, 2, 0, 0, 2, 2, 0, 0, 1, 1, -1, -1, 1, 1, -1, -1]
    assert ddx == [0, -2, 0, -2, -1, -3, -1, -3, 0, -2, 0, -2, -1, -3, -1, -3]
