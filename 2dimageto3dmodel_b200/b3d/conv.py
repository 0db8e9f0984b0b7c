"""Dense conv2d over libb3d's tcgen05 implicit-GEMM kernel (NHWC fp32 activations, tf32 tensor cores).

Reference call sites: nn.Conv2d layers of /root/reference/code/models/gan.py (:57-65, :163-177, :294-302,
:359, :364) — 3x3 / 1x1 / 5x5 stride 1 and 4x4 stride 2, zero padding along y only (x padding is explicit:
replicate / circular pads are materialised by the caller exactly as the reference does)."""
import ctypes
import os

import torch

from . import B3DError, check, dev, last_variant, lib, ptr, stream_ptr

VARIANT_LOG = None      # tests set this to a list: every kernel template instance the conv entry points launch is appended


def _conv_call(fn, *args):
    """One convolution entry point of libb3d; records which kernel instances it launched when VARIANT_LOG is a list."""
    rc = fn(*args)
    if VARIANT_LOG is not None and rc == 0:
        VARIANT_LOG.extend(v for v in last_variant().split(";") if v)
    return rc


def _ints(v):
    return (ctypes.c_int * len(v))(*v)


def taps_layout(weight):
    """[Cout,Cin,kh,kw] -> tap-major K-major rows [kh*kw, Cout, Cin]."""
    co, ci, kh, kw = weight.shape
    return weight.permute(2, 3, 0, 1).reshape(kh * kw, co, ci).contiguous()


def _thin(Cout, Cin, kh, kw, stride):
    return Cout <= 4 and Cin % 64 == 0 and kh == 5 and kw == 5 and stride == 1 and not os.environ.get("B3D_NO_THIN")


def conv2d_nhwc(x, weight, bias=None, pad_y=0, stride=1, leaky=1.0, wt=None, cin_major=False, pad_out=0, pad_mode=1,
                x_crop=0):
    """x [N,H,W,Cin] (Cin % 32 == 0), weight [Cout,Cin,kh,kw] -> [N,Hout,Wout,Cout]; zero pad along y only.
    pad_out > 0: the result is written into the interior of a [N,Hout,Wout + 2*pad_out,Cout] buffer whose pad columns
    are then filled in place (replicate / circular) — the next convolution's padded input without a copy.
    x_crop > 0 (stride 1): convolve x[:, :, x_crop:W - x_crop] without materialising the slice (taps are shifted)."""
    x = dev(x, "x")
    N, H, W, Cin = x.shape
    Cout, Cin_w, kh, kw = weight.shape
    if Cin_w != Cin:
        raise B3DError(f"conv2d: input has {Cin} channels, weight expects {Cin_w}")
    if wt is None:
        wt = weight.permute(2, 3, 1, 0).reshape(kh * kw, Cin, Cout).contiguous() if cin_major else taps_layout(weight)
    wt = dev(wt, "weight")
    Hout = (H + 2 * pad_y - kh) // stride + 1
    if x_crop and stride != 1:
        raise B3DError("conv2d: x_crop needs stride 1")
    Wout = (W - 2 * x_crop - kw) // stride + 1
    OW = Wout + 2 * pad_out
    out = torch.empty(N, Hout, OW, Cout, device=x.device, dtype=torch.float32)
    optr = ctypes.c_void_p(out.data_ptr() + 4 * pad_out * Cout)          # pixel (n, y, pad_out) of the padded buffer
    if pad_out and Cout % 4:
        raise B3DError("conv2d: pad_out needs Cout % 4 == 0")
    wide_head = Wout >= 128 and N * Hout * (Wout // 128) >= 8 * 148 and not os.environ.get("B3D_THIN_HEAD_CUDA_CORES")
    if _thin(Cout, Cin, kh, kw, stride) and not cin_major and not wide_head:
        # 1-4 output channels: fp32 CUDA-core reduction kernel (csrc/thin_kernels.cu), not a 64-wide MMA tile
        # (wide heads — conv_final at 256 x 128 — take the row-window tensor-core kernel with N = 16 tiles instead)
        check(_conv_call(lib.b3d_conv2d_thin_fwd, ptr(x), ptr(wt), ptr(dev(bias, "bias") if bias is not None else None), optr, N, H, W,
                                      Cin, Hout, Wout, Cout, kh, kw, pad_y, x_crop, OW, Cout, float(leaky), stream_ptr(x)))
        if pad_out:
            check(lib.b3d_wrap_x_inplace(ptr(out), N * Hout, Wout, Cout, pad_out, pad_mode, stream_ptr(x)))
        return out
    dy = [r - pad_y for r in range(kh) for _ in range(kw)]
    dx = [s + x_crop for _ in range(kh) for s in range(kw)]
    b = dev(bias, "bias") if bias is not None else None
    # the halo-staged kernel wins on wide-N layers with enough tiles to fill the GPU twice; elsewhere the per-tap kernel
    # (2 CTAs / SM) is as fast or faster (profiles/r1_conv_layers.md)
    use_flat = stride == 1 and not cin_major and Cout > 64 and N * Hout * W >= 2 * 148 * 384 and not x_crop
    if os.environ.get("B3D_CONV_FLAT"):
        use_flat = stride == 1 and not cin_major and os.environ["B3D_CONV_FLAT"] == "1"
    if use_flat:
        # halo-staged kernel (tc_conv2.cu); falls through to the per-tap kernel when the halo does not fit in smem
        rc = _conv_call(lib.b3d_conv2d_flat_tf32, ptr(x), ptr(wt), ptr(b), optr, N, H, W, Cin, Hout, Wout, Cout, kh * kw,
                                      _ints(dy), _ints(dx), Hout, OW, Cout, float(leaky), stream_ptr(x))
        if rc != 0 and b"does not fit" not in lib.b3d_last_error():
            check(rc)
    if not use_flat or rc != 0:
        check(_conv_call(lib.b3d_conv2d_tf32, ptr(x), ptr(wt), ptr(b), optr, N, H, W, Cin, Hout, Wout, Cout, kh * kw, _ints(dy),
                                  _ints(dx), stride, stride, Hout, OW, Cout, 1, 1, 0, 0, float(leaky), int(cin_major), None, 0, None, 0, 0,
                                  None, stream_ptr(x)))
    if pad_out:
        check(lib.b3d_wrap_x_inplace(ptr(out), N * Hout, Wout, Cout, pad_out, pad_mode, stream_ptr(x)))
    return out


def stride2_classes(kh, kw, pad_y, H, W):
    """Output-parity decomposition of the input gradient of a stride-2 convolution (pure index arithmetic, unit-tested on
    the CPU): input pixel (y', x') = (2a + cy, 2b + cx) receives dY[a + dy_t, b + dx_t] * W[:, :, r_t, s_t] summed over the
    taps t of its class.  From y' = 2*yo + r - pad_y: only taps with (cy + pad_y - r) even take part, at yo = a + (cy +
    pad_y - r) / 2; likewise along x (no x padding: the input is pre-padded).  Returns one tuple per class:
    (cy, cx, [(r, s)], [dy], [dx], Ha, Wa) with Ha x Wa the number of input pixels of that parity."""
    out = []
    for cy in range(2):
        for cx in range(2):
            rs = [(r, s) for r in range(kh) for s in range(kw) if (cy + pad_y - r) % 2 == 0 and (cx - s) % 2 == 0]
            out.append((cy, cx, rs, [(cy + pad_y - r) // 2 for r, s in rs], [(cx - s) // 2 for r, s in rs],
                        (H - cy + 1) // 2, (W - cx + 1) // 2))
    return out


def conv2d_dgrad_nhwc(dy_, weight, in_hw, pad_y=0, stride=1, x_crop=0):
    """Gradient w.r.t. the (x-padded) input [N,H,W,Cin] of conv2d_nhwc, from dy_ [N,Hout,Wout,Cout] (Cout % 32 == 0)."""
    g = dev(dy_, "grad_output")
    N, Hout, Wout, Cout = g.shape
    Cout_w, Cin, kh, kw = weight.shape
    H, W = in_hw
    dxo = torch.empty(N, H, W, Cin, device=g.device, dtype=torch.float32)
    st = stream_ptr(g)
    if stride == 1:
        wt = weight.permute(2, 3, 1, 0).reshape(kh * kw, Cin, Cout).contiguous()        # [tap][Cin][Cout]
        dy = [pad_y - r for r in range(kh) for _ in range(kw)]
        dx = [-s - x_crop for _ in range(kh) for s in range(kw)]
        check(_conv_call(lib.b3d_conv2d_tf32, ptr(g), ptr(wt), None, ptr(dxo), N, Hout, Wout, Cout, H, W, Cin, kh * kw, _ints(dy),
                                  _ints(dx), 1, 1, H, W, Cin, 1, 1, 0, 0, 1.0, 0, None, 0, None, 0, 0, None, st))
        return dxo
    if stride != 2 or x_crop:
        raise B3DError("conv2d_dgrad: stride must be 1 or 2 (x_crop: stride 1 only)")
    for cy, cx, rs, dy, dx, Ha, Wa in stride2_classes(kh, kw, pad_y, H, W):
        if not rs:
            dxo[:, cy::2, cx::2] = 0
            continue
        wt = torch.stack([weight[:, :, r, s].t() for r, s in rs]).contiguous()      # [taps][Cin][Cout]
        check(_conv_call(lib.b3d_conv2d_tf32, ptr(g), ptr(wt), None, ptr(dxo), N, Hout, Wout, Cout, Ha, Wa, Cin, len(rs),
                                  _ints(dy), _ints(dx), 1, 1, H, W, Cin, 2, 2, cy, cx, 1.0, 0, None, 0, None, 0, 0, None, st))
    return dxo


def conv2d_wgrad_nhwc(dy_, x, kh, kw, pad_y=0, stride=1, x_crop=0):
    """dW [Cout,Cin,kh,kw] from dy_ [N,Hout,Wout,Cout] and the (x-padded) input x [N,H,W,Cin], both NHWC
    (channel counts that are not multiples of 32 are zero-padded here)."""
    co_real, ci_real = dy_.shape[3], x.shape[3]
    if _thin(co_real, ci_real, kh, kw, stride):
        g, x = dev(dy_, "grad_output"), dev(x, "input")
        N, Hout, Wout, _ = g.shape
        dw = torch.zeros(co_real, ci_real, kh, kw, device=g.device, dtype=torch.float32)
        check(_conv_call(lib.b3d_conv2d_thin_wgrad, ptr(g), ptr(x), ptr(dw), N, x.shape[1], x.shape[2], ci_real, Hout, Wout, co_real, kh, kw,
                                        pad_y, x_crop, 0, stream_ptr(g)))
        return dw
    g, x = dev(_pad_last(dy_, 32), "grad_output"), dev(_pad_last(x, 32), "input")
    N, Hout, Wout, Cout = g.shape
    _, H, W, Cin = x.shape
    dw = torch.zeros(Cout, Cin, kh, kw, device=g.device, dtype=torch.float32)
    check(_conv_call(lib.b3d_conv2d_wgrad_tf32, ptr(g), ptr(x), ptr(dw), N, H, W, Cin, Hout, Wout, Cout, kh, kw, pad_y, stride,
                                    x_crop, 0, 0, 0, stream_ptr(g)))
    return dw if (co_real, ci_real) == (Cout, Cin) else dw[:co_real, :ci_real]


# ------------------------------------------------------------------------------------------------------------------
# autograd: y = conv(x, w) + b on NHWC tensors; fprop / dgrad / wgrad all on the tcgen05 kernels
# ------------------------------------------------------------------------------------------------------------------
def _pad_last(t, mult):
    c = t.shape[-1]
    return t if c % mult == 0 else torch.nn.functional.pad(t, (0, mult - c % mult))


class _Conv2dNHWC(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, pad_y, stride, leaky=1.0, pad_out=0, pad_mode=1, x_crop=0):
        """pad_out > 0 (needs Cout = 4 * power of two): also applies the NEXT layer's x padding — the result is
        [N,Hout,Wout + 2*pad_out,Cout] — and the backward undoes padding, activation and bias in one fused pass."""
        x = dev(x.detach(), "x")
        w = weight.detach()
        Cin = x.shape[3]
        if Cin % 32:                                    # thin inputs (discriminator stems: 8 / 11 channels): zero-pad K
            x = _pad_last(x, 32)
            w = torch.nn.functional.pad(w, (0, 0, 0, 0, 0, x.shape[3] - Cin))
        y = conv2d_nhwc(x, w, bias.detach() if bias is not None else None, pad_y=pad_y, stride=stride, leaky=leaky,
                        pad_out=pad_out, pad_mode=pad_mode, x_crop=x_crop)
        if leaky != 1.0 or pad_out:
            ctx.save_for_backward(x, w, y)
        else:
            ctx.save_for_backward(x, w)
        ctx.cfg = (pad_y, stride, Cin, bias is not None, leaky, pad_out, pad_mode, x_crop)
        return y

    @staticmethod
    def backward(ctx, gy):
        pad_y, stride, Cin, has_bias, leaky, pad_out, pad_mode, x_crop = ctx.cfg
        gb = None
        want_gb = has_bias and ctx.needs_input_grad[2]
        if pad_out:                       # padding + LeakyReLU + bias gradient in one pass over the padded gradient
            x, w, y = ctx.saved_tensors
            gy = dev(gy, "grad_output")
            N, Ho, OW, Co = y.shape
            masked = torch.empty(N, Ho, OW - 2 * pad_out, Co, device=gy.device, dtype=torch.float32)
            gb = torch.zeros(Co, device=gy.device, dtype=torch.float32) if want_gb else None
            check(lib.b3d_pad_leaky_bias_bwd(ptr(gy), ptr(y), ptr(masked), ptr(gb), N * Ho, OW - 2 * pad_out, Co, pad_out,
                                             pad_mode, float(leaky), stream_ptr(gy)))
            gy = masked
        elif leaky != 1.0:                # LeakyReLU was fused into the epilogue: mask the incoming gradient by sign(y)
            x, w, y = ctx.saved_tensors
            gy = dev(gy, "grad_output")
            masked = torch.empty_like(gy)
            check(lib.b3d_leaky_bwd(ptr(gy), ptr(y), ptr(masked), gy.numel(), float(leaky), stream_ptr(gy)))
            gy = masked
        else:
            x, w = ctx.saved_tensors
        Cout, _, kh, kw = w.shape
        gy = dev(gy, "grad_output")
        if gb is None and want_gb:
            gb = gy.sum(dim=(0, 1, 2))
        gyp, wp = gy, w
        if Cout % 32:                                   # heads with 1 / 3 output channels: zero-pad the reduction dim
            gyp = _pad_last(gy, 32)
            wp = torch.nn.functional.pad(w, (0, 0, 0, 0, 0, 0, 0, gyp.shape[3] - Cout))
        gx = gw = None
        if ctx.needs_input_grad[0]:
            gx = conv2d_dgrad_nhwc(gyp, wp, (x.shape[1], x.shape[2]), pad_y=pad_y, stride=stride, x_crop=x_crop)[..., :Cin]
        if ctx.needs_input_grad[1]:
            gw = conv2d_wgrad_nhwc(gy if _thin(Cout, x.shape[3], kh, kw, stride) else gyp, x, kh, kw, pad_y=pad_y,
                                   stride=stride, x_crop=x_crop)[:Cout, :Cin]
        return gx, gw, gb, None, None, None, None, None, None


def fold_kh_weight(weight, cpad=0):
    """[Cout,Cin,kh,kw] -> [Cout, kh*Cin + cpad, 1, kw] matching fold_rows: channel r*Cin + c of the folded input is
    row tap r of input channel c (pure torch; unit-tested on the CPU against the unfolded convolution)."""
    Cout, Cin, kh, kw = weight.shape
    w = weight.permute(0, 2, 1, 3).reshape(Cout, kh * Cin, 1, kw)
    return torch.nn.functional.pad(w, (0, 0, 0, 0, 0, cpad)) if cpad else w


_FOLD = os.environ.get("B3D_FOLD", "kh")


def conv2d(x_nchw, weight, bias=None, pad_y=0, stride=1, leaky=1.0, pad_out=0, pad_mode=1, x_crop=0):
    """Drop-in for F.conv2d(x, w, b, stride, padding=(pad_y, 0)) on logically-NCHW tensors: runs on the tcgen05
    kernels over the channels-last storage (a no-copy view when x is already channels_last) and returns a
    logically-NCHW, channels-last tensor."""
    x = x_nchw.permute(0, 2, 3, 1)
    Cout, Cin, kh, kw = weight.shape
    if stride == 1 and kh > 1 and Cin * kh <= 64 and _FOLD == "kh":
        # thin stems (discriminator conv1: 8 or 11 input channels, 5x5): fold the kh vertical taps into the channel
        # dimension — X'[n,y,x, r*Cin + c] = X[n, y+r-pad_y, x, c] (zero rows = the y padding) — so the tensor cores see
        # kw taps of kh*Cin real channels instead of kh*kw taps of Cin channels zero-padded to 32.  The remaining taps
        # are horizontal: the weight-gradient kernel covers a whole row of taps per CTA (one pass over dY and X').
        from .ew import fold_rows
        cpad = (-kh * Cin) % 32                            # ... and round up to the 32-channel K slice in the same pass
        x = fold_rows(x, kh, pad_y, kh * Cin + cpad)
        weight = fold_kh_weight(weight, cpad)
        pad_y = 0
    elif stride == 1 and kw > 1 and Cin * kw <= 64:
        # same fold along x (B3D_FOLD=kw): X'[n,y,x, s*Cin + c] = X[n,y,x+s,c], kh vertical taps remain
        Wout = x.shape[2] - kw + 1
        cpad = (-kw * Cin) % 32
        parts = [x[:, :, s:s + Wout, :] for s in range(kw)]
        if cpad:
            parts.append(x.new_zeros(x.shape[0], x.shape[1], Wout, cpad))
        x = torch.cat(parts, dim=3)
        weight = weight.permute(0, 3, 1, 2).reshape(Cout, kw * Cin, kh, 1)          # [co, s*Cin + c, r, 0]
        if cpad:
            weight = torch.nn.functional.pad(weight, (0, 0, 0, 0, 0, cpad))
    y = _Conv2dNHWC.apply(x, weight, bias, int(pad_y), int(stride), float(leaky), int(pad_out), int(pad_mode), int(x_crop))
    return y.permute(0, 3, 1, 2)


# ------------------------------------------------------------------------------------------------------------------
# Banked convolution: the weights arrive from b3d.bank.WeightBank already normalised and laid out for the kernels
# (F [T'][Cout][Cin'] for fprop, D [T'][Cin'][Cout'] for the input gradient); the weight gradient is accumulated
# straight into the bank's F-layout gradient sink.  No per-call permute / contiguous / zeros.
# ------------------------------------------------------------------------------------------------------------------
class _ConvOpts(ctypes.Structure):
    """b3d_conv_opts (include/b3d.h)."""
    _fields_ = [("mask", ctypes.c_void_p), ("mask_slope", ctypes.c_float), ("stats_sum_only", ctypes.c_int),
                ("x_row_pitch", ctypes.c_int), ("nclass", ctypes.c_int), ("class_ooy", ctypes.c_int * 4), ("class_oox", ctypes.c_int * 4)]


class ActLink:
    """Hand-over between two chained banked convolutions  conv_L -> bias -> LeakyReLU -> x padding -> conv_L+1  (the
    discriminators, models/gan.py:163-177,294-302) for the backward pass.  The producer (conv_L, `link_out`) records its
    padded output; the consumer (conv_L+1, `link_in`), whose saved input IS that tensor, runs its input-gradient kernels
    with the LeakyReLU adjoint in their epilogue (mask = the activated tensor), folds the pad columns back
    (b3d_wrap_x_bwd_inplace) and leaves the bias gradient here — the producer's backward then reads the interior of the
    padded gradient in place (row-pitch tensor maps) instead of running b3d_pad_leaky_bias_bwd over it.
    Only valid when conv_L+1 is the ONLY consumer of conv_L's output: the caller creates a link exactly then."""
    __slots__ = ("armed", "slope", "pad", "mode", "ptr", "shape", "want_gb", "gb", "done")

    def __init__(self):
        self.armed = self.done = False
        self.gb = None


class _ConvBanked(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, wf, bias, lw, pad_y, stride, leaky, pad_out, pad_mode, x_crop, stats=None, fold_raw=0, link_in=None,
                link_out=None):
        """fold_raw = kh > 0: x is the RAW 8-channel stem input [N,H,W,8]; the kernels fold the kh vertical taps into the K
        dimension on the fly (TMA boxes of 4 rows x 8 channels) — the folded tensor never exists (pad_y = the fold's y padding)."""
        x = dev(x.detach(), "x")
        N, H, W, Cx = x.shape
        fold_pad = 0
        if fold_raw:
            if not lw.fold or Cx != 8 or lw.Cin != 8 or stride != 1 or x_crop:
                raise B3DError("banked conv: on-the-fly fold needs a folded 8-channel stride-1 stem")
            fold_pad = pad_y
        elif Cx != lw.Cinp:
            if lw.fold or Cx > lw.Cinp:
                raise B3DError(f"banked conv: input has {Cx} channels, the layer expects {lw.Cinp}")
            x = _pad_last(x, 32)                                      # thin un-folded inputs (512^2 stem): zero-pad K
        kh, kw = (1, lw.kw) if lw.fold else (lw.kh, lw.kw)
        if lw.fold:
            pad_y = 0
        Cout, Cin = lw.Cout, lw.Cinp
        wt = dev(wf.detach(), "weight")
        b = dev(bias.detach(), "bias") if bias is not None else None
        Hout = (H + 2 * fold_pad - lw.kh + 1) if fold_raw else (H + 2 * pad_y - kh) // stride + 1
        if x_crop and stride != 1:
            raise B3DError("conv2d: x_crop needs stride 1")
        Wout = (W - 2 * x_crop - kw) // stride + 1
        OW = Wout + 2 * pad_out
        if pad_out and Cout % 4:
            raise B3DError("conv2d: pad_out needs Cout % 4 == 0")
        out = torch.empty(N, Hout, OW, Cout, device=x.device, dtype=torch.float32)
        optr = ctypes.c_void_p(out.data_ptr() + 4 * pad_out * Cout)
        st = stream_ptr(x)
        thin = _thin(Cout, Cin, kh, kw, stride)
        # wide thin heads (conv_final: 64 -> 3 at 256 x 128) go to the row-window tensor-core kernel with N = 16 tiles
        thin_fwd = thin and not (Wout >= 128 and N * Hout * (Wout // 128) >= 8 * 148 and not os.environ.get("B3D_THIN_HEAD_CUDA_CORES"))
        if thin_fwd:
            check(_conv_call(lib.b3d_conv2d_thin_fwd, ptr(x), ptr(wt), ptr(b), optr, N, H, W, Cin, Hout, Wout, Cout, kh, kw, pad_y,
                             x_crop, OW, Cout, float(leaky), st))
        else:
            dy = [r - pad_y for r in range(kh) for _ in range(kw)]
            dx = [s + x_crop for _ in range(kh) for s in range(kw)]
            use_flat = stride == 1 and Cout > 64 and N * Hout * W >= 2 * 148 * 384 and not x_crop and not fold_raw
            if os.environ.get("B3D_CONV_FLAT"):
                use_flat = stride == 1 and os.environ["B3D_CONV_FLAT"] == "1" and not fold_raw
            if stats is not None:                 # the statistics epilogue lives in the persistent / row-window kernels
                use_flat = False
                if bias is not None or leaky != 1.0 or stride != 1:
                    raise B3DError("banked conv: output statistics are taken before bias / activation (plain stride-1 convs only)")
            rc = -1
            if use_flat:
                rc = _conv_call(lib.b3d_conv2d_flat_tf32, ptr(x), ptr(wt), ptr(b), optr, N, H, W, Cin, Hout, Wout, Cout, kh * kw,
                                _ints(dy), _ints(dx), Hout, OW, Cout, float(leaky), st)
                if rc != 0 and b"does not fit" not in lib.b3d_last_error():
                    check(rc)
            if rc != 0:
                check(_conv_call(lib.b3d_conv2d_tf32, ptr(x), ptr(wt), ptr(b), optr, N, H, W, Cin, Hout, Wout, Cout, kh * kw,
                                 _ints(dy), _ints(dx), stride, stride, Hout, OW, Cout, 1, 1, 0, 0, float(leaky), 0, None, 0, ptr(stats),
                                 fold_raw, fold_pad, None, st))
        if pad_out:
            check(lib.b3d_wrap_x_inplace(ptr(out), N * Hout, Wout, Cout, pad_out, pad_mode, st))
        ctx.save_for_backward(x, out if (leaky != 1.0 or pad_out) else None)
        ctx.lw = lw
        ctx.cfg = (pad_y, stride, Cx, bias is not None, leaky, pad_out, pad_mode, x_crop, kh, kw, thin, fold_raw, fold_pad)
        # chained activation adjoint (ActLink): usable as a consumer when x is exactly the producer's padded output
        ctx.link_in = link_in if (link_in is not None and link_in.armed and link_in.ptr == x.data_ptr() and link_in.shape == tuple(x.shape)
                                  and Cx == Cin and Cin % 32 == 0 and not fold_raw and not thin) else None
        ctx.link_out = None
        if link_out is not None and pad_out and leaky != 1.0 and Cout % 32 == 0 and not thin:
            link_out.armed, link_out.slope, link_out.pad, link_out.mode = True, float(leaky), int(pad_out), int(pad_mode)
            link_out.ptr, link_out.shape, link_out.done = out.data_ptr(), tuple(out.shape), False
            link_out.want_gb = bias is not None and bool(ctx.needs_input_grad[2])     # frozen discriminator (generator step): no bias sums
            ctx.link_out = link_out
        return out

    @staticmethod
    def backward(ctx, gy):
        x, y = ctx.saved_tensors
        lw = ctx.lw
        pad_y, stride, Cx, has_bias, leaky, pad_out, pad_mode, x_crop, kh, kw, thin, fold_raw, fold_pad = ctx.cfg
        Cout, Cin = lw.Cout, lw.Cinp
        N, H, W, _ = x.shape
        gy = dev(gy, "grad_output")
        st = stream_ptr(gy)
        gb = None
        want_gb = has_bias and ctx.needs_input_grad[2]
        g_pitch, g_off = 0, 0                                          # gy as a window of wider rows (pixels): pitch, first column
        link_out = ctx.link_out
        if link_out is not None and link_out.done:
            # the consumer's input-gradient epilogue already applied LeakyReLU', folded the pad columns and summed the bias
            # gradient: gy is the PADDED gradient [N,Ho,Wo + 2 pad,C]; its interior is read in place
            link_out.done = False
            if tuple(gy.shape) != tuple(y.shape):
                raise B3DError("banked conv: chained gradient has the wrong shape")
            g_pitch, g_off = y.shape[2], pad_out
            gb = link_out.gb if want_gb else None
            link_out.gb = None
            gy = gy[:, :, pad_out:y.shape[2] - pad_out]                # a view: shapes below are the interior's
        elif pad_out:
            _, Ho, OW, _ = y.shape
            masked = torch.empty(N, Ho, OW - 2 * pad_out, Cout, device=gy.device, dtype=torch.float32)
            gb = torch.zeros(Cout, device=gy.device, dtype=torch.float32) if want_gb else None
            check(lib.b3d_pad_leaky_bias_bwd(ptr(gy), ptr(y), ptr(masked), ptr(gb), N * Ho, OW - 2 * pad_out, Cout, pad_out,
                                             pad_mode, float(leaky), st))
            gy = masked
        elif leaky != 1.0:
            masked = torch.empty_like(gy)
            check(lib.b3d_leaky_bwd(ptr(gy), ptr(y), ptr(masked), gy.numel(), float(leaky), st))
            gy = masked
        if gb is None and want_gb:
            gb = gy.sum(dim=(0, 1, 2))
        _, Hout, Wout, _ = gy.shape
        gx = gw = None
        if ctx.needs_input_grad[0]:
            if lw.wd is None:
                raise B3DError("banked conv: this layer was registered without an input gradient (no_dgrad)")
            gyp = gy if g_pitch else _pad_last(gy, 32)                 # heads with 1 / 3 output channels: zero-pad K
            gptr = ctypes.c_void_p(gy.data_ptr()) if g_pitch else ptr(gyp)     # (the view's data_ptr = first interior pixel)
            Cop = lw.Coutp
            Hraw = H
            if fold_raw:
                H = Hout                                               # gradient w.r.t. the (virtual) folded tensor [N, Hout, W, Cin]
            gx = torch.empty(N, H, W, Cin, device=gy.device, dtype=torch.float32)
            wd = lw.wd
            link_in = ctx.link_in if (stride == 1 or (stride == 2 and not x_crop)) else None
            opts, sums = None, None
            classes = stride2_classes(kh, kw, pad_y, H, W) if (stride == 2 and not x_crop) else []
            # one launch for the four parity classes when they have the same extent and tap count (even H, W; 4x4 kernels)
            merged = (len(classes) == 4 and all(c[2] for c in classes) and len({(len(c[2]), c[5], c[6]) for c in classes}) == 1
                      and not os.environ.get("B3D_DGRAD_PER_CLASS"))
            if g_pitch or link_in is not None or merged:
                opts = _ConvOpts(None, 1.0, 0, g_pitch, 0)
                if link_in is not None:                                # LeakyReLU adjoint of the PRODUCER of x in this epilogue
                    if link_in.want_gb:
                        sums = torch.zeros(2 * Cin, device=gy.device, dtype=torch.float64)
                    opts.mask, opts.mask_slope, opts.stats_sum_only = x.data_ptr(), link_in.slope, 1
            optr_ = ctypes.cast(ctypes.pointer(opts), ctypes.c_void_p) if opts is not None else None
            if stride == 1:
                dy = [pad_y - r for r in range(kh) for _ in range(kw)]
                dx = [-s - x_crop for _ in range(kh) for s in range(kw)]
                check(_conv_call(lib.b3d_conv2d_tf32, gptr, ptr(wd), None, ptr(gx), N, Hout, Wout, Cop, H, W, Cin, kh * kw,
                                 _ints(dy), _ints(dx), 1, 1, H, W, Cin, 1, 1, 0, 0, 1.0, 0, None, 0, ptr(sums), 0, 0, optr_, st))
            elif merged:
                opts.nclass = 4
                for i, c in enumerate(classes):
                    opts.class_ooy[i], opts.class_oox[i] = c[0], c[1]
                dy = [v for c in classes for v in c[3]]
                dx = [v for c in classes for v in c[4]]
                taps = [r * kw + s for c in classes for r, s in c[2]]   # rows of the tap-major D array: no gathered copy
                check(_conv_call(lib.b3d_conv2d_tf32, gptr, ptr(wd), None, ptr(gx), N, Hout, Wout, Cop, classes[0][5], classes[0][6], Cin,
                                 len(taps), _ints(dy), _ints(dx), 1, 1, H, W, Cin, 2, 2, 0, 0, 1.0, 0, _ints(taps), kh * kw,
                                 ptr(sums), 0, 0, optr_, st))
            elif stride == 2 and not x_crop:
                for cy, cx, rs, dy, dx, Ha, Wa in classes:
                    if not rs:
                        gx[:, cy::2, cx::2] = 0
                        continue
                    taps = [r * kw + s for r, s in rs]                  # rows of the tap-major D array: no gathered copy
                    check(_conv_call(lib.b3d_conv2d_tf32, gptr, ptr(wd), None, ptr(gx), N, Hout, Wout, Cop, Ha, Wa, Cin,
                                     len(rs), _ints(dy), _ints(dx), 1, 1, H, W, Cin, 2, 2, cy, cx, 1.0, 0, _ints(taps), kh * kw,
                                     ptr(sums), 0, 0, optr_, st))
            else:
                raise B3DError("conv2d_dgrad: stride must be 1 or 2 (x_crop: stride 1 only)")
            if link_in is not None:
                # gx = LeakyReLU'(x) * d(padded input), pad columns included: fold them back, hand the bias gradient over
                check(lib.b3d_wrap_x_bwd_inplace(ptr(gx), N * H, W - 2 * link_in.pad, Cin, link_in.pad, link_in.mode, st))
                link_in.gb = sums[:Cin].float() if sums is not None else None
                link_in.done = True
            if fold_raw:                                               # adjoint of the fold: back to the raw 8-channel layout
                graw = torch.empty(N, Hraw, W, Cx, device=gy.device, dtype=torch.float32)
                check(lib.b3d_fold_rows_bwd(ptr(gx), ptr(graw), N, Hraw, W, Cx, lw.kh, fold_pad, Cin, st))
                gx, H = graw, Hraw
            elif Cx != Cin:
                gx = gx[..., :Cx]
        if ctx.needs_input_grad[1]:
            gw = lw.df                                                 # the bank's gradient sink (zeroed by the bank)
            if gw is None:
                raise B3DError("banked conv: weight gradient requested but the bank was run without gradients")
            if thin:
                check(_conv_call(lib.b3d_conv2d_thin_wgrad, ptr(gy), ptr(x), ptr(gw), N, H, W, Cin, Hout, Wout, Cout, kh, kw, pad_y,
                                 x_crop, 1, st))
            else:
                if Cout % 32:
                    raise B3DError(f"banked conv: weight gradient needs Cout % 32 == 0 or a thin head (Cout={Cout})")
                if fold_raw:
                    raise B3DError("banked conv: the on-the-fly fold has no weight-gradient kernel (materialise the fold)")
                check(_conv_call(lib.b3d_conv2d_wgrad_tf32, ctypes.c_void_p(gy.data_ptr()), ptr(x), ptr(gw), N, H, W, Cin, Hout, Wout,
                                 Cout, kh, kw, pad_y, stride, x_crop, 1, 0, g_pitch, st))
        return gx, gw, gb, None, None, None, None, None, None, None, None, None, None, None


def conv2d_banked(x_nchw, lw, pad_y=0, stride=1, leaky=1.0, pad_out=0, pad_mode=1, x_crop=0, stats=None, link_in=None, link_out=None):
    """conv2d for a layer whose weights come from a WeightBank (`lw` = its LayerWeights).  Thin stems registered with
    fold=True get their kh taps folded into the channels here (b3d.ew.fold_rows), as in conv2d().
    stats: optional zeroed fp64 tensor [2*Cout]; the conv epilogue accumulates the output's per-channel sum / sum of
    squares into it (the following batch norm's statistics without another pass over the tensor)."""
    x = x_nchw.permute(0, 2, 3, 1)
    fold_raw = 0
    if lw.fold:
        Wout = x.shape[2] - lw.kw + 1
        need_wgrad = torch.is_grad_enabled() and lw.wf.requires_grad
        if (lw.Cin == 8 and stride == 1 and not x_crop and Wout % 128 == 0 and x.shape[0] * x.shape[1] * (Wout // 128) >= 2 * 148
                and not need_wgrad and not os.environ.get("B3D_FOLD_MATERIALIZE")):
            # 8-channel stems of wide images when no weight gradient is taken (generator step: the discriminator is frozen):
            # the forward kernel folds the kh rows on the fly (TMA boxes of 4 rows x 8 channels), no folded tensor is written.
            # Same-box A/B inside the step graph: 41.21 ms with it, 41.45 ms with the materialised fold (B3D_FOLD_MATERIALIZE=1)
            # — although a cold-cache ncu launch of the 32-byte-swizzle kernel alone looks slower than fold + conv.
            fold_raw = lw.kh
        else:
            from .ew import fold_rows
            x = fold_rows(x, lw.kh, pad_y, lw.Cinp)
    y = _ConvBanked.apply(x, lw.wf, lw.bias, lw, int(pad_y), int(stride), float(leaky), int(pad_out), int(pad_mode), int(x_crop), stats,
                          fold_raw, link_in, link_out)
    return y.permute(0, 3, 1, 2)


# ------------------------------------------------------------------------------------------------------------------
# Up-convolution: conv3x3(up2(x)) (zero padding in y, x padding already in the input) run on x itself.  Every 2x2 block of
# the nearest-upsampled tensor holds one value, so output pixel (2i+a, 2j+b) is a 2x2 convolution of x with the class taps
# K_ab = A_a W A_b^T (A_0 = [[1,0,0],[0,1,1]], A_1 = [[1,1,0],[0,0,1]]; the bank's `up2` layouts): 4 MACs per output pixel
# and input channel instead of 9.  With x replicate-padded by one column, up2 of it is the replicate-padded up2(x), so the
# padded low-resolution tensor stands in for the padded upsampled one.
# ------------------------------------------------------------------------------------------------------------------
def upconv_taps():
    """Tap lists of the up-convolution, tap t = ((a*2 + b)*2 + u)*2 + v (class (a, b), class tap (u, v)), in the pixel
    coordinates of b3d_conv2d_tf32 (pure index arithmetic, unit-tested on the CPU):
      forward  Y[2i+a, 2j+b]  += K_ab[u][v] . Xp[i + a-1+u, j + b+v]       (Xp: x padded by one column, zero rows outside)
      dgrad    dXp[i, j]      += K_ab[u][v]^T . dY[2i + 2-a-2u, 2j - b-2v]  (input stride 2, zeros outside dY)
    The weight gradient runs b3d_conv2d_wgrad_tf32 with the operands swapped (Xp as "dy", dY as the stride-2 "x", kh = kw =
    4, pad_y = 1, x_off = -3): its tap (R, S) = (3-a-2u, 3-b-2v) is dK_ab[u][v]^T.  -> (classes, fdy, fdx, ddy, ddx)."""
    classes = [(a, b) for a in range(2) for b in range(2)]
    t = [(a, b, u, v) for a, b in classes for u in range(2) for v in range(2)]
    return (classes, [a - 1 + u for a, b, u, v in t], [b + v for a, b, u, v in t], [2 - a - 2 * u for a, b, u, v in t],
            [-b - 2 * v for a, b, u, v in t])


_UPCONV = upconv_taps()


class _UpConvBanked(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, wf, lw, stats):
        """x [N,H,W+2,Cin] (replicate-padded by one column) -> conv3x3(up2(x)) [N,2H,2W,Cout]; stats as conv2d_banked's."""
        x = dev(x.detach(), "x")
        N, H, Wp, Cin = x.shape
        if not lw.up2 or Cin != lw.Cinp or lw.Cout % 32:
            raise B3DError("upconv: the layer needs the bank's up2 class taps, Cin' input channels and Cout % 32 == 0")
        W, Cout = Wp - 2, lw.Cout
        classes, fdy, fdx, _, _ = _UPCONV
        out = torch.empty(N, 2 * H, 2 * W, Cout, device=x.device, dtype=torch.float32)
        opts = _ConvOpts(None, 1.0, 0, 0, 4)
        for i, (a, b) in enumerate(classes):
            opts.class_ooy[i], opts.class_oox[i] = a, b
        check(_conv_call(lib.b3d_conv2d_tf32, ptr(x), ptr(dev(lw.uf, "weight")), None, ptr(out), N, H, Wp, Cin, H, W, Cout, 16,
                         _ints(fdy), _ints(fdx), 1, 1, 2 * H, 2 * W, Cout, 2, 2, 0, 0, 1.0, 0, None, 0, ptr(stats), 0, 0,
                         ctypes.cast(ctypes.pointer(opts), ctypes.c_void_p), stream_ptr(x)))
        ctx.save_for_backward(x)
        ctx.lw = lw
        return out

    @staticmethod
    def backward(ctx, gy):
        x, = ctx.saved_tensors
        lw = ctx.lw
        N, H, Wp, Cin = x.shape
        Cout = lw.Cout
        gy = dev(gy, "grad_output")
        st = stream_ptr(gy)
        _, _, _, ddy, ddx = _UPCONV
        gx = gw = None
        if ctx.needs_input_grad[0]:
            gx = torch.empty(N, H, Wp, Cin, device=gy.device, dtype=torch.float32)
            check(_conv_call(lib.b3d_conv2d_tf32, ptr(gy), ptr(dev(lw.ud, "weight")), None, ptr(gx), N, 2 * H, 2 * (Wp - 2), Cout, H, Wp,
                             Cin, 16, _ints(ddy), _ints(ddx), 2, 2, H, Wp, Cin, 1, 1, 0, 0, 1.0, 0, None, 0, None, 0, 0, None, st))
        if ctx.needs_input_grad[1]:
            gw = lw.df                                                 # the bank's 3x3 gradient sink (zeroed by the bank)
            if gw is None:
                raise B3DError("upconv: weight gradient requested but the bank was run without gradients")
            dk = torch.zeros(16, Cin, Cout, device=gy.device, dtype=torch.float32)
            check(_conv_call(lib.b3d_conv2d_wgrad_tf32, ptr(x), ptr(gy), ptr(dk), N, 2 * H, 2 * (Wp - 2), Cout, H, Wp, Cin, 4, 4, 1, 2,
                             -3, 1, 0, 0, st))
            check(lib.b3d_bank_up2_grad(ptr(dk), ptr(gw), Cout, lw.Cin, lw.Cinp, st))
        return gx, gw, None, None


def upconv_banked(x_nchw, lw, stats=None):
    """conv2d_banked(up2(x), lw, pad_y=1) for a 3x3 layer the bank serves as `up2`, with x the replicate-padded input of the
    upsample (logically NCHW, channels-last) — the x4 tensor is never written."""
    y = _UpConvBanked.apply(x_nchw.permute(0, 2, 3, 1), lw.wf, lw, stats)
    return y.permute(0, 3, 1, 2)
