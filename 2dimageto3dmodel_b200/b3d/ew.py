"""One-pass NHWC helper ops between the convolutions (libb3d csrc/ew_kernels.cu), with autograd."""
import ctypes
import os

import torch

from . import B3DError, check, dev, lib, ptr, stream_ptr

REPLICATE, CIRCULAR = 0, 1


class _PadX(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x_nhwc, amount, mode):
        x = dev(x_nhwc.detach(), "x")
        N, H, W, C = x.shape
        out = torch.empty(N, H, W + 2 * amount, C, device=x.device, dtype=torch.float32)
        check(lib.b3d_pad_x_fwd(ptr(x), ptr(out), N * H, W, C, amount, mode, stream_ptr(x)))
        ctx.cfg = (amount, mode, x.shape)
        return out

    @staticmethod
    def backward(ctx, g):
        amount, mode, shape = ctx.cfg
        N, H, W, C = shape
        g = dev(g, "grad")
        gx = torch.empty(shape, device=g.device, dtype=torch.float32)
        check(lib.b3d_pad_x_bwd(ptr(g), ptr(gx), N * H, W, C, amount, mode, stream_ptr(g)))
        return gx, None, None


class _FoldRows(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x_nhwc, kh, pad_y, Cp):
        x = dev(x_nhwc.detach(), "x")
        N, H, W, C = x.shape
        out = torch.empty(N, H + 2 * pad_y - kh + 1, W, Cp, device=x.device, dtype=torch.float32)
        check(lib.b3d_fold_rows_fwd(ptr(x), ptr(out), N, H, W, C, kh, pad_y, Cp, stream_ptr(x)))
        ctx.cfg = (kh, pad_y, Cp, x.shape)
        return out

    @staticmethod
    def backward(ctx, g):
        kh, pad_y, Cp, shape = ctx.cfg
        N, H, W, C = shape
        g = dev(g, "grad")
        gx = torch.empty(shape, device=g.device, dtype=torch.float32)
        check(lib.b3d_fold_rows_bwd(ptr(g), ptr(gx), N, H, W, C, kh, pad_y, Cp, stream_ptr(g)))
        return gx, None, None, None


def fold_rows(x_nhwc, kh, pad_y, Cp):
    """[N,H,W,C] -> [N,H + 2*pad_y - kh + 1,W,Cp] with out[..., r*C + c] = x[n, y + r - pad_y, x, c] (zeros elsewhere)."""
    return _FoldRows.apply(x_nhwc, int(kh), int(pad_y), int(Cp))


class _StemInput(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x_nchw, pos, amount, mode):
        x = dev(x_nchw.detach(), "x")
        pos = dev(pos, "positions")
        N, C1, H, W = x.shape
        C2 = pos.shape[0]
        if tuple(pos.shape[1:]) != (H, W):
            raise B3DError(f"stem_input: positions {tuple(pos.shape)} do not match the image {tuple(x.shape)}")
        out = torch.empty(N, H, W + 2 * amount, C1 + C2, device=x.device, dtype=torch.float32)
        check(lib.b3d_stem_input_fwd(ptr(x), ptr(pos), ptr(out), N, C1, C2, H, W, amount, mode, stream_ptr(x)))
        ctx.cfg = (amount, mode, x.shape, C2)
        return out

    @staticmethod
    def backward(ctx, g):
        amount, mode, shape, C2 = ctx.cfg
        N, C1, H, W = shape
        g = dev(g, "grad")
        gx = torch.empty(shape, device=g.device, dtype=torch.float32)
        check(lib.b3d_stem_input_bwd(ptr(g), ptr(gx), N, C1, C2, H, W, amount, mode, stream_ptr(g)))
        return gx, None, None, None


def stem_input(x_nchw, pos, amount, mode):
    """pad_x(cat(x, pos broadcast over the batch), amount, mode) in one pass: x [N,C1,H,W] contiguous NCHW, pos [C2,H,W],
    C1 + C2 in (4, 8) -> logically-NCHW view of the NHWC tensor [N,H,W + 2*amount,C1 + C2] (what the convolutions read)."""
    return _StemInput.apply(x_nchw, pos, int(amount), int(mode)).permute(0, 3, 1, 2)


def pad_x(x_nchw, amount, mode):
    """Padding along x of a logically-NCHW (channels-last) tensor; returns the same kind of tensor."""
    if amount == 0:
        return x_nchw
    if x_nchw.shape[1] % 4:         # odd channel counts (raw RGBA+... inputs): plain torch
        if mode == REPLICATE:
            return torch.nn.functional.pad(x_nchw, (amount, amount, 0, 0), mode='replicate')
        return torch.cat((x_nchw[..., -amount:], x_nchw, x_nchw[..., :amount]), dim=3)
    return _PadX.apply(x_nchw.permute(0, 2, 3, 1), int(amount), int(mode)).permute(0, 3, 1, 2)


# ------------------------------------------------------------------------------------------------------------------
# fused conditional-batch-norm -> LeakyReLU -> (+ residual) -> (LeakyReLU) -> x2 nearest upsample -> replicate pad
# ------------------------------------------------------------------------------------------------------------------
def _dist_world():
    import torch.distributed as dist
    return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1


class CBNBatch:
    """fc_gamma / fc_beta of ALL ConditionalBatchNorm2d layers of a generator forward as one GEMM
    (models/gan.py:264-286: gamma = fc_gamma(z), beta = fc_beta(z) per layer): gb [N, 2*sum(C)], row n holds layer l's
    gamma at off[l] and beta at off[l] + C_l.  The layers' backward passes write d(gamma), d(beta) straight into one sink
    buffer of the same shape, handed to autograd once (by the layer that runs last in the backward = first in the forward;
    every other layer is downstream of it, so the data dependencies order this, not the scheduler)."""

    def __init__(self, cbns, z):
        self.offsets, off = {}, 0
        ws, bs = [], []
        for m in cbns:
            C = m.fc_gamma.out_features
            self.offsets[id(m)] = (off, off + C)
            off += 2 * C
            ws += [m.fc_gamma.weight, m.fc_beta.weight]
            bs += [m.fc_gamma.bias, m.fc_beta.bias]
        self.first = id(cbns[0])
        self.n_layers, self.done = len(cbns), 0
        self.gb = torch.nn.functional.linear(z, torch.cat(ws), torch.cat(bs))
        self.sink = None
        # fp64 [sum x | sum x^2] slots the conv epilogues accumulate into (one zero fill for all layers of the forward)
        self.stats = torch.zeros(off, device=z.device, dtype=torch.float64) if z.is_cuda else None

    def stats_slot(self, cbn):
        """The layer's zeroed statistics slot [2*C] (handed to the producing convolution), or None in eval mode."""
        if self.stats is None or not cbn.norm.training:
            return None
        goff, boff = self.offsets[id(cbn)]
        return self.stats[goff: goff + 2 * (boff - goff)]

    shared = False                                  # per-sample gamma / beta rows

    def grad_sink(self, N=None):
        if self.sink is None:
            self.sink = torch.empty_like(self.gb) if not self.shared else torch.empty(N, self.gb.shape[1], device=self.gb.device)
        return self.sink


class BNAffine(CBNBatch):
    """A plain BatchNorm2d (affine weight / bias shared by all samples; models/reconstruction.py:7-26, :52-64) expressed in
    the fused kernels' terms: one row gb = [weight - 1 | bias] read by every sample (row pitch 0); the per-sample
    d(gamma), d(beta) rows of the backward are summed over the batch."""
    shared = True

    def __init__(self, bn):
        C = bn.num_features
        self.offsets = {id(bn): (0, C)}
        self.first, self.n_layers, self.done = id(bn), 1, 0
        self.gb = torch.cat((bn.weight - 1, bn.bias)).view(1, 2 * C)
        self.sink, self.stats = None, None


class _CBNActPad(torch.autograd.Function):
    """y [N,H,W,C] (conv output, NHWC) -> out [N, up*H, up*W + 2*pad, C]; gb = CBNBatch.gb (gamma / beta of this layer at
    column offsets goff / boff).  `skip` (optional) [N,H,Ws,C] read at pixel offset skip_off; skip_half: [N,H/2,Ws,C] read at
    (y/2, x/2).  Statistics, running buffers
    and the per-sample affine come from one b3d_cbn_prepare launch (modes: 0 eval, 1 batch statistics, 2 SyncBN)."""

    @staticmethod
    def forward(ctx, y, gb, cb, key, bn, skip, skip_off, up, pad, post_leaky, sums_in=None, slope=0.2, skip_half=0):
        y = dev(y.detach(), "y")
        N, H, W, C = y.shape
        gbd = dev(gb.detach(), "gamma/beta")
        P = gbd.shape[1]
        gp = 0 if cb.shared else P                          # row pitch of gamma / beta (0: one row for all samples)
        goff, boff = cb.offsets[key]
        st = stream_ptr(y)
        mode, sums, count, sync, peers = 0, None, 1.0, False, None
        if bn.training:
            if sums_in is not None:                     # accumulated by the epilogue of the convolution that produced y
                sums = sums_in
            else:
                sums = torch.empty(2 * C, device=y.device, dtype=torch.float64)
                check(lib.b3d_bn_sums(ptr(y), N * H * W, C, ptr(sums), st))
            mode, count = 1, float(N * H * W)
            if _dist_world() > 1 and bn.__class__.__name__.startswith("Synchronized"):
                import torch.distributed as dist
                from .sync import peer_sync
                mode, count, sync = 2, count * dist.get_world_size(), True
                peers = peer_sync(y.device) if C <= 512 else None
                if peers is None:
                    dist.all_reduce(sums)                   # NCCL fallback: one collective per layer, [sum x, sum x^2] in fp64
        mean = torch.empty(C, device=y.device, dtype=torch.float32)
        invstd = torch.empty_like(mean)
        scale = torch.empty(N, C, device=y.device, dtype=torch.float32)
        shift, gt = torch.empty_like(scale), torch.empty_like(scale)
        track = bn.training and bn.track_running_stats
        if peers is not None:
            # statistics all-reduce over NVLink peer memory fused into the kernel that consumes them (csrc/ew_kernels.cu)
            check(lib.b3d_cbn_prepare_sync(peers.data, peers.flag, peers.rank, peers.world, ptr(peers.epoch), ptr(peers.err),
                                           ptr(gbd), gp, goff, boff, ptr(sums), count, float(bn.eps), float(bn.momentum or 0.0),
                                           ptr(bn.running_mean) if track else None, ptr(bn.running_var) if track else None,
                                           ptr(bn.num_batches_tracked) if track else None,
                                           ptr(mean), ptr(invstd), ptr(scale), ptr(shift), ptr(gt), N, C, st))
        else:
            check(lib.b3d_cbn_prepare(ptr(gbd), gp, goff, boff, ptr(sums), count, float(bn.eps), float(bn.momentum or 0.0), mode,
                                      ptr(bn.running_mean) if (track or mode == 0) else None,
                                      ptr(bn.running_var) if (track or mode == 0) else None,
                                      ptr(bn.num_batches_tracked) if track else None,
                                      ptr(mean), ptr(invstd), ptr(scale), ptr(shift), ptr(gt), N, C, st))
        sk = dev(skip.detach(), "skip") if skip is not None else None
        pitch = sk.shape[2] if sk is not None else 0
        out = torch.empty(N, up * H, up * W + 2 * pad, C, device=y.device, dtype=torch.float32)
        check(lib.b3d_cbn_act_fwd(ptr(y), ptr(scale), ptr(shift), ptr(sk), pitch, skip_off, ptr(out), N, H, W, C, up, pad, float(slope),
                                  int(post_leaky), int(skip_half), st))
        ctx.save_for_backward(y, gt, scale, shift, mean, invstd, sk if sk is not None else torch.empty(0))
        ctx.cb, ctx.key = cb, key
        ctx.cfg = (skip_off, up, pad, post_leaky, mode != 0, sync, count, sk is not None, skip.shape if skip is not None else None,
                   P, goff, boff, float(slope), int(skip_half))
        ctx.peers = peers
        return out

    @staticmethod
    def backward(ctx, gout):
        y, gt, scale, shift, mean, invstd, sk = ctx.saved_tensors
        skip_off, up, pad, post_leaky, batch_stats, sync, count, has_skip, skip_shape, P, goff, boff, slope, skip_half = ctx.cfg
        cb = ctx.cb
        N, H, W, C = y.shape
        gout = dev(gout, "grad")
        st = stream_ptr(y)
        ga = torch.empty_like(y)
        gskip, gpitch = None, 0
        if has_skip and ctx.needs_input_grad[5]:
            gpitch = skip_shape[2]
            dense = gpitch == W >> skip_half
            gskip = torch.empty(skip_shape, device=y.device) if dense else torch.zeros(skip_shape, device=y.device)
        want_gb = ctx.needs_input_grad[1]
        sink = cb.grad_sink(N) if want_gb else torch.empty(N, P, device=y.device)
        s1 = ctypes.c_void_p(sink.data_ptr() + 4 * boff)        # d beta  = sum ga
        s2 = ctypes.c_void_p(sink.data_ptr() + 4 * goff)        # d gamma = sum ga * xhat
        check(lib.b3d_cbn_act_bwd1(ptr(gout), ptr(y), ptr(scale), ptr(shift), ptr(sk) if has_skip else None,
                                   sk.shape[2] if has_skip else 0, skip_off, ptr(mean), ptr(invstd), ptr(ga), ptr(gskip), gpitch,
                                   skip_off, s1, s2, P, N, H, W, C, up, pad, slope, int(post_leaky), skip_half, st))
        inv_m = 0.0
        if batch_stats:
            red = torch.empty(2 * C, device=y.device, dtype=torch.float32)
            peers = ctx.peers
            if sync and peers is not None:
                check(lib.b3d_cbn_bwd_reduce_sync(peers.data, peers.flag, peers.rank, peers.world, ptr(peers.epoch), ptr(peers.err),
                                                  s1, s2, P, ptr(gt), ptr(red), N, C, st))
            else:
                check(lib.b3d_cbn_bwd_reduce(s1, s2, P, ptr(gt), ptr(red), N, C, st))
                if sync:
                    import torch.distributed as dist
                    dist.all_reduce(red)
            inv_m = 1.0 / count
        else:
            red = torch.zeros(2 * C, device=y.device, dtype=torch.float32)
        check(lib.b3d_cbn_act_bwd2(ptr(ga), ptr(y), ptr(gt), ptr(mean), ptr(invstd), ptr(red), ctypes.c_void_p(red.data_ptr() + 4 * C),
                                   inv_m, N, H, W, C, st))
        ggb = None
        if want_gb:
            cb.done += 1
            if ctx.key == cb.first:
                if cb.done != cb.n_layers:
                    raise RuntimeError(f"CBNBatch: {cb.done} of {cb.n_layers} layers ran their backward before the first layer's")
                ggb = sink.sum(dim=0, keepdim=True) if cb.shared else sink
        return ga, ggb, None, None, None, gskip, None, None, None, None, None, None, None


_BN_STATS_IMPL = os.environ.get("B3D_BN_STATS", "torch")


def bn_stats(y_nhwc, eps, impl=None):
    """(mean, invstd) per channel of an NHWC tensor = torch.batch_norm_stats on the NCHW view.  impl "b3d" = the one-pass
    libb3d kernel, "torch" = the stock op."""
    y = dev(y_nhwc, "y")
    C = y.shape[-1]
    if C % 4 or 256 % (C // 4) or (impl or _BN_STATS_IMPL) != "b3d":     # odd channel counts: always the stock op
        return torch.batch_norm_stats(y.permute(0, 3, 1, 2), eps)
    mean = torch.empty(C, device=y.device, dtype=torch.float32)
    invstd = torch.empty_like(mean)
    ws = torch.empty(2 * C, device=y.device, dtype=torch.float64)
    check(lib.b3d_bn_stats(ptr(y), y.numel() // C, C, float(eps), ptr(mean), ptr(invstd), ptr(ws), stream_ptr(y)))
    return mean, invstd


def bn_act_pad(y_nchw, bn, skip_nchw=None, skip_off=0, up=1, pad=1, post_relu=False, slope=0.0):
    """BatchNorm2d(y) (affine, batch or running statistics, SyncBN under torch.distributed) -> ReLU [-> + skip] [-> ReLU]
    [-> x2 nearest upsample] -> replicate pad in one pass (models/reconstruction.py:7-26 ResBlock glue), NHWC."""
    cb = BNAffine(bn)
    y = y_nchw.permute(0, 2, 3, 1)
    C = y.shape[3]
    if C % 4 or 256 % (C // 4):
        raise B3DError(f"bn_act_pad: C={C} must be 4 * a divisor of 256")
    skip = skip_nchw.permute(0, 2, 3, 1) if skip_nchw is not None else None
    out = _CBNActPad.apply(y, cb.gb, cb, id(bn), bn, skip, int(skip_off), int(up), int(pad), bool(post_relu), None, float(slope))
    return out.permute(0, 3, 1, 2)


def cbn_act_pad(y_nchw, cbn, z, skip_nchw=None, skip_off=0, up=1, pad=1, post_leaky=False, cb=None, sums=None, skip_half=False):
    """ConditionalBatchNorm2d(y, z) -> LeakyReLU(0.2) [-> + skip] [-> LeakyReLU] [-> x2 upsample] -> replicate pad, fused.
    skip_half: the skip is at half y's resolution and is added as its x2 nearest upsample.
    `cbn` is a models.gan.ConditionalBatchNorm2d whose .norm is a (Synchronized)BatchNorm2d without affine; statistics and
    running buffers follow F.batch_norm (single process) or the reference's SyncBN formulas (torch.distributed).
    cb: the forward's CBNBatch (gamma / beta of all layers from one GEMM); None = a one-layer batch built here."""
    if cb is None:
        cb = CBNBatch([cbn], z)
    y = y_nchw.permute(0, 2, 3, 1)
    C = y.shape[3]
    if C % 4 or 256 % (C // 4):
        raise B3DError(f"cbn_act_pad: C={C} must be 4 * a divisor of 256")
    skip = skip_nchw.permute(0, 2, 3, 1) if skip_nchw is not None else None
    out = _CBNActPad.apply(y, cb.gb, cb, id(cbn), cbn.norm, skip, int(skip_off), int(up), int(pad), bool(post_leaky), sums, 0.2,
                           int(bool(skip_half)))
    return out.permute(0, 3, 1, 2)
