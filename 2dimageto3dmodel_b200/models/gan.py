"""Drop-in for /root/reference/code/models/gan.py: the conv-GAN texture/mesh generator and the multi-scale
discriminators, with every nn.Conv2d running on libb3d's tcgen05 / TMA implicit-GEMM kernels
(csrc/tc_conv.cu: fprop, dgrad, wgrad; tf32 inputs, fp32 accumulate).

Module tree, parameter and buffer names equal the reference's, so its checkpoints load with strict=True
(`blk1.conv1.weight_orig / weight_u / weight_v`, `blk1.norm1.norm.running_mean`, `blk1.norm1.fc_gamma.weight`,
`emb_class.weight`, `fc.weight`, ... — SURVEY.md §8b).  Spectral normalisation is torch's own
nn.utils.spectral_norm hook (parameter plumbing, one mat-vec per layer), as in the reference.
Activations stay logically NCHW (the reference's interface) and physically channels-last, which is what the
kernels read; x-padding (replicate for the symmetric generator, circular for the discriminators) is explicit
as in the reference, y-padding is the convolution's zero padding (TMA out-of-bounds fill).
"""
import math
import os

import torch
import torch.nn as nn
import torch.nn.functional as F

from b3d import B3DError
from b3d.bank import WeightBank
from b3d.conv import conv2d as _tc_conv2d
from b3d.conv import ActLink, conv2d_banked, upconv_banked
from b3d.ew import CIRCULAR, REPLICATE, CBNBatch, cbn_act_pad, pad_x, stem_input
from rendering.utils import adjust_poles, symmetrize_texture


class TCConv2d(nn.Conv2d):
    """nn.Conv2d (same parameters / state dict) whose forward runs on the tensor-core kernels."""

    def forward(self, x, leaky=1.0, pad_out=0, pad_mode=CIRCULAR, x_crop=0):
        """`leaky` != 1 fuses LeakyReLU(leaky) into the convolution's epilogue (conv -> bias -> activation in one pass);
        `pad_out` > 0 also applies the next layer's x padding (the epilogue writes into the padded buffer)."""
        if not x.is_cuda:
            raise B3DError("models.gan convolutions run on CUDA only (libb3d tcgen05 kernels); there is no CPU fallback")
        if self.stride[0] != self.stride[1] or self.dilation != (1, 1) or self.groups != 1 or self.padding_mode != 'zeros':
            raise B3DError("TCConv2d supports zero padding, square strides, no dilation / groups")
        if self.padding[1] != 0:          # the kernels zero-pad along y (TMA fill); zero padding along x is materialised
            x = F.pad(x, (self.padding[1], self.padding[1], 0, 0))
        return _tc_conv2d(x, self.weight, self.bias, pad_y=self.padding[0], stride=self.stride[0], leaky=leaky,
                          pad_out=pad_out, pad_mode=pad_mode, x_crop=x_crop)


def positional_encoding(Ny, Nx):
    """[4, Ny, Nx] = cos/sin of the latitude (rows, 0..pi) and of the longitude (columns, -pi..pi, wrapping
    smoothly); for a half-width (symmetric) map only the central half of the longitudes is kept (reference :9-20)."""
    half = (Nx == Ny // 2)
    lat = torch.arange(Ny, dtype=torch.float64) * (math.pi / Ny)
    lon = -math.pi + torch.arange(Ny, dtype=torch.float64) * (2 * math.pi / Ny)
    rows, cols = lat.view(Ny, 1).expand(Ny, Ny), lon.view(1, Ny).expand(Ny, Ny)
    enc = torch.stack((rows.cos(), rows.sin(), cols.cos(), cols.sin()))
    if half:
        enc = enc[:, :, Ny // 4: Ny - Ny // 4]
    return enc.numpy()


def _norm_and_bias(args):
    if args.norm_d == 'instance':
        return (lambda ch: nn.InstanceNorm2d(ch, affine=True)), False
    if args.norm_d == 'none':
        return (lambda ch: None), True          # no norm layer: conv -> bias -> LeakyReLU runs in the conv epilogue
    raise ValueError(f"norm_d={args.norm_d!r}")


def _conv_norm_act(conv, norm, x, pad_next=0, lw=None, link_in=None, link_out=None):
    """pad_x(LeakyReLU(0.2)(norm(conv(x))), pad_next, circular): one fused kernel when there is no norm layer.
    lw: the layer's weights from the network's WeightBank (spectral norm + kernel layouts done for all layers at once);
    None = the module's own forward (torch's spectral-norm hook).
    link_in / link_out (b3d.conv.ActLink, banked layers only): this layer's input is the sole use of the previous layer's
    padded output / this layer's padded output has exactly one consumer, the next convolution — the backward pass then
    applies LeakyReLU', the padding's adjoint and the bias sum in the consumer's input-gradient epilogue."""
    if lw is not None:
        run = lambda **kw: conv2d_banked(x, lw, pad_y=conv.padding[0], stride=conv.stride[0], link_in=link_in, **kw)
    else:
        run = lambda **kw: conv(x, **kw)
    if norm is None and conv.out_channels in (16, 32, 64, 128, 256, 512, 1024):
        if lw is not None and pad_next:
            return run(leaky=0.2, pad_out=pad_next, pad_mode=CIRCULAR, link_out=link_out)
        return run(leaky=0.2, pad_out=pad_next, pad_mode=CIRCULAR)
    y = run(leaky=0.2) if norm is None else F.leaky_relu(norm(run()), 0.2)
    return pad_x(y, pad_next, CIRCULAR) if pad_next else y


def _head(conv, x, lw):
    return conv(x) if lw is None else conv2d_banked(x, lw, pad_y=conv.padding[0], stride=conv.stride[0])


def _bankable(m):
    """Layers a WeightBank can serve: circular variant (no zero padding along x), unit dilation / groups."""
    return isinstance(m, TCConv2d) and m.padding[1] == 0 and m.dilation == (1, 1) and m.groups == 1 and m.stride[0] == m.stride[1]


class _DiscriminatorBase(nn.Module):
    """Shared pieces of the two discriminators: wrap-around padding, positional channels, projection head."""

    def _setup(self, args, circular, positional_embeddings):
        self.args = args
        self.circular = circular
        self.positional_embeddings = positional_embeddings
        if circular:
            self.pad = lambda x: pad_x(x, 2, CIRCULAR)       # in front of the 5x5 convolutions
            self.pad2 = lambda x: pad_x(x, 1, CIRCULAR)      # in front of the 4x4 / stride-2 convolutions
        else:
            self.pad = lambda x: x
        if positional_embeddings:
            self.pos_emb = None

    def _positions(self, x):
        """[1,4,H,W] positional channels on x's device (computed for the first input's size, uploaded once)."""
        if self.pos_emb is None:
            self.pos_emb = torch.FloatTensor(positional_encoding(x.shape[2], x.shape[3])).unsqueeze(0)
        dev_copy = getattr(self, '_pos_emb_dev', None)
        if dev_copy is None or dev_copy.device != x.device:
            dev_copy = self._pos_emb_dev = self.pos_emb.to(x.device)
        return dev_copy

    def _with_positions(self, x, extra=()):
        parts = [x, *extra]
        if self.positional_embeddings:
            parts.append(self._positions(x).expand(x.shape[0], -1, -1, -1))
        return torch.cat(parts, dim=1) if len(parts) > 1 else x

    def _stem_input(self, x, amount):
        """pad_x(_with_positions(x), amount, circular) — as one kernel (b3d.ew.stem_input) for the 4 + 4 channel texture stems."""
        if (self.circular and self.positional_embeddings and x.is_cuda and x.dtype == torch.float32 and x.shape[1] == 4
                and not getattr(self, 'disable_stem_input', False)):
            pos = self._positions(x)[0]
            if tuple(pos.shape[1:]) == tuple(x.shape[2:]):
                return stem_input(x.contiguous(), pos, amount, CIRCULAR)
        x = self._with_positions(x)
        return pad_x(x, amount, CIRCULAR) if self.circular else x

    def _links(self, n, W):
        """ActLinks for the first n conv -> conv hand-overs of the stack (the last padded activation also feeds the
        projection, so it keeps the stand-alone backward pass)."""
        on = bool(W) and self.circular and not getattr(self, 'disable_act_chain', False) and not os.environ.get("B3D_NO_ACT_CHAIN")
        return [ActLink() if on else None for _ in range(n)]

    def _project(self, y, feat, c, caption):
        a = self.args
        if a.conditional_class:        # projection discriminator
            emb = self.projector(c[:, 0])
            if a.conditional_color:
                emb = emb + self.projector_col1(c[:, 1])
            y = y + (feat * emb[:, :, None, None]).sum(dim=1, keepdim=True)
        elif a.conditional_text:
            att, _ = self.att(feat, *caption)
            y = y + (feat * att).sum(dim=1, keepdim=True)
        return y


class MeshDiscriminator(_DiscriminatorBase):
    def __init__(self, args, nc, circular=True, positional_embeddings=True):
        super().__init__()
        norm_layer, bias = _norm_and_bias(args)
        self._setup(args, circular, positional_embeddings)
        if args.conditional_text:
            self.att = SpatialAttention(256, args.text_embedding_dim)
        k5pad = (2, 0) if circular else 2
        if positional_embeddings:
            nc += 4
        sn = nn.utils.spectral_norm
        self.conv1 = sn(TCConv2d(nc, 64, 5, padding=k5pad, stride=1))
        self.conv2 = sn(TCConv2d(64, 128, 4, padding=(1, 0), stride=2, bias=bias))
        self.bn2 = norm_layer(128)
        self.conv3 = sn(TCConv2d(128, 256, 4, padding=(1, 0), stride=2, bias=bias))
        self.bn3 = norm_layer(256)
        self.conv4 = sn(TCConv2d(256, 1, 5, padding=k5pad, stride=1))
        self.relu = nn.LeakyReLU(0.2, inplace=True)
        if args.conditional_class:
            self.projector = nn.Embedding(args.n_classes[0], 256)
            if args.conditional_color:
                self.projector_col1 = nn.Embedding(args.n_classes[1], 256)

    def forward(self, texture, mesh_map, c=None, caption=None, W=None, prefix="d2."):
        W = W or {}
        x = F.avg_pool2d(texture, texture.shape[2] // mesh_map.shape[2])      # texture at mesh resolution (32x32)
        x = self._with_positions(x, (mesh_map,))
        mask = None
        if self.args.mask_output:
            with torch.no_grad():
                mask = F.avg_pool2d(x[:, 3:4], 4)
        p1, p2 = (1, 2) if self.circular else (0, 0)       # x padding of the 4x4 / 5x5 layers, applied by the producer
        l1, l2 = self._links(2, W)
        x = _conv_norm_act(self.conv1, None, self.pad(x), p1, W.get(prefix + "conv1"), link_out=l1)
        x = _conv_norm_act(self.conv2, self.bn2, x, p1, W.get(prefix + "conv2"), link_in=l1, link_out=l2)
        x = _conv_norm_act(self.conv3, self.bn3, x, p2, W.get(prefix + "conv3"), link_in=l2)
        feat = x[..., p2:x.shape[3] - p2]
        y = self._project(_head(self.conv4, x, W.get(prefix + "conv4")), feat, c, caption)
        return y, mask


class TextureDiscriminator(_DiscriminatorBase):
    def __init__(self, args, nc, downsample=1, circular=True, positional_embeddings=True):
        super().__init__()
        norm_layer, bias = _norm_and_bias(args)
        self._setup(args, circular, positional_embeddings)
        if args.conditional_text:
            self.att = SpatialAttention(512, args.text_embedding_dim)
        k5pad = (2, 0) if circular else 2
        if positional_embeddings:
            nc += 4
        sn = nn.utils.spectral_norm
        # full-resolution 512^2 textures (and all 1024^2 ones) are halved by the very first layer
        self.stride_first = (downsample == 1 and args.texture_resolution >= 512) or args.texture_resolution >= 1024 \
            or args.conditional_text
        if self.stride_first:
            self.padconv1 = self.pad2
            self.conv1 = sn(TCConv2d(nc, 64, 4, padding=(1, 0), stride=2))
        else:
            self.padconv1 = self.pad
            self.conv1 = sn(TCConv2d(nc, 64, 5, padding=k5pad, stride=1))
        self.conv2 = sn(TCConv2d(64, 128, 4, padding=(1, 0), stride=2, bias=bias))
        self.bn2 = norm_layer(128)
        self.conv3 = sn(TCConv2d(128, 256, 4, padding=(1, 0), stride=2, bias=bias))
        self.bn3 = norm_layer(256)
        self.conv4 = sn(TCConv2d(256, 512, 4, padding=(1, 0), stride=2, bias=bias))
        self.bn4 = norm_layer(512)
        self.conv5 = sn(TCConv2d(512, 1, 5, padding=k5pad, stride=1))
        self.relu = nn.LeakyReLU(0.2, inplace=True)
        self.downsample = downsample
        if args.conditional_class:
            self.projector = nn.Embedding(args.n_classes[0], 512)
            if args.conditional_color:
                self.projector_col1 = nn.Embedding(args.n_classes[1], 512)

    def forward(self, x, c=None, caption=None, W=None, prefix="d1."):
        W = W or {}
        if self.downsample > 1:
            x = F.avg_pool2d(x, self.downsample)
        mask = None
        if self.args.mask_output:
            with torch.no_grad():
                mask = F.avg_pool2d(x[:, 3:4], 16 if self.stride_first else 8)
        p1, p2 = (1, 2) if self.circular else (0, 0)       # x padding of the 4x4 / 5x5 layers, applied by the producer
        l1, l2, l3 = self._links(3, W)
        x = self._stem_input(x, 1 if self.stride_first else 2)          # positional channels + the padding in front of conv1
        x = _conv_norm_act(self.conv1, None, x, p1, W.get(prefix + "conv1"), link_out=l1)
        x = _conv_norm_act(self.conv2, self.bn2, x, p1, W.get(prefix + "conv2"), link_in=l1, link_out=l2)
        x = _conv_norm_act(self.conv3, self.bn3, x, p1, W.get(prefix + "conv3"), link_in=l2, link_out=l3)
        x = _conv_norm_act(self.conv4, self.bn4, x, p2, W.get(prefix + "conv4"), link_in=l3)
        feat = x[..., p2:x.shape[3] - p2]
        y = self._project(_head(self.conv5, x, W.get(prefix + "conv5")), feat, c, caption)
        return y, mask


class MultiScaleDiscriminator(nn.Module):
    def __init__(self, args, nc):
        super().__init__()
        self.args = args
        if args.num_discriminators not in (2, 3):
            raise ValueError("num_discriminators must be 2 or 3")
        self.d1 = TextureDiscriminator(args, nc, 1)
        self.d2 = TextureDiscriminator(args, nc, 2) if args.texture_only else MeshDiscriminator(args, nc + 3)
        if args.num_discriminators == 3:
            self.d3 = TextureDiscriminator(args, nc, 4)

    def _weights(self):
        """Spectral norm + kernel layouts of every convolution of d1 / d2 / d3 in one WeightBank pass (b3d/bank.py)."""
        if getattr(self, 'disable_bank', False):
            return None
        bank = self.__dict__.get('_bank')
        if bank is None:
            convs, fold = {}, []
            for dn in ('d1', 'd2', 'd3'):
                d = getattr(self, dn, None)
                if d is None:
                    continue
                for cn in ('conv1', 'conv2', 'conv3', 'conv4', 'conv5'):
                    m = getattr(d, cn, None)
                    if m is None:
                        continue
                    if not _bankable(m):
                        self.__dict__['_bank'] = False
                        return None
                    convs[f"{dn}.{cn}"] = m
                    if cn == 'conv1' and m.stride[0] == 1 and m.kernel_size[0] > 1 and m.in_channels * m.kernel_size[0] <= 64:
                        fold.append(f"{dn}.{cn}")               # thin stem: vertical taps folded into the channels
            bank = self.__dict__['_bank'] = WeightBank(convs, fold=fold)
        return bank.forward(self.training) if bank else None

    def forward(self, x, mesh_map=None, c=None, caption=None):
        W = self._weights() if x.is_cuda else None
        d1, m1 = self.d1(x, c, caption, W=W, prefix="d1.")
        if self.args.texture_only:
            d2, m2 = self.d2(x, c, caption, W=W, prefix="d2.")
        else:
            d2, m2 = self.d2(x, mesh_map, c, caption, W=W, prefix="d2.")
        if self.args.num_discriminators == 3:
            d3, m3 = self.d3(x, c, caption, W=W, prefix="d3.")
            return [d1, d2, d3], [m1, m2, m3]
        return [d1, d2], [m1, m2]


class ConditionalBatchNorm2d(nn.Module):
    def __init__(self, args, ch, emb_dim):
        super().__init__()
        kind = args.norm_g
        if kind == 'syncbatch':
            from sync_batchnorm import SynchronizedBatchNorm2d
            self.norm = SynchronizedBatchNorm2d(ch, affine=False)
        elif kind == 'batch':
            self.norm = nn.BatchNorm2d(ch, affine=False)
        elif kind == 'instance':
            self.norm = nn.InstanceNorm2d(ch, affine=False)
        elif kind == 'none':
            self.norm = lambda x: x
        else:
            raise ValueError(f"norm_g={kind!r}")
        self.fc_gamma = nn.Linear(emb_dim, ch)
        self.fc_beta = nn.Linear(emb_dim, ch)

    def forward(self, x, z):
        g = self.fc_gamma(z)[:, :, None, None]
        b = self.fc_beta(z)[:, :, None, None]
        return self.norm(x) * (1 + g) + b


class ResBlockUp(nn.Module):
    def __init__(self, args, ch_in, ch_out, emb_dim, pad_fn):
        super().__init__()
        mid = min(ch_in, ch_out)
        self.ch_out = ch_out
        sn = nn.utils.spectral_norm
        self.conv1 = sn(TCConv2d(ch_in, mid, 3, padding=(1, 0), bias=False))
        self.conv2 = sn(TCConv2d(mid, ch_out, 3, padding=(1, 0), bias=False))
        self.norm1 = ConditionalBatchNorm2d(args, mid, emb_dim)
        self.norm2 = ConditionalBatchNorm2d(args, ch_out, emb_dim)
        self.relu = nn.LeakyReLU(0.2, inplace=True)
        self.pad = pad_fn
        self.shortcut = sn(TCConv2d(ch_in, ch_out, 1, bias=False)) if ch_in != ch_out else (lambda x: x)

    def forward(self, x, z):
        skip = self.shortcut(x)
        h = self.relu(self.norm1(self.conv1(self.pad(x, 1)), z))
        h = self.relu(self.norm2(self.conv2(self.pad(h, 1)), z))
        return h + skip

    def fusable(self):
        from torch.nn.modules.batchnorm import _BatchNorm
        return isinstance(self.norm1.norm, _BatchNorm) and isinstance(self.norm2.norm, _BatchNorm)

    def forward_fused(self, xp, z, up, pad_next, post_leaky=False, W=None, prefix="", cb=None, half_in=False):
        """Same block on an input that is ALREADY replicate-padded by 1 (xp = pad(x, 1)); returns the padded input of the
        consumer: pad(up(out), pad_next) with out = [LeakyReLU](h + skip).  Every conv output goes through exactly one fused
        elementwise kernel (b3d.ew.cbn_act_pad) instead of BN, affine, LeakyReLU, add, upsample and pad kernels.
        half_in (banked only): xp = pad(x', 1) with x = up2(x') — conv1 runs as an up-convolution on x' and the shortcut /
        identity skip at x''s resolution, read at (y/2, x/2) by the fused kernel (both commute with nearest upsampling)."""
        s1 = s2 = None
        if half_in and W is None:
            raise B3DError("ResBlockUp: a half-resolution input needs the weight bank's up-convolution taps")
        if W is not None:
            # the conv epilogues accumulate the batch-norm statistics of their output (no separate pass over y)
            if cb is not None and not getattr(self, 'disable_epilogue_stats', False):
                s1, s2 = cb.stats_slot(self.norm1), cb.stats_slot(self.norm2)
            if half_in:
                c1 = lambda t: upconv_banked(t, W[prefix + ".conv1"], stats=s1)
            else:
                c1 = lambda t: conv2d_banked(t, W[prefix + ".conv1"], pad_y=1, stats=s1)
            c2 = lambda t: conv2d_banked(t, W[prefix + ".conv2"], pad_y=1, stats=s2)
            sc = lambda t: conv2d_banked(t, W[prefix + ".shortcut"], x_crop=1)
        else:
            c1, c2, sc = self.conv1, self.conv2, (lambda t: self.shortcut(t, x_crop=1))
        y1 = c1(xp)
        a = cbn_act_pad(y1, self.norm1, z, up=1, pad=1, cb=cb, sums=s1)
        y2 = c2(a)
        if isinstance(self.shortcut, nn.Module):
            skip, off = sc(xp), 0                                    # 1x1 conv on the interior of the padded input
        else:
            skip, off = xp, 1                                        # identity: read the interior of the padded input
        return cbn_act_pad(y2, self.norm2, z, skip_nchw=skip, skip_off=off, up=up, pad=pad_next, post_leaky=post_leaky, cb=cb,
                           sums=s2, skip_half=half_in)


class Generator(nn.Module):
    def __init__(self, args, emb_dim, symmetric=True, mesh_head=True):
        super().__init__()
        self.relu = nn.LeakyReLU(0.2, inplace=True)
        self.up = lambda x: F.interpolate(x, scale_factor=2, mode='nearest')
        self.args, self.symmetric, self.mesh_head = args, symmetric, mesh_head
        self.height, self.width = 8, (4 if symmetric else 8)
        if symmetric:    # half-width map: an even-mirror border equals edge replication for 3x3 / 5x5 kernels
            self.pad = lambda x, amount: pad_x(x, amount, REPLICATE)
        else:
            self.pad = lambda x, amount: pad_x(x, amount, CIRCULAR)

        if args.conditional_class and args.conditional_color:
            self.emb_class = nn.Embedding(args.n_classes[0], emb_dim // 2)
            self.emb_color = nn.Embedding(args.n_classes[1], emb_dim // 2)
            emb_dim += emb_dim
        elif args.conditional_class:
            self.emb_class = nn.Embedding(args.n_classes[0], emb_dim)
            emb_dim += emb_dim

        self.fc = nn.Linear(emb_dim, self.height * self.width * 512)
        block = lambda cin, cout: ResBlockUp(args, cin, cout, emb_dim, self.pad)
        self.blk1 = block(512, 512)
        self.blk2 = block(512, 256)
        res = args.texture_resolution
        if res >= 256:
            self.blk3a = block(256, 256)
        if res >= 512:
            self.blk3b = block(256, 256)
        if res >= 1024:
            self.blk3c = block(256, 256)
        if args.conditional_text:
            self.att = SpatialAttention(256, args.text_embedding_dim)
        self.blk4 = block(256, 128)
        self.blk5 = block(128, 128)
        self.blk6 = block(128, 64)
        self.conv_final = TCConv2d(64, 3, 5, padding=(2, 0))
        if mesh_head:
            self.blk3_mesh = block(256, 64)
            self.conv_mesh = TCConv2d(64, 3, 5, padding=(2, 0))
            with torch.no_grad():      # start from the undeformed template
                self.conv_mesh.weight.zero_()
                self.conv_mesh.bias.zero_()

    def forward(self, z, c=None, caption=None, return_attention=False):
        a = self.args
        if a.conditional_class:
            if c is None:
                raise AssertionError("class-conditional generator needs c")
            cond = [z, self.emb_class(c[:, 0])]
            if a.conditional_color:
                cond.append(self.emb_color(c[:, 1]))
            z = torch.cat(cond, dim=1)

        x = self.fc(z).view(z.shape[0], -1, self.height, self.width)
        x = x.contiguous(memory_format=torch.channels_last)
        if self.symmetric and not a.conditional_text and self.blk1.fusable() and not getattr(self, 'disable_fusion', False):
            return self._forward_fused(x, z, return_attention)
        x = self.up(self.blk1(x, z))
        x = self.blk2(x, z)
        attention_map = None
        if a.conditional_text:
            att, attention_map = self.att(x, *caption)
            x = x + att
        x = self.up(x)

        t = x
        for name in ('blk3a', 'blk3b', 'blk3c'):
            if hasattr(self, name):
                t = self.up(getattr(self, name)(t, z))
        t = self.up(self.blk4(t, z))
        t = self.up(self.blk5(t, z))
        t = self.relu(self.blk6(t, z))
        x_tex = torch.tanh(self.conv_final(self.pad(t, 2)))

        x_mesh = None
        if self.mesh_head:
            m = self.relu(self.blk3_mesh(x, z))
            x_mesh = adjust_poles(self.conv_mesh(self.pad(m, 2)))

        if self.symmetric:
            x_tex = symmetrize_texture(x_tex)
            if x_mesh is not None:
                x_mesh = symmetrize_texture(x_mesh)
            if attention_map is not None:
                attention_map = symmetrize_texture(attention_map)
        return (x_tex, x_mesh, attention_map) if return_attention else (x_tex, x_mesh)

    def _weights(self):
        """Spectral norm + kernel layouts of every convolution of the generator in one WeightBank pass (b3d/bank.py)."""
        if getattr(self, 'disable_bank', False):
            return None
        bank = self.__dict__.get('_bank')
        if bank is None:
            convs, up2 = {}, []
            for bn in ('blk1', 'blk2', 'blk3a', 'blk3b', 'blk3c', 'blk4', 'blk5', 'blk6', 'blk3_mesh'):
                blk = getattr(self, bn, None)
                if blk is None:
                    continue
                convs[bn + ".conv1"], convs[bn + ".conv2"] = blk.conv1, blk.conv2
                if bn != 'blk1':                                  # every block after the first reads an upsampled input
                    up2.append(bn + ".conv1")
                if isinstance(blk.shortcut, nn.Module):
                    convs[bn + ".shortcut"] = blk.shortcut
            convs["conv_final"] = self.conv_final
            if self.mesh_head:
                convs["conv_mesh"] = self.conv_mesh
            bank = self.__dict__['_bank'] = WeightBank(convs, up2=up2)
        return bank.forward(self.training)

    def _forward_fused(self, x, z, return_attention):
        """The same network with the inter-convolution glue fused (replicate-padded tensors flow between the blocks) and the
        weights of all convolutions prepared by one WeightBank pass.  With the bank, the blocks hand over their output BEFORE
        the x2 upsample and every later block runs its 3x3 conv1 as an up-convolution (b3d.conv.upconv_banked)."""
        W = self._weights()
        names = [n for n in ('blk1', 'blk2', 'blk3a', 'blk3b', 'blk3c', 'blk4', 'blk5', 'blk6') if hasattr(self, n)]
        if self.mesh_head:
            names.append('blk3_mesh')
        # gamma / beta of all conditional batch norms from one GEMM (blk1.norm1 first: it closes the gradient sink)
        cb = CBNBatch([m for n in names for m in (getattr(self, n).norm1, getattr(self, n).norm2)], z)
        blk = lambda name, inp, **kw: getattr(self, name).forward_fused(inp, z, W=W, prefix=name, cb=cb, **kw)
        head = (lambda conv, name, inp: conv(inp)) if W is None else (lambda conv, name, inp: conv2d_banked(inp, W[name], pad_y=2))
        half = W is not None                                          # up2 happens inside the next block's conv1
        up = 1 if half else 2
        p = pad_x(x, 1, REPLICATE)
        p = blk('blk1', p, up=up, pad_next=1)
        p = blk('blk2', p, up=up, pad_next=1, half_in=half)          # blk2 -> up: shared by the texture and mesh branches
        t = p
        for name in ('blk3a', 'blk3b', 'blk3c'):
            if hasattr(self, name):
                t = blk(name, t, up=up, pad_next=1, half_in=half)
        t = blk('blk4', t, up=up, pad_next=1, half_in=half)
        t = blk('blk5', t, up=up, pad_next=1, half_in=half)
        t = blk('blk6', t, up=1, pad_next=2, post_leaky=True, half_in=half)
        x_tex = symmetrize_texture(torch.tanh(head(self.conv_final, "conv_final", t)))
        x_mesh = None
        if self.mesh_head:
            m = blk('blk3_mesh', p, up=1, pad_next=2, post_leaky=True, half_in=half)
            x_mesh = symmetrize_texture(adjust_poles(head(self.conv_mesh, "conv_mesh", m)))
        return (x_tex, x_mesh, None) if return_attention else (x_tex, x_mesh)


class SpatialAttention(nn.Module):
    """Word-level attention of the text-conditional variant (reference :433-481, AttnGAN-style).  Kept for
    state-dict / constructor compatibility; the text branch is dead in the reference (its RNN_Encoder is never
    defined, SURVEY App. A D12), so it runs on stock torch ops."""

    def __init__(self, input_dim, context_dim):
        super().__init__()
        self.conv_context = nn.Conv2d(context_dim, input_dim, 1, stride=1, padding=0, bias=False)
        self.sm = nn.Softmax(dim=1)

    def forward(self, input, context, mask):
        B, _, ih, iw = input.shape
        L = context.size(2)
        q = input.reshape(B, -1, ih * iw).transpose(1, 2)                    # B x HW x C
        src = self.conv_context(context.unsqueeze(3)).squeeze(3)              # B x C x L
        att = torch.bmm(q, src).view(B * ih * iw, L)
        if mask is not None:
            att = att + mask.unsqueeze(1).expand(-1, ih * iw, -1).reshape(B * ih * iw, L).float() * -10000
        att = self.sm(att).view(B, ih * iw, L).transpose(1, 2)                # B x L x HW
        out = torch.bmm(src, att).view(B, -1, ih, iw)
        return out, att.reshape(B, -1, ih, iw)
