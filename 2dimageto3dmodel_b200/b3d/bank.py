"""Weight bank: spectral normalisation and kernel weight layouts of all convolutions of a network in four launches
(libb3d csrc/sn_kernels.cu) instead of torch.nn.utils.spectral_norm's per-layer hooks (~17 tiny kernels per layer and
forward) plus per-call permute+contiguous re-layouts.

Reference semantics: torch.nn.utils.spectral_norm as used by /root/reference/code/models/gan.py:57-65,163-177,294-302 —
training mode: one power iteration updating the module's weight_u / weight_v buffers in place, sigma = u . (W v),
weight = weight_orig / sigma with u, v constants of the autograd graph; eval mode: sigma from the stored vectors.
The modules keep torch's parameter / buffer names (weight_orig, weight_u, weight_v), so state dicts are unchanged.

Per layer the bank hands the convolution kernels
  F [T'][Cout][Cin']  tap-major K-major rows (fprop operand; the weight gradient comes back in the same layout),
  D [T'][Cin'][Cout'] its per-tap transpose (input-gradient operand),
and its backward turns the F-layout gradients into gradients of weight_orig (two launches for the whole network).
Layers registered as `up2` (3x3 convolutions of a x2 nearest upsample) also get the 16 taps of the four output-parity
classes, UF [16][Cout][Cin'] and UD [16][Cin'][Cout'] (b3d.conv.upconv_forward / _UpConvBanked).
"""
import struct

import torch

from . import B3DError, check, lib, ptr, stream_ptr


def _r32(v):
    return (v + 31) // 32 * 32


def _r64(v):
    return (v + 63) // 64 * 64


class LayerWeights:
    """What one convolution needs from the bank for one forward/backward: wf (autograd output), wd, df (gradient sink)."""
    __slots__ = ("wf", "wd", "df", "uf", "ud", "Cout", "Cin", "kh", "kw", "fold", "up2", "Cinp", "Coutp", "Tp", "bias")

    def __init__(self, spec):
        for k in ("Cout", "Cin", "kh", "kw", "fold", "up2", "Cinp", "Coutp", "Tp"):
            setattr(self, k, spec[k])
        self.wf = self.wd = self.df = self.uf = self.ud = self.bias = None


class WeightBank:
    def __init__(self, convs, fold=(), no_dgrad=(), round_tf32=True, up2=()):
        """convs: ordered {name: conv module} (spectral-normalised modules expose weight_orig / weight_u / weight_v, plain
        ones weight).  fold: names whose kh vertical taps are folded into the channel dimension (thin stems).
        no_dgrad: names that never need an input gradient (no D layout is written).
        up2: 3x3 layers that also get the class taps of the convolution of a x2 nearest upsample."""
        self.names = list(convs)
        self.mods = [convs[n] for n in self.names]
        # emitted weights rounded to the nearest tf32 value (the tensor cores would otherwise truncate the fp32 words)
        self.round_tf32 = bool(round_tf32)
        self.specs = []
        off_out = off_scr = off_w = 0
        for n, m in zip(self.names, self.mods):
            sn = hasattr(m, "weight_orig")
            w = m.weight_orig if sn else m.weight
            Cout, Cin, kh, kw = w.shape
            fd = n in fold
            Cinp = _r32(kh * Cin if fd else Cin)
            Tp = kw if fd else kh * kw
            u2 = n in up2
            if u2 and (fd or (kh, kw) != (3, 3)):
                raise B3DError(f"bank: {n}: up2 class taps need an unfolded 3x3 layer")
            sp = dict(name=n, sn=sn, Cout=Cout, Cin=Cin, kh=kh, kw=kw, fold=int(fd), up2=int(u2), Cinp=Cinp, Coutp=_r32(Cout), Tp=Tp,
                      K=Cin * kh * kw, need_d=n not in no_dgrad)
            sp["wf_off"] = off_out
            off_out += _r64(Tp * Cout * Cinp)
            self.specs.append(sp)
        self.f_total = off_out                                  # the dF buffer mirrors the F region
        for sp in self.specs:
            sp["wd_off"] = -1
            if sp["need_d"]:
                sp["wd_off"] = off_out
                off_out += _r64(sp["Tp"] * sp["Cinp"] * sp["Coutp"])
        for sp in self.specs:
            sp["uf_off"] = sp["ud_off"] = -1
            if sp["up2"]:
                sp["uf_off"] = off_out
                off_out += _r64(16 * sp["Cout"] * sp["Cinp"])
                sp["ud_off"] = off_out
                off_out += _r64(16 * sp["Cinp"] * sp["Coutp"])
        for sp in self.specs:
            sp["u_off"], sp["v_off"], sp["scal_off"] = off_out, off_out + _r64(sp["Cout"]), off_out + _r64(sp["Cout"]) + _r64(sp["K"])
            off_out = sp["scal_off"] + 64
            sp["t_off"], sp["s_off"] = off_scr, off_scr + _r64(2 * sp["K"])       # t: K int64 fixed-point accumulators
            off_scr = sp["s_off"] + _r64(sp["Cout"])
            sp["dw_off"] = off_w
            off_w += _r64(sp["Cout"] * sp["K"])
        self.out_total, self.scr_total, self.w_total = off_out, off_scr, off_w
        self._ptrs = None
        self._dev = None

    # ------------------------------------------------------------------------------------------------------------
    def params(self):
        return [m.weight_orig if sp["sn"] else m.weight for m, sp in zip(self.mods, self.specs)]

    def _build(self, device):
        if lib.b3d_bank_layer_bytes() != 160:
            raise B3DError("bank: BankLayer record size mismatch between b3d/bank.py and csrc/sn_kernels.cu")
        rec, wtu, wv, emit, dot = [], [], [], [], []
        ptrs = []
        for i, (m, sp) in enumerate(zip(self.mods, self.specs)):
            w = m.weight_orig if sp["sn"] else m.weight
            u = m.weight_u if sp["sn"] else None
            v = m.weight_v if sp["sn"] else None
            for t in (w, u, v):
                if t is not None and (not t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous()):
                    raise B3DError(f"bank: {sp['name']}: parameters must be contiguous CUDA fp32 tensors (no CPU fallback)")
            ptrs.append((w.data_ptr(), u.data_ptr() if u is not None else 0, v.data_ptr() if v is not None else 0))
            rec.append(struct.pack("<3Q11q12i", ptrs[-1][0], ptrs[-1][1], ptrs[-1][2], sp["t_off"], sp["s_off"], sp["wf_off"],
                                   sp["wd_off"], sp["u_off"], sp["v_off"], sp["scal_off"], sp["wf_off"], sp["dw_off"],
                                   sp["uf_off"], sp["ud_off"],
                                   sp["Cout"], sp["Cin"], sp["kh"], sp["kw"], sp["fold"], sp["Cinp"], sp["Coutp"], sp["Tp"],
                                   int(sp["sn"]), sp["up2"], 0, 0))
            if sp["sn"]:
                wtu += [(i, a, b, 0) for a in range(-(-sp["K"] // 256)) for b in range(-(-sp["Cout"] // 64))]
                wv += [(i, a, 0, 0) for a in range(-(-sp["Cout"] // 8))]
                dot += [(i, a, 0, 0) for a in range(-(-(sp["Tp"] * sp["Cout"] * sp["Cinp"]) // 4096))]
            emit += [(i, a, b, 0) for a in range(sp["Coutp"] // 32) for b in range(sp["Cinp"] // 32)]

        def dev_bytes(b):
            return torch.frombuffer(bytearray(b), dtype=torch.uint8).to(device)

        def items(lst):
            return torch.tensor(lst if lst else [(0, 0, 0, 0)], dtype=torch.int32).to(device), len(lst)

        self._table = dev_bytes(b"".join(rec))
        self._wtu, self._wv, self._emit, self._dot = items(wtu), items(wv), items(emit), items(dot)
        self._scratch = torch.zeros(max(self.scr_total, 64), device=device)
        self._ptrs, self._dev = ptrs, device

    def _check(self):
        ps = self.params()
        device = ps[0].device
        if self._ptrs is None or self._dev != device:
            self._build(device)
            return
        for (pw, pu, pv), m, sp in zip(self._ptrs, self.mods, self.specs):
            w = m.weight_orig if sp["sn"] else m.weight
            if w.data_ptr() != pw or (sp["sn"] and (m.weight_u.data_ptr() != pu or m.weight_v.data_ptr() != pv)):
                self._build(device)                              # parameters were re-allocated (load / .to()): re-pack
                return

    # ------------------------------------------------------------------------------------------------------------
    def forward(self, training):
        """-> {name: LayerWeights}.  Differentiable w.r.t. the weight_orig / weight parameters."""
        self._check()
        ps = self.params()
        need_grad = torch.is_grad_enabled() and any(p.requires_grad for p in ps)
        outs = _BankFn.apply(self, bool(training), need_grad, *ps)
        n = len(self.specs)
        res = {}
        df_flat = outs[2 * n] if need_grad else None
        for i, sp in enumerate(self.specs):
            lw = LayerWeights(sp)
            lw.wf = outs[i]
            lw.wd = outs[n + i] if sp["need_d"] else None
            if sp["up2"]:
                lw.uf, lw.ud = outs[2 * n + 1 + 2 * i], outs[2 * n + 2 + 2 * i]
            if need_grad:
                sz = sp["Tp"] * sp["Cout"] * sp["Cinp"]
                lw.df = df_flat[sp["wf_off"]: sp["wf_off"] + sz].view(sp["Tp"], sp["Cout"], sp["Cinp"])
            lw.bias = getattr(self.mods[i], "bias", None)
            res[sp["name"]] = lw
        return res


class _BankFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, bank, training, need_grad, *weights):
        device = weights[0].device
        out = torch.empty(bank.out_total, device=device, dtype=torch.float32)
        st = stream_ptr(weights[0])
        check(lib.b3d_bank_forward(ptr(bank._table), ptr(bank._wtu[0]), bank._wtu[1], ptr(bank._wv[0]), bank._wv[1],
                                   ptr(bank._emit[0]), bank._emit[1], ptr(bank._scratch), bank._scratch.numel() * 4,
                                   ptr(out), int(training) | (2 if bank.round_tf32 else 0), st))
        wfs, wds = [], []
        for sp in bank.specs:
            wfs.append(out[sp["wf_off"]: sp["wf_off"] + sp["Tp"] * sp["Cout"] * sp["Cinp"]].view(sp["Tp"], sp["Cout"], sp["Cinp"]))
            if sp["need_d"]:
                wds.append(out[sp["wd_off"]: sp["wd_off"] + sp["Tp"] * sp["Cinp"] * sp["Coutp"]].view(sp["Tp"], sp["Cinp"], sp["Coutp"]))
            else:
                wds.append(out.new_empty(0))
        df = torch.zeros(bank.f_total, device=device, dtype=torch.float32) if need_grad else out.new_empty(0)
        ups = []                                            # (UF, UD) per layer (empty for layers without up2)
        for sp in bank.specs:
            if sp["up2"]:
                ups.append(out[sp["uf_off"]: sp["uf_off"] + 16 * sp["Cout"] * sp["Cinp"]].view(16, sp["Cout"], sp["Cinp"]))
                ups.append(out[sp["ud_off"]: sp["ud_off"] + 16 * sp["Cinp"] * sp["Coutp"]].view(16, sp["Cinp"], sp["Coutp"]))
            else:
                ups += [out.new_empty(0), out.new_empty(0)]
        ctx.bank, ctx.out, ctx.df = bank, out, df
        ctx.mark_non_differentiable(*wds, df, *ups)
        return (*wfs, *wds, df, *ups)

    @staticmethod
    def backward(ctx, *grads):
        bank, out, df = ctx.bank, ctx.out, ctx.df
        n = len(bank.specs)
        if df.numel() == 0:
            return (None, None, None) + (None,) * n
        for sp, g in zip(bank.specs, grads[:n]):
            if g is None:
                continue
            sz = sp["Tp"] * sp["Cout"] * sp["Cinp"]
            if g.data_ptr() != df.data_ptr() + 4 * sp["wf_off"]:          # gradient did not come from the sink: copy it in
                df[sp["wf_off"]: sp["wf_off"] + sz].copy_(g.reshape(-1))
        dw = torch.zeros(bank.w_total, device=df.device, dtype=torch.float32)    # zeros: alignment gaps are all-reduced too
        bank.last_dw = dw                                   # flat gradient of all conv weights (in-place all-reduce under DDP)
        check(lib.b3d_bank_backward(ptr(bank._table), ptr(bank._dot[0]), bank._dot[1], ptr(bank._emit[0]), bank._emit[1],
                                    ptr(out), ptr(df), ptr(dw), stream_ptr(df)))
        gws = []
        for sp, need in zip(bank.specs, ctx.needs_input_grad[3:]):
            gws.append(dw[sp["dw_off"]: sp["dw_off"] + sp["Cout"] * sp["K"]].view(sp["Cout"], sp["Cin"], sp["kh"], sp["kw"])
                       if need else None)
        return (None, None, None, *gws)
