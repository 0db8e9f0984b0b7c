"""Generate the goldens that let the host-logic tests compare with the original project without its checkout:
    python tests/golden/make_golden_reference_state.py <original project's code directory> [gan recon flops pseudogt]
Each part runs in its own process (the original project and this package both have top-level `models`, `utils`, `data`).

  gan       gan_init_reference.npz: the original models.gan Generator / MultiScaleDiscriminator built with
            gan_common.build's seed (256^2, nd = 2) -> state-dict probes (state_probes below); positional_encoding probes;
            the names and shapes of the shipped CUB checkpoint's generator_running_avg.
  recon     recon_init_reference.npz: the original models.reconstruction network built with recon_common.build's seed
            -> state-dict probes.
  flops     bench_flops_reference.npz: dense-conv GFLOPs of one image through the original modules, measured with forward
            hooks on every nn.Conv2d (the numerators of bench.py's tensor-core roofline).
  pseudogt  pseudogt_dataset_reference.npz: a record written by this package's data/pseudo_gt.py, read back by the original
            AbstractDataset.load_pseudo_ground_truth; its mirror_tex of the texture."""
import os
import re
import subprocess
import sys
import types

import numpy as np
import torch
import torch.nn as nn

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
PARTS = ("gan", "recon", "flops", "pseudogt")
sys.path.insert(0, HERE)


def state_probes(sd, prefix):
    """Names, shapes, float64 sums and 64 values at seeded flat positions of every tensor: same-seed construction is
    checked value for value at those positions and in aggregate everywhere, in a few kB instead of tens of MB."""
    from state_probes import probe
    out = {prefix + ".names": np.array(list(sd))}
    for k, v in sd.items():
        idx, val, s = probe(v)
        out[f"{prefix}.{k}.shape"] = np.array(v.shape, dtype=np.int64)
        out[f"{prefix}.{k}.idx"], out[f"{prefix}.{k}.val"], out[f"{prefix}.{k}.sum"] = idx, val, s
    return out


def part_gan(ref):
    import gan_common as GC
    from models import gan as ref_gan
    G, D = GC.build(ref_gan, GC.make_args(256, 2))
    out = {**state_probes(G.state_dict(), "G"), **state_probes(D.state_dict(), "D")}
    for ny, nx in ((32, 32), (32, 16), (256, 128)):
        out[f"pe_{ny}x{nx}"] = ref_gan.positional_encoding(ny, nx)[:, ::4, ::4]
    ck = torch.load(os.path.join(ref, "gan_weights/pretrained_weights_cub/checkpoint_latest.pth"), map_location="cpu")
    sd = ck["generator_running_avg"]
    out["ckpt_names"] = np.array(list(sd))
    out["ckpt_shapes"] = np.array([",".join(map(str, v.shape)) for v in sd.values()])
    return "gan_init_reference.npz", out


def part_recon(ref):
    import recon_common as RC
    from models import reconstruction as ref_recon
    return "recon_init_reference.npz", state_probes(RC.build(ref_recon).state_dict(), "net")


def conv_gflops(module, run):
    tot, hooks = {}, []
    for name, m in module.named_modules():
        if isinstance(m, nn.Conv2d):
            def hook(mod, inp, out, name=name):
                kh, kw = mod.kernel_size
                tot[name] = tot.get(name, 0.0) + 2.0 * out.numel() * mod.in_channels * kh * kw / 1e9
            hooks.append(m.register_forward_hook(hook))
    with torch.no_grad():
        run()
    for h in hooks:
        h.remove()
    return tot


def part_flops(ref):
    import gan_common as GC
    import recon_common as RC
    from models import gan as ref_gan
    from models import reconstruction as ref_recon
    out = {}
    for res, nd in ((256, 2), (512, 3)):
        args = GC.make_args(res, nd)
        G, D = GC.build(ref_gan, args)
        G.eval(); D.eval()
        z, c, alpha, tex, mesh = GC.inputs(args, B=1)
        g = conv_gflops(G, lambda: G(z, c))
        d = conv_gflops(D, lambda: D(torch.cat((tex * alpha, alpha), 1), mesh, c))
        out[f"g{res}"] = np.float64(sum(g.values()))
        out[f"d{res}"] = np.float64(sum(d.values()))
        out[f"d_first{res}"] = np.float64(sum(v for k, v in d.items() if re.fullmatch(r"d\d\.conv1", k)))
    net = RC.build(ref_recon, texture_res=128).eval()
    r = conv_gflops(net, lambda: net(torch.rand(1, 4, 256, 256)))
    out["recon"], out["recon_first"] = np.float64(sum(r.values())), np.float64(r["conv1e"])
    return "bench_flops_reference.npz", out


def _load(name, path):
    import importlib.util
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def part_pseudogt(ref):
    import tempfile
    ours = _load("pseudo_gt", os.path.join(ROOT, "2dimageto3dmodel_b200", "data", "pseudo_gt.py"))
    theirs = _load("ref_abstract_dataset", os.path.join(ref, "data", "abstract_dataset.py"))
    from pseudogt_common import record
    cache = os.path.join(tempfile.mkdtemp(), "cache", "cub")
    ours.save_pseudo_gt(ours.pseudo_gt_dir(cache, 32), 0, record(ours.make_record, seed=3))
    ds = object.__new__(theirs.AbstractDataset)                  # bypass __init__ (it globs the real dataset)
    ds.args = types.SimpleNamespace(texture_resolution=32)
    ds.cache_dir = cache
    got = ds.load_pseudo_ground_truth(0)
    out = {k: v.numpy() for k, v in got.items()}
    out["mirror_texture"] = theirs.AbstractDataset.mirror_tex(got["texture"]).numpy()
    return "pseudogt_dataset_reference.npz", out


if __name__ == "__main__":
    ref = os.path.abspath(sys.argv[1])
    which = sys.argv[2:] or list(PARTS)
    if len(which) > 1:
        for p in which:
            subprocess.run([sys.executable, __file__, ref, p], check=True)
        sys.exit(0)
    if which[0] != "pseudogt":
        sys.path.insert(0, ref)
    torch.set_num_threads(8)
    fname, out = globals()["part_" + which[0]](ref)
    path = os.path.join(HERE, fname)
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")
