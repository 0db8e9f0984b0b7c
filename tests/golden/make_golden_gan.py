"""Generate tests/golden/gan_reference.npz from the REFERENCE's own modules (authoring container only):
    python tests/golden/make_golden_gan.py
Imports models/gan.py and utils/losses.py unmodified from /root/reference/code (they run on CPU, SURVEY §8c),
builds G and D with the seeds of tests/golden/gan_common.py, runs one generator step and one discriminator step
(ModelWrapper.forward modes 'g' and 'd', main.py:476-521) in training mode and stores output probes, losses and
per-parameter gradient norms.  The CUDA modules are built with the same seeds on the GPU box (their initial
values equal the reference's — checked by tests/test_gan_hostlogic.py when /root/reference is present)."""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, "/root/reference/code")
import gan_common as GC                                     # noqa: E402
from models import gan as ref_gan                           # noqa: E402  (reference)
from utils.losses import GANLoss                            # noqa: E402  (reference)


def make(fname, res, nd, B, probe):
    """One generator step + one discriminator step of the reference modules -> tests/golden/<fname>.
    probe: spatial stride of the stored activation probes (full tensors for the small B=2 golden)."""
    torch.set_num_threads(8)
    args = GC.make_args(res, nd)
    G, D = GC.build(ref_gan, args)
    G.train(); D.train()
    crit = GANLoss('hinge', tensor=torch.FloatTensor)
    z, c, alpha, tex, mesh = GC.inputs(args, B=B)
    out = {"res": np.int64(res), "nd": np.int64(nd), "B": np.int64(B), "probe": np.int64(probe)}
    # ---- generator step
    loss, pred_tex, pred_mesh, dout, mask = GC.g_step(G, D, crit, z, c, alpha)
    loss.mean().backward()
    out["g_loss"] = loss.detach().numpy()
    out["tex_probe"] = pred_tex.detach()[:, :, ::16, ::16].numpy()
    out["tex_sum"] = np.float64(pred_tex.detach().double().sum())
    out["mesh"] = pred_mesh.detach()[:, :, ::probe, ::probe].numpy()
    for i in range(nd):
        out[f"d_out{i}"] = dout[i].detach()[:, :, ::probe, ::probe].numpy()
        out[f"mask{i}"] = mask[i][:, :, ::probe, ::probe].numpy()
    names = [n for n, p in G.named_parameters() if p.grad is not None]
    out["g_grad_names"] = np.array(names)
    out["g_grad_norms"] = np.array([float(dict(G.named_parameters())[n].grad.norm()) for n in names])
    out["g_grad_probe"] = G.blk5.conv1.weight_orig.grad[:4, :4].numpy()
    out["sn_u_blk1"] = G.blk1.conv1.weight_u.numpy().copy()
    out["bn_mean_blk6"] = G.blk6.norm2.norm.running_mean.numpy().copy()
    G.zero_grad(); D.zero_grad()
    # ---- discriminator step (same modules, second forward: spectral-norm u/v advance again, as in training)
    lf, lr, dout = GC.d_step(G, D, crit, z, c, alpha, tex, mesh)
    (lf.mean() + lr.mean()).backward()
    out["d_loss_fake"], out["d_loss_real"] = lf.detach().numpy(), lr.detach().numpy()
    out["dd_out0"] = dout[0].detach()[:, :, ::probe, ::probe].numpy()
    names = [n for n, p in D.named_parameters() if p.grad is not None]
    out["d_grad_names"] = np.array(names)
    out["d_grad_norms"] = np.array([float(dict(D.named_parameters())[n].grad.norm()) for n in names])
    path = os.path.join(HERE, fname)
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes; g_loss", out["g_loss"], "d losses", out["d_loss_fake"], out["d_loss_real"])


def checkpoint_kat():
    """Known-answer test of a checkpoint load (SURVEY §8c(1)): the reference Generator, eval mode, loading strictly
    gan_common.checkpoint_standin (the shipped CUB checkpoint's layout, seeded values; the 52 MB checkpoint itself cannot
    travel with the tests) -> probes."""
    args = GC.make_args(512, 3)
    G = ref_gan.Generator(args, 64, symmetric=True, mesh_head=True)
    G.load_state_dict(GC.checkpoint_standin(ref_gan), strict=True)
    G.eval()
    torch.manual_seed(1234)
    z, c = torch.randn(2, 64), torch.tensor([[3], [77]])
    with torch.no_grad():
        tex, mesh = G(z, c)
    out = {"z": z.numpy(), "c": c.numpy(), "tex_probe": tex[:, :, ::16, ::16].numpy(), "tex_px": tex[0, :, 100, 200].numpy(),
           "mesh": mesh.numpy(), "tex_sum": np.float64(tex.double().sum())}
    path = os.path.join(HERE, "gan_checkpoint_kat.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes; tex[0,:,100,200]", out["tex_px"], "sum", out["tex_sum"])


if __name__ == "__main__":
    which = sys.argv[1:] or ["b2", "b32", "r512", "kat"]
    if "b2" in which:
        make("gan_reference.npz", 256, 2, 2, 1)            # the small golden (full tensors)
    if "b32" in which:
        make("gan_reference_b32.npz", 256, 2, 32, 4)       # cfg3's batch: reaches the kernels bench.py dispatches
    if "r512" in which:
        make("gan_reference_r512.npz", 512, 3, 2, 1)       # cfg5's architecture (512^2, three discriminators)
    if "kat" in which:
        checkpoint_kat()
