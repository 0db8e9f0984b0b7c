"""The CUDA GAN (tcgen05 convs) against golden vectors produced by the reference's modules on the CPU
(tests/golden/make_golden_gan.py): same seeds -> same weights, same inputs; one generator step and one
discriminator step in training mode (spectral-norm power iteration, batch statistics, hinge losses, backward).

Tolerance: the reference golden is exact fp32; the tensor cores compute in tf32 (10-bit mantissa, the class
cuDNN uses by default).  Through ~25 stacked convolutions we allow 2e-2 of the largest magnitude for
activations, 2e-2 relative for losses, and 6e-2 relative (+ 2e-3 of the largest norm, for the scalar
biases whose gradient is a cancelling sum over all pixels) for per-parameter gradient norms."""
import os
import sys

import numpy as np
import pytest
import torch

from conftest import GOLDEN

sys.path.insert(0, GOLDEN)
import gan_common as GC          # noqa: E402

pytestmark = pytest.mark.gpu


def close(a, ref, tol):
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else a
    err = float(np.abs(a - ref).max())
    lim = tol * max(float(np.abs(ref).max()), 1e-6)
    assert err <= lim, (err, lim)


@pytest.mark.parametrize("fname", ["gan_reference.npz", "gan_reference_b32.npz", "gan_reference_r512.npz"])
def test_gan_steps_match_reference_golden(fname):
    """gan_reference.npz: 256^2, nd=2, B=2.  gan_reference_b32.npz: cfg3's batch of 32 (the generator convolutions run at
    N=32, the discriminators at N=32 / 64: the kernel variants bench.py dispatches).  gan_reference_r512.npz: cfg5's
    architecture (512^2, three discriminators, stride-2 stem)."""
    from models import gan
    from utils.losses import GANLoss
    d = np.load(os.path.join(GOLDEN, fname))
    res, nd, B, pr = (int(d[k]) for k in ("res", "nd", "B", "probe"))
    args = GC.make_args(res, nd)
    G, D = GC.build(gan, args)
    G.cuda().train(); D.cuda().train()
    crit = GANLoss('hinge', tensor=torch.cuda.FloatTensor)
    z, c, alpha, tex, mesh = [t.cuda() for t in GC.inputs(args, B=B)]
    loss, pred_tex, pred_mesh, dout, mask = GC.g_step(G, D, crit, z, c, alpha)
    loss.mean().backward()
    close(pred_tex[:, :, ::16, ::16], d["tex_probe"], 2e-2)
    # mean signed deviation of the whole texture (a bias, so it scales with n, not sqrt(n)): tf32 operand rounding
    assert abs(float(pred_tex.double().sum()) - float(d["tex_sum"])) / pred_tex.numel() < 1e-3
    close(pred_mesh[:, :, ::pr, ::pr], d["mesh"], 2e-2)
    for i in range(nd):
        close(dout[i][:, :, ::pr, ::pr], d[f"d_out{i}"], 2e-2)
        close(mask[i][:, :, ::pr, ::pr], d[f"mask{i}"], 1e-6)
    assert abs(float(loss) - float(d["g_loss"])) < 2e-2 * abs(float(d["g_loss"]))
    params = dict(G.named_parameters())
    floor = 2e-3 * float(d["g_grad_norms"].max())      # scalar biases are cancelling sums over all pixels
    for name, ref in zip(d["g_grad_names"], d["g_grad_norms"]):
        got = float(params[str(name)].grad.norm())
        assert abs(got - ref) <= 6e-2 * ref + floor, (str(name), got, ref)
    close(G.blk5.conv1.weight_orig.grad[:4, :4], d["g_grad_probe"], 6e-2)
    close(G.blk1.conv1.weight_u, d["sn_u_blk1"], 1e-4)
    close(G.blk6.norm2.norm.running_mean, d["bn_mean_blk6"], 2e-2)
    G.zero_grad(); D.zero_grad()
    lf, lr, dout = GC.d_step(G, D, crit, z, c, alpha, tex, mesh)
    (lf.mean() + lr.mean()).backward()
    assert abs(float(lf) - float(d["d_loss_fake"])) < 2e-2 * abs(float(d["d_loss_fake"]))
    assert abs(float(lr) - float(d["d_loss_real"])) < 2e-2 * abs(float(d["d_loss_real"]))
    close(dout[0][:, :, ::pr, ::pr], d["dd_out0"], 2e-2)
    params = dict(D.named_parameters())
    floor = 2e-3 * float(d["d_grad_norms"].max())
    for name, ref in zip(d["d_grad_names"], d["d_grad_norms"]):
        got = float(params[str(name)].grad.norm())
        assert abs(got - ref) <= 6e-2 * ref + floor, (str(name), got, ref)


def test_shipped_checkpoint_known_answer():
    """SURVEY §8c(1): a generator_running_avg state dict in the shipped checkpoint's layout (gan_common.checkpoint_standin:
    seeded values, since the 52 MB checkpoint cannot travel; its layout is checked against the shipped one by
    test_gan_hostlogic.py) loads strict into the CUDA Generator and its eval-mode forward reproduces the probes the REFERENCE
    Generator computed from the same state dict on the CPU (tests/golden/make_golden_gan.py:checkpoint_kat).  Eval mode: no
    batch statistics, no power iteration."""
    from models import gan
    d = np.load(os.path.join(GOLDEN, "gan_checkpoint_kat.npz"))
    G = gan.Generator(GC.make_args(512, 3), 64, symmetric=True, mesh_head=True)
    G.load_state_dict(GC.checkpoint_standin(gan), strict=True)
    G.cuda().eval()
    with torch.no_grad():
        tex, mesh = G(torch.tensor(d["z"]).cuda(), torch.tensor(d["c"]).cuda())
    close(tex[:, :, ::16, ::16], d["tex_probe"], 2e-2)
    close(tex[0, :, 100, 200], d["tex_px"], 2e-2)
    close(mesh, d["mesh"], 2e-2)
    assert abs(float(tex.double().sum()) - float(d["tex_sum"])) / tex.numel() < 1e-3


def test_shipped_size_generator_runs_and_is_symmetric():
    """512^2 generator (the shipped checkpoints' architecture), 3 discriminators: shapes, symmetry, finiteness."""
    from models import gan
    args = GC.make_args(512, 3)
    G, D = GC.build(gan, args)
    G.cuda().eval(); D.cuda().eval()
    z, c, alpha, tex, mesh = [t.cuda() for t in GC.inputs(args, B=2)]
    with torch.no_grad():
        t, m = G(z, c)
        out, masks = D(torch.cat((t * alpha, alpha), 1), m, c)
    assert t.shape == (2, 3, 512, 512) and m.shape == (2, 3, 32, 32)
    assert torch.equal(t, t.flip(3)) is False          # not trivially symmetric about the image centre ...
    w = t.shape[3]
    assert torch.allclose(t[..., : w // 4], t[..., w // 4: w // 2].flip(3))     # ... but mirrored about the seam
    assert [o.shape for o in out] == [(2, 1, 32, 32), (2, 1, 8, 8), (2, 1, 16, 16)]
    assert all(torch.isfinite(o).all() for o in out) and float(t.abs().max()) <= 1.0
