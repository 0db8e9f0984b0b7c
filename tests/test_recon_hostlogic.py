"""Host-side logic of the models.reconstruction drop-in (CPU): state-dict layout and same-seed initial values equal the
reference's (stored probes); DatasetParams against the reference golden."""
import os
import sys

import numpy as np
import pytest
import torch

from conftest import GOLDEN

sys.path.insert(0, GOLDEN)
import recon_common as RC          # noqa: E402


def test_dataset_params_match_reference_golden():
    from models.reconstruction import DatasetParams
    d = np.load(os.path.join(GOLDEN, "recon_reference.npz"))
    dp = DatasetParams(RC.dataset_args(), 10)
    with torch.no_grad():
        st = torch.tensor(d["dp_state"])
        dp.ds_translation.copy_(st[:, :2]); dp.ds_scale.copy_(st[:, 2:3]); dp.ds_z0.copy_(st[:, 3:4])
    idx = torch.tensor(d["dp_idx"])
    t, s = dp(idx, 'deltas')
    assert np.array_equal(t.detach().numpy(), d["dp_t"]) and np.array_equal(s.detach().numpy(), d["dp_s"])
    assert np.allclose(dp(idx, 'z0').detach().numpy(), d["dp_z0"], rtol=1e-6, atol=0)
    t, s = dp(None, 'deltas')
    assert np.allclose(t.detach().numpy(), d["dp_t_mean"], atol=1e-7) and np.allclose(s.detach().numpy(), d["dp_s_mean"], atol=1e-7)
    assert np.allclose(dp(None, 'z0').detach().numpy(), d["dp_z0_mean"], rtol=1e-6)
    with pytest.raises(ValueError):
        dp(idx, 'nope')
    # mirrored copies (indices >= N) flip the sign of the x translation only
    a, _ = dp(torch.tensor([3]), 'deltas')
    b, _ = dp(torch.tensor([13]), 'deltas')
    assert float(a[0, 0]) == -float(b[0, 0]) and float(a[0, 1]) == float(b[0, 1]) and float(b[0, 2]) == 0.0


def test_state_dict_layout():
    from models.reconstruction import ReconstructionNetwork
    net = RC.build(sys.modules["models.reconstruction"], texture_res=256)
    sd = net.state_dict()
    assert sd["conv1e.weight"].shape == (64, 4, 5, 5) and sd["fc1e.weight"].shape == (256, 4096)
    assert sd["blk1.shortcut.weight"].shape == (512, 256, 1, 1) and "blk3.shortcut.weight" not in sd
    assert sd["blk3c_tex.conv2.weight"].shape == (256, 256, 3, 3) and sd["conv_tex.bias"].shape == (3,)
    assert sd["bnfc3e.running_var"].shape == (1024,) and sd["fc1_tex.weight"].shape == (4 * 2 * 256, 1024)
    assert round(sum(p.numel() for p in ReconstructionNetwork(texture_res=128).parameters()) / 1e6, 2) == 15.11   # SURVEY §8e
    with pytest.raises(ValueError):
        ReconstructionNetwork(texture_res=100)


def test_same_seed_state_equals_reference():
    """tests/golden/recon_init_reference.npz (make_golden_reference_state.py): the reference's models.reconstruction built
    with the same seed -> state-dict names, shapes, probed values and sums."""
    from models import reconstruction as mine
    from state_probes import assert_state_matches
    assert_state_matches(RC.build(mine).state_dict(), np.load(os.path.join(GOLDEN, "recon_init_reference.npz")), "net")


def test_forward_wiring_matches_reference_golden_on_cpu(monkeypatch):
    """The module's wiring (layer order, paddings, flatten order, upsampling, heads, symmetrisation) with the CUDA pieces
    swapped for exact torch ops — TCConv2d -> nn.Conv2d.forward, pad_x -> F.pad / wrap-around cat — must reproduce the
    reference golden to fp32 round-off, forward and backward.  (The same golden is the target of the CUDA test.)"""
    import torch.nn as nn
    import torch.nn.functional as F
    from models import gan, reconstruction
    d = np.load(os.path.join(GOLDEN, "recon_reference.npz"))

    def pad_x_cpu(t, amount, mode):
        if mode == reconstruction.REPLICATE:
            return F.pad(t, (amount, amount, 0, 0), mode='replicate')
        return torch.cat((t[..., -amount:], t, t[..., :amount]), dim=3)

    monkeypatch.setattr(gan.TCConv2d, "forward", lambda self, x, **kw: nn.Conv2d.forward(self, x))
    monkeypatch.setattr(reconstruction, "pad_x", pad_x_cpu)
    torch.set_num_threads(8)
    net = RC.build(reconstruction).train()
    x, w_tex, w_mesh = RC.inputs()
    tex, mesh_map = net(x)
    RC.loss_of(tex, mesh_map, w_tex, w_mesh).backward()
    assert np.abs(tex.detach()[:, :, ::8, ::8].numpy() - d["tex_probe"]).max() < 2e-4
    assert np.abs(mesh_map.detach().numpy() - d["mesh_map"]).max() < 1e-4     # fp32 round-off (channels-last vs NCHW kernels)
    params = dict(net.named_parameters())
    for name, ref in zip(d["grad_names"], d["grad_norms"]):
        got = float(params[str(name)].grad.norm())
        assert abs(got - ref) <= 2e-3 * ref + 1e-6, (str(name), got, ref)
    assert np.abs(net.bn4e.running_mean.numpy() - d["bn4e_mean"]).max() < 1e-5


@pytest.mark.parametrize("tag,deltas,z0", [("deltas", True, False), ("full", True, True), ("z0", False, True)])
def test_training_iteration_matches_the_reference_loop(tag, deltas, z0, monkeypatch):
    """tests/golden/recon_step_reference.npz: the training-loop body of run_reconstruction.py (:409-465) EXECUTED from the
    script's syntax tree for four iterations on stand-in network / template / renderer (make_golden_recon_step.py).
    ReconTrainer.step — on the same stand-ins, with its fused CUDA pieces (RGBA-MSE + IoU kernel, flat-loss kernel, fused
    vertex pipeline) replaced by their torch definitions — must reproduce every iteration's loss, the warm-up factor and the
    updated network / DatasetParams parameters (two Adams)."""
    import recon_step_common as RS
    import reconstruction_training as RT
    from models.reconstruction import DatasetParams
    from oracle import mesh as OM
    d = np.load(os.path.join(GOLDEN, "recon_step_reference.npz"))
    args = RS.make_args(deltas, z0)

    def rgba_mse_iou(image, alpha, X_real):                  # b3d.mesh.rgba_mse_iou = run_reconstruction.py:429-436
        X_fake = torch.cat((image, alpha), dim=3).permute(0, 3, 1, 2)
        return torch.nn.functional.mse_loss(X_fake, X_real), OM.mean_iou(X_fake[:, 3], X_real[:, 3])
    monkeypatch.setattr(RT, "rgba_mse_iou", rgba_mse_iou)
    monkeypatch.setattr(RT, "loss_flat", lambda mesh, norms: OM.loss_flat(mesh.ff, mesh.faces.shape[0], norms))

    tpl = RS.Template()
    tpl.vertices_and_pose = lambda m, s, t, r, z=None: (lambda raw: (raw, OM.transform_vertices(raw, s, t, r, z)))(tpl.get_vertex_positions(m))
    tr = object.__new__(RT.ReconTrainer)                      # the constructor builds the CUDA network; wire the stand-ins instead
    tr.args, tr.tpl, tr.world, tr.renderer = args, tpl, 1, None
    tr.generator = RS.build_net()
    tr.optimizer = torch.optim.Adam(tr.generator.parameters(), lr=args.lr)
    tr.dataset_params = DatasetParams(args, 10)
    tr.optimizer_dataset = torch.optim.Adam(tr.dataset_params.parameters(), lr=args.lr_dataset)
    tr.flat_warmup = torch.full((), 10.0)
    losses = []
    for i, (X, s, t, r, idx) in enumerate(RS.batches()):
        loss, recon, flat, miou = tr.step(X, s, t, r, idx.squeeze(-1))
        losses.append(float(loss))
        if i == 0:
            ref = str(d[tag + ".log0"])
            assert f"recon_loss {float(recon):.5f} flat_loss {float(flat):.5f} total {float(loss):.5f} iou {float(miou):.5f}" in ref
    assert np.abs(np.array(losses) - d[tag + ".g_curve"]).max() < 2e-6
    assert abs(float(tr.flat_warmup) - float(d[tag + ".flat_warmup"])) < 1e-5     # 10 -> 9.6 (an fp32 device scalar here, a Python float there)
    for k, v in tr.generator.state_dict().items():
        # four Adam steps of 1e-2: a wrong learning rate / optimiser / loss weight moves parameters by >= 1e-3; Adam's
        # g / sqrt(v) normalisation amplifies rounding differences of small-gradient elements to ~1e-5
        assert np.abs(v.numpy().astype(np.float64) - d[f"{tag}.net.{k}"]).max() < 1e-4, k
    for k, v in tr.dataset_params.state_dict().items():
        assert np.abs(v.numpy() - d[f"{tag}.dp.{k}"]).max() < 1e-4, k
    assert any(np.abs(d[f"{tag}.dp.{k}"] - (1.0 if k == "ds_z0" else 0.0)).max() > 1e-2 for k in tr.dataset_params.state_dict())
