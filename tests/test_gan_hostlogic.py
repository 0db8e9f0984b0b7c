"""Host-side logic of the GAN drop-ins (CPU): state-dict layout, same-seed initial values and positional
encoding equal the reference's (stored probes); GANLoss vs golden."""
import os
import sys
import types

import numpy as np
import pytest
import torch

from conftest import GOLDEN

sys.path.insert(0, GOLDEN)
import gan_common as GC          # noqa: E402


def test_ganloss_matches_reference_golden():
    from utils.losses import GANLoss
    g = np.load(os.path.join(GOLDEN, "mesh_reference_pieces.npz"))
    t = lambda k: torch.tensor(g[k])
    crit = GANLoss('hinge')
    preds, masks = [t("gl_p0"), t("gl_p1")], [t("gl_m0"), t("gl_m1")]
    assert abs(float(crit(preds, True, for_discriminator=False, mask=masks, weight=[2, 1])) - float(g["gl_g"])) < 1e-7
    assert abs(float(crit(preds, False, for_discriminator=True, mask=masks)) - float(g["gl_d_fake"])) < 1e-7
    assert abs(float(crit(preds, True, for_discriminator=True, mask=masks, weight=[2, 1])) - float(g["gl_d_real"])) < 1e-7
    assert abs(float(crit(preds, True, for_discriminator=False)) - float(g["gl_g_nomask"])) < 1e-7
    with pytest.raises(ValueError):
        GANLoss('nope')


def test_state_dict_layout():
    from models import gan
    args = GC.make_args(512, 3)
    G, D = GC.build(gan, args)
    sd = G.state_dict()
    # names and shapes SURVEY §8b lists for the shipped checkpoints
    assert sd["blk1.conv1.weight_orig"].shape == (512, 512, 3, 3)
    assert sd["blk1.conv1.weight_u"].shape == (512,) and sd["blk1.conv1.weight_v"].shape == (4608,)
    assert sd["blk1.norm1.fc_gamma.weight"].shape == (512, 128) and "blk1.norm1.norm.running_mean" in sd
    assert sd["emb_class.weight"].shape == (200, 64) and sd["fc.weight"].shape == (16384, 128)
    assert len(sd) == 179                                   # SURVEY §2 #22: 179 entries in generator_running_avg
    assert sum(p.numel() for p in G.parameters()) > 13.0e6
    assert {"d1.conv1.weight_orig", "d2.conv4.bias", "d3.conv5.weight_orig", "d1.projector.weight"} <= set(D.state_dict())
    with pytest.raises(Exception, match="CUDA only|no CPU fallback"):
        G(torch.zeros(1, 64), torch.zeros(1, 1, dtype=torch.long))


def test_equal_to_reference_modules():
    """tests/golden/gan_init_reference.npz (make_golden_reference_state.py): the reference's models.gan built with the same
    seeds -> state-dict names, shapes, probed values and sums; positional encodings; the shipped checkpoint's layout."""
    from models import gan
    from state_probes import assert_state_matches
    d = np.load(os.path.join(GOLDEN, "gan_init_reference.npz"))
    Gm, Dm = GC.build(gan, GC.make_args(256, 2))
    assert_state_matches(Gm.state_dict(), d, "G")
    assert_state_matches(Dm.state_dict(), d, "D")
    for ny, nx in ((32, 32), (32, 16), (256, 128)):
        assert np.abs(d[f"pe_{ny}x{nx}"] - gan.positional_encoding(ny, nx)[:, ::4, ::4]).max() < 1e-12
    G5 = gan.Generator(GC.make_args(512, 3), 64)
    sd = G5.state_dict()
    assert list(sd) == [str(k) for k in d["ckpt_names"]]
    assert [",".join(map(str, v.shape)) for v in sd.values()] == [str(s) for s in d["ckpt_shapes"]]
    G5.load_state_dict(GC.checkpoint_standin(gan), strict=True)


def test_model_wrapper_and_running_average_match_the_reference_step_logic():
    """tests/golden/wrapper_reference.npz: main.py's ModelWrapper / divide_pred / update_generator_running_avg EXECUTED from the
    script's syntax tree on tiny stand-in networks (make_golden_wrapper.py).  The drop-in wrapper (gan_training.ModelWrapper)
    and the trainer's running-average update must reproduce losses, outputs and the averaged state dict."""
    import sys
    import types
    sys.path.insert(0, GOLDEN)
    import wrapper_common as WC
    from gan_training import GANTrainer, ModelWrapper
    d = np.load(os.path.join(GOLDEN, "wrapper_reference.npz"))
    for tag, nd, res in (("w21", 2, 512), ("unw", 2, 256), ("nd3", 3, 512)):
        args = WC.make_args(nd, res)
        gi, D = WC.build()
        mw = ModelWrapper(args, gi, D).train()
        x = WC.inputs()
        loss, tex, mesh = mw('g', None, x["X_alpha"], None, x["C"], None, x["noise"])
        lf, lr, _, _ = mw('d', x["X_tex"], x["X_alpha"], x["X_mesh"], x["C"], None, x["noise"])
        for got, key in ((loss, "_g_loss"), (tex, "_g_tex"), (mesh, "_g_mesh"), (lf, "_d_fake"), (lr, "_d_real")):
            ref = d[tag + key]
            assert got.shape == ref.shape, (tag, key, got.shape, ref.shape)       # incl. the [1]-shaped losses of list inputs
            assert np.abs(got.detach().numpy() - ref).max() < 1e-6, (tag, key)
        if tag != "w21":
            continue
        mw.eval()
        itex, imesh, attn = mw('inference', None, None, None, x["C"], None, x["noise"])
        assert attn is None and np.abs(itex.numpy() - d["inf_tex"]).max() < 1e-6 and np.abs(imesh.numpy() - d["inf_mesh"]).max() < 1e-6
        mw.train()
        with torch.no_grad():
            for p in mw.generator.parameters():
                p.add_(0.05 * torch.randn(p.shape, generator=torch.Generator().manual_seed(p.numel())))
            mw.generator.bn.num_batches_tracked.fill_(7)
        holder = types.SimpleNamespace(args=args, trainer=mw)
        for epoch in (5, 50, 500):
            GANTrainer.update_generator_running_avg(holder, epoch)
            for k, v in mw.generator_running_avg.state_dict().items():
                ref = d[f"avg{epoch}_{k}"]
                assert np.abs(v.numpy().astype(np.float64) - ref).max() < 1e-6, (epoch, k)
    assert float(d["w21_g_loss"][0]) != float(d["unw_g_loss"][0])    # the [2, 1] discriminator weights act at 512^2 / nd = 2 only


def test_training_iteration_matches_the_reference_loop(monkeypatch):
    """tests/golden/gan_loop_reference.npz: the training-loop body of main.py (:672-727) EXECUTED from the script's syntax tree for
    six iterations (G D D G D D) on stand-in networks / template (make_golden_gan_loop.py).  GANTrainer.step — same stand-ins,
    its flat-loss kernel replaced by the torch definition — must reproduce the loss curves, the generator, the discriminator and
    the running-average generator after both Adams."""
    sys.path.insert(0, GOLDEN)
    import recon_step_common as RS
    import wrapper_common as WC
    import gan_training as GT
    from oracle import mesh as OM
    d = np.load(os.path.join(GOLDEN, "gan_loop_reference.npz"))
    args = WC.make_args(2, 512)
    args.d_steps_per_g, args.mesh_regularization, args.lr_g, args.lr_d = 2, 0.0001, 0.01, 0.04
    monkeypatch.setattr(GT, "loss_flat", lambda mesh, norms: OM.loss_flat(mesh.ff, mesh.faces.shape[0], norms))
    gi, D = WC.build()
    tr = object.__new__(GT.GANTrainer)                         # the constructor builds the CUDA networks; wire the stand-ins instead
    tr.args, tr.mesh_template, tr.world, tr.total_it = args, RS.Template(map_size=8), 1, 0
    tr.trainer = GT.ModelWrapper(args, gi, D).train()
    tr.optimizer_g = torch.optim.Adam(tr.trainer.generator.parameters(), lr=args.lr_g, betas=(0.0, 0.9))
    tr.optimizer_d = torch.optim.Adam(tr.trainer.discriminator.parameters(), lr=args.lr_d, betas=(0.0, 0.9))
    torch.manual_seed(77)
    g_curve, d_curve = [], []
    for i in range(6):
        x = WC.inputs(seed=50 + i, B=4)
        out = tr.step(x["X_tex"], x["X_alpha"], x["X_mesh"], x["C"], epoch=0)
        (g_curve if i % 3 == 0 else d_curve).append(float(out))
    assert np.abs(np.array(g_curve) - d["g_curve"][1:]).max() < 2e-6
    assert np.abs(np.array(d_curve) - (d["d_fake_curve"][1:] + d["d_real_curve"][1:])).max() < 5e-6
    for name, mod in (("g", tr.trainer.generator), ("avg", tr.trainer.generator_running_avg), ("d", tr.trainer.discriminator)):
        for k, v in mod.state_dict().items():
            ref = d[f"{name}.{k}"]
            assert np.abs(v.numpy().astype(np.float64) - ref).max() < 1e-4, (name, k)      # Adam amplifies rounding to ~1e-5
    moved = max(np.abs(d[f"g.{k}"] - d[f"avg.{k}"]).max() for k in tr.trainer.generator.state_dict() if "num_batches" not in k)
    assert moved > 1e-3                                        # epoch 0: alpha^100, the average trails the live generator
