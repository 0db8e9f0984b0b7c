"""Shared recipe of the GAN golden test: identical construction (same seeds -> same weights, verified equal to the
reference's in the authoring container) and identical synthetic inputs for the reference (CPU) and the CUDA modules."""
import types

import torch


def make_args(res=256, nd=2):
    return types.SimpleNamespace(texture_resolution=res, conditional_class=True, conditional_color=False,
                                 conditional_text=False, norm_g='syncbatch', norm_d='none', n_classes=(200,),
                                 mask_output=True, texture_only=False, num_discriminators=nd, text_embedding_dim=256)


def build(gan_module, args, seed=123):
    torch.manual_seed(seed)
    G = gan_module.Generator(args, 64, symmetric=True, mesh_head=True)
    D = gan_module.MultiScaleDiscriminator(args, 4)
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():       # the mesh head is zero-initialised: give it a signal so the test sees it
        G.conv_mesh.weight.copy_(torch.randn(G.conv_mesh.weight.shape, generator=g) * 0.02)
        G.conv_mesh.bias.copy_(torch.randn(G.conv_mesh.bias.shape, generator=g) * 0.02)
    return G, D


def checkpoint_standin(gan_module, seed=2024):
    """A generator_running_avg state dict in the layout of the shipped CUB checkpoint (512^2, nd = 3), built from seeds so
    that it can travel with the tests: same-seed weights, non-trivial batch-norm running statistics, and spectral-norm
    vectors u, v from 30 float64 power iterations (eval mode divides each weight by u^T W v with the stored vectors, as it
    does with a trained checkpoint)."""
    G, _ = build(gan_module, make_args(512, 3), seed=seed)
    sd = G.state_dict()
    g = torch.Generator().manual_seed(seed + 2)
    with torch.no_grad():
        for k, v in sd.items():
            if k.endswith("running_mean"):
                v.copy_(0.1 * torch.randn(v.shape, generator=g))
            elif k.endswith("running_var"):
                v.copy_(0.5 + torch.rand(v.shape, generator=g))
        for k in [k for k in sd if k.endswith("_orig")]:
            base = k[: -len("orig")]
            W = sd[k].double().reshape(sd[k].shape[0], -1)
            u = sd[base + "u"].double()
            for _ in range(30):
                v = torch.nn.functional.normalize(W.t() @ u, dim=0)
                u = torch.nn.functional.normalize(W @ v, dim=0)
            sd[base + "u"].copy_(u)
            sd[base + "v"].copy_(v)
    return sd


def inputs(args, B=2, seed=5):
    g = torch.Generator().manual_seed(seed)
    R = args.texture_resolution
    z = torch.randn(B, 64, generator=g)
    c = torch.randint(0, 200, (B, 1), generator=g)
    alpha = (torch.rand(B, 1, R // 8, R // 8, generator=g) > 0.4).float()
    alpha = torch.nn.functional.interpolate(alpha, size=(R, R), mode='bilinear', align_corners=False)
    tex = torch.rand(B, 3, R, R, generator=g) * 2 - 1
    mesh = torch.randn(B, 3, 32, 32, generator=g) * 0.05
    return z, c, alpha, tex, mesh


def g_step(G, D, crit, z, c, alpha, d_weight=None):
    """ModelWrapper.forward mode 'g' (main.py:491-498)."""
    pred_tex, pred_mesh = G(z, c)
    x_fake = torch.cat((pred_tex * alpha, alpha), dim=1)
    out, mask = D(x_fake, pred_mesh, c)
    loss = crit(out, True, for_discriminator=False, mask=mask, weight=d_weight)
    return loss, pred_tex, pred_mesh, out, mask


def d_step(G, D, crit, z, c, alpha, tex, mesh, d_weight=None):
    """ModelWrapper.forward mode 'd' (main.py:499-521)."""
    with torch.no_grad():
        pred_tex, pred_mesh = G(z, c)
        x_fake = torch.cat((pred_tex * alpha, alpha), dim=1)
        x_real = torch.cat((tex, alpha), dim=1)
        x = torch.cat((x_fake, x_real), dim=0)
        cc = torch.cat((c, c), dim=0)
        m = torch.cat((pred_mesh, mesh), dim=0)
    out, mask = D(x, m, cc)
    B = z.shape[0]
    fake, real = [o[:B] for o in out], [o[B:] for o in out]
    mf, mr = [k[:B] for k in mask], [k[B:] for k in mask]
    loss_fake = crit(fake, False, for_discriminator=True, mask=mf, weight=d_weight)
    loss_real = crit(real, True, for_discriminator=True, mask=mr, weight=d_weight)
    return loss_fake, loss_real, out
