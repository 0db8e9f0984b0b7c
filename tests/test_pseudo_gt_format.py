"""The pseudo-ground-truth record format (data/pseudo_gt.py) on the CPU: round trip, dtypes, and that the reference's own
dataset class reads our files and mirrors textures identically (stored golden)."""
import os
import sys
import types

import numpy as np
import torch

from conftest import GOLDEN

sys.path.insert(0, GOLDEN)
import pseudogt_common as PC          # noqa: E402


def _record(seed=0, R=32):
    from data.pseudo_gt import make_record
    return PC.record(make_record, seed, R)


def test_round_trip_and_dtypes(tmp_path):
    from data.pseudo_gt import load_pseudo_ground_truth, pseudo_gt_dir, save_pseudo_gt
    rec = _record()
    assert rec['texture'].dtype == torch.float16 and rec['texture_alpha'].dtype == torch.float16
    assert rec['image'].dtype == torch.float16 and rec['mesh'].dtype == torch.float32
    save_pseudo_gt(pseudo_gt_dir(str(tmp_path), 32), 7, rec)
    assert os.path.exists(os.path.join(str(tmp_path), "pseudogt_32x32", "7.npz"))
    out = load_pseudo_ground_truth(str(tmp_path), 32, 7)
    assert set(out) == {'image', 'texture', 'texture_alpha', 'mesh'}
    assert out['image'].shape == (3, 16, 16) and out['image'].dtype == torch.float32
    assert torch.equal(out['image'], rec['image'][:3].float() / 2 + 0.5)
    assert torch.equal(out['texture'], rec['texture'].float()) and torch.equal(out['mesh'], rec['mesh'])
    assert float(out['image'].min()) >= -1e-3 and float(out['image'].max()) <= 1 + 1e-3


def test_mirror_tex_is_an_involution_with_half_turn_shift():
    from data.pseudo_gt import mirror_tex
    t = torch.arange(2 * 3 * 8, dtype=torch.float32).reshape(2, 3, 8)
    m = mirror_tex(t)
    assert m.shape == t.shape and torch.equal(mirror_tex(m), t)
    # flip, then rotate u by half a turn: each half of the map is reversed in place
    assert torch.equal(m[..., :4], t[..., :4].flip(2)) and torch.equal(m[..., 4:], t[..., 4:].flip(2))


def test_visibility_to_mask():
    from data.pseudo_gt import visibility_to_mask
    v = torch.zeros(1, 3, 8, 8)
    v[0, 1, 2:4, 2:4] = 0.5
    m = visibility_to_mask(v, 16)
    assert m.shape == (1, 16, 16, 1) and set(m.unique().tolist()) <= {0.0, 1.0}
    assert m[0, 5, 5, 0] == 1 and m[0, 0, 0, 0] == 0 and m[0, 15, 15, 0] == 0


def test_poses_metadata_round_trip(tmp_path):
    from data.pseudo_gt import load_poses_metadata, save_poses_metadata
    s, t, r = torch.rand(5, 1), torch.rand(5, 2), torch.rand(5, 4)
    save_poses_metadata(str(tmp_path), s, t, r, [f"img{i}.jpg" for i in range(5)])
    d = load_poses_metadata(str(tmp_path))
    assert torch.equal(d['scale'], s) and torch.equal(d['rotation'], r) and d['path'][3] == "img3.jpg"


def test_reference_dataset_reads_our_records(tmp_path):
    """tests/golden/pseudogt_dataset_reference.npz (make_golden_reference_state.py): the reference's own
    AbstractDataset.load_pseudo_ground_truth reading the record this module writes, and its mirror_tex of the texture."""
    from data.pseudo_gt import load_pseudo_ground_truth, mirror_tex, pseudo_gt_dir, save_pseudo_gt
    theirs = np.load(os.path.join(GOLDEN, "pseudogt_dataset_reference.npz"))
    cache = os.path.join(str(tmp_path), "cache", "cub")
    save_pseudo_gt(pseudo_gt_dir(cache, 32), 0, _record(seed=3))
    ours = load_pseudo_ground_truth(cache, 32, 0)
    assert set(theirs.files) == set(ours) | {"mirror_texture"}
    for k in ours:
        assert ours[k].dtype == torch.from_numpy(theirs[k]).dtype and np.array_equal(ours[k].numpy(), theirs[k]), k
    assert np.array_equal(mirror_tex(ours['texture']).numpy(), theirs["mirror_texture"])


def test_export_pipeline_matches_the_reference_export_loop(tmp_path):
    """tests/golden/pseudogt_reference.npz: the export loop of run_reconstruction.py (:542-604) with its nested InverseRenderer
    (:506-527) EXECUTED from the script's syntax tree through the reference's own MeshTemplate / Renderer classes
    (make_golden_pseudogt.py).  The construction the GPU tests compare the CUDA renderer with (tests/test_inverse_renderer_gpu.py:
    oracle render with a differentiable texture -> autograd visibility; UV-space render of the photograph) plus the drop-in's
    host pieces (DatasetParams, visibility_to_mask, make_record, save / load) must reproduce the records it wrote."""
    from conftest import GOLDEN
    sys.path.insert(0, GOLDEN)
    import pseudogt_common as PC
    from data.pseudo_gt import load_pseudo_ground_truth, make_record, pseudo_gt_dir, save_pseudo_gt, visibility_to_mask
    from models.reconstruction import DatasetParams
    from oracle import mesh as M
    d = np.load(os.path.join(GOLDEN, "pseudogt_reference.npz"))
    path = M.write_uvsphere_obj(str(tmp_path / "uvsphere_16rings.obj"), rings=16)
    T = M.TemplateData(M.load_obj(path), path)
    net = PC.build_net().eval()
    dp = DatasetParams(types.SimpleNamespace(optimize_deltas=True, optimize_z0=False), 10)
    with torch.no_grad():
        dp.ds_translation.copy_(torch.tensor(d["ds_translation"]))
        dp.ds_scale.copy_(torch.tensor(d["ds_scale"]))
    seen = []
    for net_image, inception_image, hd_image, s, t, q, indices in PC.batches():
        with torch.no_grad():
            pred_tex, mesh_map = net(net_image)
            td, sd = dp(indices.squeeze(-1), 'deltas')
            vtx = M.transform_vertices(M.get_vertex_positions(T, mesh_map), s, t, q, scale_delta=sd, translation_delta=td)
        tex = pred_tex.clone().requires_grad_(True)
        img, _, _ = M.forward_renderer(T, vtx, tex, PC.RENDER, PC.RENDER)
        vis, = torch.autograd.grad(img, tex, torch.ones_like(img))
        with torch.no_grad():
            B = hd_image.shape[0]
            uvs = (vtx[..., :2] + 1) / 2
            verts = torch.cat((T.uvs.unsqueeze(0) * 2 - 1, torch.zeros(1, T.uvs.shape[0], 1)), dim=-1).expand(B, -1, -1)
            outs = []
            for idx in ([0, 1, 2], [3, 3, 3]):             # three channels per pass, as the CUDA InverseRenderer does
                o, hard, _, _ = M.render(verts, T.face_textures, uvs, hd_image[:, idx], ft=T.faces, H=PC.PSEUDO, W=PC.PSEUDO, return_hardmask=True)
                outs.append(o)
            inverse_tex = torch.cat((outs[0], outs[1][..., :1]), dim=3)
            mask = visibility_to_mask(vis, PC.PSEUDO)
            inverse_tex, inverse_alpha = (inverse_tex * mask).permute(0, 3, 1, 2), (hard * mask).permute(0, 3, 1, 2)
        for i, idx in enumerate(indices.view(-1).tolist()):
            rec = make_record(mesh_map[i], inverse_tex[i], inverse_alpha[i], inception_image[i])
            assert np.abs(rec['mesh'].numpy() - d[f"{idx}.mesh"]).max() < 1e-7
            assert np.array_equal(rec['image'].numpy(), d[f"{idx}.image"])
            # fp16 records: at most one unit in the last place apart (fp32 render differences of 1e-6 can flip a rounding)
            assert np.array_equal(rec['texture_alpha'].numpy(), d[f"{idx}.texture_alpha"])
            assert np.abs(rec['texture'].float().numpy() - d[f"{idx}.texture"].astype(np.float32)).max() <= 1e-3
            assert rec['texture'].shape == (4, PC.PSEUDO, PC.PSEUDO) and rec['texture_alpha'].shape == (1, PC.PSEUDO, PC.PSEUDO)
            save_pseudo_gt(pseudo_gt_dir(str(tmp_path), PC.PSEUDO), idx, rec)
            back = load_pseudo_ground_truth(str(tmp_path), PC.PSEUDO, idx)
            assert torch.equal(back['texture_alpha'], torch.tensor(d[f"{idx}.texture_alpha"]).float())
            seen.append(idx)
    assert sorted(seen) == [0, 1, 2, 13]
    assert 0.3 < float(np.mean([float((d[f"{i}.texture_alpha"] != 0).mean()) for i in seen])) < 0.95
