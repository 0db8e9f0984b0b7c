"""MeshTemplate (SURVEY §8 row a10) against the REFERENCE's own class: tests/golden/template_reference.npz was produced by
running /root/reference/code/rendering/mesh_template.py:MeshTemplate unmodified on the CPU (make_golden_template.py: a
stand-in supplies the one kaolin call, OBJ loading, and `.cuda()`).  Checked here, on the procedural UV spheres that travel
with the repo (16 and 31 rings, symmetric and not): the oracle's restatement (oracle/mesh.py TemplateData, get_vertex_positions,
adjust_uv_and_texture, compute_normals) — which thereby becomes PINNED — and the drop-in rendering/mesh_template.py on its
torch path.  Index sets, topology maps and UVs must be identical; floating-point results within 2e-6.  The shipped OBJ templates
(stored under tests/golden/) are checked through probes."""
import os
import tempfile

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle import mesh as M

G = np.load(os.path.join(GOLDEN, "template_reference.npz"))
CASES = [(r, s) for r in (16, 31) for s in (True, False)]


def _path(rings):
    return M.write_uvsphere_obj(os.path.join(tempfile.mkdtemp(), f"uvsphere_{rings}rings.obj"), rings=rings)


def _close(a, ref, tol=2e-6):
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    assert a.shape == ref.shape, (a.shape, ref.shape)
    assert float(np.abs(a - ref).max()) <= tol, float(np.abs(a - ref).max())


@pytest.mark.parametrize("rings,sym", CASES)
def test_oracle_restatement_equals_the_reference_class(rings, sym):
    tag = f"proc{rings}_{'sym' if sym else 'asym'}"
    path = _path(rings)
    T = M.TemplateData(M.load_obj(path), path, is_symmetric=sym)
    assert np.array_equal(T.pos_indices.numpy(), G[tag + "_pos"]) and np.array_equal(T.neg_indices.numpy(), G[tag + "_neg"])
    assert np.array_equal(T.nonneg_indices.numpy(), G[tag + "_nonneg"])
    assert np.array_equal(T.ff.numpy(), G[tag + "_ff"].astype(np.int64))
    _close(T.topo_map, G[tag + "_topo"], 0.0)
    _close(T.tangent_map, G[tag + "_tangent"], 1e-7)
    _close(T.symmetry_mask, G[tag + "_symmask"], 0.0)
    dmap, tex = torch.tensor(G[tag + "_dmap"]), torch.tensor(G[tag + "_tex"])
    vtx = M.get_vertex_positions(T, dmap)
    _close(vtx, G[tag + "_vtx"])
    _close(M.compute_normals(T, vtx), G[tag + "_normals"])
    uvs, padded = M.adjust_uv_and_texture(T, tex)
    _close(uvs[0], G[tag + "_uvs"], 0.0)
    _close(padded, G[tag + "_padded"], 0.0)


@pytest.mark.parametrize("rings,sym", CASES)
def test_drop_in_template_equals_the_reference_class(rings, sym):
    from rendering.mesh_template import MeshTemplate
    tag = f"proc{rings}_{'sym' if sym else 'asym'}"
    t = MeshTemplate(_path(rings), is_symmetric=sym, device="cpu")
    assert np.array_equal(t.pos_indices.numpy(), G[tag + "_pos"]) and np.array_equal(t.neg_indices.numpy(), G[tag + "_neg"])
    assert np.array_equal(t.nonneg_indices.numpy(), G[tag + "_nonneg"])
    assert np.array_equal(t.mesh.ff.numpy(), G[tag + "_ff"].astype(np.int64))
    _close(t.topo_map, G[tag + "_topo"], 0.0)
    _close(t.tangent_map, G[tag + "_tangent"], 1e-7)
    _close(t.symmetry_mask, G[tag + "_symmask"], 0.0)
    dmap, tex, deltas = (torch.tensor(G[tag + k]) for k in ("_dmap", "_tex", "_deltas"))
    vtx = t.get_vertex_positions(dmap)
    _close(vtx, G[tag + "_vtx"])
    _close(t.compute_normals(vtx), G[tag + "_normals"])
    _close(t.deform(deltas), G[tag + "_deform"])
    uvs, padded = t.adjust_uv_and_texture(tex)
    _close(uvs[0], G[tag + "_uvs"], 0.0)
    _close(padded, G[tag + "_padded"], 0.0)
    counts = G[tag + "_counts"]
    assert (len(t.pos_indices), len(t.neg_indices), t.mesh.vertices.shape[0], t.mesh.faces.shape[0], t.mesh.uvs.shape[0]) == \
        (counts[0], counts[1], counts[3], counts[4], counts[5])


@pytest.mark.parametrize("rings", [16, 31])
def test_shipped_templates_through_probes(rings):
    path = os.path.join(GOLDEN, f"uvsphere_{rings}rings.obj")          # the reference's shipped template, stored verbatim
    from rendering.mesh_template import MeshTemplate
    tag = f"ship{rings}_sym"
    g = torch.Generator().manual_seed(int(G[tag + "_dmap_seed"][0]))
    dmap = torch.randn(2, 3, 32, 32, generator=g) * 0.05
    T = M.TemplateData(M.load_obj(path), path, is_symmetric=True)
    t = MeshTemplate(path, is_symmetric=True, device="cpu")
    for vtx, normals in ((M.get_vertex_positions(T, dmap), None), (t.get_vertex_positions(dmap), None)):
        _close(vtx[:, ::37], G[tag + "_vtx_probe"])
        assert float(np.abs(vtx.double().sum(dim=1).numpy() - G[tag + "_vtx_sum"]).max()) < 1e-4
    _close(t.compute_normals(t.get_vertex_positions(dmap))[:, ::53], G[tag + "_normals_probe"])
    assert (len(t.pos_indices), len(t.neg_indices), t.mesh.vertices.shape[0], t.mesh.faces.shape[0]) == \
        tuple(G[tag + "_counts"][[0, 1, 3, 4]])


def test_oracle_render_wiring_equals_the_reference_renderer():
    """tests/golden/renderer_reference.npz: the reference's Renderer.forward run unmodified with the oracle's rasteriser
    standing in for kaolin's (make_golden_renderer.py) — pins everything around the rasteriser in oracle/mesh.py:render."""
    d = np.load(os.path.join(GOLDEN, "renderer_reference.npz"))
    path = _path(16)
    T = M.TemplateData(M.load_obj(path), path)
    H = int(d["H"][0])
    mesh_map, q, s, t, tex, bg = (torch.tensor(d[k]) for k in ("mesh_map", "q", "s", "t", "tex", "bg"))
    vtx = M.transform_vertices(M.get_vertex_positions(T, mesh_map), s, t, q)
    p3d, p2d, nrm = M.ortho_projection(vtx, T.faces)
    for a, k in ((p3d, "p3d"), (p2d, "p2d"), (nrm, "normal")):
        _close(a, d[k], 0.0)
    uvs, padded = M.adjust_uv_and_texture(T, tex)
    img, alpha, n1, _ = M.render(vtx, T.faces, uvs, padded, T.face_textures, H, H)
    _close(img, d["img"], 0.0)
    _close(alpha, d["alpha"], 0.0)
    _close(n1, d["normal1"], 0.0)
    img_bg, hard, _, _ = M.render(vtx, T.faces, uvs, padded, T.face_textures, H, H, background_image=bg, return_hardmask=True)
    _close(img_bg, d["img_bg"], 0.0)
    _close(hard, d["hard"], 0.0)
    img_noft, _, _, _ = M.render(vtx, T.faces, uvs[:, :T.vertices.shape[0]], padded, None, H, H)
    _close(img_noft, d["img_noft"], 0.0)
    # the convenience wrapper the GPU tests call
    img2, alpha2, _ = M.forward_renderer(T, vtx, tex, H, H)
    _close(img2, d["img"], 0.0)
    _close(alpha2, d["alpha"], 0.0)
