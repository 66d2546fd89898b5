"""CPU tests: the oracle (and, on CPU, the drop-in model and renderer) is pinned against the committed golden vectors
that the UNMODIFIED reference produced (``tests/golden/make_golden.py``), bit for bit where the same torch ops run in
the same order."""
import os

import numpy as np
import pytest
import torch

import helpers
from neumesh_b200 import synth
from oracle import knn as oknn
from oracle import render as orender

GOLDEN = ["scan63like_small.npz", "nonabla_unbounded.npz"]


@pytest.mark.parametrize("name", GOLDEN)
def test_oracle_field_matches_reference_golden(golden_dir, name):
    g, mesh, cfg, sd, kw = helpers.golden_case(os.path.join(golden_dir, name))
    f = helpers.oracle_field(mesh, cfg, sd)
    xyz, view = torch.from_numpy(g["xyz"]), torch.from_numpy(g["view_dirs"])
    ds, idx, w = f.compute_distance(xyz)
    assert torch.equal(idx, torch.from_numpy(g["idx"]))
    assert torch.equal(ds, torch.from_numpy(g["ds"]))
    assert torch.equal(w, torch.from_numpy(g["w"]))
    assert torch.equal(f.forward_density_only(xyz), torch.from_numpy(g["sdf"]))
    sdf, nabla = f.forward_with_nablas(xyz)
    assert torch.equal(nabla, torch.from_numpy(g["nabla"]))
    sdf2, rgb = f.forward(xyz, view)
    assert torch.equal(rgb, torch.from_numpy(g["rgb_pts"]))
    assert torch.equal(sdf2, torch.from_numpy(g["sdf_forward"]))


@pytest.mark.parametrize("name", GOLDEN)
def test_oracle_render_matches_reference_golden(golden_dir, name):
    g, mesh, cfg, sd, kw = helpers.golden_case(os.path.join(golden_dir, name))
    f = helpers.oracle_field(mesh, cfg, sd)
    rgb, depth, ex = orender.volume_render(torch.from_numpy(g["rays_o"]), torch.from_numpy(g["rays_d"]), f,
                                           detailed_output=True, **kw)
    # bit-exact: same torch ops in the same order on the same platform
    assert torch.equal(rgb, torch.from_numpy(g["render_rgb"]))
    assert torch.equal(depth, torch.from_numpy(g["render_depth"]))
    assert torch.equal(ex["mask_volume"], torch.from_numpy(g["render_acc"]))
    assert torch.equal(ex["d_final"], torch.from_numpy(g["render_d_final"]))
    if "render_normals" in g:
        assert torch.equal(ex["normals_volume"], torch.from_numpy(g["render_normals"]))


def test_knn_oracle_brute_vs_kdtree():
    mesh = synth.icosphere_mesh(4, seed=3)
    p = torch.from_numpy(mesh.vertices).float()
    q, _ = helpers.sample_points(3000, seed=7)
    d_b, i_b = oknn.knn_exact(q, p, 8, method="brute")
    d_k, i_k = oknn.knn_exact(q, p, 8, method="kdtree")
    assert torch.equal(i_b, i_k) and torch.equal(d_b, d_k)
    assert (d_b[:, 1:] >= d_b[:, :-1]).all()
    # frnn call-site contract (mesh_grid.py:109-119): batch dim 1, squared distances, int64, 4-tuple
    dists, idxs, nn_, grid = oknn.frnn_grid_points(q[None], p[None], None, None, K=8, r=100.0, grid=None)
    assert dists.shape == (1, 3000, 8) and idxs.dtype == torch.int64 and nn_ is None and grid is not None
    assert torch.allclose(dists[0, :, 0], ((q - p[idxs[0, :, 0]]) ** 2).sum(-1), atol=1e-7)


def _pins(golden_dir):
    g, mesh, cfg, sd, _ = helpers.golden_case(os.path.join(golden_dir, "reference_pins_small.npz"))
    t = {k: torch.from_numpy(v) for k, v in g.items() if v.dtype == np.float32}
    return g, t, mesh, cfg, sd


def test_oracle_vs_unmodified_reference(golden_dir):
    """The oracle's field, renderer and inverse-CDF sampler equal, bit for bit, what the unmodified reference computed
    for the same inputs (``tests/golden/make_golden.py pins``)."""
    g, t, mesh, cfg, sd = _pins(golden_dir)
    f = helpers.oracle_field(mesh, cfg, sd)
    x, v = t["xyz"], t["view_dirs"]
    assert torch.equal(t["sdf"], f.forward_density_only(x))
    s_o, n_o = f.forward_with_nablas(x)
    assert torch.equal(t["nabla"], n_o) and torch.equal(t["sdf_with_nabla"], s_o)
    _, c_o = f.forward(x, v)
    assert torch.equal(t["rgb_pts"], c_o)
    kw = dict(calc_normal=True, white_bkgd=True, bounded_near_far=True)
    rgb_o, dep_o, ex_o = orender.volume_render(t["render_rays_o"], t["render_rays_d"], f, detailed_output=True,
                                               rayschunk=64, **kw)
    for k in ("rgb", "depth_volume", "mask_volume", "normals_volume", "d_final", "implicit_surface", "radiance"):
        assert torch.equal(t["render_" + k], ex_o[k]), k
    # sample_pdf on its own, incl. the u = 0 / u = 1 ends (SURVEY.md section 8a')
    assert torch.equal(t["pdf_samples"], orender.inverse_cdf_samples(t["pdf_bins"], t["pdf_weights"], 16))


def test_reference_renderer_and_trainer_loss_run_on_the_dropin_model(golden_dir):
    """INTEGRATION.md section 3 end to end, as far as a CPU allows: the drop-in ``neumesh_b200.NeuMesh`` loads the
    reference's state_dict and, driven by the drop-in renderer and by the oracle's restatement of the reference renderer
    (``models/renderer.py::volume_render``), renders what the reference renders with its own model; under autograd with
    ``perturb=True`` it returns every key the reference's renderer returns to the trainer, and its loss back-propagates."""
    import neumesh_b200 as nb
    g, t, mesh, cfg, sd = _pins(golden_dir)
    ours = nb.NeuMesh(helpers.OracleMeshGrid(mesh), **cfg.model_kwargs())
    ours.load_state_dict(sd, strict=True)      # identical state_dict keys
    ours.eval()
    o, d = t["dropin_rays_o"], t["dropin_rays_d"]
    rgb_r, dep_r = t["dropin_rgb"], t["dropin_depth"]
    kw = dict(calc_normal=True, white_bkgd=True, bounded_near_far=True, detailed_output=True, rayschunk=64)
    with torch.no_grad():
        rgb_o, dep_o, _ = orender.volume_render(o, d, ours, **kw)                 # reference renderer (restated), drop-in model
        rgb_n, dep_n, ex_n = nb.volume_render(o, d, ours, **kw)                   # drop-in renderer, drop-in model
    assert set(g["dropin_keys"]) <= set(ex_n.keys()) | {"near_far"}
    for a, b in ((rgb_o, rgb_r), (dep_o, dep_r), (rgb_n, rgb_r), (dep_n, dep_r)):
        assert (a - b).abs().max() < 1e-5
    # training-style call: grad enabled, perturb=True (the reference's default), samples_output for the distillation loss
    ours.train()
    ours.fused_train = False
    torch.manual_seed(3)
    rgb_t, dep_t, ex_t = nb.volume_render(o, d, ours, calc_normal=True, detailed_output=True, samples_output=True,
                                          perturb=True, rayschunk=64)
    assert {"xyz", "dirs", "density", "colors", "implicit_nablas"} <= set(g["train_keys"]) <= set(ex_t.keys())
    assert (rgb_t - t["train_rgb"]).abs().max() < 1e-5 and (dep_t - t["train_depth"]).abs().max() < 1e-5
    loss = helpers.train_loss(rgb_t, dep_t, ex_t) + ex_t["density"].abs().mean() + ex_t["colors"].mean()
    loss.backward()
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for n, p in ours.named_parameters()
               if n != "indicator_weight_raw")


def test_oracle_perturb_with_injected_uniforms_equals_reference_with_patched_rand(golden_dir):
    """perturb=True (rend_util.py:292-295) draws ``torch.rand`` once per up-sampling iteration; the oracle takes the draws
    as ``perturb_u``.  The reference, with ``torch.rand`` patched to hand it the same draws, drew them four times and
    rendered what the oracle renders, bit for bit."""
    g, t, mesh, cfg, sd = _pins(golden_dir)
    f = helpers.oracle_field(mesh, cfg, sd)
    o, d, u = t["perturb_rays_o"], t["perturb_rays_d"], t["perturb_u"]
    assert int(g["perturb_rand_calls"]) == u.shape[0] == 4
    kw = dict(calc_normal=True, white_bkgd=False, bounded_near_far=True)
    rgb_o, dep_o, ex_o = orender.volume_render(o, d, f, detailed_output=True, perturb_u=u, **kw)
    assert torch.equal(t["perturb_rgb"], rgb_o) and torch.equal(t["perturb_depth"], dep_o)
    assert torch.equal(t["perturb_d_final"], ex_o["d_final"])
    # and it differs from the deterministic render (the draws are used)
    rgb_d, _, _ = orender.volume_render(o, d, f, **kw)
    assert not torch.equal(rgb_d, rgb_o)
