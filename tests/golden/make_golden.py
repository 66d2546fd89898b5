"""Generate ``tests/golden/*.npz`` by running the UNMODIFIED reference (``/root/reference``) on CPU.

Run in the build container only:  ``python tests/golden/make_golden.py``.
The reference holds no golden vectors of its own (SURVEY.md section 4); these files are outputs of the reference's
Python for the hot path (``models/renderer.py``, ``models/frameworks/neumesh/neumesh.py``, ``models/mesh_grid.py``) with
the one absent native dependency (``frnn``) replaced by the exact-KNN restatement in ``oracle/knn.py``.
"""
from __future__ import annotations

import hashlib
import os
import sys
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
warnings.filterwarnings("ignore")
# MKL's AVX-512 path with 8 threads, as tests/conftest.py pins it for the bit-exact comparisons
os.environ["MKL_CBWR"] = "AVX512"
torch.set_num_threads(8)

import ref_harness  # noqa: E402
from neumesh_b200 import synth  # noqa: E402


def state_digest(sd) -> str:
    h = hashlib.sha256()
    for k in sorted(sd):
        h.update(k.encode())
        h.update(sd[k].detach().cpu().numpy().tobytes())
    return h.hexdigest()


def make_case(name, level, H, W, cfg, render_kwargs, seed):
    ns = ref_harness.load()
    mesh = synth.icosphere_mesh(level, seed=seed)
    sd = synth.make_state_dict(mesh, cfg, seed=seed + 1)
    model = ref_harness.build_reference_model(mesh, cfg, sd)
    o, d = synth.frame_rays(H, W, view=3)
    torch.manual_seed(seed)
    # point queries: near-surface, mid-range and far-from-mesh points
    dirs = torch.nn.functional.normalize(torch.randn(600, 3), dim=-1)
    radii = torch.cat([0.5 + 0.05 * torch.randn(300), 0.2 + 0.8 * torch.rand(200), 1.0 + torch.rand(100)])
    xyz = dirs * radii[:, None]
    view = torch.nn.functional.normalize(torch.randn(600, 3), dim=-1)
    with torch.no_grad():
        ds, idx, w = model.compute_distance(xyz)
        sdf0 = model.forward_density_only(xyz)
    sdf1, nabla = model.forward_with_nablas(xyz.clone())
    sdf2, rgb = model.forward(xyz.clone(), view)
    with torch.no_grad():
        r_rgb, r_depth, ex = ns.renderer.volume_render(o, d, model, detailed_output=True, rayschunk=4096,
                                                       **render_kwargs)
    out = dict(
        level=np.int64(level), H=np.int64(H), W=np.int64(W), seed=np.int64(seed), view=np.int64(3),
        state_digest=np.array(state_digest(sd)),
        xyz=xyz.numpy(), view_dirs=view.numpy(), ds=ds.numpy(), idx=idx.numpy(), w=w.numpy(),
        sdf=sdf0.numpy(), nabla=nabla.detach().numpy(), sdf_with_nabla=sdf1.detach().numpy(),
        rgb_pts=rgb.detach().numpy(), sdf_forward=sdf2.detach().numpy(),
        rays_o=o.numpy(), rays_d=d.numpy(), render_rgb=r_rgb.numpy(), render_depth=r_depth.numpy(),
        render_acc=ex["mask_volume"].numpy(), render_d_final=ex["d_final"].numpy(),
        render_sdf=ex["implicit_surface"].numpy(), render_radiance=ex["radiance"].numpy(),
    )
    if "normals_volume" in ex:
        out["render_normals"] = ex["normals_volume"].numpy()
    for k, v in render_kwargs.items():
        out["kw_" + k] = np.array(v)
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


def make_train_case(name, level, n_rays, seed):
    """Gradients of a training-style loss through the UNMODIFIED reference renderer + model (config 4 semantics:
    grad enabled, calc_normal, eikonal double backward; perturb=False so that the sample positions are deterministic)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import helpers
    ns = ref_harness.load()
    cfg = synth.ModelConfig()
    mesh = synth.icosphere_mesh(level, seed=seed)
    sd = synth.make_state_dict(mesh, cfg, seed=seed + 1)
    model = ref_harness.build_reference_model(mesh, cfg, sd)
    model.train()
    o, d = synth.frame_rays(24, 24, view=2)
    sel = torch.linspace(0, o.shape[0] - 1, n_rays).long()
    o, d = o[sel].contiguous(), d[sel].contiguous()
    # record the final sample depths the reference's cascade produces (d_all is not among its outputs): the points
    # handed to forward_with_nablas are rays_o + d_all * normalize(rays_d) (renderer.py:264)
    seen = {}
    fwn = model.forward_with_nablas

    def spy(xyz):
        seen["pts"] = xyz.detach().clone()
        return fwn(xyz)

    model.forward_with_nablas = spy
    rgb, depth, ex = ns.renderer.volume_render(o, d, model, rayschunk=4096, **helpers.TRAIN_KW)
    model.forward_with_nablas = fwn
    dn = torch.nn.functional.normalize(d, dim=-1)
    d_all = ((seen["pts"].reshape(o.shape[0], -1, 3) - o[:, None, :]) * dn[:, None, :]).sum(-1)
    loss = helpers.train_loss(rgb, depth, ex)
    loss.backward()
    params = dict(model.named_parameters())
    out = dict(level=np.int64(level), seed=np.int64(seed), state_digest=np.array(state_digest(sd)),
               rays_o=o.numpy(), rays_d=d.numpy(), loss=np.float64(loss.item()), d_all=d_all.numpy())
    for k in helpers.GRAD_KEYS:
        g = params[k].grad
        out["grad_" + k] = g.numpy() if g.numel() < 20000 else g.numpy()[::7]
        out["gnorm_" + k] = np.float64(g.double().norm().item())
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes; loss", loss.item())


def make_texture_case(name, seed):
    """Point colours and a small render of the UNMODIFIED ``TextureEditableNeuMesh``
    (``editing/texture_neumesh/texture_neumesh.py``) over reference ``NeuMesh`` models."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import helpers
    ns = ref_harness.load()
    case = helpers.texture_edit_case(seed)
    main = ref_harness.build_reference_model(case["main_mesh"], case["cfg"], case["main_sd"])
    refs = [ref_harness.build_reference_model(m, case["cfg"], sd) for m, sd in case["refs"]]
    model = ns.texture_neumesh.TextureEditableNeuMesh(main, refs, case["masks"], case["codes"], T_r_m_list=case["T"])
    model.eval()
    torch.manual_seed(seed)
    dirs = torch.nn.functional.normalize(torch.randn(500, 3), dim=-1)
    radii = torch.cat([0.5 + 0.04 * torch.randn(350), 0.2 + 0.8 * torch.rand(150)])
    xyz = dirs * radii[:, None]
    view = torch.nn.functional.normalize(torch.randn(500, 3), dim=-1)
    sdf, rgb = model.forward(xyz.clone(), view)
    sdf_m, rgb_m = main.forward(xyz.clone(), view)
    o, d = synth.frame_rays(10, 10, view=5)
    kw = dict(calc_normal=False, white_bkgd=True, bounded_near_far=True)
    with torch.no_grad():
        r_rgb, r_depth, ex = ns.renderer.volume_render(o, d, model, detailed_output=False, rayschunk=4096, **kw)
    changed = (rgb.detach() - rgb_m.detach()).abs().max(-1)[0] > 1e-6
    out = dict(seed=np.int64(seed), digest_main=np.array(state_digest(case["main_sd"])),
               digest_codes=np.array(state_digest({"codes": case["codes"], "masks": case["masks"].float()})),
               xyz=xyz.numpy(), view_dirs=view.numpy(), sdf=sdf.detach().numpy(), rgb=rgb.detach().numpy(),
               rgb_unedited=rgb_m.detach().numpy(), rays_o=o.numpy(), rays_d=d.numpy(), render_rgb=r_rgb.numpy(),
               render_depth=r_depth.numpy())
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes; points recoloured by the edit:", int(changed.sum()), "of 500")


def make_neus_case(name, seed):
    """Point outputs of the UNMODIFIED NeuS teacher (models/frameworks/neus/neus.py + models/base.py)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import contextlib
    import io
    import helpers
    ns = ref_harness.load()
    with contextlib.redirect_stdout(io.StringIO()):
        model = ns.neus.NeuS(**helpers.NEUS_KW)
    sd = helpers.neus_state_dict(model, seed)
    model.load_state_dict(sd, strict=True)
    model.eval()
    torch.manual_seed(seed)
    x = (torch.rand(700, 3) * 2 - 1) * 0.8
    v = torch.nn.functional.normalize(torch.randn(700, 3), dim=-1)
    with torch.no_grad():
        sdf, rad = model.forward(x.clone(), v)
        sdf2, nabla = model.forward_with_nablas(x.clone())
        dens = model.forward_density_only(x)
    out = dict(seed=np.int64(seed), keys=np.array(sorted(model.state_dict().keys())), state_digest=np.array(state_digest(sd)),
               x=x.numpy(), view_dirs=v.numpy(), sdf=sdf.numpy(), radiance=rad.numpy(), nabla=nabla.numpy(),
               density_only=dens.numpy())
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes; |sdf| max", float(sdf.abs().max()))


def make_raycast_case(name, seed):
    """``root_finding_surface_points`` / ``sphere_tracing_surface_points`` of the UNMODIFIED ``models/ray_casting.py`` over
    the reference NeuMesh field."""
    ns = ref_harness.load()
    cfg = synth.ModelConfig()
    mesh = synth.icosphere_mesh(4, seed=seed)
    sd = synth.make_state_dict(mesh, cfg, seed=seed + 1)
    model = ref_harness.build_reference_model(mesh, cfg, sd)
    o, d = synth.frame_rays(20, 20, view=6)
    d = torch.nn.functional.normalize(d, dim=-1)
    fn = lambda x: model.forward_density_only(x).squeeze(-1)   # noqa: E731
    with torch.no_grad():
        dp, pt, mask, msc = ns.ray_casting.root_finding_surface_points(fn, o.clone(), d.clone(), near=1.5, far=3.5,
                                                                        batched=False, N_steps=128, N_secant_steps=8)
    out = dict(seed=np.int64(seed), state_digest=np.array(state_digest(sd)), rays_o=o.numpy(), rays_d=d.numpy(),
               d_pred=dp.numpy(), pt_pred=pt.numpy(), mask=mask.numpy(), mask_sign_change=msc.numpy())
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes; rays hitting the surface:", int(mask.sum()), "of", mask.numel())


def make_reference_pins(name, level, seed):
    """What the UNMODIFIED reference computes for the CPU pins of ``tests/test_oracle.py``: its model's point queries,
    its renderer on three small frames (no-grad; ``perturb=True`` under grad with ``samples_output``; ``perturb=True``
    with the uniforms handed to it through a patched ``torch.rand``) and ``rend_util.sample_pdf``."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import helpers
    ns = ref_harness.load()
    cfg = synth.ModelConfig()
    mesh = synth.icosphere_mesh(level, seed=seed)
    sd = synth.make_state_dict(mesh, cfg, seed=seed + 1)
    ref = ref_harness.build_reference_model(mesh, cfg, sd)
    # inputs, stored with the outputs: point queries, three small frames, sample_pdf bins / weights, perturb uniforms
    x, v = helpers.sample_points(500, seed=1)
    torch.manual_seed(0)
    bins = torch.sort(torch.rand(64, 40), dim=-1)[0]
    wts = torch.rand(64, 39) * (torch.rand(64, 39) > 0.5)
    inp = dict(xyz=x, view_dirs=v, pdf_bins=bins, pdf_weights=wts)
    for tag, n, view in (("render", 10, 1), ("dropin", 8, 2), ("perturb", 9, 4)):
        inp[tag + "_rays_o"], inp[tag + "_rays_d"] = synth.frame_rays(n, n, view=view)
    inp["perturb_u"] = torch.rand(4, n * n, 16, generator=torch.Generator().manual_seed(11))
    out = dict(level=np.int64(level), seed=np.int64(seed), state_digest=np.array(state_digest(sd)))
    out.update({k: t.numpy() for k, t in inp.items()})
    with torch.no_grad():
        out["sdf"] = ref.forward_density_only(x).numpy()
    s, n = ref.forward_with_nablas(x.clone())
    out["sdf_with_nabla"], out["nabla"] = s.detach().numpy(), n.detach().numpy()
    _, c = ref.forward(x.clone(), v)
    out["rgb_pts"] = c.detach().numpy()
    kw = dict(calc_normal=True, white_bkgd=True, bounded_near_far=True, detailed_output=True, rayschunk=64)
    with torch.no_grad():
        _, _, ex = ns.renderer.volume_render(inp["render_rays_o"], inp["render_rays_d"], ref, **kw)
    for k in ("rgb", "depth_volume", "mask_volume", "normals_volume", "d_final", "implicit_surface", "radiance"):
        out["render_" + k] = ex[k].numpy()
    out["pdf_samples"] = ns.rend_util.sample_pdf(inp["pdf_bins"], inp["pdf_weights"], 16, det=True).numpy()
    # the keys the reference renderer returns: the drop-in renderer must return at least these
    o, d = inp["dropin_rays_o"], inp["dropin_rays_d"]
    with torch.no_grad():
        rgb, dep, ex = ns.renderer.volume_render(o, d, ref, **kw)
    out.update(dropin_rgb=rgb.numpy(), dropin_depth=dep.numpy(), dropin_keys=np.array(sorted(ex)))
    # a training-style call: grad enabled, perturb=True (draws from torch's CPU generator), samples_output
    ref.train()
    torch.manual_seed(3)
    rgb, dep, ex = ns.renderer.volume_render(o, d, ref, calc_normal=True, detailed_output=True, samples_output=True,
                                             perturb=True, rayschunk=64)
    ref.eval()
    out.update(train_rgb=rgb.detach().numpy(), train_depth=dep.detach().numpy(), train_keys=np.array(sorted(ex)))
    # perturb=True with the uniforms injected: torch.rand is patched to hand out perturb_u, one [N, 16] slab per call
    u = inp["perturb_u"]
    calls = {"n": 0}
    real_rand = torch.rand

    def fake_rand(*shape, **kw):
        shp = tuple(shape[0]) if len(shape) == 1 and isinstance(shape[0], (list, tuple)) else tuple(shape)
        r = u[calls["n"]].reshape(shp).clone()
        calls["n"] += 1
        return r

    torch.rand = fake_rand
    try:
        with torch.no_grad():
            rgb, dep, ex = ns.renderer.volume_render(inp["perturb_rays_o"], inp["perturb_rays_d"], ref,
                                                     detailed_output=True, perturb=True, rayschunk=4096,
                                                     calc_normal=True, white_bkgd=False, bounded_near_far=True)
    finally:
        torch.rand = real_rand
    out.update(perturb_rgb=rgb.numpy(), perturb_depth=dep.numpy(), perturb_d_final=ex["d_final"].numpy(),
               perturb_rand_calls=np.int64(calls["n"]))
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


def main():
    if len(sys.argv) > 1 and sys.argv[1] == "pins":
        make_reference_pins("reference_pins_small", 3, seed=5)
        return
    if len(sys.argv) > 1 and sys.argv[1] == "raycast":
        make_raycast_case("ray_casting_small", seed=60)
        return
    if len(sys.argv) > 1 and sys.argv[1] == "neus":
        make_neus_case("neus_teacher_small", seed=50)
        return
    if len(sys.argv) > 1 and sys.argv[1] == "texture":
        make_texture_case("texture_edit_small", seed=40)
        return
    if len(sys.argv) > 1 and sys.argv[1] == "train":
        make_train_case("train_step_small", 3, 48, seed=30)
        return
    cfg = synth.ModelConfig()
    make_case("scan63like_small", 4, 12, 12, cfg,
              dict(calc_normal=True, white_bkgd=True, bounded_near_far=True), seed=10)
    cfg2 = synth.ModelConfig(enable_nablas_input=False, ln_s=0.4, learn_indicator_weight=True)
    make_case("nonabla_unbounded", 3, 10, 10, cfg2,
              dict(calc_normal=False, white_bkgd=False, bounded_near_far=False), seed=20)
    make_train_case("train_step_small", 3, 48, seed=30)
    make_texture_case("texture_edit_small", seed=40)
    make_neus_case("neus_teacher_small", seed=50)
    make_raycast_case("ray_casting_small", seed=60)
    make_reference_pins("reference_pins_small", 3, seed=5)


if __name__ == "__main__":
    main()
