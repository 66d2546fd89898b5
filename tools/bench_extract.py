"""Mesh-extraction benchmark: ``python tools/bench_extract.py`` -> one JSON line.

For N = 256 and 512, the sphere-initialised NeuS teacher (``examples/train_distill.py``'s TEACHER_KW) and a synthetic
NeuMesh model (``synth`` icosphere), times the stages of ``extract_mesh`` with CUDA events: sdf grid, marching cubes,
normals + colours, PLY write (host), and the end-to-end call.  Also reports counts, the sdf GEMMs' FLOP/s (from shapes)
and the marching cubes' bytes/s (volume read twice + workspace + outputs), plus the numpy oracle's marching-cubes time
at 256^3 - the only comparison arm: the reference's path (PyMCubes + Open3D) is not installed.
Reads the device name and power limit in the same run."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import neumesh_b200 as nb  # noqa: E402
from neumesh_b200 import mesh_extraction as mx, synth  # noqa: E402
from oracle import marching_cubes as omc  # noqa: E402

TEACHER_KW = dict(variance_init=0.05, speed_factor=10.0, W_geo_feat=256, obj_bounding_radius=1.0,
                  surface_cfg=dict(embed_multires=6, radius_init=0.5, geometric_init=True, D=8, W=256, skips=[4]),
                  radiance_cfg=dict(embed_multires=-1, embed_multires_view=4, use_view_dirs=True, D=4, W=256, skips=[]))


def teacher_flops_per_point(surf):
    """2 * sum(in * out) over the value-only surface MLP (last layer: the sdf row only)."""
    f = 0
    for i, lin in enumerate(surf.surface_fc_layers):
        w = lin.weight_v if hasattr(lin, "weight_v") else lin.weight
        out = 1 if i == len(surf.surface_fc_layers) - 1 else w.shape[0]
        f += 2 * w.shape[1] * out
    return f


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    r = fn()
    b.record()
    b.synchronize()
    return r, a.elapsed_time(b)


def run(model, N, out_dir, flops_pp):
    rng = ((-1.0, 1.0),) * 3
    mx.extract_mesh(model, 64, *rng, 0.0, 2048, 1.0, out_dir, "warm")          # warm-up: modules, pools
    vol, t_sdf = timed(lambda: mx.sdf_volume(model, N, *rng))
    (V, T), t_mc = timed(lambda: mx.marching_cubes(vol, 0.0))

    def shade():
        verts = mx.map_vertices(V, N, *rng)
        n = mx._vertex_normals(verts.float(), T)
        return verts, n, mx.vertex_colors(model, verts.float(), -n)
    (verts, n, c), t_col = timed(shade)
    t0 = time.perf_counter()
    mx.write_ply(os.path.join(out_dir, "b.ply"), verts.cpu().numpy(), T.cpu().numpy(), n.double().cpu().numpy(),
                 c.double().cpu().numpy())
    t_ply = 1e3 * (time.perf_counter() - t0)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    mx.extract_mesh(model, N, *rng, 0.0, 2048, 1.0, out_dir, "e2e")
    torch.cuda.synchronize()
    e2e = time.perf_counter() - t0
    P = N ** 3
    mc_bytes = 2 * 4 * P + 4 * P + 2 * 4 * P + V.shape[0] * 24 + T.shape[0] * 24   # vol x2, ws write + reads, outputs
    r = dict(N=N, vertices=int(V.shape[0]), triangles=int(T.shape[0]), ms_sdf_grid=round(t_sdf, 3),
             ms_marching_cubes=round(t_mc, 3), ms_normals_colors=round(t_col, 3), ms_ply_write=round(t_ply, 3),
             s_end_to_end=round(e2e, 4), mc_GBps=round(mc_bytes / (t_mc * 1e-3) / 1e9, 1))
    if flops_pp:
        r["sdf_gemm_TFLOPs"] = round(flops_pp * P / (t_sdf * 1e-3) / 1e12, 2)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[256, 512])
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_extract measures the CUDA path: it needs a GPU"
    dev = torch.device("cuda:0")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    torch.manual_seed(0)
    teacher = nb.NeuS(**TEACHER_KW).to(dev).eval()
    cfg = synth.ModelConfig()
    mesh = synth.icosphere_mesh(5, seed=0)
    neumesh = nb.NeuMesh(nb.MeshGrid(mesh, dev), **cfg.model_kwargs())
    neumesh.load_state_dict(synth.make_state_dict(mesh, cfg, seed=1))
    neumesh = neumesh.to(dev).eval()
    res = dict(device=torch.cuda.get_device_name(0), nvidia_smi=q, teacher=[], neumesh=[])
    with tempfile.TemporaryDirectory() as d:
        for N in args.sizes:
            res["teacher"].append(run(teacher, N, d, teacher_flops_per_point(teacher.implicit_surface)))
            res["neumesh"].append(run(neumesh, N, d, 0))
        vol = mx.sdf_volume(teacher, 256).cpu().numpy()
    t0 = time.perf_counter()
    omc.marching_cubes(vol, 0.0)
    res["oracle_numpy_mc_256_ms"] = round(1e3 * (time.perf_counter() - t0), 1)
    res["reference_arm"] = "not run: PyMCubes and Open3D are not installed"
    print(json.dumps(res))


if __name__ == "__main__":
    main()
