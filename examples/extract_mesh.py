"""Teacher -> prior mesh -> MeshGrid -> NeuMesh, on the GPU.

    python examples/extract_mesh.py --N_grid 256 --output_dir /tmp/x [--ckpt_path teacher.pt]

Evaluates a NeuS teacher (sphere-initialised, the TEACHER_KW of examples/train_distill.py, unless a checkpoint with a
``model`` state_dict - or a bare state_dict - is given) on the dense grid, extracts the mesh with marching cubes, writes
``extracted_{obj_id}.ply`` / ``bbox_{obj_id}.json`` as the reference's extract_mesh.py does, and builds a NeuMesh on it.
"""
from __future__ import annotations

import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import neumesh_b200 as nb  # noqa: E402
from neumesh_b200 import synth  # noqa: E402

TEACHER_KW = dict(variance_init=0.05, speed_factor=10.0, W_geo_feat=256, obj_bounding_radius=1.0,
                  surface_cfg=dict(embed_multires=6, radius_init=0.5, geometric_init=True, D=8, W=256, skips=[4]),
                  radiance_cfg=dict(embed_multires=-1, embed_multires_view=4, use_view_dirs=True, D=4, W=256, skips=[]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--output_dir", required=True)
    ap.add_argument("--ckpt_path", default=None)
    ap.add_argument("--N_grid", type=int, default=256)
    ap.add_argument("--x_range", nargs=2, type=float, default=[-1.0, 1.0])
    ap.add_argument("--y_range", nargs=2, type=float, default=[-1.0, 1.0])
    ap.add_argument("--z_range", nargs=2, type=float, default=[-1.0, 1.0])
    ap.add_argument("--sdf_th", type=float, default=0.0)
    ap.add_argument("--chunk", type=int, default=2048)
    ap.add_argument("--scale_factor", type=float, default=1.0)
    ap.add_argument("--obj_id", default="0")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    teacher = nb.NeuS(**TEACHER_KW)
    if args.ckpt_path:
        ck = torch.load(args.ckpt_path, map_location="cpu")
        teacher.load_state_dict(ck.get("model", ck))
    teacher = teacher.to(dev).eval()
    mesh = nb.extract_mesh(teacher, args.N_grid, args.x_range, args.y_range, args.z_range, args.sdf_th, args.chunk,
                           args.scale_factor, args.output_dir, args.obj_id)
    grid = nb.MeshGrid(mesh, dev)
    student = nb.NeuMesh(grid, **synth.ModelConfig().model_kwargs()).to(dev).eval()   # the reference defaults
    with torch.no_grad():
        sdf = student.forward_density_only(grid.vertices[:4096])
    print("wrote %s: %d vertices, %d triangles; NeuMesh on it: %d vertices, sdf at the vertices in [%.3g, %.3g]"
          % (os.path.join(args.output_dir, "extracted_%s.ply" % args.obj_id), len(mesh.vertices), len(mesh.triangles),
             grid.vertices.shape[0], float(sdf.min()), float(sdf.max())))


if __name__ == "__main__":
    main()
