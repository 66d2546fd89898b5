"""Generate ``tests/golden/extract_mesh_small.npz`` by running the UNMODIFIED reference NeuS teacher on CPU.

Run in the build container only:  ``python tests/golden/make_extract_golden.py``.
The reference's ``extract_mesh.py`` imports mcubes and open3d at module level, so it cannot be imported; its grid
(``extract_mesh.py:113-136``) and vertex mapping (``:139-145``) lines are restated here as data-generation code.
"""
from __future__ import annotations

import contextlib
import io
import os
import sys
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(ROOT, "tests"))
warnings.filterwarnings("ignore")
# MKL's AVX-512 path with 8 threads, as tests/conftest.py pins it for the bit-exact comparisons
os.environ["MKL_CBWR"] = "AVX512"
torch.set_num_threads(8)

import helpers  # noqa: E402
import ref_harness  # noqa: E402
from oracle.marching_cubes import marching_cubes  # noqa: E402

EXTRACT_GRIDS = (
    # (tag, N, x_range, y_range, z_range, sdf_th, scale_factor): the default cube, then unequal ranges that pin the
    # reference's x/y range swap in its vertex mapping
    ("a", 32, (-1.0, 1.0), (-1.0, 1.0), (-1.0, 1.0), -0.08, 1.0),
    ("b", 24, (-0.9, 0.7), (-0.6, 1.0), (-0.8, 0.5), -0.08, 2.0),
)


def make_extract_case(name, seed):
    """The sdf grid of ``extract_mesh.py:113-136`` over the reference NeuS teacher (``model(xyz, zeros)[0]`` in 2 048-point
    chunks) for ``EXTRACT_GRIDS``, and the teacher's colours at the vertices of the oracle's marching cubes of each
    volume, mapped as ``extract_mesh.py:139-145`` maps them, with ``-normals`` (area-weighted) in float64 numpy."""
    ns = ref_harness.load()
    with contextlib.redirect_stdout(io.StringIO()):
        model = ns.neus.NeuS(**helpers.NEUS_KW)
    sd = helpers.neus_state_dict(model, seed)
    model.load_state_dict(sd, strict=True)
    model.eval()
    out = dict(seed=np.int64(seed), state_digest=np.array(helpers.state_digest(sd)))
    for tag, N, xr, yr, zr, th, scale in EXTRACT_GRIDS:
        x, y, z = np.linspace(*xr, N), np.linspace(*yr, N), np.linspace(*zr, N)
        xyz = torch.from_numpy(np.stack(np.meshgrid(x, y, z), -1).reshape(-1, 3).astype(np.float32))
        with torch.no_grad():
            sdf = torch.cat([model(xyz[i:i + 2048], torch.zeros_like(xyz[i:i + 2048]))[0]
                             for i in range(0, xyz.shape[0], 2048)], 0)
        vol = sdf.numpy().reshape(N, N, N)
        verts, tris = marching_cubes(vol, th)
        v = (verts / N).astype(np.float64)
        xw = (yr[1] - yr[0]) * v[:, 1] + yr[0]
        yw = (xr[1] - xr[0]) * v[:, 0] + xr[0]
        v[:, 0], v[:, 1] = xw, yw
        v[:, 2] = (zr[1] - zr[0]) * v[:, 2] + zr[0]
        vs = v * scale
        fn = np.cross(vs[tris[:, 1]] - vs[tris[:, 0]], vs[tris[:, 2]] - vs[tris[:, 0]])
        nrm = np.zeros_like(vs)
        for c in range(3):
            np.add.at(nrm, tris[:, c], fn)
        nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
        pts, dirs = torch.from_numpy(v.astype(np.float32)), torch.from_numpy((-nrm).astype(np.float32))
        with torch.no_grad():
            col = torch.cat([model(pts[i:i + 2048], dirs[i:i + 2048])[1] for i in range(0, pts.shape[0], 2048)], 0)
        # the mesh itself is the oracle's marching cubes of the stored volume; only the colours need the reference
        out.update({tag + "_volume": vol, tag + "_colors": col.numpy(), tag + "_ranges": np.array([xr, yr, zr]),
                    tag + "_sdf_th": np.float64(th), tag + "_scale": np.float64(scale)})
        print(tag, "sdf range", float(vol.min()), float(vol.max()), "vertices", len(v), "triangles", len(tris))
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    make_extract_case("extract_mesh_small", seed=50)
