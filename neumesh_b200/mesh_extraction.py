"""Mesh extraction on the GPU: drop-ins for ``mcubes.marching_cubes`` and the reference's ``extract_mesh.py``.

The reference makes the prior mesh NeuMesh trains on by evaluating a teacher on a dense grid, running PyMCubes on the
host and colouring / writing the mesh with Open3D.  Here:

* the sdf grid is evaluated on the library's kernels straight into a device volume - the value-only fused NeuS
  teacher (``neus._fused_surface_value``) or ``nmb_field_sdf`` of a ``NeuMesh`` - in row chunks whose size does not
  change a bit of the result;
* marching cubes is ``csrc/mcubes.cu`` (conventions in ``include/neumesh_b200.h`` and DESIGN.md section 4.8);
* vertex normals are ``nmb_vertex_normals`` and vertex colours the model's fused ``forward``;
* the PLY is written here (binary little-endian), since Open3D is not a dependency.

``extract_mesh`` keeps the reference's grid and vertex mapping verbatim (``extract_mesh.py:113-145``), including its
quirks, so its meshes are interchangeable with the reference's.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import json
import os

import numpy as np
import torch

from . import _lib
from .neumesh import NeuMesh
from .neus import NeuS, _fused_ok as _neus_fused_ok, _fused_surface_value
from .renderer import vertex_normals as _vertex_normals

# points per library call when evaluating the grid / the vertex colours (``chunk`` can only raise it): large enough to
# keep the GEMMs busy, small enough that the NeuS colour pass (4 row blocks of 256 fp32 activations) stays in a few GB
POINTS_PER_CALL = 1 << 19


def marching_cubes(volume: torch.Tensor, isovalue: float):
    """``mcubes.marching_cubes(volume, isovalue)`` on a CUDA fp32 volume [n0,n1,n2] -> (vertices [Nv,3] float64 in
    index space, triangles [Nt,3] int64), both on the volume's device.  Synchronises once (to size the outputs)."""
    _lib.require_cuda(volume, "marching_cubes")
    if volume.dim() != 3:
        raise ValueError("marching_cubes expects a 3-d volume, got shape %s" % (tuple(volume.shape),))
    vol = volume.detach().float().contiguous()
    n0, n1, n2 = vol.shape
    L = _lib.lib()
    dev = vol.device
    nbytes = int(L.nmb_mc_workspace_bytes(n0, n1, n2))
    if nbytes < 0:
        raise ValueError("neumesh_b200.marching_cubes: %s" % L.nmb_last_error().decode())
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    nv, nt = C.c_int64(0), C.c_int64(0)
    with torch.cuda.device(dev):
        s = _lib.stream_ptr(dev)
        _lib.check(L.nmb_mc_count(_lib.ptr(vol), n0, n1, n2, float(isovalue), _lib.ptr(ws), nbytes, C.byref(nv),
                                  C.byref(nt), s))
        verts = torch.empty(nv.value, 3, dtype=torch.float64, device=dev)
        tris = torch.empty(nt.value, 3, dtype=torch.int64, device=dev)
        if nv.value or nt.value:
            _lib.check(L.nmb_mc_emit(_lib.ptr(vol), n0, n1, n2, float(isovalue), _lib.ptr(ws), nbytes, _lib.ptr(verts),
                                     _lib.ptr(tris), s))
    return verts, tris


def grid_axes(N, x_range, y_range, z_range):
    """The reference's axes (extract_mesh.py:113-118): ``np.linspace`` in float64, cast to float32."""
    return tuple(np.linspace(r[0], r[1], N).astype(np.float32) for r in (x_range, y_range, z_range))


def sdf_volume(model, N, x_range=(-1.0, 1.0), y_range=(-1.0, 1.0), z_range=(-1.0, 1.0), chunk=2048,
               device=None) -> torch.Tensor:
    """sdf of ``model`` on the reference's grid -> CUDA fp32 [N,N,N] with ``vol[i, j, k] = f(x_j, y_i, z_k)``
    (``np.meshgrid``'s default 'xy' indexing).  Evaluated in whole rows of N*N points, at least ``chunk`` points per
    library call; the result is bit-identical for any ``chunk``."""
    if not isinstance(model, (NeuS, NeuMesh)):
        raise TypeError("extract_mesh supports neumesh_b200.NeuS and neumesh_b200.NeuMesh models, got %s"
                        % type(model).__name__)
    if device is None:
        device = next(model.parameters()).device
    device = torch.device(device)
    if device.type != "cuda":
        raise RuntimeError("neumesh_b200.sdf_volume needs a CUDA model: the kernels have no CPU implementation")
    sdf_rows = _sdf_evaluator(model)
    x, y, z = (torch.from_numpy(a).to(device) for a in grid_axes(N, x_range, y_range, z_range))
    vol = torch.empty(N, N, N, dtype=torch.float32, device=device)
    rows = max(1, -(-max(int(chunk), POINTS_PER_CALL) // (N * N)))
    with torch.no_grad():
        for i0 in range(0, N, rows):
            i1 = min(N, i0 + rows)
            xyz = torch.stack([x[None, :, None].expand(i1 - i0, N, N), y[i0:i1, None, None].expand(i1 - i0, N, N),
                               z[None, None, :].expand(i1 - i0, N, N)], dim=-1).reshape(-1, 3)
            vol[i0:i1] = sdf_rows(xyz).reshape(i1 - i0, N, N)
    return vol


def _sdf_evaluator(model):
    if isinstance(model, NeuS):
        surf = model.implicit_surface
        if not _neus_fused_ok(surf):
            raise NotImplementedError("this NeuS surface configuration has no fused CUDA evaluation")
        return lambda xyz: _fused_surface_value(surf, xyz)
    if isinstance(model, NeuMesh):
        field = model.packed_field()       # raises for configurations outside the fused kernels

        def run(xyz):
            out = torch.empty(xyz.shape[0], dtype=torch.float32, device=xyz.device)
            with torch.cuda.device(xyz.device):
                _lib.check(_lib.lib().nmb_field_sdf(field, _lib.ptr(xyz.contiguous()), xyz.shape[0], _lib.ptr(out), None,
                                                    _lib.stream_ptr(xyz.device)))
            return out
        return run
    raise TypeError("no sdf evaluator for %s" % type(model).__name__)


def map_vertices(vertices_index, N, x_range, y_range, z_range):
    """The reference's index -> world mapping, verbatim (extract_mesh.py:139-145): divided by N (not N - 1); world x
    from index 1 over the **y** range, world y from index 0 over the x range, z from index 2.  float64."""
    if torch.is_tensor(vertices_index):
        # a true division: torch's CUDA kernel turns division by a scalar into multiplication by its reciprocal
        v = vertices_index / torch.full_like(vertices_index, float(N))
    else:
        v = vertices_index / N
    out = v.clone() if torch.is_tensor(v) else v.copy()
    out[:, 0] = (y_range[1] - y_range[0]) * v[:, 1] + y_range[0]
    out[:, 1] = (x_range[1] - x_range[0]) * v[:, 0] + x_range[0]
    out[:, 2] = (z_range[1] - z_range[0]) * v[:, 2] + z_range[0]
    return out


def vertex_colors(model, vertices, view_dirs, chunk=2048):
    """``model(vertices, view_dirs)[1]`` in calls of at least ``chunk`` points (extract_mesh.py:158-167)."""
    per = max(int(chunk), POINTS_PER_CALL)
    out = torch.empty(vertices.shape[0], 3, dtype=torch.float32, device=vertices.device)
    with torch.no_grad():
        for i in range(0, vertices.shape[0], per):
            out[i:i + per] = model(vertices[i:i + per], view_dirs[i:i + per])[1].reshape(-1, 3)
    return out


class ExtractedMesh:
    """What ``extract_mesh`` returns: the mesh of the PLY as CPU tensors - vertices [V,3] float64 (scaled),
    triangles [T,3] int64, vertex_normals [V,3] float64, vertex_colors [V,3] float64 in [0, 1] as the model returned
    them.  ``MeshGrid(mesh, device)`` accepts it directly."""

    def __init__(self, vertices, triangles, vertex_normals, vertex_colors):
        self.vertices, self.triangles = vertices, triangles
        self.vertex_normals, self.vertex_colors = vertex_normals, vertex_colors


def extract_mesh(model, N_grid=256, x_range=(-1.0, 1.0), y_range=(-1.0, 1.0), z_range=(-1.0, 1.0), sdf_th=0.0,
                 chunk=2048, scale_factor=1.0, output_dir=".", obj_id="0") -> ExtractedMesh:
    """The reference's ``extract_mesh`` (extract_mesh.py:98-189): writes ``extracted_{obj_id}.ply`` and
    ``bbox_{obj_id}.json`` to ``output_dir`` and returns the mesh.  Raises ``ValueError`` if the grid has no surface
    at ``sdf_th``."""
    N = int(N_grid)
    vol = sdf_volume(model, N, x_range, y_range, z_range, chunk)
    verts_idx, tris = marching_cubes(vol, sdf_th)
    if tris.shape[0] == 0:
        lo, hi = torch.aminmax(vol)
        raise ValueError("no surface at sdf_th = %g: the sdf on the %d^3 grid ranges over [%g, %g]"
                         % (sdf_th, N, float(lo), float(hi)))
    verts = map_vertices(verts_idx, N, x_range, y_range, z_range)
    scaled = verts * scale_factor
    normals = _vertex_normals(scaled.float(), tris)
    colors = vertex_colors(model, verts.float(), -normals, chunk)
    mesh = ExtractedMesh(scaled.cpu(), tris.cpu(), normals.double().cpu(), colors.double().cpu())
    os.makedirs(output_dir, exist_ok=True)
    write_ply(os.path.join(output_dir, "extracted_%s.ply" % obj_id), mesh.vertices.numpy(), mesh.triangles.numpy(),
              mesh.vertex_normals.numpy(), mesh.vertex_colors.numpy())
    write_bbox_json(os.path.join(output_dir, "bbox_%s.json" % obj_id), mesh.vertices.numpy())
    return mesh


# ----------------------------------------------------------------------------------------------------------------
# files
# ----------------------------------------------------------------------------------------------------------------
_VERTEX_DTYPE = np.dtype([("x", "<f8"), ("y", "<f8"), ("z", "<f8"), ("nx", "<f8"), ("ny", "<f8"), ("nz", "<f8"),
                          ("red", "u1"), ("green", "u1"), ("blue", "u1")])
_FACE_DTYPE = np.dtype([("n", "u1"), ("v", "<i4", (3,))])


def write_ply(path, vertices, triangles, normals, colors):
    """Binary little-endian PLY: x y z, nx ny nz as double; red green blue as uchar round(clamp(c, 0, 1) * 255);
    faces as ``list uchar int vertex_indices``."""
    v = np.empty(len(vertices), dtype=_VERTEX_DTYPE)
    for i, k in enumerate("xyz"):
        v[k] = vertices[:, i]
        v["n" + k] = normals[:, i]
    c = np.rint(np.clip(colors, 0.0, 1.0) * 255.0).astype(np.uint8)
    v["red"], v["green"], v["blue"] = c[:, 0], c[:, 1], c[:, 2]
    f = np.empty(len(triangles), dtype=_FACE_DTYPE)
    f["n"] = 3
    f["v"] = triangles
    header = ("ply\nformat binary_little_endian 1.0\nelement vertex %d\n" % len(v)
              + "".join("property double %s\n" % k for k in ("x", "y", "z", "nx", "ny", "nz"))
              + "property uchar red\nproperty uchar green\nproperty uchar blue\n"
              + "element face %d\nproperty list uchar int vertex_indices\nend_header\n" % len(f))
    with open(path, "wb") as fh:
        fh.write(header.encode("ascii"))
        fh.write(v.tobytes())
        fh.write(f.tobytes())


def read_ply(path):
    """Reads what ``write_ply`` writes -> dict(vertices, normals float64 [V,3], colors uint8 [V,3], triangles int64)."""
    with open(path, "rb") as fh:
        data = fh.read()
    end = data.index(b"end_header\n") + len(b"end_header\n")
    header = data[:end].decode("ascii").split("\n")
    expect = ("ply\nformat binary_little_endian 1.0\nelement vertex {}\n"
              + "".join("property double %s\n" % k for k in ("x", "y", "z", "nx", "ny", "nz"))
              + "property uchar red\nproperty uchar green\nproperty uchar blue\n"
              + "element face {}\nproperty list uchar int vertex_indices\nend_header\n")
    nv = int(header[2].split()[-1])
    nf = int([h for h in header if h.startswith("element face")][0].split()[-1])
    if data[:end].decode("ascii") != expect.format(nv, nf):
        raise ValueError("%s: not a PLY in the layout write_ply produces" % path)
    v = np.frombuffer(data, dtype=_VERTEX_DTYPE, count=nv, offset=end)
    f = np.frombuffer(data, dtype=_FACE_DTYPE, count=nf, offset=end + nv * _VERTEX_DTYPE.itemsize)
    if nf and (f["n"] != 3).any():
        raise ValueError("%s: non-triangular face" % path)
    return dict(vertices=np.stack([v[k] for k in "xyz"], 1), normals=np.stack([v["n" + k] for k in "xyz"], 1),
                colors=np.stack([v[k] for k in ("red", "green", "blue")], 1),
                triangles=f["v"].astype(np.int64).reshape(-1, 3))


def write_bbox_json(path, vertices):
    """``bbox_{obj_id}.json`` as the reference writes it (extract_mesh.py:174-185): the axis-aligned bounds of the
    written (scaled) vertices."""
    lo, hi = vertices.min(axis=0), vertices.max(axis=0)
    with open(path, "wt") as fh:
        json.dump({"max_bound": hi.tolist(), "min_bound": lo.tolist(), "size": (hi - lo).tolist()}, fh, indent=4,
                  sort_keys=False)
