"""Marching cubes in numpy: the specification ``csrc/mcubes.cu`` is held to, bit for bit.

Same tables (parsed from ``neumesh_b200/csrc/mc_tables.cuh``), same rules, same output order:

* a grid point is inside iff ``value < iso`` (fp32 values compared in float64);
* one vertex per crossing grid edge, owned by the edge's lower end ``p``: ``p + t e_a`` with
  ``t = (iso - v(p)) / (v(p + e_a) - v(p))`` in float64 (numpy does not contract, so these are the kernel's bits);
* vertices ordered by (owner's C-order linear index, axis); triangles by (cell linear index = linear index of the
  cell's lowest corner, position in the case table);
* the right-hand normal of every triangle points toward values >= iso.
"""
from __future__ import annotations

import os
import re

import numpy as np

TABLES_PATH = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "neumesh_b200", "csrc",
                           "mc_tables.cuh")


def _array(text, name):
    m = re.search(r"static const \w+ %s\[[^=]*=\s*\{(.*?)\};" % name, text, re.S)
    return np.array([int(v, 0) for v in re.findall(r"-?0x[0-9a-fA-F]+|-?\d+", m.group(1))], dtype=np.int64)


def load_tables(path=TABLES_PATH):
    """-> dict(corner [8,3], edge [12,2], edge_table [256], tri_table [256, W]) as the CUDA header defines them."""
    with open(path) as f:
        text = f.read()
    width = int(re.search(r"#define\s+NMB_MC_TRI_WIDTH\s+(\d+)", text).group(1))
    return dict(corner=_array(text, "MC_CORNER").reshape(8, 3), edge=_array(text, "MC_EDGE").reshape(12, 2),
                edge_table=_array(text, "MC_EDGE_TABLE").reshape(256),
                tri_table=_array(text, "MC_TRI_TABLE").reshape(256, width))


TABLES = load_tables()


def edge_owner_axis(tables=TABLES):
    """-> (owner corner offset [12,3], axis [12]) of each cube edge."""
    c, e = tables["corner"], tables["edge"]
    a, b = c[e[:, 0]], c[e[:, 1]]
    lo = np.minimum(a, b)
    axis = np.argmax(a != b, axis=1)
    return lo, axis


def marching_cubes(volume, iso, tables=TABLES):
    """volume [n0,n1,n2] (fp32), iso -> (vertices [Nv,3] float64 index space, triangles [Nt,3] int64)."""
    vol = np.ascontiguousarray(volume, dtype=np.float32)
    if vol.ndim != 3 or min(vol.shape) < 2:
        raise ValueError("marching cubes needs a 3-d volume with every dimension >= 2")
    iso = float(iso)
    if not np.isfinite(iso):
        raise ValueError("the isovalue must be finite")
    n0, n1, n2 = vol.shape
    v = vol.astype(np.float64)
    inside = v < iso
    flags = np.zeros(vol.shape + (3,), dtype=bool)
    flags[:-1, :, :, 0] = inside[:-1] != inside[1:]
    flags[:, :-1, :, 1] = inside[:, :-1] != inside[:, 1:]
    flags[:, :, :-1, 2] = inside[:, :, :-1] != inside[:, :, 1:]
    flat = flags.reshape(-1, 3)
    p, a = np.nonzero(flat)                                   # C order over (point, axis)
    vid = np.full(flat.shape, -1, dtype=np.int64)
    vid[p, a] = np.arange(p.size, dtype=np.int64)
    step = np.array([n1 * n2, n2, 1], dtype=np.int64)
    vf = v.reshape(-1)
    v0, v1 = vf[p], vf[p + step[a]]
    t = (iso - v0) / (v1 - v0)
    verts = np.stack(np.unravel_index(p, vol.shape), axis=1).astype(np.float64)
    verts[np.arange(p.size), a] += t

    cs = np.zeros((n0 - 1, n1 - 1, n2 - 1), dtype=np.int64)
    for c, (dx, dy, dz) in enumerate(tables["corner"]):
        cs |= inside[dx:n0 - 1 + dx, dy:n1 - 1 + dy, dz:n2 - 1 + dz].astype(np.int64) << c
    cells = np.nonzero(cs.reshape(-1))[0]                      # C order over cells == C order over lowest corners
    ci = np.stack(np.unravel_index(cells, cs.shape), axis=1)
    rows = tables["tri_table"][cs.reshape(-1)[cells]]
    r, col = np.nonzero(rows >= 0)                             # row-major: (cell, position in the case table)
    e = rows[r, col]
    lo, axis = edge_owner_axis(tables)
    owner = ci[r] + lo[e]
    lin = (owner[:, 0] * n1 + owner[:, 1]) * n2 + owner[:, 2]
    tris = vid[lin, axis[e]].reshape(-1, 3)
    return verts, tris
