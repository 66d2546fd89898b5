"""Mesh extraction (``neumesh_b200.mesh_extraction``, ``csrc/mcubes.cu``): the marching-cubes tables, the numpy oracle
(``oracle/marching_cubes.py``) and the file formats on the CPU; on the GPU the CUDA marching cubes against the oracle bit
for bit, the dense teacher / NeuMesh sdf grids and ``extract_mesh`` end to end against the UNMODIFIED reference's
outputs (``tests/golden/extract_mesh_small.npz``, ``tests/golden/make_extract_golden.py``)."""
import ctypes
import json
import os

import numpy as np
import pytest
import torch

import helpers
from oracle import marching_cubes as omc
from neumesh_b200 import mesh_extraction as mx
from neumesh_b200.neus import NeuS


# ----------------------------------------------------------------------------------------------------------------
# helpers
# ----------------------------------------------------------------------------------------------------------------
def table_problems(tables):
    """-> list of violations of: used edges == sign-change edges; no degenerate triangle; interior sides shared twice
    with opposite direction; boundary segments on each face a function of that face's corner bits alone (crack-free);
    each boundary segment has only inside corners on its right (outward normal up) - the winding that makes triangle
    normals point toward values >= iso."""
    corner, edge, tri = tables["corner"], tables["edge"], tables["tri_table"]
    mid = (corner[edge[:, 0]] + corner[edge[:, 1]]) / 2.0
    faces = [(a, s) for a in range(3) for s in (0, 1)]
    seen = {}
    bad = []
    for c in range(256):
        inside = [(c >> k) & 1 for k in range(8)]
        row = [e for e in tri[c] if e >= 0]
        if len(row) % 3:
            bad.append((c, "row length"))
            continue
        ts = [tuple(row[i:i + 3]) for i in range(0, len(row), 3)]
        crossing = {e for e in range(12) if inside[edge[e, 0]] != inside[edge[e, 1]]}
        if set(row) != crossing:
            bad.append((c, "edges used != sign-change edges"))
        if any(len(set(t)) < 3 for t in ts):
            bad.append((c, "degenerate triangle"))
        sides = {}
        for t in ts:
            for a, b in ((t[0], t[1]), (t[1], t[2]), (t[2], t[0])):
                sides[(a, b)] = sides.get((a, b), 0) + 1
        if any(n > 1 for n in sides.values()):
            bad.append((c, "directed side used twice"))
        boundary = [s for s in sides if (s[1], s[0]) not in sides]
        for a, b in sides:
            if (b, a) in sides and any((mid[a, fa] == fs) and (mid[b, fa] == fs) for fa, fs in faces):
                bad.append((c, "interior side joins two edges of one face (the neighbour could draw it too)"))
        for fa, fs in faces:
            fc = [k for k in range(8) if corner[k, fa] == fs]
            on_face = [s for s in boundary if mid[s[0], fa] == fs and mid[s[1], fa] == fs]
            bits = tuple(sorted((tuple(np.delete(corner[k], fa)), inside[k]) for k in fc))
            key = (fa, bits)
            # undirected: the two cells sharing a face see it with opposite outward normals
            segs = frozenset(frozenset(tuple(np.delete(mid[e], fa)) for e in s) for s in on_face)
            if seen.setdefault(key, segs) != segs:
                bad.append((c, "face %s segments depend on more than its corners" % (key[0],)))
            nf = np.zeros(3)
            nf[fa] = 1.0 if fs else -1.0
            for s in on_face:
                p, q = mid[s[0]], mid[s[1]]
                for k in fc:
                    if np.dot(np.cross(nf, q - p), corner[k] - p) < -1e-9 and not inside[k]:
                        bad.append((c, "boundary segment with an outside corner on its right"))
        ends = [e for s in boundary for e in s]
        if sorted(ends) != sorted(list(crossing) * 2):
            bad.append((c, "boundary segments do not pass twice through every crossing edge"))
    return bad


def mesh_report(V, T):
    """-> dict(closed, manifold, oriented, euler) of an indexed triangle mesh."""
    T = np.asarray(T)
    d = np.concatenate([T[:, [0, 1]], T[:, [1, 2]], T[:, [2, 0]]])
    und = np.sort(d, axis=1)
    _, cnt = np.unique(und, axis=0, return_counts=True)
    dk = d[:, 0] * (len(V) + 1) + d[:, 1]
    rk = d[:, 1] * (len(V) + 1) + d[:, 0]
    consistent = np.unique(dk).size == dk.size            # no directed side twice: neighbours agree on orientation
    oriented = consistent and np.isin(rk, dk).all()
    used = np.unique(T).size
    return dict(closed=bool((cnt == 2).all()), manifold=bool((cnt <= 2).all()), oriented=bool(oriented),
                consistent=bool(consistent),
                euler=int(used - cnt.size + len(T)), all_used=used == len(V))


def face_normals(V, T):
    return np.cross(V[T[:, 1]] - V[T[:, 0]], V[T[:, 2]] - V[T[:, 0]])


def sphere(n, r, c=None, shape=None):
    shape = shape or (n, n, n)
    c = np.array(c if c is not None else [(s - 1) / 2.0 + 0.3 for s in shape])
    g = np.stack(np.meshgrid(*[np.arange(s, dtype=np.float64) for s in shape], indexing="ij"), -1)
    return (np.linalg.norm(g - c, axis=-1) - r).astype(np.float32), c


def torus(n, R, r):
    g = np.stack(np.meshgrid(*[np.arange(n, dtype=np.float64)] * 3, indexing="ij"), -1) - (n - 1) / 2.0 - 0.17
    q = np.sqrt(g[..., 0] ** 2 + g[..., 1] ** 2) - R
    return (np.sqrt(q ** 2 + g[..., 2] ** 2) - r).astype(np.float32)


def noise(shape, seed, border=True):
    v = np.random.default_rng(seed).standard_normal(shape).astype(np.float32)
    if border:
        v[0], v[-1], v[:, 0], v[:, -1], v[:, :, 0], v[:, :, -1] = 1, 1, 1, 1, 1, 1
    return v


# ----------------------------------------------------------------------------------------------------------------
# CPU
# ----------------------------------------------------------------------------------------------------------------
def test_tables_valid_for_all_cases():
    assert table_problems(omc.TABLES) == []
    assert omc.TABLES["tri_table"].shape[0] == 256


def test_table_checks_catch_one_wrong_edge_and_one_flipped_triangle():
    for case in (1, 0x5A, 0x7E):
        t = {k: v.copy() for k, v in omc.TABLES.items()}
        row = t["tri_table"][case]
        row[1] = (row[1] + 1) % 12 if (row[1] + 1) % 12 not in row[:3] else (row[1] + 2) % 12
        assert table_problems(t), "a wrong edge in case %d went unnoticed" % case
        t = {k: v.copy() for k, v in omc.TABLES.items()}
        row = t["tri_table"][case]
        row[1], row[2] = row[2], row[1]
        assert table_problems(t), "a flipped triangle in case %d went unnoticed" % case


def test_tables_match_their_generator():
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "tools", "gen_mc_tables.py")], capture_output=True,
                         text=True, check=True).stdout
    with open(omc.TABLES_PATH) as f:
        assert f.read() == out


@pytest.mark.parametrize("kind", ["sphere", "torus"])
def test_oracle_closed_oriented_surfaces(kind):
    n = 48
    if kind == "sphere":
        vol, c = sphere(n, 17.0)
    else:
        vol, c = torus(n, 14.0, 5.0), None
    V, T = omc.marching_cubes(vol, 0.0)
    r = mesh_report(V, T)
    assert r["closed"] and r["oriented"] and r["all_used"]
    assert r["euler"] == (2 if kind == "sphere" else 0)
    fn = face_normals(V, T)
    cen = V[T].mean(axis=1)
    if kind == "sphere":
        out = cen - c
    else:
        g = cen - ((n - 1) / 2.0 + 0.17)
        ring = g.copy()
        ring[:, 2] = 0
        ring = ring / np.linalg.norm(ring, axis=1, keepdims=True) * 14.0
        out = g - ring
    assert (np.einsum("ij,ij->i", fn, out) > 0).all(), "normals must point toward values >= iso (outward)"


def test_oracle_noise_with_positive_border_is_closed():
    for seed in range(3):
        V, T = omc.marching_cubes(noise((20, 17, 23), seed), 0.0)
        r = mesh_report(V, T)
        assert len(T) > 1000 and r["closed"] and r["manifold"] and r["oriented"]


def test_oracle_vertices_are_the_float64_interpolation():
    vol = noise((9, 8, 7), 5, border=False)
    iso = 0.123
    V, T = omc.marching_cubes(vol, iso)
    ip = np.floor(V).astype(np.int64)
    frac = V - ip
    axis = np.argmax(frac != 0, axis=1)
    exact = (frac == 0).all(axis=1)          # t == 1 lands on the next grid point
    axis[exact] = -1
    checked = 0
    v64 = vol.astype(np.float64)
    for n in range(len(V)):
        if axis[n] < 0:
            continue
        p = tuple(ip[n])
        q = list(p)
        q[axis[n]] += 1
        t = (iso - v64[p]) / (v64[tuple(q)] - v64[p])
        want = np.array(p, dtype=np.float64)
        want[axis[n]] += t
        assert np.array_equal(V[n], want)
        checked += 1
    assert checked > 100
    # order: (owner linear index, axis), strictly increasing
    keys = [(int(np.ravel_multi_index(tuple(ip[n]), vol.shape)), axis[n]) for n in range(len(V)) if axis[n] >= 0]
    assert keys == sorted(keys)


def test_oracle_exact_iso_values_give_a_consistent_mesh():
    n = 12
    i = np.arange(n, dtype=np.float32)[:, None, None] * np.ones((n, n, n), np.float32)
    V, T = omc.marching_cubes(i - 5.0, 0.0)            # the plane i = 5 passes through grid nodes
    r = mesh_report(V, T)
    assert r["manifold"] and r["consistent"] and len(T) == 2 * (n - 1) ** 2
    assert (V[:, 0] == 5.0).all()
    assert (face_normals(V, T)[:, 0] > 0).all()         # toward i > 5, where values >= iso
    q = np.rint(noise((14, 15, 16), 9) * 2).astype(np.float32)   # integer values: many grid values equal the iso
    q[0], q[-1], q[:, 0], q[:, -1], q[:, :, 0], q[:, :, -1] = 3, 3, 3, 3, 3, 3
    V, T = omc.marching_cubes(q, 1.0)
    r = mesh_report(V, T)
    assert r["closed"] and r["oriented"]


def test_reference_vertex_mapping():
    N = 10
    xr, yr, zr = (-0.9, 0.7), (-0.6, 1.0), (-0.8, 0.5)
    vi = np.array([[0.0, 0.0, 0.0], [2.5, 7.0, 9.0], [9.0, 3.25, 1.0]])
    want = np.stack([yr[0] + (yr[1] - yr[0]) * vi[:, 1] / N, xr[0] + (xr[1] - xr[0]) * vi[:, 0] / N,
                     zr[0] + (zr[1] - zr[0]) * vi[:, 2] / N], 1)
    got = mx.map_vertices(vi, N, xr, yr, zr)
    assert np.allclose(got, want, atol=1e-15, rtol=0)
    gt = mx.map_vertices(torch.from_numpy(vi), N, xr, yr, zr)
    assert torch.equal(gt, torch.from_numpy(got))
    # the grid: vol[i, j, k] = f(x_j, y_i, z_k), axes linspace in float64 cast to float32
    x, y, z = mx.grid_axes(N, xr, yr, zr)
    assert x.dtype == np.float32 and x[0] == np.float32(-0.9) and y[-1] == np.float32(1.0) and len(z) == N
    xyz = np.stack(np.meshgrid(x, y, z), -1)
    assert xyz[2, 5, 7, 0] == x[5] and xyz[2, 5, 7, 1] == y[2] and xyz[2, 5, 7, 2] == z[7]


def test_ply_round_trip_and_bbox(tmp_path):
    rng = np.random.default_rng(0)
    V = rng.standard_normal((50, 3))
    Nn = rng.standard_normal((50, 3))
    Cc = rng.uniform(-0.2, 1.2, (50, 3))
    T = rng.integers(0, 50, (70, 3))
    p = tmp_path / "m.ply"
    mx.write_ply(str(p), V, T, Nn, Cc)
    back = mx.read_ply(str(p))
    assert np.array_equal(back["vertices"], V) and np.array_equal(back["normals"], Nn)
    assert np.array_equal(back["triangles"], T)
    assert np.array_equal(back["colors"], np.rint(np.clip(Cc, 0, 1) * 255).astype(np.uint8))
    with open(p, "rb") as f:
        assert f.read(64).startswith(b"ply\nformat binary_little_endian 1.0\nelement vertex 50\n")
    mx.write_bbox_json(str(tmp_path / "b.json"), V)
    with open(tmp_path / "b.json") as f:
        b = json.load(f)
    assert list(b) == ["max_bound", "min_bound", "size"]
    assert np.allclose(b["min_bound"], V.min(0), rtol=0, atol=0) and np.allclose(b["size"], V.max(0) - V.min(0))


def test_entry_points_raise_without_cuda():
    vol = torch.zeros(4, 4, 4)
    with pytest.raises(RuntimeError):
        mx.marching_cubes(vol, 0.0)
    model = NeuS(**helpers.NEUS_KW)
    with pytest.raises(RuntimeError):
        mx.sdf_volume(model, 8)
    with pytest.raises(RuntimeError):
        mx.extract_mesh(model, 8, output_dir="/nonexistent")
    with pytest.raises(TypeError):
        mx.sdf_volume(torch.nn.Linear(3, 1), 8)


def test_c_abi_rejects_bad_input():
    from neumesh_b200 import _lib
    L = _lib.lib()
    assert L.nmb_mc_workspace_bytes(1, 4, 4) == -1 and b"dimension" in L.nmb_last_error()
    assert L.nmb_mc_workspace_bytes(4096, 4096, 4096) == -1 and b"2^34" in L.nmb_last_error()
    n = ctypes.c_int64()
    dummy = ctypes.c_void_p(256)
    rc = L.nmb_mc_count(dummy, 4, 4, 4, float("nan"), dummy, 1 << 20, ctypes.byref(n), ctypes.byref(n), None)
    assert rc != 0 and b"finite" in L.nmb_last_error()


# ----------------------------------------------------------------------------------------------------------------
# GPU
# ----------------------------------------------------------------------------------------------------------------
DEV = "cuda:0"


def _gpu_mc(vol, iso):
    V, T = mx.marching_cubes(torch.from_numpy(vol).to(DEV), iso)
    return V.cpu().numpy(), T.cpu().numpy()


def _assert_same(vol, iso):
    Vc, Tc = _gpu_mc(vol, iso)
    Vo, To = omc.marching_cubes(vol, iso)
    assert Vc.dtype == np.float64 and Tc.dtype == np.int64
    assert np.array_equal(Vc, Vo) and np.array_equal(Tc, To)
    return Vc, Tc


@pytest.mark.gpu
def test_cuda_marching_cubes_equals_oracle():
    _assert_same(noise((64, 48, 40), 1), 0.0)                      # non-cubic, positive border
    _assert_same(noise((33, 20, 45), 2, border=False), 0.37)       # iso != 0, surface touching the boundary
    _assert_same(sphere(128, 50.0)[0], 0.0)
    _assert_same(sphere(40, 30.0)[0], 2.5)                         # sphere cut by the volume's faces
    q = np.rint(noise((30, 31, 29), 3) * 2).astype(np.float32)     # exact iso values on grid points
    _assert_same(q, 1.0)
    _assert_same(q, 0.0)
    corners = np.array([[0, 0, 0], [1, 0, 0], [1, 1, 0], [0, 1, 0], [0, 0, 1], [1, 0, 1], [1, 1, 1], [0, 1, 1]])
    for c in range(256):                                           # every case on a single cell
        v = np.ones((2, 2, 2), np.float32)
        for k in range(8):
            if (c >> k) & 1:
                v[tuple(corners[k])] = -0.5 - 0.1 * k
        Vc, Tc = _assert_same(v, 0.0)
        assert len(Tc) == int((omc.TABLES["tri_table"][c] >= 0).sum()) // 3


@pytest.mark.gpu
def test_cuda_marching_cubes_repeatable_empty_and_large():
    from neumesh_b200 import _lib
    vol = torch.from_numpy(noise((70, 50, 60), 4)).to(DEV)
    n0 = _lib.launch_count()
    a = mx.marching_cubes(vol, 0.0)
    assert _lib.launch_count() - n0 >= 3
    b = mx.marching_cubes(vol, 0.0)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    V, T = mx.marching_cubes(torch.ones(16, 9, 5, device=DEV), 0.0)
    assert V.shape == (0, 3) and T.shape == (0, 3) and V.dtype == torch.float64 and T.dtype == torch.int64
    a = torch.arange(512, device=DEV, dtype=torch.float32) - 255.8
    big = (a[:, None, None] ** 2 + a[None, :, None] ** 2 + a[None, None, :] ** 2).sqrt() - 200.0
    V, T = (t.cpu().numpy() for t in mx.marching_cubes(big, 0.0))
    r = mesh_report(V, T)
    print("512^3 sphere: %d vertices, %d triangles" % (len(V), len(T)))
    assert r["closed"] and r["oriented"] and r["euler"] == 2
    with pytest.raises(RuntimeError):
        mx.marching_cubes(torch.zeros(4, 4, 4, device=DEV), float("inf"))
    with pytest.raises(ValueError):
        mx.marching_cubes(torch.zeros(1, 4, 4, device=DEV), 0.0)


def _golden(golden_dir):
    g = dict(np.load(os.path.join(golden_dir, "extract_mesh_small.npz"), allow_pickle=False))
    model = NeuS(**helpers.NEUS_KW)
    sd = helpers.neus_state_dict(model, int(g["seed"]))
    assert helpers.state_digest(sd) == str(g["state_digest"])
    model.load_state_dict(sd, strict=True)
    return g, model.eval().to(DEV)


def _grid(g, tag):
    vol = g[tag + "_volume"]
    r = g[tag + "_ranges"]
    return vol, vol.shape[0], tuple(r[0]), tuple(r[1]), tuple(r[2]), float(g[tag + "_sdf_th"]), float(g[tag + "_scale"])


@pytest.mark.gpu
def test_teacher_volume_vs_reference(golden_dir):
    from neumesh_b200 import neus as nneus
    from neumesh_b200.train_ops import CudaPrims
    g, model = _golden(golden_dir)
    for tag in ("a", "b"):
        vol, N, xr, yr, zr, _, _ = _grid(g, tag)
        v1 = mx.sdf_volume(model, N, xr, yr, zr, chunk=1)
        v2 = mx.sdf_volume(model, N, xr, yr, zr, chunk=N * N * N)
        assert torch.equal(v1, v2), "the volume must not depend on the chunk size"
        e = (v1.cpu() - torch.from_numpy(vol)).abs().max().item()
        print("teacher volume %s vs the unmodified reference: %.2e" % (tag, e))
        assert e <= 5e-6
    # the value-only path computes the value rows of the full fused surface, bit for bit
    x = (torch.rand(3000, 3, generator=torch.Generator().manual_seed(0)) * 2 - 1).to(DEV)
    with torch.no_grad():
        s_full = model.forward_with_nablas(x)[0]
    assert torch.equal(nneus._fused_surface_value(model.implicit_surface, x), s_full)
    # epilogue 3: bias + softplus(beta = 100, threshold = 20)
    gen = torch.Generator().manual_seed(1)
    A = (torch.randn(777, 150, generator=gen) * 0.1).to(DEV)
    W = (torch.randn(300, 150, generator=gen) * 0.1).to(DEV)
    b = (torch.randn(300, generator=gen) * 0.1).to(DEV)
    Z = torch.empty(777, 300, device=DEV)
    CudaPrims(DEV).gemm(A, 150, True, W, 150, True, Z, 300, 777, 300, 150, bias=b, epilogue=3)
    ref = torch.nn.functional.softplus(A.double() @ W.double().T + b.double(), beta=100)
    e = (Z.double() - ref).abs().max().item()
    print("epilogue 3 vs torch (float64): %.2e" % e)
    assert e <= 1e-5


@pytest.mark.gpu
def test_extract_mesh_teacher_end_to_end(golden_dir, tmp_path):
    import neumesh_b200 as nb
    from neumesh_b200 import _lib
    g, model = _golden(golden_dir)
    for tag in ("a", "b"):
        vol, N, xr, yr, zr, th, scale = _grid(g, tag)
        vc = mx.sdf_volume(model, N, xr, yr, zr).cpu().numpy()
        assert np.array_equal(vc < th, vol < th), "a grid value changed side of sdf_th: the meshes cannot match"
        n0 = _lib.launch_count()
        out = str(tmp_path / tag)
        mesh = nb.extract_mesh(model, N, xr, yr, zr, th, 2048, scale, out, tag)
        torch.cuda.synchronize()
        assert _lib.launch_count() - n0 > 10
        Vo, To = omc.marching_cubes(vol, th)
        assert np.array_equal(mesh.triangles.numpy(), To)
        # vertices: t moves by at most |dv| / |v1 - v0| along the edge, |dv| <= 5e-6 (the teacher bar) at both ends
        Vi, Ti = omc.marching_cubes(vc, th)
        assert np.array_equal(Ti, To)
        v64 = vol.astype(np.float64).reshape(-1)
        ip = np.floor(Vo).astype(np.int64)
        axis = np.argmax(Vo - ip != 0, axis=1)
        lin = np.ravel_multi_index(tuple(np.minimum(ip, N - 1).T), vol.shape)
        step = np.array([N * N, N, 1])[axis]
        dv = np.abs(v64[np.minimum(lin + step, v64.size - 1)] - v64[lin])
        bound = 1e-5 / np.maximum(dv, 1e-12)
        err_idx = np.abs(Vi - Vo).max(axis=1)
        assert (err_idx <= bound + 1e-12).all()
        want = mx.map_vertices(Vi, N, xr, yr, zr) * scale
        assert np.array_equal(mesh.vertices.numpy(), want)
        ec = np.abs(mesh.vertex_colors.numpy() - g[tag + "_colors"]).max()
        print("extract_mesh %s: %d vertices, %d triangles, max |colour - reference| = %.2e"
              % (tag, len(mesh.vertices), len(mesh.triangles), ec))
        assert ec <= 1e-4
        back = mx.read_ply(os.path.join(out, "extracted_%s.ply" % tag))
        assert np.array_equal(back["vertices"], mesh.vertices.numpy())
        assert np.array_equal(back["triangles"], To)
        with open(os.path.join(out, "bbox_%s.json" % tag)) as f:
            bb = json.load(f)
        assert np.allclose(bb["min_bound"], mesh.vertices.numpy().min(0), rtol=0, atol=0)
        grid = nb.MeshGrid(mesh, torch.device(DEV))
        assert grid.vertices.shape[0] == len(mesh.vertices)
    with pytest.raises(ValueError, match="ranges over"):
        nb.extract_mesh(model, 16, sdf_th=5.0, output_dir=str(tmp_path / "none"))


@pytest.mark.gpu
def test_extract_mesh_neumesh(tmp_path):
    import neumesh_b200 as nb
    from neumesh_b200 import synth
    cfg = synth.ModelConfig()
    mesh = synth.icosphere_mesh(3, seed=7)
    sd = synth.make_state_dict(mesh, cfg, seed=8)
    model = helpers.cuda_model(mesh, cfg, sd)
    oracle = helpers.oracle_field(mesh, cfg, sd)
    N = 40
    vol = mx.sdf_volume(model, N).cpu()
    x, y, z = (torch.from_numpy(a) for a in mx.grid_axes(N, (-1, 1), (-1, 1), (-1, 1)))
    pts = torch.stack(torch.meshgrid(y, x, z, indexing="ij"), -1)[..., [1, 0, 2]].reshape(-1, 3)
    _, idx_o, _ = oracle.compute_distance(pts)
    with torch.no_grad():
        _, idx_c, _ = model.compute_distance(pts.to(DEV))
    same = (idx_o == idx_c.cpu()).all(dim=-1)
    assert same.float().mean() > 0.999
    with torch.no_grad():
        so = oracle.forward_density_only(pts).reshape(-1)
    e = (vol.reshape(-1) - so)[same].abs().max().item()
    print("NeuMesh volume vs the oracle field: %.2e (%d KNN ties skipped)" % (e, int((~same).sum())))
    assert e <= 5e-6
    th = float(vol.median())
    res = nb.extract_mesh(model, N, sdf_th=th, output_dir=str(tmp_path), obj_id="nm")
    Vo, To = omc.marching_cubes(vol.numpy(), th)
    assert np.array_equal(res.triangles.numpy(), To)
    assert np.array_equal(res.vertices.numpy(), mx.map_vertices(Vo, N, (-1, 1), (-1, 1), (-1, 1)))
    vf = torch.from_numpy(res.vertices.numpy()).float()
    dirs = -res.vertex_normals.float()
    _, idx_o, _ = oracle.compute_distance(vf)
    with torch.no_grad():
        _, idx_c, _ = model.compute_distance(vf.to(DEV))
    same = (idx_o == idx_c.cpu()).all(dim=-1)
    with torch.no_grad():
        co = oracle.forward(vf, dirs)[1].reshape(-1, 3)
    ec = (res.vertex_colors.float() - co)[same].abs().max().item()
    print("NeuMesh extract: %d triangles, colours vs the oracle field %.2e" % (len(To), ec))
    assert ec <= 1e-5
