"""Mesh extraction on the CPU: the generated marching-cubes table (tools/gen_mc_table.py -> csrc/mc_table.h), the oracle's meshes of
analytic TSDFs (oracle/orc_mesh.c), and the mesh form of the PLY writers (C++ and Python)."""
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import mesh_cases as mc
from oracle import orc_mesh

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "tools"))
import gen_mc_table as gen  # noqa: E402

TABLE = gen.build_table()
IDENTITY = (np.eye(3, dtype=np.float32), np.zeros(3, np.float32))


def test_generator_reproduces_the_committed_header():
    assert gen.render(TABLE) == (ROOT / "dynamicfusion_b200" / "csrc" / "mc_table.h").read_text()
    assert max(len(t) for t in TABLE) == 5 and len(TABLE[0]) == len(TABLE[255]) == 0


def _inside(case, c):
    return (case >> c) & 1


def test_every_case_uses_each_crossing_edge_once():
    for case in range(256):
        polys = gen.polygons(case)
        used = sorted(e for p in polys for e in p)
        assert used == gen.crossing_edges(case), case
        assert sorted({e for t in TABLE[case] for e in t}) == gen.crossing_edges(case), case
        assert len(TABLE[case]) == sum(len(p) - 2 for p in polys)


def test_every_face_normal_points_from_inside_to_outside():
    """with the crossing edges' midpoints as vertices, each triangle's normal has a positive dot product with the sum, over its three
    edges, of the step from the edge's inside corner to its outside corner"""
    for case in range(256):
        for tri in TABLE[case]:
            p = [np.array(gen.edge_mid(e)) for e in tri]
            n = np.cross(p[1] - p[0], p[2] - p[0])
            d = np.zeros(3)
            for e in tri:
                a, b = gen.edge_corners(e)
                pa, pb = np.array(gen.corner_pos(a)), np.array(gen.corner_pos(b))
                d += (pb - pa) if _inside(case, a) else (pa - pb)
            assert n @ d > 0, (case, tri)


def test_ambiguous_faces_separate_the_inside_corners():
    """the polygon boundary of a case (triangle edges used once in the cell) runs on the cube faces; on a face with four crossings every
    boundary segment joins the two edges of one INSIDE corner; fan diagonals never lie in a face"""
    n_ambiguous = 0
    for case in range(256):
        und = {}
        for t in TABLE[case]:
            for a, b in ((t[0], t[1]), (t[1], t[2]), (t[2], t[0])):
                und[tuple(sorted((a, b)))] = und.get(tuple(sorted((a, b))), 0) + 1
        for (a, b), cnt in und.items():
            faces = [f for f in gen.FACES if a in f[4] and b in f[4]]
            if cnt == 2:
                assert not faces, (case, a, b)                      # an interior diagonal
                continue
            assert cnt == 1 and len(faces) == 1, (case, a, b)
            _, _, _, corners, fedges = faces[0]
            crossing = [e for e in fedges if e in gen.crossing_edges(case)]
            if len(crossing) == 4:
                n_ambiguous += 1
                shared = set(gen.edge_corners(a)) & set(gen.edge_corners(b))
                assert len(shared) == 1 and _inside(case, shared.pop()), (case, a, b)
    assert n_ambiguous > 0


def _mesh(orc, vol, dims, vs):
    v, k, t, (nv, nt) = orc_mesh.extract_mesh(vol, dims, (vs, vs, vs), 4 * vs, 64, IDENTITY)
    assert len(v) == nv and len(t) == nt and nt > 0
    assert np.all(np.diff(k.astype(np.int64)) > 0) and np.all(np.isfinite(v[:, :3])) and np.all(v[:, 3] == 0)
    assert t.min() >= 0 and t.max() < nv
    return v, k, t


@pytest.mark.parametrize("shape", ["sphere", "torus"])
def test_oracle_mesh_of_analytic_shapes_is_closed(orc, shape):
    dims = (48, 48, 48) if shape == "sphere" else (64, 64, 64)
    vol, vs = mc.sphere(dims) if shape == "sphere" else mc.torus(dims)
    v, k, t = _mesh(orc, vol, dims, vs)
    V, E, F = mc.check_closed_oriented(t)
    assert V == len(v)
    assert V - E + F == (2 if shape == "sphere" else 0)
    vol_mesh = mc.signed_volume(v, t)
    want = 4.0 / 3.0 * np.pi * 0.3 ** 3 if shape == "sphere" else 2 * np.pi ** 2 * 0.25 * 0.1 ** 2
    assert vol_mesh > 0 and abs(vol_mesh / want - 1) < 0.02, (vol_mesh, want)


def test_oracle_mesh_of_a_random_field_has_no_cracks(orc):
    dims = (40, 36, 44)
    vol, vs = mc.smooth_random(dims, seed=3)
    v, k, t = _mesh(orc, vol, dims, vs)
    x, y, z, axis = mc.key_coords(k, dims)
    hi = [x + (axis == 0), y + (axis == 1), z + (axis == 2)]
    border = (x == 0) | (y == 0) | (z == 0) | (hi[0] == dims[0] - 1) | (hi[1] == dims[1] - 1) | (hi[2] == dims[2] - 1)
    mc.check_closed_oriented(t, keep=lambda e: ~border[e[:, 0]] & ~border[e[:, 1]])
    assert len(t) > 2000


def _cell_cases(vol, dims):
    """case of every cell [z, y, x] (-1: a corner is inactive)"""
    Dx, Dy, Dz = dims
    a = vol.reshape(Dz, Dy, Dx)
    W = a >> 16
    F = (a & 0xffff).astype(np.uint16).view(np.float16).astype(np.float32)
    act = (W != 0) & (F != 1)
    ins = F < 0
    case = np.zeros((Dz - 1, Dy - 1, Dx - 1), np.int64)
    allact = np.ones_like(case, bool)
    for c in range(8):
        i, j, kk = c & 1, (c >> 1) & 1, c >> 2
        sl = (slice(kk, Dz - 1 + kk), slice(j, Dy - 1 + j), slice(i, Dx - 1 + i))
        case |= ins[sl].astype(np.int64) << c
        allact &= act[sl]
    return np.where(allact, case, -1)


def test_partial_observation_meshes_only_fully_observed_cells(orc):
    """unobserved (W == 0) and free-space (F == 1) corners keep their cells out of the mesh; every vertex is used by a triangle"""
    dims = (48, 40, 44)
    vol, vs = mc.sphere(dims, r=0.28)
    rng = np.random.default_rng(1)
    a = vol.reshape(dims[::-1]).copy()
    x, y, z = mc.centres(dims, vs)
    a[x > 0.62] &= 0xffff                                            # a slab never observed: W = 0
    blobs = rng.random(a.shape) < 0.02
    a[blobs] = (a[blobs] & 0xffff0000) | 0x3c00                       # scattered free-space voxels: F = 1
    vol = np.ascontiguousarray(a.reshape(-1))
    v, k, t = _mesh(orc, vol, dims, vs)
    cases = _cell_cases(vol, dims)
    meshed = (cases > 0) & (cases < 255)
    ntri = np.array([len(c) for c in TABLE])
    assert len(t) == int(ntri[cases[meshed]].sum())
    assert np.array_equal(np.unique(t), np.arange(len(v)))             # every vertex is referenced
    # every triangle lies in a meshed cell: its three edges belong to one cell with all corners active
    X, Y, Z, A = mc.key_coords(k, dims)
    for tri in t[rng.choice(len(t), 400, replace=False)]:
        ok = False
        for dy in (0, 1):
            for dz in (0, 1):
                o = [X[tri[0]], Y[tri[0]], Z[tri[0]]]
                others = [ax for ax in range(3) if ax != A[tri[0]]]
                o[others[0]] -= dy
                o[others[1]] -= dz
                if min(o) < 0 or o[0] >= dims[0] - 1 or o[1] >= dims[1] - 1 or o[2] >= dims[2] - 1 or not meshed[o[2], o[1], o[0]]:
                    continue
                off = [(X[i] - o[0], Y[i] - o[1], Z[i] - o[2]) for i in tri]
                ok |= all(0 <= c <= 1 for d in off for c in d)
        assert ok, tri


def test_oracle_counts_are_true_totals_and_overflow_writes_no_triangles(orc):
    dims = (32, 32, 32)
    vol, vs = mc.sphere(dims, r=0.25)
    v, k, t, (nv, nt) = orc_mesh.extract_mesh(vol, dims, (vs,) * 3, 4 * vs, 64, IDENTITY)
    v2, k2, t2, c2 = orc_mesh.extract_mesh(vol, dims, (vs,) * 3, 4 * vs, 64, IDENTITY, vcap=nv - 1, tcap=nt)
    assert c2 == (nv, nt) and len(v2) == nv - 1 and len(t2) == 0 and np.array_equal(v2, v[:-1])
    v3, k3, t3, c3 = orc_mesh.extract_mesh(vol, dims, (vs,) * 3, 4 * vs, 64, IDENTITY, vcap=nv, tcap=10)
    assert c3 == (nv, nt) and np.array_equal(t3, t[:10])
    empty = mc.pack(np.ones(dims[::-1]), 0)
    assert orc_mesh.extract_mesh(empty, dims, (vs,) * 3, 4 * vs, 64, IDENTITY)[3] == (0, 0)


def test_oracle_mesh_vertices_on_cloud_edges_are_cloud_points(orc):
    dims = (40, 36, 44)
    vol, vs = mc.smooth_random(dims, seed=5)
    pose = (np.array([[0, -1, 0], [1, 0, 0], [0, 0, 1]], np.float32), np.array([0.1, -0.2, 0.3], np.float32))
    v, k, t, _ = orc_mesh.extract_mesh(vol, dims, (vs,) * 3, 4 * vs, 64, pose)
    cloud = orc.extract_cloud(vol, dims, (vs,) * 3, 4 * vs, 64, pose, 10 ** 6)
    cset = {tuple(r) for r in cloud.view(np.uint32)[:, :3]}
    F = (vol & 0xffff).astype(np.uint16).view(np.float16).astype(np.float32)
    X, Y, Z, A = mc.key_coords(k, dims)
    nb = (X + (A == 0)) + dims[0] * ((Y + (A == 1)) + dims[1] * (Z + (A == 2)))
    f0, f1 = F[k.astype(np.int64) // 3], F[nb]
    strict = ((f0 > 0) & (f1 < 0)) | ((f0 < 0) & (f1 > 0))
    strict &= Z < dims[2] - 1                                          # the cloud's scan stops below the last slice
    assert strict.sum() > 1000
    assert all(tuple(r) in cset for r in v.view(np.uint32)[strict, :3])


def _read_mesh_ply(path):
    raw = Path(path).read_bytes()
    head, body = raw.split(b"end_header\n", 1)
    lines = head.decode().splitlines()
    nv = int([l for l in lines if l.startswith("element vertex")][0].split()[-1])
    nf = int([l for l in lines if l.startswith("element face")][0].split()[-1])
    props = [l.split()[-1] for l in lines if l.startswith("property float")]
    assert "property list uchar int vertex_indices" in lines
    verts = np.frombuffer(body[: nv * 4 * len(props)], "<f4").reshape(nv, len(props))
    faces = np.frombuffer(body[nv * 4 * len(props):], np.dtype([("n", "u1"), ("i", "<i4", 3)]))
    assert len(faces) == nf and np.all(faces["n"] == 3)
    return verts, props, faces["i"]


def test_mesh_ply_cpp_and_python_agree(tmp_path):
    from dynamicfusion_b200 import build
    exe = tmp_path / "ply_mesh_check"
    cmd = ["/usr/bin/g++" if Path("/usr/bin/g++").exists() else "g++", "-std=c++17", "-O1", *build.MIRROR_INC, "-o", str(exe),
           str(ROOT / "tests" / "cpp" / "ply_mesh_check.cpp")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    out = subprocess.run([str(exe), str(tmp_path)], capture_output=True, text=True)
    assert out.returncode == 0 and out.stdout.split() == ["5", "5"], out.stdout + out.stderr
    verts, props, faces = _read_mesh_ply(tmp_path / "mesh.ply")
    i = np.arange(5, dtype=np.float32)
    assert props == ["x", "y", "z", "nx", "ny", "nz"]
    assert np.array_equal(verts[:, 0], 0.25 * i) and np.array_equal(verts[:, 1], 1 - i) and np.array_equal(verts[:, 2], 0.5 + i)
    assert np.array_equal(verts[:, 3], [1, 1, 0, 1, 1])
    assert faces.tolist() == [[0, 1, 2], [2, 1, 3], [3, 4, 2]]
    v2, props2, f2 = _read_mesh_ply(tmp_path / "mesh_no_normals.ply")
    assert props2 == ["x", "y", "z"] and np.array_equal(v2, verts[:, :3]) and np.array_equal(f2, faces)
    pytest.importorskip("torch")
    from dynamicfusion_b200 import host
    vv = np.zeros((5, 4), np.float32)
    vv[:, 0], vv[:, 1], vv[:, 2] = 0.25 * i, 1 - i, 0.5 + i
    nn = np.zeros((5, 4), np.float32)
    nn[:, 0] = 1
    nn[2, 0] = np.nan
    tri = np.array([[0, 1, 2], [2, 1, 3], [3, 4, 2]], np.int32)
    assert host.save_ply(tmp_path / "py.ply", vv, nn, triangles=tri) == 5
    assert (tmp_path / "py.ply").read_bytes() == (tmp_path / "mesh.ply").read_bytes()
    assert host.save_ply(tmp_path / "py2.ply", vv, triangles=tri) == 5
    assert (tmp_path / "py2.ply").read_bytes() == (tmp_path / "mesh_no_normals.ply").read_bytes()
