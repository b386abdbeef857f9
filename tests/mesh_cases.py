"""Analytic TSDF volumes and mesh topology checks shared by tests/test_mesh_model.py (CPU oracle) and tests/test_mesh_gpu.py."""
import numpy as np


def pack(F, W) -> np.ndarray:
    """packed u32 voxels (fp16 TSDF in the low half, u16 weight in the high half), flattened in (z, y, x) order"""
    h = np.asarray(F, np.float32).astype(np.float16).view(np.uint16).astype(np.uint32)
    return np.ascontiguousarray((h | (np.asarray(W, np.uint32) << 16)).reshape(-1))


def centres(dims, vs):
    """voxel centres as arrays indexed [z, y, x] (extraction positions voxel x at (x + 0.5) * vs)"""
    z, y, x = np.meshgrid(*[(np.arange(d) + 0.5) * vs for d in dims[::-1]], indexing="ij")
    return x, y, z


def sphere(dims=(48, 48, 48), r=0.3, trunc_vox=4.0):
    """fully observed sphere of radius r (metres) in a 1 m cube; F < 0 inside"""
    vs = 1.0 / dims[0]
    x, y, z = centres(dims, vs)
    d = np.sqrt((x - 0.5) ** 2 + (y - 0.5) ** 2 + (z - 0.5) ** 2) - r
    return pack(np.clip(d / (trunc_vox * vs), -1, 1), 1), vs


def torus(dims=(64, 64, 64), R=0.25, r=0.1, trunc_vox=4.0):
    vs = 1.0 / dims[0]
    x, y, z = centres(dims, vs)
    q = np.sqrt((x - 0.5) ** 2 + (y - 0.5) ** 2) - R
    d = np.sqrt(q ** 2 + (z - 0.5) ** 2) - r
    return pack(np.clip(d / (trunc_vox * vs), -1, 1), 1), vs


def smooth_random(dims=(40, 36, 44), seed=0):
    """seeded random smooth field crossing zero all over the volume, fully observed (|F| < 1 everywhere: no free-space voxel)"""
    from scipy.ndimage import gaussian_filter
    rng = np.random.default_rng(seed)
    f = gaussian_filter(rng.standard_normal(dims[::-1]), 3.0)
    return pack(0.95 * f / np.abs(f).max(), 1), 1.0 / dims[0]


def edges_of(tris: np.ndarray):
    """directed half-edges (a -> b) of the triangles, [3m, 2]"""
    return np.concatenate([tris[:, [0, 1]], tris[:, [1, 2]], tris[:, [2, 0]]])


def check_closed_oriented(tris: np.ndarray, keep=None):
    """every undirected edge (optionally: those `keep` selects) has exactly two triangles and they traverse it in opposite directions;
    returns (V, E, F) of the referenced vertices"""
    he = edges_of(tris)
    und = np.sort(he, 1)
    uniq, inv, cnt = np.unique(und, axis=0, return_inverse=True, return_counts=True)
    sel = np.ones(len(uniq), bool) if keep is None else keep(uniq)
    assert np.all(cnt[sel] == 2), f"{np.count_nonzero(cnt[sel] != 2)} edges without exactly two triangles"
    # orientation: the two half-edges of an edge point opposite ways
    fwd = (he[:, 0] < he[:, 1]).astype(np.int64)
    nfwd = np.bincount(inv.reshape(-1), weights=fwd, minlength=len(uniq))
    assert np.all(nfwd[sel] == 1), f"{np.count_nonzero(nfwd[sel] != 1)} edges with inconsistent orientation"
    return len(np.unique(tris)), len(uniq), len(tris)


def signed_volume(verts: np.ndarray, tris: np.ndarray) -> float:
    v = verts[:, :3].astype(np.float64)
    a, b, c = v[tris[:, 0]], v[tris[:, 1]], v[tris[:, 2]]
    return float(np.einsum("ij,ij->i", a, np.cross(b, c)).sum() / 6.0)


def face_normals(verts: np.ndarray, tris: np.ndarray) -> np.ndarray:
    v = verts[:, :3].astype(np.float64)
    return np.cross(v[tris[:, 1]] - v[tris[:, 0]], v[tris[:, 2]] - v[tris[:, 0]])


def key_coords(keys: np.ndarray, dims):
    """(owner voxel x, y, z, axis) of edge keys"""
    keys = keys.astype(np.int64)
    v, axis = keys // 3, keys % 3
    return v % dims[0], (v // dims[0]) % dims[1], v // (dims[0] * dims[1]), axis
