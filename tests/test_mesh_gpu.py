"""GPU mesh extraction (dfusion.h df_extract_mesh / df_kinfu_extract_mesh) against the CPU oracle (oracle/orc_mesh.c), the cloud, the
normals and the frame loop."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from dynamicfusion_b200 import capi, host, kinfu as kf, synth  # noqa: E402
import mesh_cases as mc  # noqa: E402
from oracle import orc_mesh  # noqa: E402

K = synth.DEFAULT_K


def _umbrella_volume(dims, frames=3, track=False):
    v = host.TsdfVolume(dims, track_activity=track)
    v.setTruncDist(0.04); v.setMaxWeight(64); v.setSize((1.0, 1.0, 1.0)); v.setPose(synth.volume_pose(1.0))
    v.setGradientDeltaFactor(0.5); v.clear()
    for t in range(frames):
        dists = host.computeDists(host.u16_to_device(synth.umbrella_depth(t)), K)
        R, tr = synth.camera_drift(4 * t)
        v.integrate(dists, (R.astype(np.float32), tr.astype(np.float32)), K)
    return v


def _gpu_mesh(v, vcap=2_000_000, tcap=4_000_000, normals=False):
    verts, nrm, keys, tris, counts = v.fetchMesh(vcap, tcap, normals=normals)
    nv, nt = (int(c) for c in counts.cpu().numpy())
    n, m = min(nv, vcap), (min(nt, tcap) if nv <= vcap else 0)
    out = (verts[:n].cpu().numpy(), keys[:n].cpu().numpy().view(np.uint32), tris[:m].cpu().numpy(), (nv, nt))
    return out + ((nrm[:n].cpu().numpy(),) if normals else ())


def _oracle_mesh(orc, v):
    return orc_mesh.extract_mesh(v.data_.cpu().numpy().view(np.uint32), v.getDims(), v.getVoxelSize(), v.getTruncDist(), v.getMaxWeight(), v.pose_)


@pytest.mark.parametrize("dims", [(64, 64, 64), (96, 96, 96), (61, 50, 47)])
def test_mesh_matches_oracle_bit_for_bit(orc, dims):
    """vertices, edge keys, triangles and counts equal the oracle's, in order; the activity-map path equals the full scan
    (61 x 50 x 47: the one-voxel-per-thread path)"""
    full = _umbrella_volume(dims)
    tracked = _umbrella_volume(dims, track=True)
    assert torch.equal(full.data_, tracked.data_)
    g = _gpu_mesh(full)
    r = _oracle_mesh(orc, full)
    assert g[3] == r[3] and r[3][1] > 1000, (g[3], r[3])
    assert np.array_equal(g[0].view(np.uint32), r[0].view(np.uint32))
    assert np.array_equal(g[1], r[1]) and np.array_equal(g[2], r[2])
    a = _gpu_mesh(tracked)
    assert a[3] == g[3] and np.array_equal(a[0].view(np.uint32), g[0].view(np.uint32)) and np.array_equal(a[1], g[1]) and np.array_equal(a[2], g[2])
    # run to run: bit-identical
    b = _gpu_mesh(tracked)
    assert np.array_equal(a[0].view(np.uint32), b[0].view(np.uint32)) and np.array_equal(a[2], b[2])


def test_mesh_vertices_on_cloud_edges_are_cloud_points():
    v = _umbrella_volume((96, 96, 96))
    verts, keys, tris, _ = _gpu_mesh(v)
    pts, cnt = v.fetchCloud(1_000_000)
    cloud = pts[: int(cnt.item())].cpu().numpy()
    dims = tuple(int(d) for d in v.getDims())
    vol = v.data_.cpu().numpy().view(np.uint32)
    F = (vol & 0xffff).astype(np.uint16).view(np.float16).astype(np.float32)
    act = ((vol >> 16) != 0) & (F != 1)
    X, Y, Z, A = mc.key_coords(keys, dims)
    own = keys.astype(np.int64) // 3
    nb = (X + (A == 0)) + dims[0] * ((Y + (A == 1)) + dims[1] * (Z + (A == 2)))
    strict = (((F[own] > 0) & (F[nb] < 0)) | ((F[own] < 0) & (F[nb] > 0))) & act[own] & act[nb] & (Z < dims[2] - 1)
    assert strict.sum() > 5000
    cset = {tuple(r) for r in cloud.view(np.uint32)[:, :3]}
    assert all(tuple(r) in cset for r in verts.view(np.uint32)[strict, :3])


def test_face_normals_agree_with_extracted_normals():
    v = _umbrella_volume((96, 96, 96))
    verts, keys, tris, _, nrm = _gpu_mesh(v, normals=True)
    fn = mc.face_normals(verts, tris)
    vn = nrm[:, :3].astype(np.float64)[tris].sum(1)
    ok = np.isfinite(vn).all(1) & (np.linalg.norm(fn, axis=1) > 0)
    assert ok.mean() > 0.9
    frac = np.mean(np.einsum("ij,ij->i", fn[ok], vn[ok]) > 0)
    assert frac >= 0.99, frac


def test_capacities_counts_and_empty_volume():
    v = _umbrella_volume((64, 64, 64))
    lib = capi.load()
    ws = torch.empty(lib.df_extract_mesh_workspace_bytes(v._vol()), dtype=torch.uint8, device="cuda")
    _, _, tris_all, (nv, nt) = _gpu_mesh(v)

    def run(vcap, tcap):
        verts = torch.full((vcap + 64, 4), -7.0, device="cuda")
        keys = torch.full((vcap + 64,), -7, dtype=torch.int32, device="cuda")
        tris = torch.full((tcap + 64, 3), -7, dtype=torch.int32, device="cuda")
        counts = torch.full((2,), -1, dtype=torch.int32, device="cuda")
        capi.check(lib.df_extract_mesh(v._vol(), capi.make_aff(*v.pose_), None, verts.data_ptr(), keys.data_ptr(), vcap, tris.data_ptr(), tcap,
                                       counts.data_ptr(), ws.data_ptr(), torch.cuda.current_stream().cuda_stream))
        return verts.cpu().numpy(), keys.cpu().numpy(), tris.cpu().numpy(), tuple(int(c) for c in counts.cpu().numpy())

    verts, keys, tris, c = run(nv - 10, nt)                 # vertex overflow: true counts, no triangle at all
    assert c == (nv, nt) and np.all(verts[nv - 10:] == -7) and np.all(keys[nv - 10:] == -7) and np.all(keys[: nv - 10] >= 0)
    assert np.all(tris == -7)
    verts, keys, tris, c = run(nv, 100)                     # triangle overflow: the first 100, nothing past them
    assert c == (nv, nt) and np.array_equal(tris[:100], tris_all[:100]) and np.all(tris[100:] == -7) and np.all(verts[nv:] == -7)
    v.clear()
    assert run(16, 16)[3] == (0, 0)


def _kinfu_params(dim=128, flags=0):
    p = kf.KinFuParams.default_params_dynamicfusion()
    kf.KinFuParams.set_volume(p, dim, 1.0)
    p.max_nodes = 512
    p.cloud_capacity = 400000
    p.flags = flags
    return p


def test_kinfu_mesh_canonical_and_live():
    p = _kinfu_params()
    k = kf.KinFu(p)
    for t in range(5):
        k(synth.umbrella_depth(t))
    verts, nrm, tris, keys = k.mesh()
    assert len(tris) > 5000
    # the same volume extracted through TsdfVolume (full scan, no activity map)
    v = host.TsdfVolume((128, 128, 128))
    v.data_.copy_(torch.from_numpy(k.buffer("volume").view(np.int32)).cuda())
    v.setSize((1.0, 1.0, 1.0)); v.setTruncDist(p.tsdf_trunc_dist); v.setGradientDeltaFactor(p.gradient_delta_factor)
    v.setPose((np.array(p.volume_pose.R, np.float32).reshape(3, 3), np.array(p.volume_pose.t, np.float32)))
    gv, gk, gt, _, gn = _gpu_mesh(v, normals=True)
    assert np.array_equal(verts.view(np.uint32), gv[:, :3].view(np.uint32)) and np.array_equal(keys, gk) and np.array_equal(tris, gt)
    assert np.array_equal(nrm.view(np.uint32), gn[:, :3].view(np.uint32))
    # live: WarpField.warp of the canonical vertices and normals (rotation only), same topology
    lv, ln, lt, lk = k.mesh(live=True)
    assert np.array_equal(lt, tris) and np.array_equal(lk, keys)
    nodes = k.buffer("nodes")[: k.info()["nodes"]].copy()
    wf = host.WarpField()
    wf.setNodes(torch.from_numpy(nodes).cuda())
    pts = torch.from_numpy(np.concatenate([verts, np.zeros((len(verts), 1), np.float32)], 1)).cuda()
    nn = torch.from_numpy(np.concatenate([nrm, np.zeros((len(nrm), 1), np.float32)], 1)).cuda()
    wf.warp(pts, nn, flags=2)                                # DF_WARP_NORMAL_ROTATE_ONLY
    assert np.array_equal(lv.view(np.uint32), pts[:, :3].cpu().numpy().view(np.uint32))
    assert np.array_equal(ln.view(np.uint32), nn[:, :3].cpu().numpy().view(np.uint32))
    assert np.mean(np.any(lv != verts, 1)) > 0.5             # the field moved the surface
    k.close()


def test_kinfu_rigid_only_rejects_live_mesh():
    k = kf.KinFu(_kinfu_params(flags=kf.RIGID_ONLY))
    for t in range(2):
        k(synth.umbrella_depth(t))
    assert len(k.mesh()[2]) > 1000
    with pytest.raises(RuntimeError):
        k.mesh(live=True)
    k.close()


def test_kinfu_mesh_between_frames_leaves_the_loop_unchanged():
    runs = []
    for call_mesh in (False, True):
        k = kf.KinFu(_kinfu_params())
        digests = []
        for t in range(7):
            k(synth.umbrella_depth(t))
            if call_mesh and t >= 1:
                k.mesh()
                if k.info()["nodes"] >= 8:
                    k.mesh(live=True)
            digests.append(k.state_digest())
        pose = k.getCameraPose()
        runs.append((digests, k.buffer("volume").copy(), k.buffer("cloud").copy(), pose[0].copy(), pose[1].copy()))
        k.close()
    a, b = runs
    assert a[0] == b[0]
    assert np.array_equal(a[1], b[1]) and np.array_equal(a[2].view(np.uint32), b[2].view(np.uint32))
    assert np.array_equal(a[3], b[3]) and np.array_equal(a[4], b[4])
