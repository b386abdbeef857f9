"""Pin the CPU oracle against every golden vector the reference's own tests hold for this path
(SURVEY.md section 8c): tests/utils/test_quaternion.cc, tests/utils/test_dual_quaternion.cc,
tests/nanoflann_test.cpp (orders regenerated from the vendored nanoflann header) and the warp-solve scenarios of
tests/warp_test.cpp / tests/ceres_warp_test.cpp."""
import ctypes as C
import math

import numpy as np
import pytest


def _q(*v):
    return np.array(v, np.float32)


def test_half_roundtrip_matches_numpy(orc):
    lib = orc.load()
    rng = np.random.default_rng(0)
    vals = np.concatenate([rng.uniform(-2, 2, 20000), rng.uniform(-7e4, 7e4, 2000), rng.normal(0, 1e-5, 2000),
                           [0.0, -0.0, 1.0, -1.0, 65504.0, 65519.9, 65520.0, 1e-8, 5.96e-8, 2.98e-8, 2.9802322e-8, 6.1e-5]]).astype(np.float32)
    ref = vals.astype(np.float16)
    for v, r in zip(vals, ref):
        h = lib.orc_float2half_rn(float(v))
        assert h == int(r.view(np.uint16)), (v, h, r.view(np.uint16))
    for h in list(range(0, 0x7c00, 7)) + list(range(0x8000, 0xfc00, 13)) + [0x7c00, 0xfc00]:
        assert lib.orc_half2float(h) == float(np.uint16(h).view(np.float16))


# ---- tests/utils/test_quaternion.cc -------------------------------------------------------------------------------------------
def test_quaternion_encode_rotation(orc):          # :6-15
    q = np.zeros(4, np.float32)
    orc.load().orc_quat_encode_rotation(C.c_float(math.pi / 4), C.c_float(0), C.c_float(0), C.c_float(1), C.c_void_p(q.ctypes.data))
    np.testing.assert_allclose(q, [0.9238795, 0, 0, 0.38268346], rtol=4e-7, atol=0)


def test_quaternion_rotate_sandwich(orc):          # :17-25  (0,0,1,1) rotates (0,0,1) -> (0,2,0)
    q = _q(0, 0, 1, 1)
    v = _q(0, 0, 1)
    orc.load().orc_quat_rotate_sandwich(C.c_void_p(q.ctypes.data), C.c_void_p(v.ctypes.data))
    assert list(v) == [0, 2, 0]


def test_quaternion_product(orc):                  # :27-36
    a, b, out = _q(1, 1, 2, 2), _q(0, 0, 1, 1), np.zeros(4, np.float32)
    orc.load().orc_quat_mul(C.c_void_p(a.ctypes.data), C.c_void_p(b.ctypes.data), C.c_void_p(out.ctypes.data))
    assert list(out) == [-4, 0, 0, 2]


def test_quaternion_dot_product(orc):              # :38-43  0.5*((conj(q)*o) + q*conj(o)).w == 4
    a, b = _q(1, 1, 2, 2), _q(0, 0, 1, 1)
    ca, cb = a * _q(1, -1, -1, -1), b * _q(1, -1, -1, -1)
    o1, o2 = np.zeros(4, np.float32), np.zeros(4, np.float32)
    lib = orc.load()
    lib.orc_quat_mul(C.c_void_p(ca.ctypes.data), C.c_void_p(b.ctypes.data), C.c_void_p(o1.ctypes.data))
    lib.orc_quat_mul(C.c_void_p(a.ctypes.data), C.c_void_p(cb.ctypes.data), C.c_void_p(o2.ctypes.data))
    assert 0.5 * (o1[0] + o2[0]) == 4


def test_quaternion_normalize(orc):                # :45-50 (10,10,10,10) -> 0.5 via the rotate path's normalise
    # orc_node_translation normalises the node rotation: dual (0.5*(0,1,0,0)*r) with r = (10,10,10,10) must give t = (1,0,0)
    node = np.zeros(12, np.float32)
    node[3:7] = 10
    orc.load().orc_node_encode_translation(C.c_void_p(node.ctypes.data), C.c_float(1), C.c_float(0), C.c_float(0))
    t = np.zeros(4, np.float32)
    orc.load().orc_node_translation(C.c_void_p(node.ctypes.data), C.c_void_p(t.ctypes.data))
    # 2 * (0.5*(0,1,0,0)*r) * conj(r/|r|) = (0,1,0,0) * |r| = 20 * x
    np.testing.assert_allclose(t, [0, 20, 0, 0], atol=1e-5)


# ---- tests/utils/test_dual_quaternion.cc ----------------------------------------------------------------------------------------
def test_dual_quaternion_constructor(orc):         # :6-21
    rot, dual = np.zeros(4, np.float32), np.zeros(4, np.float32)
    orc.load().orc_dq_from_euler(C.c_float(1), C.c_float(2), C.c_float(3), C.c_float(1), C.c_float(2), C.c_float(3),
                                 C.c_void_p(rot.ctypes.data), C.c_void_p(dual.ctypes.data))
    node = np.zeros(12, np.float32)
    node[3:7], node[7:11] = rot, dual
    t = np.zeros(4, np.float32)
    orc.load().orc_node_translation(C.c_void_p(node.ctypes.data), C.c_void_p(t.ctypes.data))
    assert abs(t[0]) < 0.001 and abs(t[1] - 1) < 0.1 and abs(t[2] - 2) < 0.1 and abs(t[3] - 3) < 0.1
    np.testing.assert_allclose(rot[:3], [0.435953, -0.718287, 0.310622], atol=0.01)
    # the reference's expected z (0.454649 +- 0.01) is self-inconsistent with its own Euler formula
    # (dual_quaternion.hpp:47-48 gives 0.444435 for roll=1, pitch=2, yaw=3: off by 0.0102); pin the formula's value
    assert abs(rot[3] - 0.454649) < 0.0103 and abs(rot[3] - 0.4444351) < 1e-6


# ---- tests/nanoflann_test.cpp (orders generated from the vendored header, SURVEY 8c) ----------------------------------------------
CUBE = [(1, 1, 1), (1, 1, -1), (1, -1, 1), (1, -1, -1), (-1, 1, 1), (-1, 1, -1), (-1, -1, 1), (-1, -1, -1)]


def test_knn_orders_match_nanoflann(orc):
    nodes = orc.make_nodes(CUBE)
    q = np.array([(-1, -1, -1), (0, 0, 0), (1, 1, 1), (2, 2, 2), (3, 3, 3)], np.float32)
    idx, d2 = orc.knn8(nodes, q)
    assert idx[0].tolist() == [7, 3, 5, 6, 1, 2, 4, 0]
    assert idx[1].tolist() == [0, 1, 2, 3, 4, 5, 6, 7]
    for r in (2, 3, 4):
        assert idx[r].tolist() == [0, 1, 2, 4, 3, 5, 6, 7]
    assert d2[1].tolist() == [3.0] * 8


def test_knn_matches_reference_nanoflann_binary(orc):
    """against what oracle/_ref/knn_ref (the reference's vendored nanoflann + knn_point_cloud.hpp compiled as they lie) returned
    for these random clouds (tests/golden/knn_ref_random.npz, written by tests/golden/make_golden.py): squared distances
    bit-exact, index lists equal wherever distances are distinct"""
    from pathlib import Path
    rng = np.random.default_rng(5)
    pts = rng.uniform(-1, 1, (300, 3)).astype(np.float32)
    qs = rng.uniform(-1.2, 1.2, (200, 3)).astype(np.float32)
    golden = np.load(Path(__file__).parent / "golden" / "knn_ref_random.npz")
    ref_idx, ref_d2 = golden["idx"].astype(np.int64), golden["d2"]
    idx, d2 = orc.knn8(orc.make_nodes(pts), qs)
    assert np.array_equal(d2.view(np.uint32), ref_d2.view(np.uint32))
    distinct = np.ones(len(qs), bool)
    distinct &= (np.diff(ref_d2, axis=1) > 0).all(axis=1)
    assert np.array_equal(idx[distinct], ref_idx[distinct])


# ---- tests/warp_test.cpp / ceres_warp_test.cpp scenarios ----------------------------------------------------------------------------
# The reference asserts |warp(source) - target| < 1e-3 after the solve.  For its rigid / multi-node / non-rigid scenarios that
# bound is NOT attainable by any minimiser of its own energy: the 8-NN Gaussian weight matrix W is rank deficient there (e.g.
# rigid: 5 collinear vertices see only 4 symmetry classes of cube-corner nodes, exact least-squares residual 6.3e-3), so those
# reference tests cannot pass as written (like its `rodrigues` quaternion test).  The oracle is therefore pinned against the
# exact dense least-squares optimum of the reference's energy (numpy lstsq, float64), plus the reference's own tolerance
# wherever the optimum satisfies it (single vertex).
def _lsq_reference(node_pts, src, dst):
    P = np.array(node_pts, np.float64)
    S = np.array(src, np.float64)
    D = np.array(dst, np.float64)
    d2 = ((S[:, None, :].astype(np.float32) - P[None].astype(np.float32)) ** 2).sum(-1).astype(np.float64)
    order = np.argsort(d2, axis=1, kind="stable")[:, :8]
    W = np.zeros((len(S), len(P)))
    for v in range(len(S)):
        for k in order[v]:
            W[v, k] = math.exp(-d2[v, k] / 18.0)          # node weight 3 -> 2*w*w = 18
    T, *_ = np.linalg.lstsq(W, D - S, rcond=None)
    return S + W @ T, W, T


def _solve_and_warp(orc, node_pts, src, dst, lm_iters=300):
    nodes = orc.make_nodes(node_pts)
    src = np.array(src, np.float32)
    dst = np.array(dst, np.float32)
    nrm = np.tile(np.array([0, 0, 1], np.float32), (len(src), 1))
    stats = orc.solve_data_term(nodes, src, dst, lm_iters=lm_iters)
    warped = src.copy()
    orc.warp(nodes, warped, nrm)
    return nodes, warped, stats


def test_warp_single_vertex_closed_form(orc):      # warp_test.cpp:15-69, tol 1e-5; closed form SURVEY 8c
    nodes, warped, stats = _solve_and_warp(orc, CUBE, [(0, 0, 0)], [(0.05, 0.05, 0.05)])
    np.testing.assert_allclose(warped, [[0.05, 0.05, 0.05]], atol=1e-5)
    w = math.exp(-3.0 / 18.0)
    t = orc.node_translations(nodes)[:, 1:]
    np.testing.assert_allclose(t, np.full((8, 3), 0.05 / (8 * w)), rtol=1e-4)       # minimum-norm solution
    assert stats[1] < 1e-12


RIGID_SRC = [(-3, -3, -3), (-2, -2, -2), (0, 0, 0), (2, 2, 2), (3, 3, 3)]
RIGID_DST = [(-2.95, -2.95, -2.95), (-1.95, -1.95, -1.95), (0.05, 0.05, 0.05), (2.05, 2.05, 2.05), (3.05, 3.05, 3.05)]
NODES12 = [(1, 1, 1), (1, 2, -1), (1, -2, 1), (1, -1, -1), (-1, 1, 5), (-1, 1, -1), (-1, -1, 1), (-1, -1, -1), (2, -3, -1), (-3, -3, -2),
           (2, -3, 3), (2, 2, 4)]
MULTI_SRC = RIGID_SRC + [(3, 3, 3)]
MULTI_DST = [(-2.95, -2.95, -2.95), (-1.95, -1.95, -1.95), (0.1, 0.1, 0.1), (2, 2, 2), (3.05, 3.05, 3.05), (3.05, 3.05, 3.05)]
NONRIGID_DST = [(-2.95, -3.0, -2.95), (-1.95, -1.95, -2.0), (0.1, 0.1, 0.1), (2, 2.5, 2), (3.05, 3.05, 3.05), (3.05, 3.05, 3.05)]

SCENARIOS = {
    "rigid": (CUBE, RIGID_SRC, RIGID_DST),                 # warp_test.cpp:73-144
    "multiple_nodes": (NODES12, MULTI_SRC, MULTI_DST),     # warp_test.cpp:243-316
    "non_rigid": (NODES12[:9], MULTI_SRC, NONRIGID_DST),   # warp_test.cpp:320-390
}


@pytest.mark.parametrize("name", list(SCENARIOS))
def test_warp_scenarios_reach_exact_least_squares(orc, name):
    node_pts, src, dst = SCENARIOS[name]
    _, warped, stats = _solve_and_warp(orc, node_pts, src, dst)
    best, W, T = _lsq_reference(node_pts, src, dst)
    np.testing.assert_allclose(warped, best, atol=2e-4)
    resid = np.abs(best - np.array(dst)).max()
    if resid < 5e-4:                                       # the reference's own tolerance where it is attainable
        np.testing.assert_allclose(warped, np.array(dst, np.float32), atol=1e-3)
    cost_opt = 0.5 * ((best - np.array(dst, np.float64)) ** 2).sum()
    assert abs(stats[1] - cost_opt) <= 1e-4 * max(cost_opt, 1e-12) + 1e-10


def test_warp_and_reverse(orc):                    # warp_test.cpp:147-241: second solve returns to the start
    nodes = orc.make_nodes(CUBE)
    src, dst = np.array(RIGID_SRC, np.float32), np.array(RIGID_DST, np.float32)
    nrm = np.tile(np.array([0, 0, 1], np.float32), (len(src), 1))
    orc.solve_data_term(nodes, src, dst, lm_iters=300)
    s1 = orc.node_translations(nodes).sum(0)
    orc.solve_data_term(nodes, dst, src, lm_iters=300)
    back = dst.copy()
    orc.warp(nodes, back, nrm.copy())
    best, _, _ = _lsq_reference(CUBE, RIGID_DST, RIGID_SRC)
    np.testing.assert_allclose(back, src, atol=7e-3)        # exact least-squares residual of this scenario is 6.3e-3
    s2 = orc.node_translations(nodes).sum(0)
    # the reference accumulates the node translations printed after BOTH solves and asserts the total ~ 0 (1e-3), :236-238
    np.testing.assert_allclose((s1 + s2)[1:], 0, atol=1e-3)
