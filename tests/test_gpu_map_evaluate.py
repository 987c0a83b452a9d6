"""svnicp_map_evaluate (VoxelHashMap.Evaluate): a scan scored and linearised at caller-given poses against the device local map.

Checked against the brute-force oracle (tests/map_nn_oracle.c: exact nearest map point, same fp64 arithmetic and tie rule), scipy's
k-d tree at full size, oracle.gn_given_corr for H and b, svnicp_evaluate at the initial guess, and for the absence of side
effects on the map."""
import ctypes as C

import numpy as np
import pytest
from scipy.spatial import cKDTree

import svn_icp_b200 as sv
from svn_icp_b200 import synth
from test_map_evaluate_cpu import BOUNDARY_CASES, case_arrays, map_nn

pytestmark = pytest.mark.gpu

SEED = 0xC0FFEE
MAX_DIST = 3.0
ERR_INVALID = -1  # SVNICP_ERR_INVALID


def exp_so3(w):
    th = np.linalg.norm(w)
    K = np.array([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]])
    if th < 1e-12:
        return np.eye(3) + K
    return np.eye(3) + np.sin(th) / th * K + (1 - np.cos(th)) / th ** 2 * (K @ K)


def drive_map(sensor="32", scans=range(6), voxel=1.0, cap=20):
    world = synth.make_world(SEED)
    m = sv.VoxelHashMap(voxel, 100.0, cap)
    for k in scans:
        pts, (R, t) = synth.make_scan(world, k, sensor, SEED)
        m.AddPointCloud(pts.astype(np.float32), R, t)
    return world, m


@pytest.fixture(scope="module")
def drive():
    """map of 6 scans of the 32-beam sensor; 4000 points of scan 8 and its ground-truth pose"""
    world, m = drive_map()
    pts, (R, t) = synth.make_scan(world, 8, "32", SEED)
    sel = np.sort(np.random.default_rng(1).choice(len(pts), 4000, replace=False))
    return m, pts[sel].astype(np.float32), R, t, m.GetMap()


def world_poses(oracle, R0, t0, poses):
    """[6, M] relative poses -> R~ [M,3,3], t~ [M,3] in fp64 (oracle.so3_exp), and R_p [M,3,3]"""
    Rp = np.stack([oracle.so3_exp(poses[3:, j])[0] for j in range(poses.shape[1])])
    return np.einsum("ij,mjk->mik", R0, Rp), t0 + poses[:3].T @ R0.T, Rp


def map_index(mp, near, mask):
    """rows of GetMap() holding the returned coordinates (any duplicate holds the same point)"""
    lut = {tuple(p): i for i, p in reversed(list(enumerate(mp.astype(np.float32).tolist())))}
    idx = np.zeros(mask.shape, dtype=np.int32)
    for j in range(mask.shape[0]):
        for i in np.nonzero(mask[j])[0]:
            idx[j, i] = lut[tuple(near[j, i].tolist())]
    return idx


def sort_rows(a):
    return a[np.lexsort((a[:, 2], a[:, 1], a[:, 0]))] if len(a) else a


def check_system(H, b, cH, cb, src):
    """the bars of check_system in test_gpu_evaluate.py"""
    for blk in (slice(0, 3), slice(3, 6)):
        for blk2 in (slice(0, 3), slice(3, 6)):
            scale = np.abs(cH[:, blk, blk2]).max()
            np.testing.assert_allclose(H[:, blk, blk2], cH[:, blk, blk2], rtol=0, atol=1e-6 * scale)
    n_s = len(src)
    rng_s = np.linalg.norm(src, axis=1).mean()
    np.testing.assert_allclose(b[:, :3], cb[:, :3], rtol=0, atol=1e-6 * n_s * 0.3)
    np.testing.assert_allclose(b[:, 3:], cb[:, 3:], rtol=0, atol=1e-6 * n_s * 0.3 * rng_s)


def test_world_poses_bit_exact(oracle, drive):
    m, src, Rg, tg, mp = drive
    rng = np.random.default_rng(2)
    for k in range(4):
        R0, t0 = (Rg, tg) if k == 0 else (Rg @ exp_so3(rng.normal(0, 0.02, 3)), tg + rng.normal(0, 0.3, 3))
        ev = m.Evaluate(src, R0, t0, np.zeros(6), MAX_DIST, want_mask=True, want_nearest=True)
        q = oracle.transform_q0(src, R0, t0)
        near, d2, mask, _ = map_nn(q, mp, MAX_DIST)
        np.testing.assert_array_equal(ev["mask"], mask)
        np.testing.assert_array_equal(ev["nearest"], near)
        assert ev["inliers"] == mask.sum() > 1000
        assert ev["fitness"] == mask.sum() / len(src)
        np.testing.assert_allclose(ev["rmse"], np.sqrt(d2[mask == 1].mean()), rtol=1e-12, atol=0)


@pytest.mark.parametrize("case", BOUNDARY_CASES, ids=[c[0] for c in BOUNDARY_CASES])
def test_boundary_cases(oracle, case):
    _, v, md, pts, qs, want = case_arrays(case)
    m = sv.VoxelHashMap(v, 1000.0, 20, capacity_voxels=1 << 10)
    m.AddPointCloud(pts, np.eye(3), np.zeros(3))
    ev = m.Evaluate(qs, np.eye(3), np.zeros(3), np.zeros(6), md, want_mask=True, want_nearest=True)
    near, _, mask, _ = map_nn(qs, pts, md)
    np.testing.assert_array_equal(ev["nearest"], near)
    np.testing.assert_array_equal(ev["mask"], mask)
    np.testing.assert_array_equal(ev["mask"], want >= 0)


def relative_poses(M, seed):
    rng = np.random.default_rng(seed)
    return np.concatenate([rng.uniform(-0.5, 0.5, (3, M)), rng.uniform(-0.05, 0.05, (3, M))])


@pytest.mark.parametrize("M", [1, 31, 32, 33, 100])
def test_relative_poses(oracle, drive, M):
    m, src, Rg, tg, mp = drive
    poses = relative_poses(M, M)
    ev = m.Evaluate(src, Rg, tg, poses, MAX_DIST, want_mask=True, want_nearest=True)
    Rt, tt, _ = world_poses(oracle, Rg, tg, poses)
    for j in sorted({0, M // 2, M - 1} | ({31, 32} & set(range(M)))):  # both sides of the 32-pose blocks
        q = oracle.transform_q0(src, Rt[j], tt[j])
        near, d2, mask, _ = map_nn(q, mp, MAX_DIST)
        clear = np.abs(d2 - MAX_DIST) >= 1e-9
        np.testing.assert_array_equal(ev["mask"][j][clear], mask[clear])
        both = (ev["mask"][j] == 1) & (mask == 1)
        d2g = ((q - ev["nearest"][j].astype(np.float64)) ** 2).sum(axis=1)
        np.testing.assert_allclose(d2g[both], d2[both], rtol=1e-12, atol=0)
        diff = both & (ev["nearest"][j] != near).any(axis=1)
        d2o = ((q - near.astype(np.float64)) ** 2).sum(axis=1)
        assert (np.abs(d2g - d2o)[diff] <= 1e-9).all()
        assert ev["inliers"][j] == ev["mask"][j].sum()


def test_gauss_newton_system(oracle, drive):
    m, src, Rg, tg, mp = drive
    poses = np.concatenate([np.zeros((6, 1)), relative_poses(32, 7)], axis=1)
    ev = m.Evaluate(src, Rg, tg, poses, MAX_DIST, want_mask=True, want_nearest=True)
    _, _, Rp = world_poses(oracle, Rg, tg, poses)
    idx = map_index(mp, ev["nearest"], ev["mask"])
    cH, cb = oracle.gn_given_corr(Rp, poses[:3].T, Rg, tg, src, mp, idx, ev["mask"], MAX_DIST)
    check_system(ev["H"], ev["b"], cH, cb, src)
    no_sys = m.Evaluate(src, Rg, tg, poses, MAX_DIST, want_system=False)
    for k in ("inliers", "fitness", "rmse"):
        np.testing.assert_array_equal(no_sys[k], ev[k])


def test_agrees_with_svnicp_evaluate(oracle, drive):
    """At the initial guess the map evaluation and svnicp_evaluate (candidate table of GetMap()) pick the same map point
    wherever the nearest is unique."""
    m, src, Rg, tg, mp = drive
    R0, t0 = Rg @ exp_so3(np.array([0.002, -0.001, 0.003])), tg + np.array([0.05, -0.04, 0.02])
    icp = sv.SVNICP(sv.SteinICPParam(iterations=1, KNN_count=32, max_dist=MAX_DIST, lr=1.0, debug_corr=True), np.zeros((6, 4)))
    icp.add_cloud(src.astype(np.float64), mp, np.zeros((6, 4)))
    icp.set_initial_mean(R0, t0)
    assert icp.stein_align() == sv.ALIGN_SUCCESS
    e_tab = icp.evaluate(np.zeros(6), want_mask=True, want_idx=True)
    e_map = m.Evaluate(src, R0, t0, np.zeros(6), MAX_DIST, want_mask=True, want_nearest=True)
    q0 = oracle.transform_q0(src, R0, t0)
    cand = icp.get_candidates()
    d0 = ((q0 - mp[cand[:, 0]]) ** 2).sum(axis=1)
    d1 = ((q0 - mp[cand[:, 1]]) ** 2).sum(axis=1)
    unique = (np.abs(d0 - d1) > 1e-12 * d0) & (e_map["mask"] == 1)
    np.testing.assert_array_equal(e_map["nearest"][unique], mp[cand[unique, 0]].astype(np.float32))
    clear = np.abs(d0 - MAX_DIST) >= 1e-5
    np.testing.assert_array_equal(e_map["mask"][clear], e_tab["mask"][clear])
    check_system(e_map["H"][None], e_map["b"][None], e_tab["H"][None], e_tab["b"][None], src)


def test_full_size_scan():
    """64-beam scan (~143 k points) against a saturated 1 m / 20-point map of a drive, M = 4"""
    world, m = drive_map("64", range(0, 12, 2))
    src, (Rg, tg) = synth.make_scan(world, 12, "64", SEED)
    src = src.astype(np.float32)
    mp = m.GetMap()
    assert len(src) > 100_000
    poses = np.concatenate([np.zeros((6, 1)), relative_poses(3, 11) * 0.2], axis=1)
    ev = m.Evaluate(src, Rg, tg, poses, MAX_DIST, want_mask=True, want_nearest=True)
    tree = cKDTree(mp)
    for j in range(4):
        R, t = Rg @ exp_so3(poses[3:, j]), tg + Rg @ poses[:3, j]
        q = src.astype(np.float64) @ R.T + t
        dist, _ = tree.query(q)
        kd2 = dist ** 2
        sel = ev["mask"][j] == 1
        d2g = ((q - ev["nearest"][j].astype(np.float64)) ** 2).sum(axis=1)
        np.testing.assert_allclose(d2g[sel], kd2[sel], rtol=1e-9, atol=1e-12)
        clear = np.abs(kd2 - MAX_DIST) >= 1e-5
        np.testing.assert_array_equal(sel[clear], (kd2 < MAX_DIST)[clear])
    assert ev["fitness"][0] > 0.5


def test_independent_of_batch_and_repeatable(drive):
    m, src, Rg, tg, _ = drive
    poses = relative_poses(100, 5)
    kw = dict(want_mask=True, want_nearest=True)
    full = m.Evaluate(src, Rg, tg, poses, MAX_DIST, **kw)
    again = m.Evaluate(src, Rg, tg, poses, MAX_DIST, **kw)
    rev = m.Evaluate(src, Rg, tg, poses[:, ::-1], MAX_DIST, **kw)
    for k in full:
        np.testing.assert_array_equal(full[k], again[k])
        np.testing.assert_array_equal(full[k], rev[k][::-1])
    for j in (0, 31, 32, 57, 99):
        one = m.Evaluate(src, Rg, tg, poses[:, j], MAX_DIST, **kw)
        for k in full:
            np.testing.assert_array_equal(one[k], full[k][j])


def test_no_side_effects():
    world, m = drive_map(scans=range(4))
    _, twin = drive_map(scans=range(4))
    src, (Rg, tg) = synth.make_scan(world, 5, "32", SEED)
    before = m.GetMap()
    ptr, n = m.GetMapDevice()
    size, pts = m.Size(), m.PointCount()
    for f32 in (True, False):
        m.Evaluate(src.astype(np.float32 if f32 else np.float64), Rg, tg, relative_poses(40, 3), MAX_DIST, want_mask=True,
                   want_nearest=True)
    assert (m.Size(), m.PointCount()) == (size, pts)
    after = np.zeros((n, 3))
    assert m._lib.svnicp_map_download(m._m, after.ctypes.data_as(C.c_void_p), C.c_int64(n)) == 0
    np.testing.assert_array_equal(after, before)
    # the device pointer of the earlier GetMap still feeds the registration
    import torch
    prm = sv.SteinICPParam(iterations=4, KNN_count=32, max_dist=MAX_DIST, lr=1.0)
    init = synth.init_particles(16, np.random.default_rng(4))
    src64 = torch.from_numpy(np.ascontiguousarray(src, dtype=np.float64)).cuda()
    a = sv.SVNICP(prm, init)
    a.add_cloud_device(src64.data_ptr(), len(src), ptr, n, init)
    a.set_initial_mean(Rg, tg)
    assert a.stein_align() == sv.ALIGN_SUCCESS
    b = sv.SVNICP(prm, init)
    b.add_cloud(src, before, init)
    b.set_initial_mean(Rg, tg)
    assert b.stein_align() == sv.ALIGN_SUCCESS
    np.testing.assert_array_equal(a.get_particles(), b.get_particles())
    # the next AddPointCloud behaves as on a map that never evaluated
    m.AddPointCloud(src.astype(np.float32), Rg, tg)
    twin.AddPointCloud(src.astype(np.float32), Rg, tg)
    assert (m.Size(), m.PointCount()) == (twin.Size(), twin.PointCount())
    np.testing.assert_array_equal(sort_rows(m.GetMap()), sort_rows(twin.GetMap()))


def test_edge_cases(drive):
    m, src, Rg, tg, _ = drive
    n = len(src)
    # empty map: no inliers, H = the Q2 / Q3 diagonal
    e = sv.VoxelHashMap(1.0, 100.0, 20).Evaluate(src, Rg, tg, np.zeros(6), MAX_DIST, want_mask=True)
    assert e["inliers"] == 0 and e["fitness"] == 0 and e["rmse"] == 0 and e["mask"].sum() == 0
    np.testing.assert_array_equal(e["H"], np.diag([n + 1e-6] * 3 + [1e-6] * 3))
    np.testing.assert_array_equal(e["b"], np.zeros(6))
    # NaN poses: no correspondence, finite system; NaN source points: masked, the rest unaffected
    poses = np.concatenate([np.zeros((6, 1)), np.full((6, 1), np.nan), np.array([[0, 0, 0, np.nan, 0, 0]]).T], axis=1)
    e = m.Evaluate(src, Rg, tg, poses, MAX_DIST, want_mask=True)
    assert e["inliers"][0] > 0 and (e["inliers"][1:] == 0).all() and (e["rmse"][1:] == 0).all() and np.isfinite(e["H"]).all()
    bad = src.copy()
    bad[::7, 1] = np.nan
    e2 = m.Evaluate(bad, Rg, tg, np.zeros(6), MAX_DIST, want_mask=True)
    assert e2["mask"][::7].sum() == 0 and np.isfinite(e2["H"]).all() and np.isfinite(e2["b"]).all()
    keep = np.ones(n, bool)
    keep[::7] = False
    np.testing.assert_array_equal(e2["mask"][keep], e["mask"][0][keep])
    # far off the map
    far = m.Evaluate(src, Rg, tg + np.array([5e4, -3e4, 100.0]), np.zeros(6), MAX_DIST)
    assert far["inliers"] == 0 and far["rmse"] == 0
    # host / device, float / double: the same bits
    import torch
    ref = m.Evaluate(src, Rg, tg, relative_poses(5, 9), MAX_DIST, want_mask=True, want_nearest=True)
    for dt, f64 in ((np.float32, False), (np.float64, True)):
        host = m.Evaluate(src.astype(dt), Rg, tg, relative_poses(5, 9), MAX_DIST, want_mask=True, want_nearest=True)
        d = torch.from_numpy(np.ascontiguousarray(src, dtype=dt)).cuda()
        dev = m.EvaluateDevice(d.data_ptr(), n, f64, Rg, tg, relative_poses(5, 9), MAX_DIST, want_mask=True, want_nearest=True)
        for k in ref:
            np.testing.assert_array_equal(host[k], ref[k])
            np.testing.assert_array_equal(dev[k], ref[k])


def test_errors(drive):
    m, src, Rg, tg, _ = drive
    ok = dict(R0=Rg, t0=tg, poses=np.zeros(6))
    for md in (np.nan, np.inf, 0.0, -1.0):
        with pytest.raises(sv.SvnIcpError, match="max_dist"):
            m.Evaluate(src, max_dist=md, **ok)
    with pytest.raises(sv.SvnIcpError, match="at most 4"):
        m.Evaluate(src, max_dist=4.01 ** 2, **ok)  # v = 1 m: 5 voxels on each side
    m.Evaluate(src, max_dist=16.0, **ok)  # exactly 4 voxels
    with pytest.raises(sv.SvnIcpError, match="n_poses"):
        m.Evaluate(src, Rg, tg, np.zeros((6, 0)), MAX_DIST)
    with pytest.raises(sv.SvnIcpError, match="source points"):
        m.Evaluate(np.zeros((0, 3), np.float32), Rg, tg, np.zeros(6), MAX_DIST)
    lib, R, t, x, stats = m._lib, Rg.ravel().copy(), tg.copy(), np.zeros(6), np.zeros(3)
    p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    args = [m._m, p(src), C.c_int64(len(src)), 0, 0, p(R), p(t), 1, p(x), C.c_double(MAX_DIST), p(stats), None, None, None, None]
    assert lib.svnicp_map_evaluate(*args) == 0
    for i, bad in ((2, C.c_int64((1 << 30) + 1)), (1, None), (5, None), (6, None), (8, None), (10, None)):
        a = list(args)
        a[i] = bad
        assert lib.svnicp_map_evaluate(*a) == ERR_INVALID
    a = list(args)
    a[0] = None
    assert lib.svnicp_map_evaluate(*a) == ERR_INVALID
