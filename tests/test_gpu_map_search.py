"""svnicp_map_search (VoxelHashMap.Search): the exact top k of a grid of poses against the device local map.

Checked against svnicp_map_evaluate on every grid pose (counts bit for bit), the brute-force oracle (tests/map_nn_oracle.c), a
np.lexsort of (-count, g) for the ranking, svnicp_map_evaluate again for the winners' statistics, and for determinism, the
absence of side effects, argument errors and an end-to-end relocalisation."""
import ctypes as C

import numpy as np
import pytest

import svn_icp_b200 as sv
from svn_icp_b200 import synth
from test_gpu_map_evaluate import MAX_DIST, SEED, drive_map, exp_so3, world_poses
from test_map_evaluate_cpu import map_nn
from test_map_search_cpu import topk_lexsort

pytestmark = pytest.mark.gpu

ERR_INVALID = -1  # SVNICP_ERR_INVALID
STEPS = np.array([0.3, 0.25, 0.15, 0.02, 0.03, 0.05])
GRID_ODD = (3, 3, 1, 3, 1, 5)     # holds x = 0
GRID_MIXED = (4, 3, 2, 2, 1, 3)   # even counts: no x = 0; negative values on every axis with a count > 1


@pytest.fixture(scope="module")
def drive():
    """map of 6 scans of the 32-beam sensor; 4000 points of scan 8 and its ground-truth pose"""
    world, m = drive_map()
    pts, (R, t) = synth.make_scan(world, 8, "32", SEED)
    sel = np.sort(np.random.default_rng(1).choice(len(pts), 4000, replace=False))
    return m, pts[sel].astype(np.float32), R, t


@pytest.fixture(scope="module")
def drive64():
    """the DESIGN 10b map: scans 0-11 of the 64-beam sensor at 1 m / 20 points, and the world"""
    return drive_map("64", range(12))


def search(m, src, R0, t0, counts, steps=STEPS, k=1, want_counts=True, md=MAX_DIST):
    return m.Search(src, R0, t0, counts, steps, md, top_k=k, want_counts=want_counts)


def all_poses(counts, steps=STEPS):
    return sv.search_grid_poses(counts, steps, np.arange(int(np.prod(counts))))


def assert_same(a, b):
    for k in a:
        if a[k] is None:
            assert b[k] is None
        else:
            np.testing.assert_array_equal(a[k], b[k])


@pytest.mark.parametrize("counts", [GRID_ODD, GRID_MIXED], ids=["odd", "mixed"])
def test_counts_equal_evaluate(drive, counts):
    import torch
    m, src, Rg, tg = drive
    x = all_poses(counts)
    if counts == GRID_ODD:
        assert ((x == 0).all(axis=0)).sum() == 1
    want = m.Evaluate(src, Rg, tg, x, MAX_DIST, want_system=False)["inliers"]
    assert want.max() > 1000 and want.min() < want.max()
    for dt, f64 in ((np.float32, False), (np.float64, True)):
        host = search(m, src.astype(dt), Rg, tg, counts)
        np.testing.assert_array_equal(host["counts"].reshape(-1), want)
        assert host["counts"].shape == tuple(reversed(counts))
        d = torch.from_numpy(np.ascontiguousarray(src, dtype=dt)).cuda()
        dev = m.SearchDevice(d.data_ptr(), len(src), f64, Rg, tg, counts, STEPS, MAX_DIST, top_k=1, want_counts=True)
        assert_same(host, dev)


def test_counts_equal_brute_force(oracle, drive):
    """a few hundred poses of 400 points against the brute-force sweep over GetMap() (boundary distances excepted)"""
    m, src, Rg, tg = drive
    src = src[::10]
    counts = (5, 5, 1, 1, 1, 8)
    x = all_poses(counts)
    got = search(m, src, Rg, tg, counts)["counts"].reshape(-1)
    mp = m.GetMap()
    Rt, tt, _ = world_poses(oracle, Rg, tg, x)
    assert got.max() > 100
    for j in range(x.shape[1]):
        q = oracle.transform_q0(src, Rt[j], tt[j])
        _, d2, _, _ = map_nn(q, mp, 1e300)  # the nearest map point whatever its distance
        near_edge = int((np.abs(d2 - MAX_DIST) < 1e-9).sum())
        assert abs(int(got[j]) - int((d2 < MAX_DIST).sum())) <= near_edge


@pytest.mark.parametrize("k", [1, 7, 1024])
def test_topk_is_lexsort(drive, k):
    m, src, Rg, tg = drive
    for counts in (GRID_ODD, (41, 41, 1, 1, 1, 10)):  # 16 810 poses: two chunks, the second (426 poses) smaller than k
        M = int(np.prod(counts))
        kk = min(k, M)
        r = search(m, src, Rg, tg, counts, k=kk)
        c = r["counts"].reshape(-1)
        np.testing.assert_array_equal(r["index"], topk_lexsort(c, kk))
        np.testing.assert_array_equal(r["count"], c[r["index"]])
        np.testing.assert_array_equal(r["poses"], sv.search_grid_poses(counts, STEPS, r["index"]))


def test_far_scan_all_zero(drive):
    m, src, Rg, tg = drive
    counts = (41, 41, 1, 1, 1, 10)
    for k in (1, 7, 1024):
        r = search(m, src, Rg, tg + np.array([5e4, -3e4, 100.0]), counts, k=k)
        assert (r["counts"] == 0).all()
        np.testing.assert_array_equal(r["index"], np.arange(k))
        assert (r["count"] == 0).all() and (r["rmse"] == 0).all()


def test_stats_equal_evaluate(drive):
    m, src, Rg, tg = drive
    counts = (9, 9, 1, 1, 1, 7)
    r = search(m, src, Rg, tg, counts, k=64)
    np.testing.assert_array_equal(r["poses"], sv.search_grid_poses(counts, STEPS, r["index"]))
    ev = m.Evaluate(src, Rg, tg, r["poses"], MAX_DIST, want_system=False)
    np.testing.assert_array_equal(r["count"], ev["inliers"])
    np.testing.assert_array_equal(r["fitness"], ev["fitness"])
    np.testing.assert_array_equal(r["rmse"], ev["rmse"])


def test_full_size_scan_two_chunks(drive64):
    """143 k points: 936 poses per chunk, so a 1 089-pose grid takes two chunks"""
    world, m = drive64
    src, (Rg, tg) = synth.make_scan(world, 12, "64", SEED)
    src = src.astype(np.float32)
    counts = (11, 11, 1, 1, 1, 9)
    x = all_poses(counts)
    r = search(m, src, Rg, tg, counts, k=20)
    want = m.Evaluate(src, Rg, tg, x, MAX_DIST, want_system=False)["inliers"]
    np.testing.assert_array_equal(r["counts"].reshape(-1), want)
    np.testing.assert_array_equal(r["index"], topk_lexsort(want, 20))


def test_deterministic_and_layout_free(drive):
    m, src, Rg, tg = drive
    counts = (41, 41, 1, 1, 1, 10)
    a = search(m, src, Rg, tg, counts, k=1024)
    b = search(m, src, Rg, tg, counts, k=1024)
    twin = sv.VoxelHashMap(m.voxel_size_, m.max_range_, m.max_pointscount_, capacity_voxels=1 << 17)  # another slot layout
    twin.Import(m.Export())
    c = search(twin, src, Rg, tg, counts, k=1024)
    assert_same(a, b)
    assert_same(a, c)


def test_no_side_effects_and_errors(drive):
    m, src, Rg, tg = drive
    before = m.GetMap()
    ptr, n = m.GetMapDevice()
    size, pts = m.Size(), m.PointCount()
    ref = search(m, src, Rg, tg, GRID_ODD, k=5)
    assert (m.Size(), m.PointCount()) == (size, pts)
    after = np.zeros((n, 3))
    assert m._lib.svnicp_map_download(m._m, after.ctypes.data_as(C.c_void_p), C.c_int64(n)) == 0
    np.testing.assert_array_equal(after, before)
    assert m.GetMapDevice() == (ptr, n)
    # argument errors through the raw ABI, each followed by a valid call
    lib, R, t = m._lib, Rg.ravel().copy(), tg.copy()
    cnt, stp = np.array(GRID_ODD, np.int32), STEPS.copy()
    idx, poses, stats, grid = np.zeros(5, np.int64), np.zeros((6, 5)), np.zeros((5, 3)), np.zeros(int(np.prod(GRID_ODD)), np.int32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    args = [m._m, p(src), C.c_int64(len(src)), 0, 0, p(R), p(t), p(cnt), p(stp), C.c_double(MAX_DIST), 5, p(idx), p(poses), p(stats), p(grid)]
    assert lib.svnicp_map_search(*args) == 0
    np.testing.assert_array_equal(idx, ref["index"])

    def bad_arrays():
        out = []
        for a_cnt in ([0, 3, 1, 3, 1, 5], [3, 3, -1, 3, 1, 5], [65536, 65536, 1, 1, 1, 1]):  # < 1, < 1, M = 2^32
            out.append(("counts", np.array(a_cnt, np.int32)))
        for a_stp in ([-0.1, 0, 0, 0, 0, 0], [0, np.nan, 0, 0, 0, 0], [0, 0, np.inf, 0, 0, 0]):
            out.append(("steps", np.array(a_stp)))
        return out
    for what, arr in bad_arrays():
        a = list(args)
        a[7 if what == "counts" else 8] = p(arr)
        assert lib.svnicp_map_search(*a) == ERR_INVALID, (what, arr)
        assert lib.svnicp_map_search(*args) == 0
    for i, bad in ((0, None), (1, None), (5, None), (6, None), (7, None), (8, None), (11, None), (12, None), (13, None),
                   (2, C.c_int64(0)), (2, C.c_int64((1 << 30) + 1)), (9, C.c_double(np.nan)), (9, C.c_double(0.0)),
                   (9, C.c_double(4.01 ** 2)), (10, 0), (10, -1), (10, 1025), (10, int(np.prod(GRID_ODD)) + 1)):
        a = list(args)
        a[i] = bad
        assert lib.svnicp_map_search(*a) == ERR_INVALID, i
        assert lib.svnicp_map_search(*args) == 0
    with pytest.raises(sv.SvnIcpError, match="top_k"):
        search(m, src, Rg, tg, (1, 1, 1, 1, 1, 1), k=2)
    with pytest.raises(sv.SvnIcpError, match="at most 4"):
        search(m, src, Rg, tg, GRID_ODD, md=4.01 ** 2)
    # largest allowed k on a grid of fewer than 1024 poses: every pose, ranked
    M = int(np.prod(GRID_ODD))
    r = search(m, src, Rg, tg, GRID_ODD, k=M)
    np.testing.assert_array_equal(np.sort(r["index"]), np.arange(M))
    np.testing.assert_array_equal(r["index"], topk_lexsort(r["counts"], M))
    assert_same(search(m, src, Rg, tg, GRID_ODD, k=5), ref)


def _yaw(a):
    c, s = np.cos(a), np.sin(a)
    return np.array([[c, -s, 0], [s, c, 0], [0, 0, 1.0]])


def test_relocalise_end_to_end(tmp_path, drive64):
    """Save the 12-scan map, Load it, search scan 14 (not in the map, down-sampled on the device) around a guess that is
    (+2.1 m, -1.4 m, +20 deg) off, and register from the best grid pose."""
    import torch
    world, built = drive64
    path = str(tmp_path / "map.svnmap")
    built.Save(path)
    m = sv.VoxelHashMap.Load(path)
    assert (m.Size(), m.PointCount()) == (built.Size(), built.PointCount())
    pts, (Rg, tg) = synth.make_scan(world, 14, "64", SEED)
    pre = sv.ScanPreprocessor(len(pts))
    p1, n1 = pre.downsample_uniform(pts.astype(np.float32), 0.5)
    p2, n2 = pre.downsample_uniform(p1, 1.5, n=n1, on_device=True)
    assert 300 < n2 < 5000
    yaw = np.deg2rad(20.0)
    R0, t0 = Rg @ _yaw(yaw), tg + np.array([2.1, -1.4, 0.0])
    counts = (33, 33, 1, 1, 1, 31)  # +-4 m at 0.25 m, yaw +-30 deg at 2 deg
    steps = (0.25, 0.25, 0.0, 0.0, 0.0, np.deg2rad(2.0))
    # with the registration's r = 1.73 m a shift along the road keeps nearly every point an inlier; r = 0.5 m does not
    r = m.SearchDevice(p2, n2, False, R0, t0, counts, steps, 0.25, top_k=5)
    best = r["poses"][:, 0]
    t_true, w_true = R0.T @ (tg - t0), np.array([0.0, 0.0, -yaw])  # T0^-1 T_true: R0^T Rg = Rz(-yaw)
    assert np.all(np.abs(best[:2] - t_true[:2]) <= 0.25 + 1e-9), (best, t_true)
    assert abs(best[5] - w_true[2]) <= np.deg2rad(2.0) + 1e-9, (best, w_true)
    Rb, tb = R0 @ exp_so3(best[3:]), t0 + R0 @ best[:3]

    def register(Rs, ts):
        rng = np.random.default_rng(5)
        P = 64
        icp = sv.SVNICP(sv.SteinICPParam(iterations=30, KNN_count=32, max_dist=MAX_DIST, lr=1.0, SVN_full_grad=True),
                        synth.init_particles(P, rng))
        ptr, n_t = m.GetMapDevice(ts, 110.0)
        src = torch.from_numpy(np.ascontiguousarray(pts, dtype=np.float64)).cuda()
        init = synth.init_particles(P, rng)
        icp.add_cloud_device(src.data_ptr(), len(pts), ptr, n_t, init)
        icp.set_initial_mean(Rs, ts)
        state = icp.stein_align()
        x = icp.get_transformation()
        Rc, tc = Rs @ exp_so3(x[3:]), ts + Rs @ x[:3]
        return state, float(np.linalg.norm(tc - tg)), float(np.linalg.norm(Rc @ Rg.T - np.eye(3)))

    state, et, er = register(Rb, tb)
    _, et0, er0 = register(R0, t0)
    print(f"relocalise: best grid pose {best[:2]} m, {np.rad2deg(best[5]):.1f} deg (truth {t_true[:2]}, {np.rad2deg(w_true[2]):.1f}); "
          f"registered from it: {et:.3f} m / {er:.2e}; from the perturbed guess: {et0:.3f} m / {er0:.2e}")
    assert state == sv.ALIGN_SUCCESS
    assert et < 0.15 and er < 5e-3, (et, er)
