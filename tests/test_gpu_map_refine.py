"""svnicp_map_refine (VoxelHashMap.Refine): Gauss-Newton refinement of pose hypotheses against the device local map.

Checked against the fp64 oracle (tests/map_refine_oracle.c) one update at a time from svnicp_map_evaluate's own H and b, and over
whole runs; against chained one-iteration calls (the seeds must not matter), svnicp_map_evaluate at the returned poses, the same
pose in other batches, orders, calls and slot layouts; for its behaviour near the truth, off the map, with tol and across yaw
+-pi; and end to end after a whole-map Search."""
import ctypes as C

import numpy as np
import pytest

import svn_icp_b200 as sv
from svn_icp_b200 import synth
from test_gpu_map_evaluate import MAX_DIST, SEED, drive_map, exp_so3
from test_gpu_map_search import GRID_MIXED, GRID_ODD, STEPS, all_poses
from test_map_refine_cpu import refine_oracle, refine_update, rot_angle_between

pytestmark = pytest.mark.gpu

ERR_INVALID = -1  # SVNICP_ERR_INVALID
KEYS = ("poses", "iterations", "step", "inliers", "fitness", "rmse", "H", "b")


@pytest.fixture(scope="module")
def drive():
    """map of 6 scans of the 32-beam sensor; 4000 points of scan 8 and its ground-truth pose"""
    world, m = drive_map()
    pts, (R, t) = synth.make_scan(world, 8, "32", SEED)
    sel = np.sort(np.random.default_rng(1).choice(len(pts), 4000, replace=False))
    return m, pts[sel].astype(np.float32), R, t


@pytest.fixture(scope="module")
def drive64():
    return drive_map("64", range(12))


def perturbations(M, seed, dt=0.5, dw=np.deg2rad(5.0)):
    rng = np.random.default_rng(seed)
    return np.concatenate([rng.uniform(-dt, dt, (3, M)), rng.uniform(-dw, dw, (3, M))])


def assert_same(a, b, j=None):
    for k in a:
        got = b[k] if j is None else (b[k][:, j] if k == "poses" else b[k][j])
        np.testing.assert_array_equal(a[k], got, err_msg=k)


def world(R0, t0, x):
    return R0 @ exp_so3(x[3:]), t0 + R0 @ x[:3]


@pytest.mark.parametrize("counts", [GRID_ODD, GRID_MIXED], ids=["odd", "mixed"])
def test_one_step_against_oracle(drive, counts):
    import torch
    m, src, Rg, tg = drive
    x = all_poses(counts, STEPS)
    ev = m.Evaluate(src, Rg, tg, x, MAX_DIST)
    want = np.stack([refine_update(x[:, j], ev["H"][j], ev["b"][j])[0] for j in range(x.shape[1])], axis=1)
    dn = np.array([refine_update(x[:, j], ev["H"][j], ev["b"][j])[1] for j in range(x.shape[1])])
    ref = None
    for dt, f64 in ((np.float32, False), (np.float64, True)):
        host = m.Refine(src.astype(dt), Rg, tg, x, MAX_DIST, iterations=1, tol=0.0, want_system=True)
        d = torch.from_numpy(np.ascontiguousarray(src, dtype=dt)).cuda()
        dev = m.RefineDevice(d.data_ptr(), len(src), f64, Rg, tg, x, MAX_DIST, iterations=1, tol=0.0, want_system=True)
        assert_same(host, dev)
        if ref is None:
            ref = host
        assert_same(ref, host)
        assert np.abs(host["poses"] - want).max() <= 1e-12
        np.testing.assert_allclose(host["step"], dn, rtol=1e-12, atol=0)
        assert (host["iterations"] == 1).all()


def test_chaining_equals_one_call(drive):
    """Refine(x, 30, tol = 0) is 30 chained Refine(., 1) calls, bit for bit: the seeds change nothing.  With tol > 0 the poses and
    the iteration counts are those of chained calls stopped at the first step below tol."""
    m, src, Rg, tg = drive
    x0 = perturbations(8, 3)
    full = m.Refine(src, Rg, tg, x0, MAX_DIST, iterations=30, tol=0.0)
    x, steps = x0.copy(), []
    for _ in range(30):
        one = m.Refine(src, Rg, tg, x, MAX_DIST, iterations=1, tol=0.0)
        x = one["poses"]
        steps.append(one["step"])
    np.testing.assert_array_equal(full["poses"], x)
    np.testing.assert_array_equal(full["step"], steps[-1])
    assert (full["iterations"] == 30).all()
    tol = 1e-4
    stop = m.Refine(src, Rg, tg, x0, MAX_DIST, iterations=30, tol=tol)
    for j in range(x0.shape[1]):
        xj, its = x0[:, j], 0
        while its < 30:
            one = m.Refine(src, Rg, tg, xj, MAX_DIST, iterations=1, tol=0.0)
            xj, its = one["poses"], its + 1
            if one["step"] < tol:
                break
        np.testing.assert_array_equal(stop["poses"][:, j], xj)
        assert stop["iterations"][j] == its
        # tol stops a pose at the iteration where |delta| first drops below it
        first = next((i + 1 for i in range(30) if np.asarray(steps[i])[j] < tol), 30)
        assert its == first
    assert (stop["iterations"] < 30).any()


def test_final_outputs_equal_evaluate(drive):
    m, src, Rg, tg = drive
    r = m.Refine(src, Rg, tg, perturbations(40, 4), MAX_DIST, iterations=7, tol=1e-6, want_system=True)
    ev = m.Evaluate(src, Rg, tg, r["poses"], MAX_DIST)
    for k in ("inliers", "fitness", "rmse", "H", "b"):
        np.testing.assert_array_equal(r[k], ev[k], err_msg=k)


def test_invariance(drive):
    """one pose alone, inside 1024 poses, in shuffled order, on a map imported from its export, and on a repeated call"""
    m, src, Rg, tg = drive
    x = perturbations(1024, 5)
    kw = dict(iterations=10, tol=1e-6, want_system=True)
    full = m.Refine(src, Rg, tg, x, MAX_DIST, **kw)
    again = m.Refine(src, Rg, tg, x, MAX_DIST, **kw)
    assert_same(full, again)
    perm = np.random.default_rng(6).permutation(1024)
    shuf = m.Refine(src, Rg, tg, x[:, perm], MAX_DIST, **kw)
    twin = sv.VoxelHashMap(m.voxel_size_, m.max_range_, m.max_pointscount_, capacity_voxels=1 << 18)
    twin.Import(m.Export())
    imp = twin.Refine(src, Rg, tg, x, MAX_DIST, **kw)
    assert_same(full, imp)
    inv = np.argsort(perm)
    for k in KEYS:
        np.testing.assert_array_equal(shuf[k][:, inv] if k == "poses" else shuf[k][inv], full[k], err_msg=k)
    for j in (0, 31, 32, 511, 1023):
        assert_same(m.Refine(src, Rg, tg, x[:, j], MAX_DIST, **kw), full, j)


def test_against_fp64_oracle(drive):
    """30 iterations from perturbations within +-0.5 m and +-5 deg: the fp64 oracle (brute-force nearest point, Newton_grad_right
    on the correspondences, LDL^T, the same update) ends at the same poses after the same number of iterations"""
    m, src, Rg, tg = drive
    x0 = perturbations(6, 7)
    r = m.Refine(src, Rg, tg, x0, MAX_DIST, iterations=30)
    xo, its, step, cnt = refine_oracle(src, m.GetMap(), Rg, tg, x0, MAX_DIST, 30, sv.SteinICPParam.convergence_threshold)
    print(f"oracle: max |x - x_oracle| = {np.abs(r['poses'] - xo).max():.2e}, iterations {r['iterations'].tolist()}")
    np.testing.assert_array_equal(r["iterations"], its)
    np.testing.assert_array_equal(r["inliers"], cnt)
    assert np.abs(r["poses"] - xo).max() <= 1e-9


def test_behaviour_near_and_far(drive):
    m, src, Rg, tg = drive
    x0 = perturbations(16, 8)
    r = m.Refine(src, Rg, tg, x0, MAX_DIST, iterations=30)
    # the optimum of this 4000-point sample sits about 0.03 m / 0.3 deg from the synthetic truth: the bars are 0.15 m and 0.5 deg
    assert np.abs(r["poses"][:3]).max() < 0.15 and np.abs(r["poses"][3:]).max() < np.deg2rad(0.5), r["poses"]
    ev0 = m.Evaluate(src, Rg, tg, x0, MAX_DIST, want_system=False)
    assert (r["inliers"] >= ev0["inliers"]).all()
    far = m.Refine(src, Rg, tg + np.array([5e4, -3e4, 100.0]), x0[:, :4], MAX_DIST, iterations=5, tol=0.0, want_system=True)
    np.testing.assert_array_equal(far["poses"], x0[:, :4])
    assert (far["inliers"] == 0).all() and (far["step"] == 0).all() and (far["iterations"] == 5).all()
    assert np.isfinite(far["H"]).all() and np.isfinite(far["b"]).all()
    stop = m.Refine(src, Rg, tg + np.array([5e4, -3e4, 100.0]), x0[:, 0], MAX_DIST, iterations=5, tol=1e-9)
    assert stop["iterations"] == 1 and stop["step"] == 0.0


def _rz(a):
    c, s = np.cos(a), np.sin(a)
    return np.array([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]])


def test_yaw_across_pi(drive):
    """T0 placed so that the truth sits at a relative yaw of pi; hypotheses at pi, +-179 and -179.5 deg converge to the truth"""
    m, src, Rg, tg = drive
    R0, t0 = Rg @ _rz(np.pi).T, tg.copy()
    yaws = np.array([np.pi, np.deg2rad(179.0), np.deg2rad(-179.0), np.deg2rad(-179.5)])
    x0 = np.zeros((6, 4))
    x0[5] = yaws
    x0[0] = 0.2
    r = m.Refine(src, R0, t0, x0, MAX_DIST, iterations=30)
    assert (np.linalg.norm(r["poses"][3:], axis=0) <= np.pi + 1e-12).all()
    for j in range(4):
        Rw, tw = world(R0, t0, r["poses"][:, j])
        assert rot_angle_between(Rw, Rg) < np.deg2rad(0.3) and np.linalg.norm(tw - tg) < 0.05, (j, r["poses"][:, j])


def test_large_scan_blocks(drive64):
    """the full 64-beam scan (~143 k points): 64 poses span several pose blocks and equal single-pose calls bit for bit"""
    world_, m = drive64
    pts, (Rg, tg) = synth.make_scan(world_, 14, "64", SEED)
    src = pts.astype(np.float32)
    assert len(src) > 100_000
    x = perturbations(64, 9, 0.3, np.deg2rad(2.0))
    kw = dict(iterations=4, tol=0.0, want_system=True)
    full = m.Refine(src, Rg, tg, x, MAX_DIST, **kw)
    for j in (0, 1, 33, 34, 35, 36, 63):
        assert_same(m.Refine(src, Rg, tg, x[:, j], MAX_DIST, **kw), full, j)


def test_errors_and_side_effects(drive):
    m, src, Rg, tg = drive
    ok = dict(R0=Rg, t0=tg, poses=np.zeros(6))
    for md in (np.nan, np.inf, 0.0, -1.0):
        with pytest.raises(sv.SvnIcpError, match="max_dist"):
            m.Refine(src, max_dist=md, **ok)
    with pytest.raises(sv.SvnIcpError, match="at most 4"):
        m.Refine(src, max_dist=4.01 ** 2, **ok)
    with pytest.raises(sv.SvnIcpError, match="source points"):
        m.Refine(np.zeros((0, 3), np.float32), Rg, tg, np.zeros(6), MAX_DIST)
    with pytest.raises(sv.SvnIcpError, match="n_poses"):
        m.Refine(src, Rg, tg, np.zeros((6, 0)), MAX_DIST)
    with pytest.raises(sv.SvnIcpError, match="n_poses"):
        m.Refine(src[:10], Rg, tg, np.zeros((6, 65537)), MAX_DIST, iterations=1)
    for it in (0, -1, 1001):
        with pytest.raises(sv.SvnIcpError, match="iterations"):
            m.Refine(src, max_dist=MAX_DIST, iterations=it, **ok)
    for tol in (-1e-9, np.nan, np.inf):
        with pytest.raises(sv.SvnIcpError, match="tol"):
            m.Refine(src, max_dist=MAX_DIST, tol=tol, **ok)
    lib, R, t, x = m._lib, Rg.ravel().copy(), tg.copy(), np.zeros(6)
    xo, its, step, stats = np.zeros(6), np.zeros(1, np.int32), np.zeros(1), np.zeros(3)
    p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    args = [m._m, p(src), C.c_int64(len(src)), 0, 0, p(R), p(t), 1, p(x), C.c_double(MAX_DIST), 3, C.c_double(0.0), p(xo), p(its),
            None, p(stats), None, None]
    assert lib.svnicp_map_refine(*args) == 0
    for i in (0, 1, 5, 6, 8, 12, 13, 15):
        a = list(args)
        a[i] = None
        assert lib.svnicp_map_refine(*a) == ERR_INVALID, i
    # no side effects: Size(), the GetMap pointer and its content, the Export bytes
    before = m.GetMap()
    ptr, n = m.GetMapDevice()
    size, pts, snap = m.Size(), m.PointCount(), m.Export()
    m.Refine(src, Rg, tg, perturbations(50, 10), MAX_DIST, iterations=5, want_system=True)
    m.Refine(src.astype(np.float64), Rg, tg, perturbations(5, 11), MAX_DIST, iterations=5)
    assert (m.Size(), m.PointCount()) == (size, pts)
    after = np.zeros((n, 3))
    assert m._lib.svnicp_map_download(m._m, after.ctypes.data_as(C.c_void_p), C.c_int64(n)) == 0
    np.testing.assert_array_equal(after, before)
    assert m.GetMapDevice()[0] == ptr
    s2 = m.Export()
    for a, b in ((snap.voxels, s2.voxels), (snap.counts, s2.counts), (snap.points, s2.points)):
        assert a.tobytes() == b.tobytes()


def test_relocalise_search_then_refine(tmp_path, drive64):
    """No prior: scan 14 against the saved and reloaded 12-scan map, the whole-map grid of DESIGN 10e (0.5 m, yaw at 4 deg),
    top 5; Refine all five at max_dist = 3, then again from there at max_dist = 1; the best by count within the bars of
    test_relocalise_end_to_end, with no fine search and no registration."""
    import time
    world_, built = drive64
    path = str(tmp_path / "map.svnmap")
    built.Save(path)
    m = sv.VoxelHashMap.Load(path)
    snap = m.Export()
    v = m.voxel_size_
    lo, hi = snap.voxels.min(0)[:2] * v, (snap.voxels.max(0)[:2] + 1) * v
    pts, (Rg, tg) = synth.make_scan(world_, 14, "64", SEED)
    pre = sv.ScanPreprocessor(len(pts))
    p1, n1 = pre.downsample_uniform(pts.astype(np.float32), 0.5)
    p2, n2 = pre.downsample_uniform(p1, 1.5, n=n1, on_device=True)
    R0, t0 = np.eye(3), np.array([0.5 * (lo[0] + hi[0]), 0.5 * (lo[1] + hi[1]), tg[2]])
    counts = (int((hi[0] - lo[0]) / 0.5) + 1, int((hi[1] - lo[1]) / 0.5) + 1, 1, 1, 1, 90)
    steps = (0.5, 0.5, 0.0, 0.0, 0.0, np.deg2rad(4.0))
    t_start = time.perf_counter()
    s = m.SearchDevice(p2, n2, False, R0, t0, counts, steps, 0.25, top_k=5)
    r1 = m.RefineDevice(p1, n1, False, R0, t0, s["poses"], 3.0, iterations=30)
    r2 = m.RefineDevice(p1, n1, False, R0, t0, r1["poses"], 1.0, iterations=30)
    wall = time.perf_counter() - t_start
    order = np.lexsort((np.arange(5), -r2["inliers"]))
    best = r2["poses"][:, order[0]]
    Rb, tb = world(R0, t0, best)
    et, er = float(np.linalg.norm(tb - tg)), float(np.linalg.norm(Rb @ Rg.T - np.eye(3)))
    errs = []
    for j in range(5):
        Rj, tj = world(R0, t0, r2["poses"][:, j])
        errs.append((int(r2["inliers"][j]), round(float(np.linalg.norm(tj - tg)), 3)))
    print(f"search + refine: {wall * 1e3:.1f} ms, best by count {et:.4f} m / {er:.2e}; (count, error m) of the five: {errs}; "
          f"second best count {r2['inliers'][order[1]]} of {n1}")
    assert et < 0.15 and er < 5e-3, (et, er)
