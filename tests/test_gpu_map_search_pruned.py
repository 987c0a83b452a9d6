"""svnicp_map_search without per-pose counts: the branch-and-bound path (block bounds, best bound first, stop once the next bound
is below the k-th count) must return exactly what the exhaustive path returns.  Every comparison runs both paths on the same
map and scan: want_counts=True forces the exhaustive path, want_counts=False takes the pruned one where the grid allows blocks.
SearchInfo tells which ran, and on the pruned path how many poses exceeded their block's bound (always 0)."""
import ctypes as C

import numpy as np
import pytest

import svn_icp_b200 as sv
from svn_icp_b200 import synth
from test_gpu_map_evaluate import MAX_DIST, SEED, exp_so3
from test_gpu_map_search import GRID_MIXED, GRID_ODD, STEPS, drive, drive64  # noqa: F401  (fixtures)

pytestmark = pytest.mark.gpu

ERR_INVALID = -1  # SVNICP_ERR_INVALID
FIELDS = ("index", "poses", "count", "fitness", "rmse")


def both(m, src, R0, t0, counts, steps=STEPS, k=1, md=MAX_DIST, device=None):
    """(pruned-or-exhaustive result, its SearchInfo, exhaustive result); device = (ptr, n, f64) searches a device cloud"""
    def run(want):
        if device is None:
            return m.Search(src, R0, t0, counts, steps, md, top_k=k, want_counts=want)
        return m.SearchDevice(*device, R0, t0, counts, steps, md, top_k=k, want_counts=want)
    fast = run(False)
    info = m.SearchInfo()
    full = run(True)
    full_info = m.SearchInfo()
    M = int(np.prod(counts))
    assert full_info["path"] == 0 and full_info["poses_counted"] == M == full_info["grid_poses"] and full_info["violations"] == -1
    assert info["grid_poses"] == M
    if info["path"] == 1:
        assert info["violations"] == 0, info
        assert 0 < info["poses_counted"] <= M and 0 < info["blocks_counted"] <= info["blocks"]
        assert info["bound_queries"] == info["blocks"] * (len(src) if device is None else device[1])
    else:
        assert info["poses_counted"] == M and info["blocks"] == 0 and info["violations"] == -1
    return fast, info, full


def assert_equal(a, b):
    for f in FIELDS:
        np.testing.assert_array_equal(a[f], b[f], err_msg=f)


Z_GRID = ((9, 9, 5, 1, 1, 4), np.array([0.3, 0.25, 0.15, 0.0, 0.0, 0.05]))
ZERO_STEP = ((9, 9, 1, 1, 1, 6), np.array([0.3, 0.0, 0.15, 0.0, 0.0, 0.05]))
GRIDS = {"odd": (GRID_ODD, STEPS), "mixed": (GRID_MIXED, STEPS), "two_chunks": ((41, 41, 1, 1, 1, 10), STEPS), "z_blocks": Z_GRID,
         "zero_step": ZERO_STEP}


@pytest.mark.parametrize("grid", list(GRIDS), ids=list(GRIDS))
def test_pruned_equals_exhaustive(drive, grid):  # noqa: F811
    import torch
    m, src, Rg, tg = drive
    counts, steps = GRIDS[grid]
    M = int(np.prod(counts))
    paths = set()
    for dt, f64 in ((np.float32, False), (np.float64, True)):
        s = np.ascontiguousarray(src, dtype=dt)
        d = torch.from_numpy(s).cuda()
        for k in (1, 7, 1024):
            if k > M:
                continue
            for dev in (None, (d.data_ptr(), len(s), f64)):
                fast, info, full = both(m, s, Rg, tg, counts, steps, k=k, device=dev)
                assert_equal(fast, full)
                paths.add(info["path"])
    if grid in ("two_chunks", "z_blocks", "zero_step", "mixed"):
        assert 1 in paths, paths


def test_pruned_tight_radius(drive):  # noqa: F811
    """max_dist = 0.25: larger blocks and real pruning on the two-chunk grid"""
    m, src, Rg, tg = drive
    counts = (41, 41, 1, 1, 1, 10)
    for k in (1, 7, 1024):
        fast, info, full = both(m, src, Rg, tg, counts, k=k, md=0.25)
        assert_equal(fast, full)
        assert info["path"] == 1


def test_full_size_scan(drive64):  # noqa: F811
    """143 k points: 936 poses per chunk, blocks of up to 400 poses"""
    world, m = drive64
    src, (Rg, tg) = synth.make_scan(world, 12, "64", SEED)
    src = src.astype(np.float32)
    counts, steps = (21, 21, 1, 1, 1, 5), (0.25, 0.25, 0.0, 0.0, 0.0, np.deg2rad(2.0))
    fast, info, full = both(m, src, Rg, tg, counts, steps, k=20, md=0.25)
    assert_equal(fast, full)
    assert info["path"] == 1
    print(f"full-size scan: {info}")


def lattice_map(L=8.0, s=2.0, n=600_000):
    """A dense single-layer lattice at 0.25 m (voxels of 0.5 m) and a scan of lattice points repeated to n: every grid pose at
    0.25 m steps puts every scan point exactly on a map point, so every pose and every block bound is n."""
    g = np.arange(-L, L + 1e-9, 0.25)
    X, Y = np.meshgrid(g, g, indexing="ij")
    mp = np.stack([X.ravel(), Y.ravel(), np.full(X.size, 0.125)], 1).astype(np.float32)
    m = sv.VoxelHashMap(0.5, 1e3, 32, capacity_voxels=1 << 14)
    m.AddPointCloud(mp, np.eye(3), np.zeros(3))
    assert m.PointCount() == len(mp)
    h = np.arange(-s, s + 1e-9, 0.25)
    X, Y = np.meshgrid(h, h, indexing="ij")
    sc = np.stack([X.ravel(), Y.ravel(), np.full(X.size, 0.125)], 1).astype(np.float32)
    return m, np.ascontiguousarray(np.resize(sc, (n, 3)))


def test_ties_at_the_stop_rule():
    """All poses tie at the top count n, and so do all bounds; blocks are walked in id order, one per chunk (n = 600 k points:
    223 poses per chunk, blocks of 11 x 11).  With k = b0 + 1 the first block holds g = 0 .. b0 - 1 and g = counts[0], and
    the k-th winner g = b0 sits in the next block, whose bound equals the k-th count: a stop on an equal bound returns
    counts[0] instead."""
    m, src = lattice_map()
    counts, steps = (31, 31, 1, 1, 1, 1), (0.25, 0.25, 0.0, 0.0, 0.0, 0.0)
    R0, t0 = np.eye(3), np.zeros(3)
    fast, info, full = both(m, src, R0, t0, counts, steps, k=1, md=0.01)
    assert_equal(fast, full)
    assert info["path"] == 1 and (full["count"] == len(src)).all()
    b0 = int(round(info["poses_per_block"] ** 0.5))
    assert b0 * b0 == info["poses_per_block"] and 2 * info["poses_per_block"] > (1 << 27) // len(src)  # one block per chunk
    for k in (b0 + 1, 2 * b0 + 3):
        fast, info, full = both(m, src, R0, t0, counts, steps, k=k, md=0.01)
        assert_equal(fast, full)
        np.testing.assert_array_equal(fast["index"], np.arange(k))
        assert info["path"] == 1 and info["blocks_counted"] >= 2


def test_bound_at_the_block_corner():
    """One map point and one scan point: the only pose with an inlier is the far corner of block (0, 0) (11 x 11 blocks at
    0.25 m), at exactly rho = |(1.25, 1.25)| from the block's centre.  A bound taken anywhere but the centre misses it."""
    m = sv.VoxelHashMap(0.5, 1e3, 32, capacity_voxels=1 << 10)
    m.AddPointCloud(np.array([[-1.125, -1.125, 0.125]], np.float32), np.eye(3), np.zeros(3))
    src = np.array([[0.125, 0.125, 0.125]], np.float32)
    counts, steps = (31, 31, 1, 1, 1, 1), (0.25, 0.25, 0.0, 0.0, 0.0, 0.0)
    for k in (1, 7):
        fast, info, full = both(m, src, np.eye(3), np.zeros(3), counts, steps, k=k, md=0.01)
        assert_equal(fast, full)
        assert info["path"] == 1 and info["poses_per_block"] == 121
        assert full["index"][0] == 10 + 31 * 10 and full["count"][0] == 1


def test_edges_and_degenerate_grids(drive):  # noqa: F811
    m, src, Rg, tg = drive
    # partial edge blocks on both axes (blocks of 7 x 7 at 0.5 m)
    counts, steps = (9, 8, 1, 1, 1, 2), np.array([0.5, 0.5, 0.0, 0.0, 0.0, 0.05])
    M = int(np.prod(counts))
    for k in (1, 7):
        fast, info, full = both(m, src, Rg, tg, counts, steps, k=k)
        assert_equal(fast, full)
        assert info["path"] == 1 and info["poses_per_block"] == 49, info
    # k = M: every pose, ranked (a grid below 16 k poses: the exhaustive path)
    fast, info, full = both(m, src, Rg, tg, counts, steps, k=M)
    assert_equal(fast, full)
    assert info["path"] == 0
    # far from the map every count and every bound is 0: winners g = 0 .. k-1, nothing pruned
    for k in (1, 7, 1024):
        fast, info, full = both(m, src, Rg, tg + np.array([5e4, -3e4, 100.0]), (41, 41, 1, 1, 1, 10), k=k)
        assert_equal(fast, full)
        np.testing.assert_array_equal(fast["index"], np.arange(k))
        assert info["path"] == 1 and info["poses_counted"] == info["grid_poses"], info
    # no translation blocks: rotation only, and a radius at the 4-voxel limit
    for counts, md in (((1, 1, 1, 1, 1, 30), MAX_DIST), ((41, 41, 1, 1, 1, 2), 3.9 ** 2)):
        fast, info, full = both(m, src, Rg, tg, counts, k=3, md=md)
        assert_equal(fast, full)
        assert info["path"] == 0
    # R0 not orthonormal: rho comes from R0 itself
    fast, info, full = both(m, src, 1.01 * Rg, tg, (41, 41, 1, 1, 1, 10), k=7)
    assert_equal(fast, full)
    assert info["path"] == 1


def test_deterministic_no_side_effects_and_info(drive):  # noqa: F811
    m, src, Rg, tg = drive
    fresh = sv.VoxelHashMap(1.0, 100.0, 20)
    out = np.zeros(8, np.int64)
    assert fresh._lib.svnicp_map_search_info(fresh._m, out.ctypes.data_as(C.c_void_p)) == ERR_INVALID
    with pytest.raises(sv.SvnIcpError, match="SearchInfo"):
        fresh.SearchInfo()
    before = m.GetMap()
    ptr, n = m.GetMapDevice()
    size = (m.Size(), m.PointCount())
    counts = (41, 41, 1, 1, 1, 10)
    a = m.Search(src, Rg, tg, counts, STEPS, 0.25, top_k=1024)
    ia = m.SearchInfo()
    b = m.Search(src, Rg, tg, counts, STEPS, 0.25, top_k=1024)
    assert m.SearchInfo() == ia and ia["path"] == 1
    twin = sv.VoxelHashMap(m.voxel_size_, m.max_range_, m.max_pointscount_, capacity_voxels=1 << 17)
    twin.Import(m.Export())
    c = twin.Search(src, Rg, tg, counts, STEPS, 0.25, top_k=1024)
    assert twin.SearchInfo() == ia
    for f in FIELDS:
        np.testing.assert_array_equal(a[f], b[f])
        np.testing.assert_array_equal(a[f], c[f])
    assert (m.Size(), m.PointCount()) == size
    after = np.zeros((n, 3))
    assert m._lib.svnicp_map_download(m._m, after.ctypes.data_as(C.c_void_p), C.c_int64(n)) == 0
    np.testing.assert_array_equal(after, before)
    assert m.GetMapDevice() == (ptr, n)
    # an argument error leaves the last successful call's values
    with pytest.raises(sv.SvnIcpError):
        m.Search(src, Rg, tg, counts, STEPS, 0.25, top_k=0)
    with pytest.raises(sv.SvnIcpError):
        m.Search(src, Rg, tg, (0, 41, 1, 1, 1, 10), STEPS, 0.25, top_k=1)
    assert m.SearchInfo() == ia
    assert m._lib.svnicp_map_search_info(m._m, None) == ERR_INVALID
    assert m._lib.svnicp_map_search_info(None, out.ctypes.data_as(C.c_void_p)) == ERR_INVALID


def test_global_relocalisation(tmp_path, drive64):  # noqa: F811
    """No prior: scan 14 against the saved and reloaded 12-scan map over the map's whole x-y extent at 0.5 m and the full yaw
    circle at 4 deg, from T0 at the centre of the extent with identity yaw (z, roll and pitch at the sensor's mounting pose)."""
    import torch
    world, built = drive64
    path = str(tmp_path / "map.svnmap")
    built.Save(path)
    m = sv.VoxelHashMap.Load(path)
    snap = m.Export()
    v = m.voxel_size_
    lo, hi = snap.voxels.min(0)[:2] * v, (snap.voxels.max(0)[:2] + 1) * v
    pts, (Rg, tg) = synth.make_scan(world, 14, "64", SEED)
    pre = sv.ScanPreprocessor(len(pts))
    p1, n1 = pre.downsample_uniform(pts.astype(np.float32), 0.5)
    p2, n2 = pre.downsample_uniform(p1, 1.5, n=n1, on_device=True)
    R0, t0 = np.eye(3), np.array([0.5 * (lo[0] + hi[0]), 0.5 * (lo[1] + hi[1]), tg[2]])
    counts = (int((hi[0] - lo[0]) / 0.5) + 1, int((hi[1] - lo[1]) / 0.5) + 1, 1, 1, 1, 90)  # yaw -178 .. 178 deg
    steps = (0.5, 0.5, 0.0, 0.0, 0.0, np.deg2rad(4.0))
    M = int(np.prod(counts))
    assert 1e6 < M < 1e7
    fast, info, full = both(m, None, R0, t0, counts, steps, k=5, md=0.25, device=(p2, n2, False))
    assert_equal(fast, full)
    assert info["path"] == 1
    frac = info["poses_counted"] / M
    print(f"global relocalisation: {M} poses, {info['blocks']} blocks of {info['poses_per_block']}, "
          f"{info['blocks_counted']} blocks counted, fraction of poses counted {frac:.4f}")
    assert frac < 0.3, info  # 0.18 measured
    best = fast["poses"][:, 0]
    t_true = R0.T @ (tg - t0)
    yaw_true = np.arctan2(Rg[1, 0], Rg[0, 0])
    assert np.all(np.abs(best[:2] - t_true[:2]) <= 0.5 + 1e-9), (best, t_true)
    dyaw = (best[5] - yaw_true + np.pi) % (2 * np.pi) - np.pi
    assert abs(dyaw) <= np.deg2rad(4.0) + 1e-9, (best, yaw_true)
    # coarse to fine: +-0.5 m at 0.125 m and +-2 deg at 0.5 deg around the winner, then register from there
    Rw, tw = R0 @ exp_so3(best[3:]), t0 + R0 @ best[:3]
    fine = m.SearchDevice(p2, n2, False, Rw, tw, (9, 9, 1, 1, 1, 9), (0.125, 0.125, 0.0, 0.0, 0.0, np.deg2rad(0.5)), 0.25)
    xf = fine["poses"][:, 0]
    Rb, tb = Rw @ exp_so3(xf[3:]), tw + Rw @ xf[:3]
    rng = np.random.default_rng(5)
    P = 64
    icp = sv.SVNICP(sv.SteinICPParam(iterations=30, KNN_count=32, max_dist=MAX_DIST, lr=1.0, SVN_full_grad=True),
                    synth.init_particles(P, rng))
    ptr, n_t = m.GetMapDevice(tb, 110.0)
    src = torch.from_numpy(np.ascontiguousarray(pts, dtype=np.float64)).cuda()
    icp.add_cloud_device(src.data_ptr(), len(pts), ptr, n_t, synth.init_particles(P, rng))
    icp.set_initial_mean(Rb, tb)
    assert icp.stein_align() == sv.ALIGN_SUCCESS
    x = icp.get_transformation()
    Rc, tc = Rb @ exp_so3(x[3:]), tb + Rb @ x[:3]
    et, er = float(np.linalg.norm(tc - tg)), float(np.linalg.norm(Rc @ Rg.T - np.eye(3)))
    print(f"global relocalisation: best grid pose {best[:2]} m, {np.rad2deg(best[5]):.1f} deg (truth {t_true[:2]}, "
          f"{np.rad2deg(yaw_true):.1f}); registered from it: {et:.3f} m / {er:.2e}")
    assert et < 0.15 and er < 5e-3, (et, er)
