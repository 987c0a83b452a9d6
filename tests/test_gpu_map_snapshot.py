"""GPU tests of map snapshots (svnicp_map_export / svnicp_map_import, VoxelHashMap.Export / Import / Save / Load).
Bars: the export equals the sequential oracle's canonical export array for array, bit for bit, including the order of the
points inside each voxel; it does not depend on the slot layout; a restored map is the same map for every later call (exports,
GetMap sets, Evaluate bits, registration bits); a refused import leaves the map exactly as it was."""
import ctypes as C
import os

import numpy as np
import pytest

import svn_icp_b200 as sv
from svn_icp_b200 import synth
from test_map_snapshot_cpu import SnapshotOracle, snapshots_equal

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden", "vmap_sequence.npz")
SEED = 0xC0FFEE


def sort_rows(a):
    return a[np.lexsort((a[:, 2], a[:, 1], a[:, 0]))] if len(a) else a


def scans(ks, sensor="64", seed=SEED):
    world = synth.make_world(seed)
    for k in ks:
        pts, (R, t) = synth.make_scan(world, k, sensor, seed)
        yield pts.astype(np.float32), R, t


def dense_cloud(n=400_000, seed=3):
    """many small voxels on both sides of zero: several radix-sort tiles (4096 voxels each), every key field in play"""
    return np.random.default_rng(seed).uniform([-30, -30, -4], [30, 30, 4], (n, 3)).astype(np.float32)


def test_export_equals_oracle_on_reference_sequence():
    z = np.load(GOLD)
    voxel, max_range, cap, _ = z["params"]
    m = sv.VoxelHashMap(float(voxel), float(max_range), int(cap), capacity_voxels=1 << 14)
    o = SnapshotOracle(float(voxel), float(max_range), int(cap))
    for k in range(int(z["n_scans"][0])):
        m.AddPointCloud(z[f"cloud{k}"], z[f"R{k}"], z[f"t{k}"])
        o.AddPointCloud(z[f"cloud{k}"], z[f"R{k}"], z[f"t{k}"])
        s = m.Export()
        snapshots_equal(s, o.Export())
        assert len(s.counts) == m.Size() == int(z[f"size{k}"][0])
        np.testing.assert_array_equal(sort_rows(s.points), z[f"all{k}"])


def test_export_equals_oracle_on_full_size_drive_with_removal():
    """64-beam scans (~143 k points), 30 m range: voxels age out through RemoveFarPointCloud between the exports"""
    g = sv.VoxelHashMap(1.0, 30.0, 20)
    o = SnapshotOracle(1.0, 30.0, 20)
    removed = 0
    prev = set()
    for pts, R, t in scans(range(0, 48, 6)):
        g.AddPointCloud(pts, R, t)
        o.AddPointCloud(pts, R, t)
        s = g.Export()
        snapshots_equal(s, o.Export())
        cur = set(map(tuple, s.voxels.tolist()))
        removed += len(prev - cur)
        prev = cur
    assert removed > 500  # RemoveFar dropped voxels between exports


def test_export_equals_oracle_on_many_voxels():
    pts = dense_cloud()
    g = sv.VoxelHashMap(0.25, 1e4, 3, capacity_voxels=1 << 20)
    o = SnapshotOracle(0.25, 1e4, 3)
    for part in np.array_split(pts, 3):
        g.AddPointCloud(part, np.eye(3), np.zeros(3))
        o.AddPointCloud(part, np.eye(3), np.zeros(3))
    s = g.Export()
    assert len(s.counts) > 20 * 4096
    snapshots_equal(s, o.Export())


def test_export_independent_of_slot_layout():
    a = sv.VoxelHashMap(1.0, 30.0, 20, capacity_voxels=1 << 14)
    b = sv.VoxelHashMap(1.0, 30.0, 20, capacity_voxels=1 << 19)
    for pts, R, t in scans(range(0, 30, 6)):
        a.AddPointCloud(pts, R, t)
        b.AddPointCloud(pts, R, t)
        snapshots_equal(a.Export(), b.Export())
    c = sv.VoxelHashMap(0.25, 1e4, 3, capacity_voxels=1 << 18)
    d = sv.VoxelHashMap(0.25, 1e4, 3, capacity_voxels=1 << 21)
    pts = dense_cloud()
    c.AddPointCloud(pts, np.eye(3), np.zeros(3))
    d.AddPointCloud(pts, np.eye(3), np.zeros(3))
    snapshots_equal(c.Export(), d.Export())


def drive_map(capacity=1 << 19):
    m = sv.VoxelHashMap(1.0, 40.0, 20, capacity_voxels=capacity)
    for pts, R, t in scans(range(0, 24, 6)):
        m.AddPointCloud(pts, R, t)
    return m, t


def assert_same_map(a, b, t):
    snapshots_equal(a.Export(), b.Export())
    assert (a.Size(), a.PointCount()) == (b.Size(), b.PointCount())
    np.testing.assert_array_equal(sort_rows(a.GetMap()), sort_rows(b.GetMap()))
    np.testing.assert_array_equal(sort_rows(a.GetMap(t, 25.0)), sort_rows(b.GetMap(t, 25.0)))


def test_round_trip_and_identical_behaviour_afterwards():
    a, t = drive_map()
    s = a.Export()
    fresh = sv.VoxelHashMap(1.0, 40.0, 20, capacity_voxels=1 << 13)
    fresh.Import(s)
    busy = sv.VoxelHashMap(1.0, 40.0, 20)
    for pts, R, tt in scans(range(40, 46, 3)):
        busy.AddPointCloud(pts, R, tt)
    assert busy.Size() > 0
    busy.Import(s)
    for b in (fresh, busy):
        assert_same_map(a, b, t)
    # Evaluate: bit-identical stats, H, b, mask and nearest points at several poses
    src, Rg, tg = next(scans([24]))
    x = np.concatenate([np.zeros((6, 1)), synth.init_particles(5, np.random.default_rng(2))], axis=1)
    ea = a.Evaluate(src, Rg, tg, x, 3.0, want_system=True, want_mask=True, want_nearest=True)
    for b in (fresh, busy):
        eb = b.Evaluate(src, Rg, tg, x, 3.0, want_system=True, want_mask=True, want_nearest=True)
        for k in ea:
            assert ea[k].tobytes() == eb[k].tobytes(), k
    # the next scans of the drive, RemoveFar firing, keep all three maps the same after every step
    removed, prev = 0, set(map(tuple, s.voxels.tolist()))
    for pts, R, tt in scans(range(24, 48, 6)):
        for m in (a, fresh, busy):
            m.AddPointCloud(pts, R, tt)
        sa = a.Export()
        snapshots_equal(sa, fresh.Export())
        snapshots_equal(sa, busy.Export())
        cur = set(map(tuple, sa.voxels.tolist()))
        removed += len(prev - cur)
        prev = cur
    assert removed > 100  # RemoveFar fired on the restored maps too
    assert_same_map(a, fresh, tt)


def test_restored_map_gives_the_same_registration():
    """GetMapDevice -> add_cloud_device -> stein_align, as test_map_feeds_registration_without_leaving_the_gpu: the candidate
    table is ordered by (d0^2, map index); both maps hold the same points in each voxel in the same order, and the particles come
    out bit-identical (a tie in fp64 d0^2 between distinct points would be the only way the index order could matter)."""
    import torch
    pb = synth.make_problem(48, sensor="32", scan_index=6, n_map_scans=6, seed=SEED)
    a = sv.VoxelHashMap(1.0, 100.0, 20)
    for pts, R, t in scans(range(6), "32"):
        a.AddPointCloud(pts, R, t)
    b = sv.VoxelHashMap(1.0, 100.0, 20, capacity_voxels=1 << 16)
    b.Import(a.Export())
    prm = sv.SteinICPParam(iterations=6, KNN_count=32, max_dist=3.0, lr=1.0)
    src = torch.from_numpy(np.ascontiguousarray(pb.source)).cuda()
    out = []
    for m in (a, b):
        ptr, n_t = m.GetMapDevice(pb.t0, 100.0)
        assert n_t > 1000
        icp = sv.SVNICP(prm, pb.init_pose)
        icp.add_cloud_device(src.data_ptr(), len(pb.source), ptr, n_t, pb.init_pose)
        icp.set_initial_mean(pb.R0, pb.t0)
        assert icp.stein_align() == sv.ALIGN_SUCCESS
        out.append(icp.get_particles())
    np.testing.assert_array_equal(out[0], out[1])


def test_device_paths_equal_host_paths():
    import torch
    a, t = drive_map()
    s = a.Export()
    V, N = a.Size(), a.PointCount()
    vox = torch.zeros((V, 3), dtype=torch.int32, device="cuda")
    cnt = torch.zeros(V, dtype=torch.int32, device="cuda")
    xyz = torch.zeros((N, 3), dtype=torch.float32, device="cuda")
    a.ExportDevice(vox.data_ptr(), cnt.data_ptr(), xyz.data_ptr())
    assert vox.cpu().numpy().tobytes() == s.voxels.tobytes()
    assert cnt.cpu().numpy().tobytes() == s.counts.tobytes()
    assert xyz.cpu().numpy().tobytes() == s.points.tobytes()
    b = sv.VoxelHashMap(1.0, 40.0, 20)
    b.ImportDevice(vox.data_ptr(), cnt.data_ptr(), xyz.data_ptr(), V, N)
    assert_same_map(a, b, t)


# ---- errors leave the map untouched ------------------------------------------------------------------------------------------
def raw_import(m, vox, cnt, pts, V=None, N=None):
    """svnicp_map_import on host arrays, sizes overridable; -> (rc, last error)"""
    p = lambda x: x.ctypes.data_as(C.c_void_p) if x is not None else None  # noqa: E731
    V = len(cnt) if V is None else V
    N = len(pts) if N is None else N
    rc = m._lib.svnicp_map_import(m._m, p(vox), p(cnt), p(pts), C.c_int64(V), C.c_int64(N), C.c_int(0))
    return rc, (m._lib.svnicp_map_last_error(m._m) or b"").decode()


def offsets(s):
    return np.concatenate([[0], np.cumsum(s.counts)])


def test_refused_imports_leave_the_map_unchanged():
    a, t = drive_map()
    s = a.Export()
    before = a.Export()
    size = (a.Size(), a.PointCount())
    V, N, cap = len(s.counts), len(s.points), 20
    off = offsets(s)
    bad_count_voxel = int(np.argmax(s.counts >= 2))

    def case(vox=None, cnt=None, pts=None, **kw):
        return (s.voxels.copy() if vox is None else vox, s.counts.copy() if cnt is None else cnt,
                s.points.copy() if pts is None else pts, kw)

    cases = []
    c = s.counts.copy(); c[9] = 0; c[40] = 0
    cases.append(("count 0", case(cnt=c), "voxel 9:"))
    c = s.counts.copy(); c[7] = cap + 1; c[30] = -3
    cases.append(("count above cap", case(cnt=c), "voxel 7:"))
    v = s.voxels.copy(); v[11, 1] = 1 << 20; v[50, 0] = -(1 << 20) - 1
    cases.append(("index range", case(vox=v), "voxel 11:"))
    v = s.voxels.copy(); v[12] = v[3]; v[60] = v[3]
    cases.append(("duplicate", case(vox=v), "voxel 12:"))
    v = s.voxels.copy(); v[5], v[6] = s.voxels[6], s.voxels[5]  # swapped voxels: both hold points that are not theirs
    cases.append(("membership", case(vox=v), "voxel 5:"))
    p = s.points.copy(); p[off[8] + int(s.counts[8]) - 1, 2] += 2.5; p[off[90], 0] -= 3.0  # the last point of voxel 8 moves
    cases.append(("membership last point", case(pts=p), "voxel 8:"))
    c = s.counts.copy(); c[bad_count_voxel] -= 1
    cases.append(("sum of counts", case(cnt=c), "counts sum to"))
    cases.append(("n_points too small", case(N=N - 1), "counts sum to"))
    cases.append(("n_points above V * cap", case(N=V * cap + 1), "exceeds"))
    cases.append(("negative n_voxels", case(V=-1), "negative"))
    cases.append(("null voxels", (None, s.counts.copy(), s.points.copy(), {}), "null"))
    invalid = -1  # SVNICP_ERR_INVALID
    for name, (vox, cnt, pts, kw), msg in cases:
        rc, err = raw_import(a, vox, cnt, pts, **kw)
        assert rc == invalid, (name, rc)
        assert msg in err, (name, err)
        snapshots_equal(a.Export(), before)
        assert (a.Size(), a.PointCount()) == size, name
    # a table too small is SVNICP_ERR_OOM, not SVNICP_ERR_INVALID
    small = sv.VoxelHashMap(1.0, 40.0, 20, capacity_voxels=256)
    small.AddPointCloud(np.array([[0.5, 0.5, 0.5], [3.5, 0.5, 0.5]], dtype=np.float32), np.eye(3), np.zeros(3))
    small_before = small.Export()
    assert V > 512
    rc, err = raw_import(small, s.voxels, s.counts, s.points)
    assert rc != invalid and rc != 0 and "capacity_voxels" in err
    with pytest.raises(sv.SvnIcpError, match="capacity_voxels"):
        small.Import(s)
    snapshots_equal(small.Export(), small_before)
    assert (small.Size(), small.PointCount()) == (2, 2)
    np.testing.assert_array_equal(sort_rows(small.GetMap()), [[0.5, 0.5, 0.5], [3.5, 0.5, 0.5]])
    # the refused imports left a usable map: a restore of it is the same map
    b = sv.VoxelHashMap(1.0, 40.0, 20)
    b.Import(a.Export())
    assert_same_map(a, b, t)


def test_export_size_mismatch_and_parameter_mismatch():
    a, _ = drive_map()
    before = a.Export()
    V, N = a.Size(), a.PointCount()
    vox, cnt, pts = np.zeros((V + 1, 3), np.int32), np.zeros(V + 1, np.int32), np.zeros((N + 1, 3), np.float32)
    p = lambda x: x.ctypes.data_as(C.c_void_p)  # noqa: E731
    for v, n in ((V + 1, N), (V, N + 1), (V - 1, N), (V, N - 1)):
        rc = a._lib.svnicp_map_export(a._m, p(vox), p(cnt), p(pts), C.c_int64(v), C.c_int64(n), C.c_int(0))
        assert rc != 0 and "the map holds" in a._lib.svnicp_map_last_error(a._m).decode()
    snapshots_equal(a.Export(), before)
    # a 1 m snapshot into a 0.5 m map: the Python mirror refuses the parameters, the ABI finds points outside their voxels
    half = sv.VoxelHashMap(0.5, 40.0, 20)
    with pytest.raises(sv.SvnIcpError, match="voxel_size"):
        half.Import(before)
    rc, err = raw_import(half, before.voxels, before.counts, before.points)
    assert rc != 0 and "does not belong" in err
    assert half.Empty()


def test_empty_snapshot_round_trips_and_clears():
    a, _ = drive_map()
    e = sv.VoxelHashMap(1.0, 40.0, 20).Export()
    assert len(e.counts) == 0 and e.points.shape == (0, 3)
    a.Import(e)
    assert a.Empty() and a.PointCount() == 0 and len(a.GetMap()) == 0
    snapshots_equal(a.Export(), e)
    pts, R, t = next(scans([0]))
    a.AddPointCloud(pts, R, t)  # usable again
    b = sv.VoxelHashMap(1.0, 40.0, 20)
    b.AddPointCloud(pts, R, t)
    snapshots_equal(a.Export(), b.Export())


def test_save_load(tmp_path):
    a, t = drive_map()
    path = str(tmp_path / "map.svnmap")
    a.Save(path)
    b = sv.VoxelHashMap.Load(path, capacity_voxels=16)
    assert (b.voxel_size_, b.max_range_, b.max_pointscount_) == (1.0, 40.0, 20)
    assert_same_map(a, b, t)
    snapshots_equal(sv.read_map_snapshot(path), a.Export())
    b.Save(str(tmp_path / "again.svnmap"))
    assert open(path, "rb").read() == open(str(tmp_path / "again.svnmap"), "rb").read()
