"""svnicp_evaluate: fitness, inlier RMSE and the Gauss-Newton system of the last scan's candidate table at caller-given poses.

Checked against the scan's own iteration-0 taps (same transforms -> same correspondences, bit for bit), the fp64 oracle on the
evaluation's own correspondences, the fp64 reference semantics, and for the absence of side effects on the handle.
Run directly under torch.distributed.run, this file is also the worker of the 2-GPU case."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import svn_icp_b200 as sv  # noqa: E402
from svn_icp_b200 import synth  # noqa: E402

pytestmark = pytest.mark.gpu

POSE_TOL = 1e-5


@pytest.fixture(scope="module")
def small():
    return synth.make_uniform_problem(40, 1500, 20000, seed=5)


@pytest.fixture(scope="module")
def lidar():
    return synth.make_problem(64, sensor="32", scan_index=6, n_map_scans=6, seed=0xC0FFEE)


def scanned(pb, init, cls="svn", **kw):
    prm = dict(iterations=1, KNN_count=100, max_dist=3.0)
    prm.update(kw)
    if cls == "svn":
        icp = sv.SVNICP(sv.SteinICPParam(**prm), init)
    else:
        prm.setdefault("lr", 0.03)
        icp = sv.SVGDICP(sv.SteinICPParam(optimizer="Adam", **prm), init)
    icp.add_cloud(pb.source, pb.target, init)
    icp.set_initial_mean(pb.R0, pb.t0)
    assert icp.stein_align() == sv.ALIGN_SUCCESS
    return icp


def pose_Rt(oracle, poses, cls="svn"):
    """[6, M] poses of the class convention -> R [M, 3, 3], t [M, 3] (fp64, as the handle's particle state)."""
    M = poses.shape[1]
    if cls == "svn":
        R = np.stack([oracle.so3_exp(poses[3:, m])[0] for m in range(M)])
    else:
        R = np.stack([oracle.euler_R(*poses[3:, m]) for m in range(M)])
    return R, np.ascontiguousarray(poses[:3].T)


def check_system(H, b, cH, cb, pb):
    """the bars of test_gpu_parity.py::test_gauss_newton_system (fp32 accumulation vs fp64)"""
    for blk in (slice(0, 3), slice(3, 6)):
        for blk2 in (slice(0, 3), slice(3, 6)):
            scale = np.abs(cH[:, blk, blk2]).max()
            np.testing.assert_allclose(H[:, blk, blk2], cH[:, blk, blk2], rtol=0, atol=1e-6 * scale)
    n_s = len(pb.source)
    rng_s = np.linalg.norm(pb.source, axis=1).mean()
    np.testing.assert_allclose(b[:, :3], cb[:, :3], rtol=0, atol=1e-6 * n_s * 0.3)
    np.testing.assert_allclose(b[:, 3:], cb[:, 3:], rtol=0, atol=1e-6 * n_s * 0.3 * rng_s)


def fp64_rmse(R, t, pb, idx, mask):
    """inlier RMSE from the fp64 distances of the chosen pairs: q = R0 (R s + t) + t0 against the map point"""
    out = []
    for m in range(len(R)):
        q = (pb.source @ R[m].T + t[m]) @ np.asarray(pb.R0).T + pb.t0
        d2 = ((q - pb.target[idx[m]]) ** 2).sum(axis=1)
        sel = mask[m].astype(bool)
        out.append(np.sqrt(d2[sel].mean()) if sel.any() else 0.0)
    return np.array(out)


@pytest.mark.parametrize("P", [7, 64, 300])
def test_iteration0_identity_svn(oracle, lidar, P):
    """evaluate(init_pose) runs iteration 0's transforms: the same correspondences as the scan's own taps, bit for bit, and
    the same Gauss-Newton system up to the order of the fp32 sums."""
    init = synth.init_particles(P, np.random.default_rng(P))
    icp = scanned(lidar, init, debug_corr=True)
    ev = icp.evaluate(init, want_mask=True, want_idx=True)
    _, idx, mask = icp.get_correspondences()
    np.testing.assert_array_equal(ev["idx"], idx)
    np.testing.assert_array_equal(ev["mask"], mask)
    np.testing.assert_array_equal(ev["inliers"], mask.sum(axis=1))
    np.testing.assert_array_equal(ev["fitness"], mask.sum(axis=1) / len(lidar.source))
    H, b, _ = icp.get_gn_system()
    check_system(ev["H"], ev["b"], H, b, lidar)


def test_iteration0_identity_svgd(oracle, lidar):
    """SVGD-ICP class: Euler poses; idx / mask equal the class's own iteration-0 taps, H and b match the oracle (its records
    carry the first-order sums only)."""
    P = 24
    rng = np.random.default_rng(3)
    init = synth.init_particles(P, rng)
    icp = scanned(lidar, init, cls="svgd", debug_corr=True)
    ev = icp.evaluate(init, want_mask=True, want_idx=True)
    _, idx, mask = icp.get_correspondences()
    np.testing.assert_array_equal(ev["idx"], idx)
    np.testing.assert_array_equal(ev["mask"], mask)
    R, t = pose_Rt(oracle, init, "svgd")
    cH, cb = oracle.gn_given_corr(R, t, lidar.R0, lidar.t0, lidar.source, lidar.target, ev["idx"], ev["mask"], 3.0)
    check_system(ev["H"], ev["b"], cH, cb, lidar)


@pytest.mark.parametrize("which,M", [("small", 1), ("small", 5), ("lidar", 33), ("lidar", 70)])
def test_against_oracle(oracle, request, which, M):
    """Poses away from the particles (the scan's result, zeros, perturbed hypotheses), several pose blocks: the system on the
    evaluation's own correspondences, the count, the RMSE, and the reference semantics in fp64."""
    pb = request.getfixturevalue(which)
    icp = scanned(pb, pb.init_pose[:, :16], iterations=3, lr=1.0, debug_corr=True)
    rng = np.random.default_rng(M)
    poses = np.concatenate([icp.get_transformation()[:, None], np.zeros((6, 1)), synth.init_particles(max(M - 2, 1), rng)], axis=1)[:, :M]
    ev = icp.evaluate(poses, want_mask=True, want_idx=True)
    R, t = pose_Rt(oracle, poses)
    cH, cb = oracle.gn_given_corr(R, t, pb.R0, pb.t0, pb.source, pb.target, ev["idx"], ev["mask"], 3.0)
    check_system(ev["H"], ev["b"], cH, cb, pb)
    np.testing.assert_array_equal(ev["inliers"], ev["mask"].sum(axis=1))
    np.testing.assert_allclose(ev["rmse"], fp64_rmse(R, t, pb, ev["idx"], ev["mask"]), rtol=1e-5, atol=0)
    # reference semantics (fp64 correspondences over the MinK table)
    q0 = oracle.transform_q0(pb.source, pb.R0, pb.t0)
    mink, _ = oracle.knn_mink(q0, pb.target, 100)
    oH, ob, ridx, _ = oracle.gn(R, t, pb.R0, pb.t0, pb.source, pb.target, mink, 3.0, want_corr=True)
    assert np.mean(ridx != ev["idx"]) < 1e-4
    g = np.linalg.solve(ev["H"], ev["b"][..., None])[..., 0]
    og = np.linalg.solve(oH, ob[..., None])[..., 0]
    np.testing.assert_allclose(g, og, rtol=0, atol=POSE_TOL)
    # the (6,) form is the M = 1 case
    one = icp.evaluate(poses[:, 0], want_mask=True)
    assert one["H"].shape == (6, 6) and one["mask"].shape == (len(pb.source),)


def test_full_size_scan(oracle):
    """configs[1] size (64-beam scan, ~143 k points, K = 100), M = 1 at the result pose: oracle agreement, the same bits on a
    second call, and the registered pose fits better than the initial guess."""
    import bench
    W = bench.WORKLOAD
    P = 64
    pb, _ = bench.make_problem(P)
    icp = sv.SVNICP(sv.SteinICPParam(iterations=10, KNN_count=W["K"], max_dist=W["max_dist"], lr=W["lr"], SVN_full_grad=W["svn_full_grad"],
                                     debug_corr=True), pb.init_pose)
    icp.add_cloud(pb.source, pb.target, pb.init_pose)
    icp.set_initial_mean(pb.R0, pb.t0)
    assert icp.stein_align() == sv.ALIGN_SUCCESS
    x = icp.get_transformation()
    ev = icp.evaluate(x, want_mask=True, want_idx=True)
    again = icp.evaluate(x, want_mask=True, want_idx=True)
    for k in ev:
        np.testing.assert_array_equal(ev[k], again[k])
    R, t = pose_Rt(oracle, x[:, None])
    cH, cb = oracle.gn_given_corr(R, t, pb.R0, pb.t0, pb.source, pb.target, ev["idx"][None], ev["mask"][None], W["max_dist"])
    check_system(ev["H"][None], ev["b"][None], cH, cb, pb)
    assert ev["inliers"] == ev["mask"].sum()
    np.testing.assert_allclose(ev["rmse"], fp64_rmse(R, t, pb, ev["idx"][None], ev["mask"][None])[0], rtol=1e-5, atol=0)
    zero = icp.evaluate(np.zeros(6))
    assert ev["fitness"] >= zero["fitness"] and ev["rmse"] < zero["rmse"]
    # max_dist = 3 (d < 1.73 m) keeps every point of this scan at both poses; a tight gate separates them
    icp.set_threshold(0.01)
    tight, tight0 = icp.evaluate(x), icp.evaluate(np.zeros(6))
    assert tight["fitness"] > tight0["fitness"] and tight["rmse"] < tight0["rmse"]
    print(f"full size: n_s={len(pb.source)}; max_dist 3: fitness {zero['fitness']:.4f} -> {ev['fitness']:.4f}, rmse {zero['rmse']:.4f} -> "
          f"{ev['rmse']:.4f} m; max_dist 0.01: fitness {tight0['fitness']:.4f} -> {tight['fitness']:.4f}, rmse {tight0['rmse']:.4f} -> "
          f"{tight['rmse']:.4f} m")


def snapshot(icp):
    H, b, x = icp.get_gn_system()
    xf, idx, mask = icp.get_correspondences()
    d, h = icp.get_stein()
    return [icp.get_transformation(), icp.get_distribution(), icp.get_cov_matrix(), icp.get_particles(), icp.get_particle_weight(),
            icp.get_particle_history(), H, b, x, xf, idx, mask, d, np.array([h]), icp.get_prune_stats(),
            np.array(list(icp.get_timing().values())), np.array([icp.launch_count(), icp.iterations_done()])]


@pytest.mark.parametrize("cls", ["svn", "svgd"])
def test_no_side_effects(small, cls):
    """Every getter (timing and launch count included) returns the same bits after evaluate, and a following stein_align
    without add_cloud gives the same bits as on a twin handle that never evaluated."""
    kw = dict(iterations=4, KNN_count=40, lr=1.0 if cls == "svn" else 0.03, debug_corr=True)
    a, b = scanned(small, small.init_pose, cls, **kw), scanned(small, small.init_pose, cls, **kw)
    before = snapshot(a)
    a.evaluate(synth.init_particles(40, np.random.default_rng(1)), want_mask=True, want_idx=True)
    a.evaluate(np.zeros(6), want_system=False)
    for u, v in zip(before, snapshot(a)):
        np.testing.assert_array_equal(u, v)
    assert a.stein_align() == b.stein_align() == sv.ALIGN_SUCCESS
    for u, v in zip(snapshot(a)[:15], snapshot(b)[:15]):  # timing differs between handles
        np.testing.assert_array_equal(u, v)


def test_batch_stream_equals_single_handle(small, lidar):
    """evaluate on SVNICPBatch.stream(s) == evaluate on an ordinary handle with the same inputs."""
    prm = sv.SteinICPParam(iterations=5, KNN_count=64, max_dist=3.0, lr=1.0)
    P = 16
    inits = np.stack([synth.init_particles(P, np.random.default_rng(s)) for s in range(2)])
    batch = sv.SVNICPBatch(prm, inits)
    for s, pb in enumerate((small, lidar)):
        batch.streams[s].add_cloud(pb.source, pb.target, inits[s])
        batch.streams[s].set_initial_mean(pb.R0, pb.t0)
    assert batch.stein_align() == [sv.ALIGN_SUCCESS] * 2
    poses = synth.init_particles(9, np.random.default_rng(7))
    for s, pb in enumerate((small, lidar)):
        single = sv.SVNICP(prm, inits[s])
        single.add_cloud(pb.source, pb.target, inits[s])
        single.set_initial_mean(pb.R0, pb.t0)
        assert single.stein_align() == sv.ALIGN_SUCCESS
        np.testing.assert_array_equal(batch.streams[s].get_particles(), single.get_particles())
        e1 = batch.streams[s].evaluate(poses, want_mask=True)
        e2 = single.evaluate(poses, want_mask=True)
        for k in e1:
            np.testing.assert_array_equal(e1[k], e2[k])
    batch.close()


def test_errors(small):
    init = small.init_pose[:, :8]
    icp = sv.SVNICP(sv.SteinICPParam(iterations=2, KNN_count=20, max_dist=3.0), init)
    with pytest.raises(sv.SvnIcpError, match="candidate table"):
        icp.evaluate(np.zeros(6))  # no add_cloud yet
    icp.add_cloud(small.source, small.target, init)
    icp.set_initial_mean(small.R0, small.t0)
    with pytest.raises(sv.SvnIcpError, match="candidate table"):
        icp.evaluate(np.zeros(6))  # add_cloud, no stein_align yet
    assert icp.stein_align() == sv.ALIGN_SUCCESS
    icp.evaluate(np.zeros(6))
    with pytest.raises(sv.SvnIcpError, match="n_poses"):
        icp.evaluate(np.zeros((6, 0)))
    with pytest.raises(sv.SvnIcpError, match="debug_corr"):
        icp.evaluate(np.zeros(6), want_idx=True)
    # NaN poses: no fault, no inliers, the handle stays usable
    nan = icp.evaluate(np.full((6, 3), np.nan), want_mask=True)
    assert (nan["inliers"] == 0).all() and nan["mask"].sum() == 0
    ok = icp.evaluate(icp.get_transformation())
    assert ok["inliers"] > 0 and np.isfinite(ok["H"]).all()
    icp.set_threshold(1.5)  # the current threshold applies: fewer inliers, table still valid
    assert icp.evaluate(icp.get_transformation())["inliers"] <= ok["inliers"]
    icp.set_k(10)
    with pytest.raises(sv.SvnIcpError, match="candidate table"):
        icp.evaluate(np.zeros(6))
    assert icp.stein_align() == sv.ALIGN_SUCCESS
    icp.evaluate(np.zeros(6))
    icp.set_initial_mean(small.R0, small.t0 + 0.1)
    with pytest.raises(sv.SvnIcpError, match="candidate table"):
        icp.evaluate(np.zeros(6))
    icp.add_cloud(small.source, small.target, init)
    with pytest.raises(sv.SvnIcpError, match="candidate table"):
        icp.evaluate(np.zeros(6))


def test_sharded_same_result_on_every_rank():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29533", os.path.abspath(__file__)]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    sys.stdout.write(r.stdout[-4000:])
    sys.stderr.write(r.stderr[-4000:])
    assert r.returncode == 0


def _sharded_worker():
    """2 ranks: a particle-sharded scan, then evaluate on every rank -- identical bits everywhere, and equal to a single-GPU
    handle that evaluates the same poses on the same (bit-identical, all-gathered) candidate table."""
    import torch
    import torch.distributed as dist
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    pb = synth.make_problem(96, sensor="32", scan_index=6, n_map_scans=6, seed=0xC0FFEE)
    prm = sv.SteinICPParam(iterations=6, KNN_count=64, max_dist=3.0, lr=1.0, debug_corr=True)
    icp = sv.SVNICP(prm, pb.init_pose, device=local)
    uid = [sv.nccl_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    icp.init_sharding(uid[0], rank, world)
    icp.add_cloud(pb.source, pb.target, pb.init_pose)
    icp.set_initial_mean(pb.R0, pb.t0)
    assert icp.stein_align() == sv.ALIGN_SUCCESS
    poses = np.concatenate([np.zeros((6, 1)), synth.init_particles(40, np.random.default_rng(5))], axis=1)
    ev = icp.evaluate(poses, want_mask=True, want_idx=True)
    flat = np.concatenate([ev["inliers"].astype(np.float64), ev["fitness"], ev["rmse"], ev["H"].ravel(), ev["b"].ravel(),
                           ev["mask"].ravel().astype(np.float64), ev["idx"].ravel().astype(np.float64)])
    t = torch.from_numpy(flat).cuda()
    ref = t.clone()
    dist.broadcast(ref, src=0)
    ok = bool(torch.equal(t, ref))
    if rank == 0:
        single = sv.SVNICP(sv.SteinICPParam(iterations=0, KNN_count=64, max_dist=3.0, debug_corr=True), pb.init_pose, device=local)
        single.add_cloud(pb.source, pb.target, pb.init_pose)
        single.set_initial_mean(pb.R0, pb.t0)
        single.stein_align()
        es = single.evaluate(poses, want_mask=True, want_idx=True)
        same_single = all(np.array_equal(ev[k], es[k]) for k in ("inliers", "mask", "idx"))
        same_single &= all(np.allclose(ev[k], es[k], rtol=1e-12, atol=0) for k in ("fitness", "rmse", "H", "b"))
        print(f"sharded evaluate: same on all ranks {ok}, equal to single GPU {same_single}", flush=True)
        ok &= same_single
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    ok = bool(flag.item())
    icp.close()
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    _sharded_worker()
