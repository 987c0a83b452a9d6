"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle and the committed golden vectors.

Bars (BASELINE.json north_star):
  * correspondence indices bit-exact given identical transformed points and the documented tie-break;
  * per-particle poses, particle mean and covariance within POSE_TOL = 1e-5 (m / rad) of the fp64 reference.
"""
import numpy as np
import pytest

import oracle as orc
import svn_icp_b200 as sv
from svn_icp_b200 import synth
from conftest import golden_names, load_golden

pytestmark = pytest.mark.gpu

POSE_TOL = 1e-5  # metres / radians, stated tolerance for poses, mean and (sqrt of) covariance entries


def make_icp(pb, **kw):
    prm = sv.SteinICPParam(**kw)
    icp = sv.SVNICP(prm, pb.init_pose, sv.ParticleWeightOpt())
    icp.add_cloud(pb.source, pb.target, pb.init_pose)
    icp.set_initial_mean(pb.R0, pb.t0)
    return icp


def initial_state(oracle, init_pose):
    P = init_pose.shape[1]
    R = np.stack([oracle.so3_exp(init_pose[3:, p])[0] for p in range(P)])
    t = np.ascontiguousarray(init_pose[:3].T)
    return R, t


@pytest.fixture(scope="module")
def small():
    return synth.make_uniform_problem(40, 1500, 20000, seed=5)


@pytest.fixture(scope="module")
def lidar():
    # 32-beam x 900 column synthetic scan against a 6-scan voxel map: realistic density, oracle-sized
    return synth.make_problem(64, sensor="32", scan_index=6, n_map_scans=6, seed=0xC0FFEE)


@pytest.mark.parametrize("which,K", [("small", 20), ("small", 100), ("lidar", 100), ("lidar", 33), ("lidar", 256), ("small", 1)])
def test_candidate_table_exact(oracle, request, which, K):
    """Per-scan K-NN: same K-nearest SET as the reference's brute force (MinK), emitted ascending (d0^2, index)."""
    pb = request.getfixturevalue(which)
    icp = make_icp(pb, iterations=0, KNN_count=K, max_dist=3.0, debug_corr=True)
    assert icp.stein_align() == sv.ALIGN_SUCCESS
    idx, rel = icp.get_candidates(want_rel=True)
    q0 = oracle.transform_q0(pb.source, pb.R0, pb.t0)
    oidx, orel = oracle.cand_sorted(q0, pb.target, K)
    np.testing.assert_array_equal(idx, oidx)
    np.testing.assert_array_equal(rel, orel)
    np.testing.assert_array_equal(icp.get_source_f32(), oracle.source_f32(pb.source, pb.R0))
    # same set as the reference's MinK table (slot order differs by design)
    mink, _ = oracle.knn_mink(q0[:300], pb.target, K)
    np.testing.assert_array_equal(np.sort(mink, axis=1), np.sort(idx[:300].astype(np.int64), axis=1))


def test_candidate_table_tiny_map(oracle):
    """N_t < K: the reference zero-pads (knn.cu:343) -> padded slots point at map point 0."""
    pb = synth.make_uniform_problem(5, 60, 60, seed=16, box=8.0)
    pb.target = pb.target[:10].copy()
    icp = make_icp(pb, iterations=0, KNN_count=16, debug_corr=True)
    icp.stein_align()
    idx = icp.get_candidates()
    q0 = oracle.transform_q0(pb.source, pb.R0, pb.t0)
    oidx, _ = oracle.cand_sorted(q0, pb.target, 16)
    np.testing.assert_array_equal(idx, oidx)
    assert np.all(idx[:, 10:] == 0)


@pytest.mark.parametrize("which", ["small", "lidar", "lidar_p30"])
def test_correspondence_indices_bit_exact(oracle, request, which):
    """Indices chosen by the fused kernel == oracle restatement of the same fp32 arithmetic on the same inputs; the
    exact pruning pass must not change a single index.  lidar_p30: 30 particles (the reference's shipped regime), k_gn without
    the warp-uniform early exit (fewer than 32 particle pairs per row group)."""
    pb = request.getfixturevalue(which.split("_")[0])
    init = pb.init_pose[:, :30] if which.endswith("_p30") else pb.init_pose
    icp = sv.SVNICP(sv.SteinICPParam(iterations=1, KNN_count=100, max_dist=3.0, debug_corr=True), init)
    icp.add_cloud(pb.source, pb.target, init)
    icp.set_initial_mean(pb.R0, pb.t0)
    icp.stein_align()
    xf, idx, mask = icp.get_correspondences()
    cidx, rel = icp.get_candidates(want_rel=True)
    sp = icp.get_source_f32()
    oidx, omask = oracle.corr_f32(xf, sp, rel, cidx, 3.0)
    np.testing.assert_array_equal(idx, oidx)
    np.testing.assert_array_equal(mask, omask)
    # transforms from the fp64 state
    R, t = initial_state(oracle, init)
    np.testing.assert_allclose(xf, oracle.transforms_f32(R, t, pb.R0), rtol=0, atol=2e-7)
    # against the reference semantics in fp64 (different arithmetic): only near-ties may differ
    q0 = oracle.transform_q0(pb.source, pb.R0, pb.t0)
    mink, _ = oracle.knn_mink(q0, pb.target, 100)
    _, _, ridx, rmask = oracle.gn(R, t, pb.R0, pb.t0, pb.source, pb.target, mink, 3.0, want_corr=True)
    assert np.mean(ridx != idx) < 1e-4
    assert np.mean(rmask != mask) < 1e-4


@pytest.mark.parametrize("which,P", [("small", 40), ("lidar", 64), ("lidar", 7), ("lidar", 300)])
def test_gauss_newton_system(oracle, request, which, P):
    """H (6x6) and b (6) per particle against the fp64 oracle (Newton_grad_right, SVNICP.cpp:116-164).
    (1) arithmetic: same correspondences -> H, b agree to fp32-accumulation accuracy;
    (2) end to end vs the reference semantics (fp64 correspondences): the Newton step agrees within POSE_TOL even
        though a few near-tie correspondences (< 1e-4 of the pairs) differ between fp32 and fp64 geometry."""
    pb = request.getfixturevalue(which)
    rng = np.random.default_rng(P)
    init = synth.init_particles(P, rng)
    icp = sv.SVNICP(sv.SteinICPParam(iterations=1, KNN_count=100, max_dist=3.0, debug_corr=True), init)
    icp.add_cloud(pb.source, pb.target, init)
    icp.set_initial_mean(pb.R0, pb.t0)
    icp.stein_align()
    H, b, x = icp.get_gn_system()
    _, idx, mask = icp.get_correspondences()
    R, t = initial_state(oracle, init)
    np.testing.assert_allclose(x[:, :3], t, rtol=0, atol=1e-15)
    # (1) same correspondences
    cH, cb = oracle.gn_given_corr(R, t, pb.R0, pb.t0, pb.source, pb.target, idx, mask, 3.0)
    for blk in (slice(0, 3), slice(3, 6)):
        for blk2 in (slice(0, 3), slice(3, 6)):
            scale = np.abs(cH[:, blk, blk2]).max()
            np.testing.assert_allclose(H[:, blk, blk2], cH[:, blk, blk2], rtol=0, atol=1e-6 * scale)
    # b is a sum of signed terms: scale by the sum of magnitudes (~ n_s * |e| and n_s * |s| * |e|)
    n_s = len(pb.source)
    rng_s = np.linalg.norm(pb.source, axis=1).mean()
    np.testing.assert_allclose(b[:, :3], cb[:, :3], rtol=0, atol=1e-6 * n_s * 0.3)
    np.testing.assert_allclose(b[:, 3:], cb[:, 3:], rtol=0, atol=1e-6 * n_s * 0.3 * rng_s)
    g = np.linalg.solve(H, b[..., None])[..., 0]
    cg = np.linalg.solve(cH, cb[..., None])[..., 0]
    np.testing.assert_allclose(g, cg, rtol=0, atol=1e-7)
    # (2) reference semantics
    q0 = oracle.transform_q0(pb.source, pb.R0, pb.t0)
    mink, _ = oracle.knn_mink(q0, pb.target, 100)
    oH, ob, ridx, rmask = oracle.gn(R, t, pb.R0, pb.t0, pb.source, pb.target, mink, 3.0, want_corr=True)
    assert np.mean(ridx != idx) < 1e-4
    og = np.linalg.solve(oH, ob[..., None])[..., 0]
    np.testing.assert_allclose(g, og, rtol=0, atol=POSE_TOL)


@pytest.mark.parametrize("full", [True, False])
@pytest.mark.parametrize("P", [3, 64, 513])
def test_stein_step(oracle, lidar, full, P):
    """Kernel (c): bandwidth (exact lower median of P^2 distances) and the update delta, fp64 vs oracle on the GPU's own H,b,x."""
    rng = np.random.default_rng(100 + P)
    init = synth.init_particles(P, rng)
    icp = sv.SVNICP(sv.SteinICPParam(iterations=1, KNN_count=50, max_dist=3.0, SVN_full_grad=full, lr=0.7), init)
    icp.add_cloud(lidar.source[::4], lidar.target, init)
    icp.set_initial_mean(lidar.R0, lidar.t0)
    icp.stein_align()
    H, b, x = icp.get_gn_system()
    delta, h = icp.get_stein()
    od, oh = oracle.stein_step(x, H, b, full=full, lr=0.7)
    assert h == pytest.approx(oh, rel=1e-13)
    np.testing.assert_allclose(delta, od, rtol=1e-8, atol=1e-12)
    # pose update (SVNICP.cpp:268-279) applied to the initial state
    R, t = initial_state(oracle, init)
    R2, t2 = oracle.pose_update(R, t, od)
    want = np.concatenate([t2, np.stack([oracle.so3_log(r) for r in R2])], axis=1)  # [P,6]
    got = icp.get_particles().reshape(6, P).T
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-10)


@pytest.mark.parametrize("full", [True, False])
def test_full_scan_vs_oracle(oracle, lidar, full):
    """Whole scan, 12 iterations: poses, mean, variance, covariance, history within the stated tolerance."""
    icp = make_icp(lidar, iterations=12, KNN_count=100, max_dist=3.0, lr=1.0, SVN_full_grad=full)
    assert icp.stein_align() == sv.ALIGN_SUCCESS
    prm = orc.make_params(iterations=12, knn_count=100, max_dist=3.0, lr=1.0, svn_full_grad=full)
    o = oracle.align(prm, lidar.source, lidar.target, lidar.init_pose, lidar.R0, lidar.t0)
    P = lidar.init_pose.shape[1]
    # POSE_TOL is a PER-ITERATION bound (north_star; checked with identical inputs by test_gauss_newton_system and
    # test_stein_step).  Over a whole scan the few fp32-vs-fp64 near-tie correspondences compound through the
    # (non-contractive, repulsive) particle dynamics: individual particles get SCAN_TOL, the mean keeps POSE_TOL.
    SCAN_TOL = 5 * POSE_TOL
    np.testing.assert_allclose(icp.get_particles().reshape(6, P), o["particles"], rtol=0, atol=SCAN_TOL)
    hist = icp.get_particle_history().reshape(12, 6, P)
    np.testing.assert_allclose(hist[0], o["history"][0], rtol=0, atol=POSE_TOL)  # first iteration: identical inputs
    np.testing.assert_allclose(icp.get_transformation(), o["mean"], rtol=0, atol=POSE_TOL)
    np.testing.assert_allclose(np.sqrt(icp.get_distribution()), np.sqrt(o["var"]), rtol=0, atol=POSE_TOL)
    # |d cov_ij| <= (sigma_i + sigma_j) * tol + tol^2 when every pose moves by at most tol
    sig = np.sqrt(np.diag(o["cov"]))
    np.testing.assert_allclose(icp.get_cov_matrix().reshape(6, 6), o["cov"], rtol=0,
                               atol=float((2 * sig.max()) * POSE_TOL + POSE_TOL ** 2))
    np.testing.assert_array_equal(icp.get_particle_weight(), o["weights"])
    np.testing.assert_allclose(icp.get_particle_history().reshape(12, 6, P), o["history"], rtol=0, atol=SCAN_TOL)
    assert icp.iterations_done() == 12
    # and the scan actually registers: mean close to the planted relative motion
    assert np.abs(icp.get_transformation() - lidar.gt_rel)[:3].max() < 0.05
    assert np.abs(icp.get_transformation() - lidar.gt_rel)[3:].max() < 0.005


@pytest.mark.parametrize("K", [1, 7, 256])
def test_scan_extreme_candidate_counts(oracle, small, K):
    """KNN_count at the edges of the supported range (1 = plain nearest point of the initial guess, 256 = the ABI maximum,
    7 = not a multiple of 4: padded list rows)."""
    rng = np.random.default_rng(K)
    P = 16
    init = synth.init_particles(P, rng)
    icp = sv.SVNICP(sv.SteinICPParam(iterations=4, KNN_count=K, max_dist=3.0, lr=1.0), init)
    icp.add_cloud(small.source, small.target, init)
    icp.set_initial_mean(small.R0, small.t0)
    assert icp.stein_align() == sv.ALIGN_SUCCESS
    prm = orc.make_params(iterations=4, knn_count=K, max_dist=3.0, lr=1.0)
    o = oracle.align(prm, small.source, small.target, init, small.R0, small.t0)
    np.testing.assert_allclose(icp.get_particles().reshape(6, P), o["particles"], rtol=0, atol=5 * POSE_TOL)
    np.testing.assert_allclose(icp.get_transformation(), o["mean"], rtol=0, atol=POSE_TOL)


@pytest.mark.parametrize("name", golden_names())
def test_golden_vectors_through_c_abi(name):
    """The committed outputs of the reference's own sources (tests/golden/*.npz)."""
    g = load_golden(name)
    I, lr, md, es, thr, K, full = g["params"]
    prm = sv.SteinICPParam(iterations=int(I), lr=float(lr), max_dist=float(md), check_early_stop=bool(es),
                           convergence_threshold=float(thr), KNN_count=int(K), SVN_full_grad=bool(full))
    P = g["init_pose"].shape[1]
    icp = sv.SVNICP(prm, g["init_pose"])
    icp.add_cloud(g["source"], g["target"], g["init_pose"])
    icp.set_initial_mean(g["R0"], g["t0"])
    assert icp.stein_align() == int(g["ref_state"][0])
    got = icp.get_particles().reshape(6, P)
    nan_ref = np.isnan(g["ref_particles"])
    np.testing.assert_array_equal(np.isnan(got), nan_ref)  # P == 2: bandwidth 0 -> NaN, reference behaviour
    np.testing.assert_allclose(got, g["ref_particles"], rtol=0, atol=POSE_TOL)
    np.testing.assert_allclose(icp.get_transformation(), g["ref_mean"], rtol=0, atol=POSE_TOL)
    sig = np.sqrt(np.nanmax(np.abs(np.diag(g["ref_cov"]))))
    np.testing.assert_allclose(icp.get_cov_matrix().reshape(6, 6), g["ref_cov"], rtol=0, atol=float(2 * sig * POSE_TOL + POSE_TOL ** 2))
    np.testing.assert_array_equal(icp.get_particle_weight(), g["ref_weights"])
    hist = icp.get_particle_history().reshape(int(I), 6, P)
    np.testing.assert_allclose(hist, g["ref_history"], rtol=0, atol=POSE_TOL)
    zero_rows = np.abs(g["ref_history"]).sum(axis=(1, 2)) == 0
    assert (np.abs(hist).sum(axis=(1, 2)) == 0).tolist() == zero_rows.tolist()  # rows after an early stop stay zero
    # break happens after the update of the stopping epoch and before its history row (SVNICP.cpp:92-107)
    assert icp.iterations_done() == (int((~zero_rows).sum()) + 1 if zero_rows.any() else int(I))


def test_single_particle_is_gauss_newton_icp(oracle, small):
    """P == 1: stein_grad = -H^-1 b (SVNICP.cpp:88-89); recovers the planted transform."""
    init = np.zeros((6, 1))
    icp = sv.SVNICP(sv.SteinICPParam(iterations=8, KNN_count=20, max_dist=3.0), init)
    icp.add_cloud(small.source, small.target, init)
    icp.set_initial_mean(small.R0, small.t0)
    icp.stein_align()
    prm = orc.make_params(iterations=8, knn_count=20, max_dist=3.0)
    o = oracle.align(prm, small.source, small.target, init, small.R0, small.t0)
    np.testing.assert_allclose(icp.get_transformation(), o["mean"], rtol=0, atol=POSE_TOL)
    np.testing.assert_allclose(icp.get_transformation(), small.gt_rel, rtol=0, atol=5e-3)


def test_deterministic_and_reusable(lidar):
    """One long-lived instance reused for several scans (OdometryPipeline.h:125); identical inputs -> identical bits."""
    icp = make_icp(lidar, iterations=6, KNN_count=100, max_dist=3.0, lr=1.0)
    icp.stein_align()
    a = icp.get_particles().copy()
    other = synth.make_uniform_problem(64, 700, 9000, seed=9)
    icp.add_cloud(other.source, other.target, other.init_pose)
    icp.set_initial_mean(other.R0, other.t0)
    icp.stein_align()
    assert np.abs(icp.get_transformation() - other.gt_rel).max() < 0.02
    icp.add_cloud(lidar.source, lidar.target, lidar.init_pose)
    icp.set_initial_mean(lidar.R0, lidar.t0)
    icp.stein_align()
    np.testing.assert_array_equal(icp.get_particles(), a)


def test_errors(small):
    with pytest.raises(sv.SvnIcpError):
        sv.SVNICP(sv.SteinICPParam(KNN_count=1000), np.zeros((6, 4)))
    icp = sv.SVNICP(sv.SteinICPParam(iterations=1), np.zeros((6, 4)))
    with pytest.raises(sv.SvnIcpError, match="before add_cloud"):
        icp.stein_align()
    with pytest.raises(sv.SvnIcpError, match="empty cloud"):
        icp.add_cloud(np.zeros((0, 3)), small.target, np.zeros((6, 4)))


@pytest.mark.parametrize("P,full,es", [(64, True, False), (64, False, False), (1, True, False), (200, True, True), (9, False, True),
                                       (300, True, False), (1200, False, False)])
def test_stein_phase_layouts_vs_oracle(oracle, lidar, P, full, es):
    """k_head + k_tail (tail2.cu) over the CTA layouts the particle count selects (8 warps per particle for small P ... one
    warp per particle for large P, both Stein modes, P == 1, early stop): the scan is deterministic (bit-identical when
    repeated) and follows the fp64 oracle iteration by iteration."""
    rng = np.random.default_rng(P)
    init = synth.init_particles(P, rng)
    src = lidar.source[::6]
    I = 6
    prm = dict(iterations=I, KNN_count=50, max_dist=3.0, lr=1.0, SVN_full_grad=full, check_early_stop=es, convergence_threshold=3e-3)
    runs = []
    for _ in range(2):
        icp = sv.SVNICP(sv.SteinICPParam(**prm), init)
        icp.add_cloud(src, lidar.target, init)
        icp.set_initial_mean(lidar.R0, lidar.t0)
        assert icp.stein_align() == sv.ALIGN_SUCCESS
        runs.append((icp.get_particles(), icp.get_particle_history(), icp.iterations_done(), icp.get_cov_matrix()))
    for k in range(4):
        np.testing.assert_array_equal(runs[0][k], runs[1][k])
    o = oracle.align(orc.make_params(iterations=I, knn_count=50, max_dist=3.0, lr=1.0, svn_full_grad=full, check_early_stop=es,
                                     convergence_threshold=3e-3), src, lidar.target, init, lidar.R0, lidar.t0)
    assert runs[0][2] == o["iters_done"]
    np.testing.assert_allclose(runs[0][0].reshape(6, -1), o["particles"], atol=2 * POSE_TOL, rtol=0)
    np.testing.assert_allclose(runs[0][1].reshape(I, 6, -1), o["history"], atol=2 * POSE_TOL, rtol=0)


def test_list_reuse_same_bits(lidar):
    """k_filter_reuse (pruning the previous iteration's lists once they are short) must choose exactly the same
    correspondences as pruning the full K-slot table every iteration (SVNICP_FLAG_FILTER_FULL): bit-identical poses."""
    res = {}
    for mode in ("reuse", "full"):
        flags = sv.FLAG_REUSE_STATS | (sv.FLAG_FILTER_FULL if mode == "full" else 0)
        icp = sv.SVNICP(sv.SteinICPParam(iterations=25, KNN_count=100, max_dist=3.0, lr=1.0, flags=flags), lidar.init_pose)
        icp.add_cloud(lidar.source, lidar.target, lidar.init_pose)
        icp.set_initial_mean(lidar.R0, lidar.t0)
        icp.stein_align()
        hits = icp.get_prune_stats()
        res[mode] = (icp.get_particles(), icp.get_particle_history(), hits)
    np.testing.assert_array_equal(res["reuse"][0], res["full"][0])
    np.testing.assert_array_equal(res["reuse"][1], res["full"][1])
    assert res["reuse"][2][-1] > 0.99 and res["full"][2].max() == 0.0  # the reuse path really ran in the late iterations


@pytest.mark.parametrize("cls,es", [("svn", False), ("svn", True), ("svgd", False)])
def test_align_twice_without_add_cloud(oracle, small, cls, es):
    """stein_align may be called again without add_cloud (the reference allows it: R_/t_ persist, history rows 0..I-1 are
    rewritten, SVGDICP rebuilds its optimizer, SVGDICP.cpp:73).  The second run must restart the iteration state -- no
    history row beyond I, no stale stop flag -- and equal one continuous oracle run from the poses of the first."""
    I = 5
    if cls == "svn":
        prm = sv.SteinICPParam(iterations=I, KNN_count=20, max_dist=3.0, lr=1.0, check_early_stop=es, convergence_threshold=1e-2 if es else 1e-5)
        icp = sv.SVNICP(prm, small.init_pose)
    else:
        prm = sv.SteinICPParam(iterations=I, KNN_count=20, max_dist=3.0, lr=0.01, optimizer="Adam")
        icp = sv.SVGDICP(prm, small.init_pose)
    icp.add_cloud(small.source, small.target, small.init_pose)
    icp.set_initial_mean(small.R0, small.t0)
    assert icp.stein_align() == sv.ALIGN_SUCCESS
    it1, p1, h1 = icp.iterations_done(), icp.get_particles().reshape(6, -1).copy(), icp.get_particle_history().copy()
    assert icp.stein_align() == sv.ALIGN_SUCCESS
    it2, p2, h2 = icp.iterations_done(), icp.get_particles().reshape(6, -1), icp.get_particle_history()
    assert h2.shape == h1.shape and 0 < it2 <= I
    if cls == "svn":
        # history row e = poses after update e (SVNICP.cpp:103-107): the last row written equals the final particles
        if not es:
            np.testing.assert_allclose(h1[-1].reshape(6, -1), p1, atol=1e-6, rtol=0)
        if es:
            assert np.abs(p2 - p1).max() > 0  # a stop flag left over from the first run must not turn the second into a no-op
        else:
            assert it1 == it2 == I
            # 2 x I iterations == one oracle run of 2 I iterations
            o = oracle.align(orc.make_params(iterations=2 * I, knn_count=20, max_dist=3.0, lr=1.0, svn_full_grad=True),
                             small.source, small.target, small.init_pose, small.R0, small.t0)
            np.testing.assert_allclose(p2, o["particles"], atol=5 * POSE_TOL, rtol=0)
    else:
        assert np.isfinite(p2).all() and np.abs(p2 - p1).max() > 0


@pytest.mark.parametrize("P,full,es,flags", [(30, False, True, sv.FLAG_FORCE_GRAPH), (100, True, False, 0), (65, True, True, sv.FLAG_FORCE_GRAPH),
                                             (300, True, False, sv.FLAG_FORCE_GRAPH), (40, True, False, sv.FLAG_FILTER_FULL)])
def test_graph_replay_equals_direct_launches(lidar, P, full, es, flags):
    """Small problems replay iterations >= 1 as CUDA graphs (capi.cu: align_step).  Same kernels, same arguments: the results
    must be bit-identical to the direct launches (SVNICP_FLAG_NO_GRAPH), also on the second scan of a handle (the graphs of
    the first scan are patched in place) and with another initial mean."""
    rng = np.random.default_rng(P)
    init = synth.init_particles(P, rng)
    src = lidar.source[::5]
    out = {}
    for name, fl in (("graph", flags), ("direct", flags | sv.FLAG_NO_GRAPH)):
        prm = sv.SteinICPParam(iterations=18, KNN_count=48, max_dist=3.0, lr=1.0, SVN_full_grad=full, check_early_stop=es,
                               convergence_threshold=2e-3, flags=fl)
        icp = sv.SVNICP(prm, init)
        res = []
        for k in range(3):
            icp.add_cloud(src[k::2], lidar.target, init)
            t0 = lidar.t0 + np.array([0.01 * k, -0.02 * k, 0.0])
            icp.set_initial_mean(lidar.R0, t0)
            assert icp.stein_align() == sv.ALIGN_SUCCESS
            res.append((icp.get_particles().copy(), icp.get_particle_history().copy(), icp.iterations_done(), icp.get_cov_matrix().copy(),
                        icp.launch_count()))
        out[name] = res
        icp.close()
    for g, d in zip(out["graph"], out["direct"]):
        assert g[2] == d[2]
        if not es:  # with early stop the number of no-op iterations enqueued behind the stop may differ by one
            assert g[4] == d[4]
        np.testing.assert_array_equal(g[0], d[0])
        np.testing.assert_array_equal(g[1], d[1])
        np.testing.assert_array_equal(g[3], d[3])


def test_set_k_keeps_the_clouds(oracle, small):
    """set_k (SVGDICP.h:98) only changes K_source_: the next stein_align uses the new K on the stored clouds."""
    icp = make_icp(small, iterations=0, KNN_count=20, max_dist=3.0, debug_corr=True)
    icp.set_k(7)
    assert icp.stein_align() == sv.ALIGN_SUCCESS  # no second add_cloud
    idx = icp.get_candidates()
    assert idx.shape[1] == 7
    q0 = oracle.transform_q0(small.source, small.R0, small.t0)
    oidx, _ = oracle.cand_sorted(q0, small.target, 7)
    np.testing.assert_array_equal(idx, oidx)


def test_bench_subsample_against_stored_fp64_scan():
    """The bench problem (64-beam scan against its voxel map, K = 100) on a 6000-point subsample, P = 64, 12 iterations, against
    the stored fp64 oracle outputs of the same scan (tests/golden/bench_sub6000_p64.npz, make_golden_bench.py): our particles
    must agree within the scan tolerance and the mean within POSE_TOL.  (tests/test_gpu_fullsize.py checks the full BASELINE size.)"""
    import os
    import bench
    from test_gpu_fullsize import check_golden_inputs
    g = np.load(os.path.join(bench.ROOT, "tests", "golden", "bench_sub6000_p64.npz"))
    P, I, cap = 64, 12, 6000
    pb, _ = bench.make_problem(P)
    src = bench._subsample(pb, cap)
    check_golden_inputs(g, pb, src)
    W = bench.WORKLOAD
    icp = sv.SVNICP(sv.SteinICPParam(iterations=I, KNN_count=W["K"], max_dist=W["max_dist"], lr=W["lr"], SVN_full_grad=W["svn_full_grad"]),
                    pb.init_pose)
    icp.add_cloud(src, pb.target, pb.init_pose)
    icp.set_initial_mean(pb.R0, pb.t0)
    assert icp.stein_align() == sv.ALIGN_SUCCESS
    np.testing.assert_allclose(icp.get_particles().reshape(6, P), g["oracle_particles"], atol=5 * POSE_TOL, rtol=0)
    np.testing.assert_allclose(icp.get_transformation(), g["oracle_mean"], atol=POSE_TOL, rtol=0)
