"""GPU parity tests of the SVGD-ICP class (class_type = SVGDICP) through the C ABI, against the fp64 oracle
(oracle/svgd_oracle.c) and the reference's own outputs (tests/golden/svgd_*.npz).

Bars: same as the SVN-ICP class -- per-iteration quantities and the particle mean within POSE_TOL = 1e-5 (m / rad),
individual particles after a whole scan within SCAN_TOL = 5e-5 (fp32 geometry + near-tie correspondence flips compound).
"""
import numpy as np
import pytest

import oracle as orc
import svn_icp_b200 as sv
from svn_icp_b200 import synth
from conftest import golden_names, load_golden

pytestmark = pytest.mark.gpu

POSE_TOL = 1e-5
SCAN_TOL = 5e-5


def make_icp(pb, ctor_pose=None, **kw):
    prm = sv.SteinICPParam(**kw)
    icp = sv.SVGDICP(prm, pb.init_pose if ctor_pose is None else ctor_pose)
    icp.add_cloud(pb.source, pb.target, pb.init_pose)
    icp.set_initial_mean(pb.R0, pb.t0)
    return icp


@pytest.fixture(scope="module")
def lidar():
    return synth.make_problem(64, sensor="32", scan_index=6, n_map_scans=6, seed=0xC0FFEE)


@pytest.mark.parametrize("P", [64, 7, 300])
def test_first_order_gradient(oracle, lidar, P):
    """sgd_grad (SVGDICP.cpp:398-455) of iteration 0 for every particle: k_gn<FIRST> + k_finalize_first."""
    pb = lidar
    rng = np.random.default_rng(P)
    init = synth.init_particles(P, rng)
    icp = sv.SVGDICP(sv.SteinICPParam(iterations=1, KNN_count=33, max_dist=3.0, lr=0.03, debug_corr=True), init)
    icp.add_cloud(pb.source, pb.target, init)
    icp.set_initial_mean(pb.R0, pb.t0)
    assert icp.stein_align() == sv.ALIGN_SUCCESS
    _, g, x = icp.get_gn_system()
    np.testing.assert_array_equal(x, init.T)  # kernel positions of iteration 0 = the constructor's particles
    _, idx, mask = icp.get_correspondences()
    # (1) the arithmetic, on the SAME correspondences: fp32 geometry only
    og = oracle.svgd_grad_given_corr(init.T, pb.R0, pb.t0, pb.source, pb.target, idx, mask, 3.0)
    scale = np.abs(og).max()
    np.testing.assert_allclose(g, og, atol=2e-6 * scale, rtol=1e-5)
    # (2) the correspondences themselves against the fp64 choice: only near-tie / near-threshold pairs may differ
    q0 = oracle.transform_q0(pb.source, pb.R0, pb.t0)
    mink, _ = oracle.knn_mink(q0, pb.target, 33)
    oidx, omask = oracle.svgd_corr(init.T, pb.R0, pb.t0, pb.source, pb.target, mink, 3.0)
    assert np.mean(idx != oidx) < 2e-5 and np.mean(mask != omask) < 2e-5
    # (3) end to end against the fp64 gradient: one pair whose squared distance sits within fp32 rounding of max_dist flips
    # its mask and moves a rotation component by rho*|e|*|s|*N_s/(count+1) (up to ~3e-4 of the scale for a far point)
    full = oracle.svgd_grad(init.T, pb.R0, pb.t0, pb.source, pb.target, mink, 3.0)
    np.testing.assert_allclose(g, full, atol=1e-3 * scale, rtol=1e-5)


@pytest.mark.parametrize("optimizer,lr", [("Adam", 0.03), ("RMSprop", 0.01), ("SGD", 0.002), ("Adagrad", 0.03)])
def test_one_iteration_vs_oracle(oracle, lidar, optimizer, lr):
    """One whole iteration: gradient -> RBF median bandwidth -> svgd_grad -> optimizer step."""
    pb = lidar
    P = pb.init_pose.shape[1]
    icp = make_icp(pb, iterations=1, KNN_count=33, max_dist=3.0, lr=lr, optimizer=optimizer)
    assert icp.stein_align() == sv.ALIGN_SUCCESS
    prm = orc.make_svgd_params(iterations=1, lr=lr, max_dist=3.0, knn_count=33, optimizer=optimizer)
    ref = oracle.svgd_align(prm, pb.source, pb.target, pb.init_pose, pb.init_pose, pb.R0, pb.t0, dumps=("grad", "stein", "bandwidth"))
    d, h = icp.get_stein()
    assert abs(h - ref["bandwidth"][0]) <= 1e-12 * abs(h)
    s = np.abs(ref["stein"][0]).max()
    np.testing.assert_allclose(d, ref["stein"][0], atol=1e-4 * s, rtol=1e-5)  # same mask-flip allowance as the gradient
    got = icp.get_particles().reshape(6, P)
    np.testing.assert_allclose(got, ref["particles"], atol=POSE_TOL, rtol=0)
    np.testing.assert_allclose(icp.get_transformation(), ref["mean"], atol=POSE_TOL, rtol=0)


# P = 300 (> 64) runs the multi-CTA head chain: k_head_prep and, from iteration 1 on, the fast median path
@pytest.mark.parametrize("optimizer,lr,P", [("Adam", 0.03, 64), ("RMSprop", 0.01, 64), ("Adam", 0.03, 300)],
                         ids=["Adam-0.03", "RMSprop-0.01", "Adam-0.03-300"])
def test_full_scan_vs_oracle(oracle, lidar, optimizer, lr, P):
    pb = lidar
    init = pb.init_pose if P == pb.init_pose.shape[1] else synth.init_particles(P, np.random.default_rng(P))
    I = 12
    icp = sv.SVGDICP(sv.SteinICPParam(iterations=I, KNN_count=33, max_dist=3.0, lr=lr, optimizer=optimizer), init)
    icp.add_cloud(pb.source, pb.target, init)
    icp.set_initial_mean(pb.R0, pb.t0)
    assert icp.stein_align() == sv.ALIGN_SUCCESS
    prm = orc.make_svgd_params(iterations=I, lr=lr, max_dist=3.0, knn_count=33, optimizer=optimizer)
    ref = oracle.svgd_align(prm, pb.source, pb.target, init, init, pb.R0, pb.t0)
    got = icp.get_particles().reshape(6, P)
    # Adam / RMSprop divide the gradient by its running RMS: a near-threshold mask flip (test_first_order_gradient (3))
    # that changes a small gradient component by a few percent moves that parameter by a few percent of lr per step,
    # so single particles drift apart from the fp64 run faster than under SVN-ICP's Newton step: 4 * SCAN_TOL here.
    tol = 4 * SCAN_TOL
    np.testing.assert_allclose(got, ref["particles"], atol=tol, rtol=0)
    np.testing.assert_allclose(icp.get_transformation(), ref["mean"], atol=POSE_TOL, rtol=0)
    sd = np.sqrt(np.diag(ref["cov"]))
    assert np.all(np.abs(icp.get_distribution() - ref["var"]) <= 2 * tol * sd + tol ** 2)
    cov = icp.get_cov_matrix().reshape(6, 6)
    assert np.all(np.abs(cov - ref["cov"]) <= 2 * tol * np.add.outer(sd, sd) + tol ** 2)
    np.testing.assert_array_equal(icp.get_particle_weight(), np.ones(P))
    hist = icp.get_particle_history().reshape(I, 6, P)
    np.testing.assert_allclose(hist, ref["history"], atol=tol + 1e-6, rtol=0)
    assert icp.iterations_done() == I


@pytest.mark.parametrize("name", golden_names("svgd_"))
def test_golden_vectors_through_c_abi(name):
    """The reference's own SVGDICP outputs (tests/golden/make_golden_svgd.py) through svnicp_* with class_type SVGDICP."""
    z = load_golden(name)
    I, lr, md, es, thr, K = z["params"]
    P = z["init_pose"].shape[1]
    prm = sv.SteinICPParam(iterations=int(I), lr=float(lr), max_dist=float(md), check_early_stop=bool(es),
                           convergence_threshold=float(thr), KNN_count=int(K), optimizer=str(z["optimizer"]))
    icp = sv.SVGDICP(prm, z["ctor_pose"])
    icp.add_cloud(z["source"], z["target"], z["init_pose"])
    icp.set_initial_mean(z["R0"], z["t0"])
    state = icp.stein_align()
    if z["init_pose2"].size:
        np.testing.assert_allclose(icp.get_particles().reshape(6, P), z["ref_first_particles"], atol=SCAN_TOL, rtol=0)
        icp.add_cloud(z["source"], z["target"], z["init_pose2"])
        icp.set_initial_mean(z["R0"], z["t0"])
        state = icp.stein_align()
    assert state == int(z["ref_state"][0])
    np.testing.assert_allclose(icp.get_particles().reshape(6, P), z["ref_particles"], atol=SCAN_TOL, rtol=0, equal_nan=True)
    np.testing.assert_allclose(icp.get_transformation(), z["ref_mean"], atol=POSE_TOL, rtol=0, equal_nan=True)
    sd = np.sqrt(np.abs(z["ref_var"]))
    got_var = icp.get_distribution()
    assert np.all((np.abs(got_var - z["ref_var"]) <= 2 * SCAN_TOL * sd + SCAN_TOL ** 2) | (np.isnan(got_var) & np.isnan(z["ref_var"])))
    np.testing.assert_array_equal(icp.get_particle_weight(), z["ref_weights"])
    if state == sv.ALIGN_SUCCESS:
        hist = icp.get_particle_history().reshape(int(I), 6, P)
        np.testing.assert_allclose(hist, z["ref_history"], atol=SCAN_TOL + 1e-6, rtol=0, equal_nan=True)
        assert icp.iterations_done() == int(z["ref_runtime"][2])  # finish_iter_


def test_stale_constructor_particles_drive_iteration_zero(oracle, lidar):
    """add_cloud does not refresh pose_particles_ (SVGDICP.cpp:46-62): iteration 0 evaluates the kernel on the constructor's set."""
    pb = lidar
    P = pb.init_pose.shape[1]
    rng = np.random.default_rng(3)
    ctor = pb.init_pose + rng.normal(size=pb.init_pose.shape) * 0.05
    icp = make_icp(pb, ctor_pose=ctor, iterations=2, KNN_count=33, max_dist=3.0, lr=0.03)
    icp.stein_align()
    prm = orc.make_svgd_params(iterations=2, lr=0.03, max_dist=3.0, knn_count=33)
    ref = oracle.svgd_align(prm, pb.source, pb.target, ctor, pb.init_pose, pb.R0, pb.t0)
    fresh = oracle.svgd_align(prm, pb.source, pb.target, pb.init_pose, pb.init_pose, pb.R0, pb.t0)
    got = icp.get_particles().reshape(6, P)
    np.testing.assert_allclose(got, ref["particles"], atol=POSE_TOL, rtol=0)
    assert np.abs(ref["particles"] - fresh["particles"]).max() > 100 * POSE_TOL  # the quirk is observable


def test_no_optimizer_state_and_getters(lidar):
    pb = lidar
    icp = make_icp(pb, iterations=3, KNN_count=16, optimizer="LBFGS")
    assert icp.stein_align() == sv.NO_OPTIMIZER
    P = pb.init_pose.shape[1]
    np.testing.assert_array_equal(icp.get_particles().reshape(6, P), pb.init_pose)
    np.testing.assert_allclose(icp.get_transformation(), pb.init_pose.mean(axis=1), atol=1e-15)
    np.testing.assert_allclose(icp.get_distribution(), pb.init_pose.var(axis=1, ddof=1), rtol=1e-12)


def test_deterministic_and_reusable(lidar):
    pb = lidar
    a = make_icp(pb, iterations=5, KNN_count=33, max_dist=3.0, lr=0.03)
    a.stein_align()
    pa = a.get_particles().copy()
    b = make_icp(pb, iterations=5, KNN_count=33, max_dist=3.0, lr=0.03)
    b.stein_align()
    np.testing.assert_array_equal(pa, b.get_particles())
    # second scan on the same object: the optimizer moments restart, pose_particles_ carries over
    a.add_cloud(pb.source, pb.target, pb.init_pose)
    a.set_initial_mean(pb.R0, pb.t0)
    a.stein_align()
    assert np.all(np.isfinite(a.get_particles()))
    assert np.abs(a.get_particles() - pa).max() > 0  # iteration 0 saw the previous result as kernel positions


def test_minibatch_rejected(lidar):
    with pytest.raises(sv.SvnIcpError):
        sv.SVGDICP(sv.SteinICPParam(use_minibatch=True), lidar.init_pose)
