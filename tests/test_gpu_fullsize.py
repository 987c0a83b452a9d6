"""GPU parity at the BASELINE.json sizes (through the C ABI).

  configs[1]  P = 1000, 64-beam scan (143k points), 30 iterations: against the stored outputs of that scan
              (tests/golden/bench_full_p1000.npz): the particle mean of the REFERENCE ITSELF run on a B200 (its unmodified
              sources + its vendored knn.cu) and the particles of the fp64 oracle, asserted.
  configs[2]  P = 4096 (16 particle groups), 128-beam scan (~250k points): correspondence indices bit-exact and a short scan
              against the fp64 oracle on a 4096-point subsample of that scan; the full-size scan through size-independent
              properties (deterministic, finite, recovers the planted motion, history consistent with the particles).
"""
import os

import numpy as np
import pytest

import oracle as orc
import svn_icp_b200 as sv
from svn_icp_b200 import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
POSE_TOL = 1e-5


def check_golden_inputs(g, pb, src):
    """The seeded bench problem is still the one the golden outputs were computed on (tests/golden/make_golden_bench.py)."""
    np.testing.assert_array_equal(g["in_n"], [len(src), len(pb.target)])
    for k, v in (("in_gt_rel", pb.gt_rel), ("in_R0", pb.R0), ("in_t0", pb.t0), ("in_init_pose", pb.init_pose)):
        np.testing.assert_allclose(v, g[k], rtol=0, atol=1e-12, err_msg=k)
    np.testing.assert_allclose(src.sum(0), g["in_source_sum"], rtol=1e-12, err_msg="source")
    np.testing.assert_allclose(pb.target.sum(0), g["in_target_sum"], rtol=1e-12, err_msg="target")


def test_config1_full_size_against_the_reference_on_this_gpu():
    """Per-particle poses <= 5e-5, particle mean <= 1e-5 after 30 iterations at P = 1000, N_s = 143k (near-tie
    correspondence flips -- 1.6e-6 of the pairs -- compound through the repulsive dynamics, hence the per-particle bar).
    Against tests/golden/bench_full_p1000.npz: the particle mean of the reference's own sources run on a B200 on this scan,
    and the particles of the fp64 C restatement on the same scan."""
    import bench
    g = np.load(os.path.join(ROOT, "tests", "golden", "bench_full_p1000.npz"))
    P, I = 1000, 30
    pb, _ = bench.make_problem(P)
    check_golden_inputs(g, pb, pb.source)
    W = bench.WORKLOAD
    icp = sv.SVNICP(sv.SteinICPParam(iterations=I, KNN_count=W["K"], max_dist=W["max_dist"], lr=W["lr"], SVN_full_grad=True), pb.init_pose)
    icp.add_cloud(pb.source, pb.target, pb.init_pose)
    icp.set_initial_mean(pb.R0, pb.t0)
    assert icp.stein_align() == sv.ALIGN_SUCCESS
    ours = icp.get_particles().reshape(6, P)
    np.testing.assert_allclose(ours, g["oracle_particles"], atol=5 * POSE_TOL, rtol=0)
    np.testing.assert_allclose(icp.get_transformation(), g["reference_mean"], atol=POSE_TOL, rtol=0)
    np.testing.assert_allclose(icp.get_transformation(), g["oracle_mean"], atol=POSE_TOL, rtol=0)


@pytest.fixture(scope="module")
def c2():
    return synth.make_problem_saturated(4096, sensor="128")


def test_config2_indices_bit_exact_over_particle_groups(oracle, c2):
    rng = np.random.default_rng(3)
    sel = np.sort(rng.choice(len(c2.source), 4096, replace=False))
    src = np.ascontiguousarray(c2.source[sel])
    icp = sv.SVNICP(sv.SteinICPParam(iterations=1, KNN_count=100, max_dist=3.0, lr=1.0, debug_corr=True), c2.init_pose)
    icp.add_cloud(src, c2.target, c2.init_pose)
    icp.set_initial_mean(c2.R0, c2.t0)
    assert icp.stein_align() == sv.ALIGN_SUCCESS
    assert icp.get_scan_info()["n_pgroups"] == 4  # k_gn: 512 threads x 2 particles per CTA; 4096 particles = 4 groups over the same rows
    xf, idx, mask = icp.get_correspondences()
    cidx, rel = icp.get_candidates(want_rel=True)
    oidx, omask = oracle.corr_f32(xf, icp.get_source_f32(), rel, cidx, 3.0)
    np.testing.assert_array_equal(idx, oidx)
    np.testing.assert_array_equal(mask, omask)


def test_config2_short_scan_vs_oracle(oracle, c2):
    rng = np.random.default_rng(4)
    sel = np.sort(rng.choice(len(c2.source), 4096, replace=False))
    src = np.ascontiguousarray(c2.source[sel])
    I = 3
    icp = sv.SVNICP(sv.SteinICPParam(iterations=I, KNN_count=100, max_dist=3.0, lr=1.0), c2.init_pose)
    icp.add_cloud(src, c2.target, c2.init_pose)
    icp.set_initial_mean(c2.R0, c2.t0)
    assert icp.stein_align() == sv.ALIGN_SUCCESS
    o = oracle.align(orc.make_params(iterations=I, knn_count=100, max_dist=3.0, lr=1.0, svn_full_grad=True), src, c2.target, c2.init_pose,
                     c2.R0, c2.t0)
    np.testing.assert_allclose(icp.get_particles().reshape(6, -1), o["particles"], atol=POSE_TOL, rtol=0)
    np.testing.assert_allclose(icp.get_transformation(), o["mean"], atol=POSE_TOL, rtol=0)
    np.testing.assert_allclose(icp.get_cov_matrix().reshape(6, 6), o["cov"], atol=POSE_TOL ** 2 + 2e-5 * np.abs(o["cov"]).max(), rtol=0)


def test_config2_full_size_properties(c2):
    P, I = 4096, 12
    icp = sv.SVNICP(sv.SteinICPParam(iterations=I, KNN_count=100, max_dist=3.0, lr=1.0), c2.init_pose)
    runs = []
    for _ in range(2):
        icp.add_cloud(c2.source, c2.target, c2.init_pose)
        icp.set_initial_mean(c2.R0, c2.t0)
        assert icp.stein_align() == sv.ALIGN_SUCCESS
        runs.append((icp.get_particles().copy(), icp.get_particle_history().copy(), icp.get_transformation().copy()))
    np.testing.assert_array_equal(runs[0][0], runs[1][0])  # deterministic
    part, hist, mean = runs[0]
    assert np.isfinite(part).all() and hist.shape == (I, 6 * P)
    # history row e = poses after update e (SVNICP.cpp:103-107): without an early stop the last row is the final particle set
    np.testing.assert_array_equal(hist[-1], part.astype(np.float32))
    err = np.abs(mean - c2.gt_rel)
    assert err[:3].max() < 0.02 and err[3:].max() < 2e-3, err  # recovers the planted motion (range noise 2 cm)
    w = icp.get_particle_weight()
    np.testing.assert_array_equal(w, np.full(P, np.float64(np.float32(1.0) / np.float32(P))))
