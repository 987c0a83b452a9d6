"""svnicp_map_refine without a GPU: the principal SO(3) Log against scipy (up to and including pi), the fp64 oracle's update
(tests/map_refine_oracle.c) against the matrix exponential, the oracle loop on a synthetic map, a pose without inliers, and
VoxelHashMap::Refine of the C++ mirror compiled and linked against the C ABI.  refine_oracle, log_principal and refine_update are
also used by tests/test_gpu_map_refine.py."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest
from scipy.linalg import expm
from scipy.spatial.transform import Rotation

from conftest import ROOT

_LIB = None
_DIR = None


def _lib():
    """tests/map_refine_oracle.c, compiled once per process into a temporary directory (the tree may be read-only)"""
    global _LIB, _DIR
    if _LIB is None:
        _DIR = tempfile.TemporaryDirectory(prefix="map_refine_oracle_")
        so = os.path.join(_DIR.name, "libmap_refine_oracle.so")
        subprocess.check_call(["/usr/bin/gcc", "-O2", "-std=c11", "-fPIC", "-ffp-contract=off", "-fopenmp", "-Wall", "-Wextra", "-Werror",
                               "-shared", "-o", so, os.path.join(ROOT, "tests", "map_refine_oracle.c"), "-lm"])
        _LIB = C.CDLL(so)
        _LIB.oracle_refine_update.restype = C.c_double
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def log_principal(R):
    R = np.ascontiguousarray(R, dtype=np.float64).reshape(9)
    w = np.zeros(3)
    _lib().oracle_so3_log_principal(_p(R), _p(w))
    return w


def so3_exp(w):
    """the oracle's Exp and J_l (NaN at a zero angle, quirk Q7)"""
    w = np.ascontiguousarray(w, dtype=np.float64)
    R, J = np.zeros(9), np.zeros(9)
    _lib().oracle_so3_exp(_p(w), _p(R), _p(J))
    return R.reshape(3, 3), J.reshape(3, 3)


def refine_update(x, H, b):
    """one update of the oracle from the system at x -> (x', |delta|)"""
    x = np.ascontiguousarray(x, dtype=np.float64)
    H = np.ascontiguousarray(H, dtype=np.float64).reshape(36)
    b = np.ascontiguousarray(b, dtype=np.float64)
    out = np.zeros(6)
    dn = _lib().oracle_refine_update(_p(x), _p(H), _p(b), _p(out))
    return out, dn


def refine_oracle(src, map_xyz, R0, t0, poses, max_dist, iterations, tol):
    """the whole loop in fp64 -> poses [6, M], iterations [M], step [M], inliers [M]"""
    src = np.ascontiguousarray(src, dtype=np.float32).reshape(-1, 3)
    mp = np.ascontiguousarray(map_xyz, dtype=np.float32).reshape(-1, 3)
    x = np.ascontiguousarray(np.asarray(poses, dtype=np.float64).reshape(6, -1))
    M = x.shape[1]
    out, its, step, cnt = np.zeros((6, M)), np.zeros(M, np.int32), np.zeros(M), np.zeros(M, np.int64)
    _lib().oracle_map_refine(_p(src), C.c_int64(len(src)), _p(mp), C.c_int64(len(mp)), _p(np.ascontiguousarray(R0, dtype=np.float64)),
                             _p(np.ascontiguousarray(t0, dtype=np.float64)), C.c_int(M), _p(x), C.c_double(max_dist), C.c_int(iterations),
                             C.c_double(tol), _p(out), _p(its), _p(step), _p(cnt))
    return out, its.astype(np.int64), step, cnt


def rot_angle_between(Ra, Rb):
    return np.linalg.norm(Rotation.from_matrix(Ra.T @ Rb).as_rotvec())


def _angles_and_axes():
    rng = np.random.default_rng(0)
    axes = [np.eye(3)[k] for k in range(3)] + [v / np.linalg.norm(v) for v in rng.normal(size=(12, 3))]
    angles = [np.pi, np.pi - 1e-9, np.pi - 1e-4, 3.0, 2.0, np.pi / 2 + 1e-3, np.pi / 2, np.pi / 2 - 1e-3, 1.0, 1e-3, 1e-8, 1e-15, 0.0]
    return [(a, n) for a in angles for n in axes]


def test_log_principal_against_scipy():
    for a, n in _angles_and_axes():
        R = Rotation.from_rotvec(a * n).as_matrix()
        w = log_principal(R)
        assert np.linalg.norm(w) <= np.pi * (1 + 1e-15)
        # rotations, not rotation vectors: at exactly pi, w and -w are the same rotation
        assert rot_angle_between(Rotation.from_rotvec(w).as_matrix(), R) < 1e-13, (a, n)
        ref = Rotation.from_matrix(R).as_rotvec()
        if a < np.pi - 1e-3:
            np.testing.assert_allclose(w, ref, rtol=0, atol=1e-13)
        else:  # the axis near pi: the reference log of so3_log returns 0 or loses digits here
            assert abs(abs(w @ n) - a) < 1e-12 and np.linalg.norm(np.cross(w, n)) < 1e-12
    np.testing.assert_array_equal(log_principal(np.eye(3)), np.zeros(3))


def test_log_principal_exact_pi():
    for k in range(3):
        R = -np.eye(3)
        R[k, k] = 1.0
        w = log_principal(R)
        want = np.zeros(3)
        want[k] = np.pi
        np.testing.assert_allclose(np.abs(w), want, rtol=0, atol=1e-15)


def _hat4(d):
    v, w = d[:3], d[3:]
    return np.array([[0, -w[2], w[1], v[0]], [w[2], 0, -w[0], v[1]], [-w[1], w[0], 0, v[2]], [0, 0, 0, 0]])


def test_update_against_expm():
    """x' = [t' ; Log R'] with R' = Exp(omega) dR, t' = R' dt + t, (dR, dt) = expm of the twist delta (SVNICP.cpp:268-279)"""
    rng = np.random.default_rng(1)
    for k in range(50):
        x = np.concatenate([rng.normal(0, 2.0, 3), rng.normal(0, 0.5, 3)])
        A = rng.normal(size=(6, 6))
        H = A @ A.T + 6 * np.eye(6)
        b = rng.normal(0, 10.0 ** -rng.uniform(1, 5), 6)
        d = -np.linalg.solve(H, b)
        E = expm(_hat4(d))
        R = Rotation.from_rotvec(x[3:]).as_matrix()
        Rn = R @ E[:3, :3]
        tn = Rn @ E[:3, 3] + x[:3]
        got, dn = refine_update(x, H, b)
        assert dn == pytest.approx(np.linalg.norm(d), rel=1e-12)
        np.testing.assert_allclose(got[:3], tn, rtol=0, atol=1e-12 * (1 + np.abs(tn).max()))
        assert rot_angle_between(Rotation.from_rotvec(got[3:]).as_matrix(), Rn) < 1e-12


def test_zero_rotation_step_uses_identity_jacobian():
    """delta_w = 0 exactly: J_l = I (the reference's J_l is NaN there, Q7)"""
    _, J = so3_exp(np.zeros(3))
    assert np.isnan(J).all()
    x = np.array([1.0, -2.0, 0.5, 0.1, 0.2, -0.3])
    H = np.diag([2.0, 4.0, 8.0, 1.0, 1.0, 1.0])
    b = np.array([-2.0, 4.0, -8.0, 0.0, 0.0, 0.0])  # delta = (1, -1, 1, 0, 0, 0) exactly
    got, dn = refine_update(x, H, b)
    R = Rotation.from_rotvec(x[3:]).as_matrix()
    np.testing.assert_allclose(got[:3], R @ np.array([1.0, -1.0, 1.0]) + x[:3], rtol=0, atol=1e-14)
    np.testing.assert_allclose(got[3:], x[3:], rtol=0, atol=1e-15)
    assert dn == np.sqrt(3.0) and np.isfinite(got).all()


def _room(rng, n=20000):
    """random points of a 20 m box volume (float32), distinct structure in every direction"""
    return rng.uniform(-10, 10, (n, 3)).astype(np.float32)


def test_oracle_converges_from_offset():
    rng = np.random.default_rng(2)
    mp = _room(rng)
    R_gt = Rotation.from_rotvec([0.02, -0.01, 0.3]).as_matrix()
    t_gt = np.array([0.4, -0.3, 0.1])
    sel = rng.choice(len(mp), 2000, replace=False)
    src = ((mp[sel].astype(np.float64) - t_gt) @ R_gt).astype(np.float32)  # s = R_gt^T (p - t_gt)
    R0 = R_gt @ Rotation.from_rotvec([0.004, 0.003, -0.012]).as_matrix()
    t0 = t_gt + np.array([0.1, -0.08, 0.05])
    x, its, step, cnt = refine_oracle(src, mp, R0, t0, np.zeros(6), 1.0, 30, 1e-10)
    R = R0 @ Rotation.from_rotvec(x[3:, 0]).as_matrix()
    t = t0 + R0 @ x[:3, 0]
    assert np.linalg.norm(t - t_gt) < 1e-5 and rot_angle_between(R, R_gt) < 1e-6
    assert cnt[0] == len(src) and its[0] < 30 and step[0] < 1e-10


def test_no_inlier_pose_stays_put():
    rng = np.random.default_rng(3)
    mp = _room(rng, 2000)
    src = _room(rng, 300)
    x0 = np.array([[0.3, -0.2, 0.1, 0.01, -0.02, 0.5]]).T
    x, its, step, cnt = refine_oracle(src, mp, np.eye(3), np.array([1e4, 0, 0]), x0, 1.0, 5, 0.0)
    np.testing.assert_array_equal(x, x0)
    assert its[0] == 5 and step[0] == 0.0 and cnt[0] == 0


SRC = r"""
#include "svnicp/VoxelHashMap.hpp"
int main() {
  int reached = 0;
  try {
    svnicp::VoxelHashMap m(1.0, 100.0, 20);
    reached = 1;
    std::vector<float> xyz = {0.f, 0.f, 0.f, 1.f, 2.f, 3.f, -1.f, 0.5f, 2.f};
    svnicp::InitialMean T0;
    m.AddPointCloud(xyz, T0);
    std::vector<double> poses(12, 0.0);
    poses[0] = 0.05;  // pose 0: t_x = 0.05 ([6][M] layout)
    svnicp::VoxelHashMap::RefineResult r = m.Refine(xyz.data(), 3, T0, poses, 1.0, 5, 0.0, true);
    if (r.n_poses != 2 || r.poses.size() != 12 || r.iterations.size() != 2 || r.H.size() != 72 || r.inliers[1] != 3) return 4;
    if (r.iterations[0] != 5) return 6;
    r = m.Refine(xyz.data(), 3, T0, poses, 1.0e6);  // radius beyond 4 voxels: throws
    return 5;
  } catch (const svnicp::Error &) {
  }
  return reached ? 10 : 0;
}
"""


def test_mirror_map_refine_compiles(tmp_path):
    from svn_icp_b200 import build
    lib = build.build()
    src, exe = os.path.join(tmp_path, "map_refine.cpp"), os.path.join(tmp_path, "map_refine")
    open(src, "w").write(SRC)
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "svn_icp_b200", "include"), src,
                           "-o", exe, lib, "-Wl,-rpath," + os.path.dirname(lib)])
    import torch
    # without a GPU the constructor throws (0); on a GPU the first Refine succeeds and the second throws (10)
    assert subprocess.call([exe]) == (10 if torch.cuda.is_available() else 0)
