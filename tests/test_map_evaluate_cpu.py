"""svnicp_map_evaluate without a GPU: the brute-force nearest-map-point oracle (tests/map_nn_oracle.c) against scipy's k-d tree
and on hand-made voxel-boundary cases, and VoxelHashMap::Evaluate of the C++ mirror compiled and linked against the C ABI.
map_nn and BOUNDARY_CASES are also used by tests/test_gpu_map_evaluate.py."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest
from scipy.spatial import cKDTree

from conftest import ROOT

_NN_LIB = None
_NN_DIR = None


def _nn_lib():
    """tests/map_nn_oracle.c, compiled once per process into a temporary directory (the tree may be read-only)"""
    global _NN_LIB, _NN_DIR
    if _NN_LIB is None:
        _NN_DIR = tempfile.TemporaryDirectory(prefix="map_nn_oracle_")
        so = os.path.join(_NN_DIR.name, "libmap_nn_oracle.so")
        subprocess.check_call(["/usr/bin/gcc", "-O2", "-std=c11", "-fPIC", "-ffp-contract=off", "-fopenmp", "-Wall", "-Wextra", "-Werror",
                               "-shared", "-o", so, os.path.join(ROOT, "tests", "map_nn_oracle.c"), "-lm"])
        _NN_LIB = C.CDLL(so)
    return _NN_LIB


def map_nn(q, map_xyz, max_dist):
    """Brute-force nearest map point of fp64 queries among float map points (svnicp_map_evaluate's contract):
    -> nearest [n,3] float32, d2 [n], mask [n] uint8, idx [n] int64 (-1 where no point has d^2 < max_dist)."""
    q = np.ascontiguousarray(q, dtype=np.float64).reshape(-1, 3)
    mp = np.ascontiguousarray(map_xyz, dtype=np.float32).reshape(-1, 3)
    n = len(q)
    near = np.zeros((n, 3), dtype=np.float32)
    d2 = np.zeros(n)
    mask = np.zeros(n, dtype=np.uint8)
    idx = np.zeros(n, dtype=np.int64)
    p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    _nn_lib().oracle_map_nn(p(q), C.c_int64(n), p(mp), C.c_int64(len(mp)), C.c_double(max_dist), p(near), p(d2), p(mask), p(idx))
    return near, d2, mask, idx


# (name, voxel_size, max_dist, map points, queries, expected map row per query or -1).  Values are dyadic where a tie or a
# boundary has to be exact.
BOUNDARY_CASES = [
    # x in (-1, 1) is voxel 0 (truncation toward zero), twice as wide as voxel 1 = [1, 2) and voxel -1 = (-2, -1]
    ("zero_voxel_both_sides", 1.0, 1.0,
     [[-0.75, 0, 0], [0.75, 0, 0], [1.25, 0, 0], [-1.25, 0, 0], [0, -0.5, 0.25]],
     [[0.25, 0, 0], [-0.5, 0, 0], [-1.0, 0, 0], [1.0, 0, 0], [0, 0, 0], [0.0, 0.0, 1.0]],
     # q = -1: -0.75 (voxel 0) and -1.25 (voxel -1) tie at d^2 = 1/16 -> smaller x; q = 1: 0.75 and 1.25 tie -> 0.75;
     # (0, 0, 1): d^2 to (0, -0.5, 0.25) = 0.8125 < 1
     [1, 0, 3, 1, 4, 4]),
    ("negative_coordinates", 0.5, 0.25,
     [[-3.1, -2.2, -1.3], [-3.4, -2.2, -1.3], [-2.9, -2.6, -1.1], [-0.2, -0.3, -0.1]],
     [[-3.2, -2.2, -1.3], [-3.3, -2.25, -1.3], [-2.8, -2.5, -1.0], [-0.1, -0.1, -0.1], [-5.0, -5.0, -5.0]],
     [0, 1, 2, 3, -1]),
    # r = 1.73 v: the nearest point of the first query lies two voxels away; the second query's only point is beyond r
    ("two_voxels_away", 1.0, 1.73 ** 2,
     [[2.5, 0.5, 0.5], [3.0, -0.5, -0.5]],
     [[0.9, 0.5, 0.5], [0.5, 0.5, 0.5], [2.0, -0.25, -0.25]],
     [0, -1, 1]),
    ("radius_below_voxel", 1.0, 0.09,
     [[1.1, 0, 0], [0.5, 0.5, 0.5]],
     [[0.9, 0, 0], [0.5, 0.5, 0.85], [0.5, 0.5, 0.75]],
     [0, -1, 1]),
    # voxel 0.5; (0.25, 0.25, +-0.25) tie at d^2 = 1/16 from (0.25, 0.25, 0) -> the smaller z
    ("half_metre_voxels_tie", 0.5, 0.3,
     [[0.25, 0.25, 0.25], [0.25, 0.25, -0.25], [0.75, 0.75, 0.75], [-0.75, 0.25, 0.0]],
     [[0.25, 0.25, 0.0], [0.7, 0.7, 0.7], [-0.5, 0.25, 0.0], [-0.25, 0.25, 0.0]],
     [1, 2, 3, 3]),
]


def case_arrays(case):
    name, v, md, pts, qs, want = case
    return name, v, md, np.asarray(pts, dtype=np.float32), np.asarray(qs, dtype=np.float64), np.asarray(want)


def test_map_nn_against_kdtree():
    rng = np.random.default_rng(0)
    for n_map, n_q, max_dist in ((2000, 3000, 0.5), (50, 500, 4.0), (20000, 2000, 0.05)):
        mp = rng.uniform(-10, 10, (n_map, 3)).astype(np.float32)
        q = rng.uniform(-11, 11, (n_q, 3))
        near, d2, mask, idx = map_nn(q, mp, max_dist)
        dist, j = cKDTree(mp.astype(np.float64)).query(q)
        kd2 = dist ** 2
        clear = np.abs(kd2 - max_dist) >= 1e-12 * max_dist
        np.testing.assert_array_equal(mask[clear], (kd2 < max_dist)[clear])
        sel = mask.astype(bool)
        np.testing.assert_allclose(d2[sel], kd2[sel], rtol=1e-12, atol=0)
        np.testing.assert_array_equal(near[sel], mp[idx[sel]])
        assert (idx[~sel] == -1).all() and (near[~sel] == 0).all() and (d2[~sel] == 0).all()
        assert sel.any() and (~sel).any()


def test_map_nn_nonfinite_queries():
    mp = np.zeros((4, 3), dtype=np.float32)
    q = np.array([[np.nan, 0, 0], [np.inf, 0, 0], [0, 0, 0.5]])
    _, _, mask, idx = map_nn(q, mp, 1.0)
    np.testing.assert_array_equal(mask, [0, 0, 1])
    assert idx[2] == 0  # four identical points: the first one


@pytest.mark.parametrize("case", BOUNDARY_CASES, ids=[c[0] for c in BOUNDARY_CASES])
def test_boundary_cases(case):
    _, v, md, pts, qs, want = case_arrays(case)
    assert np.ceil(np.sqrt(md) / v) <= 4
    near, d2, mask, idx = map_nn(qs, pts, md)
    np.testing.assert_array_equal(idx, want)
    np.testing.assert_array_equal(mask, want >= 0)
    np.testing.assert_array_equal(near[want >= 0], pts[want[want >= 0]])


SRC = r"""
#include "svnicp/VoxelHashMap.hpp"
int main() {
  int reached = 0;
  try {
    svnicp::VoxelHashMap m(1.0, 100.0, 20);
    reached = 1;
    std::vector<float> xyz = {0.f, 0.f, 0.f, 1.f, 2.f, 3.f};
    svnicp::InitialMean T0;
    m.AddPointCloud(xyz, T0);
    svnicp::SVGDICP::Evaluation e = m.Evaluate(xyz.data(), 2, T0, std::vector<double>(12, 0.0), 1.0, true, true);
    if (e.n_poses != 2 || e.inliers.size() != 2 || e.H.size() != 72 || e.mask.size() != 4) return 4;
    e = m.Evaluate(xyz.data(), 2, T0, std::vector<double>(6, 0.0), 1.0e6);  // radius beyond 4 voxels: throws
    return 5;
  } catch (const svnicp::Error &) {
  }
  return reached ? 10 : 0;
}
"""


def test_mirror_map_evaluate_compiles(tmp_path):
    from svn_icp_b200 import build
    lib = build.build()
    src, exe = os.path.join(tmp_path, "map_eval.cpp"), os.path.join(tmp_path, "map_eval")
    open(src, "w").write(SRC)
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "svn_icp_b200", "include"), src,
                           "-o", exe, lib, "-Wl,-rpath," + os.path.dirname(lib)])
    import torch
    # without a GPU the constructor throws (0); on a GPU the first Evaluate succeeds and the second throws (10)
    assert subprocess.call([exe]) == (10 if torch.cuda.is_available() else 0)
