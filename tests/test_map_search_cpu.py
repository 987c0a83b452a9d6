"""svnicp_map_search without a GPU: the grid formula of search_grid_poses, the (count descending, g ascending) order restated
on hand-made counts, and VoxelHashMap::Search of the C++ mirror compiled and linked against the C ABI."""
import os
import subprocess

import numpy as np
import pytest

import svn_icp_b200 as sv
from conftest import ROOT


def topk_lexsort(counts, k):
    """The ranking of the ABI: count descending, then flat grid index ascending"""
    counts = np.asarray(counts).reshape(-1)
    return np.lexsort((np.arange(len(counts)), -counts.astype(np.int64)))[:k]


@pytest.mark.parametrize("counts", [(1, 1, 1, 1, 1, 1), (3, 1, 1, 1, 1, 5), (4, 2, 1, 1, 1, 6), (5, 4, 3, 2, 3, 7), (2, 3, 1, 4, 1, 1)])
def test_grid_poses_formula(counts):
    steps = np.array([0.25, 0.5, 0.1, 0.01, 0.02, np.deg2rad(5.0)])
    M = int(np.prod(counts))
    g = np.arange(M)
    x = sv.search_grid_poses(counts, steps, g)
    assert x.shape == (6, M)
    # the flat index: axis 0 fastest, i.e. the C-order index of the reversed counts
    idx = np.unravel_index(g, tuple(reversed(counts)))[::-1]
    for a in range(6):
        want = (idx[a].astype(np.float64) - 0.5 * (counts[a] - 1)) * steps[a]
        np.testing.assert_array_equal(x[a], want)
        vals = np.unique(x[a])
        assert len(vals) == counts[a]
        np.testing.assert_array_equal(vals, -vals[::-1])  # centred on T0
        assert (0.0 in vals) == (counts[a] % 2 == 1)  # odd counts hold x_a = 0, even ones do not
    zero = np.flatnonzero((x == 0).all(axis=0))
    if all(c % 2 == 1 for c in counts):
        assert len(zero) == 1 and zero[0] == sum(((c - 1) // 2) * int(np.prod(counts[:a])) for a, c in enumerate(counts))
    else:
        assert len(zero) == 0
    # one index alone gives the same pose
    for j in (0, M // 2, M - 1):
        np.testing.assert_array_equal(sv.search_grid_poses(counts, steps, j)[:, 0], x[:, j])


def test_grid_poses_zero_step():
    x = sv.search_grid_poses((3, 1, 1, 1, 1, 2), (0.0, 0, 0, 0, 0, 0.1), np.arange(6))
    assert (x[0] == 0).all() and (x[:5] == 0).all()
    np.testing.assert_array_equal(x[5], [-0.05] * 3 + [0.05] * 3)


def test_topk_order_with_ties():
    """The unique key ((n - count) << 32) | g of the kernels sorts as the lexsort of (-count, g): many ties, all-equal counts,
    and counts at the ends of [0, n]."""
    rng = np.random.default_rng(0)
    n = 900
    cases = [rng.integers(0, 4, 5000), np.zeros(3000, np.int64), np.full(2000, n), rng.integers(0, n + 1, 40000),
             np.repeat(rng.integers(0, 50, 300), 37)]
    for c in cases:
        keys = ((n - c.astype(np.uint64)) << np.uint64(32)) | np.arange(len(c), dtype=np.uint64)
        assert len(np.unique(keys)) == len(c)
        for k in (1, 7, 1024):
            want = topk_lexsort(c, k)
            np.testing.assert_array_equal(np.sort(keys)[:k] & np.uint64(0xFFFFFFFF), want.astype(np.uint64))
            # ties resolved by g: within a run of equal counts, indices ascend
            got = want
            assert (np.diff(c[got]) <= 0).all()
            same = np.diff(c[got]) == 0
            assert (np.diff(got)[same] > 0).all()
    # every count zero: the winners are g = 0 .. k-1
    np.testing.assert_array_equal(topk_lexsort(np.zeros(5000), 1024), np.arange(1024))


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
    const int32_t counts[6] = {3, 3, 1, 1, 1, 5};
    const double steps[6] = {2.0, 2.0, 0.0, 0.0, 0.0, 1.0};  // only x = 0 keeps both points within 1 m
    svnicp::VoxelHashMap::SearchResult r = m.Search(xyz.data(), 2, T0, counts, steps, 1.0, 7, true);
    if (r.k != 7 || r.index.size() != 7 || r.poses.size() != 42 || r.count.size() != 7 || r.counts.size() != 45) return 4;
    if (r.index[0] != 22 || r.count[0] != 2) return 6;  // x = 0 (g = 1 + 3 * (1 + 3 * 2)) holds both points
    r = m.Search(xyz.data(), 2, T0, counts, steps, 1.0e6);  // radius beyond 4 voxels: throws
    return 5;
  } catch (const svnicp::Error &) {
  }
  return reached ? 10 : 0;
}
"""


def test_mirror_map_search_compiles(tmp_path):
    from svn_icp_b200 import build
    lib = build.build()
    src, exe = os.path.join(tmp_path, "map_search.cpp"), os.path.join(tmp_path, "map_search")
    open(src, "w").write(SRC)
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "svn_icp_b200", "include"), src,
                           "-o", exe, lib, "-Wl,-rpath," + os.path.dirname(lib)])
    import torch
    # without a GPU the constructor throws (0); on a GPU the first Search succeeds and the second throws (10)
    assert subprocess.call([exe]) == (10 if torch.cuda.is_available() else 0)
