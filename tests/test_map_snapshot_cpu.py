"""Map snapshots without a GPU: the oracle's canonical export (tests/map_snapshot_oracle.c) on hand-made voxels, the snapshot file
format shared by the Python and C++ mirrors, and VoxelHashMap Export / Import / Save / Load of the C++ mirror compiled against the
C ABI.  SnapshotOracle is also the pin of tests/test_gpu_map_snapshot.py."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import oracle as orc
import svn_icp_b200 as sv
from conftest import ROOT

_LIB = None
_LIB_DIR = None


def _oracle_lib():
    """tests/map_snapshot_oracle.c (oracle/voxelmap_oracle.c plus the export), compiled once per process into a temporary
    directory (the tree may be read-only) with the flags of oracle/Makefile"""
    global _LIB, _LIB_DIR
    if _LIB is None:
        _LIB_DIR = tempfile.TemporaryDirectory(prefix="map_snapshot_oracle_")
        so = os.path.join(_LIB_DIR.name, "libmap_snapshot_oracle.so")
        subprocess.check_call(["/usr/bin/gcc", "-O2", "-std=c11", "-fPIC", "-ffp-contract=off", "-Wall", "-Wextra", "-Werror", "-shared",
                               "-o", so, os.path.join(ROOT, "tests", "map_snapshot_oracle.c"), "-lm"])
        _LIB = C.CDLL(so)
    return _LIB


class SnapshotOracle(orc.VoxelMapOracle):
    """orc.VoxelMapOracle (same sources, same methods) with Export(): the live voxels sorted by (vx, vy, vz) on the host."""

    def __init__(self, voxel_size=1.0, max_range=80.0, max_pointscount=20):
        self.lib = _oracle_lib()
        self.lib.oracle_vmap_create.restype = C.c_void_p
        self.lib.oracle_vmap_get.restype = C.c_int64
        self.lib.oracle_vmap_size.restype = C.c_int64
        self.params = (float(voxel_size), float(max_range), int(max_pointscount))
        self.m = C.c_void_p(self.lib.oracle_vmap_create(C.c_double(voxel_size), C.c_double(max_range), C.c_int(max_pointscount)))

    def Export(self) -> sv.MapSnapshot:
        V, N = C.c_int64(0), C.c_int64(0)
        self.lib.oracle_vmap_snapshot_size(self.m, C.byref(V), C.byref(N))
        vox = np.zeros((V.value, 3), dtype=np.int32)
        cnt = np.zeros(V.value, dtype=np.int32)
        pts = np.zeros((N.value, 3), dtype=np.float32)
        p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
        assert self.lib.oracle_vmap_export(self.m, p(vox), p(cnt), p(pts)) == 0
        return sv.MapSnapshot(*self.params, vox, cnt, pts)


def snapshots_equal(a: sv.MapSnapshot, b: sv.MapSnapshot):
    """array for array, bit for bit (NaN points included)"""
    assert (a.voxel_size, a.max_range, a.max_pointscount) == (b.voxel_size, b.max_range, b.max_pointscount)
    for name in ("voxels", "counts", "points"):
        x, y = getattr(a, name), getattr(b, name)
        assert x.dtype == y.dtype and x.shape == y.shape, name
        assert x.tobytes() == y.tobytes(), name


def expected_snapshot(pts, voxel_size, cap):
    """independent restatement for an identity pose: voxel = trunc(p / float(v)) in float32, first `cap` points per voxel in
    arrival order, voxels sorted lexicographically"""
    pts = np.asarray(pts, dtype=np.float32)
    vox = np.trunc(pts / np.float32(voxel_size)).astype(np.int32)
    groups = {}
    for v, p in zip(map(tuple, vox), pts):
        g = groups.setdefault(v, [])
        if len(g) < cap:
            g.append(p)
    keys = sorted(groups)
    return (np.array(keys, dtype=np.int32).reshape(-1, 3), np.array([len(groups[k]) for k in keys], dtype=np.int32),
            np.array([p for k in keys for p in groups[k]], dtype=np.float32).reshape(-1, 3))


def test_oracle_export_hand_made_voxels():
    # voxel 0 is (-1, 1) on each axis (truncation toward zero): -0.75 and 0.5 share it, -1.25 is voxel -1, 1.25 voxel 1
    pts = [[0.5, -0.25, 0.0], [-0.75, 0.5, -0.5], [-1.25, -2.5, 3.5], [1.25, 0.0, 0.0], [-0.5, -0.5, -0.5],
           [-1.5, -2.75, 3.25], [-3.5, 4.0, -7.25], [0.25, 0.25, 0.25], [-1.75, -2.25, 3.75], [1.5, 0.5, -0.5],
           [-0.125, 0.0, 0.0], [-1.0625, -2.0625, 3.0625]]
    o = SnapshotOracle(1.0, 1000.0, 3)
    o.AddPointCloud(np.asarray(pts, dtype=np.float32), np.eye(3), np.zeros(3))
    s = o.Export()
    vox, cnt, xyz = expected_snapshot(pts, 1.0, 3)
    np.testing.assert_array_equal(s.voxels, vox)
    np.testing.assert_array_equal(s.counts, cnt)
    np.testing.assert_array_equal(s.points, xyz)
    # voxel 0 holds its first three arrivals, from both sides of zero; (0.25, 0.25, 0.25) and (-0.125, 0, 0) came too late, and
    # voxel (-1, -2, 3) refused its fourth point likewise
    assert [-1, -2, 3] in s.voxels.tolist() and [0, 0, 0] in s.voxels.tolist()
    z = s.voxels.tolist().index([0, 0, 0])
    off = int(s.counts[:z].sum())
    np.testing.assert_array_equal(s.points[off:off + 3], np.asarray([pts[0], pts[1], pts[4]], dtype=np.float32))
    assert s.counts.sum() == len(s.points) == len(o.GetMap()) and len(s.counts) == o.Size()


def test_oracle_export_half_metre_voxels_and_removal():
    rng = np.random.default_rng(5)
    o = SnapshotOracle(0.5, 6.0, 4)
    clouds = [rng.uniform(-4, 4, (300, 3)).astype(np.float32) for _ in range(3)]
    for k, c in enumerate(clouds):
        o.AddPointCloud(c, np.eye(3), np.array([2.0 * k, 0.0, 0.0]))
    s = o.Export()
    # ascending lexicographic voxels, no duplicate, counts within [1, cap], every point in its voxel
    keys = [tuple(v) for v in s.voxels.tolist()]
    assert keys == sorted(set(keys))
    assert (s.counts >= 1).all() and (s.counts <= 4).all()
    per_point = np.repeat(s.voxels, s.counts, axis=0)
    np.testing.assert_array_equal(np.trunc(s.points / np.float32(0.5)).astype(np.int32), per_point)
    # RemoveFar ran: the first point of every voxel is within max_range of the last position
    first = s.points[np.concatenate([[0], np.cumsum(s.counts)[:-1]])].astype(np.float64)
    assert (np.sum((first - [4.0, 0, 0]) ** 2, axis=1) <= 36.0).all()
    assert len(s.counts) == o.Size()


def _snap_example():
    pts = np.array([[0.25, -0.5, 3.0], [np.nan, 0.0, 0.0], [-0.0, 1.5, -2.25], [7.0, 7.0, 7.0]], dtype=np.float32)
    return sv.MapSnapshot(0.5, 42.25, 7, np.array([[-3, 0, 2], [0, 0, 0], [1, -(1 << 20), (1 << 20) - 1]], dtype=np.int32),
                          np.array([1, 2, 1], dtype=np.int32), pts)


def test_python_file_round_trip(tmp_path):
    p = str(tmp_path / "a.svnmap")
    s = _snap_example()
    sv.write_map_snapshot(p, s)
    data = open(p, "rb").read()
    assert data[:8] == b"SVNMAP01" and len(data) == 48 + 16 * 3 + 12 * 4
    snapshots_equal(sv.read_map_snapshot(p), s)
    q = str(tmp_path / "b.svnmap")
    sv.write_map_snapshot(q, sv.read_map_snapshot(p))
    assert open(q, "rb").read() == data
    e = sv.MapSnapshot(1.0, 80.0, 20, np.zeros((0, 3), np.int32), np.zeros(0, np.int32), np.zeros((0, 3), np.float32))
    sv.write_map_snapshot(p, e)
    assert len(open(p, "rb").read()) == 48
    snapshots_equal(sv.read_map_snapshot(p), e)


def corrupt_files(tmp_path, good: bytes):
    """(name, path) of files both readers must reject"""
    out = []
    for name, data in (("magic", b"SVNMAP02" + good[8:]), ("version", good[:8] + (2).to_bytes(4, "little") + good[12:]),
                       ("truncated_header", good[:40]), ("truncated_body", good[:-4]), ("trailing_byte", good + b"\0"),
                       ("empty", b"")):
        p = str(tmp_path / f"bad_{name}.svnmap")
        open(p, "wb").write(data)
        out.append((name, p))
    return out


def test_python_reader_rejects(tmp_path):
    p = str(tmp_path / "a.svnmap")
    sv.write_map_snapshot(p, _snap_example())
    for name, bad in corrupt_files(tmp_path, open(p, "rb").read()):
        with pytest.raises(sv.SvnIcpError):
            sv.read_map_snapshot(bad)


FILE_SRC = r"""
#include <cstring>
#include "svnicp/VoxelHashMap.hpp"
int main(int argc, char **argv) {
  try {
    if (argc == 3 && !std::strcmp(argv[1], "write")) {
      svnicp::MapSnapshot s;
      s.voxel_size = 0.5; s.max_range = 42.25; s.max_pointscount = 7;
      s.voxels = {-3, 0, 2, 0, 0, 0, 1, -1048576, 1048575};
      s.counts = {1, 2, 1};
      s.xyz = {0.25f, -0.5f, 3.0f, 1.0f, 0.0f, 0.0f, -0.0f, 1.5f, -2.25f, 7.0f, 7.0f, 7.0f};
      svnicp::write_map_snapshot(argv[2], s);
      return 0;
    }
    if (argc == 4 && !std::strcmp(argv[1], "copy")) {
      svnicp::write_map_snapshot(argv[3], svnicp::read_map_snapshot(argv[2]));
      return 0;
    }
  } catch (const svnicp::Error &e) {
    std::fprintf(stderr, "%s\n", e.what());
    return 3;
  }
  return 2;
}
"""


@pytest.fixture(scope="module")
def snapfile_exe(tmp_path_factory):
    from svn_icp_b200 import build
    lib = build.build()
    d = tmp_path_factory.mktemp("snapfile")
    src, exe = str(d / "snapfile.cpp"), str(d / "snapfile")
    open(src, "w").write(FILE_SRC)
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "svn_icp_b200", "include"), src,
                           "-o", exe, lib, "-Wl,-rpath," + os.path.dirname(lib)])
    return exe


def test_cpp_and_python_files_are_the_same_bytes(tmp_path, snapfile_exe):
    c = str(tmp_path / "c.svnmap")
    subprocess.check_call([snapfile_exe, "write", c])
    s = sv.read_map_snapshot(c)
    want = _snap_example()
    want.points[1, 0] = 1.0  # the C++ example has no NaN literal
    snapshots_equal(s, want)
    assert np.signbit(s.points[2, 0])  # -0.0 kept
    py = str(tmp_path / "py.svnmap")
    sv.write_map_snapshot(py, s)
    assert open(py, "rb").read() == open(c, "rb").read()
    # and the C++ reader / writer reproduces a Python file (NaN included) byte for byte
    sv.write_map_snapshot(py, _snap_example())
    cc = str(tmp_path / "cc.svnmap")
    subprocess.check_call([snapfile_exe, "copy", py, cc])
    assert open(cc, "rb").read() == open(py, "rb").read()


def test_cpp_reader_rejects(tmp_path, snapfile_exe):
    p = str(tmp_path / "a.svnmap")
    sv.write_map_snapshot(p, _snap_example())
    for name, bad in corrupt_files(tmp_path, open(p, "rb").read()):
        r = subprocess.run([snapfile_exe, "copy", bad, str(tmp_path / "out.svnmap")], capture_output=True, text=True)
        assert r.returncode == 3, (name, r.stderr)


MIRROR_SRC = r"""
#include <cstring>
#include "svnicp/VoxelHashMap.hpp"
int main(int argc, char **argv) {
  if (argc != 2) return 2;
  int reached = 0;
  try {
    svnicp::VoxelHashMap m(1.0, 100.0, 20);
    reached = 1;
    std::vector<float> xyz = {0.5f, 0.5f, 0.5f, 1.5f, 2.5f, -3.5f, 0.25f, 0.5f, 0.5f};
    svnicp::InitialMean T0;
    m.AddPointCloud(xyz, T0);
    const svnicp::VoxelHashMap::Snapshot s = m.Export();
    if (s.counts.size() != 2 || s.voxels.size() != 6 || s.xyz.size() != 9) return 4;
    m.Save(argv[1]);
    std::unique_ptr<svnicp::VoxelHashMap> b = svnicp::VoxelHashMap::Load(argv[1], 16);
    const svnicp::VoxelHashMap::Snapshot t = b->Export();
    if (t.voxels != s.voxels || t.counts != s.counts || std::memcmp(t.xyz.data(), s.xyz.data(), 9 * sizeof(float)) != 0) return 5;
    try {
      b->Import(svnicp::MapSnapshot{});  // max_range 80 differs from the map's 100
      return 6;
    } catch (const svnicp::Error &) {
      return 10;
    }
  } catch (const svnicp::Error &) {
  }
  return reached ? 7 : 0;
}
"""


def test_mirror_map_snapshot_compiles(tmp_path):
    from svn_icp_b200 import build
    lib = build.build()
    src, exe = os.path.join(tmp_path, "map_snap.cpp"), os.path.join(tmp_path, "map_snap")
    open(src, "w").write(MIRROR_SRC)
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "svn_icp_b200", "include"), src,
                           "-o", exe, lib, "-Wl,-rpath," + os.path.dirname(lib)])
    import torch
    # without a GPU the constructor throws (0); on a GPU export, save, load and the refused import all run (10)
    assert subprocess.call([exe, os.path.join(tmp_path, "m.svnmap")]) == (10 if torch.cuda.is_available() else 0)
