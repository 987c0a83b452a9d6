// svnicp/VoxelHashMap.hpp -- header-only C++ mirror of the reference's local map (svn-icp/include/core/VoxelHashMap.h:28-72)
// over the C ABI of include/svnicp_b200.h (svnicp_map_*).  Same member names and meaning; the map lives in HBM, and
// GetMap hands back a DEVICE cloud that add_cloud consumes without a host round trip (the reference re-uploads the whole
// map every scan: OdometryPipeline.cpp:577-581).  Poses are passed as svnicp::InitialMean (row-major R, t).
#pragma once
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "svnicp/SVNICP.hpp"

namespace svnicp {

/** A local map's content in canonical form (svnicp_map_export): voxels [V][3] ascending (vx, vy, vz), counts [V], xyz [Npts][3]
 *  with each voxel's points in stored order, and the parameters of the map it came from. */
struct MapSnapshot {
  double voxel_size = 1.0;
  double max_range = 80;
  int max_pointscount = 20;
  std::vector<int32_t> voxels;
  std::vector<int32_t> counts;
  std::vector<float> xyz;
};

/** The snapshot file, shared with the Python mirror: little-endian header "SVNMAP01", u32 version 1, u32 max_pointscount,
 *  f64 voxel_size, f64 max_range, i64 V, i64 Npts; then voxels int32 [V][3], counts int32 [V], xyz float [Npts][3].  No GPU. */
constexpr uint32_t kMapSnapshotVersion = 1;

namespace detail {
inline bool host_is_little_endian() {
  const uint16_t one = 1;
  unsigned char b;
  std::memcpy(&b, &one, 1);
  return b == 1;
}
}  // namespace detail

inline void write_map_snapshot(const std::string &path, const MapSnapshot &s) {
  if (!detail::host_is_little_endian()) throw Error("write_map_snapshot: the file format is little-endian, this host is not");
  if (s.voxels.size() != 3 * s.counts.size() || s.xyz.size() % 3 != 0) throw Error("write_map_snapshot: voxels, counts and xyz disagree");
  std::unique_ptr<FILE, int (*)(FILE *)> f(std::fopen(path.c_str(), "wb"), &std::fclose);
  if (!f) throw Error("write_map_snapshot: cannot open " + path);
  const uint32_t head32[2] = {kMapSnapshotVersion, (uint32_t)s.max_pointscount};
  const double headf[2] = {s.voxel_size, s.max_range};
  const int64_t sizes[2] = {(int64_t)s.counts.size(), (int64_t)(s.xyz.size() / 3)};
  bool ok = std::fwrite("SVNMAP01", 1, 8, f.get()) == 8 && std::fwrite(head32, sizeof(head32), 1, f.get()) == 1 &&
            std::fwrite(headf, sizeof(headf), 1, f.get()) == 1 && std::fwrite(sizes, sizeof(sizes), 1, f.get()) == 1;
  ok = ok && std::fwrite(s.voxels.data(), sizeof(int32_t), s.voxels.size(), f.get()) == s.voxels.size();
  ok = ok && std::fwrite(s.counts.data(), sizeof(int32_t), s.counts.size(), f.get()) == s.counts.size();
  ok = ok && std::fwrite(s.xyz.data(), sizeof(float), s.xyz.size(), f.get()) == s.xyz.size();
  if (!ok || std::fflush(f.get()) != 0) throw Error("write_map_snapshot: cannot write " + path);
}

/** Rejects a wrong magic or version and a file whose length does not match the sizes. */
inline MapSnapshot read_map_snapshot(const std::string &path) {
  if (!detail::host_is_little_endian()) throw Error("read_map_snapshot: the file format is little-endian, this host is not");
  std::unique_ptr<FILE, int (*)(FILE *)> f(std::fopen(path.c_str(), "rb"), &std::fclose);
  if (!f) throw Error("read_map_snapshot: cannot open " + path);
  char magic[8];
  uint32_t head32[2];
  double headf[2];
  int64_t sizes[2];
  if (std::fread(magic, 1, 8, f.get()) != 8 || std::memcmp(magic, "SVNMAP01", 8) != 0) throw Error(path + ": not a map snapshot (magic)");
  if (std::fread(head32, sizeof(head32), 1, f.get()) != 1 || std::fread(headf, sizeof(headf), 1, f.get()) != 1 ||
      std::fread(sizes, sizeof(sizes), 1, f.get()) != 1)
    throw Error(path + ": not a map snapshot (shorter than its header)");
  if (head32[0] != kMapSnapshotVersion) throw Error(path + ": map snapshot version " + std::to_string(head32[0]) + ", this reader knows 1");
  const int64_t V = sizes[0], N = sizes[1];
  if (std::fseek(f.get(), 0, SEEK_END) != 0) throw Error("read_map_snapshot: cannot seek in " + path);
  const long long len = std::ftell(f.get());
  // sizes bounded before they are multiplied: 2^40 points are far beyond any file this could be
  if (V < 0 || N < 0 || V > (1ll << 40) || N > (1ll << 40) || len != 48 + 16 * V + 12 * N)
    throw Error(path + ": map snapshot length does not match V = " + std::to_string(V) + ", Npts = " + std::to_string(N));
  std::fseek(f.get(), 48, SEEK_SET);
  MapSnapshot s;
  s.max_pointscount = (int)head32[1];
  s.voxel_size = headf[0];
  s.max_range = headf[1];
  s.voxels.resize((size_t)V * 3);
  s.counts.resize((size_t)V);
  s.xyz.resize((size_t)N * 3);
  if (std::fread(s.voxels.data(), sizeof(int32_t), s.voxels.size(), f.get()) != s.voxels.size() ||
      std::fread(s.counts.data(), sizeof(int32_t), s.counts.size(), f.get()) != s.counts.size() ||
      std::fread(s.xyz.data(), sizeof(float), s.xyz.size(), f.get()) != s.xyz.size())
    throw Error("read_map_snapshot: cannot read " + path);
  return s;
}

struct VoxelHashMap {
  double voxel_size_ = 1.0;   // VoxelHashMap.h:32-34
  double max_range_ = 80;
  int max_pointscount_ = 20;

  explicit VoxelHashMap(double voxel_size = 1.0, double max_range = 80, int max_pointscount = 20, int64_t capacity_voxels = 1 << 19,
                        int device = -1)
      : voxel_size_(voxel_size), max_range_(max_range), max_pointscount_(max_pointscount) {
    if (svnicp_map_create(&m_, voxel_size, max_range, max_pointscount, capacity_voxels, device) != SVNICP_OK)
      throw Error(std::string("svnicp_map_create: ") + svnicp_map_last_error(nullptr));
  }
  ~VoxelHashMap() {
    if (m_) svnicp_map_destroy(m_);
  }
  VoxelHashMap(const VoxelHashMap &) = delete;
  VoxelHashMap &operator=(const VoxelHashMap &) = delete;

  void Clear() { check(svnicp_map_clear(m_), "Clear"); }  // VoxelHashMap.h:54
  [[nodiscard]] bool Empty() const { return Size() == 0; }
  [[nodiscard]] size_t Size() const {
    int64_t v = 0;
    check(svnicp_map_size(m_, &v, nullptr), "Size");
    return (size_t)v;
  }

  /** AddPointCloud (VoxelHashMap.cpp:22-43): float xyz triples in the sensor frame (pcl::PointXYZI without the intensity) */
  void AddPointCloud(const float *xyz, int64_t n, const InitialMean &new_pose, bool on_device = false) {
    check(svnicp_map_add_cloud(m_, xyz, n, 0, on_device, new_pose.R.data(), new_pose.t.data()), "AddPointCloud");
  }
  void AddPointCloud(const std::vector<float> &xyz, const InitialMean &new_pose) { AddPointCloud(xyz.data(), (int64_t)(xyz.size() / 3), new_pose); }

  /** GetMap() (VoxelHashMap.cpp:45-51): device cloud, valid until the next call on this map */
  CloudView GetMap() {
    const double *p = nullptr;
    int64_t n = 0;
    check(svnicp_map_get(m_, nullptr, 0.0, &p, &n), "GetMap");
    return CloudView{p, n, true};
  }
  /** GetMap(pose, max_range) (VoxelHashMap.cpp:53-63) */
  CloudView GetMap(const InitialMean &pose, const double &max_range) {
    const double *p = nullptr;
    int64_t n = 0;
    check(svnicp_map_get(m_, pose.t.data(), max_range, &p, &n), "GetMap");
    return CloudView{p, n, true};
  }
  /** host copy of the last GetMap result, xyz doubles */
  std::vector<double> Download(const CloudView &last) {
    std::vector<double> v((size_t)last.n * 3);
    check(svnicp_map_download(m_, v.data(), last.n), "Download");
    return v;
  }

  /** Registration objective of a scan at M poses against this map (svnicp_map_evaluate; no reference counterpart).  xyz: n float
   *  xyz triples in the sensor frame (host, or device with on_device).  poses_6xM: [6][M] x = [t ; omega] relative to T0, the
   *  SVN-ICP particle convention (zeros score T0 itself).  Each point's exact nearest map point with d^2 < max_dist (squared
   *  metres, as the registration's threshold).  Returns the result type of SVGDICP::evaluate.  Changes no state of the map. */
  SVGDICP::Evaluation Evaluate(const float *xyz, int64_t n, const InitialMean &T0, const std::vector<double> &poses_6xM, double max_dist,
                               bool want_system = true, bool want_mask = false, bool on_device = false) {
    if (poses_6xM.empty() || poses_6xM.size() % 6 != 0) throw Error("Evaluate: poses must hold 6*M doubles");
    SVGDICP::Evaluation r;
    r.n_poses = (int)(poses_6xM.size() / 6);
    const size_t M = (size_t)r.n_poses;
    std::vector<double> stats(3 * M);
    if (want_system) { r.H.resize(36 * M); r.b.resize(6 * M); }
    if (want_mask && n > 0) r.mask.resize(M * (size_t)n);
    check(svnicp_map_evaluate(m_, xyz, n, 0, on_device, T0.R.data(), T0.t.data(), r.n_poses, poses_6xM.data(), max_dist, stats.data(),
                              want_system ? r.H.data() : nullptr, want_system ? r.b.data() : nullptr,
                              want_mask ? r.mask.data() : nullptr, nullptr),
          "Evaluate");
    for (size_t m = 0; m < M; m++) {
      r.inliers.push_back((int64_t)stats[3 * m]);
      r.fitness.push_back(stats[3 * m + 1]);
      r.rmse.push_back(stats[3 * m + 2]);
    }
    return r;
  }

  /** Result of Search: the k winners, best first (index = flat grid index g, poses [6][k] the grid values relative to T0,
   *  count / fitness / rmse Evaluate's values for them), and with want_counts the score of every grid pose in g order. */
  struct SearchResult {
    int k = 0;
    std::vector<int64_t> index;
    std::vector<double> poses;
    std::vector<int64_t> count;
    std::vector<double> fitness, rmse;
    std::vector<int32_t> counts;
  };
  /** Exact search of a scan over a grid of poses around T0 (svnicp_map_search; no reference counterpart): counts[a] values
   *  x_a(i) = (i - 0.5 (counts[a] - 1)) steps[a] per axis of x = [t ; omega], flat index g with axis 0 fastest.  Score = the
   *  inlier count of Evaluate; ranked by count descending, then g ascending.  Changes no state of the map.  Without want_counts
   *  a grid with translation blocks is searched by branch and bound (SearchInfo), with the same result. */
  SearchResult Search(const float *xyz, int64_t n, const InitialMean &T0, const int32_t (&counts)[6], const double (&steps)[6],
                      double max_dist, int top_k = 1, bool want_counts = false, bool on_device = false) {
    int64_t M = 1;  // capped at 2^31: the ABI refuses larger grids
    for (int a = 0; a < 6; a++) {
      M *= counts[a] > 0 ? counts[a] : 0;
      if (M > INT32_MAX) M = (int64_t)INT32_MAX + 1;
    }
    if (top_k < 1 || (int64_t)top_k > M) throw Error("Search: need 1 <= top_k <= the number of grid poses");
    SearchResult r;
    r.k = top_k;
    r.index.resize((size_t)top_k);
    r.poses.resize(6 * (size_t)top_k);
    std::vector<double> stats(3 * (size_t)top_k);
    if (want_counts && M <= INT32_MAX) r.counts.resize((size_t)M);
    check(svnicp_map_search(m_, xyz, n, 0, on_device, T0.R.data(), T0.t.data(), counts, steps, max_dist, top_k, r.index.data(),
                            r.poses.data(), stats.data(), want_counts ? r.counts.data() : nullptr),
          "Search");
    for (int j = 0; j < top_k; j++) {
      r.count.push_back((int64_t)stats[3 * j]);
      r.fitness.push_back(stats[3 * j + 1]);
      r.rmse.push_back(stats[3 * j + 2]);
    }
    return r;
  }

  /** Result of Refine, per pose in input order: the final x (poses [6][M]), the updates applied, |delta| of the last one, and
   *  Evaluate's inliers / fitness / rmse (and with want_system H [M][36], b [M][6]) at the final x, bit for bit. */
  struct RefineResult {
    int n_poses = 0;
    std::vector<double> poses;
    std::vector<int32_t> iterations;
    std::vector<double> step;
    std::vector<int64_t> inliers;
    std::vector<double> fitness, rmse, H, b;
  };
  /** Gauss-Newton refinement of M pose hypotheses of a scan against this map (svnicp_map_refine; no reference counterpart): up
   *  to `iterations` single-particle SVN-ICP steps per pose on exact correspondences, stopping after the first step with
   *  |delta| < tol.  poses_6xM: [6][M] x relative to T0, as in Evaluate; Search's poses may be passed in unchanged.  Chain two
   *  calls to tighten max_dist.  Changes no state of the map. */
  RefineResult Refine(const float *xyz, int64_t n, const InitialMean &T0, const std::vector<double> &poses_6xM, double max_dist,
                      int iterations = 30, double tol = 1e-5, bool want_system = false, bool on_device = false) {
    if (poses_6xM.empty() || poses_6xM.size() % 6 != 0) throw Error("Refine: poses must hold 6*M doubles");
    RefineResult r;
    r.n_poses = (int)(poses_6xM.size() / 6);
    const size_t M = (size_t)r.n_poses;
    r.poses.resize(6 * M);
    r.iterations.resize(M);
    r.step.resize(M);
    std::vector<double> stats(3 * M);
    if (want_system) { r.H.resize(36 * M); r.b.resize(6 * M); }
    check(svnicp_map_refine(m_, xyz, n, 0, on_device, T0.R.data(), T0.t.data(), r.n_poses, poses_6xM.data(), max_dist, iterations, tol,
                            r.poses.data(), r.iterations.data(), r.step.data(), stats.data(), want_system ? r.H.data() : nullptr,
                            want_system ? r.b.data() : nullptr),
          "Refine");
    for (size_t m = 0; m < M; m++) {
      r.inliers.push_back((int64_t)stats[3 * m]);
      r.fitness.push_back(stats[3 * m + 1]);
      r.rmse.push_back(stats[3 * m + 2]);
    }
    return r;
  }

  /** The work of the last successful Search (svnicp_map_search_info): path 0 counted every pose, path 1 pruned by block bounds */
  struct SearchWork {
    int64_t path = 0, grid_poses = 0, poses_per_block = 0, blocks = 0, blocks_counted = 0, poses_counted = 0, bound_queries = 0,
            violations = 0;
  };
  SearchWork SearchInfo() const {
    int64_t v[8];
    check(svnicp_map_search_info(m_, v), "SearchInfo");
    return SearchWork{v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7]};
  }

  using Snapshot = MapSnapshot;
  /** The content in canonical form (svnicp_map_export; no reference counterpart) */
  Snapshot Export() const {
    int64_t V = 0, N = 0;
    check(svnicp_map_size(m_, &V, &N), "Export");
    Snapshot s;
    s.voxel_size = voxel_size_;
    s.max_range = max_range_;
    s.max_pointscount = max_pointscount_;
    s.voxels.resize((size_t)V * 3);
    s.counts.resize((size_t)V);
    s.xyz.resize((size_t)N * 3);
    check(svnicp_map_export(m_, s.voxels.data(), s.counts.data(), s.xyz.data(), V, N, 0), "Export");
    return s;
  }
  /** Replace the content by a snapshot of a map with the same parameters (svnicp_map_import; all or nothing) */
  void Import(const Snapshot &s) {
    if (s.voxel_size != voxel_size_ || s.max_range != max_range_ || s.max_pointscount != max_pointscount_)
      throw Error("Import: the snapshot's voxel_size, max_range or max_pointscount differ from this map's");
    if (s.voxels.size() != 3 * s.counts.size() || s.xyz.size() % 3 != 0) throw Error("Import: voxels, counts and xyz disagree");
    check(svnicp_map_import(m_, s.voxels.data(), s.counts.data(), s.xyz.data(), (int64_t)s.counts.size(), (int64_t)(s.xyz.size() / 3), 0),
          "Import");
  }
  void Save(const std::string &path) const { write_map_snapshot(path, Export()); }
  /** A new map with the file's parameters, a capacity of at least its voxel count, and its content */
  static std::unique_ptr<VoxelHashMap> Load(const std::string &path, int64_t capacity_voxels = 1 << 19, int device = -1) {
    const Snapshot s = read_map_snapshot(path);
    const int64_t V = (int64_t)s.counts.size();
    std::unique_ptr<VoxelHashMap> m(new VoxelHashMap(s.voxel_size, s.max_range, s.max_pointscount, capacity_voxels > V ? capacity_voxels : V, device));
    m->Import(s);
    return m;
  }

 private:
  void check(int rc, const char *what) const {
    if (rc < 0) throw Error(std::string(what) + ": " + svnicp_map_last_error(m_));
  }
  svnicp_map m_ = nullptr;
};

}  // namespace svnicp
