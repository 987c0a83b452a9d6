// svnicp/VoxelHashMap.hpp -- header-only C++ mirror of the reference's local map (svn-icp/include/core/VoxelHashMap.h:28-72)
// over the C ABI of include/svnicp_b200.h (svnicp_map_*).  Same member names and meaning; the map lives in HBM, and
// GetMap hands back a DEVICE cloud that add_cloud consumes without a host round trip (the reference re-uploads the whole
// map every scan: OdometryPipeline.cpp:577-581).  Poses are passed as svnicp::InitialMean (row-major R, t).
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "svnicp/SVNICP.hpp"

namespace svnicp {

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

 private:
  void check(int rc, const char *what) const {
    if (rc < 0) throw Error(std::string(what) + ": " + svnicp_map_last_error(m_));
  }
  svnicp_map m_ = nullptr;
};

}  // namespace svnicp
