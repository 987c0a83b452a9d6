// SVNICP.hpp -- header-only C++ mirror of the reference's registration classes over the C ABI.
//
// Same class, method and struct names, argument order and return conventions as the reference
// (svn-icp/include/core/SVGDICP.h:41-211, SVNICP.h:25-80), so a caller written against the reference
// (OdometryPipeline.cpp:282-288, 582-607) compiles against this header with its tensor arguments
// replaced by plain buffers:
//   torch::Tensor [N,3] f64 (cuda)  ->  svnicp::CloudView {const double*, int64_t n, bool on_device}
//   torch::Tensor [6,P,1] f64       ->  const std::vector<double>& (6*P, component major)
//   gtsam::Pose3                    ->  svnicp::InitialMean {R row-major 3x3, t}
//   torch::Tensor [6]               ->  std::vector<double> (6)
// Errors: the reference throws c10::Error; this mirror throws svnicp::Error (std::runtime_error) carrying
// svnicp_last_error().  stein_align() returns SteinICPState exactly like the reference.
#pragma once
#include <array>
#include <cstring>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../../include/svnicp_b200.h"

namespace svnicp {

enum CovFilterType { MEAN, MAX_SLIDING_WINDOW, NONE };  // SVGDICP.h:39

struct SteinICPParam {  // SVGDICP.h:41-57, same defaults
  int iterations = 50;
  bool use_minibatch = false;
  int batch_size = 50;
  double lr = 0.02;
  double max_dist = 1.0;
  bool normalize_cloud = true;
  std::string optimizer = "Adam";
  bool check_early_stop = false;
  int convergence_steps = 5;
  double convergence_threshold = 1e-5;
  int KNN_count = 100;
  bool SVN_full_grad = true;
  CovFilterType cov_filter_type = NONE;
};

enum SteinICPState { ALIGN_SUCCESS = 1, NO_OPTIMIZER = 2 };  // SVGDICP.h:59-62

struct ParticleWeightOpt {  // SVNICP.h:25-27
  bool use_weight_mean = false;
};

struct Error : std::runtime_error {
  using std::runtime_error::runtime_error;
};

struct CloudView {
  const double *xyz;  // [n][3] row-major float64
  int64_t n;
  bool on_device = false;
};

struct InitialMean {
  std::array<double, 9> R{1, 0, 0, 0, 1, 0, 0, 0, 1};  // row-major, = gtsam::Pose3::rotation().matrix()
  std::array<double, 3> t{0, 0, 0};
};

// initialize_particles / initialize_particles_gaussian (ICPUtils.cpp:45-75); returns [6][P]
inline std::vector<double> initialize_particles(int particle_count, const std::array<double, 6> &ub, const std::array<double, 6> &lb,
                                                uint64_t seed = 0) {
  std::vector<double> out((size_t)6 * particle_count);
  if (svnicp_initialize_particles(particle_count, ub.data(), lb.data(), seed, out.data()) != SVNICP_OK) throw Error("initialize_particles");
  return out;
}
inline std::vector<double> initialize_particles_gaussian(int particle_count, const std::array<double, 6> &cov, uint64_t seed = 0) {
  std::vector<double> out((size_t)6 * particle_count);
  if (svnicp_initialize_particles_gaussian(particle_count, cov.data(), seed, out.data()) != SVNICP_OK) throw Error("initialize_particles_gaussian");
  return out;
}

class SVGDICP {  // the base interface the node holds (OdometryPipeline.h:125)
 public:
  /** SVGDICP::SVGDICP (SVGDICP.cpp:22-44): the first-order class itself (`class_type: SVGDICP`, OdometryPipeline.cpp:282-288) */
  explicit SVGDICP(const SteinICPParam &parameters, const std::vector<double> &init_pose, int device = -1)
      : SVGDICP(parameters, init_pose, ParticleWeightOpt{}, SVNICP_CLASS_SVGDICP, device) {}
  virtual ~SVGDICP() {
    if (h_ && owned_) svnicp_destroy(h_);
  }
  SVGDICP(const SVGDICP &) = delete;
  SVGDICP &operator=(const SVGDICP &) = delete;

  /** SVGDICP::add_cloud (SVGDICP.cpp:46-62): clouds are copied, the caller may free them immediately. */
  void add_cloud(const CloudView &new_cloud, const CloudView &target, const std::vector<double> &init_pose) {
    if ((int)init_pose.size() != 6 * particle_size_) throw Error("add_cloud: init_pose must hold 6*P doubles (P is fixed at construction)");
    check(svnicp_add_cloud(h_, new_cloud.xyz, new_cloud.n, new_cloud.on_device, target.xyz, target.n, target.on_device, init_pose.data()),
          "add_cloud");
  }
  /** SVGDICP::set_initial_mean (SVGDICP.h:102-110) */
  void set_initial_mean(const InitialMean &pose) { check(svnicp_set_initial_mean(h_, pose.R.data(), pose.t.data()), "set_initial_mean"); }
  /** stein_align (SVNICP.cpp:41-114) */
  virtual SteinICPState stein_align() {
    const int rc = svnicp_align(h_);
    check(rc, "stein_align");
    return static_cast<SteinICPState>(rc);
  }
  std::vector<double> get_particles() const {  // 6P, [6][P] (SVGDICP.cpp:515-520)
    std::vector<double> v((size_t)6 * particle_size_);
    check(svnicp_get_particles(h_, v.data()), "get_particles");
    return v;
  }
  virtual std::vector<double> get_transformation() {
    std::vector<double> v(6);
    check(svnicp_get_transformation(h_, v.data()), "get_transformation");
    return v;
  }
  virtual std::vector<double> get_distribution() {
    std::vector<double> v(6);
    check(svnicp_get_distribution(h_, v.data()), "get_distribution");
    return v;
  }
  virtual std::vector<double> get_cov_matrix() {
    std::vector<double> v(36);
    check(svnicp_get_cov_matrix(h_, v.data()), "get_cov_matrix");
    return v;
  }
  std::vector<std::vector<float>> get_particle_history() const {  // iterations x 6P float (SVGDICP.cpp:526-534)
    int32_t rows = 0;
    check(svnicp_get_particle_history(h_, nullptr, &rows), "get_particle_history");
    std::vector<float> flat((size_t)(rows > 0 ? rows : 1) * 6 * particle_size_);
    check(svnicp_get_particle_history(h_, flat.data(), &rows), "get_particle_history");
    std::vector<std::vector<float>> out;
    for (int i = 0; i < rows; i++) out.emplace_back(flat.begin() + (size_t)i * 6 * particle_size_, flat.begin() + (size_t)(i + 1) * 6 * particle_size_);
    return out;
  }
  virtual std::vector<double> get_particle_weight() {
    std::vector<double> v((size_t)particle_size_);
    check(svnicp_get_particle_weight(h_, v.data()), "get_particle_weight");
    return v;
  }
  std::vector<double> get_runtime() {  // {knn s, update s, finish_iter} (SVGDICP.h:94-96), filled from CUDA events
    std::vector<double> v(3);
    check(svnicp_get_runtime(h_, v.data()), "get_runtime");
    return v;
  }
  void set_k(const int k) { check(svnicp_set_k(h_, k), "set_k"); }
  void set_threshold(const double max_dist) { check(svnicp_set_threshold(h_, max_dist), "set_threshold"); }

  /** Registration objective of the last scan at M poses (svnicp_evaluate; no reference counterpart).  poses_6xM: [6][M] in the
   *  class's particle convention, relative to the initial mean (get_transformation() and zeros are valid).  Per pose: inlier
   *  count, fitness = inlier fraction, inlier RMSE (m); with want_system the Gauss-Newton system H [M][36], b [M][6]; with
   *  want_mask the inlier mask [M][N_s].  Changes no state of the instance. */
  struct Evaluation {
    int n_poses = 0;
    std::vector<int64_t> inliers;
    std::vector<double> fitness, rmse;
    std::vector<double> H, b;
    std::vector<uint8_t> mask;
  };
  Evaluation evaluate(const std::vector<double> &poses_6xM, bool want_system = true, bool want_mask = false) const {
    if (poses_6xM.empty() || poses_6xM.size() % 6 != 0) throw Error("evaluate: poses must hold 6*M doubles");
    Evaluation r;
    r.n_poses = (int)(poses_6xM.size() / 6);
    const size_t M = (size_t)r.n_poses;
    int64_t info[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    check(svnicp_get_scan_info(h_, info), "evaluate");
    std::vector<double> stats(3 * M);
    if (want_system) { r.H.resize(36 * M); r.b.resize(6 * M); }
    if (want_mask) r.mask.resize(M * (size_t)info[0]);
    check(svnicp_evaluate(h_, r.n_poses, poses_6xM.data(), stats.data(), want_system ? r.H.data() : nullptr,
                          want_system ? r.b.data() : nullptr, want_mask ? r.mask.data() : nullptr, nullptr),
          "evaluate");
    for (size_t m = 0; m < M; m++) {
      r.inliers.push_back((int64_t)stats[3 * m]);
      r.fitness.push_back(stats[3 * m + 1]);
      r.rmse.push_back(stats[3 * m + 2]);
    }
    return r;
  }

  svnicp_handle native_handle() const { return h_; }

 protected:
  SVGDICP(const SteinICPParam &p, const std::vector<double> &init_pose, const ParticleWeightOpt &opt, int class_type, int device) {
    if (init_pose.size() % 6 != 0 || init_pose.empty()) throw Error("init_pose must hold 6*P doubles");
    particle_size_ = (int)(init_pose.size() / 6);
    svnicp_params c;
    svnicp_default_params(&c);
    c.iterations = p.iterations;
    c.use_minibatch = p.use_minibatch;
    c.batch_size = p.batch_size;
    c.lr = p.lr;
    c.max_dist = p.max_dist;
    c.normalize_cloud = p.normalize_cloud;
    std::strncpy(c.optimizer, p.optimizer.c_str(), sizeof(c.optimizer) - 1);
    c.check_early_stop = p.check_early_stop;
    c.convergence_steps = p.convergence_steps;
    c.convergence_threshold = p.convergence_threshold;
    c.KNN_count = p.KNN_count;
    c.SVN_full_grad = p.SVN_full_grad;
    c.use_weight_mean = opt.use_weight_mean;
    const int rc = svnicp_create(&h_, &c, particle_size_, init_pose.data(), class_type, device);
    if (rc != SVNICP_OK) throw Error(std::string("svnicp_create: ") + svnicp_last_error(nullptr));
  }
  void check(int rc, const char *what) const {
    if (rc < 0) throw Error(std::string(what) + ": " + svnicp_last_error(h_));
  }
  /** a view of a handle owned by someone else (SVNICPBatch) */
  SVGDICP(svnicp_handle borrowed, int particle_size) : h_(borrowed), particle_size_(particle_size), owned_(false) {}
  svnicp_handle h_ = nullptr;
  int particle_size_ = 0;
  bool owned_ = true;
  friend class SVNICPBatch;
};

class SVNICP final : public SVGDICP {  // SVNICP.h:29-80
 public:
  explicit SVNICP(const SteinICPParam &param, const std::vector<double> &init_pose, const ParticleWeightOpt &opt = {}, int device = -1)
      : SVGDICP(param, init_pose, opt, SVNICP_CLASS_SVNICP, device) {}

 private:
  SVNICP(svnicp_handle borrowed, int particle_size) : SVGDICP(borrowed, particle_size) {}
  friend class SVNICPBatch;
};

/** The hand-off after the getters in ICP mode: updater_ (OdometryPipeline.cpp:37-45) with tensor2gtsamPose3 (ICPUtils.cpp:84-98):
 *  pose = initial_guess * Pose3(Rot3::Expmap(mean[3:6]), mean[0:3]), mean = get_transformation(). */
inline InitialMean compose_pose(const InitialMean &initial_guess, const std::vector<double> &mean6) {
  InitialMean out;
  if (mean6.size() != 6 || svnicp_pose_compose(initial_guess.R.data(), initial_guess.t.data(), mean6.data(), out.R.data(), out.t.data()) != SVNICP_OK)
    throw Error("compose_pose: mean must hold 6 doubles");
  return out;
}

/** Throughput mode (BASELINE.json configs[3]; no reference counterpart): S independent SVN-ICP streams on one GPU.  stream(s)
 *  is an ordinary SVNICP bound to stream s (add_cloud / set_initial_mean / getters); stein_align() runs the scans of all streams
 *  interleaved so that they overlap on the GPU.  Every stream's result is bit-identical to SVNICP::stein_align on its own. */
class SVNICPBatch {
 public:
  /** init_poses: [S][6][P] */
  SVNICPBatch(const SteinICPParam &p, int n_streams, int particle_size, const std::vector<double> &init_poses, int device = -1) {
    if ((int64_t)init_poses.size() != (int64_t)n_streams * 6 * particle_size) throw Error("SVNICPBatch: init_poses must hold S*6*P doubles");
    svnicp_params c;
    svnicp_default_params(&c);
    c.iterations = p.iterations;
    c.lr = p.lr;
    c.max_dist = p.max_dist;
    c.check_early_stop = p.check_early_stop;
    c.convergence_threshold = p.convergence_threshold;
    c.KNN_count = p.KNN_count;
    c.SVN_full_grad = p.SVN_full_grad;
    if (svnicp_batch_create(&b_, &c, n_streams, particle_size, init_poses.data(), device) != SVNICP_OK)
      throw Error(std::string("svnicp_batch_create: ") + svnicp_last_error(nullptr));
    for (int s = 0; s < n_streams; s++) streams_.emplace_back(new SVNICP(svnicp_batch_stream(b_, s), particle_size));
  }
  ~SVNICPBatch() {
    streams_.clear();
    if (b_) svnicp_batch_destroy(b_);
  }
  SVNICPBatch(const SVNICPBatch &) = delete;
  SVNICPBatch &operator=(const SVNICPBatch &) = delete;
  int size() const { return (int)streams_.size(); }
  SVNICP &stream(int s) { return *streams_.at((size_t)s); }
  std::vector<SteinICPState> stein_align() {
    std::vector<int32_t> st(streams_.size());
    if (svnicp_batch_align(b_, st.data()) < 0) throw Error(std::string("batch stein_align: ") + svnicp_batch_last_error(b_));
    std::vector<SteinICPState> out;
    for (int32_t v : st) out.push_back(static_cast<SteinICPState>(v));
    return out;
  }

 private:
  svnicp_batch b_ = nullptr;
  std::vector<std::unique_ptr<SVNICP>> streams_;
};

}  // namespace svnicp
