// capi.cu -- the C ABI (include/svnicp_b200.h) and the host-side scan driver.
//
// Host logic mirrors the call order the reference's caller uses (OdometryPipeline.cpp:582-607):
// add_cloud -> set_initial_mean -> stein_align -> getters.  Everything heavy is a kernel launch on one
// CUDA stream; the host only sequences launches, one ncclAllGather per iteration when sharded, and one
// small device->host copy at the end of the scan.  No CPU compute path exists.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <math.h>
#include <nccl.h>
#include <stdarg.h>
#include <stdio.h>
#include <time.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <string>
#include <vector>

#include "../../include/svnicp_b200.h"
#include "common.cuh"
#include "kernels.h"

using namespace svn;

static thread_local std::string g_create_error;

// ---- NCCL through dlopen (no link-time dependency; torch's bundled libnccl is reused when loaded) ----
struct NcclApi {
  void *lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  const char *(*GetErrorString)(ncclResult_t) = nullptr;
  bool load(std::string &err) {
    if (lib) return true;
    const char *names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char *n : names) {
      lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
      if (lib) break;
    }
    if (!lib) { err = std::string("cannot dlopen libnccl.so.2: ") + dlerror(); return false; }
    GetUniqueId = (decltype(GetUniqueId))dlsym(lib, "ncclGetUniqueId");
    CommInitRank = (decltype(CommInitRank))dlsym(lib, "ncclCommInitRank");
    AllGather = (decltype(AllGather))dlsym(lib, "ncclAllGather");
    CommDestroy = (decltype(CommDestroy))dlsym(lib, "ncclCommDestroy");
    GetErrorString = (decltype(GetErrorString))dlsym(lib, "ncclGetErrorString");
    if (!GetUniqueId || !CommInitRank || !AllGather || !CommDestroy || !GetErrorString) { err = "libnccl lacks required symbols"; return false; }
    return true;
  }
};
static NcclApi g_nccl;

template <class T>
struct DevBuf {
  T *p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t n, bool zero = false) {
    if (n <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = n + n / 8 + 64;
    cudaError_t e = cudaMalloc((void **)&p, want * sizeof(T));
    if (e != cudaSuccess) return e;
    cap = want;
    if (zero) e = cudaMemset(p, 0, want * sizeof(T));
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct svnicp_handle_t {
  svnicp_params prm;
  int class_type = 0;
  int device = 0;
  int sm_count = 148;
  int P = 0, p_lo = 0, P_l = 0, P_pad = 0, P_l_max = 0;
  int rank = 0, n_ranks = 1;
  ncclComm_t comm = nullptr;
  cudaStream_t own_stream = nullptr, stream = nullptr;
  // SVN-ICP class: k_head runs on a high-priority side stream and overlaps the correspondence + Gauss-Newton pass
  cudaStream_t head_stream = nullptr;
  cudaEvent_t ev_x = nullptr, ev_head = nullptr;
  // small problems: iterations >= 1 run as two CUDA graphs (one per list-buffer parity), see align_step
  cudaGraphExec_t gexec[2] = {nullptr, nullptr};
  int glaunches[2] = {0, 0};
  bool graph_off = false;  // a capture failed once: direct launches for the rest of the handle's life
  cudaEvent_t ev_cfork = nullptr, ev_chead = nullptr;
  // record block: [2][rec_stride] doubles (double buffered by iteration parity) + the peer-exchange flag block; one cudaMalloc,
  // exported to the other ranks through CUDA IPC when sharded
  unsigned char *shared_blk = nullptr;
  size_t rec_records = 0, rec_stride = 0;
  double *rec = nullptr;
  unsigned *flags_dev = nullptr;
  void *peer_base[MAX_RANKS] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  bool peer_mode = false;  // sharded: peer-memory exchange (true) or one ncclAllGather per iteration (false)
  unsigned seq = 0;        // sequence number of the last published exchange (monotonic over scans, identical on every rank)
  PeerTable pt;
  std::string err;
  int K = 100;
  double max_dist = 1.0;
  // scan inputs
  int64_t n_s = 0, n_t = 0;
  int n_pad = 0;
  bool have_cloud = false, aligned = false, shape_dirty = false;
  ScanConst sc;
  // device buffers
  DevBuf<double> src64, tgt64, q0, sxyz, R, t, dnorm, part, xs, delta, Hbar_inv, stats, particles, init_pose, prep_scratch_d;
  DevBuf<int> prep_scratch_i;
  DevBuf<double> stamps;  // k_tail phase stamps of the last iteration (profiling on)
  // SVGD-ICP class state (class_type = SVGDICP): parameters, pose_particles_ carried between scans, optimizer moments
  DevBuf<double> pose6, prev, opt_state;
  int optimizer = -1;
  DevBuf<float4> sp, cand, clist;
  // list reuse across iterations (k_filter): second list buffer, true list lengths and the balls the lists are exact for
  DevBuf<float4> clist2, ball[2];
  DevBuf<float4> hdr, hdr2;  // row headers of the pruned lists (ping-pong with the lists)
  DevBuf<int> cbase[2];
  int filter_reuse = 1;
  // internal particle order (compute_particle_order): internal index i holds the caller's particle perm[i]
  std::vector<int> perm;
  std::vector<double> perm_stage;
  bool permuted = false;
  int rows_per_rank = 0;
  DevBuf<int> counts, starts, fill, pt_slot, sidx, misc, cand_idx;
  int Kp = 100;  // misc: [0] cursor, [1] fallback count
  DevBuf<unsigned long long> keys, kept_hist;
  DevBuf<float> xf, history, dbg_xf;
  DevBuf<unsigned> hist;
  DevBuf<Ctrl> ctrl;
  DevBuf<int32_t> dbg_idx, med_path;
  DevBuf<uint8_t> dbg_mask;
  // pinned host mirrors
  double *h_stats = nullptr;      // 48
  double *h_particles = nullptr;  // 6P
  float *h_history = nullptr;     // I*6*P
  Ctrl *h_ctrl = nullptr;
  int *h_stop = nullptr;          // per-iteration stop snapshots
  unsigned long long *h_kept = nullptr;
  int32_t *h_med = nullptr;       // per-iteration median path (svnicp_get_median_paths)
  size_t h_hist_cap = 0, h_stop_cap = 0;
  std::vector<cudaEvent_t> iter_events;
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  // results
  int iters_done = 0;
  int enqueued_iters = 0;
  double ms_setup = 0, ms_iter = 0, ms_epi = 0, ms_total = 0;
  int64_t launches = 0;
  int fallback_queries = 0;
  // optional per-phase device timing (svnicp_set_profiling): events around every launch group
  int profile = 0;
  std::vector<cudaEvent_t> prof_events;  // 7 per iteration
  double phase_ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};  // prep, filter, gn, finalize, gather, stein(decide+median+stein+update), setup, iterations executed
  // launch shape
  int TB = 16, stages = 3, n_slices = 1, n_pgroups = 1, PG = 512, RG = 1;
  size_t gn_smem = 0;
  // svnicp_evaluate: the candidate table (cand, sp, R0, K) of the last stein_align is still the scan's current one -- set by a
  // completed stein_align, cleared by add_cloud / set_initial_mean / set_k / init_sharding; and the evaluation's own scratch
  bool eval_ok = false;
  DevBuf<double> ev_pose, ev_R, ev_part, ev_out;
  DevBuf<float> ev_xf;
  DevBuf<uint8_t> ev_mask;
  DevBuf<int32_t> ev_idx;
};

static int fail(svnicp_handle h, int code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (h) h->err = buf;
  else g_create_error = buf;
  return code;
}

#define CU(call)                                                                                              \
  do {                                                                                                        \
    cudaError_t e__ = (call);                                                                                 \
    if (e__ != cudaSuccess)                                                                                   \
      return fail(h, e__ == cudaErrorMemoryAllocation ? SVNICP_ERR_OOM : SVNICP_ERR_CUDA, "%s: %s (%s:%d)", #call, \
                  cudaGetErrorString(e__), __FILE__, __LINE__);                                               \
  } while (0)

#define NC(call)                                                                                         \
  do {                                                                                                   \
    ncclResult_t r__ = (call);                                                                           \
    if (r__ != ncclSuccess) return fail(h, SVNICP_ERR_NCCL, "%s: %s", #call, g_nccl.GetErrorString(r__)); \
  } while (0)

extern "C" {

int svnicp_abi_version(void) { return SVNICP_B200_ABI_VERSION; }

void svnicp_default_params(svnicp_params *p) {
  memset(p, 0, sizeof(*p));
  p->iterations = 50;
  p->use_minibatch = 0;
  p->batch_size = 50;
  p->lr = 0.02;
  p->max_dist = 1.0;
  p->normalize_cloud = 1;
  strcpy(p->optimizer, "Adam");
  p->check_early_stop = 0;
  p->convergence_steps = 5;
  p->convergence_threshold = 1e-5;
  p->KNN_count = 100;
  p->SVN_full_grad = 1;
  p->use_weight_mean = 0;
  p->grid_cell = 0.0;
  p->debug_corr = 0;
  p->flags = 0;
  p->gn_stages = 0;
  p->gn_smem_kb = 0;
}

const char *svnicp_last_error(svnicp_handle h) { return h ? h->err.c_str() : g_create_error.c_str(); }

static void set_slice(svnicp_handle h) {
  h->P_l_max = (h->P + h->n_ranks - 1) / h->n_ranks;
  h->P_pad = h->P_l_max * h->n_ranks;
  h->p_lo = h->rank * h->P_l_max;
  int hi = h->p_lo + h->P_l_max;
  if (hi > h->P) hi = h->P;
  h->P_l = hi > h->p_lo ? hi - h->p_lo : 0;
}

static SvgdArgs svgd_args(svnicp_handle h) {
  SvgdArgs s;
  s.P = h->P; s.p_lo = h->p_lo; s.P_l = h->P_l;
  s.optimizer = h->optimizer; s.lr = h->prm.lr;
  s.pose6 = h->pose6.p; s.prev = h->prev.p; s.opt_state = h->opt_state.p;
  return s;
}

// Internal particle order.  The particle -> thread (and, sharded, particle -> GPU) assignment is free, and k_gn's exact early
// exit is a WARP vote: 32 particles that sit close together in pose space agree earlier, and a rank whose slice is a compact
// cluster gets a smaller pruning ball.  So the particles are laid out in Morton order of (x, y, yaw) quantised to 3 bits
// each (measured at configs[1]: k_gn 30.7 -> 28.4 ms per scan); every getter maps back to the caller's order.  The Stein step
// sums over all particles either way; only the order of its fp64 sums changes.  SVNICP_FLAG_NO_PARTICLE_SORT keeps the
// caller's order (A/B measurements).  Not applied to the SVGD-ICP class (its pose_particles_ state spans scans).
static void compute_particle_order(svnicp_handle h, const double *init_pose) {
  const int P = h->P;
  h->perm.resize(P);
  for (int p = 0; p < P; p++) h->perm[p] = p;
  h->permuted = false;
  // Sharded handles: the order is applied INSIDE each rank's slice, so every rank keeps the same (representative) particles
  // it had before.  Measured on 8 GPUs at configs[1] with the order applied ACROSS ranks instead: each slice becomes a compact
  // cluster (kept candidates 72 -> 47, k_gn 4.34 -> 3.94 ms per scan) but the clusters differ in cost and the wait at the
  // per-iteration all-gather grows from 0.9 to 2.2 ms: 95.6 -> 90.5 scans/s.
  if (!init_pose || P < 64 || h->class_type != SVNICP_CLASS_SVNICP || (h->prm.flags & SVNICP_FLAG_NO_PARTICLE_SORT)) return;
  const int comps[3] = {0, 1, 5};
  std::vector<int> code(P, 0);
  for (int blk = 0; blk < h->n_ranks; blk++) {  // identical on every rank: depends on init_pose and the slice bounds only
    const int b_lo = blk * h->P_l_max, b_hi = std::min(P, b_lo + h->P_l_max);
    if (b_hi - b_lo < 64) continue;
    for (int j = 0; j < 3; j++) {
      const double *v = init_pose + (size_t)comps[j] * P;
      double lo = v[b_lo], hi = v[b_lo];
      for (int p = b_lo + 1; p < b_hi; p++) { lo = v[p] < lo ? v[p] : lo; hi = v[p] > hi ? v[p] : hi; }
      if (!(hi > lo) || !std::isfinite(hi - lo)) continue;
      for (int p = b_lo; p < b_hi; p++) {
        int q = (int)((v[p] - lo) / (hi - lo) * 8.0);
        q = q < 0 ? 0 : (q > 7 ? 7 : q);
        for (int b = 0; b < 3; b++) code[p] |= ((q >> b) & 1) << (3 * b + j);
      }
    }
    std::stable_sort(h->perm.begin() + b_lo, h->perm.begin() + b_hi, [&](int a, int b) { return code[a] < code[b]; });
  }
  for (int p = 0; p < P; p++)
    if (h->perm[p] != p) { h->permuted = true; break; }
}

static int upload_particles(svnicp_handle h, const double *init_pose) {
  const size_t n = (size_t)6 * h->P;
  CU(h->init_pose.ensure(n));
  compute_particle_order(h, init_pose);
  if (init_pose && h->permuted) {
    h->perm_stage.resize(n);
    for (int c = 0; c < 6; c++)
      for (int i = 0; i < h->P; i++) h->perm_stage[(size_t)c * h->P + i] = init_pose[(size_t)c * h->P + h->perm[i]];
    CU(cudaMemcpyAsync(h->init_pose.p, h->perm_stage.data(), n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  } else if (init_pose) CU(cudaMemcpyAsync(h->init_pose.p, init_pose, n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  else CU(cudaMemsetAsync(h->init_pose.p, 0, n * sizeof(double), h->stream));
  if (h->class_type == SVNICP_CLASS_SVGDICP) {
    SvgdArgs s = svgd_args(h);
    launch_svgd_init(s, h->init_pose.p, h->R.p, h->t.p, h->dnorm.p, h->ctrl.p, h->stream);
  } else {
    launch_init_particles(h->R.p, h->t.p, h->init_pose.p, h->P, h->dnorm.p, h->p_lo, h->P_l, h->ctrl.p, h->stream);
  }
  CU(cudaGetLastError());
  // the copy source is caller memory: finish before returning (the reference clones synchronously too)
  CU(cudaStreamSynchronize(h->stream));
  return SVNICP_OK;
}

static int alloc_particle_state(svnicp_handle h) {
  const size_t P = (size_t)h->P_pad;
  CU(h->R.ensure(9 * P, true));
  CU(h->t.ensure(3 * P, true));
  CU(h->dnorm.ensure(P, true));
  if (!h->shared_blk) {
    // sized once for any later sharding (P_pad <= P + n_ranks - 1): never reallocated, so IPC mappings stay valid
    h->rec_records = (((size_t)h->P + MAX_RANKS + REC_TILE_PAD - 1) / REC_TILE_PAD) * REC_TILE_PAD + REC_TILE_PAD;
    h->rec_stride = h->rec_records * REC;
    const size_t bytes = 2 * h->rec_stride * sizeof(double) + 256;
    CU(cudaMalloc((void **)&h->shared_blk, bytes));
    CU(cudaMemset(h->shared_blk, 0, bytes));
    h->rec = reinterpret_cast<double *>(h->shared_blk);
    h->flags_dev = reinterpret_cast<unsigned *>(h->shared_blk + 2 * h->rec_stride * sizeof(double));
  }
  memset(&h->pt, 0, sizeof(h->pt));
  h->pt.n_ranks = 1; h->pt.rank = 0;
  h->pt.rec[0] = h->rec; h->pt.flag[0] = h->flags_dev;
  h->pt.timeout_ns = 4000000000ull;
  CU(h->xs.ensure(6 * P));  // SoA copy of x at the head of the iteration (k_head_*)
  CU(h->delta.ensure(6 * P, true));
  CU(h->Hbar_inv.ensure(36));
  CU(h->stats.ensure(48));
  CU(h->particles.ensure(6 * P));
  CU(h->xf.ensure(12 * P));
  CU(h->hist.ensure((size_t)2 * MED_PASSES * MED_BINS, true));  // fast-path scratch + radix histograms (k_head_*)
  CU(h->prep_scratch_d.ensure((size_t)(h->P_l_max > h->sm_count ? h->P_l_max : h->sm_count) * 12 + 64, true));  // per-CTA centre partials of k_tail
  CU(h->prep_scratch_i.ensure(PRUNE_BINS + 8, true));
  CU(h->stamps.ensure(8, true));
  CU(h->ctrl.ensure(1, true));
  CU(h->misc.ensure(8, true));
  const size_t I = (size_t)(h->prm.iterations > 0 ? h->prm.iterations : 1);
  CU(h->history.ensure(I * 6 * h->P));
  CU(h->kept_hist.ensure(I + 2, true));
  CU(h->med_path.ensure(I + 2));
  if (h->class_type == SVNICP_CLASS_SVGDICP) {
    CU(h->pose6.ensure(6 * P, true));
    CU(h->prev.ensure(6 * P, true));
    CU(h->opt_state.ensure(12 * (size_t)(h->P_l_max > 0 ? h->P_l_max : 1), true));
  }
  return SVNICP_OK;
}

static int parse_optimizer(const char *name) {  // SVGDICP.cpp:142-170
  char buf[17];
  memcpy(buf, name, 16);
  buf[16] = 0;
  if (!strcmp(buf, "Adam")) return SVGD_OPT_ADAM;
  if (!strcmp(buf, "RMSprop")) return SVGD_OPT_RMSPROP;
  if (!strcmp(buf, "SGD")) return SVGD_OPT_SGD;
  if (!strcmp(buf, "Adagrad")) return SVGD_OPT_ADAGRAD;
  return -1;  // "No optimizer chosen": stein_align returns NO_OPTIMIZER
}

int svnicp_create(svnicp_handle *out, const svnicp_params *params, int particle_count, const double *init_pose, int class_type,
                  int device) {
  if (!out || !params) return fail(nullptr, SVNICP_ERR_INVALID, "null argument");
  *out = nullptr;
  if (particle_count < 1) return fail(nullptr, SVNICP_ERR_INVALID, "particle_count must be >= 1");
  if (particle_count > SVNICP_MAX_PARTICLES)  // k_head_* count the P^2 pairwise distances in 32-bit histogram bins (tail2.cu)
    return fail(nullptr, SVNICP_ERR_INVALID,
                "particle_count %d exceeds %d: the bandwidth median counts the P^2 pairwise distances in 32-bit histograms",
                particle_count, SVNICP_MAX_PARTICLES);
  if (class_type != SVNICP_CLASS_SVNICP && class_type != SVNICP_CLASS_SVGDICP)
    return fail(nullptr, SVNICP_ERR_INVALID, "class_type must be SVNICP_CLASS_SVNICP or SVNICP_CLASS_SVGDICP");
  if (params->use_minibatch)
    return fail(nullptr, SVNICP_ERR_INVALID, "use_minibatch is not supported (the reference never enables it, SVGDICP.cpp:178-185)");
  if (params->KNN_count < 1 || params->KNN_count > 256) return fail(nullptr, SVNICP_ERR_INVALID, "KNN_count must be in [1,256]");
  if (params->iterations < 0) return fail(nullptr, SVNICP_ERR_INVALID, "iterations must be >= 0");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(nullptr, SVNICP_ERR_NO_DEVICE, "no CUDA device: this library has no CPU fallback");
  if (device < 0) cudaGetDevice(&device);
  if (device >= ndev) return fail(nullptr, SVNICP_ERR_NO_DEVICE, "device %d out of range (%d devices)", device, ndev);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return fail(nullptr, SVNICP_ERR_CUDA, "cudaGetDeviceProperties failed");
  if (prop.major != 10) return fail(nullptr, SVNICP_ERR_NO_DEVICE, "device %d is sm_%d%d; kernels are built for sm_100a only", device, prop.major, prop.minor);
  svnicp_handle h = new svnicp_handle_t();
  h->prm = *params;
  h->class_type = class_type;
  h->optimizer = parse_optimizer(params->optimizer);
  h->device = device;
  h->sm_count = prop.multiProcessorCount;
  h->P = particle_count;
  h->K = params->KNN_count;
  h->max_dist = params->max_dist;
  memset(&h->sc, 0, sizeof(h->sc));
  h->sc.R0[0] = h->sc.R0[4] = h->sc.R0[8] = 1.0;  // SVGDICP.cpp:38-39
  set_slice(h);
  int rc = SVNICP_OK;
  auto body = [&]() -> int {
    CU(cudaSetDevice(device));
    CU(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
    h->stream = h->own_stream;
    {
      int lo = 0, hi = 0;
      CU(cudaDeviceGetStreamPriorityRange(&lo, &hi));
      CU(cudaStreamCreateWithPriority(&h->head_stream, cudaStreamNonBlocking, hi));
    }
    CU(cudaEventCreateWithFlags(&h->ev_x, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&h->ev_head, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&h->ev_cfork, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&h->ev_chead, cudaEventDisableTiming));
    for (int i = 0; i < 4; i++) CU(cudaEventCreate(&h->ev[i]));
    init_iter_kernels();
    init_eval_kernels();
    CU(cudaGetLastError());
    int r = alloc_particle_state(h);
    if (r) return r;
    CU(cudaMallocHost((void **)&h->h_stats, 48 * sizeof(double)));
    CU(cudaMallocHost((void **)&h->h_particles, (size_t)6 * h->P * sizeof(double)));
    CU(cudaMallocHost((void **)&h->h_ctrl, sizeof(Ctrl)));
    memset(h->h_stats, 0, 48 * sizeof(double));
    memset(h->h_particles, 0, (size_t)6 * h->P * sizeof(double));
    if (h->class_type == SVNICP_CLASS_SVGDICP && init_pose) {
      // pose_particles_ as the constructor leaves it (SVGDICP.cpp:33-35): add_cloud never refreshes it
      std::vector<double> pp((size_t)6 * h->P);
      for (int p = 0; p < h->P; p++)
        for (int c = 0; c < 6; c++) pp[(size_t)p * 6 + c] = init_pose[(size_t)c * h->P + p];
      CU(cudaMemcpy(h->prev.p, pp.data(), pp.size() * sizeof(double), cudaMemcpyHostToDevice));
    }
    return upload_particles(h, init_pose);
  };
  rc = body();
  if (rc != SVNICP_OK) {
    g_create_error = h->err;
    svnicp_destroy(h);
    return rc;
  }
  *out = h;
  return SVNICP_OK;
}

void svnicp_destroy(svnicp_handle h) {
  if (!h) return;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  if (h->head_stream) cudaStreamSynchronize(h->head_stream);
  for (int r = 0; r < MAX_RANKS; r++)
    if (h->peer_base[r]) cudaIpcCloseMemHandle(h->peer_base[r]);
  if (h->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm);
  if (h->shared_blk) cudaFree(h->shared_blk);
  if (h->ev_x) cudaEventDestroy(h->ev_x);
  if (h->ev_head) cudaEventDestroy(h->ev_head);
  if (h->ev_cfork) cudaEventDestroy(h->ev_cfork);
  if (h->ev_chead) cudaEventDestroy(h->ev_chead);
  for (int q = 0; q < 2; q++)
    if (h->gexec[q]) cudaGraphExecDestroy(h->gexec[q]);
  if (h->head_stream) cudaStreamDestroy(h->head_stream);
  DevBuf<double> *d[] = {&h->src64, &h->tgt64, &h->q0, &h->sxyz, &h->R, &h->t, &h->dnorm, &h->part, &h->xs, &h->delta,
                         &h->Hbar_inv, &h->stats, &h->particles, &h->init_pose, &h->prep_scratch_d, &h->pose6, &h->prev, &h->opt_state};
  h->prep_scratch_i.release();
  h->stamps.release();
  for (auto *b : d) b->release();
  h->sp.release(); h->cand.release(); h->clist.release();
  h->clist2.release(); h->hdr.release(); h->hdr2.release();
  for (int i = 0; i < 2; i++) { h->ball[i].release(); h->cbase[i].release(); }
  h->cand_idx.release();
  h->counts.release(); h->starts.release(); h->fill.release(); h->pt_slot.release(); h->sidx.release(); h->misc.release();
  h->keys.release(); h->kept_hist.release(); h->med_path.release(); h->xf.release(); h->dbg_xf.release(); h->history.release(); h->hist.release(); h->ctrl.release();
  h->dbg_idx.release(); h->dbg_mask.release();
  h->ev_pose.release(); h->ev_R.release(); h->ev_part.release(); h->ev_out.release(); h->ev_xf.release(); h->ev_mask.release(); h->ev_idx.release();
  if (h->h_stats) cudaFreeHost(h->h_stats);
  if (h->h_particles) cudaFreeHost(h->h_particles);
  if (h->h_history) cudaFreeHost(h->h_history);
  if (h->h_ctrl) cudaFreeHost(h->h_ctrl);
  if (h->h_stop) cudaFreeHost(h->h_stop);
  if (h->h_kept) cudaFreeHost(h->h_kept);
  if (h->h_med) cudaFreeHost(h->h_med);
  for (auto e : h->iter_events) cudaEventDestroy(e);
  for (auto e : h->prof_events) cudaEventDestroy(e);
  for (int i = 0; i < 4; i++) if (h->ev[i]) cudaEventDestroy(h->ev[i]);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  delete h;
}

int svnicp_set_stream(svnicp_handle h, void *cuda_stream) {
  if (!h) return SVNICP_ERR_INVALID;
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  h->stream = cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream;
  return SVNICP_OK;
}

int svnicp_nccl_unique_id(void *id128) {
  std::string err;
  if (!id128) return SVNICP_ERR_INVALID;
  if (!g_nccl.load(err)) return fail(nullptr, SVNICP_ERR_NCCL, "%s", err.c_str());
  ncclUniqueId id;
  ncclResult_t r = g_nccl.GetUniqueId(&id);
  if (r != ncclSuccess) return fail(nullptr, SVNICP_ERR_NCCL, "ncclGetUniqueId: %s", g_nccl.GetErrorString(r));
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId size");
  memcpy(id128, &id, 128);
  return SVNICP_OK;
}

int svnicp_init_sharding(svnicp_handle h, const void *unique_id128, int rank, int n_ranks) {
  if (!h || !unique_id128) return SVNICP_ERR_INVALID;
  if (n_ranks < 1 || rank < 0 || rank >= n_ranks) return fail(h, SVNICP_ERR_INVALID, "bad rank %d / %d", rank, n_ranks);
  if (h->P < n_ranks) return fail(h, SVNICP_ERR_INVALID, "need at least one particle per rank (P=%d, ranks=%d)", h->P, n_ranks);
  if (h->comm) return fail(h, SVNICP_ERR_INVALID, "sharding already initialised");
  CU(cudaSetDevice(h->device));
  if (n_ranks > 1) {
    std::string err;
    if (!g_nccl.load(err)) return fail(h, SVNICP_ERR_NCCL, "%s", err.c_str());
    ncclUniqueId id;
    memcpy(&id, unique_id128, 128);
    NC(g_nccl.CommInitRank(&h->comm, n_ranks, id, rank));
  }
  h->rank = rank;
  h->n_ranks = n_ranks;
  set_slice(h);
  if ((h->P_l_max * n_ranks - h->P) >= h->P_l_max) return fail(h, SVNICP_ERR_INVALID, "P=%d leaves a rank without particles", h->P);
  int r = alloc_particle_state(h);
  if (r) return r;
  h->have_cloud = false;
  h->eval_ok = false;
  h->peer_mode = false;
  if (n_ranks > 1 && n_ranks <= MAX_RANKS && h->class_type == SVNICP_CLASS_SVNICP && !(h->prm.flags & SVNICP_FLAG_NCCL_GATHER)) {
    // Peer-memory exchange: map every rank's record block here through CUDA IPC (handles travel over the NCCL communicator
    // that exists anyway).  Any failure on any rank -> all ranks fall back to one ncclAllGather per iteration.
    struct Slot { cudaIpcMemHandle_t hdl; int ok; int pad[15]; };
    static_assert(sizeof(Slot) == 128, "Slot size");
    Slot *dev = nullptr;
    std::vector<Slot> host((size_t)n_ranks);
    CU(cudaMalloc((void **)&dev, sizeof(Slot) * n_ranks));
    Slot mine;
    memset(&mine, 0, sizeof(mine));
    mine.ok = cudaIpcGetMemHandle(&mine.hdl, h->shared_blk) == cudaSuccess ? 1 : 0;
    if (!mine.ok) cudaGetLastError();
    CU(cudaMemcpyAsync(dev + rank, &mine, sizeof(Slot), cudaMemcpyHostToDevice, h->stream));
    NC(g_nccl.AllGather(dev + rank, dev, sizeof(Slot), ncclChar, h->comm, h->stream));
    CU(cudaMemcpyAsync(host.data(), dev, sizeof(Slot) * n_ranks, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    int ok = 1;
    for (int q = 0; q < n_ranks; q++) ok &= host[q].ok;
    if (ok)
      for (int q = 0; q < n_ranks && ok; q++) {
        if (q == rank) continue;
        if (cudaIpcOpenMemHandle(&h->peer_base[q], host[q].hdl, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
          cudaGetLastError();
          h->peer_base[q] = nullptr;
          ok = 0;
        }
      }
    // second round: everybody must have mapped everybody
    mine.ok = ok;
    CU(cudaMemcpyAsync(dev + rank, &mine, sizeof(Slot), cudaMemcpyHostToDevice, h->stream));
    NC(g_nccl.AllGather(dev + rank, dev, sizeof(Slot), ncclChar, h->comm, h->stream));
    CU(cudaMemcpyAsync(host.data(), dev, sizeof(Slot) * n_ranks, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    cudaFree(dev);
    for (int q = 0; q < n_ranks; q++) ok &= host[q].ok;
    if (ok) {
      h->peer_mode = true;
      h->pt.n_ranks = n_ranks;
      h->pt.rank = rank;
      for (int q = 0; q < n_ranks; q++) {
        unsigned char *base = q == rank ? h->shared_blk : (unsigned char *)h->peer_base[q];
        h->pt.rec[q] = reinterpret_cast<double *>(base);
        h->pt.flag[q] = reinterpret_cast<unsigned *>(base + 2 * h->rec_stride * sizeof(double));
      }
    } else {
      for (int q = 0; q < MAX_RANKS; q++)
        if (h->peer_base[q]) { cudaIpcCloseMemHandle(h->peer_base[q]); h->peer_base[q] = nullptr; }
    }
  }
  return SVNICP_OK;
}

static int choose_shape(svnicp_handle h) {
  const int Kp = (h->K + 3) & ~3;
  h->Kp = Kp;
  int TB = 32;
  int S = 4;
  // one CTA of k_gn per SM: its tile ring may take ~110 KB next to the 64 KB of second-level accumulators, which leaves room
  // for the small side-stream kernels (k_head_*, 33 KB) on the same SM
  size_t budget = 110 * 1024;
  if ((h->prm.gn_stages & 255) > 1) S = h->prm.gn_stages & 255;  // tuning knobs (svnicp_params extensions, bench sweeps)
  if (h->prm.gn_smem_kb > 0) budget = (size_t)(h->prm.gn_smem_kb < 150 ? h->prm.gn_smem_kb : 150) * 1024;
  const int consumers = GN_CONSUMERS;  // every consumer thread of k_gn carries two particles (packed fp32 pairs)
  while (TB > 4 && gn_stage_bytes(TB, Kp) * S > budget) TB >>= 1;
  h->TB = TB;
  h->stages = S;
  h->gn_smem = gn_smem_bytes(TB, Kp, S);
  const int pairs = (h->P_l + 1) / 2;
  int PG = 1;  // particle pairs (threads) per row group
  while (PG < pairs && PG < consumers) PG <<= 1;
  h->PG = PG;
  h->RG = consumers / PG;
  h->n_pgroups = (pairs + PG - 1) / PG;
  if (h->n_pgroups < 1) h->n_pgroups = 1;
  return SVNICP_OK;
}

// Everything whose size depends on (n_s, n_t, K, P_l): launch shape of the Gauss-Newton kernel, candidate table, pruned lists,
// voxel hash of the map.  Runs at add_cloud, and again at the head of stein_align when set_k changed K in between
// (SVGDICP.h:98: K_source_ takes effect at the next stein_align; the stored clouds stay valid).
static int prepare_scan(svnicp_handle h) {
  const int64_t n_s = h->n_s, n_t = h->n_t;
  choose_shape(h);
  const int TB = h->TB;
  const int n_pad = (int)(((n_s + TB - 1) / TB) * TB);
  h->n_pad = n_pad;
  CU(h->q0.ensure((size_t)3 * n_s));
  CU(h->sp.ensure((size_t)n_pad + 64));
  // candidate rows are built sharded across the ranks and all-gathered once per scan: n_ranks blocks of rows_per_rank rows
  h->rows_per_rank = (int)((n_s + h->n_ranks - 1) / h->n_ranks);
  CU(h->cand.ensure((size_t)h->rows_per_rank * h->n_ranks * h->K));
  // global map index per slot: only the parity taps read it (svnicp_get_candidates / _get_correspondences)
  if (h->prm.debug_corr) CU(h->cand_idx.ensure((size_t)h->rows_per_rank * h->n_ranks * h->K));
  CU(h->clist.ensure((size_t)n_pad * h->Kp));
  CU(h->hdr.ensure((size_t)n_pad + 64));
  CU(cudaMemsetAsync(h->hdr.p, 0, ((size_t)n_pad + 64) * sizeof(float4), h->stream));  // rows [n_s, n_pad) stay padding rows
  // SVNICP_FLAG_FILTER_FULL: prune from the full K-slot table every iteration (A/B measurements, roofline of the streaming pass)
  h->filter_reuse = (h->prm.flags & SVNICP_FLAG_FILTER_FULL) ? 0 : 1;
  if (h->filter_reuse) {
    CU(h->clist2.ensure((size_t)n_pad * h->Kp));
    CU(h->hdr2.ensure((size_t)n_pad + 64));
    CU(cudaMemsetAsync(h->hdr2.p, 0, ((size_t)n_pad + 64) * sizeof(float4), h->stream));
    for (int i = 0; i < 2; i++) {
      CU(h->ball[i].ensure((size_t)n_pad + 64));
      CU(h->cbase[i].ensure((size_t)n_pad + 64));
    }
  }
  size_t table = 1024;
  while (table < (size_t)2 * n_t) table <<= 1;
  CU(h->keys.ensure(table));
  CU(h->counts.ensure(table));
  CU(h->starts.ensure(table));
  CU(h->fill.ensure(table));
  CU(h->pt_slot.ensure((size_t)n_t));
  CU(h->sidx.ensure((size_t)n_t));
  CU(h->sxyz.ensure((size_t)3 * n_t));
  const int n_tiles = n_pad / TB;
  int n_slices = h->sm_count / h->n_pgroups;  // one CTA of k_gn per SM
  if (n_slices < 1) n_slices = 1;
  if (n_slices > n_tiles) n_slices = n_tiles;
  h->n_slices = n_slices;
  CU(h->part.ensure((size_t)n_slices * h->RG * (h->P_l > 0 ? h->P_l : 1) * NACC));
  if (h->prm.debug_corr) {
    CU(h->dbg_idx.ensure((size_t)h->P_l * n_s));
    CU(h->dbg_mask.ensure((size_t)h->P_l * n_s));
  }
  h->shape_dirty = false;
  return SVNICP_OK;
}

int svnicp_add_cloud(svnicp_handle h, const double *source, int64_t n_s, int source_on_device, const double *target, int64_t n_t,
                     int target_on_device, const double *init_pose) {
  if (!h) return SVNICP_ERR_INVALID;
  if (!source || !target || n_s < 1 || n_t < 1) return fail(h, SVNICP_ERR_INVALID, "add_cloud: empty cloud (n_s=%lld, n_t=%lld)", (long long)n_s, (long long)n_t);
  if (n_s > (1ll << 30) || n_t > (1ll << 30)) return fail(h, SVNICP_ERR_INVALID, "add_cloud: cloud too large");
  CU(cudaSetDevice(h->device));
  CU(h->src64.ensure((size_t)3 * n_s));
  CU(h->tgt64.ensure((size_t)3 * n_t));
  CU(cudaMemcpyAsync(h->src64.p, source, (size_t)3 * n_s * sizeof(double), source_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(h->tgt64.p, target, (size_t)3 * n_t * sizeof(double), target_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, h->stream));
  h->n_s = n_s;
  h->n_t = n_t;
  const int rc = prepare_scan(h);
  if (rc) return rc;
  h->have_cloud = true;
  h->aligned = false;
  h->eval_ok = false;
  return upload_particles(h, init_pose);  // SVGDICP.cpp:47-61 (also synchronises the cloud copies)
}

int svnicp_set_initial_mean(svnicp_handle h, const double R0[9], const double t0[3]) {
  if (!h || !R0 || !t0) return SVNICP_ERR_INVALID;
  h->eval_ok = false;  // the candidate table is relative to the previous initial mean
  memcpy(h->sc.R0, R0, 9 * sizeof(double));
  memcpy(h->sc.t0, t0, 3 * sizeof(double));
  return SVNICP_OK;
}

int svnicp_set_k(svnicp_handle h, int k) {
  if (!h) return SVNICP_ERR_INVALID;
  if (k < 1 || k > 256) return fail(h, SVNICP_ERR_INVALID, "set_k: K must be in [1,256]");
  if (k != h->K) h->shape_dirty = true;
  h->eval_ok = false;  // SVGDICP.h:98: K_source_ takes effect at the next stein_align; the stored clouds stay
  h->K = k;
  return SVNICP_OK;
}

int svnicp_set_threshold(svnicp_handle h, double max_dist) {
  if (!h) return SVNICP_ERR_INVALID;
  h->max_dist = max_dist;  // SVGDICP.h:100
  return SVNICP_OK;
}

static int do_allgather(svnicp_handle h, int buf = 0) {
  if (h->n_ranks <= 1) return SVNICP_OK;
  // in place: this rank's block already sits at rec + p_lo*REC
  double *base = h->rec + (size_t)buf * h->rec_stride;
  NC(g_nccl.AllGather(base + (size_t)h->p_lo * REC, base, (size_t)h->P_l_max * REC, ncclDouble, h->comm, h->stream));
  return SVNICP_OK;
}

// One scan = begin (setup + head of the scan) -> step x iterations -> epilogue (enqueue) -> finish (synchronise, read back).
// svnicp_align runs them back to back; svnicp_batch_align interleaves the steps of several handles so that their streams
// overlap on the GPU (throughput mode).
struct AlignState {
  IterArgs ia;
  SteinArgs sa;
  SvgdArgs sv;
  PeerTable pt;
  bool svgd = false, overlap = false, realign = false, special = false, enqueue_done = false;
  bool use_graph = false, graph_ready[2] = {false, false};
  unsigned seq0 = 0;
  int I = 0, e = 0;
};

static int align_begin(svnicp_handle h, AlignState &S) {
  if (!h->have_cloud) return fail(h, SVNICP_ERR_INVALID, "stein_align before add_cloud");
  h->eval_ok = false;  // the candidate table is rebuilt (or, NO_OPTIMIZER, not built): valid again once the scan completes
  CU(cudaSetDevice(h->device));
  cudaStream_t st = h->stream;
  const int I = S.I = h->prm.iterations;
  h->launches = 0;
  const bool realign = S.realign = h->aligned;  // stein_align again without a fresh add_cloud: continue from the current poses
  if (h->shape_dirty) {
    const int rc = prepare_scan(h);
    if (rc) return rc;
  }
  // host mirrors sized for this run
  if (h->h_hist_cap < (size_t)(I > 0 ? I : 1) * 6 * h->P) {
    if (h->h_history) cudaFreeHost(h->h_history);
    h->h_hist_cap = (size_t)(I > 0 ? I : 1) * 6 * h->P;
    CU(cudaMallocHost((void **)&h->h_history, h->h_hist_cap * sizeof(float)));
  }
  if (h->h_stop_cap < (size_t)I + 4) {
    if (h->h_stop) cudaFreeHost(h->h_stop);
    if (h->h_kept) cudaFreeHost(h->h_kept);
    if (h->h_med) cudaFreeHost(h->h_med);
    h->h_stop_cap = (size_t)I + 4;
    CU(cudaMallocHost((void **)&h->h_stop, h->h_stop_cap * sizeof(int)));
    CU(cudaMallocHost((void **)&h->h_kept, h->h_stop_cap * sizeof(unsigned long long)));
    CU(cudaMallocHost((void **)&h->h_med, h->h_stop_cap * sizeof(int32_t)));
  }
  while ((int)h->iter_events.size() < I + 1) {
    cudaEvent_t e;
    CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    h->iter_events.push_back(e);
  }
  CU(h->history.ensure((size_t)(I > 0 ? I : 1) * 6 * h->P));
  CU(h->kept_hist.ensure((size_t)I + 2, true));
  CU(h->med_path.ensure((size_t)I + 2));
  CU(cudaMemsetAsync(h->history.p, 0, (size_t)(I > 0 ? I : 1) * 6 * h->P * sizeof(float), st));  // SVGDICP.cpp:172-174
  CU(cudaMemsetAsync(h->kept_hist.p, 0, ((size_t)I + 2) * sizeof(unsigned long long), st));
  CU(cudaMemsetAsync(h->med_path.p, 0xff, ((size_t)I + 2) * sizeof(int32_t), st));  // -1: no median computed
  CU(cudaMemsetAsync(h->misc.p, 0, 8 * sizeof(int), st));
  const bool svgd = S.svgd = h->class_type == SVNICP_CLASS_SVGDICP;
  // A scan may be run again without a fresh add_cloud (the reference keeps R_/t_ and rewrites history rows 0..I-1; SVGDICP
  // rebuilds its optimizer in every stein_align, SVGDICP.cpp:73): restart the device-side iteration state, keep the poses.
  h->launches += launch_align_reset(h->ctrl.p, svgd ? h->opt_state.p : nullptr, svgd ? (size_t)12 * h->P_l : 0, st);
  S.sv = svgd ? svgd_args(h) : SvgdArgs();
  if (svgd && h->optimizer < 0) {
    // SVGDICP.cpp:73-75: "No optimizer chosen" -> NO_OPTIMIZER before anything moves; the getters then describe the
    // untouched pose_particles_ (every rank holds all of it)
    SteinArgs sa0;
    memset(&sa0, 0, sizeof(sa0));
    sa0.P = h->P; sa0.rec = h->rec; sa0.stats = h->stats.p; sa0.particles = h->particles.p;
    h->launches += launch_svgd_rec(h->rec, h->prev.p, nullptr, 0, h->P, 0, st);
    h->launches += launch_stats_svgd(sa0, nullptr, st);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(h->h_stats, h->stats.p, 48 * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(h->h_particles, h->particles.p, (size_t)6 * h->P * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    memset(h->h_ctrl, 0, sizeof(Ctrl));
    memset(h->h_kept, 0, ((size_t)I + 2) * sizeof(unsigned long long));
    memset(h->h_med, 0xff, ((size_t)I + 2) * sizeof(int32_t));
    h->iters_done = 0;
    h->enqueued_iters = 0;
    h->ms_setup = h->ms_iter = h->ms_epi = h->ms_total = 0;
    h->aligned = true;
    S.special = true;
    return SVNICP_NO_OPTIMIZER;
  }

  CU(cudaEventRecord(h->ev[0], st));
  // ---- per-scan setup: candidate table (SVGDICP.cpp:176-215) ----
  CandBuildArgs cb;
  cb.src64 = h->src64.p; cb.tgt64 = h->tgt64.p;
  cb.n_s = (int)h->n_s; cb.n_pad = h->n_pad; cb.n_t = (int)h->n_t; cb.K = h->K;
  cb.sc = h->sc;
  cb.cell = h->prm.grid_cell > 0 ? h->prm.grid_cell : 1.5;
  cb.q0 = h->q0.p; cb.sp = h->sp.p;
  cb.keys = h->keys.p; cb.counts = h->counts.p; cb.starts = h->starts.p; cb.fill = h->fill.p; cb.pt_slot = h->pt_slot.p;
  cb.cursor = h->misc.p; cb.fallback_count = h->misc.p + 1;
  size_t table = 1024;
  while (table < (size_t)2 * h->n_t) table <<= 1;
  cb.table_size = (int)table;
  cb.sxyz = h->sxyz.p; cb.sidx = h->sidx.p; cb.cand = h->cand.p; cb.cand_idx = h->prm.debug_corr ? h->cand_idx.p : nullptr;
  cb.sm_count = h->sm_count;
  cb.row_lo = h->rank * h->rows_per_rank;
  cb.row_hi = cb.row_lo + h->rows_per_rank < (int)h->n_s ? cb.row_lo + h->rows_per_rank : (int)h->n_s;
  if (cb.row_hi < cb.row_lo) cb.row_hi = cb.row_lo;
  h->launches += launch_cand_build(cb, st);
  if (h->n_ranks > 1) {
    // per-scan exchange: every rank built the K-NN rows of its block only (exact and deterministic, so the gathered
    // table equals the single-GPU table bit for bit); in place, this rank's block already sits at its offset
    const size_t blk = (size_t)h->rows_per_rank * h->K;
    NC(g_nccl.AllGather(h->cand.p + (size_t)h->rank * blk, h->cand.p, blk * 4, ncclFloat, h->comm, st));
    // the global map indices only feed the parity taps (svnicp_get_candidates / _get_correspondences): 20 % of the volume
    if (h->prm.debug_corr) NC(g_nccl.AllGather(h->cand_idx.p + (size_t)h->rank * blk, h->cand_idx.p, blk, ncclInt32, h->comm, st));
  }
  CU(cudaGetLastError());
  CU(cudaEventRecord(h->ev[1], st));

  IterArgs &ia = S.ia;
  memset(&ia, 0, sizeof(ia));
  ia.n_s = (int)h->n_s; ia.n_pad = h->n_pad; ia.K = h->K; ia.Kp = h->Kp; ia.cand_idx = h->prm.debug_corr ? h->cand_idx.p : nullptr;
  ia.P = h->P; ia.p_lo = h->p_lo; ia.P_l = h->P_l;
  ia.sc = h->sc;
  ia.max_dist = (float)h->max_dist;
  ia.sp = h->sp.p; ia.cand = h->cand.p; ia.clist = h->clist.p; ia.hdr = h->hdr.p;
  ia.R = h->R.p; ia.t = h->t.p; ia.xf = h->xf.p; ia.dnorm = h->dnorm.p; ia.part = h->part.p; ia.rec = h->rec; ia.rec_stride = h->rec_stride; ia.ctrl = h->ctrl.p;
  ia.TB = h->TB; ia.stages = h->stages; ia.n_slices = h->n_slices; ia.n_pgroups = h->n_pgroups; ia.PG = h->PG; ia.RG = h->RG;
  ia.gn_lag = (h->prm.gn_stages >> 8) ? (h->prm.gn_stages >> 8) : ((h->stages >= 4) ? 2 : 1);
  ia.gn_smem = h->gn_smem; ia.sm_count = h->sm_count; ia.svn_full_grad = h->prm.SVN_full_grad;
  ia.first_order = svgd ? 1 : 0;
  ia.dbg_idx = h->prm.debug_corr ? h->dbg_idx.p : nullptr;
  ia.dbg_mask = h->prm.debug_corr ? h->dbg_mask.p : nullptr;

  SteinArgs &sa = S.sa;
  memset(&sa, 0, sizeof(sa));
  sa.P = h->P; sa.p_lo = h->p_lo; sa.P_l = h->P_l; sa.I = I;
  sa.svn_full_grad = h->prm.SVN_full_grad; sa.check_early_stop = h->prm.check_early_stop;
  sa.lr = h->prm.lr; sa.threshold = h->prm.convergence_threshold;
  sa.rec = h->rec; sa.rec_stride = h->rec_stride; sa.xs = h->xs.p; sa.delta = h->delta.p; sa.dnorm = h->dnorm.p; sa.R = h->R.p; sa.t = h->t.p;
  sa.Hbar_inv = h->Hbar_inv.p; sa.hist = h->hist.p; sa.history = h->history.p; sa.ctrl = h->ctrl.p;
  sa.stats = h->stats.p; sa.particles = h->particles.p; sa.sm_count = h->sm_count;
  sa.kept_hist = h->kept_hist.p;
  sa.med_path = h->med_path.p;
  if (svgd) sa.rec_stride = 0;  // one record buffer: k_head_* read buffer 0 whatever the iteration's parity
  sa.prep_scratch_d = h->prep_scratch_d.p;
  sa.prep_scratch_i = h->prep_scratch_i.p;
  sa.stamps = h->profile ? h->stamps.p : nullptr;
  // SVN-ICP class: k_head (decide + median) on the side stream as soon as the poses of the iteration are final, overlapping
  // k_filter / k_gn; k_finalize and k_tail follow on the main stream.  Sharded without the peer exchange (NCCL fallback):
  // finalize -> ncclAllGather of the records -> k_head -> k_tail, all on the main stream.
  const bool overlap = S.overlap = !svgd && (h->n_ranks == 1 || h->peer_mode);
  S.pt = h->pt;  // n_ranks == 1 view unless the peer exchange is up
  S.seq0 = h->seq;  // sequence numbers of the peer exchange run on across scans (stale flags of the last scan must never satisfy a wait)
  // Small problems without early stop are bound by the host's enqueue rate (~13 API calls per iteration against ~50 us of
  // kernels), so iterations >= 1 are captured once per scan into one CUDA graph per list-buffer parity and replayed with one
  // launch each.  Same kernels, same arguments, same order.  Measured on 868-point scans: 100 particles x 30 iterations 3.49 ->
  // 3.00 ms; with early stop (the host follows the stop flag three iterations behind, so it is never the bottleneck) the two
  // captures per scan cost more than they save (4.15 -> 4.49 ms), and big problems have nothing to gain: both keep the direct
  // launches, and the per-phase events stay usable.
  S.use_graph = overlap && h->n_ranks == 1 && !h->profile && !h->prm.debug_corr && !h->graph_off &&
                !(h->prm.flags & (SVNICP_FLAG_DEBUG_SYNC | SVNICP_FLAG_NO_GRAPH)) &&
                ((h->prm.flags & SVNICP_FLAG_FORCE_GRAPH) || (!h->prm.check_early_stop && I >= 16 && (double)h->n_s * (double)h->P_l <= 1.0e7));

  if (h->profile)
    while (h->prof_events.size() < (size_t)I * 7) {
      cudaEvent_t pe;
      CU(cudaEventCreate(&pe));
      h->prof_events.push_back(pe);
    }
  if (!svgd) {
    // head of the scan: x of every particle into record buffer 0, transforms and pruning ball of the local slice
    const double *x_src = (realign && h->n_ranks > 1) ? h->rec + (size_t)(h->iters_done & 1) * h->rec_stride : nullptr;
    h->launches += launch_prep(ia, st, 1, x_src);
    if (overlap) CU(cudaEventRecord(h->ev_x, st));
  }
  S.e = 0;
  S.enqueue_done = I <= 0;
  return SVNICP_OK;
}

// Sequence number s of the peer exchange.  Without the exchange (pt.n_ranks == 1) no kernel waits on or publishes one, so it is
// 0 there: a captured iteration then depends on e only through its list-buffer parity, and one graph per parity replays all.
static unsigned peer_seq(const AlignState &S, int s) { return S.pt.n_ranks > 1 ? S.seq0 + (unsigned)s : 0u; }

// The head chain of iteration e (epilogue: after the last one) on stream s; adds its launches to n.  Iteration 0 waits for no
// peer: every rank's k_prep wrote the x of all particles.
static int head_chain(svnicp_handle h, const AlignState &S, int e, int epilogue, cudaStream_t s, int &n) {
  const int k = launch_head(S.sa, S.pt, e > 0 ? peer_seq(S, e) : 0u, epilogue, s);
  if (k < 0) return fail(h, SVNICP_ERR_CUDA, "launch of k_head failed: %s", cudaGetErrorString(cudaGetLastError()));
  n += k;
  return SVNICP_OK;
}

// List buffers of iteration e.  With list reuse they ping-pong by parity: iteration e prunes the lists of iteration e-1
// wherever its ball still covers this one's.
static void select_lists(svnicp_handle h, IterArgs &ia, int e) {
  const int cur = h->filter_reuse ? e & 1 : 0;
  ia.clist = cur ? h->clist2.p : h->clist.p;
  ia.hdr = cur ? h->hdr2.p : h->hdr.p;
  if (!h->filter_reuse) return;
  ia.cbase = h->cbase[cur].p;
  ia.ball = h->ball[cur].p;
  ia.clist_prev = e > 0 ? (cur ? h->clist.p : h->clist2.p) : nullptr;
  ia.cbase_prev = h->cbase[cur ^ 1].p;
  ia.ball_prev = h->ball[cur ^ 1].p;
  ia.kept_hist = h->kept_hist.p;
}

// Before phase k of iteration e: the per-phase event (svnicp_set_profiling), and with SVNICP_FLAG_DEBUG_SYNC a wait for the
// device that is reported on stderr (localises a hang or a fault).  Both keep a scan off the graphs, so neither runs in a capture.
static int phase_mark(svnicp_handle h, int e, int k) {
  if (h->profile) CU(cudaEventRecord(h->prof_events[(size_t)e * 7 + k], h->stream));
  if (h->prm.flags & SVNICP_FLAG_DEBUG_SYNC) {
    fprintf(stderr, "[svnicp] iteration %d: before phase %d ...", e, k);
    fflush(stderr);
    const cudaError_t e1 = cudaStreamSynchronize(h->stream), e2 = cudaStreamSynchronize(h->head_stream);
    fprintf(stderr, " main %s, head %s\n", cudaGetErrorString(e1), cudaGetErrorString(e2));
    fflush(stderr);
  }
  return SVNICP_OK;
}

// Enqueue iteration e (SVNICP.cpp:52-108) of either class; returns its number of launches or a negative status.  Graph capture
// and direct launches both run this code.  The side-stream head chain (overlap) forks from ev_fork, recorded on the main stream
// in the same capture (or outside any), and joins it through ev_join.
static int enqueue_iteration(svnicp_handle h, AlignState &S, int e, cudaEvent_t ev_fork, cudaEvent_t ev_join) {
  IterArgs &ia = S.ia;
  SteinArgs &sa = S.sa;
  cudaStream_t st = h->stream, hs = h->head_stream;
  int n = 0;
  if (int rc = phase_mark(h, e, 0)) return rc;
  if (S.svgd) n += launch_prep(ia, st, 0, nullptr);
  else if (S.overlap) {
    CU(cudaStreamWaitEvent(hs, ev_fork, 0));
    if (int rc = head_chain(h, S, e, 0, hs, n)) return rc;
    CU(cudaEventRecord(ev_join, hs));
  }
  if (int rc = phase_mark(h, e, 1)) return rc;
  select_lists(h, ia, e);
  n += launch_filter(ia, st);
  if (int rc = phase_mark(h, e, 2)) return rc;
  n += launch_gn(ia, st);
  if (h->prm.debug_corr) {  // parity tap: the transforms this iteration's correspondences were computed with
    CU(h->dbg_xf.ensure((size_t)(h->P_l > 0 ? h->P_l : 1) * 12));
    CU(cudaMemcpyAsync(h->dbg_xf.p, h->xf.p, (size_t)h->P_l * 12 * sizeof(float), cudaMemcpyDeviceToDevice, st));
  }
  if (int rc = phase_mark(h, e, 3)) return rc;
  if (S.svgd) {
    n += launch_finalize_first(ia, S.sv, st);
    if (int rc = phase_mark(h, e, 4)) return rc;
    if (int rc = do_allgather(h)) return rc;
    if (int rc = phase_mark(h, e, 5)) return rc;
    if (int rc = head_chain(h, S, e, 0, st, n)) return rc;
    n += launch_stein_first(sa, st);
    n += launch_update_opt(sa, S.sv, e + 1, st);
  } else {
    // k_finalize does not wait for the head chain: it needs neither the bandwidth nor (for correctness) the stop flag -- if
    // the stop fires concurrently it writes one more (b, H) into the record buffer of the NEXT parity, which nobody reads
    n += launch_finalize(ia, S.pt, peer_seq(S, e + 1), st);
    if (int rc = phase_mark(h, e, 4)) return rc;
    if (!S.overlap) {
      if (int rc = do_allgather(h, e & 1)) return rc;  // NCCL fallback: whole records (x of this iteration + b, H, g)
      if (int rc = head_chain(h, S, e, 0, st, n)) return rc;
    }
    if (int rc = phase_mark(h, e, 5)) return rc;
    if (S.overlap) CU(cudaStreamWaitEvent(st, ev_join, 0));  // stop flag and bandwidth of this iteration
    n += launch_tail(sa, ia, S.pt, peer_seq(S, e + 1), peer_seq(S, e + 1), st);
  }
  if (int rc = phase_mark(h, e, 6)) return rc;
  CU(cudaGetLastError());
  return n;
}

// Capture iteration e into the CUDA graph of its parity and return whether that graph can be replayed.  A failure (e.g. a
// caller's stream that cannot be captured) is not an error of the scan: its error is cleared, direct launches take over.
static bool capture_iteration(svnicp_handle h, AlignState &S, int e) {
  const int par = e & 1;
  cudaStream_t st = h->stream;
  const std::string err = h->err;
  cudaGraph_t g = nullptr;
  int n = -1;
  if (cudaStreamBeginCapture(st, cudaStreamCaptureModeRelaxed) == cudaSuccess) {
    // fork from an event recorded in this capture: waiting on ev_x, recorded outside it, would invalidate the capture
    if (cudaEventRecord(h->ev_cfork, st) == cudaSuccess) n = enqueue_iteration(h, S, e, h->ev_cfork, h->ev_chead);
    if (cudaStreamEndCapture(st, &g) != cudaSuccess) n = -1;  // always end the capture, also after a failure inside it
  }
  bool ok = n >= 0 && g;
  if (ok && h->gexec[par]) {  // same topology as the last scan's: patch the arguments in place
    cudaGraphExecUpdateResultInfo info;
    if (cudaGraphExecUpdate(h->gexec[par], g, &info) != cudaSuccess) {
      cudaGraphExecDestroy(h->gexec[par]);
      h->gexec[par] = nullptr;
    }
  }
  if (ok && !h->gexec[par]) ok = cudaGraphInstantiate(&h->gexec[par], g, 0) == cudaSuccess;
  if (g) cudaGraphDestroy(g);
  cudaGetLastError();
  h->err = err;
  h->glaunches[par] = ok ? n : 0;
  return ok;
}

// enqueue iteration S.e: replay its graph or launch it directly, then what the host follows it by (ev_x, stop flag)
static int align_step(svnicp_handle h, AlignState &S) {
  const int LAG = 3;
  const int e = S.e;
  cudaStream_t st = h->stream;
  if (h->prm.check_early_stop && e >= LAG) {
    // deterministic host cut: the stop flag as of the END of iteration e-LAG decides (identical on every rank)
    CU(cudaEventSynchronize(h->iter_events[e - LAG]));
    if (h->h_stop[e - LAG]) { S.enqueue_done = true; return SVNICP_OK; }
  }
  bool replayed = false;
  if (S.use_graph && e >= 1) {
    const int par = e & 1;
    if (!S.graph_ready[par]) S.graph_ready[par] = capture_iteration(h, S, e);
    if (S.graph_ready[par]) {
      CU(cudaGraphLaunch(h->gexec[par], st));
      h->launches += h->glaunches[par];
      replayed = true;
    } else {
      // The graph could not be built: this handle keeps the direct launches of the same kernels from here on.  Nothing
      // captured was executed; the head chain below must wait for everything enqueued so far, hence a fresh ev_x.
      S.use_graph = false;
      h->graph_off = true;
      if (h->gexec[par]) { cudaGraphExecDestroy(h->gexec[par]); h->gexec[par] = nullptr; }
      CU(cudaEventRecord(h->ev_x, st));
    }
  }
  if (!replayed) {
    const int n = enqueue_iteration(h, S, e, h->ev_x, h->ev_head);
    if (n < 0) return n;
    h->launches += n;
  }
  // Sharded handles: the stop flag as of the END of iteration e must be copied BEFORE ev_x lets the head chain of iteration
  // e+1 (which may set it) start on the side stream -- every rank then reads the same value, enqueues the same number of
  // iterations and keeps the same sequence numbers.  Unsharded handles release the head chain first: one no-op iteration more
  // or less behind the stop is harmless there, and the 4-byte copy in front of the head chain cost 10 us per iteration on
  // small scans (3.47 -> 4.03 ms in the shipped regime).  A replayed iteration records no ev_x: nothing that follows waits on it.
  const bool release_head = S.overlap && !replayed, strict_cut = h->n_ranks > 1;
  if (release_head && !strict_cut) CU(cudaEventRecord(h->ev_x, st));
  if (h->prm.check_early_stop) {
    CU(cudaMemcpyAsync(&h->h_stop[e], &h->ctrl.p->stop, sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(cudaEventRecord(h->iter_events[e], st));
  }
  if (release_head && strict_cut) CU(cudaEventRecord(h->ev_x, st));
  S.e = e + 1;
  if (S.e >= S.I) S.enqueue_done = true;
  return SVNICP_OK;
}

static int align_epilogue(svnicp_handle h, AlignState &S) {
  cudaStream_t st = h->stream;
  const int e = S.e;
  h->enqueued_iters = e;
  h->seq = S.seq0 + (unsigned)e + 1u;
  CU(cudaEventRecord(h->ev[2], st));
  // ---- epilogue: last stop decision / history row, getters (SVNICP.cpp:111, :281-308) ----
  int n = 0;
  if (S.svgd) {
    n += launch_svgd_rec(h->rec, h->pose6.p, h->dnorm.p, h->p_lo, h->P_l, h->p_lo, st);
    if (int rc = do_allgather(h)) return rc;
  } else if (!S.overlap && h->n_ranks > 1) {
    // the final x of every particle already sits in the record buffer of parity (updates applied & 1) on every rank; NCCL
    // fallback: the device knows which buffer is final (early stop), so gather both
    for (int b2 = 0; b2 < 2; b2++)
      if (int rc = do_allgather(h, b2)) return rc;
  }
  if (int rc = head_chain(h, S, e, 1, st, n)) return rc;
  n += S.svgd ? launch_stats_svgd(S.sa, h->prev.p, st) : launch_stats(S.sa, 1, st);
  h->launches += n;
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(h->h_stats, h->stats.p, 48 * sizeof(double), cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(h->h_particles, h->particles.p, (size_t)6 * h->P * sizeof(double), cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(h->h_ctrl, h->ctrl.p, sizeof(Ctrl), cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(h->h_kept, h->kept_hist.p, ((size_t)S.I + 2) * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(h->h_med, h->med_path.p, ((size_t)S.I + 2) * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CU(cudaEventRecord(h->ev[3], st));
  return SVNICP_OK;
}

static int align_finish(svnicp_handle h, AlignState &S) {
  cudaStream_t st = h->stream, hs = h->head_stream;
  if (h->prm.flags & SVNICP_FLAG_WATCHDOG) {  // diagnostic watchdog: poll instead of blocking, report which stream is stuck and the device-side state
    const double t0 = (double)clock() / CLOCKS_PER_SEC;
    bool done = false;
    while ((double)clock() / CLOCKS_PER_SEC - t0 < 8.0) {
      if (cudaStreamQuery(st) == cudaSuccess && cudaStreamQuery(hs) == cudaSuccess) { done = true; break; }
    }
    if (!done) {
      cudaStream_t aux;
      cudaStreamCreateWithFlags(&aux, cudaStreamNonBlocking);
      Ctrl c;
      memset(&c, 0, sizeof(c));
      cudaMemcpyAsync(&c, h->ctrl.p, sizeof(Ctrl), cudaMemcpyDeviceToHost, aux);
      cudaStreamSynchronize(aux);
      fprintf(stderr, "[svnicp watchdog] main %s, head %s; ctrl: stop %d iter %d iters_done %d error %d fin_ticket %u tail_ticket %u kept_total %llu bandwidth %g enqueued %d\n",
              cudaGetErrorString(cudaStreamQuery(st)), cudaGetErrorString(cudaStreamQuery(hs)), c.stop, c.iter, c.iters_done, c.error, c.fin_ticket,
              c.tail_ticket, c.kept_total, c.bandwidth, S.e);
      fflush(stderr);
      return fail(h, SVNICP_ERR_CUDA, "watchdog: scan did not finish");
    }
  }
  CU(cudaStreamSynchronize(st));
  h->iters_done = h->h_ctrl->iters_done;
  if (h->h_ctrl->error >= 100) return fail(h, SVNICP_ERR_CUDA, "device bounds check %d failed (SVN_DEBUG_BOUNDS build)", h->h_ctrl->error - 100);
  if (h->h_ctrl->error) return fail(h, SVNICP_ERR_CUDA, "peer exchange timed out: another rank did not publish its records (rank %d of %d)", h->rank, h->n_ranks);
  float ms = 0;
  cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]); h->ms_setup = ms;
  cudaEventElapsedTime(&ms, h->ev[1], h->ev[2]); h->ms_iter = ms;
  cudaEventElapsedTime(&ms, h->ev[2], h->ev[3]); h->ms_epi = ms;
  cudaEventElapsedTime(&ms, h->ev[0], h->ev[3]); h->ms_total = ms;
  if (h->profile) {
    for (int k = 0; k < 8; k++) h->phase_ms[k] = 0;
    for (int it = 0; it < h->enqueued_iters; it++)
      for (int k = 0; k < 6; k++) {
        cudaEventElapsedTime(&ms, h->prof_events[(size_t)it * 7 + k], h->prof_events[(size_t)it * 7 + k + 1]);
        h->phase_ms[k] += ms;
      }
    h->phase_ms[6] = h->ms_setup;
    h->phase_ms[7] = (double)h->enqueued_iters;
  }
  int misc[2] = {0, 0};
  CU(cudaMemcpy(misc, h->misc.p, sizeof(misc), cudaMemcpyDeviceToHost));
  h->fallback_queries = misc[1];
  h->aligned = true;
  h->eval_ok = true;
  return SVNICP_ALIGN_SUCCESS;
}


int svnicp_align(svnicp_handle h) {
  if (!h) return SVNICP_ERR_INVALID;
  AlignState S;
  int rc = align_begin(h, S);
  if (rc != SVNICP_OK) return rc;  // error, or SVNICP_NO_OPTIMIZER (SVGDICP.cpp:73-75)
  while (!S.enqueue_done) {
    rc = align_step(h, S);
    if (rc != SVNICP_OK) return rc;
  }
  rc = align_epilogue(h, S);
  if (rc != SVNICP_OK) return rc;
  return align_finish(h, S);
}

#define NEED_ALIGNED(out)                                                              \
  if (!h) return SVNICP_ERR_INVALID;                                                   \
  if (!(out)) return fail(h, SVNICP_ERR_INVALID, "null output pointer");               \
  if (!h->aligned) return fail(h, SVNICP_ERR_INVALID, "no result yet: call svnicp_align first");

int svnicp_get_transformation(svnicp_handle h, double out6[6]) {
  NEED_ALIGNED(out6);
  memcpy(out6, h->h_stats, 6 * sizeof(double));
  return SVNICP_OK;
}
int svnicp_get_distribution(svnicp_handle h, double out6[6]) {
  NEED_ALIGNED(out6);
  memcpy(out6, h->h_stats + 6, 6 * sizeof(double));
  return SVNICP_OK;
}
int svnicp_get_cov_matrix(svnicp_handle h, double out36[36]) {
  NEED_ALIGNED(out36);
  memcpy(out36, h->h_stats + 12, 36 * sizeof(double));
  return SVNICP_OK;
}
int svnicp_get_particles(svnicp_handle h, double *out) {
  NEED_ALIGNED(out);
  if (!h->permuted) {
    memcpy(out, h->h_particles, (size_t)6 * h->P * sizeof(double));
  } else {  // back to the caller's particle order
    for (int c = 0; c < 6; c++)
      for (int i = 0; i < h->P; i++) out[(size_t)c * h->P + h->perm[i]] = h->h_particles[(size_t)c * h->P + i];
  }
  return SVNICP_OK;
}
int svnicp_get_particle_weight(svnicp_handle h, double *out) {
  if (!h) return SVNICP_ERR_INVALID;
  if (!out) return fail(h, SVNICP_ERR_INVALID, "null output pointer");
  // SVNICP.cpp:46 + :281-284: float32 weights widened to double; SVGDICP.cpp:522-524: a vector of ones
  const double w = h->class_type == SVNICP_CLASS_SVGDICP ? 1.0 : (double)(1.0f / (float)h->P);
  for (int p = 0; p < h->P; p++) out[p] = w;
  return SVNICP_OK;
}
int svnicp_get_particle_history(svnicp_handle h, float *out, int32_t *rows) {
  if (!h) return SVNICP_ERR_INVALID;
  if (!h->aligned) return fail(h, SVNICP_ERR_INVALID, "no result yet");
  const int I = h->prm.iterations;
  if (rows) *rows = I;
  if (out && I > 0) {
    CU(cudaSetDevice(h->device));
    CU(cudaMemcpy(out, h->history.p, (size_t)I * 6 * h->P * sizeof(float), cudaMemcpyDeviceToHost));
    if (h->permuted) {  // rows are [6][P] in internal order: back to the caller's particle order
      std::vector<float> row((size_t)h->P);
      for (size_t r = 0; r < (size_t)I * 6; r++) {
        float *p = out + r * h->P;
        memcpy(row.data(), p, (size_t)h->P * sizeof(float));
        for (int i = 0; i < h->P; i++) p[h->perm[i]] = row[i];
      }
    }
  }
  return SVNICP_OK;
}
int svnicp_get_runtime(svnicp_handle h, double out3[3]) {
  if (!h || !out3) return SVNICP_ERR_INVALID;
  // SVGDICP.h:94-96 {knn_duration_, update_duration_, finish_iter_}; SVNICP never fills them (Q12) -- we do, from CUDA events.
  out3[0] = h->ms_setup * 1e-3;
  out3[1] = h->ms_iter * 1e-3;
  out3[2] = (double)(h->aligned ? h->iters_done : h->prm.iterations);
  return SVNICP_OK;
}

// ---- counter-based RNG for the particle initialisers (ICPUtils.cpp:45-75) ----
static inline uint64_t splitmix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
static inline double u01(uint64_t seed, uint64_t i) { return (double)(splitmix64(seed ^ splitmix64(i)) >> 11) * (1.0 / 9007199254740992.0); }

int svnicp_initialize_particles(int P, const double ub[6], const double lb[6], uint64_t seed, double *out) {
  if (P < 1 || !ub || !lb || !out) return SVNICP_ERR_INVALID;
  for (int c = 0; c < 6; c++)
    for (int p = 0; p < P; p++) out[(size_t)c * P + p] = (P == 1) ? 0.0 : (ub[c] - lb[c]) * u01(seed, (uint64_t)c * P + p) + lb[c];
  return SVNICP_OK;
}

int svnicp_initialize_particles_gaussian(int P, const double cov_diag[6], uint64_t seed, double *out) {
  if (P < 1 || !cov_diag || !out) return SVNICP_ERR_INVALID;
  for (int c = 0; c < 6; c++) {
    const double sd = sqrt(cov_diag[c]);
    for (int p = 0; p < P; p++) {
      if (P == 1) { out[(size_t)c * P + p] = 0.0; continue; }
      const double u1 = u01(seed, 2 * ((uint64_t)c * P + p)), u2 = u01(seed, 2 * ((uint64_t)c * P + p) + 1);
      double z = sqrt(-2.0 * log(u1 > 1e-300 ? u1 : 1e-300)) * cos(6.283185307179586 * u2) * sd;
      if (z > 3 * sd) z = 3 * sd;   // clamp(-3 sigma, 3 sigma), ICPUtils.cpp:72-74
      if (z < -3 * sd) z = -3 * sd;
      out[(size_t)c * P + p] = z;
    }
  }
  return SVNICP_OK;
}

// ---- parity / debug taps ----
int svnicp_iterations_done(svnicp_handle h, int32_t *out) {
  if (!h || !out) return SVNICP_ERR_INVALID;
  *out = h->iters_done;
  return SVNICP_OK;
}

int svnicp_get_candidates(svnicp_handle h, int32_t *out_idx, float *out_rel) {
  if (!h || !h->aligned) return fail(h, SVNICP_ERR_INVALID, "no scan yet");
  if (out_idx && !h->prm.debug_corr)
    return fail(h, SVNICP_ERR_INVALID, "handle created without debug_corr: the map-index table is only written for the parity taps");
  CU(cudaSetDevice(h->device));
  const size_t n = (size_t)h->n_s * h->K;
  if (out_idx) CU(cudaMemcpy(out_idx, h->cand_idx.p, n * sizeof(int32_t), cudaMemcpyDeviceToHost));
  if (out_rel) {
    std::vector<float4> tmp(n);
    CU(cudaMemcpy(tmp.data(), h->cand.p, n * sizeof(float4), cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < n; i++) { out_rel[3 * i] = tmp[i].x; out_rel[3 * i + 1] = tmp[i].y; out_rel[3 * i + 2] = tmp[i].z; }
  }
  return SVNICP_OK;
}

int svnicp_get_source_f32(svnicp_handle h, float *out) {
  if (!h || !h->aligned) return fail(h, SVNICP_ERR_INVALID, "no scan yet");
  CU(cudaSetDevice(h->device));
  std::vector<float4> tmp((size_t)h->n_s);
  CU(cudaMemcpy(tmp.data(), h->sp.p, (size_t)h->n_s * sizeof(float4), cudaMemcpyDeviceToHost));
  for (int64_t i = 0; i < h->n_s; i++) { out[3 * i] = tmp[i].x; out[3 * i + 1] = tmp[i].y; out[3 * i + 2] = tmp[i].z; }
  return SVNICP_OK;
}

int svnicp_get_correspondences(svnicp_handle h, float *out_xf, int32_t *out_idx, uint8_t *out_mask) {
  if (!h || !h->aligned) return fail(h, SVNICP_ERR_INVALID, "no scan yet");
  if (!h->prm.debug_corr) return fail(h, SVNICP_ERR_INVALID, "created without debug_corr");
  CU(cudaSetDevice(h->device));
  // rows are local particles in INTERNAL order; on an unsharded handle they are handed out in the caller's order
  const bool unperm = h->permuted && h->n_ranks == 1;
  auto fetch_rows = [&](void *out, const void *dev, size_t row_bytes) -> cudaError_t {
    if (!unperm) return cudaMemcpy(out, dev, (size_t)h->P_l * row_bytes, cudaMemcpyDeviceToHost);
    std::vector<unsigned char> tmp((size_t)h->P_l * row_bytes);
    const cudaError_t e = cudaMemcpy(tmp.data(), dev, tmp.size(), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return e;
    for (int i = 0; i < h->P_l; i++) memcpy((unsigned char *)out + (size_t)h->perm[i] * row_bytes, tmp.data() + (size_t)i * row_bytes, row_bytes);
    return cudaSuccess;
  };
  if (out_xf) CU(fetch_rows(out_xf, h->dbg_xf.p, 12 * sizeof(float)));
  if (out_idx) CU(fetch_rows(out_idx, h->dbg_idx.p, (size_t)h->n_s * sizeof(int32_t)));
  if (out_mask) CU(fetch_rows(out_mask, h->dbg_mask.p, (size_t)h->n_s));
  return SVNICP_OK;
}

int svnicp_get_gn_system(svnicp_handle h, double *out_H, double *out_b, double *out_x) {
  if (!h || !h->aligned) return fail(h, SVNICP_ERR_INVALID, "no scan yet");
  CU(cudaSetDevice(h->device));
  std::vector<double> rec((size_t)h->P * REC);
  // SVN-ICP class: the record of the last executed iteration k = iters_done - 1 (x at its head, b, H) is in buffer k & 1
  const int buf = (h->class_type == SVNICP_CLASS_SVNICP && h->iters_done > 0) ? ((h->iters_done - 1) & 1) : 0;
  CU(cudaMemcpy(rec.data(), h->rec + (size_t)buf * h->rec_stride, rec.size() * sizeof(double), cudaMemcpyDeviceToHost));
  // SVGD-ICP class: x at the head of the last executed iteration lives in xs [6][P] (the epilogue rewrites rec's x)
  std::vector<double> xs((size_t)6 * h->P);
  if (h->class_type != SVNICP_CLASS_SVNICP) CU(cudaMemcpy(xs.data(), h->xs.p, xs.size() * sizeof(double), cudaMemcpyDeviceToHost));
  else
    for (int i = 0; i < h->P; i++)
      for (int c = 0; c < 6; c++) xs[(size_t)c * h->P + i] = rec[(size_t)i * REC + REC_X + c];
  for (int i = 0; i < h->P; i++) {  // i: internal order, p: the caller's particle index
    const double *r = rec.data() + (size_t)i * REC;
    const size_t p = h->permuted ? (size_t)h->perm[i] : (size_t)i;
    if (out_x)
      for (int c = 0; c < 6; c++) out_x[6 * p + c] = xs[(size_t)c * h->P + i];
    if (out_b) memcpy(out_b + 6 * p, r + REC_B, 6 * sizeof(double));
    if (out_H)
      for (int a = 0; a < 6; a++)
        for (int c = 0; c < 6; c++) out_H[36 * p + 6 * a + c] = r[REC_H + (a <= c ? tri(a, c) : tri(c, a))];
  }
  return SVNICP_OK;
}

int svnicp_get_stein(svnicp_handle h, double *out_delta, double *out_bandwidth) {
  if (!h || !h->aligned) return fail(h, SVNICP_ERR_INVALID, "no scan yet");
  CU(cudaSetDevice(h->device));
  if (out_delta) {
    if (h->permuted && h->n_ranks == 1) {  // unsharded: the caller's particle order (sharded: the local slice in internal order)
      std::vector<double> tmp((size_t)h->P_l * 6);
      CU(cudaMemcpy(tmp.data(), h->delta.p, tmp.size() * sizeof(double), cudaMemcpyDeviceToHost));
      for (int i = 0; i < h->P_l; i++) memcpy(out_delta + 6 * (size_t)h->perm[i], tmp.data() + 6 * (size_t)i, 6 * sizeof(double));
    } else {
      CU(cudaMemcpy(out_delta, h->delta.p, (size_t)h->P_l * 6 * sizeof(double), cudaMemcpyDeviceToHost));
    }
  }
  if (out_bandwidth) *out_bandwidth = h->h_ctrl->bandwidth;
  return SVNICP_OK;
}

int svnicp_get_prune_stats(svnicp_handle h, double *out_mean_kept, int32_t *rows) {
  if (!h || !h->aligned) return fail(h, SVNICP_ERR_INVALID, "no scan yet");
  const int I = h->prm.iterations;
  if (rows) *rows = I;
  if (out_mean_kept)
    for (int i = 0; i < I; i++) {
      const unsigned long long v = h->h_kept[i];
      const double den = (double)(h->n_s > 0 ? h->n_s : 1);
      // SVNICP_FLAG_REUSE_STATS: fraction of rows pruned from the previous list instead of mean kept candidates (tuning aid)
      out_mean_kept[i] = (h->prm.flags & SVNICP_FLAG_REUSE_STATS) ? (double)(v >> 40) / den : (double)(v & ((1ull << 40) - 1ull)) / den;
    }
  return SVNICP_OK;
}

int svnicp_get_median_paths(svnicp_handle h, int32_t *out, int32_t *rows) {
  if (!h || !h->aligned) return fail(h, SVNICP_ERR_INVALID, "no scan yet");
  const int I = h->prm.iterations;
  if (rows) *rows = I;
  if (out) memcpy(out, h->h_med, (size_t)I * sizeof(int32_t));
  return SVNICP_OK;
}

int svnicp_get_timing(svnicp_handle h, double out4[4]) {
  if (!h || !out4) return SVNICP_ERR_INVALID;
  out4[0] = h->ms_setup; out4[1] = h->ms_iter; out4[2] = h->ms_epi; out4[3] = h->ms_total;
  return SVNICP_OK;
}

int svnicp_get_slice(svnicp_handle h, int32_t *lo, int32_t *hi) {
  if (!h) return SVNICP_ERR_INVALID;
  if (lo) *lo = h->p_lo;
  if (hi) *hi = h->p_lo + h->P_l;
  return SVNICP_OK;
}

int svnicp_set_profiling(svnicp_handle h, int on) {
  if (!h) return SVNICP_ERR_INVALID;
  h->profile = on ? 1 : 0;
  return SVNICP_OK;
}

int svnicp_get_phase_times(svnicp_handle h, double out8[8]) {
  if (!h || !out8) return SVNICP_ERR_INVALID;
  for (int k = 0; k < 8; k++) out8[k] = h->phase_ms[k];
  return SVNICP_OK;
}

int svnicp_get_scan_info(svnicp_handle h, int64_t out8[8]) {
  if (!h || !out8) return SVNICP_ERR_INVALID;
  out8[0] = h->n_s; out8[1] = h->n_t; out8[2] = h->K; out8[3] = h->fallback_queries;
  out8[4] = h->TB; out8[5] = h->n_slices; out8[6] = h->n_pgroups; out8[7] = h->enqueued_iters;
  return SVNICP_OK;
}

int svnicp_get_tail_stamps(svnicp_handle h, double out8[8]) {
  if (!h || !out8) return SVNICP_ERR_INVALID;
  CU(cudaSetDevice(h->device));
  CU(cudaMemcpy(out8, h->stamps.p, 8 * sizeof(double), cudaMemcpyDeviceToHost));
  return SVNICP_OK;
}

int svnicp_get_launch_count(svnicp_handle h, int64_t *out) {
  if (!h || !out) return SVNICP_ERR_INVALID;
  *out = h->launches;
  return SVNICP_OK;
}

// ---- svnicp_evaluate: registration objective of the last scan at caller-given poses (eval_kernels.cu) ----
// Reads the candidate table, the fp32 source and R0 of the last stein_align; writes only its own scratch (ev_*).  No launch
// is counted in launch_count() and no event of the scan's timing is recorded.
int svnicp_evaluate(svnicp_handle h, int n_poses, const double *poses_6xM, double *out_stats, double *out_H, double *out_b,
                    uint8_t *out_mask, int32_t *out_idx) {
  if (!h) return SVNICP_ERR_INVALID;
  if (n_poses < 1) return fail(h, SVNICP_ERR_INVALID, "evaluate: n_poses must be >= 1 (got %d)", n_poses);
  if (!poses_6xM || !out_stats) return fail(h, SVNICP_ERR_INVALID, "evaluate: null poses or out_stats");
  if (!h->eval_ok)
    return fail(h, SVNICP_ERR_INVALID, "evaluate: no candidate table of the current scan (stein_align must complete after add_cloud / "
                                       "set_initial_mean / set_k)");
  if (out_idx && !h->prm.debug_corr)
    return fail(h, SVNICP_ERR_INVALID, "evaluate: out_idx needs a handle created with debug_corr (the map-index table is only kept for it)");
  CU(cudaSetDevice(h->device));
  cudaStream_t st = h->stream;
  const int M = n_poses, n_s = (int)h->n_s;
  const int n_blk = M < EV_BLOCK ? M : EV_BLOCK;
  CU(h->ev_pose.ensure((size_t)6 * M));
  CU(h->ev_xf.ensure((size_t)12 * M));
  CU(h->ev_R.ensure((size_t)9 * M));
  CU(h->ev_out.ensure((size_t)EV_OUT * M));
  CU(h->ev_part.ensure((size_t)eval_parts(n_s, h->K, h->sm_count) * n_blk * EV_NS));
  if (out_mask) CU(h->ev_mask.ensure((size_t)n_blk * n_s));
  if (out_idx) CU(h->ev_idx.ensure((size_t)n_blk * n_s));
  CU(cudaMemcpyAsync(h->ev_pose.p, poses_6xM, (size_t)6 * M * sizeof(double), cudaMemcpyHostToDevice, st));
  launch_eval_prep(h->ev_pose.p, M, h->class_type == SVNICP_CLASS_SVGDICP ? 1 : 0, h->sc, h->ev_xf.p, h->ev_R.p, st);
  EvalArgs a;
  memset(&a, 0, sizeof(a));
  a.n_s = n_s; a.K = h->K; a.max_dist = (float)h->max_dist;
  a.sp = h->sp.p; a.cand = h->cand.p; a.cand_idx = out_idx ? h->cand_idx.p : nullptr;
  a.part = h->ev_part.p;
  a.mask = out_mask ? h->ev_mask.p : nullptr;
  a.idx = out_idx ? h->ev_idx.p : nullptr;
  for (int m0 = 0; m0 < M; m0 += EV_BLOCK) {
    a.MB = M - m0 < EV_BLOCK ? M - m0 : EV_BLOCK;
    a.G = 1;
    while (a.G < a.MB) a.G <<= 1;
    a.xf = h->ev_xf.p + (size_t)12 * m0;
    launch_eval_block(a, out_H || out_b, h->sc, h->ev_R.p + (size_t)9 * m0, h->ev_out.p + (size_t)EV_OUT * m0, h->sm_count, st);
    CU(cudaGetLastError());
    // [M][n_s] outputs: the rows of this block are contiguous in the caller's array
    if (out_mask) CU(cudaMemcpyAsync(out_mask + (size_t)m0 * n_s, h->ev_mask.p, (size_t)a.MB * n_s, cudaMemcpyDeviceToHost, st));
    if (out_idx) CU(cudaMemcpyAsync(out_idx + (size_t)m0 * n_s, h->ev_idx.p, (size_t)a.MB * n_s * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  }
  std::vector<double> res((size_t)EV_OUT * M);
  CU(cudaMemcpyAsync(res.data(), h->ev_out.p, res.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  for (int m = 0; m < M; m++) {
    const double *r = res.data() + (size_t)EV_OUT * m;
    memcpy(out_stats + (size_t)3 * m, r, 3 * sizeof(double));
    if (out_H) memcpy(out_H + (size_t)36 * m, r + 3, 36 * sizeof(double));
    if (out_b) memcpy(out_b + (size_t)6 * m, r + 39, 6 * sizeof(double));
  }
  return SVNICP_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Throughput mode (BASELINE.json configs[3]): several independent odometry streams on one GPU.  A batch owns one ordinary
// handle per stream (own CUDA streams, own buffers); svnicp_batch_align enqueues the scans of all streams iteration by
// iteration, round robin, so the short latency-bound kernels of one stream (pruning, finalize, Stein phase) run under
// the Gauss-Newton pass of another.  Results are bit-identical to running each stream's handle on its own.
// ---------------------------------------------------------------------------------------------------------------
struct svnicp_batch_t {
  std::vector<svnicp_handle> hs;
  std::string err;
};

int svnicp_batch_create(svnicp_batch *out, const svnicp_params *params, int n_streams, int particle_count, const double *init_pose, int device) {
  if (!out || !params || n_streams < 1 || n_streams > 4096) return fail(nullptr, SVNICP_ERR_INVALID, "svnicp_batch_create: bad argument");
  *out = nullptr;
  svnicp_batch b = new svnicp_batch_t();
  for (int s = 0; s < n_streams; s++) {
    svnicp_handle h = nullptr;
    const int rc = svnicp_create(&h, params, particle_count, init_pose ? init_pose + (size_t)s * 6 * particle_count : nullptr, SVNICP_CLASS_SVNICP, device);
    if (rc != SVNICP_OK) {
      svnicp_batch_destroy(b);
      return rc;  // message in svnicp_last_error(NULL)
    }
    b->hs.push_back(h);
  }
  *out = b;
  return SVNICP_OK;
}

void svnicp_batch_destroy(svnicp_batch b) {
  if (!b) return;
  for (svnicp_handle h : b->hs) svnicp_destroy(h);
  delete b;
}

const char *svnicp_batch_last_error(svnicp_batch b) { return b ? b->err.c_str() : g_create_error.c_str(); }

int svnicp_batch_size(svnicp_batch b) { return b ? (int)b->hs.size() : SVNICP_ERR_INVALID; }

svnicp_handle svnicp_batch_stream(svnicp_batch b, int s) { return (b && s >= 0 && s < (int)b->hs.size()) ? b->hs[(size_t)s] : nullptr; }

int svnicp_batch_align(svnicp_batch b, int32_t *states) {
  if (!b) return SVNICP_ERR_INVALID;
  const size_t n = b->hs.size();
  std::vector<AlignState> S(n);
  std::vector<int> rc(n, SVNICP_OK);
  auto note = [&](size_t s, int code) {
    rc[s] = code;
    if (code < 0) b->err = "stream " + std::to_string(s) + ": " + b->hs[s]->err;
  };
  for (size_t s = 0; s < n; s++) note(s, align_begin(b->hs[s], S[s]));
  bool any = true;
  while (any) {
    any = false;
    for (size_t s = 0; s < n; s++) {
      if (rc[s] != SVNICP_OK || S[s].enqueue_done) continue;
      note(s, align_step(b->hs[s], S[s]));
      any = true;
    }
  }
  for (size_t s = 0; s < n; s++)
    if (rc[s] == SVNICP_OK) note(s, align_epilogue(b->hs[s], S[s]));
  int worst = SVNICP_ALIGN_SUCCESS;
  for (size_t s = 0; s < n; s++) {
    if (rc[s] == SVNICP_OK) note(s, align_finish(b->hs[s], S[s]));
    if (states) states[s] = rc[s];
    if (rc[s] < 0) worst = rc[s];
  }
  for (size_t s = 0; s < n; s++)  // a stream that failed midway may still have work in flight
    if (rc[s] < 0) { cudaSetDevice(b->hs[s]->device); cudaStreamSynchronize(b->hs[s]->stream); cudaStreamSynchronize(b->hs[s]->head_stream); }
  return worst;
}

}  // extern "C"
