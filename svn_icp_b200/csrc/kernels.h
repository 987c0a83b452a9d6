// kernels.h -- host-callable launchers of the hand-written sm_100a kernels (internal).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "common.cuh"

namespace svn {

struct CandBuildArgs {
  const double *src64, *tgt64;
  int n_s, n_pad, n_t, K;
  int row_lo, row_hi;  // source rows whose candidates THIS rank builds (sharded across ranks, then all-gathered)
  ScanConst sc;
  double cell;
  double *q0;     // [n_s][3]
  float4 *sp;     // [n_pad]
  // voxel hash of the map
  unsigned long long *keys;
  int *counts, *starts, *fill, *pt_slot, *cursor;
  int table_size;  // power of two >= 2*n_t
  double *sxyz;    // [n_t][3] cell-sorted map
  int *sidx;       // [n_t] original indices
  float4 *cand;    // [n_s][K]  (m - q0 in fp32, w = lower bound of |m - q0|)
  int *cand_idx;   // [n_s][K]  global map index per slot
  int *fallback_count;
  int sm_count;
};
int launch_cand_build(const CandBuildArgs &a, cudaStream_t st);
size_t knn_smem_bytes();

struct IterArgs {
  // sizes
  int n_s, n_pad, K;
  int Kp;           // K rounded up to a multiple of 4: row stride of the pruned lists
  const int *cand_idx;  // [n_s][K] global map index per candidate slot (debug taps only)
  int P;            // all particles
  int p_lo, P_l;    // local slice
  // geometry
  ScanConst sc;
  float max_dist;
  // buffers
  const float4 *sp, *cand;
  float4 *clist;
  float4 *hdr;          // [n_pad] row headers of the pruned lists: (R0 s).xyz, w = (padded length << 16 | true length) bits; 0 = padding row
  // list reuse (k_filter): the previous iteration's pruned lists, their true lengths and the ball (centre query, radius)
  // they are exact for; null = always prune from the full table.  cbase / ball: the same for THIS iteration's output.
  const float4 *clist_prev;
  const int *cbase_prev;
  const float4 *ball_prev;
  int *cbase;
  float4 *ball;
  const unsigned long long *kept_hist;  // [I] kept candidates per iteration (low 40 bits): picks the pruning kernel, see filter_use_reuse
  double *R, *t;       // [P][9], [P][3]
  float *xf;           // [P_l][12]
  double *dnorm;       // [P_l]
  double *part;        // [n_slices*RG][P_l][NACC]
  double *rec;         // [2][rec_stride]: records [P_rec][REC], double buffered by iteration parity (SVGD-ICP class: buffer 0 only)
  size_t rec_stride;   // doubles per record buffer
  Ctrl *ctrl;
  // launch shape of the Gauss-Newton kernel
  int TB, stages, n_slices, n_pgroups, PG, RG;
  int gn_lag;          // k_gn: a tile's stage is refilled gn_lag tiles after it was consumed (1 or 2)
  size_t gn_smem;
  int sm_count;
  int svn_full_grad;
  int first_order;     // 1: SVGD-ICP class -- k_gn sums the first-order quantities only (svgd_class.cu)
  // debug taps (may be null)
  int32_t *dbg_idx;
  uint8_t *dbg_mask;
};
#ifdef __CUDACC__
// Fixed-order fp64 sum of the Gauss-Newton partial rows of local particle l (k_finalize, k_finalize_first): one CTA of
// nw = blockDim.x / 32 warps per particle (fin_threads: 4 warps, 8 when there are many partial rows -- small particle counts,
// where k_gn runs many row groups).  Lane (j = lane & 15, half = lane >> 4) of warp w sums partial rows half + 2 (w + nw k) of sum
// j over four independent chains, the odd half joins the even one, then the warps are added in ascending order.
// The order depends only on the number of partial rows, never on timing.  Result: v[0..NACC) valid in EVERY thread of the CTA.
constexpr int FIN_WARPS = 8;  // at most
__host__ __device__ inline int fin_rows(const IterArgs &a) { return a.n_slices * (a.RG < a.TB ? a.RG : a.TB); }  // row groups beyond TB own no rows
inline int fin_threads(const IterArgs &a) { return fin_rows(a) > 512 ? FIN_WARPS * 32 : 128; }
__device__ __forceinline__ void gn_sum_partials(const IterArgs &a, int l, double v[NACC]) {
  __shared__ double s_fin[FIN_WARPS][NACC];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int nrows = fin_rows(a);
  const int j16 = lane & 15, half = lane >> 4;
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  const int step = 2 * nw;
  int r = half + 2 * w;
  for (; r + 3 * step < nrows; r += 4 * step) {
    s0 += a.part[((size_t)r * a.P_l + l) * NACC + j16];
    s1 += a.part[((size_t)(r + step) * a.P_l + l) * NACC + j16];
    s2 += a.part[((size_t)(r + 2 * step) * a.P_l + l) * NACC + j16];
    s3 += a.part[((size_t)(r + 3 * step) * a.P_l + l) * NACC + j16];
  }
  for (; r < nrows; r += step) s0 += a.part[((size_t)r * a.P_l + l) * NACC + j16];
  double s = (s0 + s1) + (s2 + s3);
  s += __shfl_down_sync(0xffffffffu, s, 16);
  if (lane < NACC) s_fin[w][lane] = s;
  __syncthreads();
#pragma unroll
  for (int j = 0; j < NACC; j++) {
    double t = s_fin[0][j];
    for (int ww = 1; ww < nw; ww++) t += s_fin[ww][j];
    v[j] = t;
  }
}
#endif
int launch_prep(const IterArgs &a, cudaStream_t st, int all_x, const double *x_src);
int launch_filter(const IterArgs &a, cudaStream_t st);
int launch_gn(const IterArgs &a, cudaStream_t st);
int launch_finalize(const IterArgs &a, const PeerTable &pt, unsigned seq_h, cudaStream_t st);
void init_iter_kernels();
// bytes of one shared-memory stage of k_gn: TB pruned rows of K float4 + TB row headers + 3 row-class masks, 128-byte aligned
__host__ __device__ inline size_t gn_stage_bytes(int TB, int K) { return ((size_t)TB * K * 16 + (size_t)TB * 16 + 16 + 127) & ~(size_t)127; }
// k_gn launch shape: one CTA per SM of GN_CONSUMERS threads (each carries two particles; the warps take turns loading tiles).
// Dynamic shared memory: [S] stages, 2*S mbarriers, then the second-level accumulators [NACC][GN_CONSUMERS] fp32 pairs.
constexpr int GN_CONSUMERS = 512;
constexpr int GN_THREADS = GN_CONSUMERS;
__host__ __device__ inline size_t gn_dacc_offset(int TB, int K, int S) { return (gn_stage_bytes(TB, K) * S + 2 * (size_t)S * 8 + 127) & ~(size_t)127; }
__host__ __device__ inline size_t gn_smem_bytes(int TB, int K, int S) { return gn_dacc_offset(TB, K, S) + (size_t)NACC * GN_CONSUMERS * 8; }

struct SteinArgs {
  int P, p_lo, P_l, I;
  int svn_full_grad, check_early_stop;
  double lr, threshold;
  double *rec;       // [2][rec_stride] (see IterArgs)
  size_t rec_stride; // SVN-ICP class: doubles per record buffer; SVGD-ICP class: 0, one buffer
  double *xs;        // [6][P] SoA copy of x at the head of the iteration (median sweeps, get_gn_system of the SVGD-ICP class)
  double *delta;     // [P_l][6]
  double *dnorm;     // [P_l]
  double *R, *t;
  double *Hbar_inv;  // [36]
  unsigned *hist;    // [MED_PASSES][MED_BINS]
  float *history;    // [I][6][P]
  Ctrl *ctrl;
  double *stats;     // [6 + 6 + 36] mean, var, cov
  double *particles; // [6][P]
  unsigned long long *kept_hist;  // [I] candidates kept by the prune pass per iteration (statistics)
  int32_t *med_path;              // [I + 2] how k_head_* settled each iteration's median (MED_PATH_*; -1 = not computed)
  double *prep_scratch_d;         // [sm_count][12] per-CTA partial sums of the fused tail kernel
  int *prep_scratch_i;            // [PRUNE_BINS + 3] envelope / alpha / beta / NaN flag maxima (bit patterns)
  double *stamps;                 // [8] globaltimer stamps of k_tail's phases (tuning aid; null = off)
  int sm_count;
};
// Stein phase (tail2.cu): k_head_* = early-stop decision + history row + exact median bandwidth (a chain of small ordinary
// kernels; both classes), k_tail = Stein step + pose update + next iteration's transforms and pruning ball (SVN-ICP class).
// seq_x / seq_h / seq_x_out: sequence numbers of the peer exchange (0 = nothing to wait for).  Return launches or -1.
int launch_head(const SteinArgs &a, const PeerTable &pt, unsigned seq_x, int epilogue, cudaStream_t st);
int launch_tail(const SteinArgs &a, const IterArgs &ia, const PeerTable &pt, unsigned seq_h, unsigned seq_x_out, cudaStream_t st);
// getters from the record buffer; parity_from_ctrl: read the buffer of parity (iters_done & 1) (SVN-ICP class)
int launch_stats(const SteinArgs &a, int parity_from_ctrl, cudaStream_t st);
// restart of the device-side iteration state at the head of every stein_align (poses are kept)
int launch_align_reset(Ctrl *ctrl, double *opt_state, size_t n_opt, cudaStream_t st);
int launch_init_particles(double *R, double *t, const double *init_pose_dev, int P, double *dnorm, int p_lo, int P_l, Ctrl *ctrl,
                          cudaStream_t st);


// ---- svnicp_evaluate (eval_kernels.cu): registration objective of the last scan's candidate table at given poses ----
constexpr int EV_NS = NACC + 2;  // per-pose sums: the 16 Gauss-Newton sums, inlier count, sum of inlier d^2
constexpr int EV_OUT = 45;       // per-pose result: {count, fraction, rmse}, H [36], b [6]
constexpr int EV_BLOCK = 32;     // poses per pass over the table
struct EvalArgs {
  int n_s, K;
  float max_dist;
  const float4 *sp, *cand;
  const int *cand_idx;  // [n_s][K] global map index per slot (only read when idx != null)
  const float *xf;      // [MB][12] fp32 transforms of the block's poses
  int MB, G;            // poses in the block (<= EV_BLOCK); lane groups = MB rounded up to a power of two
  double *part;         // [eval_parts][MB][EV_NS] per-CTA partial sums
  uint8_t *mask;        // [MB][n_s] or null
  int32_t *idx;         // [MB][n_s] or null
};
int eval_parts(int n_s, int K, int sm_count);  // CTAs of the correspondence pass = partial slots per pose
int launch_eval_prep(const double *poses, int M, int euler, const ScanConst &sc, float *xf, double *R, cudaStream_t st);
int launch_eval_block(const EvalArgs &a, bool want_system, const ScanConst &sc, const double *R_blk, double *out_blk, int sm_count,
                      cudaStream_t st);
// k_eval_fin alone: per-CTA partials part [n_parts][MB][EV_NS] -> out_blk [MB][EV_OUT] (stats, then H and b by gn_assemble with
// sc.R0 and the poses' rotations R_blk [MB][9]).  Also the back end of svnicp_map_evaluate (voxel_map.cu).
int launch_eval_fin(const double *part, int n_parts, int MB, int n_s, const ScanConst &sc, const double *R_blk, double *out_blk,
                    cudaStream_t st);
void init_eval_kernels();

// ---- SVGD-ICP class (class_type = SVGDICP, svgd_class.cu): first-order gradient + torch::optim-style update ----
enum { SVGD_OPT_ADAM = 0, SVGD_OPT_RMSPROP = 1, SVGD_OPT_SGD = 2, SVGD_OPT_ADAGRAD = 3 };
struct SvgdArgs {
  int P, p_lo, P_l;
  int optimizer;       // SVGD_OPT_*
  double lr;
  double *pose6;       // [P_pad][6] the parameters x_,y_,z_,rx_,ry_,rz_ (global particle index; local slice is live)
  double *prev;        // [P][6] pose_particles_ as stein_align finds it (constructor / previous scan; SVGDICP.cpp:46-62)
  double *opt_state;   // [P_l][12] optimizer moments, zeroed per scan (SVGDICP.cpp:73)
};
int launch_svgd_init(const SvgdArgs &s, const double *init_pose_dev, double *R, double *t, double *dnorm, Ctrl *ctrl, cudaStream_t st);
int launch_finalize_first(const IterArgs &a, const SvgdArgs &s, cudaStream_t st);
int launch_svgd_rec(double *rec, const double *src6, const double *dnorm, int lo, int n, int dn_off, cudaStream_t st);
int launch_stein_first(const SteinArgs &a, cudaStream_t st);
int launch_update_opt(const SteinArgs &a, const SvgdArgs &s, int step, cudaStream_t st);
int launch_stats_svgd(const SteinArgs &a, double *prev_out, cudaStream_t st);

}  // namespace svn
