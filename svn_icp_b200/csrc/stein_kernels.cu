// stein_kernels.cu -- particle initialisation, the per-scan reset and the getters.
// (The Stein phase runs in tail2.cu -- k_head_* for both classes, k_tail for SVN-ICP -- and svgd_class.cu.)
//
//   k_particles_init     SVGDICP::add_cloud :46-61 with SVNICP's Exp (SVNICP.cpp:166-194)
//   k_align_reset        head of every stein_align
//   k_stats              getters :281-308  weighted mean / variance / covariance
// All fp64.
#include "common.cuh"
#include "kernels.h"

namespace svn {

// ---------------------------------------------------------------------------------------------
// k_particles_init: SVGDICP::add_cloud (SVGDICP.cpp:46-61) with SVNICP's Exp (SVNICP.cpp:166-194)
// ---------------------------------------------------------------------------------------------
__global__ void k_particles_init(double *R, double *t, const double *init_pose, int P, double *dnorm, int p_lo, int P_l, Ctrl *ctrl) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p == 0) {
    ctrl->stop = 0; ctrl->iter = 0; ctrl->iters_done = 0; ctrl->bandwidth = 0.0; ctrl->kept_total = 0ull;
  }
  if (p >= P) return;
  const double r[3] = {init_pose[3 * P + p], init_pose[4 * P + p], init_pose[5 * P + p]};
  double Rm[9];
  so3_exp(r, Rm, nullptr);
  for (int i = 0; i < 9; i++) R[9 * (size_t)p + i] = Rm[i];
  for (int i = 0; i < 3; i++) t[3 * (size_t)p + i] = init_pose[i * P + p];
  if (p >= p_lo && p < p_lo + P_l) dnorm[p - p_lo] = 0.0;
}

// k_align_reset: head of every stein_align.  A second scan without add_cloud continues from the current poses (as the
// reference does) but with fresh iteration counters, stop flag and -- SVGD-ICP class -- optimizer moments (SVGDICP.cpp:73).
__global__ void k_align_reset(Ctrl *ctrl, double *opt_state, size_t n_opt) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0) {
    ctrl->stop = 0; ctrl->iter = 0; ctrl->iters_done = 0; ctrl->kept_total = 0ull;
    ctrl->error = 0; ctrl->fin_ticket = 0u; ctrl->tail_ticket = 0u;
  }
  for (size_t k = i; k < n_opt; k += (size_t)gridDim.x * blockDim.x) opt_state[k] = 0.0;
}

// ---------------------------------------------------------------------------------------------
// k_stats: getters (SVNICP.cpp:281-308) from the gathered record.  One CTA.
// weights = float32(1)/P promoted to double (SVNICP.cpp:46, :281-284).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) k_stats(SteinArgs a, int parity_from_ctrl) {
  // SVN-ICP class: the final poses sit in the record buffer of parity (number of updates applied & 1)
  if (parity_from_ctrl) a.rec += (size_t)(a.ctrl->iters_done & 1) * a.rec_stride;
  __shared__ double s_red[32][36];
  __shared__ double s_mean[6];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
  const double w = (double)(1.0f / (float)a.P);
  for (int i = tid; i < 6 * a.P; i += blockDim.x) {
    const int comp = i / a.P, p = i % a.P;
    a.particles[i] = a.rec[(size_t)p * REC + REC_X + comp];  // get_particles: [6][P] (SVGDICP.cpp:515-520)
  }
  double acc[36];
#pragma unroll
  for (int q = 0; q < 6; q++) acc[q] = 0.0;
  for (int p = tid; p < a.P; p += blockDim.x)
#pragma unroll
    for (int q = 0; q < 6; q++) acc[q] += a.rec[(size_t)p * REC + REC_X + q] * w;  // :288
#pragma unroll
  for (int q = 0; q < 6; q++) acc[q] = warp_sum(acc[q]);
  if (lane == 0)
#pragma unroll
    for (int q = 0; q < 6; q++) s_red[warp][q] = acc[q];
  __syncthreads();
  if (tid < 6) {
    double s = 0.0;
    for (int ww = 0; ww < nw; ww++) s += s_red[ww][tid];
    s_mean[tid] = s;
    a.stats[tid] = s;
  }
  __syncthreads();
#pragma unroll
  for (int q = 0; q < 36; q++) acc[q] = 0.0;
  for (int p = tid; p < a.P; p += blockDim.x) {
    double d[6];
#pragma unroll
    for (int q = 0; q < 6; q++) d[q] = a.rec[(size_t)p * REC + REC_X + q] - s_mean[q];
#pragma unroll
    for (int r = 0; r < 6; r++)
#pragma unroll
      for (int cc = 0; cc < 6; cc++) acc[6 * r + cc] += w * (d[r] * d[cc]);  // :302-304
  }
#pragma unroll
  for (int q = 0; q < 36; q++) acc[q] = warp_sum(acc[q]);
  __syncthreads();
  if (lane == 0)
#pragma unroll
    for (int q = 0; q < 36; q++) s_red[warp][q] = acc[q];
  __syncthreads();
  if (tid < 36) {
    double s = 0.0;
    for (int ww = 0; ww < nw; ww++) s += s_red[ww][tid];
    a.stats[12 + tid] = s;                     // covariance, row-major 36 (:305-306)
    if (tid % 7 == 0) a.stats[6 + tid / 7] = s;  // variance (:294-295) = diagonal of the same weighted sum
  }
}

// ---------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------
static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

int launch_align_reset(Ctrl *ctrl, double *opt_state, size_t n_opt, cudaStream_t st) {
  k_align_reset<<<n_opt > 4096 ? 32 : 1, 256, 0, st>>>(ctrl, opt_state, n_opt);
  return 1;
}

int launch_init_particles(double *R, double *t, const double *init_pose_dev, int P, double *dnorm, int p_lo, int P_l, Ctrl *ctrl,
                          cudaStream_t st) {
  k_particles_init<<<cdiv(P, 128), 128, 0, st>>>(R, t, init_pose_dev, P, dnorm, p_lo, P_l, ctrl);
  return 1;
}

int launch_stats(const SteinArgs &a, int parity_from_ctrl, cudaStream_t st) {
  k_stats<<<1, 1024, 0, st>>>(a, parity_from_ctrl);
  return 1;
}

}  // namespace svn
