// svgd_class.cu -- the SVGD-ICP class (`class_type = SVGDICP`, OdometryPipeline.cpp:282-288) on the same device
// pipeline as SVN-ICP.  Replaces, per iteration of SVGDICP::stein_align (reference svn-icp/src/core/SVGDICP.cpp:81-134):
//   to_rotation_tensor   :226-260  ZYX Euler -> R                                  (k_svgd_init, k_update_opt)
//   transform + get_correspondence_fast + point_filter :94-101, :300-333           (k_prep/k_filter/k_gn, shared)
//   partial_derivative + sgd_grad :335-455                                         (k_gn<FIRST> + k_finalize_first)
//   rbf_kernel + svgd_grad :457-474                                                (k_head_* shared, k_stein_first)
//   pose_update :476-494 = torch::optim::{Adam,RMSprop,SGD,Adagrad}::step          (k_update_opt)
//   early stop :123-131, history :133, getters :497-534                            (k_head_* shared, k_stats_svgd)
//
// Why the SVN-ICP correspondence kernel serves unchanged: each Euler partial is dR/dtheta_k = [omega_k]x R with
//   omega_roll = R(:,0) of Rz Ry = (cp cy, cp sy, -sp),  omega_pitch = (-sy, cy, 0),  omega_yaw = (0, 0, 1),
// so  sum_b rho e . (R0 dR_k s) = (R0 omega_k) . sum_b rho (w x e),  w = R0 R s  -- the cross-product sum C that k_gn
// already accumulates (sums 13..15), next to E = sum rho e (sums 10..12).  Only the pair count is new (sum 0).
#include "common.cuh"
#include "kernels.h"

namespace svn {

__device__ __forceinline__ void euler_R(const double *x6, double *R) {  // SVGDICP.cpp:226-260
  double sr, cr, sp, cp, sy, cy;
  sincos(x6[3], &sr, &cr);
  sincos(x6[4], &sp, &cp);
  sincos(x6[5], &sy, &cy);
  R[0] = cp * cy; R[1] = sr * sp * cy - cr * sy; R[2] = sr * sy + cr * sp * cy;
  R[3] = cp * sy; R[4] = cr * cy + sr * sp * sy; R[5] = cr * sp * sy - sr * cy;
  R[6] = -sp;     R[7] = sr * cp;                R[8] = cr * cp;
}

// SVGDICP::add_cloud (:46-61): parameters from init_pose [6][P]; optimizer moments cleared (set_optimizer, :73, :142-170)
__global__ void k_svgd_init(SvgdArgs s, const double *init_pose, double *R, double *t, double *dnorm, Ctrl *ctrl) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p == 0) {
    ctrl->stop = 0; ctrl->iter = 0; ctrl->iters_done = 0; ctrl->bandwidth = 0.0; ctrl->kept_total = 0ull;
  }
  if (p >= s.P) return;
  double x[6];
  for (int c = 0; c < 6; c++) { x[c] = init_pose[(size_t)c * s.P + p]; s.pose6[(size_t)p * 6 + c] = x[c]; }
  double Rm[9];
  euler_R(x, Rm);
  for (int i = 0; i < 9; i++) R[9 * (size_t)p + i] = Rm[i];
  for (int i = 0; i < 3; i++) t[3 * (size_t)p + i] = x[i];
  if (p >= s.p_lo && p < s.p_lo + s.P_l) {
    dnorm[p - s.p_lo] = 0.0;
    for (int i = 0; i < 12; i++) s.opt_state[(size_t)(p - s.p_lo) * 12 + i] = 0.0;
  }
}

// partial sums -> sgd_grad of one particle (one warp each), into the gathered record:
//   rec.x = the particle's KERNEL position (pose_particles_: `prev` in iteration 0, the parameters afterwards)
//   rec.b = sgd_gradient * gradient_scaling_factor_   (:454)
__global__ void __launch_bounds__(FIN_WARPS * 32) k_finalize_first(IterArgs a, SvgdArgs s) {
  if (a.ctrl->stop) return;
  const int l = blockIdx.x;  // one CTA (FIN_WARPS warps) per local particle, same fixed order as k_finalize
  double v[NACC];
  gn_sum_partials(a, l, v);
  if (threadIdx.x != 0) return;
  const int p = a.p_lo + l;
  const double *R0 = a.sc.R0;
  const double *x = s.pose6 + (size_t)p * 6;
  double sp, cp, sy, cy;
  sincos(x[4], &sp, &cp);
  sincos(x[5], &sy, &cy);
  const double om[3][3] = {{cp * cy, cp * sy, -sp}, {-sy, cy, 0.0}, {0.0, 0.0, 1.0}};
  const double den = v[0] + 1.0;                // nonzero_count + 1 (:414-416)
  const double scale = (double)a.n_s;           // gradient_scaling_factor_ (:58)
  const double E[3] = {v[10], v[11], v[12]}, C[3] = {v[13], v[14], v[15]};
  double g[6];
#pragma unroll
  for (int c = 0; c < 3; c++) g[c] = (E[0] * R0[c] + E[1] * R0[3 + c] + E[2] * R0[6 + c]) / den * scale;  // error.sum(1).matmul(R0_)
#pragma unroll
  for (int k = 0; k < 3; k++) {
    double w[3];
#pragma unroll
    for (int rr = 0; rr < 3; rr++) w[rr] = R0[3 * rr] * om[k][0] + R0[3 * rr + 1] * om[k][1] + R0[3 * rr + 2] * om[k][2];
    g[3 + k] = (w[0] * C[0] + w[1] * C[1] + w[2] * C[2]) / den * scale;
  }
  double *rec = a.rec + (size_t)p * REC;
  const double *kp = (a.ctrl->iter == 0) ? s.prev + (size_t)p * 6 : x;
#pragma unroll
  for (int i = 0; i < 6; i++) { rec[REC_X + i] = kp[i]; rec[REC_B + i] = g[i]; }
  rec[REC_DNORM] = a.dnorm[l];
}

// rec.x <- src6 rows [lo, lo+n) (scan epilogue: the final parameters; NO_OPTIMIZER: the untouched pose_particles_)
__global__ void k_svgd_rec(double *rec, const double *src6, const double *dnorm, int lo, int n, int dn_off) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int p = lo + i;
  for (int c = 0; c < 6; c++) rec[(size_t)p * REC + REC_X + c] = src6[(size_t)p * 6 + c];
  rec[(size_t)p * REC + REC_DNORM] = dnorm ? dnorm[p - dn_off] : 0.0;
}

// SVGDICP::svgd_grad (:457-462): stein_i = ( sum_j K_ij (-g_j) + (2/h) sum_j (x_i - x_j) K_ij ) / P ; P == 1: -g (:112)
constexpr int SF_WARPS = 8, SF_TJ = 32;
static_assert(REC_X == 0 && REC_B == 6, "k_stein_first stages x and b as record doubles 0..11");
__global__ void __launch_bounds__(SF_WARPS * 32) k_stein_first(SteinArgs a) {
  Ctrl *c = a.ctrl;
  if (c->stop) return;
  __shared__ double s_rec[12][SF_TJ + 1];
  const double h = c->bandwidth;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int l = blockIdx.x * SF_WARPS + warp;
  const bool active = l < a.P_l;
  const int i = a.p_lo + (active ? l : 0);
  if (a.P == 1) {
    if (active && lane == 0)
      for (int d = 0; d < 6; d++) a.delta[d] = -a.rec[(size_t)i * REC + REC_B + d];
    return;
  }
  double xi[6];
#pragma unroll
  for (int d = 0; d < 6; d++) xi[d] = a.rec[(size_t)i * REC + REC_X + d];
  double rep[6], kg[6];
#pragma unroll
  for (int d = 0; d < 6; d++) { rep[d] = 0.0; kg[d] = 0.0; }
  for (int j0 = 0; j0 < a.P; j0 += SF_TJ) {
    __syncthreads();
    for (int e = tid; e < 12 * SF_TJ; e += blockDim.x) {
      const int q = e / SF_TJ, jj = e % SF_TJ;  // s_rec rows 0..5 = x, 6..11 = b (the gradient)
      s_rec[q][jj] = (j0 + jj < a.P) ? a.rec[(size_t)(j0 + jj) * REC + q] : 0.0;
    }
    __syncthreads();
    if (active && j0 + lane < a.P) {
      double dl[6], D = 0.0;
#pragma unroll
      for (int d = 0; d < 6; d++) { dl[d] = xi[d] - s_rec[d][lane]; D += dl[d] * dl[d]; }  // :465-468
      const double kij = exp(-D / h);                                                       // :472
#pragma unroll
      for (int d = 0; d < 6; d++) { rep[d] += dl[d] * kij; kg[d] -= kij * s_rec[6 + d][lane]; }
    }
  }
#pragma unroll
  for (int d = 0; d < 6; d++) { rep[d] = warp_sum(rep[d]); kg[d] = warp_sum(kg[d]); }
  if (active && lane == 0) {
    const double f = 2.0 / h;
    for (int d = 0; d < 6; d++) a.delta[(size_t)l * 6 + d] = (kg[d] + f * rep[d]) / (double)a.P;
  }
}

// one torch::optim step on one scalar (libtorch 2.11 adam.cpp / rmsprop.cpp / sgd.cpp / adagrad.cpp with the options of
// SVGDICP.cpp:142-170); m = st[0], v = st[1]; step is 1-based
__device__ __forceinline__ double opt_step(int opt, double lr, int step, double p, double grad, double *st) {
  switch (opt) {
    case SVGD_OPT_ADAM: {
      const double b1 = 0.9, b2 = 0.999, eps = 1e-8;
      const double bc1 = 1.0 - pow(b1, (double)step), bc2 = 1.0 - pow(b2, (double)step);
      st[0] = st[0] * b1 + grad * (1.0 - b1);
      st[1] = st[1] * b2 + grad * grad * (1.0 - b2);
      const double denom = sqrt(st[1]) / sqrt(bc2) + eps;
      return p + -(lr / bc1) * (st[0] / denom);
    }
    case SVGD_OPT_RMSPROP: {
      const double alpha = 0.99, eps = 1e-8, wd = 1e-8, mom = 0.9;
      grad = grad + wd * p;
      st[0] = st[0] * alpha + grad * grad * (1.0 - alpha);
      const double avg = sqrt(st[0]) + eps;
      st[1] = st[1] * mom + grad / avg;
      return p + -lr * st[1];
    }
    case SVGD_OPT_SGD:
      return p + -lr * grad;
    default: {  // Adagrad
      st[0] += grad * grad;
      const double sd = sqrt(st[0]) + 1e-10;
      return p + -lr * (grad / sd);
    }
  }
}

// SVGDICP::pose_update (:476-494) for the local slice; parameter gradient = -stein_grad
__global__ void k_update_opt(SteinArgs a, SvgdArgs s, int step) {  // step = epoch + 1 (host-known: kernels past a stop are no-ops)
  Ctrl *c = a.ctrl;
  if (c->stop) return;
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l < a.P_l) {
    const int p = a.p_lo + l;
    double x[6], n2 = 0.0;
    for (int i = 0; i < 6; i++) {
      const double old_kernel_pos = a.rec[(size_t)p * REC + REC_X + i];  // pose_particles_old (:114)
      x[i] = opt_step(s.optimizer, s.lr, step, s.pose6[(size_t)p * 6 + i], -a.delta[(size_t)l * 6 + i], s.opt_state + (size_t)l * 12 + 2 * i);
      s.pose6[(size_t)p * 6 + i] = x[i];
      const double df = x[i] - old_kernel_pos;                          // pose_difference (:122)
      n2 += df * df;
    }
    double Rm[9];
    euler_R(x, Rm);                                                      // :88-89 of the next iteration
    for (int i = 0; i < 9; i++) a.R[9 * (size_t)p + i] = Rm[i];
    for (int i = 0; i < 3; i++) a.t[3 * (size_t)p + i] = x[i];
    a.dnorm[l] = sqrt(n2);                                               // :124 norm(2, 0)
  }
  if (l == 0) {
    if (a.kept_hist) a.kept_hist[step - 1] = c->kept_total;  // candidates kept by this iteration's pruning pass
    c->iter = step;
  }
}

// getters (:497-524): plain mean, UNBIASED variance (torch::var), covariance / P; also refreshes pose_particles_ (`prev`)
__global__ void __launch_bounds__(1024) k_stats_svgd(SteinArgs a, double *prev_out) {
  __shared__ double s_red[32][36];
  __shared__ double s_mean[6];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
  for (int i = tid; i < 6 * a.P; i += blockDim.x) {
    const int comp = i / a.P, p = i % a.P;
    const double v = a.rec[(size_t)p * REC + REC_X + comp];
    a.particles[i] = v;                          // get_particles [6][P] (:515-520)
    if (prev_out) prev_out[(size_t)p * 6 + comp] = v;  // pose_particles_ carried into the next scan (:136-138)
  }
  double acc[36];
#pragma unroll
  for (int q = 0; q < 6; q++) acc[q] = 0.0;
  for (int p = tid; p < a.P; p += blockDim.x)
#pragma unroll
    for (int q = 0; q < 6; q++) acc[q] += a.rec[(size_t)p * REC + REC_X + q];
#pragma unroll
  for (int q = 0; q < 6; q++) acc[q] = warp_sum(acc[q]);
  if (lane == 0)
#pragma unroll
    for (int q = 0; q < 6; q++) s_red[warp][q] = acc[q];
  __syncthreads();
  if (tid < 6) {
    double sum = 0.0;
    for (int ww = 0; ww < nw; ww++) sum += s_red[ww][tid];
    s_mean[tid] = sum / (double)a.P;             // :497-499
    a.stats[tid] = s_mean[tid];
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
      for (int cc = 0; cc < 6; cc++) acc[6 * r + cc] += d[r] * d[cc];
  }
#pragma unroll
  for (int q = 0; q < 36; q++) acc[q] = warp_sum(acc[q]);
  __syncthreads();
  if (lane == 0)
#pragma unroll
    for (int q = 0; q < 36; q++) s_red[warp][q] = acc[q];
  __syncthreads();
  if (tid < 36) {
    double sum = 0.0;
    for (int ww = 0; ww < nw; ww++) sum += s_red[ww][tid];
    a.stats[12 + tid] = sum / (double)a.P;                              // :505-509
    if (tid % 7 == 0) a.stats[6 + tid / 7] = sum / (double)(a.P - 1);   // :501-503 (P == 1: 0/0 = NaN like torch::var)
  }
}

static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

int launch_svgd_init(const SvgdArgs &s, const double *init_pose_dev, double *R, double *t, double *dnorm, Ctrl *ctrl, cudaStream_t st) {
  k_svgd_init<<<cdiv(s.P, 128), 128, 0, st>>>(s, init_pose_dev, R, t, dnorm, ctrl);
  return 1;
}
int launch_finalize_first(const IterArgs &a, const SvgdArgs &s, cudaStream_t st) {
  if (a.P_l > 0) k_finalize_first<<<a.P_l, fin_threads(a), 0, st>>>(a, s);
  return 1;
}
int launch_svgd_rec(double *rec, const double *src6, const double *dnorm, int lo, int n, int dn_off, cudaStream_t st) {
  if (n < 1) return 0;
  k_svgd_rec<<<cdiv(n, 128), 128, 0, st>>>(rec, src6, dnorm, lo, n, dn_off);
  return 1;
}
int launch_stein_first(const SteinArgs &a, cudaStream_t st) {
  k_stein_first<<<cdiv(a.P_l > 0 ? a.P_l : 1, SF_WARPS), SF_WARPS * 32, 0, st>>>(a);
  return 1;
}
int launch_update_opt(const SteinArgs &a, const SvgdArgs &s, int step, cudaStream_t st) {
  k_update_opt<<<cdiv(a.P_l > 0 ? a.P_l : 1, 128), 128, 0, st>>>(a, s, step);
  return 1;
}
int launch_stats_svgd(const SteinArgs &a, double *prev_out, cudaStream_t st) {
  k_stats_svgd<<<1, 1024, 0, st>>>(a, prev_out);
  return 1;
}

}  // namespace svn
