// iter_kernels.cu -- the per-iteration correspondence + Gauss-Newton pass (north_star kernels (a)+(b)).
//
// Replaces, per iteration of SVNICP::stein_align (reference svn-icp/src/core/SVNICP.cpp:52-71):
//   transform            SVNICP.cpp:58-64
//   get_correspondence_fast + KNearestNeighborKernelV3<double,3,1>   SVGDICP.cpp:300-329, knn.cu:204-251
//   point_filter         SVGDICP.cpp:331-333
//   Newton_grad_right    SVNICP.cpp:116-164  (J [P,B,3,6] is never materialised)
//
//   k_prep     fp64 particle state -> fp32 transforms in coordinates RELATIVE to q0_b, plus the ball
//              (centre transform, alpha, beta) that bounds every particle's query around the centre query.
//   k_filter   HBM-streaming pass over the candidate table: per source point keeps exactly the candidates
//              that can be the nearest neighbour of ANY particle of the slice (triangle inequality around
//              the centre query), in slot order.  Reads 16*N_s*(K+1) bytes: the HBM-roofline kernel.
//   k_gn       fused transform + 1-NN over the pruned lists + robust weight + Gauss-Newton reduction.
//              Lists are staged through shared memory with 1-D TMA bulk copies (cp.async.bulk +
//              mbarrier, S stages, the 16 warps of the CTA take turns as producer); one thread owns TWO
//              particles in packed fp32 pairs (FFMA2 / FADD2 / FMUL2) and keeps their 16 sums in registers
//              (fp32 per 32 rows, folded into fp32 shared-memory slots, then fp64), so no cross-thread
//              reduction is needed until the per-CTA partials are summed by k_finalize.
//   k_finalize fixed-order fp64 sum of the partials -> H (21), b (6) of the reference's system.
//
// Arithmetic that decides a correspondence index is written with explicit _rn intrinsics and is restated
// operation by operation in oracle/svn_oracle.c (oracle_corr_f32) for the bit-exact index parity test.
#include "common.cuh"
#include "kernels.h"
#include "ptx.cuh"

namespace svn {

// ---------------------------------------------------------------------------------------------
// k_prep
// ---------------------------------------------------------------------------------------------
// all_x (SVN-ICP class, head of a scan): x = [t ; Log R] of EVERY particle goes into record buffer 0 -- each rank can do that
// alone because add_cloud gives every rank all initial poses; x_src != null (stein_align called again without add_cloud on a
// sharded handle, where R, t of the other ranks' particles are stale): their x is carried over from the previous result.
__global__ void __launch_bounds__(1024) k_prep(IterArgs a, int all_x, const double *x_src) {
  if (a.ctrl->stop) return;
  __shared__ double s_red[32][12];
  __shared__ float s_center[12];
  __shared__ double s_max[32][2];
  __shared__ int s_env[PRUNE_BINS];
  __shared__ int s_nan;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const double *R0 = a.sc.R0;
  double acc[12];
#pragma unroll
  for (int i = 0; i < 12; i++) acc[i] = 0.0;
  for (int l = tid; l < a.P_l; l += blockDim.x) {
    const int p = a.p_lo + l;
    double R[9], t[3], w[3];
#pragma unroll
    for (int i = 0; i < 9; i++) R[i] = a.R[9 * (size_t)p + i];
#pragma unroll
    for (int i = 0; i < 3; i++) t[i] = a.t[3 * (size_t)p + i];
    so3_log(R, w);  // SVNICP.cpp:74-77
    double *rec = a.rec + (size_t)p * REC;
#pragma unroll
    for (int i = 0; i < 3; i++) { rec[REC_X + i] = t[i]; rec[REC_X + 3 + i] = w[i]; }
    rec[REC_DNORM] = a.dnorm[l];
    float f[12];
    rel_transform_f32(R0, R, t, f);  // A' = R0 (R - I) R0^T, tau = R0 t
    float *xf = a.xf + (size_t)l * 12;
#pragma unroll
    for (int i = 0; i < 12; i++) { xf[i] = f[i]; acc[i] += (double)f[i]; }
  }
  if (all_x)
    for (int p = tid; p < a.P; p += blockDim.x) {
      if (p >= a.p_lo && p < a.p_lo + a.P_l) continue;
      double *rec = a.rec + (size_t)p * REC;
      if (x_src) {
#pragma unroll
        for (int i = 0; i < 6; i++) rec[REC_X + i] = x_src[(size_t)p * REC + REC_X + i];
      } else {
        double R[9], w[3];
#pragma unroll
        for (int i = 0; i < 9; i++) R[i] = a.R[9 * (size_t)p + i];
        so3_log(R, w);
#pragma unroll
        for (int i = 0; i < 3; i++) { rec[REC_X + i] = a.t[3 * (size_t)p + i]; rec[REC_X + 3 + i] = w[i]; }
      }
      rec[REC_DNORM] = 0.0;
    }
#pragma unroll
  for (int i = 0; i < 12; i++) acc[i] = warp_sum(acc[i]);
  if (lane == 0)
#pragma unroll
    for (int i = 0; i < 12; i++) s_red[warp][i] = acc[i];
  __syncthreads();
  if (tid < 12) {
    double s = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) s += s_red[w][tid];
    s_center[tid] = __double2float_rn(s / (double)a.P_l);
  }
  __syncthreads();
  for (int i = tid; i < PRUNE_BINS; i += blockDim.x) s_env[i] = 0;
  __syncthreads();
  double ma = 0.0, mb = 0.0;
  for (int l = tid; l < a.P_l; l += blockDim.x) {
    const float *xf = a.xf + (size_t)l * 12;
    double M[9], db = 0;
#pragma unroll
    for (int i = 0; i < 9; i++) M[i] = (double)xf[i] - (double)s_center[i];
#pragma unroll
    for (int i = 9; i < 12; i++) { const double d = (double)xf[i] - (double)s_center[i]; db += d * d; }
    // |(A_p - Abar) s| <= sigma_max(A_p - Abar) |s|: largest eigenvalue of M^T M (trigonometric closed form)
    double da = sym3_max_eig_MtM(M);
    // NaN state (e.g. the reference's P == 2 bandwidth-0 quirk) must poison the radius, not vanish in fmax
    ma = (da != da) ? da : fmax(ma, da);
    mb = (db != db) ? db : fmax(mb, db);
    // per-range-bin envelope max_p (sigma_p r + beta_p) at the bin's upper edge r (tighter than max sigma * r + max beta)
    if (da == da && db == db) {
      const double sg = sqrt(da) * (1.0 + 1e-6), bt = sqrt(db) * (1.0 + 1e-6);
      for (int i = 0; i < PRUNE_BINS; i++) {
        const float v = __double2float_ru(sg * ((double)(i + 1) * PRUNE_BIN_W) + bt);
        atomicMax(&s_env[i], __float_as_int(v));  // non-negative floats order like their bit patterns
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double oa = __shfl_xor_sync(0xffffffffu, ma, o), ob = __shfl_xor_sync(0xffffffffu, mb, o);
    ma = (oa != oa || ma != ma) ? NAN : fmax(ma, oa);
    mb = (ob != ob || mb != mb) ? NAN : fmax(mb, ob);
  }
  if (lane == 0) { s_max[warp][0] = ma; s_max[warp][1] = mb; }
  __syncthreads();
  if (tid == 0) {
    double fa = 0, fb = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) {
      fa = (s_max[w][0] != s_max[w][0] || fa != fa) ? NAN : fmax(fa, s_max[w][0]);
      fb = (s_max[w][1] != s_max[w][1] || fb != fb) ? NAN : fmax(fb, s_max[w][1]);
    }
    Ctrl *c = a.ctrl;
    for (int i = 0; i < 9; i++) c->Abar[i] = s_center[i];
    for (int i = 0; i < 3; i++) c->taubar[i] = s_center[9 + i];
    c->alpha = __double2float_ru(sqrt(fa) * (1.0 + 1e-6));
    c->beta = __double2float_ru(sqrt(fb) * (1.0 + 1e-6));
    c->kept_total = 0ull;
    s_nan = (fa != fa || fb != fb) ? 1 : 0;
  }
  __syncthreads();
  for (int i = tid; i < PRUNE_BINS; i += blockDim.x) a.ctrl->env[i] = s_nan ? NAN : __int_as_float(s_env[i]);
}

// ---------------------------------------------------------------------------------------------
// k_filter: exact candidate pruning, one warp per source point (the HBM-streaming kernel)
// ---------------------------------------------------------------------------------------------
constexpr float PRUNE_MARGIN = 1e-4f;  // metres; absorbs every fp32 rounding in q, qbar and the norms

// Which pruning kernel runs this iteration (both are launched, one returns at once; decided on the device because the
// host runs ahead of the GPU): while the lists are long (mean kept > FR_SWITCH) streaming the K-slot table with a warp per
// row is faster (52 us, HBM bound); once they are short, k_filter_reuse prunes the previous lists with a thread per row.
constexpr int FR_SWITCH = 12;
__device__ __forceinline__ bool filter_use_reuse(const IterArgs &a) {
  if (!a.clist_prev || !a.kept_hist) return false;
  const int it = a.ctrl->iter;
  if (it < 1) return false;
  const unsigned long long kept_prev = a.kept_hist[it - 1] & ((1ull << 40) - 1ull);
  return kept_prev <= (unsigned long long)FR_SWITCH * (unsigned long long)a.n_s;
}

template <int NCH>
__global__ void __launch_bounds__(256, 4) k_filter(IterArgs a) {  // 64 registers: four CTAs per SM keep the HBM pipe full
  if (a.ctrl->stop) return;
  if (filter_use_reuse(a)) return;  // k_filter_reuse takes this iteration
  const int lane = lane_id();
  const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
  const Ctrl *c = a.ctrl;
  float A[9], tb[3];
#pragma unroll
  for (int i = 0; i < 9; i++) A[i] = c->Abar[i];
#pragma unroll
  for (int i = 0; i < 3; i++) tb[i] = c->taubar[i];
  const float alpha = c->alpha, beta = c->beta;
  const int K = a.K, Kp = a.Kp;
  const unsigned lt = (1u << lane) - 1u;
  unsigned long long kept = 0;
  for (int b = gw; b < a.n_s; b += nw) {
    const float4 s = a.sp[b];
    const float qx = fmaf(A[0], s.x, fmaf(A[1], s.y, fmaf(A[2], s.z, tb[0])));
    const float qy = fmaf(A[3], s.x, fmaf(A[4], s.y, fmaf(A[5], s.z, tb[1])));
    const float qz = fmaf(A[6], s.x, fmaf(A[7], s.y, fmaf(A[8], s.z, tb[2])));
    // radius of the ball that holds every particle's query for this point: the per-range-bin envelope where it
    // applies, never worse than sigma_max * |s| + beta_max
    float rho = fmaf(alpha, s.w, beta);
    const int rbin = (int)(s.w * (float)(1.0 / PRUNE_BIN_W));
    if (rbin < PRUNE_BINS) rho = fminf(rho, c->env[rbin]);  // fminf: a NaN env entry leaves rho (itself NaN then) alone
    const float4 *row = a.cand + (size_t)b * K;
    float4 e[NCH];
    float d2[NCH];
    float dmin = INFINITY;
#pragma unroll
    for (int ch = 0; ch < NCH; ch++) {
      const int k = ch * 32 + lane;
      if (k < K) {
        e[ch] = __ldcs(row + k);  // streamed once per iteration: do not keep in L2
        const float dx = qx - e[ch].x, dy = qy - e[ch].y, dz = qz - e[ch].z;
        d2[ch] = fmaf(dz, dz, fmaf(dy, dy, dx * dx));
        dmin = fminf(dmin, d2[ch]);  // fminf drops NaN: a NaN d2 never becomes the minimum
      } else {
        d2[ch] = INFINITY;
      }
    }
    dmin = warp_min(dmin);
    // any candidate farther than d_min + 2 rho from the centre query cannot be (or tie with) the
    // nearest neighbour of a query within rho of it
    const float lim = sqrtf(dmin) + 2.0f * rho + PRUNE_MARGIN;
    const float thr = lim * lim * (1.0f + 1e-5f);
    float4 *out = a.clist + (size_t)b * Kp;
    int base = 0;
#pragma unroll
    for (int ch = 0; ch < NCH; ch++) {
      const int k = ch * 32 + lane;
      const bool keep = (k < K) && !(d2[ch] > thr);  // NaN anywhere keeps everything (NaN must propagate)
      const unsigned m = __ballot_sync(0xffffffffu, keep);
      if (keep) out[base + __popc(m & lt)] = e[ch];
      base += __popc(m);
    }
    // pad to a multiple of 4 with sentinels that can never win (d = inf, strict '<') so k_gn scans in chunks of 4
    const int padded = (base <= 2) ? 2 : ((base + 3) & ~3);  // k_gn scans 2, then chunks of 4
    SVN_CHECK(a.ctrl, padded <= a.Kp && b < a.n_pad, 10);
    if (lane < padded - base) out[base + lane] = make_float4(INFINITY, INFINITY, INFINITY, INFINITY);
    if (lane == 0) {
      a.hdr[b] = make_float4(s.x, s.y, s.z, __int_as_float((padded << 16) | base));  // row header of k_gn: source point + list length
      kept += (unsigned long long)base;
      if (a.ball) { a.cbase[b] = base; a.ball[b] = make_float4(qx, qy, qz, rho); }  // what this list is exact for (k_filter_reuse)
    }
  }
  if (lane == 0 && kept) atomicAdd(&a.ctrl->kept_total, kept);
}

// ---------------------------------------------------------------------------------------------
// k_filter_reuse: the same exact pruning, fed from the PREVIOUS iteration's pruned list where that is provably enough.
// The list of iteration e-1 is exact for every query inside the ball (centre query, rho) it was built for.  If the ball of
// iteration e lies inside it, the nearest candidate of every query of iteration e -- and of the new centre query -- is in
// that list, so pruning it instead of the K-slot row yields the same exact superset (a subsequence, so slot order and the
// ascending-norm property are kept) for a fraction of the HBM traffic.  Measured at configs[1]: the particle cloud contracts
// monotonically and every row takes this path from iteration 2 on.  Rows that fail the containment test (NaN included)
// are pruned from the full row.
// Mapping: a warp takes 32 consecutive rows.  Rows whose previous list is short (<= FR_FAST entries: almost all of them
// once the cloud has contracted) are pruned by ONE THREAD each -- a warp per row would spend ~250 issue slots on three
// candidates, which made the kernel issue bound at ~60 us.  The remaining rows (long lists, failed containment) are then
// pruned one after the other by the whole warp, exactly like k_filter.
// ---------------------------------------------------------------------------------------------
#ifndef SVN_FR_FAST
#define SVN_FR_FAST 256  // measured at configs[1] (late iterations, ncu): 16 -> 30 us (the few long rows serialise whole warps), 128+ -> 19 us
#endif
constexpr int FR_FAST = SVN_FR_FAST;

struct FrRow {
  float sx, sy, sz;
  float qx, qy, qz, rho;
  bool from_prev;
  int n_prev;
};

__device__ __forceinline__ FrRow fr_row_setup(const IterArgs &a, const float *A, const float *tb, float alpha, float beta, int b) {
  const Ctrl *c = a.ctrl;
  const float4 s = a.sp[b];
  const float4 pb = a.ball_prev[b];
  FrRow r;
  r.sx = s.x; r.sy = s.y; r.sz = s.z;
  r.n_prev = a.cbase_prev[b];
  r.qx = fmaf(A[0], s.x, fmaf(A[1], s.y, fmaf(A[2], s.z, tb[0])));
  r.qy = fmaf(A[3], s.x, fmaf(A[4], s.y, fmaf(A[5], s.z, tb[1])));
  r.qz = fmaf(A[6], s.x, fmaf(A[7], s.y, fmaf(A[8], s.z, tb[2])));
  float rho = fmaf(alpha, s.w, beta);
  const int rbin = (int)(s.w * (float)(1.0 / PRUNE_BIN_W));
  if (rbin < PRUNE_BINS) rho = fminf(rho, c->env[rbin]);
  r.rho = rho;
  const float cx = r.qx - pb.x, cy = r.qy - pb.y, cz = r.qz - pb.z;
  const float move = sqrtf(fmaf(cz, cz, fmaf(cy, cy, cx * cx)));
  r.from_prev = fmaf(move, 1.00001f, rho) + 1e-6f <= pb.w;  // ball(q', rho) inside ball(q_prev, rho_prev); NaN -> false
  return r;
}

__global__ void __launch_bounds__(256, 4) k_filter_reuse(IterArgs a) {
  if (a.ctrl->stop) return;
  if (!filter_use_reuse(a)) return;  // k_filter (streaming, warp per row) takes this iteration
  __shared__ unsigned long long s_kept;
  if (threadIdx.x == 0) s_kept = 0ull;
  __syncthreads();
  const int lane = lane_id();
  const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
  const Ctrl *c = a.ctrl;
  float A[9], tb[3];
#pragma unroll
  for (int i = 0; i < 9; i++) A[i] = c->Abar[i];
#pragma unroll
  for (int i = 0; i < 3; i++) tb[i] = c->taubar[i];
  const float alpha = c->alpha, beta = c->beta;
  const int K = a.K, Kp = a.Kp;
  const unsigned lt = (1u << lane) - 1u;
  unsigned long long kept = 0;
  for (int b0 = gw * 32; b0 < a.n_s; b0 += nw * 32) {
    const int b = b0 + lane;
    const bool valid = b < a.n_s;
    FrRow r;
    r.from_prev = false;
    r.n_prev = 0;
    if (valid) r = fr_row_setup(a, A, tb, alpha, beta, b);
    const bool fast = valid && r.from_prev && r.n_prev <= FR_FAST;
    if (fast) {
      // ---- one thread, one row: two passes over <= FR_FAST entries (the second one hits L1)
      const float4 *prow = a.clist_prev + (size_t)b * Kp;
      float dmin = INFINITY;
      for (int k = 0; k < r.n_prev; k++) {
        const float4 e = prow[k];
        const float dx = r.qx - e.x, dy = r.qy - e.y, dz = r.qz - e.z;
        dmin = fminf(dmin, fmaf(dz, dz, fmaf(dy, dy, dx * dx)));
      }
      const float lim = sqrtf(dmin) + 2.0f * r.rho + PRUNE_MARGIN;
      const float thr = lim * lim * (1.0f + 1e-5f);
      float4 *out = a.clist + (size_t)b * Kp;
      int base = 0;
      for (int k = 0; k < r.n_prev; k++) {
        const float4 e = prow[k];
        const float dx = r.qx - e.x, dy = r.qy - e.y, dz = r.qz - e.z;
        const float d2 = fmaf(dz, dz, fmaf(dy, dy, dx * dx));
        if (!(d2 > thr)) out[base++] = e;
      }
      const int padded = (base <= 2) ? 2 : ((base + 3) & ~3);
      SVN_CHECK(a.ctrl, padded <= a.Kp && b < a.n_pad, 11);
      for (int k = base; k < padded; k++) out[k] = make_float4(INFINITY, INFINITY, INFINITY, INFINITY);
      a.hdr[b] = make_float4(r.sx, r.sy, r.sz, __int_as_float((padded << 16) | base));
      a.cbase[b] = base;
      a.ball[b] = make_float4(r.qx, r.qy, r.qz, r.rho);
      kept += (unsigned long long)base + (1ull << 40);  // high bits: rows served by the previous list
    }
    // ---- the other rows, one after the other, by the whole warp (as k_filter)
    unsigned slow = __ballot_sync(0xffffffffu, valid && !fast);
    while (slow) {
      const int src_lane = __ffs(slow) - 1;
      slow &= slow - 1;
      const int bb = b0 + src_lane;
      const float qx = __shfl_sync(0xffffffffu, r.qx, src_lane), qy = __shfl_sync(0xffffffffu, r.qy, src_lane);
      const float qz = __shfl_sync(0xffffffffu, r.qz, src_lane), rho = __shfl_sync(0xffffffffu, r.rho, src_lane);
      const float sx = __shfl_sync(0xffffffffu, r.sx, src_lane), sy = __shfl_sync(0xffffffffu, r.sy, src_lane), sz = __shfl_sync(0xffffffffu, r.sz, src_lane);
      const bool from_prev = __shfl_sync(0xffffffffu, (int)r.from_prev, src_lane) != 0;
      const int n_src = from_prev ? __shfl_sync(0xffffffffu, r.n_prev, src_lane) : K;
      const float4 *row = from_prev ? a.clist_prev + (size_t)bb * Kp : a.cand + (size_t)bb * K;
      float dmin = INFINITY;
      for (int k = lane; k < n_src; k += 32) {
        const float4 e = row[k];
        const float dx = qx - e.x, dy = qy - e.y, dz = qz - e.z;
        dmin = fminf(dmin, fmaf(dz, dz, fmaf(dy, dy, dx * dx)));
      }
      dmin = warp_min(dmin);
      const float lim = sqrtf(dmin) + 2.0f * rho + PRUNE_MARGIN;
      const float thr = lim * lim * (1.0f + 1e-5f);
      float4 *out = a.clist + (size_t)bb * Kp;
      int base = 0;
      for (int k0 = 0; k0 < n_src; k0 += 32) {
        const int k = k0 + lane;
        float4 e = make_float4(0.f, 0.f, 0.f, 0.f);
        bool keep = false;
        if (k < n_src) {
          e = row[k];
          const float dx = qx - e.x, dy = qy - e.y, dz = qz - e.z;
          const float d2 = fmaf(dz, dz, fmaf(dy, dy, dx * dx));
          keep = !(d2 > thr);
        }
        const unsigned m = __ballot_sync(0xffffffffu, keep);
        if (keep) out[base + __popc(m & lt)] = e;
        base += __popc(m);
      }
      const int padded = (base <= 2) ? 2 : ((base + 3) & ~3);
      SVN_CHECK(a.ctrl, padded <= a.Kp && bb < a.n_pad, 12);
      if (lane < padded - base) out[base + lane] = make_float4(INFINITY, INFINITY, INFINITY, INFINITY);
      if (lane == 0) {
        a.hdr[bb] = make_float4(sx, sy, sz, __int_as_float((padded << 16) | base));
        a.cbase[bb] = base;
        a.ball[bb] = make_float4(qx, qy, qz, rho);
        kept += (unsigned long long)base + (from_prev ? (1ull << 40) : 0ull);
      }
    }
  }
  // one global atomic per CTA (the statistic is not worth thousands of same-address atomics per launch)
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) kept += __shfl_xor_sync(0xffffffffu, kept, o);
  if (lane == 0 && kept) atomicAdd(&s_kept, kept);
  __syncthreads();
  if (threadIdx.x == 0 && s_kept) atomicAdd(&a.ctrl->kept_total, s_kept);
}

// ---------------------------------------------------------------------------------------------
// k_gn: fused transform + 1-NN + robust weight + Gauss-Newton reduction
// ---------------------------------------------------------------------------------------------
constexpr int GN_FLUSH_ROWS = 32;
// Three-level accumulation of the 16 Gauss-Newton sums: fp32 registers over GN_FLUSH_ROWS rows -> fp32 in shared memory (the
// thread's own 16 slots: 32 registers less per thread, which is what lets 16 consumer warps share an SM) over GN_FLUSH2 such
// flushes -> the thread's fp64 partial slot.  fp32 second level: measured 30.3 vs 35.5 ms per scan at configs[1] against an
// fp64 second level (round 1), at <= ~5e-7 relative error in H and b.
constexpr int GN_FLUSH2 = 64;

__device__ __forceinline__ float sqrt_approx(float x) {
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));  // one MUFU; feeds only the robust weight and the exit bound
  return r;
}
__device__ __forceinline__ float rcp_approx(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// ---- packed fp32 pairs (sm_100 FFMA2 / FADD2 / FMUL2): one instruction issues the same IEEE-rn operation on two independent
// floats held in an aligned register pair.  The FMA pipe retires the same 128 results/clk/SM either way
// (scripts/ubench/ffma2.cu), but k_gn is bound by instruction ISSUE (75 % issue-slot use at 50 % FMA-pipe use with scalar
// code): a thread that carries two particles needs one issue slot per two flops, and every per-row operand (source point,
// candidate) enters as a broadcast register (`R.F32` operand form: no packing instruction).  Each half is rounded exactly as
// the scalar instruction would round it, so the correspondence indices stay bit-exact.
typedef unsigned long long f2;
__device__ __forceinline__ f2 pk(float a, float b) { f2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ float lo(f2 v) { float a; asm("{ .reg .f32 t; mov.b64 {%0, t}, %1; }" : "=f"(a) : "l"(v)); return a; }
__device__ __forceinline__ float hi(f2 v) { float a; asm("{ .reg .f32 t; mov.b64 {t, %0}, %1; }" : "=f"(a) : "l"(v)); return a; }
__device__ __forceinline__ f2 bc(float s) { return pk(s, s); }
__device__ __forceinline__ f2 fma2(f2 a, f2 b, f2 c) { f2 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ f2 add2(f2 a, f2 b) { f2 r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f2 sub2(f2 a, f2 b) { f2 r; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f2 mul2(f2 a, f2 b) { f2 r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f2 neg2(f2 a) { return pk(-lo(a), -hi(a)); }  // folds into the operand's negate modifier
__device__ __forceinline__ f2 sel2(bool p0, bool p1, f2 a, f2 b) { return pk(p0 ? lo(a) : lo(b), p1 ? hi(a) : hi(b)); }
__device__ __forceinline__ f2 min4_2(f2 a, f2 b, f2 c, f2 d) {  // fminf drops NaN, like a strict '<' against +inf
  return pk(fminf(fminf(lo(a), lo(b)), fminf(lo(c), lo(d))), fminf(fminf(hi(a), hi(b)), fminf(hi(c), hi(d))));
}

// parity tap (debug_corr handles only): the slot of the winner in the un-pruned table = first slot with identical coordinates
__device__ __noinline__ void gn_dbg_tap(const IterArgs &a, int row, int l, float qx, float qy, float qz, float ex, float ey, float ez, bool valid) {
  const float4 *full_row = a.cand + (size_t)row * a.K;
  const float wx_ = __fsub_rn(qx, ex), wy_ = __fsub_rn(qy, ey), wz_ = __fsub_rn(qz, ez);
  int slot = 0;
  float bd_ = INFINITY;
  for (int kk = 0; kk < a.K; kk++) {  // q - (q - c) is c up to one rounding: take the nearest table entry
    const float4 f = full_row[kk];
    const float dd_ = fabsf(f.x - wx_) + fabsf(f.y - wy_) + fabsf(f.z - wz_);
    if (dd_ < bd_) { bd_ = dd_; slot = kk; }
  }
  a.dbg_idx[(size_t)l * a.n_s + row] = a.cand_idx[(size_t)row * a.K + slot];
  a.dbg_mask[(size_t)l * a.n_s + row] = valid ? 1 : 0;
}

// long lists, one particle: the first slot of chunk [bk, bk+4) whose distance IS the minimum -- what slot-by-slot strict '<'
// would have kept.  Scalar, once per row; operation order as in SVN_DIST.
__device__ __forceinline__ void gn_recover(const float4 *e, int bk, float qx, float qy, float qz, float best, float &ex, float &ey, float &ez) {
  const float4 c0 = e[bk], c1 = e[bk + 1], c2 = e[bk + 2], c3 = e[bk + 3];
#define SVN_D1(C, T)                                                                                      \
  const float T##x = __fsub_rn(qx, (C).x), T##y = __fsub_rn(qy, (C).y), T##z = __fsub_rn(qz, (C).z);       \
  const float T##d = __fmaf_rn(T##z, T##z, __fmaf_rn(T##y, T##y, __fmul_rn(T##x, T##x)));
  SVN_D1(c0, u) SVN_D1(c1, v) SVN_D1(c2, w) SVN_D1(c3, z)
#undef SVN_D1
  (void)zd;
  const bool h0 = ud == best, h1 = vd == best, h2 = wd == best;
  ex = h0 ? ux : h1 ? vx : h2 ? wx : zx;
  ey = h0 ? uy : h1 ? vy : h2 ? wy : zy;
  ez = h0 ? uz : h1 ? vz : h2 ? wz : zz;
  if (best == INFINITY) { ex = ux; ey = uy; ez = uz; }  // nothing compared below +inf (NaN query): slot 0
}

// UNI: every lane of a warp works on the same source point (PG >= 32) -> the early exit is a warp vote.
// FIRST: first-order mode of the SVGD-ICP class (SVGDICP::sgd_grad, SVGDICP.cpp:398-455): sum 0 counts the unmasked
// pairs (nonzero_count, :404) and the second-moment sums 1..9 are not needed -- the gradient is E and C alone because
// every Euler partial is [omega_k]x R (see svgd_class.cu).
// Stage layout: [TB][Kp] float4 pruned lists, then [TB] float4 row headers (source point R0 s, w = list length bits: padded
// length << 16 | true length; 0 = padding row), then three 32-bit row masks written by the warp that loads the tile: rows whose padded list
// length is 2, 4, and more.  The consumers walk the three classes one after the other with a loop body specialised for the
// class (no data-dependent branch inside the two short-list bodies: control flow was 18 of 122 instructions per row).
// Thread -> particles: consumer thread pl of particle group y carries particles 2*(y*PG + pl) and the next one (neighbours in
// the pose-space ordering of the slice: their scan lengths are similar); .x of every pair is the even particle.
template <bool DBG, bool UNI, bool FIRST>
__global__ void __launch_bounds__(GN_THREADS, 1) k_gn(IterArgs a) {  // 16 warps x 128 registers
  if (a.ctrl->stop) return;
  extern __shared__ __align__(128) unsigned char smem[];
  const int TB = a.TB, Kp = a.Kp, S = a.stages;
  const size_t stage_bytes = gn_stage_bytes(TB, Kp);
  uint64_t *full = reinterpret_cast<uint64_t *>(smem + (size_t)S * stage_bytes);
  uint64_t *empty = full + S;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n_tiles = a.n_pad / TB;
  const int slice = blockIdx.x, n_slices = gridDim.x;
  const int n_my = (slice < n_tiles) ? (n_tiles - slice + n_slices - 1) / n_slices : 0;
  const size_t hdr_off = (size_t)TB * Kp * 16, msk_off = hdr_off + (size_t)TB * 16;

  if (tid == 0) {
    for (int s = 0; s < S; s++) { mbar_init(full + s, 1); mbar_init(empty + s, GN_CONSUMERS / 32); }
    fence_barrier_init();
  }
  __syncthreads();

  // ---------------- tile loads: 1-D TMA bulk copies of the pruned lists + the row-class masks ----------------
  // There is no producer warp (a 17th warp would round the CTA's register allocation up to 20 warps: 96 registers per
  // thread).  The warps take turns instead: at tile i, warp i % 16 refills the stage that tile i-LAG left with tile i+AHEAD
  // (AHEAD = S - LAG tiles in flight ahead of the slowest warp).  With S >= 4 the stage it refills was left TWO tiles ago, so
  // the wait for the slowest warp is normally over before it starts (with LAG = 1 it was 9 % of all stall samples; measured
  // 22.4 -> 21.6 ms per scan at configs[1]); the tile's list lengths were fetched one tile earlier.
  constexpr int NW = GN_CONSUMERS / 32;
  auto tile_cnt = [&](int j) -> int {  // padded list length of row `lane` of this CTA's j-th tile
    return (lane < TB) ? (__float_as_int(__ldg(&a.hdr[(size_t)(slice + j * n_slices) * TB + lane].w)) >> 16) : 0;
  };
  auto tile_issue = [&](int j, int cnt) {  // whole warp
    const int s = j % S;
    const int row0 = (slice + j * n_slices) * TB;
    unsigned char *st = smem + (size_t)s * stage_bytes;
    const unsigned m2 = __ballot_sync(0xffffffffu, cnt == 2), m4 = __ballot_sync(0xffffffffu, cnt == 4), ml = __ballot_sync(0xffffffffu, cnt > 4);
    const int bytes = cnt * 16;
    SVN_CHECK(a.ctrl, cnt >= 0 && cnt <= Kp && row0 + TB <= a.n_pad, 1);
    int total = bytes;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) total += __shfl_xor_sync(0xffffffffu, total, o);
    total += TB * 16;
    if (lane == 0) {
      unsigned *msk = reinterpret_cast<unsigned *>(st + msk_off);
      msk[0] = m2; msk[1] = m4; msk[2] = ml;
      mbar_expect_tx(full + s, (uint32_t)total);  // arrive = release: the masks are visible to whoever sees the phase complete
    }
    __syncwarp();
    if (lane < TB && cnt > 0) bulk_g2s(st + (size_t)lane * Kp * 16, a.clist + (size_t)(row0 + lane) * Kp, (uint32_t)bytes, full + s);
    if (lane == 0) bulk_g2s(st + hdr_off, a.hdr + row0, (uint32_t)(TB * 16), full + s);
  };
  const int LAG = (a.gn_lag < S) ? a.gn_lag : 1, AHEAD = S - LAG;
  for (int j = 0; j < AHEAD && j < n_my; j++)
    if (warp == j % NW) tile_issue(j, tile_cnt(j));
  int cnt_pref = (warp == 0 && AHEAD < n_my) ? tile_cnt(AHEAD) : 0;

  // ---------------- consumers: one thread = two particles (x RG row groups) ----------------
  const int PG = a.PG, RG = a.RG;  // PG = consumer threads (particle PAIRS) per row group
  const int pl = tid % PG, rg = tid / PG;
  const int l0 = 2 * (blockIdx.y * PG + pl), l1 = l0 + 1;  // local particle indices
  const bool active0 = l0 < a.P_l, active1 = l1 < a.P_l;
  f2 A0 = 0, A1 = 0, A2 = 0, A3 = 0, A4 = 0, A5 = 0, A6 = 0, A7 = 0, A8 = 0, t0 = 0, t1 = 0, t2 = 0;
  if (active0) {
    const float *xa = a.xf + (size_t)l0 * 12, *xb = a.xf + (size_t)(active1 ? l1 : l0) * 12;  // an odd tail pairs with itself
    A0 = pk(xa[0], xb[0]); A1 = pk(xa[1], xb[1]); A2 = pk(xa[2], xb[2]); A3 = pk(xa[3], xb[3]); A4 = pk(xa[4], xb[4]);
    A5 = pk(xa[5], xb[5]); A6 = pk(xa[6], xb[6]); A7 = pk(xa[7], xb[7]); A8 = pk(xa[8], xb[8]);
    t0 = pk(xa[9], xb[9]); t1 = pk(xa[10], xb[10]); t2 = pk(xa[11], xb[11]);
  }
  const float Dm = a.max_dist;
  f2 acc[NACC];  // first accumulation level, both particles
  f2 *dacc = reinterpret_cast<f2 *>(smem + gn_dacc_offset(TB, Kp, S)) + tid;  // second level: slot j at dacc[j * GN_CONSUMERS]
#pragma unroll
  for (int i = 0; i < NACC; i++) { acc[i] = 0; dacc[i * GN_CONSUMERS] = 0; }
  int rows_in_acc = 0, flushes2 = 0;
  bool wrote = false;
  const int RGe = RG < TB ? RG : TB;  // row groups that own rows (rg >= TB: none, they neither accumulate nor write partials)
  const bool active = active0 && rg < RGe;
  double *out = a.part + (((size_t)slice * RGe + (rg < RGe ? rg : 0)) * a.P_l + (active ? l0 : 0)) * NACC;  // particle l1: out + NACC
  SVN_CHECK(a.ctrl, PG * RG == GN_CONSUMERS && (int)gridDim.x == a.n_slices && gn_smem_bytes(TB, Kp, S) <= 227 * 1024, 4);
  // rows of a tile this thread owns: r = rg, rg + RG, ... (RG is a power of two dividing TB or larger than it)
  unsigned rgmask = 0;
  for (int r = rg; r < TB; r += RG) rgmask |= 1u << r;

// a = A' s' ; q = a + tau : query relative to q0_b.  Order fixed (index parity with oracle_corr_f32).
#define SVN_QUERY                                                                 \
  const f2 sx = bc(sv.x), sy = bc(sv.y), sz = bc(sv.z);                           \
  const f2 ax = fma2(A0, sx, fma2(A1, sy, mul2(A2, sz)));                         \
  const f2 ay = fma2(A3, sx, fma2(A4, sy, mul2(A5, sz)));                         \
  const f2 az = fma2(A6, sx, fma2(A7, sy, mul2(A8, sz)));                         \
  const f2 qx = add2(ax, t0), qy = add2(ay, t1), qz = add2(az, t2);
// residual and squared distance to one candidate: fixed operation order (index parity)
#define SVN_DIST(C, T)                                                                                    \
  const f2 T##x = sub2(qx, bc((C).x)), T##y = sub2(qy, bc((C).y)), T##z = sub2(qz, bc((C).z));            \
  const f2 T##d = fma2(T##z, T##z, fma2(T##y, T##y, mul2(T##x, T##x)));
// robust weight + the 16 Gauss-Newton sums for the matched pairs (residual ex, ey, ez, squared distance best: packed).
// LIVE = false turns the row into a no-op (the phantom second row of an odd-sized pair, see the two-candidate class).
#define SVN_ACCUM(LIVE)                                                                                                      \
  {                                                                                                                          \
    const float b0_ = lo(best), b1_ = hi(best);                                                                              \
    const bool v0_ = b0_ < Dm, v1_ = b1_ < Dm; /* SVGDICP.cpp:332: squared distance vs un-squared max_dist (Q1) */           \
    if (DBG) {                                                                                                               \
      const int row = (slice + i * n_slices) * TB + r;                                                                       \
      if (active && (LIVE)) gn_dbg_tap(a, row, l0, lo(qx), lo(qy), lo(qz), lo(ex), lo(ey), lo(ez), v0_);                      \
      if (active1 && (LIVE)) gn_dbg_tap(a, row, l1, hi(qx), hi(qy), hi(qz), hi(ex), hi(ey), hi(ez), v1_);                     \
    }                                                                                                                        \
    /* rho = (D / (D + 3 |e|))^2  (SVNICP.cpp:120-122); masked pairs: rho' = 0 and +1 on the translation block (Q2) */       \
    const f2 en = pk(sqrt_approx(b0_), sqrt_approx(b1_));                                                                    \
    const f2 den = fma2(bc(3.0f), en, bc(Dm));                                                                               \
    const f2 wq = mul2(bc(Dm), pk(rcp_approx(lo(den)), rcp_approx(hi(den))));                                                \
    const f2 rho = mul2(wq, wq);                                                                                             \
    const f2 rp = pk((v0_ && (LIVE)) ? lo(rho) : 0.0f, (v1_ && (LIVE)) ? hi(rho) : 0.0f);                                    \
    if (FIRST) {                                                                                                             \
      acc[0] = add2(acc[0], pk((v0_ && (LIVE)) ? 1.0f : 0.0f, (v1_ && (LIVE)) ? 1.0f : 0.0f));                               \
    } else {                                                                                                                 \
      acc[0] = add2(acc[0], pk((LIVE) ? (v0_ ? lo(rho) : 1.0f) : 0.0f, (LIVE) ? (v1_ ? hi(rho) : 1.0f) : 0.0f));             \
      const f2 gx = mul2(rp, sx), gy = mul2(rp, sy), gz = mul2(rp, sz);                                                      \
      acc[1] = add2(acc[1], gx); acc[2] = add2(acc[2], gy); acc[3] = add2(acc[3], gz);                                       \
      acc[4] = fma2(gx, sx, acc[4]); acc[5] = fma2(gx, sy, acc[5]); acc[6] = fma2(gx, sz, acc[6]);                           \
      acc[7] = fma2(gy, sy, acc[7]); acc[8] = fma2(gy, sz, acc[8]); acc[9] = fma2(gz, sz, acc[9]);                           \
    }                                                                                                                        \
    const f2 fx = mul2(rp, ex), fy = mul2(rp, ey), fz = mul2(rp, ez); /* multiplication (not select): NaN must propagate */  \
    acc[10] = add2(acc[10], fx); acc[11] = add2(acc[11], fy); acc[12] = add2(acc[12], fz);                                   \
    const f2 wx = add2(ax, sx), wy = add2(ay, sy), wz = add2(az, sz); /* R~ s in the world-oriented frame */                 \
    acc[13] = fma2(wy, fz, fma2(neg2(wz), fy, acc[13]));                                                                     \
    acc[14] = fma2(wz, fx, fma2(neg2(wx), fz, acc[14]));                                                                     \
    acc[15] = fma2(wx, fy, fma2(neg2(wy), fx, acc[15]));                                                                     \
  }

  for (int i = 0; i < n_my; i++) {
    const int s = i % S, k = i / S;
    {
      const int j = i + AHEAD;  // the tile that takes over the stage of tile i-LAG
      if (warp == i % NW && j < n_my) {
        if (j >= S) mbar_wait(empty + j % S, (uint32_t)((j / S - 1) & 1));  // every warp has left tile j-S = i-LAG
        tile_issue(j, cnt_pref);
      }
      if (warp == (i + 1) % NW && j + 1 < n_my) cnt_pref = tile_cnt(j + 1);
    }
    mbar_wait(full + s, (uint32_t)(k & 1));
    const unsigned char *st = smem + (size_t)s * stage_bytes;
    const float4 *hdr = reinterpret_cast<const float4 *>(st + hdr_off);
    const float4 *lists = reinterpret_cast<const float4 *>(st);
    if (UNI || active) {
      const unsigned *msk = reinterpret_cast<const unsigned *>(st + msk_off);
      unsigned m2 = msk[0] & rgmask, m4 = msk[1] & rgmask, ml = msk[2] & rgmask;
      rows_in_acc += __popc(m2 | m4 | ml);
      // ---- lists of one or two candidates (padded to 2: a one-candidate list carries a +inf sentinel that never wins).
      // Two rows per trip, written as one straight-line block so that the scheduler interleaves the two independent
      // chains; an odd last row gets a single-row body (pairing it with a dead copy of itself wasted a row's worth of
      // arithmetic: 5 % of this class at 16 rows per thread and tile, 40 % at 2 rows -- the sharded slices).
#define SVN_ROW2(SV, CA, CB)                                                                                            \
  {                                                                                                                     \
    const float4 sv = (SV);                                                                                             \
    SVN_QUERY                                                                                                           \
    SVN_DIST(CA, u) SVN_DIST(CB, v)                                                                                     \
    /* strict '<': the first slot wins ties (mink.cuh:141); NaN compares false -> slot 0 */                             \
    const bool p0 = lo(vd) < lo(ud), p1 = hi(vd) < hi(ud);                                                              \
    const f2 best = sel2(p0, p1, vd, ud), ex = sel2(p0, p1, vx, ux), ey = sel2(p0, p1, vy, uy), ez = sel2(p0, p1, vz, uz); \
    SVN_ACCUM(true)                                                                                                     \
  }
      while (m2 & (m2 - 1)) {  // at least two rows left
        const int r0 = __ffs(m2) - 1;
        m2 &= m2 - 1;
        const int r1 = __ffs(m2) - 1;
        m2 &= m2 - 1;
        const float4 sv0 = hdr[r0], sv1 = hdr[r1];
        const float4 *e0 = lists + r0 * Kp, *e1 = lists + r1 * Kp;
        const float4 c00 = e0[0], c01 = e0[1], c10 = e1[0], c11 = e1[1];
        { const int r = r0; (void)r; SVN_ROW2(sv0, c00, c01) }
        { const int r = r1; (void)r; SVN_ROW2(sv1, c10, c11) }
      }
      if (m2) {
        const int r = __ffs(m2) - 1;
        const float4 *e0 = lists + r * Kp;
        const float4 sv0 = hdr[r], c00 = e0[0], c01 = e0[1];
        SVN_ROW2(sv0, c00, c01)
      }
#undef SVN_ROW2
      // ---- three or four candidates (padded to 4)
      while (m4) {
        const int r = __ffs(m4) - 1;
        m4 &= m4 - 1;
        const float4 sv = hdr[r];
        const float4 *e = lists + r * Kp;
        const float4 c0 = e[0], c1 = e[1], c2 = e[2], c3 = e[3];
        SVN_QUERY
        SVN_DIST(c0, u) SVN_DIST(c1, v) SVN_DIST(c2, w) SVN_DIST(c3, z)
        // tournament with strict '<' at every node: among equal distances the lowest slot wins, as slot-by-slot '<' would decide
        const bool p10 = lo(vd) < lo(ud), p11 = hi(vd) < hi(ud), p30 = lo(zd) < lo(wd), p31 = hi(zd) < hi(wd);
        const f2 m01 = sel2(p10, p11, vd, ud), m23 = sel2(p30, p31, zd, wd);
        const f2 e01x = sel2(p10, p11, vx, ux), e01y = sel2(p10, p11, vy, uy), e01z = sel2(p10, p11, vz, uz);
        const f2 e23x = sel2(p30, p31, zx, wx), e23y = sel2(p30, p31, zy, wy), e23z = sel2(p30, p31, zz, wz);
        const bool p0 = lo(m23) < lo(m01), p1 = hi(m23) < hi(m01);
        const f2 best = sel2(p0, p1, m23, m01), ex = sel2(p0, p1, e23x, e01x), ey = sel2(p0, p1, e23y, e01y), ez = sel2(p0, p1, e23z, e01z);
        SVN_ACCUM(true)
      }
      // ---- longer lists: chunks of four, exact warp-voted early exit
      while (ml) {
        const int r = __ffs(ml) - 1;
        ml &= ml - 1;
        const float4 sv = hdr[r];
        const float4 *e = lists + r * Kp;
        const int n = __float_as_int(sv.w) >> 16;
        SVN_CHECK(a.ctrl, n > 4 && n <= Kp && (n & 3) == 0 && r < TB, 2);
        float4 c0 = e[0], c1 = e[1], c2 = e[2], c3 = e[3];
        SVN_QUERY
        float best0, best1;
        int bk0 = 0, bk1 = 0;  // first slot of the chunk that holds the running minimum (per particle)
        {
          SVN_DIST(c0, u) SVN_DIST(c1, v) SVN_DIST(c2, w) SVN_DIST(c3, z)
          const f2 m_ = min4_2(ud, vd, wd, zd);
          best0 = lo(m_); best1 = hi(m_);
          if (!(best0 == best0)) best0 = INFINITY;
          if (!(best1 == best1)) best1 = INFINITY;
        }
        // upper bound of |q| (distance of each particle's query from the initial-guess query q0_b)
        const f2 qq = fma2(qz, qz, fma2(qy, qy, mul2(qx, qx)));
        const f2 qn = fma2(pk(sqrt_approx(lo(qq)), sqrt_approx(hi(qq))), bc(1.00001f), bc(1e-7f));
        for (int k0 = 4; k0 < n; k0 += 4) {
          c0 = e[k0]; c1 = e[k0 + 1]; c2 = e[k0 + 2]; c3 = e[k0 + 3];
          // exact early exit: slots ascend in |c| (= c.w, a lower bound) and |q - c| >= |c| - |q|, so once
          // (|c| - |q|)^2 > best no later slot can win or tie.  NaN anywhere compares false -> no exit.  A particle whose
          // partner (or warp) is not done yet keeps scanning: later slots cannot change its minimum.
          const f2 tt = sub2(bc(c0.w), qn);
          const f2 tb = mul2(mul2(tt, tt), bc(0.99999f));
          const bool done = (lo(tt) > 0.f) && (lo(tb) > best0) && (hi(tt) > 0.f) && (hi(tb) > best1);
          if (UNI) { if (__all_sync(0xffffffffu, done)) break; }
          else { if (done) break; }
          // only the chunk minimum enters the running comparison; the slot inside the winning chunk is recovered afterwards
          SVN_DIST(c0, u) SVN_DIST(c1, v) SVN_DIST(c2, w) SVN_DIST(c3, z)
          const f2 m_ = min4_2(ud, vd, wd, zd);
          if (lo(m_) < best0) { best0 = lo(m_); bk0 = k0; }
          if (hi(m_) < best1) { best1 = hi(m_); bk1 = k0; }
        }
        SVN_CHECK(a.ctrl, bk0 >= 0 && bk0 + 3 < n && bk1 >= 0 && bk1 + 3 < n, 3);
        float ex0, ey0, ez0, ex1, ey1, ez1;
        gn_recover(e, bk0, lo(qx), lo(qy), lo(qz), best0, ex0, ey0, ez0);
        gn_recover(e, bk1, hi(qx), hi(qy), hi(qz), best1, ex1, ey1, ez1);
        const f2 best = pk(best0, best1), ex = pk(ex0, ex1), ey = pk(ey0, ey1), ez = pk(ez0, ez1);
        SVN_ACCUM(true)
      }
      if (rows_in_acc >= GN_FLUSH_ROWS) {
#pragma unroll
        for (int j = 0; j < NACC; j++) { dacc[j * GN_CONSUMERS] = add2(dacc[j * GN_CONSUMERS], acc[j]); acc[j] = 0; }
        rows_in_acc = 0;
        if (++flushes2 >= GN_FLUSH2 && active) {
          // third level: fold into the two particles' own fp64 partial slots (global, L2-resident) so that the fp32
          // second level never carries more than GN_FLUSH2 * GN_FLUSH_ROWS rows, whatever the slice length
#pragma unroll
          for (int j = 0; j < NACC; j++) {
            const f2 d = dacc[j * GN_CONSUMERS];
            out[j] = (wrote ? out[j] : 0.0) + (double)lo(d);
            if (active1) out[NACC + j] = (wrote ? out[NACC + j] : 0.0) + (double)hi(d);
            dacc[j * GN_CONSUMERS] = 0;
          }
          wrote = true;
          flushes2 = 0;
        }
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(empty + s);
  }
#undef SVN_QUERY
#undef SVN_DIST
#undef SVN_ACCUM
  if (active) {
#pragma unroll
    for (int j = 0; j < NACC; j++) {
      const f2 d = dacc[j * GN_CONSUMERS];
      out[j] = (wrote ? out[j] : 0.0) + ((double)lo(d) + (double)lo(acc[j]));
      if (active1) out[NACC + j] = (wrote ? out[NACC + j] : 0.0) + ((double)hi(d) + (double)hi(acc[j]));
    }
  }
}

// ---------------------------------------------------------------------------------------------
// k_finalize: partials -> reference H (upper triangle) and b; one CTA per particle.  The record fields it produces (b, H, g)
// go into the record buffer of this iteration's parity on EVERY rank (peer stores over NVLink when sharded); the CTA that
// finishes last publishes the sequence number in the peers' flag blocks (k_tail waits for it).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(FIN_WARPS * 32) k_finalize(IterArgs a, PeerTable pt, unsigned seq_h) {
  Ctrl *ctl = a.ctrl;
  if (ctl->stop) return;
  __shared__ double s_out[REC];
  __shared__ int s_last;
  const int l = blockIdx.x;  // one CTA (FIN_WARPS warps) per local particle
  double v[NACC];
  gn_sum_partials(a, l, v);
  const int p = a.p_lo + l;
  SVN_CHECK(ctl, l < a.P_l && p < a.P && (size_t)(p + 1) * REC <= a.rec_stride, 20);
  const size_t buf_off = (size_t)(ctl->iter & 1) * a.rec_stride;
  if (threadIdx.x == 0) {
    double Rp[9], H[36], b[6];
#pragma unroll
    for (int i = 0; i < 9; i++) Rp[i] = a.R[9 * (size_t)p + i];
    gn_assemble(a.sc.R0, Rp, v, H, b);
#pragma unroll
    for (int i = 0; i < 6; i++) s_out[REC_B + i] = b[i];
#pragma unroll
    for (int r = 0; r < 6; r++)
#pragma unroll
      for (int c = r; c < 6; c++) s_out[REC_H + tri(r, c)] = H[6 * r + c];
    double g[6];
#pragma unroll
    for (int i = 0; i < 6; i++) g[i] = 0.0;
    if (!a.svn_full_grad) {  // g = H^-1 b, SVNICP.cpp:162 (only consumed by the pre-conditioned SVGD step)
#pragma unroll
      for (int i = 0; i < 6; i++) g[i] = b[i];
      ldl_solve6_reg(H, g);  // SPD (+ 1e-6 I), register resident (the record fields were taken from H above)
    }
#pragma unroll
    for (int i = 0; i < 6; i++) s_out[REC_G + i] = g[i];
  }
  __syncthreads();
  // fields [REC_B, REC_DNORM) and [REC_G, REC_G + 6) of the particle's record on every rank; x and |delta| belong to k_tail
  for (int u = threadIdx.x; u < pt.n_ranks * 33; u += blockDim.x) {
    const int r = u / 33, f = u % 33;
    const int field = f < 27 ? REC_B + f : REC_G + (f - 27);
    pt.rec[r][buf_off + (size_t)p * REC + field] = s_out[field];
  }
  if (pt.n_ranks <= 1) return;
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) s_last = (atomicAdd(&ctl->fin_ticket, 1u) == gridDim.x - 1) ? 1 : 0;
  __syncthreads();
  if (!s_last) return;
  if ((int)threadIdx.x < pt.n_ranks && (int)threadIdx.x != pt.rank) {
    __threadfence_system();
    st_release_sys(pt.flag[threadIdx.x] + FLAG_H * MAX_RANKS + pt.rank, seq_h);
  }
  if (threadIdx.x == 0) ctl->fin_ticket = 0u;
}

// ---------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------
static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

void init_iter_kernels() {
// dynamic shared memory up to 200 KB, and the SM configured for the maximum shared-memory carve-out while k_gn runs: its two
// CTAs take ~156 KB, and the small side-stream kernels (k_head_*, 33 KB each) must find room NEXT to them instead of waiting for
// a k_gn CTA to retire (with the default carve-out the head chain finished ~26 us after k_gn, on the critical path)
#define SVN_GN_ATTR(D, U, F)                                                                                  \
  do {                                                                                                        \
    cudaFuncSetAttribute(k_gn<D, U, F>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);             \
    cudaFuncSetAttribute(k_gn<D, U, F>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared); \
  } while (0)
  SVN_GN_ATTR(false, true, false); SVN_GN_ATTR(true, true, false); SVN_GN_ATTR(false, false, false); SVN_GN_ATTR(true, false, false);
  SVN_GN_ATTR(false, true, true); SVN_GN_ATTR(true, true, true); SVN_GN_ATTR(false, false, true); SVN_GN_ATTR(true, false, true);
#undef SVN_GN_ATTR
}

int launch_prep(const IterArgs &a, cudaStream_t st, int all_x, const double *x_src) {
  k_prep<<<1, 1024, 0, st>>>(a, all_x, x_src);
  return 1;
}

int launch_filter(const IterArgs &a, cudaStream_t st) {
  const int nch = (a.K + 31) / 32;
  int grid = cdiv((long long)a.n_s * 32, 256);
  const int max_grid = a.sm_count * 8;
  if (grid > max_grid) grid = max_grid;
  if (grid < 1) grid = 1;
  int launches = 1;
  if (a.clist_prev) {  // iterations >= 1: both pruning kernels are enqueued, filter_use_reuse() lets exactly one of them work
    int g = cdiv(a.n_s, 32 * 8);  // a warp takes 32 consecutive rows per trip
    const int resident = a.sm_count * 4;  // __launch_bounds__(256, 4): one wave, grid-stride over the rows
    if (g > resident) g = resident;
    k_filter_reuse<<<g < 1 ? 1 : g, 256, 0, st>>>(a);
    launches = 2;
  }
  switch (nch) {
    case 1: k_filter<1><<<grid, 256, 0, st>>>(a); break;
    case 2: k_filter<2><<<grid, 256, 0, st>>>(a); break;
    case 3: k_filter<3><<<grid, 256, 0, st>>>(a); break;
    case 4: k_filter<4><<<grid, 256, 0, st>>>(a); break;
    case 5: k_filter<5><<<grid, 256, 0, st>>>(a); break;
    case 6: k_filter<6><<<grid, 256, 0, st>>>(a); break;
    case 7: k_filter<7><<<grid, 256, 0, st>>>(a); break;
    default: k_filter<8><<<grid, 256, 0, st>>>(a); break;
  }
  return launches;
}

int launch_gn(const IterArgs &a, cudaStream_t st) {
  dim3 grid(a.n_slices, a.n_pgroups);
  const bool uni = a.PG >= 32;
#define SVN_GN_GO(D, U, F) k_gn<D, U, F><<<grid, GN_THREADS, a.gn_smem, st>>>(a)
  if (a.first_order) {
    if (a.dbg_idx) { if (uni) SVN_GN_GO(true, true, true); else SVN_GN_GO(true, false, true); }
    else { if (uni) SVN_GN_GO(false, true, true); else SVN_GN_GO(false, false, true); }
  } else {
    if (a.dbg_idx) { if (uni) SVN_GN_GO(true, true, false); else SVN_GN_GO(true, false, false); }
    else { if (uni) SVN_GN_GO(false, true, false); else SVN_GN_GO(false, false, false); }
  }
#undef SVN_GN_GO
  return 1;
}

int launch_finalize(const IterArgs &a, const PeerTable &pt, unsigned seq_h, cudaStream_t st) {
  if (a.P_l > 0) k_finalize<<<a.P_l, fin_threads(a), 0, st>>>(a, pt, seq_h);
  return 1;
}

}  // namespace svn
