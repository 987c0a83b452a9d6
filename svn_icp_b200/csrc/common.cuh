// common.cuh -- shared device-side declarations of the B200 SVN-ICP inner loop.
//
// Data layout in HBM (one handle = one GPU = one particle slice; see DESIGN.md):
//   src64  [N_s][3] f64   clone of the source cloud           (SVGDICP.cpp:56)
//   tgt64  [N_t][3] f64   clone of the target cloud           (SVGDICP.cpp:55)
//   sp     [N_s]   float4 (R0*s).xyz, w = |R0*s| rounded up   per scan
//   cand   [N_s][K] float4 candidate m - q0 (fp32), w = global map index bits; ascending (d0^2, index)
//   clist  [N_s][K] float4 per-iteration exactly pruned candidate lists, ccount [N_s]
//   R,t    [P][9],[P][3] f64 particle state (only the local slice is authoritative)
//   xf     [P_l][12] f32  per-iteration particle transforms A' = R0 (R_p - I) R0^T, tau = R0 t_p
//   part   [slices*RG][P_l][16] f64 Gauss-Newton partial sums
//   rec    [P_pad][REC] f64 packed per-particle record (the all-gather payload)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

namespace svn {

// packed per-particle record, REC doubles.  41, not 40: tiles of records are staged AoS in shared memory by 1-D bulk TMA and
// read with lane = particle; an odd stride in doubles makes those reads bank-conflict free (40 would be a 16-way conflict)
constexpr int REC = 41;
constexpr int REC_TILE_PAD = 256;  // the record buffers hold a multiple of this many records, zero filled: every tile copy is full size
constexpr int REC_X = 0;       // [0,6)   x = [t ; Log R] at the head of the iteration
constexpr int REC_B = 6;       // [6,12)  b = sum J^T rho e
constexpr int REC_H = 12;      // [12,33) H upper triangle, row-major
constexpr int REC_DNORM = 33;  // |delta| of the previous iteration (early stop, SVNICP.cpp:95-101)
constexpr int REC_G = 34;      // [34,40) g = H^-1 b (pre-conditioned SVGD mode only, SVNICP.cpp:162)

constexpr int NACC = 16;  // W, S1(3), S2(6: xx xy xz yy yz zz), E(3), C(3)

constexpr int MED_PASSES = 5;  // 11 + 13 + 13 + 13 + 13 = 63 key bits
constexpr int MED_BINS = 8192;

constexpr int PRUNE_BINS = 64;        // range bins of the pruning-radius envelope
constexpr double PRUNE_BIN_W = 2.0;   // metres per bin (points beyond PRUNE_BINS*PRUNE_BIN_W use alpha*|s|+beta)

struct Ctrl {
  int stop;         // 1 once the early stop fired (all later kernels return immediately)
  int iter;         // iterations whose pose update has been applied
  int iters_done;   // == iter at the moment of the stop
  int error;        // 1: a wait on a peer's flag timed out (sharded handles); >= 100: a device-side bounds check of the
                    // -DSVN_DEBUG_BOUNDS build failed (code = 100 + check id); the host reports it after the scan
  unsigned fin_ticket, tail_ticket;  // CTAs of k_finalize / k_tail that have finished (the last one publishes)
  unsigned pad1, pad2;
  double bandwidth;  // h of the last Stein step
  // exact-pruning ball of the local particle slice (k_prep): |q_pb - qbar_b| <= alpha*|s'_b| + beta
  float Abar[9];
  float taubar[3];
  float alpha;
  float beta;
  float env[PRUNE_BINS];  // env[i] >= max_p (sigma_p r + beta_p) for every r <= (i+1)*PRUNE_BIN_W
  // median radix select (lower median of P^2 pairwise squared distances, SVNICP.cpp:262)
  unsigned long long sel_prefix[MED_PASSES + 1];
  unsigned long long sel_rank[MED_PASSES + 1];
  unsigned med_ticket[MED_PASSES];  // CTAs that finished pass s (the last one selects)
  unsigned long long kept_total;  // sum of ccount over rows (prune statistics)
  // k_head_* (tail2.cu): fast median path around the previous iteration's median
  unsigned fast_ticket[2];
  int med_done;                   // 1: the bandwidth of this iteration is final (the radix passes return at once)
  int pad3;
  unsigned long long fast_bin, fast_rank;  // bin of the linear histogram that holds the median (0 / MED_BINS-1: miss) and the rank inside it
};

// ---- peer-memory exchange of the per-particle records between the GPUs of one box (sharded handles) -----------------
// Every rank owns a block [2][rec_stride] doubles (records, double buffered by iteration parity) + a flag block, mapped
// into every other rank through CUDA IPC.  The owner of a particle stores its record fields straight into every rank's
// buffer over NVLink and then publishes a sequence number in that rank's flag block; consumers spin on their LOCAL flags.
constexpr int MAX_RANKS = 8;
constexpr int FLAG_H = 0;  // "b, H (g) of iteration seq are in your buffer"   (k_finalize -> k_tail)
constexpr int FLAG_X = 1;  // "x, |delta| after update seq are in your buffer" (k_tail -> k_head)
// Device-side bounds checks of the debug build (build.py --debug-bounds -> libsvnicp_b200_dbg.so; compute-sanitizer is not
// available on the target pool).  A failed check records 100 + id in ctrl->error (first failure wins) and the access is skipped
// or clamped by the caller; svnicp_align then fails with the id in its message.  The release build compiles them away.
#ifdef SVN_DEBUG_BOUNDS
#define SVN_CHECK(ctrl, cond, id) do { if (!(cond)) atomicCAS(&(ctrl)->error, 0, 100 + (id)); } while (0)
#else
#define SVN_CHECK(ctrl, cond, id) do { } while (0)
#endif

struct PeerTable {
  int n_ranks, rank;
  double *rec[MAX_RANKS];     // record block of rank r as mapped HERE (rec[rank] = the local block)
  unsigned *flag[MAX_RANKS];  // flag block of rank r: [kind * MAX_RANKS + source rank]
  unsigned long long timeout_ns;
};

struct ScanConst {  // per-scan constants, passed by value
  double R0[9];
  double t0[3];
};

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ---- 6x6 dense helpers in fp64 (Stein step, finalize) ------------------------------------------
// Compile-time loop: every index below is a constant, so the 6x6 operands stay in registers (nvcc leaves `#pragma unroll`
// loops of this depth rolled and puts the matrix on the stack, hence the template recursion).
template <int I, int N, class F>
__device__ __forceinline__ void static_for(F &&f) {
  if constexpr (I < N) { f(std::integral_constant<int, I>{}); static_for<I + 1, N>(f); }
}

// Symmetric positive definite 6x6 solve A x = b by LDL^T, every index a compile-time constant (registers only), one reciprocal
// per column and no pivot search.  The matrices solved on the hot path are SPD by construction -- the Gauss-Newton Hessian
// carries + 1e-6 I (SVNICP.cpp:153) and the Stein Hessian is a kernel-weighted sum of those plus outer products -- so this is
// the same solution as the reference's LU-based linalg::solve / inv up to rounding (cond * 1e-16), at a quarter of the
// dependent instruction chain of a pivoted LU (which cost 12 us per particle in k_tail).  NaN / Inf inputs propagate.
// Only the upper triangle of A (row-major 6x6) is read; A is overwritten.
__device__ __forceinline__ void ldl_solve6_reg(double (&A)[36], double (&b)[6]) {
  double L[36];   // strict lower triangle, L[i*6+k], k < i
  double iD[6];   // 1 / d_j
  static_for<0, 6>([&](auto J) {
    constexpr int j = decltype(J)::value;
    double w[6];  // w_k = L_jk d_k, k < j
    double d = A[j * 6 + j];
    static_for<0, j>([&](auto K) {
      constexpr int k = decltype(K)::value;
      w[k] = L[j * 6 + k] * A[k * 6 + k];  // A's diagonal holds d_k once column k is done
      d -= L[j * 6 + k] * w[k];
    });
    A[j * 6 + j] = d;
    iD[j] = 1.0 / d;
    static_for<j + 1, 6>([&](auto I_) {
      constexpr int i = decltype(I_)::value;
      double sum = A[j * 6 + i];  // upper triangle: A_ji = A_ij
      static_for<0, j>([&](auto K) { constexpr int k = decltype(K)::value; sum -= L[i * 6 + k] * w[k]; });
      L[i * 6 + j] = sum * iD[j];
    });
  });
  static_for<1, 6>([&](auto I_) {  // L y = b
    constexpr int i = decltype(I_)::value;
    static_for<0, i>([&](auto K) { constexpr int k = decltype(K)::value; b[i] -= L[i * 6 + k] * b[k]; });
  });
  static_for<0, 6>([&](auto I_) { constexpr int i = decltype(I_)::value; b[i] *= iD[i]; });  // D z = y
  static_for<0, 5>([&](auto II) {  // L^T x = z
    constexpr int i = 4 - decltype(II)::value;
    static_for<i + 1, 6>([&](auto K) { constexpr int k = decltype(K)::value; b[i] -= L[k * 6 + i] * b[k]; });
  });
}

// upper-triangle index of (r,c), r <= c, row-major packing of a symmetric 6x6
__host__ __device__ __forceinline__ int tri(int r, int c) { return r * 6 - (r * (r - 1)) / 2 + (c - r); }

// SO(3) Exp and left Jacobian exactly as SVNICP::to_rotation_tensor (SVNICP.cpp:166-194),
// NaN at angle == 0 for J_l included (quirk Q7).
__device__ inline void so3_exp(const double r[3], double R[9], double *Jl) {
  const double a = sqrt(r[0] * r[0] + r[1] * r[1] + r[2] * r[2]);
  double n[3];
  const double ia = 1.0 / a;  // one division (inf at a == 0: sa, ca below become NaN exactly as s / a, (1 - c) / a do -- quirk Q7)
  if (a < 1e-12) { n[0] = n[1] = n[2] = 0.0; }
  else { n[0] = r[0] * ia; n[1] = r[1] * ia; n[2] = r[2] * ia; }
  double s, c;
  sincos(a, &s, &c);
  const double ah[9] = {0, -n[2], n[1], n[2], 0, -n[0], -n[1], n[0], 0};
  const double sa = s * ia, ca = (1.0 - c) * ia;
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int j = 0; j < 3; j++) {
      const double id = (i == j) ? 1.0 : 0.0, nn = n[i] * n[j];
      R[3 * i + j] = c * id + (1.0 - c) * nn + s * ah[3 * i + j];
      if (Jl) Jl[3 * i + j] = sa * id + (1.0 - sa) * nn + ca * ah[3 * i + j];
    }
}

// SO(3) Log exactly as SVNICP::rotm_to_ypr_tensor (SVNICP.cpp:196-215).
__device__ inline void so3_log(const double R[9], double w[3]) {
  double v = 0.5 * (R[0] + R[4] + R[8] - 1.0);
  v = fmin(fmax(v, -1.0), 1.0);
  const double a = acos(v), s = sin(a);
  if (fabs(s) > 1e-12) {
    const double f = 0.5 / s * a;
    w[0] = f * (R[7] - R[5]);
    w[1] = f * (R[2] - R[6]);
    w[2] = f * (R[3] - R[1]);
  } else {
    w[0] = w[1] = w[2] = 0.0;
  }
}

// largest eigenvalue of M^T M (M 3x3 row-major) = sigma_max(M)^2, rounded up; NaN propagates
__device__ inline double sym3_max_eig_MtM(const double M[9]) {
  double B[6];  // 00 01 02 11 12 22
  B[0] = M[0] * M[0] + M[3] * M[3] + M[6] * M[6];
  B[1] = M[0] * M[1] + M[3] * M[4] + M[6] * M[7];
  B[2] = M[0] * M[2] + M[3] * M[5] + M[6] * M[8];
  B[3] = M[1] * M[1] + M[4] * M[4] + M[7] * M[7];
  B[4] = M[1] * M[2] + M[4] * M[5] + M[7] * M[8];
  B[5] = M[2] * M[2] + M[5] * M[5] + M[8] * M[8];
  const double tr = B[0] + B[3] + B[5];
  const double q = tr / 3.0;
  const double p1 = B[1] * B[1] + B[2] * B[2] + B[4] * B[4];
  const double p2 = (B[0] - q) * (B[0] - q) + (B[3] - q) * (B[3] - q) + (B[5] - q) * (B[5] - q) + 2.0 * p1;
  const double p = sqrt(p2 / 6.0);
  if (!(p > 1e-300)) return (tr != tr) ? tr : q * (1.0 + 1e-9);
  const double ip = 1.0 / p;  // one division (the result carries a 1e-9 relative safety margin; a reciprocal multiply costs 1e-16)
  const double c00 = (B[0] - q) * ip, c11 = (B[3] - q) * ip, c22 = (B[5] - q) * ip, c01 = B[1] * ip, c02 = B[2] * ip, c12 = B[4] * ip;
  double r = 0.5 * (c00 * (c11 * c22 - c12 * c12) - c01 * (c01 * c22 - c12 * c02) + c02 * (c01 * c12 - c11 * c02));
  r = fmin(fmax(r, -1.0), 1.0);
  const double lam = q + 2.0 * p * cos(acos(r) / 3.0);
  // never above the Frobenius bound (= trace), never optimistic: 1e-9 relative + absolute guard for rounding
  return fmin(tr, lam * (1.0 + 1e-9) + 1e-30) * (tr == tr ? 1.0 : NAN);
}

}  // namespace svn
