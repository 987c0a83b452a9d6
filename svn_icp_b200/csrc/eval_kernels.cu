// eval_kernels.cu -- svnicp_evaluate: the registration objective of the last scan at caller-given poses.
//
// Per pose x (the handle's particle convention) and per source point b, against the candidate table of the last stein_align:
//   1-NN among the K candidates of b (the fp32 arithmetic and tie-break of k_gn / oracle_corr_f32: first strictly smaller
//   squared distance in slot order), inlier mask d^2 < max_dist (Q1), and over all points the inlier count, the sum of
//   inlier d^2 and the 16 Gauss-Newton sums of k_gn -> H, b of Newton_grad_right (SVNICP.cpp:116-164, Q1-Q3).
//
//   k_eval_prep   pose -> R, t (so3_exp as k_particles_init, or euler_R as k_svgd_init) -> fp32 A', tau (rel_transform_f32)
//   k_eval_corr   one warp per source row, streaming the K-slot table once per block of <= 32 poses.  With G lane groups
//                 (G = poses of the block rounded up to a power of two) 32 / G lanes share a pose's K slots.  G == 1: every
//                 lane scans its own slots straight from registers; G > 1: the row is staged in shared memory and the lanes
//                 of a group scan slots sub, sub + 32/G, ...  The lanes of a group combine their minima by (distance, slot).
//                 Sums: fp32 over EV_FLUSH rows, then fp64 per (warp, pose) in shared memory, then fixed-order per CTA.
//   k_eval_fin    fixed-order fp64 sum of the per-CTA partials, then H, b (gn_assemble, shared with k_finalize) and stats.
// Nothing of the scan's own state (particles, records, transforms, pruned lists, ctrl, history) is read or written
// except the inputs of the table (sp, cand, cand_idx).
#include "common.cuh"
#include "kernels.h"

namespace svn {

constexpr int EV_WARPS = 4;
constexpr int EV_FLUSH = 32;  // rows per fp32 accumulation level (as GN_FLUSH_ROWS of k_gn)
// CTAs per SM that k_eval_corr is compiled for: 5 (96 registers) up to K = 128; longer rows need 128 registers to stay spill free
__host__ __device__ constexpr int ev_min_blocks(int nch) { return nch <= 4 ? 5 : 4; }

__global__ void k_eval_prep(const double *poses, int M, int euler, ScanConst sc, float *xf, double *R) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M) return;
  double x[6], Rm[9];
#pragma unroll
  for (int c = 0; c < 6; c++) x[c] = poses[(size_t)c * M + m];
  if (euler) euler_R(x, Rm);
  else so3_exp(x + 3, Rm, nullptr);
  float f[12];
  rel_transform_f32(sc.R0, Rm, x, f);
#pragma unroll
  for (int i = 0; i < 12; i++) xf[(size_t)m * 12 + i] = f[i];
#pragma unroll
  for (int i = 0; i < 9; i++) R[(size_t)m * 9 + i] = Rm[i];
}

__device__ __forceinline__ float ev_sqrt_approx(float x) {
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float ev_rcp_approx(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// dynamic shared memory: [EV_WARPS][G][EV_NS] fp64 sums, then (G > 1) [EV_WARPS][K] float4 staged rows
template <int NCH, bool SYS>
__global__ void __launch_bounds__(EV_WARPS * 32, ev_min_blocks(NCH)) k_eval_corr(EvalArgs a) {
  extern __shared__ __align__(16) unsigned char ev_smem[];
  const int G = a.G, L = 32 / G, MB = a.MB, K = a.K;
  double *s_acc = reinterpret_cast<double *>(ev_smem);
  float4 *s_row = reinterpret_cast<float4 *>(ev_smem + (size_t)EV_WARPS * G * EV_NS * sizeof(double));
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane / L, sub = lane % L;
  const bool live = g < MB;
  for (int i = tid; i < EV_WARPS * G * EV_NS; i += blockDim.x) s_acc[i] = 0.0;
  __syncthreads();
  float A[12];
  {
    const float *x = a.xf + (size_t)(live ? g : 0) * 12;
#pragma unroll
    for (int i = 0; i < 12; i++) A[i] = x[i];
  }
  const float Dm = a.max_dist;
  float acc[EV_NS];
#pragma unroll
  for (int j = 0; j < EV_NS; j++) acc[j] = 0.f;
  double *my_acc = s_acc + ((size_t)warp * G + g) * EV_NS;
  float4 *row_buf = s_row + (size_t)warp * K;
  int rows = 0;
  const int gw = blockIdx.x * EV_WARPS + warp, nw = gridDim.x * EV_WARPS;
  for (int b = gw; b < a.n_s; b += nw) {
    const float4 *row = a.cand + (size_t)b * K;
    float4 e[NCH];
#pragma unroll
    for (int ch = 0; ch < NCH; ch++) {
      const int k = ch * 32 + lane;
      e[ch] = (k < K) ? __ldcs(row + k) : make_float4(0.f, 0.f, 0.f, 0.f);  // streamed: the table exceeds L2 at full size
    }
    const float4 sv = a.sp[b];
    // query relative to q0: a = A' s', q = a + tau; operation order of k_gn's SVN_QUERY (index parity with oracle_corr_f32)
    const float ax = __fmaf_rn(A[0], sv.x, __fmaf_rn(A[1], sv.y, __fmul_rn(A[2], sv.z)));
    const float ay = __fmaf_rn(A[3], sv.x, __fmaf_rn(A[4], sv.y, __fmul_rn(A[5], sv.z)));
    const float az = __fmaf_rn(A[6], sv.x, __fmaf_rn(A[7], sv.y, __fmul_rn(A[8], sv.z)));
    const float qx = __fadd_rn(ax, A[9]), qy = __fadd_rn(ay, A[10]), qz = __fadd_rn(az, A[11]);
    // this lane's first strictly smaller distance in ascending slot order (NaN never wins; slot K = none)
    float best = INFINITY, ex = 0.f, ey = 0.f, ez = 0.f;
    int slot = K;
#define EV_CAND(C, KK)                                                                                        \
  {                                                                                                           \
    const float dx = __fsub_rn(qx, (C).x), dy = __fsub_rn(qy, (C).y), dz = __fsub_rn(qz, (C).z);             \
    const float d = __fmaf_rn(dz, dz, __fmaf_rn(dy, dy, __fmul_rn(dx, dx)));                                  \
    if (d < best) { best = d; slot = (KK); ex = dx; ey = dy; ez = dz; }                                      \
  }
    if (G == 1) {
#pragma unroll
      for (int ch = 0; ch < NCH; ch++) {
        const int k = ch * 32 + lane;
        if (k < K) EV_CAND(e[ch], k)
      }
    } else {
      __syncwarp();  // the previous row's readers are done with the buffer
#pragma unroll
      for (int ch = 0; ch < NCH; ch++) {
        const int k = ch * 32 + lane;
        if (k < K) row_buf[k] = e[ch];
      }
      __syncwarp();
      for (int k = sub; k < K; k += L) EV_CAND(row_buf[k], k)
    }
#undef EV_CAND
    // the group's minimum by (distance, slot): the first strictly smaller distance in slot order over all K slots
    for (int o = L >> 1; o > 0; o >>= 1) {
      const float ob = __shfl_xor_sync(0xffffffffu, best, o);
      const int os = __shfl_xor_sync(0xffffffffu, slot, o);
      const float ox = __shfl_xor_sync(0xffffffffu, ex, o), oy = __shfl_xor_sync(0xffffffffu, ey, o), oz = __shfl_xor_sync(0xffffffffu, ez, o);
      if (ob < best || (ob == best && os < slot)) { best = ob; slot = os; ex = ox; ey = oy; ez = oz; }
    }
    if (slot == K) {  // nothing below +inf (NaN or infinite query): slot 0, as the strict '<' scan from +inf decides
      const float4 c0 = a.cand[(size_t)b * K];
      slot = 0;
      ex = __fsub_rn(qx, c0.x); ey = __fsub_rn(qy, c0.y); ez = __fsub_rn(qz, c0.z);
    }
    const bool v = best < Dm;  // SVGDICP.cpp:332: squared distance vs un-squared max_dist (Q1)
    if (live && sub == 0) {
      if (a.mask) a.mask[(size_t)g * a.n_s + b] = v ? 1 : 0;
      if (a.idx) a.idx[(size_t)g * a.n_s + b] = a.cand_idx[(size_t)b * K + slot];
    }
    acc[16] += v ? 1.0f : 0.0f;
    acc[17] += v ? best : 0.0f;
    if (SYS) {  // SVN_ACCUM of k_gn (second-order mode), one pose
      const float en = ev_sqrt_approx(best);
      const float wq = Dm * ev_rcp_approx(__fmaf_rn(3.0f, en, Dm));
      const float rho = wq * wq;  // (D / (D + 3 |e|))^2, SVNICP.cpp:120-122
      const float rp = v ? rho : 0.0f;
      acc[0] += v ? rho : 1.0f;  // masked pairs: +1 on the translation block (Q2)
      const float gx = rp * sv.x, gy = rp * sv.y, gz = rp * sv.z;
      acc[1] += gx; acc[2] += gy; acc[3] += gz;
      acc[4] = __fmaf_rn(gx, sv.x, acc[4]); acc[5] = __fmaf_rn(gx, sv.y, acc[5]); acc[6] = __fmaf_rn(gx, sv.z, acc[6]);
      acc[7] = __fmaf_rn(gy, sv.y, acc[7]); acc[8] = __fmaf_rn(gy, sv.z, acc[8]); acc[9] = __fmaf_rn(gz, sv.z, acc[9]);
      const float fx = rp * ex, fy = rp * ey, fz = rp * ez;  // multiplication (not select): NaN must propagate
      acc[10] += fx; acc[11] += fy; acc[12] += fz;
      const float wx = ax + sv.x, wy = ay + sv.y, wz = az + sv.z;  // R~ s in the world-oriented frame
      acc[13] = __fmaf_rn(wy, fz, __fmaf_rn(-wz, fy, acc[13]));
      acc[14] = __fmaf_rn(wz, fx, __fmaf_rn(-wx, fz, acc[14]));
      acc[15] = __fmaf_rn(wx, fy, __fmaf_rn(-wy, fx, acc[15]));
    }
    if (++rows == EV_FLUSH) {
      if (live && sub == 0)
#pragma unroll
        for (int j = 0; j < EV_NS; j++) my_acc[j] += (double)acc[j];
#pragma unroll
      for (int j = 0; j < EV_NS; j++) acc[j] = 0.f;
      rows = 0;
    }
  }
  if (live && sub == 0)
#pragma unroll
    for (int j = 0; j < EV_NS; j++) my_acc[j] += (double)acc[j];
  __syncthreads();
  // per-CTA partial: warps in ascending order
  for (int i = tid; i < MB * EV_NS; i += blockDim.x) {
    const int m = i / EV_NS, j = i % EV_NS;
    double s = 0.0;
    for (int w = 0; w < EV_WARPS; w++) s += s_acc[((size_t)w * G + m) * EV_NS + j];
    a.part[((size_t)blockIdx.x * MB + m) * EV_NS + j] = s;
  }
}

// one CTA of EV_NS warps per pose of the block: warp j sums partial j over the CTAs (lane-strided, then a fixed butterfly)
__global__ void __launch_bounds__(EV_NS * 32) k_eval_fin(const double *part, int n_parts, int MB, int n_s, ScanConst sc,
                                                         const double *R, double *out) {
  __shared__ double s_v[EV_NS];
  const int m = blockIdx.x, lane = threadIdx.x & 31, j = threadIdx.x >> 5;
  double s = 0.0;
  for (int c = lane; c < n_parts; c += 32) s += part[((size_t)c * MB + m) * EV_NS + j];
  s = warp_sum(s);
  if (lane == 0) s_v[j] = s;
  __syncthreads();
  if (threadIdx.x != 0) return;
  double *o = out + (size_t)m * EV_OUT;
  const double cnt = s_v[16];
  o[0] = cnt;
  o[1] = cnt / (double)n_s;
  o[2] = cnt > 0.0 ? sqrt(s_v[17] / cnt) : 0.0;
  double v[NACC], Rp[9], H[36], b[6];
#pragma unroll
  for (int i = 0; i < NACC; i++) v[i] = s_v[i];
#pragma unroll
  for (int i = 0; i < 9; i++) Rp[i] = R[(size_t)m * 9 + i];
  gn_assemble(sc.R0, Rp, v, H, b);
#pragma unroll
  for (int i = 0; i < 36; i++) o[3 + i] = H[i];
#pragma unroll
  for (int i = 0; i < 6; i++) o[39 + i] = b[i];
}

static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

int eval_parts(int n_s, int K, int sm_count) {
  int grid = cdiv(n_s, EV_WARPS);
  const int max_grid = sm_count * ev_min_blocks((K + 31) / 32);  // one wave, grid-stride over the rows
  return grid < 1 ? 1 : (grid > max_grid ? max_grid : grid);
}

size_t eval_smem_bytes(int G, int K) {
  return (size_t)EV_WARPS * G * EV_NS * sizeof(double) + (G > 1 ? (size_t)EV_WARPS * K * sizeof(float4) : 0);
}

int launch_eval_prep(const double *poses, int M, int euler, const ScanConst &sc, float *xf, double *R, cudaStream_t st) {
  k_eval_prep<<<cdiv(M, 128), 128, 0, st>>>(poses, M, euler, sc, xf, R);
  return 1;
}

template <bool SYS>
static void go_corr(const EvalArgs &a, int grid, size_t smem, cudaStream_t st) {
  switch ((a.K + 31) / 32) {
    case 1: k_eval_corr<1, SYS><<<grid, EV_WARPS * 32, smem, st>>>(a); break;
    case 2: k_eval_corr<2, SYS><<<grid, EV_WARPS * 32, smem, st>>>(a); break;
    case 3: k_eval_corr<3, SYS><<<grid, EV_WARPS * 32, smem, st>>>(a); break;
    case 4: k_eval_corr<4, SYS><<<grid, EV_WARPS * 32, smem, st>>>(a); break;
    case 5: k_eval_corr<5, SYS><<<grid, EV_WARPS * 32, smem, st>>>(a); break;
    case 6: k_eval_corr<6, SYS><<<grid, EV_WARPS * 32, smem, st>>>(a); break;
    case 7: k_eval_corr<7, SYS><<<grid, EV_WARPS * 32, smem, st>>>(a); break;
    default: k_eval_corr<8, SYS><<<grid, EV_WARPS * 32, smem, st>>>(a); break;
  }
}

void init_eval_kernels() {
#define SVN_EV_ATTR(N)                                                                                     \
  cudaFuncSetAttribute(k_eval_corr<N, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);      \
  cudaFuncSetAttribute(k_eval_corr<N, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
  SVN_EV_ATTR(1) SVN_EV_ATTR(2) SVN_EV_ATTR(3) SVN_EV_ATTR(4) SVN_EV_ATTR(5) SVN_EV_ATTR(6) SVN_EV_ATTR(7) SVN_EV_ATTR(8)
#undef SVN_EV_ATTR
}

int launch_eval_block(const EvalArgs &a, bool want_system, const ScanConst &sc, const double *R_blk, double *out_blk, int sm_count,
                      cudaStream_t st) {
  const int grid = eval_parts(a.n_s, a.K, sm_count);
  const size_t smem = eval_smem_bytes(a.G, a.K);
  if (want_system) go_corr<true>(a, grid, smem, st);
  else go_corr<false>(a, grid, smem, st);
  launch_eval_fin(a.part, grid, a.MB, a.n_s, sc, R_blk, out_blk, st);
  return 2;
}

int launch_eval_fin(const double *part, int n_parts, int MB, int n_s, const ScanConst &sc, const double *R_blk, double *out_blk,
                    cudaStream_t st) {
  k_eval_fin<<<MB, EV_NS * 32, 0, st>>>(part, n_parts, MB, n_s, sc, R_blk, out_blk);
  return 1;
}

}  // namespace svn
