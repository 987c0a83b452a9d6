// preprocess.cu -- the scan pre-processing that runs immediately before add_cloud in the reference's node, on the device
// (SURVEY.md 8(f) row 3): OdometryPipeline::crop_pointcloud (svn-icp/src/core/OdometryPipeline.cpp:692-704) and
// OdometryPipeline::downsample_uniform (:684-690 = pcl::UniformSampling with leaf size = the "radius", applied twice:
// 0.5 * voxel_size for the cloud that goes into the map, then 1.5 * voxel_size for the registration source, :559-560).
//
// Semantics kept:
//   crop       keep p iff min_range^2 < x*x + y*y + z*z < max_range^2 (norm in float, compared in double), input order kept;
//              also reports max over ALL points of that float norm -- the reference stores this SQUARED value in
//              scan_max_range_ (:699) and later uses it as a range in metres (:577): the caller keeps the running maximum.
//   uniform    PCL 1.12 filters/impl/uniform_sampling.hpp (PCL is absent from this image: restated from its published source):
//              ijk = floor(p * (1.0f / float(leaf))) per axis; per leaf the point with the smallest
//              (x - i)^2 + (y - j)^2 + (z - k)^2 wins -- PCL measures the distance to the leaf's INTEGER INDEX, not to its
//              centre -- the first point on ties (strict '<' in cloud order).  Output order is PCL's unordered_map iteration
//              order, i.e. not part of the contract; here it is hash-slot order.
// All of it is streaming integer/byte work: one pass to mark or vote (atomicMin on (distance bits, point index) packs the
// sequential rule "strictly closer, else the earlier point" into one 64-bit key), a block scan, one pass to emit.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <string>

#include "../../include/svnicp_b200.h"
#include "block_scan.cuh"
#include "voxel_hash.cuh"

namespace {

constexpr int PB = svn::SCAN_BLOCK;  // threads per block of every kernel here (the block scans need SCAN_BLOCK)

__device__ __forceinline__ bool crop_keep(const float *p, double lo2, double hi2, float *norm_out) {
  // :697, evaluated as the host compiler does for a baseline x86-64 build: three products, two adds, no fused multiply-add
  const float norm = __fadd_rn(__fadd_rn(__fmul_rn(p[0], p[0]), __fmul_rn(p[1], p[1])), __fmul_rn(p[2], p[2]));
  *norm_out = norm;
  return (double)norm < hi2 && (double)norm > lo2;               // :700
}

__global__ void __launch_bounds__(PB) k_crop_count(const float *xyz, int n, double lo2, double hi2, int *sums, unsigned *max_bits) {
  const int i = blockIdx.x * PB + threadIdx.x;
  int c = 0;
  float norm = 0.f;
  if (i < n) c = crop_keep(xyz + 3 * (size_t)i, lo2, hi2, &norm) ? 1 : 0;
  // max of the (non-negative) float norms: their bit patterns order like the values; NaN (bits above +inf) propagates as in a max
  unsigned nb = (i < n) ? __float_as_uint(norm) : 0u;
  for (int o = 16; o > 0; o >>= 1) nb = max(nb, __shfl_xor_sync(0xffffffffu, nb, o));
  if ((threadIdx.x & 31) == 0) atomicMax(max_bits, nb);
  svn::block_sum_int(c, &sums[blockIdx.x]);
}

__global__ void __launch_bounds__(PB) k_crop_emit(const float *xyz, int n, double lo2, double hi2, const int *offs, float *out) {
  const int i = blockIdx.x * PB + threadIdx.x;
  float norm;
  const int c = (i < n && crop_keep(xyz + 3 * (size_t)i, lo2, hi2, &norm)) ? 1 : 0;
  const int off = offs[blockIdx.x] + svn::block_exclusive_scan<int>(c, nullptr);
  if (c)
    for (int k = 0; k < 3; k++) out[3 * (size_t)off + k] = xyz[3 * (size_t)i + k];
}

// first pass of UniformSampling::applyFilter: every point votes for its leaf with (distance bits, index)
__global__ void k_us_vote(const float *xyz, int n, float inv_leaf, unsigned long long *keys, unsigned long long *best, unsigned mask) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  const float x = xyz[3 * (size_t)p], y = xyz[3 * (size_t)p + 1], z = xyz[3 * (size_t)p + 2];
  const int i = (int)floorf(x * inv_leaf), j = (int)floorf(y * inv_leaf), k = (int)floorf(z * inv_leaf);
  const float dx = x - (float)i, dy = y - (float)j, dz = z - (float)k;
  // distance to the leaf INDEX (PCL's rule), unfused left-to-right like the restatement in oracle/preprocess_oracle.c;
  // NaN points vote last
  const float diff = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
  const unsigned long long vote = ((unsigned long long)__float_as_uint(diff) << 32) | (unsigned)p;
  bool created;
  const int slot = svn::hash_insert(keys, mask, svn::pack_voxel_key(i, j, k), &created);  // never -1: slots >= 2 n
  atomicMin(&best[slot], vote);  // smaller distance wins; equal distances: the earlier point (strict '<' in cloud order)
}

__global__ void __launch_bounds__(PB) k_us_count(const unsigned long long *keys, int slots, int *sums) {
  const int s = blockIdx.x * PB + threadIdx.x;
  svn::block_sum_int((s < slots && keys[s] != svn::EMPTY_KEY) ? 1 : 0, &sums[blockIdx.x]);
}

__global__ void __launch_bounds__(PB) k_us_emit(const float *xyz, const unsigned long long *keys, const unsigned long long *best, int slots,
                                                const int *offs, float *out) {
  const int s = blockIdx.x * PB + threadIdx.x;
  const int c = (s < slots && keys[s] != svn::EMPTY_KEY) ? 1 : 0;
  const int off = offs[blockIdx.x] + svn::block_exclusive_scan<int>(c, nullptr);
  if (c) {
    const unsigned p = (unsigned)(best[s] & 0xFFFFFFFFull);
    for (int k = 0; k < 3; k++) out[3 * (size_t)off + k] = xyz[3 * (size_t)p + k];
  }
}

__global__ void k_f32_to_f64(const float *in, double *out, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (double)in[i];
}

}  // namespace


// ---------------------------------------------------------------------------------------------
// De-skewing: OdometryPipeline::deskew_pointcloud (OdometryPipeline.cpp:357-447).  Two streaming kernels (HBM bound:
// 12 + 8 B read, 12 B written per point): stamps (+ the KITTI tilt) and their min / max; then one SE(3) exponential per point.
// The Pose3 Exp / Log closed forms are GTSAM 4.2's (gtsam/geometry/Pose3.cpp, SO3.cpp), twist order [omega ; v].
// ---------------------------------------------------------------------------------------------
__host__ __device__ inline void se3_rot_exp(const double w[3], double R[9]) {
  const double theta2 = w[0] * w[0] + w[1] * w[1] + w[2] * w[2];
  const double W[9] = {0, -w[2], w[1], w[2], 0, -w[0], -w[1], w[0], 0};
  if (theta2 <= 2.220446049250313e-16) {
    for (int i = 0; i < 9; i++) R[i] = ((i % 4 == 0) ? 1.0 : 0.0) + W[i];
    return;
  }
  const double theta = sqrt(theta2), sn = sin(theta), s2 = sin(0.5 * theta), omc = 2.0 * s2 * s2;
  double K[9];
  for (int i = 0; i < 9; i++) K[i] = W[i] / theta;
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) {
      const double kk = K[3 * r] * K[c] + K[3 * r + 1] * K[3 + c] + K[3 * r + 2] * K[6 + c];
      R[3 * r + c] = ((r == c) ? 1.0 : 0.0) + sn * K[3 * r + c] + omc * kk;
    }
}
__host__ __device__ inline void se3_exp(const double xi[6], double R[9], double t[3]) {
  const double *w = xi, *v = xi + 3;
  se3_rot_exp(w, R);
  const double theta2 = w[0] * w[0] + w[1] * w[1] + w[2] * w[2];
  if (theta2 > 2.220446049250313e-16) {
    const double wv = w[0] * v[0] + w[1] * v[1] + w[2] * v[2];
    const double c[3] = {w[1] * v[2] - w[2] * v[1], w[2] * v[0] - w[0] * v[2], w[0] * v[1] - w[1] * v[0]};
    for (int r = 0; r < 3; r++) t[r] = (c[r] - (R[3 * r] * c[0] + R[3 * r + 1] * c[1] + R[3 * r + 2] * c[2]) + w[r] * wv) / theta2;
  } else {
    t[0] = v[0]; t[1] = v[1]; t[2] = v[2];
  }
}
static void se3_rot_log(const double R[9], double w[3]) {
  const double pi = 3.14159265358979323846;
  const double tr = R[0] + R[4] + R[8];
  if (tr + 1.0 < 1e-10) {
    if (fabs(R[8] + 1.0) > 1e-5) { const double f = pi / sqrt(2.0 + 2.0 * R[8]); w[0] = f * R[2]; w[1] = f * R[5]; w[2] = f * (1.0 + R[8]); }
    else if (fabs(R[4] + 1.0) > 1e-5) { const double f = pi / sqrt(2.0 + 2.0 * R[4]); w[0] = f * R[1]; w[1] = f * (1.0 + R[4]); w[2] = f * R[7]; }
    else { const double f = pi / sqrt(2.0 + 2.0 * R[0]); w[0] = f * (1.0 + R[0]); w[1] = f * R[3]; w[2] = f * R[6]; }
    return;
  }
  const double tr_3 = tr - 3.0;
  double mag;
  if (tr_3 < -1e-7) { const double theta = acos((tr - 1.0) / 2.0); mag = theta / (2.0 * sin(theta)); }
  else mag = 0.5 - tr_3 / 12.0;
  w[0] = mag * (R[7] - R[5]); w[1] = mag * (R[2] - R[6]); w[2] = mag * (R[3] - R[1]);
}
// delta_pose = Pose3::Logmap(start^-1 * finish), OdometryPipeline.cpp:424
static void se3_delta_log(const double Rs[9], const double ts[3], const double Rf[9], const double tf[3], double xi[6]) {
  double R[9], T[3], w[3];
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) R[3 * r + c] = Rs[r] * Rf[c] + Rs[3 + r] * Rf[3 + c] + Rs[6 + r] * Rf[6 + c];
  const double d[3] = {tf[0] - ts[0], tf[1] - ts[1], tf[2] - ts[2]};
  for (int r = 0; r < 3; r++) T[r] = Rs[r] * d[0] + Rs[3 + r] * d[1] + Rs[6 + r] * d[2];
  se3_rot_log(R, w);
  const double t = sqrt(w[0] * w[0] + w[1] * w[1] + w[2] * w[2]);
  xi[0] = w[0]; xi[1] = w[1]; xi[2] = w[2];
  if (t < 1e-10) { xi[3] = T[0]; xi[4] = T[1]; xi[5] = T[2]; return; }
  const double k[3] = {w[0] / t, w[1] / t, w[2] / t};
  const double WT[3] = {k[1] * T[2] - k[2] * T[1], k[2] * T[0] - k[0] * T[2], k[0] * T[1] - k[1] * T[0]};
  const double WWT[3] = {k[1] * WT[2] - k[2] * WT[1], k[2] * WT[0] - k[0] * WT[2], k[0] * WT[1] - k[1] * WT[0]};
  const double Tan = tan(0.5 * t);
  for (int i = 0; i < 3; i++) xi[3 + i] = T[i] - (0.5 * t) * WT[i] + (1.0 - t / (2.0 * Tan)) * WWT[i];
}

// doubles order like these unsigned keys (NaN excluded by the caller's data contract: stamps are finite)
__device__ __forceinline__ unsigned long long ord_key(double d) {
  const unsigned long long b = (unsigned long long)__double_as_longlong(d);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double ord_val(unsigned long long k) {
  return __longlong_as_double((long long)((k >> 63) ? (k & 0x7FFFFFFFFFFFFFFFull) : ~k));
}

struct Twist6 { double xi[6]; };

// pass 1: (KITTI: tilt the point, stamp from its azimuth, :385-399) stamps -> st, block min / max -> global
__global__ void __launch_bounds__(PB) k_deskew_stamps(const float *__restrict__ xyz, const double *__restrict__ stamps, long long n, int kitti,
                                                      float *__restrict__ pts, double *__restrict__ st, unsigned long long *minmax) {
  __shared__ unsigned long long s_mn[PB / 32], s_mx[PB / 32];
  const long long i = (long long)blockIdx.x * PB + threadIdx.x;
  unsigned long long kmn = ~0ull, kmx = 0ull;
  if (i < n) {
    double s;
    if (kitti) {
      const double pi = 3.14159265358979323846, off = (0.205 * pi) / 180.0;
      const double p[3] = {(double)xyz[3 * i], (double)xyz[3 * i + 1], (double)xyz[3 * i + 2]};
      double a[3] = {p[1], -p[0], 0.0};  // pt.cross(unit z)
      const double an = sqrt(a[0] * a[0] + a[1] * a[1]);
      if (an > 0) { a[0] /= an; a[1] /= an; }
      const double c = cos(off), sn = sin(off), ad = a[0] * p[0] + a[1] * p[1] + a[2] * p[2];
      const double cr[3] = {a[1] * p[2] - a[2] * p[1], a[2] * p[0] - a[0] * p[2], a[0] * p[1] - a[1] * p[0]};
      float q[3];
      for (int k = 0; k < 3; k++) { q[k] = (float)(c * p[k] + sn * cr[k] + (1.0 - c) * ad * a[k]); pts[3 * i + k] = q[k]; }
      const double yaw = -atan2((double)q[1], (double)q[0]);
      s = 0.5 * (yaw / pi + 1.0);
    } else {
      for (int k = 0; k < 3; k++) pts[3 * i + k] = xyz[3 * i + k];
      s = stamps[i];
    }
    st[i] = s;
    kmn = kmx = ord_key(s);
  }
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long a = __shfl_xor_sync(0xffffffffu, kmn, o), b = __shfl_xor_sync(0xffffffffu, kmx, o);
    kmn = a < kmn ? a : kmn;
    kmx = b > kmx ? b : kmx;
  }
  if ((threadIdx.x & 31) == 0) { s_mn[threadIdx.x >> 5] = kmn; s_mx[threadIdx.x >> 5] = kmx; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < PB / 32; w++) { kmn = s_mn[w] < kmn ? s_mn[w] : kmn; kmx = s_mx[w] > kmx ? s_mx[w] : kmx; }
    atomicMin(minmax, kmn);
    atomicMax(minmax + 1, kmx);
  }
}

// pass 2: p' = Expmap((stamp_normalised - 0.5) * delta_pose).transformFrom(p), :417-439; all stamps equal -> the input cloud (:415)
__global__ void __launch_bounds__(PB) k_deskew_apply(const float *__restrict__ xyz, const float *__restrict__ pts, const double *__restrict__ st,
                                                     long long n, const unsigned long long *__restrict__ minmax, Twist6 d, float *__restrict__ out) {
  const long long i = (long long)blockIdx.x * PB + threadIdx.x;
  if (i >= n) return;
  const double mn = ord_val(minmax[0]), mx = ord_val(minmax[1]);
  if (mn == mx) {
    for (int k = 0; k < 3; k++) out[3 * i + k] = xyz[3 * i + k];
    return;
  }
  const double f = (st[i] - mn) / (mx - mn) - 0.5;
  double tw[6], R[9], t[3];
  for (int k = 0; k < 6; k++) tw[k] = f * d.xi[k];
  se3_exp(tw, R, t);
  const double p[3] = {(double)pts[3 * i], (double)pts[3 * i + 1], (double)pts[3 * i + 2]};
  for (int r = 0; r < 3; r++) out[3 * i + r] = (float)(R[3 * r] * p[0] + R[3 * r + 1] * p[1] + R[3 * r + 2] * p[2] + t[r]);
}

struct svnicp_pre_t {
  int device = 0;
  size_t cap = 0;  // points
  float *in = nullptr, *buf[2] = {nullptr, nullptr};
  double *f64 = nullptr;
  double *stamps = nullptr;            // [2][cap]: staged time stamps, stamps in use (lazily allocated by svnicp_pre_deskew)
  unsigned long long *d_minmax = nullptr;  // ordered-bits min / max of the stamps
  unsigned long long *keys = nullptr, *best = nullptr;
  size_t slots = 0;
  int *sums = nullptr;
  long long *d_total = nullptr;
  unsigned *d_max = nullptr;
  long long *h_total = nullptr;  // pinned: [0] count, [1] max bits
  int last = 1;                  // buffer holding the last output
  cudaStream_t stream = nullptr;
  std::string err;
};

static thread_local std::string g_pre_create_error;

static int pfail(svnicp_pre p, int code, const char *what, cudaError_t e = cudaSuccess) {
  char b[256];
  snprintf(b, sizeof(b), "%s%s%s", what, e != cudaSuccess ? ": " : "", e != cudaSuccess ? cudaGetErrorString(e) : "");
  if (p) p->err = b;
  else g_pre_create_error = b;
  return code;
}
#define PCU(call)                                                                                                  \
  do {                                                                                                             \
    cudaError_t e__ = (call);                                                                                      \
    if (e__ != cudaSuccess) return pfail(p, e__ == cudaErrorMemoryAllocation ? SVNICP_ERR_OOM : SVNICP_ERR_CUDA, #call, e__); \
  } while (0)

// input staging: host clouds are copied in; a device cloud is used where it lies.  Output goes to the buffer that is not the input.
static int stage_input(svnicp_pre p, const float *xyz, int64_t n, int on_device, const float **src, int *out_buf) {
  if ((size_t)n > p->cap) return pfail(p, SVNICP_ERR_INVALID, "cloud larger than max_points given to svnicp_pre_create");
  if (!on_device) {
    PCU(cudaMemcpyAsync(p->in, xyz, (size_t)n * 3 * sizeof(float), cudaMemcpyHostToDevice, p->stream));
    *src = p->in;
    *out_buf = p->last ^ 1;
  } else {
    *src = xyz;
    *out_buf = (xyz == p->buf[0]) ? 1 : (xyz == p->buf[1]) ? 0 : (p->last ^ 1);
  }
  return SVNICP_OK;
}

extern "C" {

int svnicp_pre_create(svnicp_pre *out, int64_t max_points, int device) {
  if (!out) return SVNICP_ERR_INVALID;
  *out = nullptr;
  if (max_points < 1 || max_points > (1ll << 30)) return pfail(nullptr, SVNICP_ERR_INVALID, "svnicp_pre_create: bad max_points");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return pfail(nullptr, SVNICP_ERR_NO_DEVICE, "no CUDA device: this library has no CPU fallback");
  if (device < 0) cudaGetDevice(&device);
  if (device >= ndev) return pfail(nullptr, SVNICP_ERR_NO_DEVICE, "device out of range");
  svnicp_pre p = new svnicp_pre_t();
  p->device = device;
  p->cap = (size_t)max_points;
  size_t slots = 1024;
  while (slots < 2 * p->cap) slots <<= 1;
  p->slots = slots;
  auto body = [&]() -> int {
    PCU(cudaSetDevice(device));
    PCU(cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking));
    PCU(cudaMalloc((void **)&p->in, p->cap * 3 * sizeof(float)));
    for (int i = 0; i < 2; i++) PCU(cudaMalloc((void **)&p->buf[i], p->cap * 3 * sizeof(float)));
    PCU(cudaMalloc((void **)&p->f64, p->cap * 3 * sizeof(double)));
    PCU(cudaMalloc((void **)&p->keys, slots * sizeof(unsigned long long)));
    PCU(cudaMalloc((void **)&p->best, slots * sizeof(unsigned long long)));
    PCU(cudaMalloc((void **)&p->sums, ((slots + PB - 1) / PB + 2) * sizeof(int)));
    PCU(cudaMalloc((void **)&p->d_total, sizeof(long long)));
    PCU(cudaMalloc((void **)&p->d_max, sizeof(unsigned)));
    PCU(cudaMallocHost((void **)&p->h_total, 2 * sizeof(long long)));
    return SVNICP_OK;
  };
  const int rc = body();
  if (rc != SVNICP_OK) {
    g_pre_create_error = p->err;
    svnicp_pre_destroy(p);
    return rc;
  }
  *out = p;
  return SVNICP_OK;
}

void svnicp_pre_destroy(svnicp_pre p) {
  if (!p) return;
  cudaSetDevice(p->device);
  if (p->stream) cudaStreamSynchronize(p->stream);
  cudaFree(p->in); cudaFree(p->buf[0]); cudaFree(p->buf[1]); cudaFree(p->f64); cudaFree(p->keys); cudaFree(p->best);
  cudaFree(p->sums); cudaFree(p->d_total); cudaFree(p->d_max); cudaFree(p->stamps); cudaFree(p->d_minmax);
  if (p->h_total) cudaFreeHost(p->h_total);
  if (p->stream) cudaStreamDestroy(p->stream);
  delete p;
}

const char *svnicp_pre_last_error(svnicp_pre p) { return p ? p->err.c_str() : g_pre_create_error.c_str(); }

int svnicp_pre_crop(svnicp_pre p, const float *xyz, int64_t n, int on_device, double min_range, double max_range, const float **dev_out,
                    int64_t *n_out, double *max_sq_norm) {
  if (!p || !n_out || (n > 0 && !xyz) || n < 0) return SVNICP_ERR_INVALID;
  PCU(cudaSetDevice(p->device));
  const float *src = nullptr;
  int ob = 0;
  int rc = stage_input(p, xyz, n, on_device, &src, &ob);
  if (rc) return rc;
  const int nb = (int)((n + PB - 1) / PB);
  PCU(cudaMemsetAsync(p->d_max, 0, sizeof(unsigned), p->stream));
  PCU(cudaMemsetAsync(p->d_total, 0, sizeof(long long), p->stream));
  const double lo2 = min_range * min_range, hi2 = max_range * max_range;
  if (n > 0) {
    k_crop_count<<<nb, PB, 0, p->stream>>>(src, (int)n, lo2, hi2, p->sums, p->d_max);
    svn::k_scan_block_sums<int><<<1, PB, 0, p->stream>>>(p->sums, nb, p->d_total);
    k_crop_emit<<<nb, PB, 0, p->stream>>>(src, (int)n, lo2, hi2, p->sums, p->buf[ob]);
    PCU(cudaGetLastError());
  }
  PCU(cudaMemcpyAsync(&p->h_total[0], p->d_total, sizeof(long long), cudaMemcpyDeviceToHost, p->stream));
  PCU(cudaMemcpyAsync(&p->h_total[1], p->d_max, sizeof(unsigned), cudaMemcpyDeviceToHost, p->stream));
  PCU(cudaStreamSynchronize(p->stream));
  p->last = ob;
  *n_out = p->h_total[0];
  if (dev_out) *dev_out = p->buf[ob];
  if (max_sq_norm) {
    const unsigned bits = (unsigned)(p->h_total[1] & 0xFFFFFFFFll);
    float f;
    memcpy(&f, &bits, sizeof(f));
    *max_sq_norm = (double)f;
  }
  return SVNICP_OK;
}

int svnicp_pre_downsample_uniform(svnicp_pre p, const float *xyz, int64_t n, int on_device, double leaf, const float **dev_out, int64_t *n_out) {
  if (!p || !n_out || (n > 0 && !xyz) || n < 0) return SVNICP_ERR_INVALID;
  if (!(leaf > 0)) return pfail(p, SVNICP_ERR_INVALID, "svnicp_pre_downsample_uniform: leaf size must be positive");
  PCU(cudaSetDevice(p->device));
  const float *src = nullptr;
  int ob = 0;
  int rc = stage_input(p, xyz, n, on_device, &src, &ob);
  if (rc) return rc;
  PCU(cudaMemsetAsync(p->keys, 0xFF, p->slots * sizeof(unsigned long long), p->stream));
  PCU(cudaMemsetAsync(p->best, 0xFF, p->slots * sizeof(unsigned long long), p->stream));
  PCU(cudaMemsetAsync(p->d_total, 0, sizeof(long long), p->stream));
  if (n > 0) {
    const float inv_leaf = 1.0f / (float)leaf;  // inverse_leaf_size_ = Array4f::Ones() / leaf_size_.array()
    const int nb = (int)((p->slots + PB - 1) / PB);
    k_us_vote<<<(unsigned)((n + 255) / 256), 256, 0, p->stream>>>(src, (int)n, inv_leaf, p->keys, p->best, (unsigned)(p->slots - 1));
    k_us_count<<<nb, PB, 0, p->stream>>>(p->keys, (int)p->slots, p->sums);
    svn::k_scan_block_sums<int><<<1, PB, 0, p->stream>>>(p->sums, nb, p->d_total);
    k_us_emit<<<nb, PB, 0, p->stream>>>(src, p->keys, p->best, (int)p->slots, p->sums, p->buf[ob]);
    PCU(cudaGetLastError());
  }
  PCU(cudaMemcpyAsync(&p->h_total[0], p->d_total, sizeof(long long), cudaMemcpyDeviceToHost, p->stream));
  PCU(cudaStreamSynchronize(p->stream));
  p->last = ob;
  *n_out = p->h_total[0];
  if (dev_out) *dev_out = p->buf[ob];
  return SVNICP_OK;
}

int svnicp_pre_deskew(svnicp_pre p, const float *xyz, int64_t n, int on_device, const double *stamps, int stamps_on_device, int kitti,
                      const double R_start[9], const double t_start[3], const double R_finish[9], const double t_finish[3],
                      const float **dev_out, int32_t *moved) {
  if (!p || n < 0 || (n > 0 && !xyz) || !R_start || !t_start || !R_finish || !t_finish) return SVNICP_ERR_INVALID;
  if (!kitti && n > 0 && !stamps) return pfail(p, SVNICP_ERR_INVALID, "svnicp_pre_deskew: per-point time stamps needed unless kitti != 0");
  PCU(cudaSetDevice(p->device));
  const float *src = nullptr;
  int ob = 0;
  int rc = stage_input(p, xyz, n, on_device, &src, &ob);
  if (rc) return rc;
  if (!p->stamps) {
    PCU(cudaMalloc((void **)&p->stamps, 2 * p->cap * sizeof(double)));
    PCU(cudaMalloc((void **)&p->d_minmax, 2 * sizeof(unsigned long long)));
  }
  const double *st_in = nullptr;
  if (!kitti && n > 0) {
    if (stamps_on_device) st_in = stamps;
    else {
      PCU(cudaMemcpyAsync(p->stamps, stamps, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, p->stream));
      st_in = p->stamps;
    }
  }
  const unsigned long long init[2] = {~0ull, 0ull};
  PCU(cudaMemcpyAsync(p->d_minmax, init, sizeof(init), cudaMemcpyHostToDevice, p->stream));
  Twist6 d;
  se3_delta_log(R_start, t_start, R_finish, t_finish, d.xi);
  // the tilted copy (KITTI) / plain copy goes to the third float buffer; the result to the output buffer
  float *pts = (src == p->in) ? p->buf[ob ^ 1] : p->in;
  if (n > 0) {
    const unsigned nb = (unsigned)((n + PB - 1) / PB);
    k_deskew_stamps<<<nb, PB, 0, p->stream>>>(src, st_in, (long long)n, kitti, pts, p->stamps + p->cap, p->d_minmax);
    k_deskew_apply<<<nb, PB, 0, p->stream>>>(src, pts, p->stamps + p->cap, (long long)n, p->d_minmax, d, p->buf[ob]);
    PCU(cudaGetLastError());
  }
  unsigned long long mm[2] = {0, 0};
  PCU(cudaMemcpyAsync(mm, p->d_minmax, sizeof(mm), cudaMemcpyDeviceToHost, p->stream));
  PCU(cudaStreamSynchronize(p->stream));
  p->last = ob;
  if (dev_out) *dev_out = p->buf[ob];
  if (moved) *moved = (n > 0 && mm[0] != mm[1]) ? 1 : 0;
  return SVNICP_OK;
}

// updater_ of the ICP estimator (OdometryPipeline.cpp:37-45) with tensor2gtsamPose3 (ICPUtils.cpp:84-98):
// pose = initial_guess * Pose3(Rot3::Expmap(mean[3:6]), mean[0:3]).  Host arithmetic on 12 + 6 doubles.
int svnicp_pose_compose(const double R0[9], const double t0[3], const double mean6[6], double R_out[9], double t_out[3]) {
  if (!R0 || !t0 || !mean6 || !R_out || !t_out) return SVNICP_ERR_INVALID;
  double Rc[9];
  se3_rot_exp(mean6 + 3, Rc);
  for (int r = 0; r < 3; r++) {
    for (int c = 0; c < 3; c++) R_out[3 * r + c] = R0[3 * r] * Rc[c] + R0[3 * r + 1] * Rc[3 + c] + R0[3 * r + 2] * Rc[6 + c];
    t_out[r] = R0[3 * r] * mean6[0] + R0[3 * r + 1] * mean6[1] + R0[3 * r + 2] * mean6[2] + t0[r];
  }
  return SVNICP_OK;
}

int svnicp_pre_to_f64(svnicp_pre p, const float *dev_xyz, int64_t n, const double **dev_out) {
  if (!p || !dev_out || n < 0 || (size_t)n > p->cap) return SVNICP_ERR_INVALID;
  PCU(cudaSetDevice(p->device));
  if (n > 0) {
    k_f32_to_f64<<<(unsigned)(((size_t)n * 3 + 255) / 256), 256, 0, p->stream>>>(dev_xyz, p->f64, (size_t)n * 3);
    PCU(cudaGetLastError());
  }
  PCU(cudaStreamSynchronize(p->stream));
  *dev_out = p->f64;
  return SVNICP_OK;
}

int svnicp_pre_download(svnicp_pre p, const float *dev_xyz, int64_t n, float *out) {
  if (!p || n < 0 || (n > 0 && (!dev_xyz || !out))) return SVNICP_ERR_INVALID;
  PCU(cudaSetDevice(p->device));
  if (n > 0) PCU(cudaMemcpy(out, dev_xyz, (size_t)n * 3 * sizeof(float), cudaMemcpyDeviceToHost));
  return SVNICP_OK;
}

}  // extern "C"
