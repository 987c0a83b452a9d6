// cand_build.cu -- per-scan candidate builder (north_star kernel (a), per-scan part).
//
// Replaces SVGDICP::knn_source_cloud + the index_select gathers of mini_batch_pair_generator
// (reference svn-icp/src/core/SVGDICP.cpp:176-215), i.e. the brute-force
// KNearestNeighborKernelV1<double,3> (src/core/knn/knn.cu:68-111): for every source point
// q0_b = R0 s_b + t0 the K = KNN_count nearest map points.
//
// B200 design: a voxel hash of the map is rebuilt per scan (3 streaming kernels, no sort), then one
// warp per source point gathers the cells of growing Chebyshev rings, keeps (d^2, index) pairs in
// shared memory and stops as soon as K points lie inside the radius the visited cube is known to
// cover completely.  The result is EXACT: the same K-nearest set as the brute force (fp64 distances,
// identical fma order), emitted in ascending (d0^2, map index) order.  Queries whose ring search
// exceeds RING_MAX fall back to a brute-force sweep of the whole map inside the same kernel.
// Documented difference to the reference: slot ORDER (the reference leaves MinK replacement order,
// mink.cuh:62-83); parity is therefore stated on global map indices, ties between exactly equal
// fp32 distances go to the earlier slot of OUR order (see DESIGN.md "tie-break").
#include "block_scan.cuh"
#include "common.cuh"
#include "kernels.h"
#include "voxel_hash.cuh"

namespace svn {

constexpr int RING_MAX = 6;
constexpr int KNN_WARPS = 4;
#ifndef SVN_KNN_CAP
#define SVN_KNN_CAP 512
#endif
// (d^2, pos, idx) entries per warp, power of two (bitonic sort).  The kernel is latency bound, so resident warps matter:
// 1024 entries = 16 KB per warp -> 12 warps/SM; 512 -> 24 warps/SM, with buffer overflows relieved by a histogram cut
// (warp_cut) instead of a full sort (measured at configs[1]: see DESIGN.md section 4).
constexpr int KNN_CAP = SVN_KNN_CAP;
constexpr int KNN_BINS = 64;

struct Ent {
  double d;
  int pos;
  int idx;
};

__device__ __forceinline__ int cell_of(double x, double inv_cell) { return (int)floor(x * inv_cell); }
// q0 = R0 s + t0 (SVGDICP.cpp:204) in the fma order shared with oracle_transform_q0; sp = fp32(R0 s).
__global__ void k_q0(const double *__restrict__ src, int n_s, ScanConst sc, double *__restrict__ q0, float4 *__restrict__ sp,
                     int n_pad) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_pad) return;
  if (i >= n_s) { sp[i] = make_float4(0.f, 0.f, 0.f, 0.f); return; }
  const double x = src[3 * i], y = src[3 * i + 1], z = src[3 * i + 2];
  double r[3];
#pragma unroll
  for (int a = 0; a < 3; a++) {
    q0[3 * i + a] = affine_row_fma(sc.R0, sc.t0, a, x, y, z);
    r[a] = fma(sc.R0[3 * a], x, fma(sc.R0[3 * a + 1], y, sc.R0[3 * a + 2] * z));
  }
  const float fx = __double2float_rn(r[0]), fy = __double2float_rn(r[1]), fz = __double2float_rn(r[2]);
  const double nrm = sqrt((double)fx * fx + (double)fy * fy + (double)fz * fz);
  sp[i] = make_float4(fx, fy, fz, __double2float_ru(nrm * (1.0 + 1e-7)));
}

__global__ void k_grid_clear(unsigned long long *keys, int *counts, int *fill, int table_size, int *cursor) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < table_size) { keys[i] = EMPTY_KEY; counts[i] = 0; fill[i] = 0; }
  if (i == 0) *cursor = 0;
}

__global__ void k_grid_count(const double *__restrict__ tgt, int n_t, double inv_cell, unsigned long long *keys, int *counts,
                             int *pt_slot, unsigned mask) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_t) return;
  const unsigned long long key = pack_voxel_key(cell_of(tgt[3 * j], inv_cell), cell_of(tgt[3 * j + 1], inv_cell), cell_of(tgt[3 * j + 2], inv_cell));
  bool created;
  const int slot = hash_insert(keys, mask, key, &created);  // never -1: table_size >= 2 n_t
  atomicAdd(&counts[slot], 1);
  pt_slot[j] = slot;
}

__global__ void k_grid_alloc(const int *counts, int *starts, int table_size, int *cursor) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= table_size) return;
  const int c = counts[i];
  if (c > 0) starts[i] = atomicAdd(cursor, c);
}

__global__ void k_grid_scatter(const double *__restrict__ tgt, int n_t, const int *__restrict__ pt_slot, const int *__restrict__ starts,
                               int *fill, double *__restrict__ sxyz, int *__restrict__ sidx) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_t) return;
  const int slot = pt_slot[j];
  const int pos = starts[slot] + atomicAdd(&fill[slot], 1);
  sxyz[3 * pos] = tgt[3 * j];
  sxyz[3 * pos + 1] = tgt[3 * j + 1];
  sxyz[3 * pos + 2] = tgt[3 * j + 2];
  sidx[pos] = j;
}

__device__ __forceinline__ bool ent_less(const Ent &a, const Ent &b) { return a.d < b.d || (a.d == b.d && a.idx < b.idx); }

// warp bitonic sort of buf[0..n) (n power of two), ascending (d, idx)
__device__ void warp_sort(Ent *buf, int n) {
  const int lane = lane_id();
  for (int k = 2; k <= n; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      // one lane per compare-exchange PAIR (n/2 pairs), so no lane idles
      for (int t = lane; t < (n >> 1); t += 32) {
        const int i = (t & (j - 1)) | ((t & ~(j - 1)) << 1);
        const int ixj = i | j;
        const Ent a = buf[i], b = buf[ixj];
        const bool up = (i & k) == 0;
        if (ent_less(b, a) == up) { buf[i] = b; buf[ixj] = a; }
      }
      __syncwarp();
    }
}

// The same bitonic network with the elements in REGISTERS (NPER per lane, blocked: element NPER*lane + r): partner distances
// below NPER are register-to-register exchanges, the others four 32-bit shuffles per element; no shared-memory round trip and
// no __syncwarp per stage.  ncu on the shared-memory version: the sort is ~60 % of k_knn's 1e9 warp instructions and the
// kernel stalls 5.2 warps per issue on the short scoreboard (LDS/STS).  Sorts buf[0 .. 32*NPER) ascending (d, idx).
__device__ __forceinline__ Ent ent_shfl_xor(const Ent &e, int lane_mask) {
  Ent r;
  const int lo = __shfl_xor_sync(0xffffffffu, __double2loint(e.d), lane_mask);
  const int hi = __shfl_xor_sync(0xffffffffu, __double2hiint(e.d), lane_mask);
  r.d = __hiloint2double(hi, lo);
  r.pos = __shfl_xor_sync(0xffffffffu, e.pos, lane_mask);
  r.idx = __shfl_xor_sync(0xffffffffu, e.idx, lane_mask);
  return r;
}

template <int NPER>
__device__ void warp_sort_regs(Ent *buf) {
  const int lane = lane_id();
  constexpr int n = 32 * NPER;
  Ent e[NPER];
#pragma unroll
  for (int r = 0; r < NPER; r++) e[r] = buf[NPER * lane + r];
#pragma unroll
  for (int k = 2; k <= n; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
      if (j >= NPER) {
        const int lm = j / NPER;
        const bool lower = (lane & lm) == 0;
#pragma unroll
        for (int r = 0; r < NPER; r++) {
          const bool asc = (((NPER * lane + r) & k) == 0);
          const Ent o = ent_shfl_xor(e[r], lm);
          // the lower index of the pair keeps the smaller element when ascending (the larger when descending)
          const bool take = (lower == asc) ? ent_less(o, e[r]) : ent_less(e[r], o);
          if (take) e[r] = o;
        }
      } else {
#pragma unroll
        for (int r = 0; r < NPER; r++) {
          const int rp = r ^ j;
          if (rp > r) {
            const bool asc = (((NPER * lane + r) & k) == 0);
            const bool swap = asc ? ent_less(e[rp], e[r]) : ent_less(e[r], e[rp]);
            if (swap) { const Ent t = e[r]; e[r] = e[rp]; e[rp] = t; }
          }
        }
      }
    }
  }
  __syncwarp();
#pragma unroll
  for (int r = 0; r < NPER; r++) buf[NPER * lane + r] = e[r];
  __syncwarp();
}

// keep the K smallest of buf[0..count); returns the new count (<= K); *tau = K-th key if full
__device__ int warp_compact(Ent *buf, int count, int K, double *tau) {
  const int lane = lane_id();
  int n = 32;
  while (n < count) n <<= 1;
  for (int i = count + lane; i < n; i += 32) { buf[i].d = INFINITY; buf[i].pos = -1; buf[i].idx = 0x7fffffff; }
  __syncwarp();
  switch (n) {  // register-resident up to 256 elements (8 per lane); larger buffers (rare: overflow fallbacks) sort in shared memory
    case 32: warp_sort_regs<1>(buf); break;
    case 64: warp_sort_regs<2>(buf); break;
    case 128: warp_sort_regs<4>(buf); break;
    case 256: warp_sort_regs<8>(buf); break;
    default: warp_sort(buf, n); break;
  }
  const int c = count < K ? count : K;
  if (c == K) *tau = buf[K - 1].d;
  return c;
}

// Cheap overflow relief (no sort): 64-bin histogram of d over [0, max d in the buffer]; keep every entry up to the bin
// that holds the K-th smallest -- an exact superset of the K nearest seen so far.  The bin function is monotone in d, so
// a later point may be dropped iff its bin exceeds *cut_bin under the same *cut_scale.  Returns the new count (unchanged
// when the cut cannot shrink the buffer: all keys in one bin).
__device__ __forceinline__ int cut_bin_of(double d, double scale) { return min(KNN_BINS - 1, (int)(d * scale)); }

__device__ int warp_cut(Ent *buf, int count, int K, double *cut_scale, int *cut_bin, int *hist) {
  const int lane = lane_id();
  const unsigned lt_mask = (1u << lane) - 1u;
  double dmax = 0.0;
  for (int i = lane; i < count; i += 32) dmax = fmax(dmax, buf[i].d);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) dmax = fmax(dmax, __shfl_xor_sync(0xffffffffu, dmax, o));
  if (!(dmax > 0.0) || dmax == INFINITY) return count;
  const double scale = (double)KNN_BINS / dmax;
  hist[lane] = 0;
  hist[lane + 32] = 0;
  __syncwarp();
  for (int i = lane; i < count; i += 32) atomicAdd(&hist[cut_bin_of(buf[i].d, scale)], 1);
  __syncwarp();
  const int h0 = hist[2 * lane], h1 = hist[2 * lane + 1];
  const int incl = warp_inclusive_scan(h0 + h1);
  const int before = incl - h0 - h1;
  int tbin = KNN_BINS;
  if (before < K && before + h0 >= K) tbin = 2 * lane;
  else if (before + h0 < K && incl >= K) tbin = 2 * lane + 1;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) tbin = min(tbin, __shfl_xor_sync(0xffffffffu, tbin, o));
  __syncwarp();
  if (tbin >= KNN_BINS - 1) return count;  // fewer than K entries, or the K-th sits in the last bin: nothing to drop
  int m_out = 0;
  for (int i0 = 0; i0 < count; i0 += 32) {
    const int i = i0 + lane;
    Ent e;
    bool keep = false;
    if (i < count) {
      e = buf[i];
      keep = cut_bin_of(e.d, scale) <= tbin;
    }
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    __syncwarp();
    if (keep) buf[m_out + __popc(m & lt_mask)] = e;
    m_out += __popc(m);
    __syncwarp();
  }
  *cut_scale = scale;
  *cut_bin = tbin;
  return m_out;
}

__global__ void __launch_bounds__(KNN_WARPS * 32)
k_knn(const double *__restrict__ q0, int row_lo, int row_hi, const double *__restrict__ tgt, int n_t, const double *__restrict__ sxyz,
      const int *__restrict__ sidx, const unsigned long long *__restrict__ keys, const int *__restrict__ starts,
      const int *__restrict__ counts, unsigned mask, double cell, int K, float4 *__restrict__ cand, int *__restrict__ cand_idx,
      int *__restrict__ fallback_count) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = lane_id();
  Ent *buf = reinterpret_cast<Ent *>(smem_raw) + (size_t)warp * KNN_CAP;
  __shared__ int s_start[KNN_WARPS][32], s_excl[KNN_WARPS][33], s_hist[KNN_WARPS][KNN_BINS];
  const double inv_cell = 1.0 / cell;
  const unsigned lt_mask = (1u << lane) - 1u;

  for (int b = row_lo + blockIdx.x * KNN_WARPS + warp; b < row_hi; b += gridDim.x * KNN_WARPS) {
    const double q[3] = {q0[3 * b], q0[3 * b + 1], q0[3 * b + 2]};
    const int c0[3] = {cell_of(q[0], inv_cell), cell_of(q[1], inv_cell), cell_of(q[2], inv_cell)};
    int count = 0;
    double tau = INFINITY, rs2_done = 0.0;
    double cut_scale = 0.0;       // histogram cut in force (warp_cut): drop d when cut_bin_of(d, cut_scale) > cut_bin
    int cut_bin = KNN_BINS;
    bool done = false;
    // overflow: first the cheap histogram cut, the full sort only if that could not make room
#define SVN_KNN_RELIEVE()                                                                         \
  if (count + 32 > KNN_CAP) {                                                                     \
    count = warp_cut(buf, count, K, &cut_scale, &cut_bin, s_hist[warp]);                          \
    if (count + 32 > KNN_CAP) count = warp_compact(buf, count, K, &tau);                          \
  }

    for (int r = 0; r <= RING_MAX && !done; r++) {
      const int side = 2 * r + 1, ncube = side * side * side;
      for (int base = 0; base < ncube; base += 32) {
        const int ci = base + lane;
        int st = 0, cn = 0;
        if (ci < ncube) {
          const int dz = ci / (side * side) - r, dy = (ci / side) % side - r, dx = ci % side - r;
          const int ch = max(abs(dx), max(abs(dy), abs(dz)));
          if (ch == r) {
            const int slot = hash_find(keys, mask, pack_voxel_key(c0[0] + dx, c0[1] + dy, c0[2] + dz));
            if (slot >= 0) { st = starts[slot]; cn = counts[slot]; }
          }
        }
        const int incl = warp_inclusive_scan(cn);
        const int total = __shfl_sync(0xffffffffu, incl, 31);
        s_start[warp][lane] = st;
        s_excl[warp][lane] = incl - cn;
        if (lane == 31) s_excl[warp][32] = total;
        __syncwarp();
        for (int t0 = 0; t0 < total; t0 += 32) {
          const int t = t0 + lane;
          bool keep = false;
          Ent e;
          if (t < total) {
            int lo = 0, hi = 31;  // largest l with excl[l] <= t
            while (lo < hi) {
              const int mid = (lo + hi + 1) >> 1;
              if (s_excl[warp][mid] <= t) lo = mid; else hi = mid - 1;
            }
            const int pos = s_start[warp][lo] + (t - s_excl[warp][lo]);
            e.d = dist2(q, sxyz + 3 * (size_t)pos);
            e.pos = pos;
            e.idx = sidx[pos];
            keep = e.d <= tau && (cut_bin >= KNN_BINS || cut_bin_of(e.d, cut_scale) <= cut_bin);
          }
          const unsigned m = __ballot_sync(0xffffffffu, keep);
          if (keep) buf[count + __popc(m & lt_mask)] = e;
          count += __popc(m);
          __syncwarp();
          SVN_KNN_RELIEVE()
        }
        __syncwarp();
      }
      // every unvisited point is farther than rs from q: the cube of radius r around q's cell is complete
      double rs = INFINITY;
#pragma unroll
      for (int a = 0; a < 3; a++) {
        rs = fmin(rs, q[a] - (double)(c0[a] - r) * cell);
        rs = fmin(rs, (double)(c0[a] + r + 1) * cell - q[a]);
      }
      rs = fmax(0.0, rs - 1e-6 * cell);
      const double rs2 = rs * rs;
      int nin = 0;
      for (int i = lane; i < count; i += 32) nin += (buf[i].d < rs2) ? 1 : 0;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) nin += __shfl_xor_sync(0xffffffffu, nin, o);
      if (nin >= K) { done = true; rs2_done = rs2; }
    }

    if (!done) {  // sparse neighbourhood (or N_t < K): exact brute-force sweep of the whole map
      if (lane == 0) atomicAdd(fallback_count, 1);
      count = 0;
      tau = INFINITY;
      cut_bin = KNN_BINS;
      for (int t0 = 0; t0 < n_t; t0 += 32) {
        const int t = t0 + lane;
        bool keep = false;
        Ent e;
        if (t < n_t) {
          e.d = dist2(q, sxyz + 3 * (size_t)t);
          e.pos = t;
          e.idx = sidx[t];
          keep = e.d <= tau && (cut_bin >= KNN_BINS || cut_bin_of(e.d, cut_scale) <= cut_bin);
        }
        const unsigned m = __ballot_sync(0xffffffffu, keep);
        if (keep) buf[count + __popc(m & lt_mask)] = e;
        count += __popc(m);
        __syncwarp();
        SVN_KNN_RELIEVE()
      }
    }
#undef SVN_KNN_RELIEVE
    if (done) {
      // >= K points lie inside rs2_done.  Cut the buffer down before sorting: 64-bin histogram of d over [0, rs2),
      // keep everything up to the bin in which the K-th smallest falls (exact superset of the K nearest).
      int *hist = s_hist[warp];
      hist[lane] = 0;
      hist[lane + 32] = 0;
      __syncwarp();
      const double scale = (double)KNN_BINS / rs2_done;
      for (int i = lane; i < count; i += 32) {
        const double d = buf[i].d;
        if (d < rs2_done) atomicAdd(&hist[min(KNN_BINS - 1, (int)(d * scale))], 1);
      }
      __syncwarp();
      // inclusive prefix over the 64 bins (2 per lane)
      const int h0 = hist[2 * lane], h1 = hist[2 * lane + 1];
      const int incl = warp_inclusive_scan(h0 + h1);
      const int before = incl - h0 - h1;
      int tbin = KNN_BINS;  // first bin whose inclusive count reaches K
      if (before < K && before + h0 >= K) tbin = 2 * lane;
      else if (before + h0 < K && incl >= K) tbin = 2 * lane + 1;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) tbin = min(tbin, __shfl_xor_sync(0xffffffffu, tbin, o));
      // in-place compaction (write index never passes the read index)
      int m_out = 0;
      for (int i0 = 0; i0 < count; i0 += 32) {
        const int i = i0 + lane;
        Ent e;
        bool keep = false;
        if (i < count) {
          e = buf[i];
          keep = (e.d < rs2_done) && (min(KNN_BINS - 1, (int)(e.d * scale)) <= tbin);
        }
        const unsigned m = __ballot_sync(0xffffffffu, keep);
        __syncwarp();
        if (keep) buf[m_out + __popc(m & lt_mask)] = e;
        m_out += __popc(m);
        __syncwarp();
      }
      count = m_out;
    }
    count = warp_compact(buf, count, K, &tau);

    // emit: relative fp32 coordinates m - q0 (w = lower bound of their norm: slots ascend in it, which k_gn's exact
    // early exit relies on) and the global map index; zero padding -> map point 0 (knn.cu:343)
    for (int k = lane; k < K; k += 32) {
      const double *m;
      int gi;
      if (k < count) { m = sxyz + 3 * (size_t)buf[k].pos; gi = buf[k].idx; }
      else { m = tgt; gi = 0; }
      const float cx = __double2float_rn(m[0] - q[0]), cy = __double2float_rn(m[1] - q[1]), cz = __double2float_rn(m[2] - q[2]);
      const double nrm = sqrt((double)cx * cx + (double)cy * cy + (double)cz * cz);
      const float w = (k < count) ? __double2float_rd(nrm * (1.0 - 1e-6)) : INFINITY;  // padded duplicates never need a visit
      cand[(size_t)b * K + k] = make_float4(cx, cy, cz, w);
      if (cand_idx) cand_idx[(size_t)b * K + k] = gi;  // parity taps only (debug_corr)
    }
    __syncwarp();
  }
}

// ---- host side -----------------------------------------------------------------------------
static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

size_t knn_smem_bytes() { return (size_t)KNN_WARPS * KNN_CAP * sizeof(Ent); }

int launch_cand_build(const CandBuildArgs &a, cudaStream_t st) {
  int launches = 0;
  const int T = 256;
  k_q0<<<cdiv(a.n_pad, T), T, 0, st>>>(a.src64, a.n_s, a.sc, a.q0, a.sp, a.n_pad); launches++;
  k_grid_clear<<<cdiv(a.table_size, T), T, 0, st>>>(a.keys, a.counts, a.fill, a.table_size, a.cursor); launches++;
  k_grid_count<<<cdiv(a.n_t, T), T, 0, st>>>(a.tgt64, a.n_t, 1.0 / a.cell, a.keys, a.counts, a.pt_slot, (unsigned)(a.table_size - 1)); launches++;
  k_grid_alloc<<<cdiv(a.table_size, T), T, 0, st>>>(a.counts, a.starts, a.table_size, a.cursor); launches++;
  k_grid_scatter<<<cdiv(a.n_t, T), T, 0, st>>>(a.tgt64, a.n_t, a.pt_slot, a.starts, a.fill, a.sxyz, a.sidx); launches++;
  // per scan, not once per process: the attribute is per device, and a process may hold handles on several devices
  if (knn_smem_bytes() > 48 * 1024) cudaFuncSetAttribute(k_knn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)knn_smem_bytes());
  int grid = cdiv(a.row_hi - a.row_lo, KNN_WARPS);
  const int max_grid = a.sm_count * 12;
  if (grid > max_grid) grid = max_grid;
  if (grid < 1) grid = 1;
  k_knn<<<grid, KNN_WARPS * 32, knn_smem_bytes(), st>>>(a.q0, a.row_lo, a.row_hi, a.tgt64, a.n_t, a.sxyz, a.sidx, a.keys, a.starts, a.counts,
                                                         (unsigned)(a.table_size - 1), a.cell, a.K, a.cand, a.cand_idx, a.fallback_count);
  launches++;
  return launches;
}

}  // namespace svn
