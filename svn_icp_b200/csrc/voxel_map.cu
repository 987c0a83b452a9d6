// voxel_map.cu -- device-resident local map: the reference's svnicp::VoxelHashMap (svn-icp/include/core/VoxelHashMap.h:28-72,
// src/core/VoxelHashMap.cpp:22-101) kept in HBM, so that the per-scan target cloud handed to add_cloud never leaves the GPU
// (the reference rebuilds it on the host and re-uploads it every scan, OdometryPipeline.cpp:577-581).  SURVEY.md 8(f) row 1.
//
// Semantics kept (VoxelHashMap.cpp):
//   AddPointCloud :22-43   p_map = float(T * p) (pcl::transformPointCloud with a double matrix); voxel index =
//                          (p_map / float(voxel_size)).cast<int>() -- truncation toward zero; a voxel keeps its FIRST
//                          max_pointscount points in arrival order; then RemoveFarPointCloud(translation)
//   GetMap()      :45-51   all points;  GetMap(pose, r) :53-63: voxels whose FIRST point is closer than r to the position
//   RemoveFar     :93-101  voxels whose first point is farther than max_range are dropped
// "Arrival order" is made deterministic on the GPU by ranking the points of one AddPointCloud batch by their index in the
// cloud (what the reference's sequential loop does): pass 1 links every point into its voxel's list and elects the lowest
// index as the voxel's walker; pass 2 lets the walker keep the (cap - count) lowest indices, ascending.
// The table is the voxel hash of voxel_hash.cuh (open addressing over packed 3x21-bit voxel indices); RemoveFar rebuilds into
// the twin table (no tombstones).  Point output order of GetMap is slot order: arbitrary like the reference's robin_map iteration.
//
// svnicp_map_evaluate (DESIGN.md section 10b) scores a scan at caller-given poses against the table itself: an exact
// nearest-map-point search per (source point, pose) by read-only probes of the same hash (k_map_eval), then the fixed-order
// reduction of svnicp_evaluate (k_eval_fin, eval_kernels.cu).
//
// svnicp_map_search (DESIGN.md section 10d) ranks a regular grid of poses by the same inlier count: an existence test per
// (source point, pose) with an early exit (k_map_search_count), integer counts per pose and a deterministic running top k
// (k_map_search_topk); the winners' statistics come from svnicp_map_evaluate itself.
//
// svnicp_map_refine (DESIGN.md section 10f) runs Gauss-Newton steps of many poses against the table: k_map_refine_eval (the
// sums of k_map_eval, each search seeded with the previous iteration's map point), k_eval_fin, k_map_refine_step (solve and
// update), the whole loop enqueued without a host round trip; the final statistics come from svnicp_map_evaluate itself.
//
// svnicp_map_export / svnicp_map_import (DESIGN.md section 10c) save and restore the content in canonical form -- voxels in
// ascending (vx, vy, vz), each voxel's points in stored order -- independent of the slot layout: a radix sort of the live keys
// on the way out, a rebuild into the twin table with full validation on the way in.
#include <cuda_runtime.h>
#include <limits.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/svnicp_b200.h"
#include "block_scan.cuh"
#include "kernels.h"
#include "voxel_hash.cuh"

namespace {

using svn::EMPTY_KEY;
using svn::SCAN_BLOCK;
using svn::block_exclusive_scan;

constexpr int MAX_CAP = 32;

struct MapTable {
  unsigned long long *keys;  // [slots]
  int *count;                // [slots]
  float *pts;                // [slots][cap][3]
};

struct MapDev {
  MapTable tab;
  int *head, *walker;        // [slots] per-batch list head / elected walker (restored to -1 / INT_MAX after every batch)
  long long *counters;       // [0] voxels, [1] points, [2] far voxels (scratch), [3] dropped (table full)
  int slots_mask, cap;
  float voxel_size_f;
};

// The voxel a stored point belongs to (VoxelHashMap.cpp:30): (int)(p / float(voxel_size)) per axis -- truncation toward zero,
// so (-v, v) is voxel 0, and NaN converts to 0 -- packed.  k_map_insert_link files points with it and svnicp_map_import checks
// membership with it, so the two cannot drift.
__device__ __forceinline__ unsigned long long voxel_key(const float q[3], float voxel_size_f) {
  return svn::pack_voxel_key((int)(q[0] / voxel_size_f), (int)(q[1] / voxel_size_f), (int)(q[2] / voxel_size_f));
}

// pass 1: transform (VoxelHashMap.cpp:23-26), voxel index (:30), slot lookup, link into the voxel's batch list
template <typename T>
__global__ void k_map_insert_link(MapDev m, const T *xyz, int n, const double *Rt /*R[9], t[3]*/, float *wxyz, int *pt_slot, int *next) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double p[3] = {(double)xyz[3 * (size_t)i], (double)xyz[3 * (size_t)i + 1], (double)xyz[3 * (size_t)i + 2]};
  float q[3];
#pragma unroll
  for (int r = 0; r < 3; r++) q[r] = (float)(Rt[3 * r] * p[0] + Rt[3 * r + 1] * p[1] + Rt[3 * r + 2] * p[2] + Rt[9 + r]);
#pragma unroll
  for (int r = 0; r < 3; r++) wxyz[3 * (size_t)i + r] = q[r];
  bool created;
  const int slot = svn::hash_insert(m.tab.keys, (unsigned)m.slots_mask, voxel_key(q, m.voxel_size_f), &created);
  pt_slot[i] = slot;
  if (slot < 0) { atomicAdd((unsigned long long *)&m.counters[3], 1ull); return; }
  if (created) atomicAdd((unsigned long long *)&m.counters[0], 1ull);
  if (m.tab.count[slot] >= m.cap) { pt_slot[i] = -2; return; }  // voxel already full before this cloud (:33)
  next[i] = atomicExch(&m.head[slot], i);
  atomicMin(&m.walker[slot], i);
}

// pass 2: the lowest-index point of each touched voxel appends the (cap - count) lowest indices in ascending order
__global__ void k_map_insert_place(MapDev m, const float *wxyz, const int *pt_slot, const int *next, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int slot = pt_slot[i];
  if (slot < 0 || m.walker[slot] != i) return;
  const int have = m.tab.count[slot];
  const int need = m.cap - have;
  int best[MAX_CAP];
  int nb = 0;
  for (int j = m.head[slot]; j >= 0; j = next[j]) {
    if (nb < need) {
      int k = nb++;
      while (k > 0 && best[k - 1] > j) { best[k] = best[k - 1]; k--; }
      best[k] = j;
    } else if (j < best[nb - 1]) {
      int k = nb - 1;
      while (k > 0 && best[k - 1] > j) { best[k] = best[k - 1]; k--; }
      best[k] = j;
    }
  }
  float *dst = m.tab.pts + ((size_t)slot * m.cap + have) * 3;
  for (int k = 0; k < nb; k++)
    for (int c = 0; c < 3; c++) dst[3 * k + c] = wxyz[3 * (size_t)best[k] + c];
  m.tab.count[slot] = have + nb;
  m.head[slot] = -1;
  m.walker[slot] = INT_MAX;
  atomicAdd((unsigned long long *)&m.counters[1], (unsigned long long)nb);
}

__device__ __forceinline__ bool front_within(const MapTable &t, int cap, int slot, const double *pos, double r2, bool strict_less) {
  const float *f = t.pts + (size_t)slot * cap * 3;
  const double dx = (double)f[0] - pos[0], dy = (double)f[1] - pos[1], dz = (double)f[2] - pos[2];
  const double d2 = dx * dx + dy * dy + dz * dz;
  return strict_less ? (d2 < r2) : !(d2 > r2);
}

// RemoveFarPointCloud (:93-101): count the voxels to drop
__global__ void k_map_count_far(MapDev m, const double *pos, double r2) {
  const size_t s = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s > (size_t)m.slots_mask) return;
  if (m.tab.keys[s] == EMPTY_KEY || m.tab.count[s] == 0) return;
  if (!front_within(m.tab, m.cap, s, pos, r2, false)) atomicAdd((unsigned long long *)&m.counters[2], 1ull);
}

// ... and rebuild the survivors into the twin table (one warp per old slot: coalesced copy of the voxel's points)
__global__ void k_map_rebuild(MapDev old, MapDev neu, const double *pos, double r2) {
  const size_t w = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;  // 64-bit: slots * 32 exceeds 2^32 beyond 2^27 slots
  const int lane = threadIdx.x & 31;
  if (w > (size_t)old.slots_mask) return;
  const unsigned long long key = old.tab.keys[w];
  const int cnt = old.tab.count[w];
  if (key == EMPTY_KEY || cnt == 0) return;
  if (!front_within(old.tab, old.cap, w, pos, r2, false)) return;
  int slot = 0;
  if (lane == 0) {
    bool created;
    slot = svn::hash_insert(neu.tab.keys, (unsigned)neu.slots_mask, key, &created);
    if (slot >= 0) {
      neu.tab.count[slot] = cnt;
      atomicAdd((unsigned long long *)&neu.counters[0], 1ull);
      atomicAdd((unsigned long long *)&neu.counters[1], (unsigned long long)cnt);
    }
  }
  slot = __shfl_sync(0xffffffffu, slot, 0);
  if (slot < 0) return;
  const float *src = old.tab.pts + (size_t)w * old.cap * 3;
  float *dst = neu.tab.pts + (size_t)slot * neu.cap * 3;
  for (int e = lane; e < cnt * 3; e += 32) dst[e] = src[e];
}

// GetMap (:45-63): three-step deterministic compaction in slot order; output fp64 xyz ready for add_cloud
__device__ __forceinline__ int slot_emit_count(const MapDev &m, int s, const double *pos, double r2, int all) {
  if (s > m.slots_mask || m.tab.keys[s] == EMPTY_KEY) return 0;
  const int c = m.tab.count[s];
  if (c == 0) return 0;
  return (all || front_within(m.tab, m.cap, s, pos, r2, true)) ? c : 0;
}

__global__ void __launch_bounds__(SCAN_BLOCK) k_getmap_count(MapDev m, const double *pos, double r2, int all, int *block_sums) {
  svn::block_sum_int(slot_emit_count(m, blockIdx.x * SCAN_BLOCK + threadIdx.x, pos, r2, all), &block_sums[blockIdx.x]);
}

__global__ void __launch_bounds__(SCAN_BLOCK) k_getmap_emit(MapDev m, const double *pos, double r2, int all, const int *block_offs, double *out) {
  const int s = blockIdx.x * SCAN_BLOCK + threadIdx.x;
  const int c = slot_emit_count(m, s, pos, r2, all);
  const int off = block_offs[blockIdx.x] + block_exclusive_scan<int>(c, nullptr);
  if (c == 0) return;
  const float *src = m.tab.pts + (size_t)s * m.cap * 3;
  double *dst = out + (size_t)off * 3;
  for (int e = 0; e < c * 3; e++) dst[e] = (double)src[e];
}

__global__ void k_fill_i32(int *p, int v, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

// ---- svnicp_map_export / svnicp_map_import (DESIGN.md section 10c) ----------------------------------------------------------
// Export: live slots -> (canonical key, slot) pairs (count -> single-block scan -> emit, as GetMap) -> stable LSD radix sort
// by canonical key -> int64 point offsets in that order -> one warp per voxel gathers index, count and points.
// Import: int64 point offsets of the snapshot -> one warp per voxel builds into the twin table and checks it -> duplicates.
constexpr int RADIX_BITS = 8;
constexpr int RADIX_DIGITS = 1 << RADIX_BITS;
constexpr int RADIX_THREADS = 256;  // == RADIX_DIGITS: one thread per digit in the histogram and offset steps
constexpr int RADIX_IPT = 16;       // keys per thread
constexpr int RADIX_TILE = RADIX_THREADS * RADIX_IPT;
constexpr int CANON_BITS = 63;      // three 21-bit fields
static_assert(((CANON_BITS + RADIX_BITS - 1) / RADIX_BITS) % 2 == 0, "an even pass count leaves the sorted pairs in buffer 0");
constexpr unsigned long long SNAP_NO_ERROR = ~0ull;
enum { SNAP_BAD_COUNT = 1, SNAP_BAD_INDEX = 2, SNAP_DUPLICATE = 3, SNAP_NOT_MEMBER = 4 };  // the reason in the low 3 bits

// The packed key with the x and z fields swapped: each field holds index + 2^20, so ascending canonical keys are ascending
// lexicographic (vx, vy, vz).  The swap is its own inverse.
__device__ __forceinline__ unsigned long long canon_key(unsigned long long k) {
  const unsigned long long F = 0x1FFFFFull;
  return ((k & F) << 42) | (k & (F << 21)) | ((k >> 42) & F);
}

__device__ __forceinline__ bool slot_live(const MapDev &m, int s) {
  return s <= m.slots_mask && m.tab.keys[s] != EMPTY_KEY && m.tab.count[s] > 0;
}

__global__ void __launch_bounds__(SCAN_BLOCK) k_snap_count(MapDev m, int *block_sums) {
  const int c = __syncthreads_count(slot_live(m, blockIdx.x * SCAN_BLOCK + threadIdx.x));
  if (threadIdx.x == 0) block_sums[blockIdx.x] = c;
}

// (canonical key, slot) of every live slot, in slot order; at most V are written
__global__ void __launch_bounds__(SCAN_BLOCK) k_snap_emit(MapDev m, const int *block_offs, long long V, unsigned long long *keys, int *slots) {
  const int s = blockIdx.x * SCAN_BLOCK + threadIdx.x;
  const int live = slot_live(m, s) ? 1 : 0;
  const int off = block_offs[blockIdx.x] + block_exclusive_scan<int>(live, nullptr);
  if (!live || off >= V) return;
  keys[off] = canon_key(m.tab.keys[s]);
  slots[off] = s;
}

// Radix pass, step 1: digit histogram of each tile of RADIX_TILE keys, digit-major ([digit][tile]) so that one exclusive scan
// gives every (digit, tile) its output offset.
__global__ void __launch_bounds__(RADIX_THREADS) k_radix_hist(const unsigned long long *keys, int n, int shift, int n_tiles, int *hist) {
  __shared__ int s_h[RADIX_DIGITS];
  s_h[threadIdx.x] = 0;
  __syncthreads();
  const int base = blockIdx.x * RADIX_TILE;
  for (int k = threadIdx.x; k < RADIX_TILE && base + k < n; k += RADIX_THREADS)
    atomicAdd(&s_h[(keys[base + k] >> shift) & (RADIX_DIGITS - 1)], 1);
  __syncthreads();
  hist[(size_t)threadIdx.x * n_tiles + blockIdx.x] = s_h[threadIdx.x];
}

// Radix pass, step 3: stable scatter.  Warp w of a tile owns keys [w * 32 * IPT, (w + 1) * 32 * IPT) of it, 32 consecutive keys
// per round; a key's rank among the equal digits before it comes from __match_any_sync within the round plus the warp's running
// per-digit count, and the lower warps' counts are added once the tile is counted.
__global__ void __launch_bounds__(RADIX_THREADS) k_radix_scatter(const unsigned long long *keys_in, const int *vals_in, unsigned long long *keys_out,
                                                                int *vals_out, int n, int shift, int n_tiles, const int *offs) {
  __shared__ int s_cnt[RADIX_THREADS / 32][RADIX_DIGITS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int d = lane; d < RADIX_DIGITS; d += 32) s_cnt[warp][d] = 0;
  __syncwarp();
  const int base = blockIdx.x * RADIX_TILE + warp * 32 * RADIX_IPT + lane;
  const unsigned below = (1u << lane) - 1u;
  int dig[RADIX_IPT], rank[RADIX_IPT];
#pragma unroll
  for (int r = 0; r < RADIX_IPT; r++) {
    const int i = base + 32 * r;
    const int d = i < n ? (int)((keys_in[i] >> shift) & (RADIX_DIGITS - 1)) : RADIX_DIGITS;  // RADIX_DIGITS: no key
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    rank[r] = s_cnt[warp][d & (RADIX_DIGITS - 1)] + __popc(peers & below);
    __syncwarp();
    if (d < RADIX_DIGITS && (peers & below) == 0) s_cnt[warp][d] += __popc(peers);
    __syncwarp();
    dig[r] = d;
  }
  __syncthreads();
  {
    const int d = threadIdx.x;
    int run = offs[(size_t)d * n_tiles + blockIdx.x];
    for (int w = 0; w < RADIX_THREADS / 32; w++) {
      const int c = s_cnt[w][d];
      s_cnt[w][d] = run;
      run += c;
    }
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < RADIX_IPT; r++) {
    if (dig[r] == RADIX_DIGITS) continue;
    const int i = base + 32 * r, dst = s_cnt[warp][dig[r]] + rank[r];
    keys_out[dst] = keys_in[i];
    vals_out[dst] = vals_in[i];
  }
}

// Point count of voxel i: the table's through the sorted slots (export), or the snapshot's, taken as 0 outside [1, cap] so that
// the offsets stay in bounds (import; k_map_import reports such a count).
__device__ __forceinline__ int snap_count(const int32_t *counts, const int *slots, const int *tab_count, int cap, long long i, long long V) {
  if (i >= V) return 0;
  if (slots) return tab_count[slots[i]];
  const int c = counts[i];
  return c >= 1 && c <= cap ? c : 0;
}

__global__ void __launch_bounds__(SCAN_BLOCK) k_snap_pts_count(const int32_t *counts, const int *slots, const int *tab_count, int cap, long long V,
                                                             long long *block_sums) {
  const long long c = snap_count(counts, slots, tab_count, cap, (long long)blockIdx.x * SCAN_BLOCK + threadIdx.x, V);
  long long tot;
  block_exclusive_scan<long long>(c, &tot);
  if (threadIdx.x == 0) block_sums[blockIdx.x] = tot;
}

__global__ void __launch_bounds__(SCAN_BLOCK) k_snap_pts_offsets(const int32_t *counts, const int *slots, const int *tab_count, int cap, long long V,
                                                               const long long *block_offs, long long *off) {
  const long long i = (long long)blockIdx.x * SCAN_BLOCK + threadIdx.x;
  const long long c = snap_count(counts, slots, tab_count, cap, i, V);
  const long long o = block_offs[blockIdx.x] + block_exclusive_scan<long long>(c, nullptr);
  if (i < V) off[i] = o;
}

// one warp per sorted voxel: index, count, and the points in stored order (the coalesced copy of k_map_rebuild)
__global__ void k_snap_gather(MapTable t, int cap, const unsigned long long *keys, const int *slots, const long long *off, long long V, long long N,
                              int32_t *voxels, int32_t *counts, float *xyz) {
  const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (i >= V) return;
  const int s = slots[i], c = t.count[s];
  if (lane < 3) voxels[3 * i + lane] = (int)((keys[i] >> (42 - 21 * lane)) & 0x1FFFFFull) - (1 << 20);
  if (lane == 3) counts[i] = c;
  const long long o = off[i];
  if (o + c > N) return;  // the table disagrees with the counters: reported by the caller, nothing written out of bounds
  const float *src = t.pts + (size_t)s * cap * 3;
  float *dst = xyz + o * 3;
  for (int e = lane; e < 3 * c; e += 32) dst[e] = src[e];
}

__device__ __forceinline__ void snap_flag(unsigned long long *err, long long i, int reason) {
  atomicMin(err, ((unsigned long long)i << 3) | (unsigned long long)reason);
}

// One warp per snapshot voxel into the (cleared) twin table: hash_insert, count, points; every point's membership is
// checked with voxel_key.  words: [0] lowest (voxel << 3 | reason) of the count and index errors, [2] voxels refused by a full
// table, [3] lowest of the duplicate and membership errors (meaningful only when the counts are valid and sum to N, since the
// point offsets come from them).  Each voxel's slot goes to slot_of (-1 when not inserted) and the lowest voxel index per slot
// to walker, for k_map_import_dups.
__global__ void k_map_import(MapDev neu, const int32_t *voxels, const int32_t *counts, const float *xyz, long long V, long long N,
                             const long long *off, int *slot_of, unsigned long long *words) {
  const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (i >= V) return;
  const int vx = voxels[3 * i], vy = voxels[3 * i + 1], vz = voxels[3 * i + 2], c = counts[i];
  const int lim = 1 << 20;
  const bool count_ok = c >= 1 && c <= neu.cap;
  const bool index_ok = vx >= -lim && vx < lim && vy >= -lim && vy < lim && vz >= -lim && vz < lim;
  const unsigned long long key = svn::pack_voxel_key(vx, vy, vz);
  int slot = -1;
  if (lane == 0) {
    if (!count_ok) snap_flag(words, i, SNAP_BAD_COUNT);
    else if (!index_ok) snap_flag(words, i, SNAP_BAD_INDEX);
    else {
      bool created;
      slot = svn::hash_insert(neu.tab.keys, (unsigned)neu.slots_mask, key, &created);
      if (slot < 0) atomicAdd(&words[2], 1ull);
      else {
        atomicMin(&neu.walker[slot], (int)i);
        neu.tab.count[slot] = c;
      }
    }
    slot_of[i] = slot;
  }
  slot = __shfl_sync(0xffffffffu, slot, 0);
  if (!count_ok || !index_ok) return;
  const long long o = off[i];
  if (o + c > N) return;  // the counts sum past n_points: reported from the sum
  const float *src = xyz + o * 3;
  for (int k = lane; k < c; k += 32) {
    const float q[3] = {src[3 * k], src[3 * k + 1], src[3 * k + 2]};
    if (voxel_key(q, neu.voxel_size_f) != key) snap_flag(words + 3, i, SNAP_NOT_MEMBER);
  }
  if (slot < 0) return;
  float *dst = neu.tab.pts + (size_t)slot * neu.cap * 3;
  for (int e = lane; e < 3 * c; e += 32) dst[e] = src[e];
}

// A voxel whose slot was claimed by a lower index repeats that voxel; the lowest index of each slot is not a duplicate.
__global__ void k_map_import_dups(const int *walker, const int *slot_of, long long V, unsigned long long *words) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= V) return;
  const int s = slot_of[i];
  if (s >= 0 && walker[s] != (int)i) snap_flag(words + 3, i, SNAP_DUPLICATE);
}

__global__ void k_map_import_reset(int *walker, const int *slot_of, long long V) {  // walker back to INT_MAX, as after a batch
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= V) return;
  const int s = slot_of[i];
  if (s >= 0) walker[s] = INT_MAX;
}

// ---- svnicp_map_evaluate ----------------------------------------------------------------------------------------------------
constexpr int MEV_THREADS = 128;     // 4 warps; a warp holds 32 consecutive source points of one pose (ring order: shared voxels)
constexpr int MEV_CTAS_PER_SM = 8;   // partial slots per SM (the grid-stride over the source points depends on n and SMs only)
constexpr int MEV_MAX_REACH = 4;     // ceil(sqrt(max_dist) / voxel_size) allowed: at most 9^3 voxels per query
constexpr int MEV_SPAN = 2 * MEV_MAX_REACH + 4;  // voxels per axis of a search box beyond which a query sweeps the whole table
constexpr double MEV_MARGIN = 1.0 + 1e-12;       // search radii exceed sqrt(d^2) by far more than dist2's rounding (< 4 ulp)

// Read-only probe: the slot holding key, or -1 when the voxel is absent or holds no point.  There are no tombstones (far voxels
// leave by a rebuild into the twin table), so the walk may stop at the first empty slot.
__device__ __forceinline__ int map_find(const MapTable &t, int slots_mask, unsigned long long key) {
  const int slot = svn::hash_find(t.keys, (unsigned)slots_mask, key);
  return slot < 0 || __ldg(t.count + slot) > 0 ? slot : -1;
}

// One pose x = [t ; omega] relative to T0 = (R0, t0): R~ = R0 Exp(omega), t~ = t0 + R0 t -> o [12] (R~ row-major, t~), and
// R_p = Exp(omega) -> R [9].  x = 0 gives R_p = I exactly, and (R0, t0) is stored as given, so the query of a pose x = 0 is
// q0 bit for bit (the products would turn a -0 entry of R0 into +0).  The one place this is computed: svnicp_map_evaluate
// (k_map_eval_prep) and svnicp_map_search (k_map_search_prep) cannot drift apart.
__device__ __forceinline__ void map_pose(const double *x, const svn::ScanConst &sc, double *o, double R[9]) {
  svn::so3_exp(x + 3, R, nullptr);
  const bool zero = x[0] == 0.0 && x[1] == 0.0 && x[2] == 0.0 && x[3] == 0.0 && x[4] == 0.0 && x[5] == 0.0;
#pragma unroll
  for (int r = 0; r < 3; r++) {
#pragma unroll
    for (int c = 0; c < 3; c++)
      o[3 * r + c] = zero ? sc.R0[3 * r + c] : sc.R0[3 * r] * R[c] + sc.R0[3 * r + 1] * R[3 + c] + sc.R0[3 * r + 2] * R[6 + c];
    o[9 + r] = zero ? sc.t0[r] : sc.t0[r] + (sc.R0[3 * r] * x[0] + sc.R0[3 * r + 1] * x[1] + sc.R0[3 * r + 2] * x[2]);
  }
}

// Per pose of a block: Rt [MB][12] and Rp [MB][9] (for gn_assemble) by map_pose
__global__ void k_map_eval_prep(const double *x6 /*[MB][6]*/, int MB, svn::ScanConst sc, double *Rt, double *Rp) {
  const int p = threadIdx.x;
  if (p >= MB) return;
  double R[9];
  map_pose(x6 + 6 * p, sc, Rt + 12 * p, R);
#pragma unroll
  for (int i = 0; i < 9; i++) Rp[9 * p + i] = R[i];
}

// Voxel range [lo, hi] of one axis that holds every stored point p with |p_a - q_a| <= rad.  A point was filed under
// trunc(fl32(p_a / v)) (k_map_insert_link, VoxelHashMap.cpp:30).  With lo_f = fl32 of (q_a - rad) rounded down, both roundings
// downward, and hi_f likewise upward, lo_f <= p_a <= hi_f, because p_a is itself a float.  fp32 division by v > 0 (round to
// nearest) is monotone and so is truncation toward zero, hence trunc(fl32(lo_f / v)) <= voxel_a(p) <= trunc(fl32(hi_f / v)).
// Truncation files (-v, v) under voxel 0, which is twice as wide as the others; monotonicity holds across it, so a box that
// straddles zero contains voxel 0 and none of its points are skipped.  Saturating conversions (|q| beyond 2^31 v) stay monotone.
__device__ __forceinline__ void box_axis(double q, double rad, float v, int &lo, int &hi) {
  lo = (int)__fdiv_rn(__double2float_rd(__dsub_rd(q, rad)), v);
  hi = (int)__fdiv_rn(__double2float_ru(__dadd_ru(q, rad)), v);
}

struct NearestState {
  double q[3];
  double bd;  // best d^2 so far (max_dist until a point qualifies: d^2 < max_dist)
  float bx, by, bz;
  bool found;
};

// every point of one voxel: smaller d^2 wins, an exact tie goes to the lexicographically smaller (x, y, z) -- data only
__device__ __forceinline__ void visit_slot(const MapTable &t, int cap, int slot, NearestState &s) {
  const int c = __ldg(t.count + slot);
  const float *p = t.pts + (size_t)slot * cap * 3;
  for (int k = 0; k < c; k++) {
    const float px = __ldg(p + 3 * k), py = __ldg(p + 3 * k + 1), pz = __ldg(p + 3 * k + 2);
    const double mp[3] = {(double)px, (double)py, (double)pz};
    const double d = svn::dist2(s.q, mp);
    const bool lex = px < s.bx || (px == s.bx && (py < s.by || (py == s.by && pz < s.bz)));
    if (d < s.bd || (s.found && d == s.bd && lex)) { s.bd = d; s.bx = px; s.by = py; s.bz = pz; s.found = true; }
  }
}

// Exact nearest stored point of a finite query within d^2 < max_dist (the same choice as a brute-force sweep over GetMap()).
// The query's own voxel first; then the box shrinks to the best distance found and every other voxel of it is visited.
__device__ __forceinline__ void map_nearest(const MapDev &m, double r, NearestState &s) {
  const float v = m.voxel_size_f;
  int lo[3], hi[3];
  bool wide = false;
#pragma unroll
  for (int a = 0; a < 3; a++) {
    box_axis(s.q[a], r, v, lo[a], hi[a]);
    wide |= (long long)hi[a] - lo[a] >= MEV_SPAN;
  }
  if (wide) {  // float spacing of q coarser than the voxels (|q| >~ 2^24 v): sweep the table, still exact
    for (int slot = 0; slot <= m.slots_mask; slot++)
      if (__ldg(m.tab.keys + slot) != EMPTY_KEY) visit_slot(m.tab, m.cap, slot, s);
    return;
  }
  int own[3];
#pragma unroll
  for (int a = 0; a < 3; a++) own[a] = (int)__fdiv_rn(__double2float_rn(s.q[a]), v);
  int slot = map_find(m.tab, m.slots_mask, svn::pack_voxel_key(own[0], own[1], own[2]));
  if (slot >= 0) visit_slot(m.tab, m.cap, slot, s);
  if (s.found) {
    const double rb = fmin(r, sqrt(s.bd) * MEV_MARGIN);
#pragma unroll
    for (int a = 0; a < 3; a++) box_axis(s.q[a], rb, v, lo[a], hi[a]);
  }
  for (int z = lo[2]; z <= hi[2]; z++)
    for (int y = lo[1]; y <= hi[1]; y++)
      for (int x = lo[0]; x <= hi[0]; x++) {
        if (x == own[0] && y == own[1] && z == own[2]) continue;
        slot = map_find(m.tab, m.slots_mask, svn::pack_voxel_key(x, y, z));
        if (slot >= 0) visit_slot(m.tab, m.cap, slot, s);
      }
}

// One thread per (source point, pose): grid.x = partial slots (grid-stride over the points), grid.y = the poses of the block.
// Sums per pose, as k_eval_corr: the 16 Gauss-Newton sums in the world-oriented frame (s' = R0 s, e = q - m, R~ s), the inlier
// count and the inlier sum of d^2; fp64 per thread, a fixed butterfly per warp, the warps in ascending order per CTA.
// Queries without a correspondence (no point with d^2 < max_dist, or a non-finite query) add only +1 to W (Q2).
// Launch bounds: with the system 128 registers (4 CTAs per SM), without it 64 (8 CTAs); below that ptxas spills.
template <typename T, bool SYS>
__global__ void __launch_bounds__(MEV_THREADS, SYS ? 4 : 8) k_map_eval(MapDev m, const T *__restrict__ src, int n, const double *__restrict__ Rt,
                                                          svn::ScanConst sc, double max_dist, double r, double *part,
                                                          uint8_t *mask, float *nearest) {
  using svn::EV_NS;
  __shared__ double s_w[MEV_THREADS / 32][EV_NS];
  const int p = blockIdx.y, MB = gridDim.y;
  const double *P = Rt + 12 * p;
  double Rtl[9], ttl[3];
#pragma unroll
  for (int i = 0; i < 9; i++) Rtl[i] = P[i];
#pragma unroll
  for (int i = 0; i < 3; i++) ttl[i] = P[9 + i];
  const double D = max_dist;
  double acc[EV_NS];
#pragma unroll
  for (int j = 0; j < EV_NS; j++) acc[j] = 0.0;
  for (int i = blockIdx.x * MEV_THREADS + threadIdx.x; i < n; i += gridDim.x * MEV_THREADS) {
    const double x = (double)src[3 * (size_t)i], y = (double)src[3 * (size_t)i + 1], z = (double)src[3 * (size_t)i + 2];
    NearestState s;
#pragma unroll
    for (int a = 0; a < 3; a++) s.q[a] = svn::affine_row_fma(Rtl, ttl, a, x, y, z);
    s.bd = max_dist;
    s.bx = s.by = s.bz = 0.f;
    s.found = false;
    if (isfinite(s.q[0]) && isfinite(s.q[1]) && isfinite(s.q[2])) map_nearest(m, r, s);
    if (mask) mask[(size_t)p * n + i] = s.found ? 1 : 0;
    if (nearest) {
      float *o = nearest + ((size_t)p * n + i) * 3;
      o[0] = s.bx; o[1] = s.by; o[2] = s.bz;
    }
    if (!s.found) {
      if (SYS) acc[0] += 1.0;  // masked: +1 on the translation block (Q2); nothing else, so a NaN never reaches the sums
      continue;
    }
    acc[16] += 1.0;
    acc[17] += s.bd;
    if (SYS) {
      double sp[3], w[3];
#pragma unroll
      for (int a = 0; a < 3; a++) {
        sp[a] = fma(sc.R0[3 * a], x, fma(sc.R0[3 * a + 1], y, sc.R0[3 * a + 2] * z));  // s' = R0 s
        w[a] = fma(Rtl[3 * a], x, fma(Rtl[3 * a + 1], y, Rtl[3 * a + 2] * z));        // R~ s
      }
      const double e[3] = {s.q[0] - (double)s.bx, s.q[1] - (double)s.by, s.q[2] - (double)s.bz};
      const double wq = D / (D + 3.0 * sqrt(s.bd));
      const double rho = wq * wq;  // (D / (D + 3 |e|))^2, SVNICP.cpp:120-122
      acc[0] += rho;
      const double g[3] = {rho * sp[0], rho * sp[1], rho * sp[2]};
      acc[1] += g[0]; acc[2] += g[1]; acc[3] += g[2];
      acc[4] += g[0] * sp[0]; acc[5] += g[0] * sp[1]; acc[6] += g[0] * sp[2];
      acc[7] += g[1] * sp[1]; acc[8] += g[1] * sp[2]; acc[9] += g[2] * sp[2];
      const double f[3] = {rho * e[0], rho * e[1], rho * e[2]};
      acc[10] += f[0]; acc[11] += f[1]; acc[12] += f[2];
      acc[13] += w[1] * f[2] - w[2] * f[1];
      acc[14] += w[2] * f[0] - w[0] * f[2];
      acc[15] += w[0] * f[1] - w[1] * f[0];
    }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int j = 0; j < EV_NS; j++) {
    const double v = svn::warp_sum(acc[j]);
    if (lane == 0) s_w[warp][j] = v;
  }
  __syncthreads();
  if (threadIdx.x < EV_NS) {
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < MEV_THREADS / 32; w++) t += s_w[w][threadIdx.x];
    part[((size_t)blockIdx.x * MB + p) * EV_NS + threadIdx.x] = t;
  }
}

// ---- svnicp_map_refine (DESIGN.md section 10f) --------------------------------------------------------------------------------
// Per pose block and iteration: k_map_refine_eval (k_map_eval<T, true>'s sums of the active poses) -> k_eval_fin (the fixed-order
// sum and gn_assemble of svnicp_map_evaluate, unchanged) -> k_map_refine_step (solve, update, stop rule, next R~ t~).
// Seeding (SVN_RF_SEED, default on; the A/B measurement is in DESIGN.md section 10f): each (pose, point) keeps the map point it
// chose last iteration and starts the next search from it.
#ifndef SVN_RF_SEED
#define SVN_RF_SEED 1
#endif
constexpr bool RF_SEED = SVN_RF_SEED != 0;
constexpr int RF_MAX_BLOCK = 1024;              // poses per block at most (k_map_eval_prep runs one thread per pose)
constexpr size_t RF_BLOCK_BYTES = 64ull << 20;  // partials + seeds of one pose block, at most (one pose exceeds it only beyond ~5 M points)

// k_map_refine_eval's share of one source point in the per-pose sums, once its nearest point s is settled: the arithmetic of
// k_map_eval's loop body, which keeps its own copy so that its SASS stays as measured in DESIGN.md section 10b (a shared helper
// changes its instruction schedule).
// Queries without a correspondence (no point with d^2 < max_dist, or a non-finite query) add only +1 to W (Q2).
template <bool SYS>
__device__ __forceinline__ void map_eval_accum(const NearestState &s, double x, double y, double z, const double Rtl[9],
                                               const svn::ScanConst &sc, double D, double (&acc)[svn::EV_NS]) {
  if (!s.found) {
    if (SYS) acc[0] += 1.0;  // masked: +1 on the translation block (Q2); nothing else, so a NaN never reaches the sums
    return;
  }
  acc[16] += 1.0;
  acc[17] += s.bd;
  if (SYS) {
    double sp[3], w[3];
#pragma unroll
    for (int a = 0; a < 3; a++) {
      sp[a] = fma(sc.R0[3 * a], x, fma(sc.R0[3 * a + 1], y, sc.R0[3 * a + 2] * z));  // s' = R0 s
      w[a] = fma(Rtl[3 * a], x, fma(Rtl[3 * a + 1], y, Rtl[3 * a + 2] * z));        // R~ s
    }
    const double e[3] = {s.q[0] - (double)s.bx, s.q[1] - (double)s.by, s.q[2] - (double)s.bz};
    const double wq = D / (D + 3.0 * sqrt(s.bd));
    const double rho = wq * wq;  // (D / (D + 3 |e|))^2, SVNICP.cpp:120-122
    acc[0] += rho;
    const double g[3] = {rho * sp[0], rho * sp[1], rho * sp[2]};
    acc[1] += g[0]; acc[2] += g[1]; acc[3] += g[2];
    acc[4] += g[0] * sp[0]; acc[5] += g[0] * sp[1]; acc[6] += g[0] * sp[2];
    acc[7] += g[1] * sp[1]; acc[8] += g[1] * sp[2]; acc[9] += g[2] * sp[2];
    const double f[3] = {rho * e[0], rho * e[1], rho * e[2]};
    acc[10] += f[0]; acc[11] += f[1]; acc[12] += f[2];
    acc[13] += w[1] * f[2] - w[2] * f[1];
    acc[14] += w[2] * f[0] - w[0] * f[2];
    acc[15] += w[0] * f[1] - w[1] * f[0];
  }
}

// The CTA's partial slot of pose p, in k_map_eval's order: a fixed butterfly per warp, then the warps in ascending order
__device__ __forceinline__ void map_eval_store(const double (&acc)[svn::EV_NS], double (&s_w)[MEV_THREADS / 32][svn::EV_NS], double *part,
                                               int p, int MB) {
  using svn::EV_NS;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int j = 0; j < EV_NS; j++) {
    const double v = svn::warp_sum(acc[j]);
    if (lane == 0) s_w[warp][j] = v;
  }
  __syncthreads();
  if (threadIdx.x < EV_NS) {
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < MEV_THREADS / 32; w++) t += s_w[w][threadIdx.x];
    part[((size_t)blockIdx.x * MB + p) * EV_NS + threadIdx.x] = t;
  }
}

// The seeded search gives map_nearest's result bit for bit.  The seed is a stored point (the map does not change during a
// call).  When its d^2 at the new query is < max_dist, it starts the search as the current best, and the box radius becomes
// sqrt(d^2_seed) * MEV_MARGIN.  Then:
//  - The true nearest point p* has d^2(p*) <= d^2_seed.  By the box argument of box_axis, which holds for any radius that bounds
//    the nearest distance with the margin over dist2's rounding, the box holds p*.  map_nearest itself relies on the same
//    argument when it shrinks the box to the best distance found in the query's own voxel.
//  - Every visit compares (d^2, lexicographic (x, y, z)), a total order on the data alone, and keeps the smaller; the seed's
//    own voxel lies inside the box, so revisiting the seed leaves an exact tie with itself unchanged.  The result is the
//    minimum of the visited set plus the seed, which contains p*: p* itself.
//  - A seed with d^2 >= max_dist, NaN (no point last iteration: the store writes NaN) or a non-finite query is not used, and
//    the search is map_nearest's from max_dist.
// The inlier bit, d^2 and the chosen point are therefore those of k_map_eval, and so are the sums.
template <typename T>
__global__ void __launch_bounds__(MEV_THREADS, 4) k_map_refine_eval(MapDev m, const T *__restrict__ src, int n, const double *__restrict__ Rt,
                                                                    svn::ScanConst sc, double max_dist, double r, const int *__restrict__ active,
                                                                    double *part, float *seed) {
  using svn::EV_NS;
  __shared__ double s_w[MEV_THREADS / 32][EV_NS];
  const int p = blockIdx.y, MB = gridDim.y;
  if (!active[p]) return;  // the whole CTA: the pose stopped
  const double *P = Rt + 12 * p;
  double Rtl[9], ttl[3];
#pragma unroll
  for (int i = 0; i < 9; i++) Rtl[i] = P[i];
#pragma unroll
  for (int i = 0; i < 3; i++) ttl[i] = P[9 + i];
  double acc[EV_NS];
#pragma unroll
  for (int j = 0; j < EV_NS; j++) acc[j] = 0.0;
  for (int i = blockIdx.x * MEV_THREADS + threadIdx.x; i < n; i += gridDim.x * MEV_THREADS) {
    const double x = (double)src[3 * (size_t)i], y = (double)src[3 * (size_t)i + 1], z = (double)src[3 * (size_t)i + 2];
    NearestState s;
#pragma unroll
    for (int a = 0; a < 3; a++) s.q[a] = svn::affine_row_fma(Rtl, ttl, a, x, y, z);
    s.bd = max_dist;
    s.bx = s.by = s.bz = 0.f;
    s.found = false;
    float *sd = RF_SEED ? seed + ((size_t)p * n + i) * 3 : nullptr;
    if (isfinite(s.q[0]) && isfinite(s.q[1]) && isfinite(s.q[2])) {
      double rs = r;
      if (RF_SEED) {
        const float px = sd[0], py = sd[1], pz = sd[2];
        const double mp[3] = {(double)px, (double)py, (double)pz};
        const double d = svn::dist2(s.q, mp);
        if (d < max_dist) {
          s.bd = d; s.bx = px; s.by = py; s.bz = pz; s.found = true;
          rs = fmin(r, sqrt(d) * MEV_MARGIN);
        }
      }
      map_nearest(m, rs, s);
    }
    if (RF_SEED) {
      const float nan = __int_as_float(0x7fffffff);
      sd[0] = s.found ? s.bx : nan; sd[1] = s.found ? s.by : nan; sd[2] = s.found ? s.bz : nan;
    }
    map_eval_accum<true>(s, x, y, z, Rtl, sc, max_dist, acc);
  }
  map_eval_store(acc, s_w, part, p, MB);
}

// One thread per pose of the block: delta = -H^-1 b from k_eval_fin's H and b (ldl_solve6_reg), the update of SVNICP.cpp:268-279
// in tail2.cu's operation order with J_l = I at delta_omega = 0 (not the reference's NaN, Q7), x' = [t' ; so3_log_principal(R')],
// |delta| in the order of tail2.cu, then the stop rule (update, then test) and R~ t~, R_p of x' for the next iteration.
// An exactly zero delta (e.g. no inlier: b = 0) leaves x as it is, bit for bit.
__global__ void k_map_refine_step(const double *__restrict__ ev, int MB, svn::ScanConst sc, int iterations, double tol, int *active,
                                  int *iters, double *step, double *x6, double *Rt, double *Rp) {
  using svn::EV_OUT;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= MB || !active[p]) return;
  const double *o = ev + (size_t)EV_OUT * p;
  double A[36], d[6];
#pragma unroll
  for (int i = 0; i < 36; i++) A[i] = o[3 + i];
#pragma unroll
  for (int i = 0; i < 6; i++) d[i] = o[39 + i];
  svn::ldl_solve6_reg(A, d);
#pragma unroll
  for (int i = 0; i < 6; i++) d[i] = -d[i];
  double *x = x6 + 6 * p;
  const bool zero = d[0] == 0.0 && d[1] == 0.0 && d[2] == 0.0 && d[3] == 0.0 && d[4] == 0.0 && d[5] == 0.0;
  if (!zero) {
    double dR[9], Jl[9], Rn[9], dt[3], t[3], w[3];
    const double *R = Rp + 9 * p;  // Exp(omega) of the current x (map_pose)
    svn::so3_exp(d + 3, dR, Jl);
    const bool rot0 = d[3] == 0.0 && d[4] == 0.0 && d[5] == 0.0;
#pragma unroll
    for (int r = 0; r < 3; r++) dt[r] = rot0 ? d[r] : Jl[3 * r] * d[0] + Jl[3 * r + 1] * d[1] + Jl[3 * r + 2] * d[2];
#pragma unroll
    for (int r = 0; r < 3; r++)
#pragma unroll
      for (int c = 0; c < 3; c++) Rn[3 * r + c] = R[3 * r] * dR[c] + R[3 * r + 1] * dR[3 + c] + R[3 * r + 2] * dR[6 + c];
#pragma unroll
    for (int r = 0; r < 3; r++) t[r] = (Rn[3 * r] * dt[0] + Rn[3 * r + 1] * dt[1] + Rn[3 * r + 2] * dt[2]) + x[r];
    svn::so3_log_principal(Rn, w);
#pragma unroll
    for (int q = 0; q < 3; q++) { x[q] = t[q]; x[3 + q] = w[q]; }
  }
  const double dn = sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2] + d[3] * d[3] + d[4] * d[4] + d[5] * d[5]);
  const int it = iters[p] + 1;
  iters[p] = it;
  step[p] = dn;
  if (dn < tol || it >= iterations) active[p] = 0;
  double R[9];
  map_pose(x, sc, Rt + 12 * p, R);
#pragma unroll
  for (int i = 0; i < 9; i++) Rp[9 * p + i] = R[i];
}

// ---- svnicp_map_search (DESIGN.md section 10d) -------------------------------------------------------------------------------
// Per chunk of grid poses: k_map_search_prep (grid value -> R~ t~ by map_pose) -> k_map_search_count (inlier count per pose)
// -> k_map_search_topk (running top k of the keys ((n - count) << 32) | g).
constexpr int MS_CHUNK = 16384;      // poses per chunk at most (scratch: 100 B per pose); fewer for large scans, see svnicp_map_search
constexpr int MS_MAX_K = 1024;       // top_k limit: the winners are sorted in one block of MS_TOPK_THREADS
constexpr int MS_TOPK_THREADS = 1024;

// Grid value i of an axis with `count` values and step `step`: ((double)i - 0.5 (count - 1)) * step.  The difference is exact
// (half integers below 2^31), so the one rounding is the product's, as in search_grid_poses of the Python mirror and the host
// decode in svnicp_map_search.  A 64-bit i is the pruned path's virtual block end, which may lie past the axis (below 2^32).
template <typename I>
__host__ __device__ __forceinline__ double grid_value(I i, int count, double step) {
  return ((double)i - 0.5 * (double)(count - 1)) * step;
}

struct GridSpec {
  int counts[6];
  double steps[6];
};

// R~ t~ of grid poses g0 .. g0 + Mc - 1 -> Rt [Mc][12], the bits k_map_eval_prep gives the same x
__global__ void k_map_search_prep(GridSpec gs, long long g0, int Mc, svn::ScanConst sc, double *Rt) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= Mc) return;
  long long g = g0 + p;
  double x[6], R[9];
#pragma unroll
  for (int a = 0; a < 6; a++) {
    const int i = (int)(g % gs.counts[a]);
    g /= gs.counts[a];
    x[a] = grid_value(i, gs.counts[a], gs.steps[a]);
  }
  map_pose(x, sc, Rt + 12 * (size_t)p, R);
}

// Does the voxel hold a point with d^2 < max_dist?
__device__ __forceinline__ bool slot_any_within(const MapTable &t, int cap, int slot, const double q[3], double max_dist) {
  const int c = __ldg(t.count + slot);
  const float *p = t.pts + (size_t)slot * cap * 3;
  for (int k = 0; k < c; k++) {
    const double mp[3] = {(double)__ldg(p + 3 * k), (double)__ldg(p + 3 * k + 1), (double)__ldg(p + 3 * k + 2)};
    if (svn::dist2(q, mp) < max_dist) return true;
  }
  return false;
}

// Is there a stored point with d^2 < max_dist for the finite query q?  The box, the probes and dist2 are map_nearest's, but the
// walk stops at the first such point and the box never shrinks.  This is map_nearest's `found`, bit for bit: map_nearest sets
// found exactly when it visits a point with dist2 < max_dist (its running bound starts at max_dist), and both walks visit every
// voxel of the initial box until then -- map_nearest shrinks the box only once found is set.  By the box argument of box_axis,
// the initial box (radius r = sqrt(max_dist) * MEV_MARGIN) holds every point whose dist2 can fall below max_dist, dist2's
// rounding being far below the margin.  So both are "some stored point has dist2(q, p) < max_dist", evaluated on the same q
// with the same dist2: the inlier count svnicp_map_evaluate reports.
__device__ __forceinline__ bool map_any_within(const MapDev &m, double r, double max_dist, const double q[3]) {
  const float v = m.voxel_size_f;
  int lo[3], hi[3];
  bool wide = false;
#pragma unroll
  for (int a = 0; a < 3; a++) {
    box_axis(q[a], r, v, lo[a], hi[a]);
    wide |= (long long)hi[a] - lo[a] >= MEV_SPAN;
  }
  if (wide) {  // map_nearest's sweep of the whole table, with the early exit
    for (int slot = 0; slot <= m.slots_mask; slot++)
      if (__ldg(m.tab.keys + slot) != EMPTY_KEY && slot_any_within(m.tab, m.cap, slot, q, max_dist)) return true;
    return false;
  }
  int own[3];
#pragma unroll
  for (int a = 0; a < 3; a++) own[a] = (int)__fdiv_rn(__double2float_rn(q[a]), v);
  int slot = map_find(m.tab, m.slots_mask, svn::pack_voxel_key(own[0], own[1], own[2]));
  if (slot >= 0 && slot_any_within(m.tab, m.cap, slot, q, max_dist)) return true;
  for (int z = lo[2]; z <= hi[2]; z++)
    for (int y = lo[1]; y <= hi[1]; y++)
      for (int x = lo[0]; x <= hi[0]; x++) {
        if (x == own[0] && y == own[1] && z == own[2]) continue;
        slot = map_find(m.tab, m.slots_mask, svn::pack_voxel_key(x, y, z));
        if (slot >= 0 && slot_any_within(m.tab, m.cap, slot, q, max_dist)) return true;
      }
  return false;
}

// Flat over (pose, point): warp w of the chunk holds 32 consecutive source points of pose w / wpp (wpp = warps per pose), as
// k_map_eval's warps, so that neighbouring lanes probe the same voxels; a 900-point scan gives 29 warps per pose and a chunk
// of 16 k poses fills the GPU.  q in k_map_eval's fma order; a non-finite q is not an inlier.  Integer counts: one
// warp-aggregated atomicAdd per warp, the same sum in any order.
template <typename T>
__global__ void __launch_bounds__(MEV_THREADS) k_map_search_count(MapDev m, const T *__restrict__ src, int n, int wpp, int Mc,
                                                                 const double *__restrict__ Rt, double max_dist, double r, int *cnt) {
  const long long w = ((long long)blockIdx.x * MEV_THREADS + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const int p = (int)(w / wpp);
  if (p >= Mc) return;  // whole warps: MEV_THREADS is a multiple of 32
  const int i = (int)(w - (long long)p * wpp) * 32 + lane;
  bool in = false;
  if (i < n) {
    const double *P = Rt + 12 * (size_t)p;
    double Rtl[9], ttl[3];
#pragma unroll
    for (int k = 0; k < 9; k++) Rtl[k] = __ldg(P + k);
#pragma unroll
    for (int k = 0; k < 3; k++) ttl[k] = __ldg(P + 9 + k);
    const double x = (double)src[3 * (size_t)i], y = (double)src[3 * (size_t)i + 1], z = (double)src[3 * (size_t)i + 2];
    double q[3];
#pragma unroll
    for (int a = 0; a < 3; a++) q[a] = svn::affine_row_fma(Rtl, ttl, a, x, y, z);
    if (isfinite(q[0]) && isfinite(q[1]) && isfinite(q[2])) in = map_any_within(m, r, max_dist, q);
  }
  const unsigned b = __ballot_sync(0xffffffffu, in);
  if (lane == 0 && b) atomicAdd(cnt + p, __popc(b));
}

// The running top k: the kk = min(k, n_best + Mc) smallest of the carried keys best [n_best] (sorted) and the chunk's keys
// ((n - cnt[p]) << 32) | (g0 + p), sorted ascending back into best.  Keys are unique (g is), so the kk smallest are one set:
// an MSB-first radix select over 8-bit digits finds the kk-th smallest key T exactly (integer histograms: no order dependence),
// the keys <= T are compacted (exactly kk of them, in any order) and a bitonic sort in shared memory orders them.
// LIST (the pruned path): pose p of the chunk is grid pose gl[p], or no pose at all when gl[p] < 0 (a slot of a partial edge
// block).  Such a slot's key is MS_NO_POSE, above every real key (n - cnt < 2^31); it may repeat, so the compaction skips it:
// the real keys are still unique, at most kk of them are <= T, and the rest of best is padded with MS_NO_POSE.
constexpr unsigned long long MS_NO_POSE = ~0ull;

template <bool LIST>
__device__ __forceinline__ unsigned long long search_key(const int *cnt, const int *gl, int p, long long g0, long long n) {
  if (LIST) return gl[p] < 0 ? MS_NO_POSE : ((unsigned long long)(n - cnt[p]) << 32) | (unsigned long long)gl[p];
  return ((unsigned long long)(n - cnt[p]) << 32) | (unsigned long long)(g0 + p);
}

template <bool LIST>
__global__ void __launch_bounds__(MS_TOPK_THREADS) k_map_search_topk(const int *cnt, int Mc, long long g0, long long n,
                                                                     unsigned long long *best, int n_best, int k, const int *gl) {
  __shared__ int s_hist[RADIX_DIGITS];
  __shared__ unsigned long long s_sel[MS_TOPK_THREADS];
  __shared__ unsigned long long s_prefix, s_mask;
  __shared__ int s_need, s_n;
  const int tid = threadIdx.x, total = n_best + Mc, kk = total < k ? total : k;
  auto key = [&](int j) { return j < n_best ? best[j] : search_key<LIST>(cnt, gl, j - n_best, g0, n); };
  if (tid == 0) { s_prefix = 0; s_mask = 0; s_need = kk; s_n = 0; }
  __syncthreads();
  if (kk < total) {
    for (int shift = 64 - RADIX_BITS; shift >= 0; shift -= RADIX_BITS) {
      for (int d = tid; d < RADIX_DIGITS; d += MS_TOPK_THREADS) s_hist[d] = 0;
      __syncthreads();
      const unsigned long long prefix = s_prefix, mask = s_mask;
      for (int j = tid; j < total; j += MS_TOPK_THREADS) {
        const unsigned long long kj = key(j);
        if ((kj & mask) == prefix) atomicAdd(&s_hist[(kj >> shift) & (RADIX_DIGITS - 1)], 1);
      }
      __syncthreads();
      if (tid == 0) {  // the digit of the need-th smallest key among those matching the prefix
        int need = s_need, d = 0;
        while (s_hist[d] < need) need -= s_hist[d++];
        s_need = need;
        s_prefix = prefix | ((unsigned long long)d << shift);
        s_mask = mask | ((unsigned long long)(RADIX_DIGITS - 1) << shift);
      }
      __syncthreads();
    }
  } else if (tid == 0) {
    s_prefix = ~0ull;  // every candidate is kept
  }
  __syncthreads();
  const unsigned long long T = s_prefix;
  for (int j = tid; j < total; j += MS_TOPK_THREADS) {
    const unsigned long long kj = key(j);
    if (kj <= T && (!LIST || kj != MS_NO_POSE)) s_sel[atomicAdd(&s_n, 1)] = kj;
  }
  __syncthreads();
  if (tid >= s_n) s_sel[tid] = ~0ull;  // s_n == kk <= MS_TOPK_THREADS
  __syncthreads();
  for (int size = 2; size <= MS_TOPK_THREADS; size <<= 1)
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      const int j = tid ^ stride;
      if (j > tid) {
        const unsigned long long a = s_sel[tid], b = s_sel[j];
        if ((a > b) == ((tid & size) == 0)) { s_sel[tid] = b; s_sel[j] = a; }
      }
      __syncthreads();
    }
  if (tid < kk) best[tid] = s_sel[tid];
}

// ---- svnicp_map_search, pruned path (DESIGN.md section 10e) ----------------------------------------------------------------
// The translation axes are cut into blocks of b[0] x b[1] x b[2] consecutive grid indices; a block is (block coordinates, one
// rotation index), id = c0 + nb[0] (c1 + nb[1] (c2 + nb[2] rot)), with rot the flat index of (i3, i4, i5) -- so g and id agree on
// the rotation.  Edge blocks are partial: every block is treated as the virtual full block starting at c_a b[a].
// k_map_search_bound_prep (R~ t~ of each block's centre) -> k_map_search_count at the bound radius (an upper bound of every
// count in the block, see svnicp_map_search) -> k_map_search_keys + the export's LSD radix sort (best bound first) ->
// per chunk of whole blocks: k_map_search_expand (grid poses) -> k_map_search_count -> k_map_search_violations -> the running top k.
struct BlockSpec {
  int b[3];   // grid indices per block on axes 0..2
  int nb[3];  // blocks per axis: ceil(counts[a] / b[a])
};

// Centre of each block id0 .. id0 + Mc - 1: per translation axis the fp64 midpoint of the virtual block's first and last grid
// values, the rotation's grid values, then map_pose -> Rt [Mc][12]
__global__ void k_map_search_bound_prep(GridSpec gs, BlockSpec bs, long long id0, int Mc, svn::ScanConst sc, double *Rt) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= Mc) return;
  long long id = id0 + p;
  double x[6], R[9];
#pragma unroll
  for (int a = 0; a < 3; a++) {
    const long long first = (id % bs.nb[a]) * bs.b[a], last = first + bs.b[a] - 1;
    id /= bs.nb[a];
    x[a] = 0.5 * (grid_value(first, gs.counts[a], gs.steps[a]) + grid_value(last, gs.counts[a], gs.steps[a]));
  }
#pragma unroll
  for (int a = 3; a < 6; a++) {
    x[a] = grid_value((int)(id % gs.counts[a]), gs.counts[a], gs.steps[a]);
    id /= gs.counts[a];
  }
  map_pose(x, sc, Rt + 12 * (size_t)p, R);
}

// Sort keys ((n - bound) << id_bits) | id, unique and ascending in (bound descending, id ascending); the values are the ids
__global__ void k_map_search_keys(const int *bound, int B, long long n, int id_bits, unsigned long long *keys, int *ids) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  keys[i] = ((unsigned long long)(n - bound[i]) << id_bits) | (unsigned long long)i;
  ids[i] = i;
}

// The grid poses of the chunk's blocks ids[0 .. Mc / ppb): slot p = j ppb + l0 + b0 (l1 + b1 l2) of block ids[j].  A pose
// inside the grid gets gl[p] = g and the R~ t~ k_map_search_prep gives that g (the same integers into the same arithmetic); a
// slot past the edge of a partial block gets gl[p] = -1 and a NaN translation, so that k_map_search_count finds no inlier for it
// without a probe.  The number of real poses is added to *counted.
__global__ void k_map_search_expand(GridSpec gs, BlockSpec bs, const int *ids, int Mc, int ppb, svn::ScanConst sc, double *Rt, int *gl,
                                    unsigned long long *counted) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  bool real = false;
  if (p < Mc) {
    const int j = p / ppb;
    int l = p - j * ppb;
    long long id = ids[j], g = 0, stride = 1;
    double x[6], R[9];
    real = true;
#pragma unroll
    for (int a = 0; a < 3; a++) {
      const long long i = (id % bs.nb[a]) * bs.b[a] + l % bs.b[a];
      id /= bs.nb[a];
      l /= bs.b[a];
      real &= i < gs.counts[a];
      x[a] = grid_value(i, gs.counts[a], gs.steps[a]);
      g += i * stride;
      stride *= gs.counts[a];
    }
    g += id * stride;  // id is now the rotation index
#pragma unroll
    for (int a = 3; a < 6; a++) {
      x[a] = grid_value((int)(id % gs.counts[a]), gs.counts[a], gs.steps[a]);
      id /= gs.counts[a];
    }
    double *o = Rt + 12 * (size_t)p;
    if (real) {
      map_pose(x, sc, o, R);
    } else {
#pragma unroll
      for (int c = 0; c < 12; c++) o[c] = __longlong_as_double(0x7FF8000000000000ll);  // NaN
    }
    gl[p] = real ? (int)g : -1;
  }
  const int c = __syncthreads_count(real);
  if (threadIdx.x == 0 && c) atomicAdd(counted, (unsigned long long)c);
}

// The self-check of the bound: a counted pose whose count exceeds its block's bound (keys in walk order, from the chunk's first)
__global__ void k_map_search_violations(const int *cnt, const int *gl, const unsigned long long *keys, int Mc, int ppb, long long n, int id_bits,
                                        unsigned long long *violations) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  const bool bad = p < Mc && gl[p] >= 0 && cnt[p] > n - (long long)(keys[p / ppb] >> id_bits);
  const int c = __syncthreads_count(bad);
  if (threadIdx.x == 0 && c) atomicAdd(violations, (unsigned long long)c);
}

// max |coordinate| over the finite coordinates of the scan, as the bits of a non-negative double (ordered like the values).  A
// point with a non-finite coordinate has a non-finite query at every pose and is an inlier nowhere, so it does not enter the slack.
template <typename T>
__global__ void k_max_abs_finite(const T *src, long long n3, unsigned long long *out) {
  double v = 0.0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n3; i += (long long)gridDim.x * blockDim.x) {
    const double a = fabs((double)src[i]);
    if (isfinite(a) && a > v) v = a;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  if ((threadIdx.x & 31) == 0 && v > 0.0) atomicMax(out, (unsigned long long)__double_as_longlong(v));
}

}  // namespace

struct svnicp_map_t {
  int device = 0;
  double voxel_size = 1.0, max_range = 80.0;
  int cap = 20;
  size_t slots = 0;
  MapTable tab[2] = {{nullptr, nullptr, nullptr}, {nullptr, nullptr, nullptr}};
  int cur = 0;
  int *head = nullptr, *walker = nullptr;
  long long *counters = nullptr;  // device [4]
  long long *h_counters = nullptr;  // pinned [4]
  // batch scratch
  void *batch_in = nullptr;
  float *wxyz = nullptr;
  int *pt_slot = nullptr, *next = nullptr;
  size_t batch_cap = 0;
  double *d_pose = nullptr;  // [12] R,t  + [3] position at offset 12
  // GetMap output
  double *out = nullptr;
  size_t out_cap = 0;
  int *block_sums = nullptr;
  long long last_n = 0;
  // svnicp_map_evaluate scratch (grown on demand; nothing above is touched by it)
  void *ev_src = nullptr;
  double *ev_pose = nullptr;  // [EV_BLOCK][6] x, [EV_BLOCK][12] R~ t~, [EV_BLOCK][9] R_p
  double *ev_part = nullptr, *ev_out = nullptr;
  uint8_t *ev_mask = nullptr;
  float *ev_near = nullptr;
  size_t ev_src_cap = 0, ev_part_cap = 0, ev_mask_cap = 0, ev_near_cap = 0;
  // svnicp_map_search scratch (grown on demand): R~ t~ [chunk][12], counts [chunk], the running top k [MS_MAX_K]
  double *ms_rt = nullptr;
  int *ms_cnt = nullptr;
  unsigned long long *ms_best = nullptr;
  size_t ms_rt_cap = 0, ms_cnt_cap = 0, ms_best_cap = 0;
  // ... and of its pruned path, indexed by MP_*: the block bounds, the sort's key and id buffers and histograms, the chunk's
  // grid indices, and device words; with the work done by the last successful call (svnicp_map_search_info)
  void *mp[8] = {};
  size_t mp_cap[8] = {};
  long long ms_info[8] = {};
  bool ms_info_valid = false;
  // svnicp_map_export / svnicp_map_import scratch (grown on demand; nothing above is touched by it), indexed by SN_*
  void *sn[11] = {};
  size_t sn_cap[11] = {};
  // svnicp_map_refine scratch (grown on demand; nothing above is touched by it), indexed by RF_*
  void *rf[9] = {};
  size_t rf_cap[9] = {};
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  std::string err;
};

static thread_local std::string g_map_create_error;

static int mfail(svnicp_map m, int code, const char *what, cudaError_t e = cudaSuccess) {
  char buf[256];
  snprintf(buf, sizeof(buf), "%s%s%s", what, e != cudaSuccess ? ": " : "", e != cudaSuccess ? cudaGetErrorString(e) : "");
  if (m) m->err = buf;
  else g_map_create_error = buf;
  return code;
}
#define MCU(call)                                                                                                  \
  do {                                                                                                             \
    cudaError_t e__ = (call);                                                                                      \
    if (e__ != cudaSuccess) return mfail(m, e__ == cudaErrorMemoryAllocation ? SVNICP_ERR_OOM : SVNICP_ERR_CUDA, #call, e__); \
  } while (0)

static MapDev dev_view(svnicp_map m, int which) {
  MapDev d;
  d.tab = m->tab[which];
  d.head = m->head; d.walker = m->walker; d.counters = m->counters;
  d.slots_mask = (int)(m->slots - 1); d.cap = m->cap;
  d.voxel_size_f = (float)m->voxel_size;  // Eigen promotes the double scalar to the vector's float (VoxelHashMap.cpp:30)
  return d;
}

static int clear_table(svnicp_map m, int which) {
  MCU(cudaMemsetAsync(m->tab[which].keys, 0xFF, m->slots * sizeof(unsigned long long), m->stream));
  MCU(cudaMemsetAsync(m->tab[which].count, 0, m->slots * sizeof(int), m->stream));
  return SVNICP_OK;
}

extern "C" {

int svnicp_map_create(svnicp_map *out, double voxel_size, double max_range, int max_pointscount, int64_t capacity_voxels, int device) {
  if (!out) return SVNICP_ERR_INVALID;
  *out = nullptr;
  if (!(voxel_size > 0) || max_pointscount < 1 || max_pointscount > MAX_CAP || capacity_voxels < 1)
    return mfail(nullptr, SVNICP_ERR_INVALID, "svnicp_map_create: need voxel_size > 0, 1 <= max_pointscount <= 32, capacity_voxels >= 1");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return mfail(nullptr, SVNICP_ERR_NO_DEVICE, "no CUDA device: this library has no CPU fallback");
  if (device < 0) cudaGetDevice(&device);
  if (device >= ndev) return mfail(nullptr, SVNICP_ERR_NO_DEVICE, "device out of range");
  svnicp_map m = new svnicp_map_t();
  m->device = device; m->voxel_size = voxel_size; m->max_range = max_range; m->cap = max_pointscount;
  size_t slots = 1024;
  while (slots < (size_t)capacity_voxels * 2) slots <<= 1;
  if (slots > (1ull << 30)) { delete m; return mfail(nullptr, SVNICP_ERR_INVALID, "capacity_voxels too large"); }
  m->slots = slots;
  auto body = [&]() -> int {
    MCU(cudaSetDevice(device));
    MCU(cudaDeviceGetAttribute(&m->sm_count, cudaDevAttrMultiProcessorCount, device));
    MCU(cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking));
    for (int w = 0; w < 2; w++) {
      MCU(cudaMalloc((void **)&m->tab[w].keys, slots * sizeof(unsigned long long)));
      MCU(cudaMalloc((void **)&m->tab[w].count, slots * sizeof(int)));
      MCU(cudaMalloc((void **)&m->tab[w].pts, slots * (size_t)m->cap * 3 * sizeof(float)));
    }
    MCU(cudaMalloc((void **)&m->head, slots * sizeof(int)));
    MCU(cudaMalloc((void **)&m->walker, slots * sizeof(int)));
    MCU(cudaMalloc((void **)&m->counters, 4 * sizeof(long long)));
    MCU(cudaMalloc((void **)&m->d_pose, 16 * sizeof(double)));
    MCU(cudaMalloc((void **)&m->ev_pose, (size_t)svn::EV_BLOCK * 27 * sizeof(double)));
    MCU(cudaMalloc((void **)&m->ev_out, (size_t)svn::EV_BLOCK * svn::EV_OUT * sizeof(double)));
    MCU(cudaMalloc((void **)&m->block_sums, ((slots + SCAN_BLOCK - 1) / SCAN_BLOCK + 1) * sizeof(int)));
    MCU(cudaMallocHost((void **)&m->h_counters, 4 * sizeof(long long)));
    memset(m->h_counters, 0, 4 * sizeof(long long));
    return SVNICP_OK;
  };
  int rc = body();
  if (rc == SVNICP_OK) rc = svnicp_map_clear(m);
  if (rc != SVNICP_OK) {
    g_map_create_error = m->err;
    svnicp_map_destroy(m);
    return rc;
  }
  *out = m;
  return SVNICP_OK;
}

void svnicp_map_destroy(svnicp_map m) {
  if (!m) return;
  cudaSetDevice(m->device);
  if (m->stream) cudaStreamSynchronize(m->stream);
  for (int w = 0; w < 2; w++) { cudaFree(m->tab[w].keys); cudaFree(m->tab[w].count); cudaFree(m->tab[w].pts); }
  cudaFree(m->head); cudaFree(m->walker); cudaFree(m->counters); cudaFree(m->d_pose); cudaFree(m->block_sums);
  cudaFree(m->batch_in); cudaFree(m->wxyz); cudaFree(m->pt_slot); cudaFree(m->next); cudaFree(m->out);
  cudaFree(m->ev_src); cudaFree(m->ev_pose); cudaFree(m->ev_part); cudaFree(m->ev_out); cudaFree(m->ev_mask); cudaFree(m->ev_near);
  cudaFree(m->ms_rt); cudaFree(m->ms_cnt); cudaFree(m->ms_best);
  for (void *p : m->mp) cudaFree(p);
  for (void *p : m->sn) cudaFree(p);
  for (void *p : m->rf) cudaFree(p);
  if (m->h_counters) cudaFreeHost(m->h_counters);
  if (m->stream) cudaStreamDestroy(m->stream);
  delete m;
}

const char *svnicp_map_last_error(svnicp_map m) { return m ? m->err.c_str() : g_map_create_error.c_str(); }

int svnicp_map_clear(svnicp_map m) {  // VoxelHashMap::Clear, VoxelHashMap.h:54
  if (!m) return SVNICP_ERR_INVALID;
  MCU(cudaSetDevice(m->device));
  m->cur = 0;
  int rc = clear_table(m, 0);
  if (rc) return rc;
  const unsigned grid = (unsigned)((m->slots + 255) / 256);
  k_fill_i32<<<grid, 256, 0, m->stream>>>(m->head, -1, m->slots);
  k_fill_i32<<<grid, 256, 0, m->stream>>>(m->walker, INT_MAX, m->slots);
  MCU(cudaMemsetAsync(m->counters, 0, 4 * sizeof(long long), m->stream));
  MCU(cudaGetLastError());
  MCU(cudaStreamSynchronize(m->stream));
  memset(m->h_counters, 0, 4 * sizeof(long long));
  m->last_n = 0;
  return SVNICP_OK;
}

static int sync_counters(svnicp_map m) {
  MCU(cudaMemcpyAsync(m->h_counters, m->counters, 4 * sizeof(long long), cudaMemcpyDeviceToHost, m->stream));
  MCU(cudaStreamSynchronize(m->stream));
  return SVNICP_OK;
}

int svnicp_map_add_cloud(svnicp_map m, const void *xyz, int64_t n, int dtype_f64, int on_device, const double R[9], const double t[3]) {
  if (!m || !R || !t || (n > 0 && !xyz)) return SVNICP_ERR_INVALID;
  if (n < 0 || n > (1ll << 30)) return mfail(m, SVNICP_ERR_INVALID, "svnicp_map_add_cloud: bad point count");
  MCU(cudaSetDevice(m->device));
  const size_t esz = dtype_f64 ? sizeof(double) : sizeof(float);
  if ((size_t)n > m->batch_cap) {
    cudaFree(m->batch_in); cudaFree(m->wxyz); cudaFree(m->pt_slot); cudaFree(m->next);
    m->batch_in = nullptr; m->wxyz = nullptr; m->pt_slot = nullptr; m->next = nullptr;
    const size_t cap = (size_t)n + (size_t)n / 4 + 1024;
    m->batch_cap = 0;
    MCU(cudaMalloc(&m->batch_in, cap * 3 * sizeof(double)));
    MCU(cudaMalloc((void **)&m->wxyz, cap * 3 * sizeof(float)));
    MCU(cudaMalloc((void **)&m->pt_slot, cap * sizeof(int)));
    MCU(cudaMalloc((void **)&m->next, cap * sizeof(int)));
    m->batch_cap = cap;
  }
  double pose[15];
  memcpy(pose, R, 9 * sizeof(double));
  memcpy(pose + 9, t, 3 * sizeof(double));
  memcpy(pose + 12, t, 3 * sizeof(double));  // current_pos = new_pose.translation() (:26)
  MCU(cudaMemcpyAsync(m->d_pose, pose, sizeof(pose), cudaMemcpyHostToDevice, m->stream));
  const MapDev d = dev_view(m, m->cur);
  // points that found no free voxel slot in THIS call (reported below; not sticky: RemoveFar may free room for the next cloud)
  MCU(cudaMemsetAsync(m->counters + 3, 0, sizeof(long long), m->stream));
  if (n > 0) {
    const void *src = xyz;
    if (!on_device) {
      MCU(cudaMemcpyAsync(m->batch_in, xyz, (size_t)n * 3 * esz, cudaMemcpyHostToDevice, m->stream));
      src = m->batch_in;
    }
    const unsigned grid = (unsigned)((n + 255) / 256);
    if (dtype_f64) k_map_insert_link<double><<<grid, 256, 0, m->stream>>>(d, (const double *)src, (int)n, m->d_pose, m->wxyz, m->pt_slot, m->next);
    else k_map_insert_link<float><<<grid, 256, 0, m->stream>>>(d, (const float *)src, (int)n, m->d_pose, m->wxyz, m->pt_slot, m->next);
    k_map_insert_place<<<grid, 256, 0, m->stream>>>(d, m->wxyz, m->pt_slot, m->next, (int)n);
    MCU(cudaGetLastError());
  }
  // RemoveFarPointCloud(current_pos) (:42, :93-101)
  MCU(cudaMemsetAsync(m->counters + 2, 0, sizeof(long long), m->stream));
  const double r2 = m->max_range * m->max_range;
  k_map_count_far<<<(unsigned)((m->slots + 255) / 256), 256, 0, m->stream>>>(d, m->d_pose + 12, r2);
  MCU(cudaGetLastError());
  int rc = sync_counters(m);  // also makes the host copy safe to reuse (the caller may free xyz)
  if (rc) return rc;
  const long long dropped = m->h_counters[3];
  if (m->h_counters[2] > 0) {
    const int nxt = m->cur ^ 1;
    rc = clear_table(m, nxt);
    if (rc) return rc;
    MCU(cudaMemsetAsync(m->counters, 0, 2 * sizeof(long long), m->stream));
    const MapDev dn = dev_view(m, nxt);
    k_map_rebuild<<<(unsigned)((m->slots * 32 + 255) / 256), 256, 0, m->stream>>>(d, dn, m->d_pose + 12, r2);
    MCU(cudaGetLastError());
    m->cur = nxt;
    rc = sync_counters(m);
    if (rc) return rc;
  }
  // the far voxels are gone and the counters are current either way; the points that did not fit are simply not in the map
  if (dropped > 0) return mfail(m, SVNICP_ERR_OOM, "voxel table full: some points of this cloud were dropped; create the map with a larger capacity_voxels");
  return SVNICP_OK;
}

int svnicp_map_get(svnicp_map m, const double position[3], double max_range, const double **device_xyz, int64_t *n_out) {
  if (!m || !n_out) return SVNICP_ERR_INVALID;
  MCU(cudaSetDevice(m->device));
  const size_t need = (size_t)(m->h_counters[1] > 0 ? m->h_counters[1] : 1);
  if (need > m->out_cap) {
    cudaFree(m->out);
    m->out = nullptr;
    m->out_cap = 0;
    MCU(cudaMalloc((void **)&m->out, (need + need / 4 + 1024) * 3 * sizeof(double)));
    m->out_cap = need + need / 4 + 1024;
  }
  const int all = position ? 0 : 1;  // GetMap() (:45-51) vs GetMap(pose, max_range) (:53-63)
  if (position) MCU(cudaMemcpyAsync(m->d_pose + 12, position, 3 * sizeof(double), cudaMemcpyHostToDevice, m->stream));
  const MapDev d = dev_view(m, m->cur);
  const int n_blocks = (int)((m->slots + SCAN_BLOCK - 1) / SCAN_BLOCK);
  const double r2 = max_range * max_range;
  k_getmap_count<<<n_blocks, SCAN_BLOCK, 0, m->stream>>>(d, m->d_pose + 12, r2, all, m->block_sums);
  svn::k_scan_block_sums<int><<<1, SCAN_BLOCK, 0, m->stream>>>(m->block_sums, n_blocks, m->counters + 2);
  k_getmap_emit<<<n_blocks, SCAN_BLOCK, 0, m->stream>>>(d, m->d_pose + 12, r2, all, m->block_sums, m->out);
  MCU(cudaGetLastError());
  int rc = sync_counters(m);
  if (rc) return rc;
  m->last_n = m->h_counters[2];
  *n_out = m->last_n;
  if (device_xyz) *device_xyz = m->out;
  return SVNICP_OK;
}

int svnicp_map_download(svnicp_map m, double *out_xyz, int64_t n) {
  if (!m || (n > 0 && !out_xyz)) return SVNICP_ERR_INVALID;
  if (n > m->last_n) return mfail(m, SVNICP_ERR_INVALID, "svnicp_map_download: more points requested than the last svnicp_map_get produced");
  MCU(cudaSetDevice(m->device));
  if (n > 0) MCU(cudaMemcpy(out_xyz, m->out, (size_t)n * 3 * sizeof(double), cudaMemcpyDeviceToHost));
  return SVNICP_OK;
}

int svnicp_map_size(svnicp_map m, int64_t *voxels, int64_t *points) {  // VoxelHashMap::Size / Empty, VoxelHashMap.h:55-56
  if (!m) return SVNICP_ERR_INVALID;
  if (voxels) *voxels = m->h_counters[0];
  if (points) *points = m->h_counters[1];
  return SVNICP_OK;
}

}  // extern "C"

// device scratch of svnicp_map_evaluate: (re)allocate *p to hold at least `bytes`
static int ev_grow(svnicp_map m, void **p, size_t *cap, size_t bytes) {
  if (bytes <= *cap) return SVNICP_OK;
  cudaFree(*p);
  *p = nullptr;
  *cap = 0;
  MCU(cudaMalloc(p, bytes));
  *cap = bytes;
  return SVNICP_OK;
}

// The scan and threshold checks shared by svnicp_map_evaluate and svnicp_map_search: n, max_dist and the search-radius limit
static int check_scan_args(svnicp_map m, const char *fn, int64_t n, double max_dist) {
  char buf[256];
  if (n < 1 || n > (1ll << 30)) {
    snprintf(buf, sizeof(buf), "%s: need 1 <= n <= 2^30 source points", fn);
    return mfail(m, SVNICP_ERR_INVALID, buf);
  }
  if (!isfinite(max_dist) || !(max_dist > 0)) {
    snprintf(buf, sizeof(buf), "%s: max_dist must be finite and > 0", fn);
    return mfail(m, SVNICP_ERR_INVALID, buf);
  }
  const double r = sqrt(max_dist);
  if (ceil(r / m->voxel_size) > MEV_MAX_REACH) {
    snprintf(buf, sizeof(buf), "%s: search radius sqrt(max_dist) = %g m spans %g voxels of %g m on each side of the "
             "query; at most %d are supported", fn, r, ceil(r / m->voxel_size), m->voxel_size, MEV_MAX_REACH);
    return mfail(m, SVNICP_ERR_INVALID, buf);
  }
  return SVNICP_OK;
}

template <bool SYS>
static void go_map_eval(const MapDev &d, const void *src, int dtype_f64, dim3 grid, int n, const double *Rt, const svn::ScanConst &sc,
                        double max_dist, double r, double *part, uint8_t *mask, float *nearest, cudaStream_t st) {
  if (dtype_f64)
    k_map_eval<double, SYS><<<grid, MEV_THREADS, 0, st>>>(d, (const double *)src, n, Rt, sc, max_dist, r, part, mask, nearest);
  else
    k_map_eval<float, SYS><<<grid, MEV_THREADS, 0, st>>>(d, (const float *)src, n, Rt, sc, max_dist, r, part, mask, nearest);
}

extern "C" int svnicp_map_evaluate(svnicp_map m, const void *source, int64_t n, int dtype_f64, int on_device, const double R0[9],
                                   const double t0[3], int n_poses, const double *poses_6xM, double max_dist, double *out_stats,
                                   double *out_H, double *out_b, uint8_t *out_mask, float *out_nearest) {
  using svn::EV_BLOCK;
  using svn::EV_NS;
  using svn::EV_OUT;
  if (!m) return SVNICP_ERR_INVALID;
  if (!source || !R0 || !t0 || !poses_6xM || !out_stats)
    return mfail(m, SVNICP_ERR_INVALID, "svnicp_map_evaluate: null source, R0, t0, poses or out_stats");
  int rc = check_scan_args(m, "svnicp_map_evaluate", n, max_dist);
  if (rc) return rc;
  if (n_poses < 1) return mfail(m, SVNICP_ERR_INVALID, "svnicp_map_evaluate: n_poses must be >= 1");
  const double r = sqrt(max_dist);
  MCU(cudaSetDevice(m->device));
  cudaStream_t st = m->stream;
  const int ni = (int)n, M = n_poses;
  const int mb_max = M < EV_BLOCK ? M : EV_BLOCK;
  int parts = (int)((n + MEV_THREADS - 1) / MEV_THREADS);
  if (parts > m->sm_count * MEV_CTAS_PER_SM) parts = m->sm_count * MEV_CTAS_PER_SM;
  const size_t esz = dtype_f64 ? sizeof(double) : sizeof(float);
  if ((rc = ev_grow(m, (void **)&m->ev_part, &m->ev_part_cap, (size_t)parts * mb_max * EV_NS * sizeof(double))) ||
      (!on_device && (rc = ev_grow(m, &m->ev_src, &m->ev_src_cap, (size_t)n * 3 * esz))) ||
      (out_mask && (rc = ev_grow(m, (void **)&m->ev_mask, &m->ev_mask_cap, (size_t)mb_max * n))) ||
      (out_nearest && (rc = ev_grow(m, (void **)&m->ev_near, &m->ev_near_cap, (size_t)mb_max * n * 3 * sizeof(float)))))
    return rc;
  const void *src = source;
  if (!on_device) {
    MCU(cudaMemcpyAsync(m->ev_src, source, (size_t)n * 3 * esz, cudaMemcpyHostToDevice, st));
    src = m->ev_src;
  }
  svn::ScanConst sc;
  memcpy(sc.R0, R0, sizeof(sc.R0));
  memcpy(sc.t0, t0, sizeof(sc.t0));
  double *x_blk = m->ev_pose, *Rt_blk = m->ev_pose + 6 * EV_BLOCK, *Rp_blk = m->ev_pose + 18 * EV_BLOCK;
  const MapDev d = dev_view(m, m->cur);
  const bool sys = out_H || out_b;
  std::vector<double> hx((size_t)6 * EV_BLOCK), res((size_t)EV_OUT * EV_BLOCK);
  for (int m0 = 0; m0 < M; m0 += EV_BLOCK) {
    const int MB = M - m0 < EV_BLOCK ? M - m0 : EV_BLOCK;
    for (int j = 0; j < MB; j++)
      for (int c = 0; c < 6; c++) hx[(size_t)6 * j + c] = poses_6xM[(size_t)c * M + m0 + j];
    MCU(cudaMemcpyAsync(x_blk, hx.data(), (size_t)6 * MB * sizeof(double), cudaMemcpyHostToDevice, st));
    k_map_eval_prep<<<1, EV_BLOCK, 0, st>>>(x_blk, MB, sc, Rt_blk, Rp_blk);
    const dim3 grid((unsigned)parts, (unsigned)MB);
    uint8_t *mk = out_mask ? m->ev_mask : nullptr;
    float *nr = out_nearest ? m->ev_near : nullptr;
    if (sys) go_map_eval<true>(d, src, dtype_f64, grid, ni, Rt_blk, sc, max_dist, r * MEV_MARGIN, m->ev_part, mk, nr, st);
    else go_map_eval<false>(d, src, dtype_f64, grid, ni, Rt_blk, sc, max_dist, r * MEV_MARGIN, m->ev_part, mk, nr, st);
    svn::launch_eval_fin(m->ev_part, parts, MB, ni, sc, Rp_blk, m->ev_out, st);
    MCU(cudaGetLastError());
    MCU(cudaMemcpyAsync(res.data(), m->ev_out, (size_t)EV_OUT * MB * sizeof(double), cudaMemcpyDeviceToHost, st));
    // [M][n] outputs: the rows of this block are contiguous in the caller's arrays
    if (out_mask) MCU(cudaMemcpyAsync(out_mask + (size_t)m0 * n, m->ev_mask, (size_t)MB * n, cudaMemcpyDeviceToHost, st));
    if (out_nearest)
      MCU(cudaMemcpyAsync(out_nearest + (size_t)m0 * n * 3, m->ev_near, (size_t)MB * n * 3 * sizeof(float), cudaMemcpyDeviceToHost, st));
    MCU(cudaStreamSynchronize(st));  // the host block buffers are refilled next
    for (int j = 0; j < MB; j++) {
      const double *o = res.data() + (size_t)EV_OUT * j;
      const size_t g = (size_t)m0 + j;
      memcpy(out_stats + 3 * g, o, 3 * sizeof(double));
      if (out_H) memcpy(out_H + 36 * g, o + 3, 36 * sizeof(double));
      if (out_b) memcpy(out_b + 6 * g, o + 39, 6 * sizeof(double));
    }
  }
  return SVNICP_OK;
}

// ---- svnicp_map_search --------------------------------------------------------------------------------------------------------
// Scratch of the pruned path (DESIGN.md section 10e), grown on demand: 28 B per block (the bound, two key and two id buffers of
// the sort) + 4 B per 16 blocks of radix histogram + 4 B per chunk pose + 32 B of words.
enum { MP_BOUND, MP_KEY0, MP_KEY1, MP_ID0, MP_ID1, MP_HIST, MP_GL, MP_WORDS, MP_COUNT };
static_assert(MP_COUNT == sizeof(svnicp_map_t::mp) / sizeof(void *), "one scratch buffer per MP_* index");
// Selection rule: a grid of fewer than MS_POSES_PER_K * top_k poses takes the exhaustive path.  The walk cannot stop before k
// poses are counted and stops only on a bound below the k-th count, which a k that large keeps low: on the 143 k-point scan
// with k = 1024 of 3 969 poses nothing was pruned and the bound pass made the call 2 % slower (DESIGN.md section 10e).  The
// define is for A/B builds through SVNICP_NVCC_DEFS, as the other SVN_* switches (0: every grid with blocks is pruned).
#ifndef SVN_MS_POSES_PER_K
#define SVN_MS_POSES_PER_K 16
#endif
constexpr long long MS_POSES_PER_K = SVN_MS_POSES_PER_K;

static int mp_grow(svnicp_map m, int k, size_t bytes) { return ev_grow(m, &m->mp[k], &m->mp_cap[k], bytes > 0 ? bytes : 1); }

static void launch_search_count(const MapDev &d, const void *src, int dtype_f64, int n, int wpp, int Mc, const double *Rt, double max_dist,
                                double r, int *cnt, cudaStream_t st) {
  const unsigned blocks = (unsigned)(((long long)Mc * wpp + MEV_THREADS / 32 - 1) / (MEV_THREADS / 32));
  if (dtype_f64) k_map_search_count<double><<<blocks, MEV_THREADS, 0, st>>>(d, (const double *)src, n, wpp, Mc, Rt, max_dist, r, cnt);
  else k_map_search_count<float><<<blocks, MEV_THREADS, 0, st>>>(d, (const float *)src, n, wpp, Mc, Rt, max_dist, r, cnt);
}

struct BlockPlan {
  BlockSpec bs;
  int ppb;            // poses per full block
  long long B;        // blocks
  double max_dist_b;  // the bound's threshold r_B^2, rounded up
  double r_b;         // its box radius sqrt(max_dist_b) * MEV_MARGIN
};

// rho = max |R0 d| over the corners d = (+-h0, +-h1, +-h2) of the block's translation box, in fp64.  |R0 d| is convex in d, so
// its maximum over the box is at a corner; R0 need not be orthonormal (nothing checks it).
static double corner_radius(const double R0[9], const double h[3]) {
  double rho = 0.0;
  for (int c = 0; c < 8; c++) {
    const double dv[3] = {c & 1 ? h[0] : -h[0], c & 2 ? h[1] : -h[1], c & 4 ? h[2] : -h[2]};
    double s = 0.0;
    for (int r = 0; r < 3; r++) {
      const double v = R0[3 * r] * dv[0] + R0[3 * r + 1] * dv[1] + R0[3 * r + 2] * dv[2];
      s += v * v;
    }
    rho = fmax(rho, sqrt(s));
  }
  return rho;
}

// Why no pose of a block counts more inliers than the block's bound.  Let c be the block's centre and x one of its poses; they
// share omega, so map_pose gives them the same R~ (as values: x = 0 stores R0 itself, which equals R0 Exp(0) up to the sign
// of zeros), and t~_x - t~_c = R0 (t_x - t_c) up to the rounding of map_pose.  t_x - t_c lies in the box [-h, h], h_a =
// 0.5 (b_a - 1) steps[a], up to the rounding of grid_value and of the midpoint, so |R0 (t_x - t_c)| <= rho.  The queries of a
// source point s, q_x and q_c, are formed by the same affine_row_fma from the same R~ and s, so |q_x - q_c| <= rho + delta,
// where delta bounds every rounding above: each is a few ulp of |t0|, ||R0|| max|t| or ||R~ s|| <= ||R0|| |s| (fp64, relative
// 2^-53 each), and delta = 1e-9 (1 + |t0| + ||R0||_F max|t| + ||R0||_F sqrt(3) max|s|) exceeds their sum by a factor of about
// 10^6 (max|t| over the virtual blocks, which end at most 1.5 (counts - 1) steps from the centre; max|s| over the finite
// coordinates: a point with a non-finite one has no finite query anywhere).  If s is an inlier of x, a stored p has
// dist2(q_x, p) < max_dist; dist2 is within 4 ulp of |q_x - p|^2, so |q_x - p| < sqrt(max_dist) MEV_MARGIN and
//   |q_c - p| <= |q_c - q_x| + |q_x - p| < sqrt(max_dist) MEV_MARGIN + rho + delta = r_B.
// With max_dist_B = r_B^2 MEV_MARGIN, dist2(q_c, p) < max_dist_B (dist2 again within 4 ulp), and map_any_within at that
// threshold with its box at sqrt(max_dist_B) MEV_MARGIN finds such a point (map_any_within's own argument): s is an inlier of
// the bound query at c.  So count(x) <= bound(block), for every x of the block.  k_map_search_violations checks it on every
// counted pose.
//
// Block sizes: equal metric half-extents H on the translation axes with counts > 1, b_a = min(counts[a], 1 + floor(2 H /
// steps[a])) (a zero step adds nothing to rho and takes the finest positive step as its unit), and the largest H for which
// ceil(box radius / voxel_size) <= MEV_MAX_REACH -- so the bound queries never reach map_any_within's whole-table sweep -- and a
// block fits one chunk.  rho and the block count grow with H, so a bisection finds it.  False: the grid gets no blocks (every
// b_a = 1) and takes the exhaustive path.
static bool plan_blocks(double voxel_size, const int32_t counts[6], const double steps[6], const double R0[9], const double t0[3],
                        double max_dist, double max_abs_s, int chunk, BlockPlan *pl) {
  double nR = 0.0, tmax = 0.0, t0n = 0.0;
  for (int i = 0; i < 9; i++) nR += R0[i] * R0[i];
  for (int a = 0; a < 3; a++) {
    const double e = 1.5 * (double)(counts[a] - 1) * steps[a];
    tmax += e * e;
    t0n += t0[a] * t0[a];
  }
  nR = sqrt(nR);
  const double delta = 1e-9 * (1.0 + sqrt(t0n) + nR * sqrt(tmax) + nR * sqrt(3.0) * max_abs_s);
  const double base = sqrt(max_dist) * MEV_MARGIN + delta;
  if (!isfinite(base)) return false;
  double s_ref = 0.0;
  for (int a = 0; a < 3; a++)
    if (counts[a] > 1 && steps[a] > 0 && (s_ref == 0.0 || steps[a] < s_ref)) s_ref = steps[a];
  if (s_ref == 0.0) s_ref = voxel_size;
  auto sizes = [&](double H, BlockPlan &q) {  // true when the bound's box stays within MEV_MAX_REACH and a block fits a chunk
    double h[3];
    long long ppb = 1;
    for (int a = 0; a < 3; a++) {
      const double f = 2.0 * H / (steps[a] > 0 ? steps[a] : s_ref);
      const long long b = f >= (double)(counts[a] - 1) ? counts[a] : 1 + (long long)floor(f);
      q.bs.b[a] = (int)b;
      q.bs.nb[a] = (int)((counts[a] + b - 1) / b);
      h[a] = 0.5 * (double)(b - 1) * steps[a];
      ppb *= b;
    }
    const double rb = base + corner_radius(R0, h);
    q.ppb = (int)(ppb < chunk ? ppb : chunk);
    q.max_dist_b = rb * rb * MEV_MARGIN;
    q.r_b = sqrt(q.max_dist_b) * MEV_MARGIN;
    return ppb <= chunk && isfinite(q.r_b) && ceil(q.r_b / voxel_size) <= MEV_MAX_REACH;
  };
  double lo = 0.0, hi = 0.0;
  for (int a = 0; a < 3; a++) hi = fmax(hi, (double)counts[a] * (steps[a] > 0 ? steps[a] : s_ref));
  BlockPlan q;
  if (!sizes(lo, q)) return false;
  if (sizes(hi, q)) lo = hi;
  for (int it = 0; it < 100 && lo < hi; it++) {
    const double mid = 0.5 * (lo + hi);
    if (mid <= lo || mid >= hi) break;
    (sizes(mid, q) ? lo : hi) = mid;
  }
  sizes(lo, q);
  if (q.ppb == 1) return false;
  q.B = (long long)q.bs.nb[0] * q.bs.nb[1] * q.bs.nb[2] * counts[3] * counts[4] * counts[5];
  *pl = q;
  return true;
}

// The exhaustive path: every grid pose, in chunks of g
static int search_exhaustive(svnicp_map m, const MapDev &d, const void *src, int dtype_f64, int n, int wpp, int chunk, const GridSpec &gs,
                             const svn::ScanConst &sc, long long M, double max_dist, double r, int top_k, int32_t *out_counts,
                             long long info[8]) {
  cudaStream_t st = m->stream;
  int n_best = 0;
  for (long long g0 = 0; g0 < M; g0 += chunk) {
    const int Mc = (int)(M - g0 < chunk ? M - g0 : chunk);
    k_map_search_prep<<<(Mc + 127) / 128, 128, 0, st>>>(gs, g0, Mc, sc, m->ms_rt);
    MCU(cudaMemsetAsync(m->ms_cnt, 0, (size_t)Mc * sizeof(int), st));
    launch_search_count(d, src, dtype_f64, n, wpp, Mc, m->ms_rt, max_dist, r, m->ms_cnt, st);
    k_map_search_topk<false><<<1, MS_TOPK_THREADS, 0, st>>>(m->ms_cnt, Mc, g0, n, m->ms_best, n_best, top_k, nullptr);
    MCU(cudaGetLastError());
    if (out_counts) MCU(cudaMemcpyAsync(out_counts + g0, m->ms_cnt, (size_t)Mc * sizeof(int), cudaMemcpyDeviceToHost, st));
    n_best = n_best + Mc < top_k ? n_best + Mc : top_k;
  }
  const long long w[8] = {0, M, 0, 0, 0, M, 0, -1};
  memcpy(info, w, sizeof(w));
  return SVNICP_OK;
}

// The pruned path: block bounds, blocks sorted by bound, exact counts block by block until the next bound is below the k-th count
static int search_pruned(svnicp_map m, const MapDev &d, const void *src, int dtype_f64, int n, int wpp, int chunk, const GridSpec &gs,
                         const svn::ScanConst &sc, long long M, const BlockPlan &pl, double max_dist, double r, int top_k,
                         long long info[8]) {
  cudaStream_t st = m->stream;
  const long long B = pl.B;
  int id_bits = 1, n_bits = 1;
  while ((1ll << id_bits) < B) id_bits++;
  while ((1ll << n_bits) <= n) n_bits++;  // n - bound lies in [0, n]
  const int n_tiles = (int)((B + RADIX_TILE - 1) / RADIX_TILE);
  int rc;
  if ((rc = mp_grow(m, MP_BOUND, B * 4)) || (rc = mp_grow(m, MP_KEY0, B * 8)) || (rc = mp_grow(m, MP_KEY1, B * 8)) ||
      (rc = mp_grow(m, MP_ID0, B * 4)) || (rc = mp_grow(m, MP_ID1, B * 4)) || (rc = mp_grow(m, MP_HIST, (size_t)RADIX_DIGITS * n_tiles * 4)) ||
      (rc = mp_grow(m, MP_GL, (size_t)chunk * 4)))
    return rc;
  int *bound = (int *)m->mp[MP_BOUND], *gl = (int *)m->mp[MP_GL], *hist = (int *)m->mp[MP_HIST];
  unsigned long long *key[2] = {(unsigned long long *)m->mp[MP_KEY0], (unsigned long long *)m->mp[MP_KEY1]};
  int *id[2] = {(int *)m->mp[MP_ID0], (int *)m->mp[MP_ID1]};
  unsigned long long *words = (unsigned long long *)m->mp[MP_WORDS];  // [0] violations, [1] poses counted, [3] sink of the scans
  MCU(cudaMemsetAsync(words, 0, 2 * sizeof(unsigned long long), st));
  for (long long c0 = 0; c0 < B; c0 += chunk) {
    const int Mc = (int)(B - c0 < chunk ? B - c0 : chunk);
    k_map_search_bound_prep<<<(Mc + 127) / 128, 128, 0, st>>>(gs, pl.bs, c0, Mc, sc, m->ms_rt);
    MCU(cudaMemsetAsync(bound + c0, 0, (size_t)Mc * sizeof(int), st));
    launch_search_count(d, src, dtype_f64, n, wpp, Mc, m->ms_rt, pl.max_dist_b, pl.r_b, bound + c0, st);
  }
  k_map_search_keys<<<(unsigned)((B + 255) / 256), 256, 0, st>>>(bound, (int)B, n, id_bits, key[0], id[0]);
  int a = 0;
  for (int shift = 0; shift < id_bits + n_bits; shift += RADIX_BITS, a ^= 1) {
    k_radix_hist<<<n_tiles, RADIX_THREADS, 0, st>>>(key[a], (int)B, shift, n_tiles, hist);
    svn::k_scan_block_sums<int><<<1, SCAN_BLOCK, 0, st>>>(hist, RADIX_DIGITS * n_tiles, (long long *)words + 3);
    k_radix_scatter<<<n_tiles, RADIX_THREADS, 0, st>>>(key[a], id[a], key[a ^ 1], id[a ^ 1], (int)B, shift, n_tiles, hist);
  }
  MCU(cudaGetLastError());
  const unsigned long long *keys = key[a];
  const int *ids = id[a];
  // Stop rule: once k poses are counted, stop before the next block if its bound is strictly below the k-th count.  The blocks
  // left have bounds no higher, so none of their poses can reach the k-th count; on an equal bound a pose with that count and a
  // lower g might follow, so an equal bound does not stop the walk.
  const int per = chunk / pl.ppb;
  long long pos = 0;
  int n_best = 0;
  while (pos < B) {
    const int nbc = (int)(B - pos < per ? B - pos : per), Mc = nbc * pl.ppb;
    k_map_search_expand<<<(Mc + 127) / 128, 128, 0, st>>>(gs, pl.bs, ids + pos, Mc, pl.ppb, sc, m->ms_rt, gl, words + 1);
    MCU(cudaMemsetAsync(m->ms_cnt, 0, (size_t)Mc * sizeof(int), st));
    launch_search_count(d, src, dtype_f64, n, wpp, Mc, m->ms_rt, max_dist, r, m->ms_cnt, st);
    k_map_search_violations<<<(Mc + 127) / 128, 128, 0, st>>>(m->ms_cnt, gl, keys + pos, Mc, pl.ppb, n, id_bits, words);
    k_map_search_topk<true><<<1, MS_TOPK_THREADS, 0, st>>>(m->ms_cnt, Mc, 0, n, m->ms_best, n_best, top_k, gl);
    MCU(cudaGetLastError());
    n_best = n_best + Mc < top_k ? n_best + Mc : top_k;
    pos += nbc;
    if (pos < B && n_best == top_k) {
      unsigned long long h[2];  // the next block's key, the k-th best key (MS_NO_POSE until k real poses are counted)
      MCU(cudaMemcpyAsync(h, keys + pos, sizeof(h[0]), cudaMemcpyDeviceToHost, st));
      MCU(cudaMemcpyAsync(h + 1, m->ms_best + top_k - 1, sizeof(h[1]), cudaMemcpyDeviceToHost, st));
      MCU(cudaStreamSynchronize(st));
      if (h[1] != MS_NO_POSE && n - (long long)(h[0] >> id_bits) < n - (long long)(h[1] >> 32)) break;
    }
  }
  unsigned long long w[2];
  MCU(cudaMemcpyAsync(w, words, sizeof(w), cudaMemcpyDeviceToHost, st));
  MCU(cudaStreamSynchronize(st));
  const long long v[8] = {1, M, pl.ppb, B, pos, (long long)w[1], B * n, (long long)w[0]};
  memcpy(info, v, sizeof(v));
  return SVNICP_OK;
}

extern "C" int svnicp_map_search(svnicp_map m, const void *source, int64_t n, int dtype_f64, int on_device, const double R0[9],
                                 const double t0[3], const int32_t counts[6], const double steps[6], double max_dist, int top_k,
                                 int64_t *out_index, double *out_poses_6xK, double *out_stats, int32_t *out_counts) {
  if (!m) return SVNICP_ERR_INVALID;
  if (!source || !R0 || !t0 || !counts || !steps || !out_index || !out_poses_6xK || !out_stats)
    return mfail(m, SVNICP_ERR_INVALID, "svnicp_map_search: null source, R0, t0, counts, steps, out_index, out_poses or out_stats");
  int rc = check_scan_args(m, "svnicp_map_search", n, max_dist);
  if (rc) return rc;
  long long M = 1;
  for (int a = 0; a < 6; a++) {
    if (counts[a] < 1) return mfail(m, SVNICP_ERR_INVALID, "svnicp_map_search: every grid count must be >= 1");
    if (!isfinite(steps[a]) || !(steps[a] >= 0)) return mfail(m, SVNICP_ERR_INVALID, "svnicp_map_search: every grid step must be finite and >= 0");
    M *= counts[a];
    if (M > INT_MAX) return mfail(m, SVNICP_ERR_INVALID, "svnicp_map_search: the grid holds more than 2^31 - 1 poses");
  }
  if (top_k < 1 || top_k > MS_MAX_K || top_k > M) {
    char buf[160];
    snprintf(buf, sizeof(buf), "svnicp_map_search: top_k = %d is outside [1, min(%lld grid poses, %d)]", top_k, M, MS_MAX_K);
    return mfail(m, SVNICP_ERR_INVALID, buf);
  }
  MCU(cudaSetDevice(m->device));
  cudaStream_t st = m->stream;
  // poses per chunk: at most MS_CHUNK, and about 2^27 queries for large scans (one pose at least)
  const long long by_n = (1ll << 27) / n;
  const int chunk = (int)(by_n < 1 ? 1 : by_n < MS_CHUNK ? by_n : MS_CHUNK);
  const int wpp = (int)((n + 31) / 32);
  const size_t esz = dtype_f64 ? sizeof(double) : sizeof(float);
  if ((rc = ev_grow(m, (void **)&m->ms_rt, &m->ms_rt_cap, (size_t)chunk * 12 * sizeof(double))) ||
      (rc = ev_grow(m, (void **)&m->ms_cnt, &m->ms_cnt_cap, (size_t)chunk * sizeof(int))) ||
      (rc = ev_grow(m, (void **)&m->ms_best, &m->ms_best_cap, (size_t)MS_MAX_K * sizeof(unsigned long long))) ||
      (!on_device && (rc = ev_grow(m, &m->ev_src, &m->ev_src_cap, (size_t)n * 3 * esz))))
    return rc;
  const void *src = source;
  if (!on_device) {
    MCU(cudaMemcpyAsync(m->ev_src, source, (size_t)n * 3 * esz, cudaMemcpyHostToDevice, st));
    src = m->ev_src;
  }
  svn::ScanConst sc;
  memcpy(sc.R0, R0, sizeof(sc.R0));
  memcpy(sc.t0, t0, sizeof(sc.t0));
  GridSpec gs;
  memcpy(gs.counts, counts, sizeof(gs.counts));
  memcpy(gs.steps, steps, sizeof(gs.steps));
  const MapDev d = dev_view(m, m->cur);
  const double r = sqrt(max_dist) * MEV_MARGIN;  // k_map_eval's radius
  // Path: the per-pose counts need every pose counted; without them a grid with blocks takes the pruned path.  Both return the
  // same bits.
  BlockPlan pl;
  bool pruned = false;
  if (!out_counts && (counts[0] > 1 || counts[1] > 1 || counts[2] > 1) && M >= MS_POSES_PER_K * top_k) {
    if ((rc = mp_grow(m, MP_WORDS, 4 * sizeof(unsigned long long)))) return rc;
    unsigned long long *words = (unsigned long long *)m->mp[MP_WORDS], max_abs_bits;
    MCU(cudaMemsetAsync(words + 2, 0, sizeof(unsigned long long), st));
    const long long n3 = 3 * n;
    const unsigned grid = (unsigned)(n3 < 256ll * m->sm_count * 4 ? (n3 + 255) / 256 : m->sm_count * 4);
    if (dtype_f64) k_max_abs_finite<double><<<grid, 256, 0, st>>>((const double *)src, n3, words + 2);
    else k_max_abs_finite<float><<<grid, 256, 0, st>>>((const float *)src, n3, words + 2);
    MCU(cudaGetLastError());
    MCU(cudaMemcpyAsync(&max_abs_bits, words + 2, sizeof(max_abs_bits), cudaMemcpyDeviceToHost, st));
    MCU(cudaStreamSynchronize(st));
    double max_abs_s;
    memcpy(&max_abs_s, &max_abs_bits, sizeof(max_abs_s));
    pruned = plan_blocks(m->voxel_size, counts, steps, R0, t0, max_dist, max_abs_s, chunk, &pl);
  }
  long long info[8];
  rc = pruned ? search_pruned(m, d, src, dtype_f64, (int)n, wpp, chunk, gs, sc, M, pl, max_dist, r, top_k, info)
              : search_exhaustive(m, d, src, dtype_f64, (int)n, wpp, chunk, gs, sc, M, max_dist, r, top_k, out_counts, info);
  if (rc) return rc;
  std::vector<unsigned long long> best((size_t)top_k);
  MCU(cudaMemcpyAsync(best.data(), m->ms_best, (size_t)top_k * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
  MCU(cudaStreamSynchronize(st));
  for (int j = 0; j < top_k; j++) {
    long long g = (long long)(best[j] & 0xFFFFFFFFull);
    out_index[j] = g;
    for (int a = 0; a < 6; a++) {
      out_poses_6xK[(size_t)a * top_k + j] = grid_value((int)(g % counts[a]), counts[a], steps[a]);
      g /= counts[a];
    }
  }
  // the winners' statistics are svnicp_map_evaluate's by construction: the same call on the grid values (source already on device)
  rc = svnicp_map_evaluate(m, src, n, dtype_f64, 1, R0, t0, top_k, out_poses_6xK, max_dist, out_stats, nullptr, nullptr, nullptr, nullptr);
  if (rc) return rc;
  memcpy(m->ms_info, info, sizeof(info));  // svnicp_map_search_info: the last call that succeeded
  m->ms_info_valid = true;
  return SVNICP_OK;
}

extern "C" int svnicp_map_search_info(svnicp_map m, int64_t out8[8]) {
  if (!m) return SVNICP_ERR_INVALID;
  if (!out8) return mfail(m, SVNICP_ERR_INVALID, "svnicp_map_search_info: null output");
  if (!m->ms_info_valid) return mfail(m, SVNICP_ERR_INVALID, "svnicp_map_search_info: no svnicp_map_search has succeeded on this map yet");
  for (int i = 0; i < 8; i++) out8[i] = m->ms_info[i];
  return SVNICP_OK;
}

// ---- svnicp_map_refine ----------------------------------------------------------------------------------------------------------
// Scratch per pose block of MB poses: x [MB][6], R~ t~ [MB][12], R_p [MB][9], k_eval_fin's output [MB][EV_OUT], the active flags,
// iteration counts and last |delta| (about 640 B per pose), the partials [parts][MB][EV_NS] and the seeds [MB][n][3] float.
enum { RF_X, RF_RT, RF_RP, RF_OUT, RF_ACTIVE, RF_ITERS, RF_STEP, RF_PART, RF_SEEDS, RF_COUNT };
static_assert(RF_COUNT == sizeof(svnicp_map_t::rf) / sizeof(void *), "one scratch buffer per RF_* index");

static int rf_grow(svnicp_map m, int k, size_t bytes) { return ev_grow(m, &m->rf[k], &m->rf_cap[k], bytes > 0 ? bytes : 1); }

extern "C" int svnicp_map_refine(svnicp_map m, const void *source, int64_t n, int dtype_f64, int on_device, const double R0[9],
                                 const double t0[3], int n_poses, const double *poses_6xM, double max_dist, int iterations, double tol,
                                 double *out_poses_6xM, int32_t *out_iterations, double *out_step, double *out_stats, double *out_H,
                                 double *out_b) {
  using svn::EV_BLOCK;
  using svn::EV_NS;
  using svn::EV_OUT;
  if (!m) return SVNICP_ERR_INVALID;
  if (!source || !R0 || !t0 || !poses_6xM || !out_poses_6xM || !out_iterations || !out_stats)
    return mfail(m, SVNICP_ERR_INVALID, "svnicp_map_refine: null source, R0, t0, poses, out_poses, out_iterations or out_stats");
  int rc = check_scan_args(m, "svnicp_map_refine", n, max_dist);
  if (rc) return rc;
  if (n_poses < 1 || n_poses > 65536) return mfail(m, SVNICP_ERR_INVALID, "svnicp_map_refine: n_poses must be in [1, 65536]");
  if (iterations < 1 || iterations > 1000) return mfail(m, SVNICP_ERR_INVALID, "svnicp_map_refine: iterations must be in [1, 1000]");
  if (!isfinite(tol) || tol < 0) return mfail(m, SVNICP_ERR_INVALID, "svnicp_map_refine: tol must be finite and >= 0");
  MCU(cudaSetDevice(m->device));
  cudaStream_t st = m->stream;
  const int ni = (int)n, M = n_poses;
  int parts = (int)((n + MEV_THREADS - 1) / MEV_THREADS);  // svnicp_map_evaluate's partial slots: the same sums
  if (parts > m->sm_count * MEV_CTAS_PER_SM) parts = m->sm_count * MEV_CTAS_PER_SM;
  const size_t per_pose = (size_t)parts * EV_NS * sizeof(double) + (RF_SEED ? (size_t)n * 3 * sizeof(float) : 0);
  const size_t by_bytes = RF_BLOCK_BYTES / per_pose;
  const int mb_max = (int)std::min<size_t>({(size_t)M, (size_t)RF_MAX_BLOCK, std::max<size_t>(by_bytes, 1)});
  const size_t esz = dtype_f64 ? sizeof(double) : sizeof(float);
  const size_t mb = (size_t)mb_max;
  if ((rc = rf_grow(m, RF_X, mb * 6 * sizeof(double))) || (rc = rf_grow(m, RF_RT, mb * 12 * sizeof(double))) ||
      (rc = rf_grow(m, RF_RP, mb * 9 * sizeof(double))) || (rc = rf_grow(m, RF_OUT, mb * EV_OUT * sizeof(double))) ||
      (rc = rf_grow(m, RF_ACTIVE, mb * sizeof(int))) || (rc = rf_grow(m, RF_ITERS, mb * sizeof(int))) ||
      (rc = rf_grow(m, RF_STEP, mb * sizeof(double))) || (rc = rf_grow(m, RF_PART, (size_t)parts * mb * EV_NS * sizeof(double))) ||
      (RF_SEED && (rc = rf_grow(m, RF_SEEDS, mb * (size_t)n * 3 * sizeof(float)))) ||
      (!on_device && (rc = ev_grow(m, &m->ev_src, &m->ev_src_cap, (size_t)n * 3 * esz))))
    return rc;
  const void *src = source;
  if (!on_device) {
    MCU(cudaMemcpyAsync(m->ev_src, source, (size_t)n * 3 * esz, cudaMemcpyHostToDevice, st));
    src = m->ev_src;
  }
  svn::ScanConst sc;
  memcpy(sc.R0, R0, sizeof(sc.R0));
  memcpy(sc.t0, t0, sizeof(sc.t0));
  const MapDev d = dev_view(m, m->cur);
  const double r = sqrt(max_dist) * MEV_MARGIN;  // k_map_eval's radius
  double *x = (double *)m->rf[RF_X], *Rt = (double *)m->rf[RF_RT], *Rp = (double *)m->rf[RF_RP], *ev = (double *)m->rf[RF_OUT];
  double *part = (double *)m->rf[RF_PART], *step = (double *)m->rf[RF_STEP];
  int *active = (int *)m->rf[RF_ACTIVE], *iters = (int *)m->rf[RF_ITERS];
  float *seed = (float *)m->rf[RF_SEEDS];
  std::vector<double> hx(mb * 6), hstep(mb);
  std::vector<int> hit(mb);
  for (int m0 = 0; m0 < M; m0 += mb_max) {
    const int MB = M - m0 < mb_max ? M - m0 : mb_max;
    for (int j = 0; j < MB; j++)
      for (int c = 0; c < 6; c++) hx[(size_t)6 * j + c] = poses_6xM[(size_t)c * M + m0 + j];
    MCU(cudaMemcpyAsync(x, hx.data(), (size_t)6 * MB * sizeof(double), cudaMemcpyHostToDevice, st));
    MCU(cudaMemsetAsync(iters, 0, (size_t)MB * sizeof(int), st));
    if (RF_SEED) MCU(cudaMemsetAsync(seed, 0xFF, (size_t)MB * n * 3 * sizeof(float), st));  // NaN: no seed
    k_fill_i32<<<(MB + 255) / 256, 256, 0, st>>>(active, 1, (size_t)MB);
    for (int j = 0; j < MB; j += EV_BLOCK)
      k_map_eval_prep<<<1, EV_BLOCK, 0, st>>>(x + 6 * j, MB - j < EV_BLOCK ? MB - j : EV_BLOCK, sc, Rt + 12 * j, Rp + 9 * j);
    const dim3 grid((unsigned)parts, (unsigned)MB);
    for (int it = 0; it < iterations; it++) {
      if (dtype_f64) k_map_refine_eval<double><<<grid, MEV_THREADS, 0, st>>>(d, (const double *)src, ni, Rt, sc, max_dist, r, active, part, seed);
      else k_map_refine_eval<float><<<grid, MEV_THREADS, 0, st>>>(d, (const float *)src, ni, Rt, sc, max_dist, r, active, part, seed);
      svn::launch_eval_fin(part, parts, MB, ni, sc, Rp, ev, st);  // a stopped pose's row is stale and unread
      k_map_refine_step<<<(MB + 127) / 128, 128, 0, st>>>(ev, MB, sc, iterations, tol, active, iters, step, x, Rt, Rp);
    }
    MCU(cudaGetLastError());
    MCU(cudaMemcpyAsync(hx.data(), x, (size_t)6 * MB * sizeof(double), cudaMemcpyDeviceToHost, st));
    MCU(cudaMemcpyAsync(hit.data(), iters, (size_t)MB * sizeof(int), cudaMemcpyDeviceToHost, st));
    MCU(cudaMemcpyAsync(hstep.data(), step, (size_t)MB * sizeof(double), cudaMemcpyDeviceToHost, st));
    MCU(cudaStreamSynchronize(st));  // the host block buffers are refilled next
    for (int j = 0; j < MB; j++) {
      for (int c = 0; c < 6; c++) out_poses_6xM[(size_t)c * M + m0 + j] = hx[(size_t)6 * j + c];
      out_iterations[m0 + j] = hit[j];
      if (out_step) out_step[m0 + j] = hstep[j];
    }
  }
  // the statistics and the system at the final poses are svnicp_map_evaluate's by construction: the same call (source on device)
  return svnicp_map_evaluate(m, src, n, dtype_f64, 1, R0, t0, M, out_poses_6xM, max_dist, out_stats, out_H, out_b, nullptr, nullptr);
}

// ---- svnicp_map_export / svnicp_map_import -----------------------------------------------------------------------------------
enum { SN_KEY0, SN_KEY1, SN_SLOT0, SN_SLOT1, SN_OFF, SN_PSUM, SN_HIST, SN_WORDS, SN_VOX, SN_CNT, SN_XYZ, SN_COUNT };
static_assert(SN_COUNT == sizeof(svnicp_map_t::sn) / sizeof(void *), "one scratch buffer per SN_* index");

static int sn_grow(svnicp_map m, int k, size_t bytes) { return ev_grow(m, &m->sn[k], &m->sn_cap[k], bytes > 0 ? bytes : 1); }

// int64 exclusive scan of the V voxels' point counts into sn[SN_OFF] (the table's counts through slots, or a snapshot's counts);
// the total goes to the device word *total
static void launch_point_offsets(svnicp_map m, const int32_t *counts, const int *slots, const int *tab_count, long long V, long long *total) {
  const int nb = (int)((V + SCAN_BLOCK - 1) / SCAN_BLOCK);
  long long *psum = (long long *)m->sn[SN_PSUM], *off = (long long *)m->sn[SN_OFF];
  k_snap_pts_count<<<nb, SCAN_BLOCK, 0, m->stream>>>(counts, slots, tab_count, m->cap, V, psum);
  svn::k_scan_block_sums<long long><<<1, SCAN_BLOCK, 0, m->stream>>>(psum, nb, total);
  k_snap_pts_offsets<<<nb, SCAN_BLOCK, 0, m->stream>>>(counts, slots, tab_count, m->cap, V, psum, off);
}

extern "C" int svnicp_map_export(svnicp_map m, int32_t *voxels, int32_t *counts, float *xyz, int64_t n_voxels, int64_t n_points, int on_device) {
  if (!m) return SVNICP_ERR_INVALID;
  const long long V = m->h_counters[0], N = m->h_counters[1];
  if (n_voxels != V || n_points != N) {
    char buf[256];
    snprintf(buf, sizeof(buf), "svnicp_map_export: n_voxels = %lld and n_points = %lld, but the map holds %lld voxels and %lld points",
             (long long)n_voxels, (long long)n_points, V, N);
    return mfail(m, SVNICP_ERR_INVALID, buf);
  }
  if ((V > 0 && (!voxels || !counts)) || (N > 0 && !xyz)) return mfail(m, SVNICP_ERR_INVALID, "svnicp_map_export: null output");
  if (V == 0) return SVNICP_OK;
  MCU(cudaSetDevice(m->device));
  cudaStream_t st = m->stream;
  const int n_tiles = (int)((V + RADIX_TILE - 1) / RADIX_TILE);
  const int slot_blocks = (int)((m->slots + SCAN_BLOCK - 1) / SCAN_BLOCK);
  const size_t hist_n = (size_t)RADIX_DIGITS * n_tiles > (size_t)slot_blocks ? (size_t)RADIX_DIGITS * n_tiles : (size_t)slot_blocks;
  int rc;
  if ((rc = sn_grow(m, SN_KEY0, V * 8)) || (rc = sn_grow(m, SN_KEY1, V * 8)) || (rc = sn_grow(m, SN_SLOT0, V * 4)) ||
      (rc = sn_grow(m, SN_SLOT1, V * 4)) || (rc = sn_grow(m, SN_OFF, V * 8)) || (rc = sn_grow(m, SN_PSUM, (V / SCAN_BLOCK + 2) * 8)) ||
      (rc = sn_grow(m, SN_HIST, hist_n * 4)) || (rc = sn_grow(m, SN_WORDS, 4 * 8)) ||
      (!on_device && ((rc = sn_grow(m, SN_VOX, V * 12)) || (rc = sn_grow(m, SN_CNT, V * 4)) || (rc = sn_grow(m, SN_XYZ, N * 12)))))
    return rc;
  unsigned long long *key[2] = {(unsigned long long *)m->sn[SN_KEY0], (unsigned long long *)m->sn[SN_KEY1]};
  int *slot[2] = {(int *)m->sn[SN_SLOT0], (int *)m->sn[SN_SLOT1]};
  int *hist = (int *)m->sn[SN_HIST];
  long long *words = (long long *)m->sn[SN_WORDS];  // [0] live slots, [1] their points, [3] sink of the radix scans
  MCU(cudaMemsetAsync(words, 0, 4 * sizeof(long long), st));
  const MapDev d = dev_view(m, m->cur);
  k_snap_count<<<slot_blocks, SCAN_BLOCK, 0, st>>>(d, hist);
  svn::k_scan_block_sums<int><<<1, SCAN_BLOCK, 0, st>>>(hist, slot_blocks, words);
  k_snap_emit<<<slot_blocks, SCAN_BLOCK, 0, st>>>(d, hist, V, key[0], slot[0]);
  for (int shift = 0, a = 0; shift < CANON_BITS; shift += RADIX_BITS, a ^= 1) {
    k_radix_hist<<<n_tiles, RADIX_THREADS, 0, st>>>(key[a], (int)V, shift, n_tiles, hist);
    svn::k_scan_block_sums<int><<<1, SCAN_BLOCK, 0, st>>>(hist, RADIX_DIGITS * n_tiles, words + 3);
    k_radix_scatter<<<n_tiles, RADIX_THREADS, 0, st>>>(key[a], slot[a], key[a ^ 1], slot[a ^ 1], (int)V, shift, n_tiles, hist);
  }
  launch_point_offsets(m, nullptr, slot[0], d.tab.count, V, words + 1);
  int32_t *ov = on_device ? voxels : (int32_t *)m->sn[SN_VOX], *oc = on_device ? counts : (int32_t *)m->sn[SN_CNT];
  float *ox = on_device ? xyz : (float *)m->sn[SN_XYZ];
  k_snap_gather<<<(unsigned)((V * 32 + 255) / 256), 256, 0, st>>>(d.tab, m->cap, key[0], slot[0], (const long long *)m->sn[SN_OFF], V, N, ov, oc, ox);
  MCU(cudaGetLastError());
  if (!on_device) {
    MCU(cudaMemcpyAsync(voxels, ov, (size_t)V * 3 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    MCU(cudaMemcpyAsync(counts, oc, (size_t)V * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (N > 0) MCU(cudaMemcpyAsync(xyz, ox, (size_t)N * 3 * sizeof(float), cudaMemcpyDeviceToHost, st));
  }
  long long h[2];
  MCU(cudaMemcpyAsync(h, words, sizeof(h), cudaMemcpyDeviceToHost, st));
  MCU(cudaStreamSynchronize(st));
  if (h[0] != V || h[1] != N) {
    char buf[256];
    snprintf(buf, sizeof(buf), "svnicp_map_export: the table holds %lld voxels and %lld points, the counters %lld and %lld", h[0], h[1], V, N);
    return mfail(m, SVNICP_ERR_CUDA, buf);
  }
  return SVNICP_OK;
}

extern "C" int svnicp_map_import(svnicp_map m, const int32_t *voxels, const int32_t *counts, const float *xyz, int64_t n_voxels,
                                 int64_t n_points, int on_device) {
  if (!m) return SVNICP_ERR_INVALID;
  char buf[256];
  if (n_voxels < 0 || n_points < 0) return mfail(m, SVNICP_ERR_INVALID, "svnicp_map_import: negative n_voxels or n_points");
  if ((n_voxels > 0 && (!voxels || !counts)) || (n_points > 0 && !xyz)) return mfail(m, SVNICP_ERR_INVALID, "svnicp_map_import: null input");
  const long long V = n_voxels, N = n_points;
  if ((size_t)V > m->slots / 2) {
    snprintf(buf, sizeof(buf), "svnicp_map_import: %lld voxels do not fit a table of %zu voxels; create the map with a larger capacity_voxels",
             V, m->slots / 2);
    return mfail(m, SVNICP_ERR_OOM, buf);
  }
  if (N > V * m->cap) {
    snprintf(buf, sizeof(buf), "svnicp_map_import: n_points = %lld exceeds n_voxels * max_pointscount = %lld, so it is not the sum of the counts",
             N, V * m->cap);
    return mfail(m, SVNICP_ERR_INVALID, buf);
  }
  if (V == 0) return svnicp_map_clear(m);  // N == 0 here
  MCU(cudaSetDevice(m->device));
  cudaStream_t st = m->stream;
  int rc;
  if ((rc = sn_grow(m, SN_SLOT0, V * 4)) || (rc = sn_grow(m, SN_OFF, V * 8)) || (rc = sn_grow(m, SN_PSUM, (V / SCAN_BLOCK + 2) * 8)) ||
      (rc = sn_grow(m, SN_WORDS, 4 * 8)) ||
      (!on_device && ((rc = sn_grow(m, SN_VOX, V * 12)) || (rc = sn_grow(m, SN_CNT, V * 4)) || (rc = sn_grow(m, SN_XYZ, N * 12)))))
    return rc;
  if (!on_device) {
    MCU(cudaMemcpyAsync(m->sn[SN_VOX], voxels, (size_t)V * 3 * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    MCU(cudaMemcpyAsync(m->sn[SN_CNT], counts, (size_t)V * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    if (N > 0) MCU(cudaMemcpyAsync(m->sn[SN_XYZ], xyz, (size_t)N * 3 * sizeof(float), cudaMemcpyHostToDevice, st));
    voxels = (const int32_t *)m->sn[SN_VOX];
    counts = (const int32_t *)m->sn[SN_CNT];
    xyz = (const float *)m->sn[SN_XYZ];
  }
  // build into the twin table (the one RemoveFar rebuilds into); the map's own table, cur and counters stay as they are
  const int nxt = m->cur ^ 1;
  if ((rc = clear_table(m, nxt))) return rc;
  // [0] lowest count / index error, [1] sum of the valid counts, [2] voxels refused, [3] lowest duplicate / membership error
  long long *words = (long long *)m->sn[SN_WORDS];
  MCU(cudaMemsetAsync(words, 0xFF, 4 * sizeof(long long), st));
  MCU(cudaMemsetAsync(words + 1, 0, 2 * sizeof(long long), st));
  launch_point_offsets(m, counts, nullptr, nullptr, V, words + 1);
  const MapDev dn = dev_view(m, nxt);
  int *slot_of = (int *)m->sn[SN_SLOT0];
  k_map_import<<<(unsigned)((V * 32 + 255) / 256), 256, 0, st>>>(dn, voxels, counts, xyz, V, N, (const long long *)m->sn[SN_OFF], slot_of,
                                                                 (unsigned long long *)words);
  const unsigned grid = (unsigned)((V + 255) / 256);
  k_map_import_dups<<<grid, 256, 0, st>>>(m->walker, slot_of, V, (unsigned long long *)words);
  k_map_import_reset<<<grid, 256, 0, st>>>(m->walker, slot_of, V);
  MCU(cudaGetLastError());
  unsigned long long h[4];
  MCU(cudaMemcpyAsync(h, words, sizeof(h), cudaMemcpyDeviceToHost, st));
  MCU(cudaStreamSynchronize(st));
  // the counts and indices first, then their sum (which places the points), then what the points say: each names its lowest voxel
  static const char *why[] = {"", "its count is outside [1, max_pointscount]", "its index is outside [-2^20, 2^20)",
                              "it repeats an earlier voxel", "a point does not belong to it"};
  const bool sum_ok = (long long)h[1] == N;
  const unsigned long long e = h[0] != SNAP_NO_ERROR ? h[0] : sum_ok ? h[3] : SNAP_NO_ERROR;
  if (e != SNAP_NO_ERROR) {
    snprintf(buf, sizeof(buf), "svnicp_map_import: voxel %llu: %s", e >> 3, why[e & 7]);
    return mfail(m, SVNICP_ERR_INVALID, buf);
  }
  if (!sum_ok) {
    snprintf(buf, sizeof(buf), "svnicp_map_import: n_points = %lld, but the counts sum to %lld", N, (long long)h[1]);
    return mfail(m, SVNICP_ERR_INVALID, buf);
  }
  if (h[2] > 0) return mfail(m, SVNICP_ERR_OOM, "svnicp_map_import: the voxel table is full");
  long long size[2] = {V, N};
  MCU(cudaMemcpyAsync(m->counters, size, sizeof(size), cudaMemcpyHostToDevice, st));
  MCU(cudaStreamSynchronize(st));
  m->h_counters[0] = V;
  m->h_counters[1] = N;
  m->cur = nxt;
  return SVNICP_OK;
}
