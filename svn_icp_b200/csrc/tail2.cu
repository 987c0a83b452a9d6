// tail2.cu -- the "Stein phase" of one SVN iteration as two kernels without a grid-wide barrier on the critical path.
//
//   k_head_* (side stream, a chain of small ordinary kernels; overlaps the correspondence + Gauss-Newton pass of the same iteration)
//           early-stop decision for the previous update + its history row          SVNICP.cpp:95-107
//           exact lower median of the P^2 pairwise squared distances -> bandwidth h   SVNICP.cpp:254-266
//           Everything here depends only on the particle positions x, which are final as soon as the previous update is.
//           The SVGD-ICP class runs the same chain on its main stream, on the gathered record (svgd_class.cu).
//   k_tail  (main stream, ordinary launch, one CTA per NI particles)
//           Stein step: full SVN / pre-conditioned SVGD / P == 1                    SVNICP.cpp:218-252, 88-89
//           pose update                                                             SVNICP.cpp:268-279
//           next iteration's x = [t ; Log R], fp32 transforms, exact-pruning ball   SVNICP.cpp:58-59,74-77
//           Records of all particles stream through shared memory as AoS tiles (1-D bulk TMA + mbarrier ring); the CTA
//           that finishes last publishes the ball and the iteration counter.
//
// Sharded handles: k_finalize stores (b, H, g) and k_tail stores (x, |delta|) of the local particles straight into every
// rank's record buffer over NVLink (PeerTable, common.cuh), followed by a sequence number in the peer's flag block; k_tail /
// k_head spin on their local flags.  Records are double buffered by iteration parity, which is what makes the exchange
// safe without a second handshake (see DESIGN.md section 5).  No NCCL call on the per-iteration path.
#include "block_scan.cuh"
#include "common.cuh"
#include "kernels.h"
#include "ptx.cuh"

namespace svn {

// ---------------------------------------------------------------------------------------------
// k_head_*: a chain of ordinary (non-cooperative) kernels on the side stream.  Each has a small footprint (128 threads,
// <= 64 registers, 32 KB of shared memory) so that one CTA fits on every SM NEXT TO the two resident CTAs of k_gn and the
// chain never pushes k_gn's persistent single-wave grid into a second wave; phases that need all CTAs to be done are
// separated by kernel boundaries, and the CTA that finishes last (ticket) does the serial part.
//   k_head_prep    peers' x arrived? -> early-stop decision for the previous update, its history row, SoA copy of x,
//                  reset of the median scratch
//   k_head_fast1/2 the median moves little between iterations: histogram LINEARLY around the previous one (8190 bins over
//                  [0.5, 1.5) x previous median, one bin below, one above); then gather the few dozen values of the bin that
//                  holds the rank and pick the exact order statistic.  Same value as the radix select (the lower median is
//                  unique), so the bandwidth is bit-identical to the 5-pass path
//   k_head_radix   x 5: exact radix select on the fp64 bit pattern (11 + 13 + 13 + 13 + 13 bits); returns at once when the fast
//                  path already produced the median (first iteration of a scan, tiny particle sets and misses take this path)
// (An earlier version was ONE cooperative kernel with grid-wide barriers; with the host blocked in cudaStreamSynchronize on the
// main stream, the cooperative launch on the side stream did not start on small problems -- a hang that disappeared when the host
// polled instead.  Plain launches have no such dependence.)
// ---------------------------------------------------------------------------------------------
constexpr int HD_THREADS = 128;
constexpr int HD_WARPS = HD_THREADS / 32;
constexpr int HD_COLLECT_CAP = 4096;  // doubles staged in the 32 KB histogram buffer
static_assert(HD_COLLECT_CAP * sizeof(double) <= MED_BINS * sizeof(unsigned), "collected values are staged in the histogram buffer");
// how the median of an iteration was settled, recorded in SteinArgs::med_path[iter] (svnicp_get_median_paths)
enum { MED_PATH_SORT = 0,      // k_head_small: sort of all pairs (P <= HD_SMALL_P)
       MED_PATH_FAST = 1,      // k_head_fast1/2: linear histogram around the previous median, then the bin's values
       MED_PATH_RADIX = 2,     // k_head_radix: no fast path this iteration (iteration 0, no usable previous median) or a window miss
       MED_PATH_OVERFLOW = 3 };  // k_head_radix after the fast path found the bin but could not pick (more than HD_COLLECT_CAP values)

__device__ __forceinline__ int hd_pass_bits(int s) { return s == 0 ? 11 : 13; }
__device__ __forceinline__ int hd_bits_before(int s) { return s == 0 ? 0 : 11 + 13 * (s - 1); }

// (prefix, rank) after a pass from its finished global histogram (run by the last CTA of the pass)
__device__ void hd_select(const unsigned *hist, unsigned long long prefix_in, unsigned long long rank_in, int nbins, int bits,
                          unsigned long long *prefix_out, unsigned long long *rank_out, unsigned long long *s_warp,
                          unsigned long long *s_res) {
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5;
  const int per = (nbins + nt - 1) / nt;  // contiguous run of bins per thread (64 for 8192 bins)
  unsigned long long loc = 0;
  for (int i0 = 0; i0 < per; i0 += 16) {  // 16 loads in flight at a time
    unsigned v[16];
#pragma unroll
    for (int u = 0; u < 16; u++) {
      const int b = tid * per + i0 + u;
      v[u] = (i0 + u < per && b < nbins) ? __ldcg(hist + b) : 0u;
    }
#pragma unroll
    for (int u = 0; u < 16; u++) loc += v[u];
  }
  const unsigned long long incl = warp_inclusive_scan(loc);
  if (lane == 31) s_warp[warp] = incl;
  if (tid == 0) { s_res[0] = (prefix_in << bits) | (unsigned long long)(nbins - 1); s_res[1] = 0ull; }
  __syncthreads();
  unsigned long long wbase = 0;
  for (int w = 0; w < warp; w++) wbase += s_warp[w];
  const unsigned long long excl = wbase + incl - loc;
  if (loc > 0 && excl <= rank_in && rank_in < excl + loc) {  // exactly one thread owns the rank: it walks its (cache-hot) run again
    unsigned long long cum = excl;
    int b = tid * per;
    for (int i = 0; i < per; i++) {
      const unsigned v = (tid * per + i < nbins) ? __ldcg(hist + tid * per + i) : 0u;
      if (cum + v > rank_in) break;
      cum += v;
      b = tid * per + i + 1;
    }
    s_res[0] = (prefix_in << bits) | (unsigned long long)b;
    s_res[1] = rank_in - cum;
  }
  __syncthreads();
  *prefix_out = s_res[0];
  *rank_out = s_res[1];
  __syncthreads();
}

// true in exactly one CTA: the one that finishes last.  All global writes of the other CTAs are visible to it.
__device__ __forceinline__ bool hd_last_cta(unsigned *ticket, int *s_flag) {
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) *s_flag = (atomicAdd(ticket, 1u) == gridDim.x - 1) ? 1 : 0;
  __syncthreads();
  if (!*s_flag) return false;
  __threadfence();
  return true;
}

__global__ void __launch_bounds__(HD_THREADS, 8) k_head_prep(SteinArgs a, PeerTable pt, unsigned seq_x, int epilogue) {
  Ctrl *c = a.ctrl;
  if (c->stop) return;  // set by an earlier launch: identical for every CTA
  __shared__ double s_red[HD_WARPS];
  __shared__ int s_stop;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int gtid = blockIdx.x * blockDim.x + tid, gn = gridDim.x * blockDim.x;
  const int P = a.P;
  // x of every particle after the previous update must have arrived (the first iteration's x is computed locally by k_prep)
  if (seq_x) peer_wait(pt, FLAG_X, seq_x, c);
  const int it = c->iter;
  const double *rec = a.rec + (size_t)(it & 1) * a.rec_stride;
  // decide (redundantly per CTA: same data, same order)
  double s = 0.0;
  for (int p = tid; p < P; p += blockDim.x) s += __ldcg(rec + (size_t)p * REC + REC_DNORM);
  s = warp_sum(s);
  if (lane == 0) s_red[warp] = s;
  __syncthreads();
  if (tid == 0) {
    double tot = 0.0;
    for (int w = 0; w < HD_WARPS; w++) tot += s_red[w];
    s_stop = (a.check_early_stop && it > 0 && tot / (double)P < a.threshold) ? 1 : 0;  // SVNICP.cpp:95-101
  }
  __syncthreads();
  const bool stop = s_stop != 0;
  if (!stop && it > 0 && it - 1 < a.I) {  // the history row of a stopping iteration is NOT written (Q9)
    float *row = a.history + (size_t)(it - 1) * 6 * P;  // SVNICP.cpp:103-107
    for (int i = gtid; i < 6 * P; i += gn) {
      const int comp = i / P, p = i % P;
      row[i] = (float)__ldcg(rec + (size_t)p * REC + REC_X + comp);
    }
  }
  if (!stop && !epilogue && P >= 2) {
    for (int i = gtid; i < 6 * P; i += gn) {
      const int comp = i / P, p = i % P;
      a.xs[i] = __ldcg(rec + (size_t)p * REC + REC_X + comp);
    }
    for (int i = gtid; i < 2 * MED_PASSES * MED_BINS; i += gn) a.hist[i] = 0u;  // fast-path scratch + radix histograms
  }
  if (gtid == 0) {
    // Ctrl is written last and by one thread: every CTA of this launch has read `stop` at its top (possibly still 0), and the
    // decision above does not depend on it
    if (stop) { c->stop = 1; c->iters_done = it; }
    else if (epilogue) c->iters_done = it;
    c->med_done = 0;
    c->fast_bin = 0ull;
    c->fast_rank = 0ull;
    c->fast_ticket[0] = c->fast_ticket[1] = 0u;
    for (int q = 0; q < MED_PASSES; q++) c->med_ticket[q] = 0u;
    c->sel_prefix[0] = 0ull;
    c->sel_rank[0] = ((unsigned long long)P * (unsigned long long)P - 1ull) / 2ull;  // lower median
  }
}

// ---- the pair sweeps, shared by the multi-CTA chain and the single-CTA kernel (cta / n_cta: this CTA's share of the rows) ----
struct HdWindow {  // linear histogram window of the fast path: [0.5, 1.5) x the previous median
  double lo, hi, scale;
  __device__ __forceinline__ unsigned bin(double d2) const {  // monotone non-decreasing in d; NaN sorts last like its bit pattern
    if (d2 < lo) return 0u;
    if (!(d2 < hi)) return (unsigned)(MED_BINS - 1);
    return 1u + (unsigned)min((int)((d2 - lo) * scale), MED_BINS - 3);
  }
};
__device__ __forceinline__ HdWindow hd_window(double med_guess) {
  HdWindow w;
  w.lo = 0.5 * med_guess; w.hi = 1.5 * med_guess; w.scale = (double)(MED_BINS - 2) / (w.hi - w.lo);
  return w;
}
// lanes that fall into the same bin are aggregated with match.any before the shared-memory atomic
__device__ __forceinline__ void hd_hist_add(unsigned *s_hist, bool on, unsigned bin, int lane) {
  const unsigned mm = __ballot_sync(0xffffffffu, on);
  if (on) {
    const unsigned peers = __match_any_sync(mm, bin);
    if ((peers & ((1u << lane) - 1u)) == 0) atomicAdd(&s_hist[bin], 2u * (unsigned)__popc(peers));  // D_ij = D_ji: counted twice
  }
}
// Upper-triangle sweep shared by all passes: CTA `cta` of `n_cta` takes rows i = cta, cta + n_cta, ...; x_i stays in registers and
// four pairs per thread are in flight before `f(valid, d2)` consumes them (the passes are latency bound: one pair at a time left
// the fp64 pipe 2 % busy).  f is called by all 32 lanes of a warp together (it may vote).
template <class F>
__device__ __forceinline__ void hd_sweep(const double *__restrict__ X, int P, int cta, int n_cta, F &&f) {
  const int tid = threadIdx.x, nt = blockDim.x;
  for (int i = cta; i < P; i += n_cta) {
    double xi[6];
#pragma unroll
    for (int d = 0; d < 6; d++) xi[d] = X[d * P + i];
    for (int j0 = i + 1; j0 < P; j0 += 4 * nt) {
      double d2[4];
      bool on[4];
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const int j = j0 + u * nt + tid;
        on[u] = j < P;
        double s = 0.0;
        if (on[u]) {
          double df[6];
#pragma unroll
          for (int d = 0; d < 6; d++) df[d] = xi[d] - X[d * P + j];
          // SVNICP.cpp:257-260, rounding spelled out: this is what nvcc made of `s += df * df` from s = 0 (it fused the first
          // square into the second), written as explicit fma so that the order cannot change with the compiler and the CPU
          // oracle (oracle_pair_median_kernel_order) can restate the exact values the median is selected from
          s = fma(df[0], df[0], df[1] * df[1]);
#pragma unroll
          for (int d = 2; d < 6; d++) s = fma(df[d], df[d], s);
        }
        d2[u] = s;
      }
#pragma unroll
      for (int u = 0; u < 4; u++)
        if (j0 + u * nt < P) f(on[u], d2[u]);  // warp-uniform guard
    }
  }
}
__device__ void hd_fast_hist(const double *X, int P, const HdWindow &w, unsigned *s_hist, int cta, int n_cta) {
  const int lane = threadIdx.x & 31;
  hd_sweep(X, P, cta, n_cta, [&](bool on, double d2) { hd_hist_add(s_hist, on, on ? w.bin(d2) : 0u, lane); });
  if (cta == 0 && threadIdx.x == 0) atomicAdd(&s_hist[0], (unsigned)P);  // the diagonal: exact zeros, below lo
}
// values of bin tbin, once per unordered pair (each stands for two entries of the P x P matrix)
__device__ void hd_fast_gather(const double *X, int P, const HdWindow &w, unsigned tbin, double *list, unsigned *cursor, int cta, int n_cta) {
  hd_sweep(X, P, cta, n_cta, [&](bool on, double d2) {
    if (on && w.bin(d2) == tbin) {
      const unsigned k = atomicAdd(cursor, 1u);
      if (k < (unsigned)HD_COLLECT_CAP) list[k] = d2;
    }
  });
}
// exact order statistic `target` (ascending, among the n_c collected values) -> *out; returns false if none found (cannot happen)
__device__ bool hd_pick(const double *s_list, unsigned n_c, unsigned target, unsigned long long *s_val, int *s_found, double *out) {
  if (threadIdx.x == 0) *s_found = 0;
  __syncthreads();
  for (unsigned k = threadIdx.x; k < n_c; k += blockDim.x) {
    const double v = s_list[k];
    unsigned less = 0, eq = 0;
    for (unsigned u = 0; u < n_c; u++) {
      const double x = s_list[u];
      less += (x < v) ? 1u : 0u;
      eq += (x == v) ? 1u : 0u;
    }
    if (less <= target && target < less + eq) { *s_val = (unsigned long long)__double_as_longlong(v); *s_found = 1; }
  }
  __syncthreads();
  if (*s_found) *out = __longlong_as_double((long long)*s_val);
  return *s_found != 0;
}
// one radix pass: upper triangle, D_ij = D_ji counted twice, diagonal once (exact zeros: key 0)
__device__ void hd_radix_hist(const double *X, int P, int s, unsigned long long prefix, unsigned *s_hist, int cta, int n_cta) {
  const int lane = threadIdx.x & 31;
  const int consumed = hd_bits_before(s), nb = 1 << hd_pass_bits(s);
  const int shift = 63 - consumed - hd_pass_bits(s);
  const unsigned bmask = (unsigned)(nb - 1);
  hd_sweep(X, P, cta, n_cta, [&](bool on, double d2) {
    const unsigned long long key = (unsigned long long)__double_as_longlong(d2);
    const bool match = on && ((consumed == 0) || ((key >> (63 - consumed)) == prefix));
    hd_hist_add(s_hist, match, (unsigned)(key >> shift) & bmask, lane);
  });
  if (cta == 0 && threadIdx.x == 0 && (consumed == 0 || prefix == 0ull)) atomicAdd(&s_hist[0], (unsigned)P);
}

__global__ void __launch_bounds__(HD_THREADS, 8) k_head_fast1(SteinArgs a) {
  Ctrl *c = a.ctrl;
  const int P = a.P, it = c->iter;
  if (c->stop || P < 8 || it == 0) return;
  const double med_guess = c->bandwidth * log((double)(P + 1));  // previous iteration's median
  if (!(med_guess > 0.0 && med_guess < INFINITY)) return;
  __shared__ __align__(16) unsigned s_hist[MED_BINS];
  __shared__ unsigned long long s_warp[32], s_res[2];
  __shared__ int s_flag;
  const int tid = threadIdx.x;
  for (int i = tid; i < MED_BINS; i += blockDim.x) s_hist[i] = 0u;
  __syncthreads();
  hd_fast_hist(a.xs, P, hd_window(med_guess), s_hist, blockIdx.x, gridDim.x);
  __syncthreads();
  for (int i = tid; i < MED_BINS; i += blockDim.x)
    if (s_hist[i]) atomicAdd(&a.hist[i], s_hist[i]);
  if (!hd_last_cta(&c->fast_ticket[0], &s_flag)) return;
  unsigned long long tbin = 0ull, trank = 0ull;
  hd_select(a.hist, 0ull, ((unsigned long long)P * (unsigned long long)P - 1ull) / 2ull, MED_BINS, 13, &tbin, &trank, s_warp, s_res);
  if (tid == 0) { c->fast_bin = tbin; c->fast_rank = trank; }
}

__global__ void __launch_bounds__(HD_THREADS, 8) k_head_fast2(SteinArgs a) {
  Ctrl *c = a.ctrl;
  const int P = a.P;
  if (c->stop || P < 8) return;
  const unsigned long long tbin = c->fast_bin;
  if (tbin == 0ull || tbin == (unsigned long long)(MED_BINS - 1)) return;  // no fast path this iteration, or the median left the window
  __shared__ __align__(16) double s_list[HD_COLLECT_CAP];
  __shared__ int s_flag, s_found;
  __shared__ unsigned long long s_val;
  const int tid = threadIdx.x;
  unsigned *cursor = a.hist + MED_BINS;                              // zeroed by k_head_prep
  double *list = reinterpret_cast<double *>(a.hist + 2 * MED_BINS);  // rows 2..4: 12288 doubles
  hd_fast_gather(a.xs, P, hd_window(c->bandwidth * log((double)(P + 1))), (unsigned)tbin, list, cursor, blockIdx.x, gridDim.x);
  if (!hd_last_cta(&c->fast_ticket[1], &s_flag)) return;
  const unsigned n_c = __ldcg(cursor);
  if (n_c < 1u || n_c > (unsigned)HD_COLLECT_CAP) return;  // degenerate bin: the radix passes take over
  for (unsigned k = tid; k < n_c; k += blockDim.x) s_list[k] = __ldcg(list + k);
  double median = 0.0;
  // index among the distinct pairs of the bin, ascending: every value stands for two entries of the matrix
  if (hd_pick(s_list, n_c, (unsigned)(c->fast_rank >> 1), &s_val, &s_found, &median) && tid == 0) {
    c->bandwidth = median / log((double)(P + 1));  // SVNICP.cpp:262 (Q4)
    c->med_done = 1;
    if (a.med_path) a.med_path[c->iter] = MED_PATH_FAST;
  }
}

// one radix-select pass; the last CTA turns the histogram into the next (prefix, rank) and, after the final pass, into the bandwidth
__global__ void __launch_bounds__(HD_THREADS, 8) k_head_radix(SteinArgs a, int s) {
  Ctrl *c = a.ctrl;
  const int P = a.P;
  if (c->stop || c->med_done || P < 2) return;
  __shared__ __align__(16) unsigned s_hist[MED_BINS];
  __shared__ unsigned long long s_warp[32], s_res[2];
  __shared__ int s_flag;
  const int tid = threadIdx.x;
  const unsigned long long prefix = c->sel_prefix[s];
  const int nb = 1 << hd_pass_bits(s);
  for (int i = tid; i < nb; i += blockDim.x) s_hist[i] = 0u;
  __syncthreads();
  hd_radix_hist(a.xs, P, s, prefix, s_hist, blockIdx.x, gridDim.x);
  __syncthreads();
  unsigned *gh = a.hist + (size_t)(MED_PASSES + s) * MED_BINS;  // the radix histograms sit behind the fast-path scratch
  for (int i = tid; i < nb; i += blockDim.x)
    if (s_hist[i]) atomicAdd(&gh[i], s_hist[i]);
  if (!hd_last_cta(&c->med_ticket[s], &s_flag)) return;
  unsigned long long np, nr;
  hd_select(gh, prefix, c->sel_rank[s], nb, hd_pass_bits(s), &np, &nr, s_warp, s_res);
  if (tid == 0) {
    c->sel_prefix[s + 1] = np;
    c->sel_rank[s + 1] = nr;
    if (s == MED_PASSES - 1) {
      c->bandwidth = __longlong_as_double((long long)np) / log((double)(P + 1));  // SVNICP.cpp:262 (Q4)
      const bool miss = c->fast_bin == 0ull || c->fast_bin == (unsigned long long)(MED_BINS - 1);
      if (a.med_path) a.med_path[c->iter] = miss ? MED_PATH_RADIX : MED_PATH_OVERFLOW;
    }
  }
}

// Small particle sets (P <= HD_SMALL_P): the whole chain in ONE CTA -- one launch instead of eight, no inter-CTA hand-over.
// Same decision, same history row, same pair distances (hd_sweep); the median comes from a sort of all pairs in shared memory.
constexpr int HD_SMALL_P = 64;  // one CTA of 128 threads: 2016 pairs; beyond that the chain over many CTAs is faster (measured at 100 and 256)
__global__ void __launch_bounds__(HD_THREADS, 8) k_head_small(SteinArgs a, PeerTable pt, unsigned seq_x, int epilogue) {
  Ctrl *c = a.ctrl;
  if (c->stop) return;
  __shared__ __align__(16) unsigned s_hist[MED_BINS];      // the pair distances as 64-bit keys (32 KB = 4096 slots)
  __shared__ __align__(16) double s_x[6 * HD_SMALL_P];     // 3 KB
  __shared__ double s_red[HD_WARPS];
  __shared__ unsigned s_cursor;
  __shared__ int s_stop;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int P = a.P;
  if (seq_x) peer_wait(pt, FLAG_X, seq_x, c);
  const int it = c->iter;
  const double *rec = a.rec + (size_t)(it & 1) * a.rec_stride;
  double s = 0.0;
  for (int p = tid; p < P; p += blockDim.x) s += __ldcg(rec + (size_t)p * REC + REC_DNORM);
  s = warp_sum(s);
  if (lane == 0) s_red[warp] = s;
  __syncthreads();
  if (tid == 0) {
    double tot = 0.0;
    for (int w = 0; w < HD_WARPS; w++) tot += s_red[w];
    const int stop = (a.check_early_stop && it > 0 && tot / (double)P < a.threshold) ? 1 : 0;  // SVNICP.cpp:95-101
    s_stop = stop;
    if (stop) { c->stop = 1; c->iters_done = it; }
    else if (epilogue) c->iters_done = it;
  }
  __syncthreads();
  if (s_stop) return;  // break BEFORE the history row of that iteration (Q9)
  for (int i = tid; i < 6 * P; i += blockDim.x) {
    const int comp = i / P, p = i % P;
    const double v = __ldcg(rec + (size_t)p * REC + REC_X + comp);
    s_x[i] = v;
    if (!epilogue) a.xs[i] = v;  // x at the head of the last executed iteration (svnicp_get_gn_system, SVGD-ICP class)
    if (it > 0 && it - 1 < a.I) a.history[(size_t)(it - 1) * 6 * P + i] = (float)v;  // SVNICP.cpp:103-107
  }
  if (epilogue || P < 2) return;
  __syncthreads();
  // P <= 64: at most 2016 unordered pairs.  Sort them (bitonic network in shared memory; keys = bit patterns: non-negative
  // doubles order like their bits and NaN sorts last -- exactly the order the radix select of the multi-CTA chain uses) and
  // read the order statistic off: the P x P matrix holds P exact zeros and every pair twice.  ~2 us at P = 30 (the histogram
  // passes this replaces took 43 us on average and sat on the critical path of small scans).
  unsigned long long *s_key = reinterpret_cast<unsigned long long *>(s_hist);  // MED_BINS / 2 = 4096 slots
  const unsigned n_c = (unsigned)(P * (P - 1) / 2);
  unsigned n2 = 2u;
  while (n2 < n_c) n2 <<= 1;
  if (tid == 0) s_cursor = 0u;
  for (unsigned i = n_c + tid; i < n2; i += blockDim.x) s_key[i] = ~0ull;
  __syncthreads();
  hd_sweep(s_x, P, 0, 1, [&](bool on, double d2) {
    if (on) s_key[atomicAdd(&s_cursor, 1u)] = (unsigned long long)__double_as_longlong(d2);
  });
  __syncthreads();
  for (unsigned k = 2u; k <= n2; k <<= 1)
    for (unsigned j = k >> 1; j > 0u; j >>= 1) {
      for (unsigned i = tid; i < n2; i += blockDim.x) {
        const unsigned o = i ^ j;
        if (o > i) {
          const unsigned long long u = s_key[i], v = s_key[o];
          if (((i & k) == 0u) ? (u > v) : (u < v)) { s_key[i] = v; s_key[o] = u; }
        }
      }
      __syncthreads();
    }
  if (tid == 0) {
    const unsigned long long rank0 = ((unsigned long long)P * (unsigned long long)P - 1ull) / 2ull;  // lower median of P^2 entries
    const unsigned long long key = rank0 < (unsigned long long)P ? 0ull : s_key[(rank0 - (unsigned long long)P) / 2ull];
    c->bandwidth = __longlong_as_double((long long)key) / log((double)(P + 1));  // SVNICP.cpp:262 (Q4)
    if (a.med_path) a.med_path[it] = MED_PATH_SORT;
  }
}

// ---------------------------------------------------------------------------------------------
// k_tail
// ---------------------------------------------------------------------------------------------
constexpr int TL_CONSUMERS = 256;
constexpr int TL_WARPS = TL_CONSUMERS / 32;
constexpr int TL_THREADS = TL_CONSUMERS + 32;  // + one producer warp (bulk TMA)
constexpr int TL_ENV_CHUNK = 1024;             // particles per pass of the envelope reduction (last CTA)

// dynamic shared memory: [stages][tile_records * REC] doubles, then the mbarriers
// MODE: 0 = single particle (Gauss-Newton step), 1 = full SVN, 2 = pre-conditioned SVGD.  A template parameter, not a run-time
// branch: each instantiation carries only its own code (the three modes together were 15k instructions, and the single-thread
// sections of this kernel run cold -- instruction fetch is what they cost)
template <int MODE>
__global__ void __launch_bounds__(TL_THREADS, 1) k_tail(SteinArgs a, IterArgs ia, PeerTable pt, unsigned seq_h, unsigned seq_x_out, int NI,
                                                        int JQ, int stages) {
  Ctrl *c = a.ctrl;
  if (c->stop) return;  // decided by k_head of this iteration (ordered before this launch) or earlier
  extern __shared__ __align__(128) unsigned char s_dyn[];
  __shared__ double s_part[TL_WARPS][28];
  __shared__ double s_Hbar[TL_WARPS][21];
  __shared__ double s_Hinv[36];
  __shared__ double s_xf[TL_WARPS][12];
  __shared__ float s_center[12];
  __shared__ int s_envmax[4][PRUNE_BINS];
  __shared__ int s_ab[2];
  __shared__ int s_flag[2];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int P = a.P;
  // phase stamps (ns, tuning aid): CTA 0 stamps 0..3, the last CTA 4..5
#define TL_STAMP(k) do { if (a.stamps && tid == 0) a.stamps[k] = (double)global_timer_ns(); } while (0)
  if (blockIdx.x == 0) TL_STAMP(0);
  const int TJ = 32 * JQ;                                   // records per tile
  const size_t tile_bytes = (size_t)TJ * REC * sizeof(double);
  uint64_t *full = reinterpret_cast<uint64_t *>(s_dyn + (size_t)stages * tile_bytes);
  uint64_t *empty = full + stages;
  const int n_tiles = (P + TJ - 1) / TJ;

  if (tid == 0) {
    for (int s = 0; s < stages; s++) { mbar_init(full + s, 1); mbar_init(empty + s, TL_WARPS); }
    fence_barrier_init();
  }
  // (b, H, g) of every particle must have arrived; x arrived before k_head of this iteration ran
  peer_wait(pt, FLAG_H, seq_h, c);  // ends with __syncthreads: also publishes the barrier init
  const int it = c->iter;
  const double *rec = a.rec + (size_t)(it & 1) * a.rec_stride;
  const size_t nxt_off = (size_t)((it + 1) & 1) * a.rec_stride;
  const double h = c->bandwidth;
  if (blockIdx.x == 0) TL_STAMP(1);

  if (warp == TL_WARPS) {
    // ---------------- producer warp: AoS record tiles, one bulk copy each ----------------
    if (MODE != 0)
      for (int t = 0; t < n_tiles; t++) {
        const int s = t % stages, k = t / stages;
        mbar_wait_backoff(empty + s, (uint32_t)((k & 1) ^ 1));
        if (lane == 0) {
          mbar_expect_tx(full + s, (uint32_t)tile_bytes);
          bulk_g2s(s_dyn + (size_t)s * tile_bytes, rec + (size_t)t * TJ * REC, (uint32_t)tile_bytes, full + s);
        }
        __syncwarp();
      }
  } else {
    // ---------------- consumers: warp = (particle ii, j-quarter jq); lane = j ----------------
    const int ii = warp / JQ, jq = warp % JQ;
    const int l = blockIdx.x * NI + ii;
    const bool active = ii < NI && l < a.P_l;
    const int i = a.p_lo + (active ? l : 0);
    SVN_CHECK(c, i < P && (size_t)n_tiles * TJ * REC <= a.rec_stride && NI * JQ == TL_WARPS, 30);
    double xi[6];
#pragma unroll
    for (int d = 0; d < 6; d++) xi[d] = __ldcg(rec + (size_t)i * REC + REC_X + d);
    if constexpr (MODE == 1) {
      double Hm[21], v[6];
#pragma unroll
      for (int q = 0; q < 21; q++) Hm[q] = 0.0;
#pragma unroll
      for (int q = 0; q < 6; q++) v[q] = 0.0;
      const double two_over_h = 2.0 / h;
      for (int t = 0; t < n_tiles; t++) {
        const int s = t % stages, k = t / stages;
        mbar_wait(full + s, (uint32_t)(k & 1));
        const double *tile = reinterpret_cast<const double *>(s_dyn + (size_t)s * tile_bytes);
        const int jj = jq * 32 + lane;
        if (active && t * TJ + jj < P) {
          const double *r = tile + (size_t)jj * REC;
          double dl[6], D = 0.0;
#pragma unroll
          for (int d = 0; d < 6; d++) { dl[d] = xi[d] - r[REC_X + d]; D += dl[d] * dl[d]; }
          const double kij = exp(-D / h);  // :264
          const double k2 = kij * kij;     // :238
          double gv[6];
#pragma unroll
          for (int d = 0; d < 6; d++) gv[d] = two_over_h * (dl[d] * kij);  // :233
          int q = 0;
#pragma unroll
          for (int rr = 0; rr < 6; rr++)
#pragma unroll
            for (int cc = rr; cc < 6; cc++, q++) Hm[q] += k2 * r[REC_H + q] + gv[rr] * gv[cc];  // :236-242
#pragma unroll
          for (int d = 0; d < 6; d++) v[d] += gv[d] - kij * r[REC_B + d];  // :244 with b' = -b
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(empty + s);
      }
#pragma unroll
      for (int q = 0; q < 21; q++) Hm[q] = warp_sum(Hm[q]);
#pragma unroll
      for (int q = 0; q < 6; q++) v[q] = warp_sum(v[q]);
      if (lane == 0) {
#pragma unroll
        for (int q = 0; q < 21; q++) s_part[warp][q] = Hm[q];
#pragma unroll
        for (int q = 0; q < 6; q++) s_part[warp][21 + q] = v[q];
      }
    } else if constexpr (MODE == 2) {
      // pre-conditioned SVGD (SVNICP.cpp:85, :218-227); the warps of particle 0 of the CTA also sum H over all j (mean Hessian)
      double gs[6], kn[6], ks = 0.0, Hs[21];
#pragma unroll
      for (int d = 0; d < 6; d++) { gs[d] = 0.0; kn[d] = 0.0; }
#pragma unroll
      for (int q = 0; q < 21; q++) Hs[q] = 0.0;
      for (int t = 0; t < n_tiles; t++) {
        const int s = t % stages, k = t / stages;
        mbar_wait(full + s, (uint32_t)(k & 1));
        const double *tile = reinterpret_cast<const double *>(s_dyn + (size_t)s * tile_bytes);
        const int jj = jq * 32 + lane;
        if (t * TJ + jj < P) {
          const double *r = tile + (size_t)jj * REC;
          if (ii == 0) {
#pragma unroll
            for (int q = 0; q < 21; q++) Hs[q] += r[REC_H + q];
          }
          if (active) {
            double dl[6], D = 0.0;
#pragma unroll
            for (int d = 0; d < 6; d++) { dl[d] = xi[d] - r[REC_X + d]; D += dl[d] * dl[d]; }
            const double kij = exp(-D / h);
            ks += kij;  // :226
#pragma unroll
            for (int d = 0; d < 6; d++) { gs[d] += dl[d] * kij; kn[d] -= kij * r[REC_G + d]; }  // :221-224
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(empty + s);
      }
      ks = warp_sum(ks);
#pragma unroll
      for (int d = 0; d < 6; d++) { gs[d] = warp_sum(gs[d]); kn[d] = warp_sum(kn[d]); }
      if (ii == 0) {
#pragma unroll
        for (int q = 0; q < 21; q++) Hs[q] = warp_sum(Hs[q]);
      }
      if (lane == 0) {
#pragma unroll
        for (int d = 0; d < 6; d++) { s_part[warp][d] = gs[d]; s_part[warp][6 + d] = kn[d]; }
        s_part[warp][12] = ks;
        if (ii == 0)
#pragma unroll
          for (int q = 0; q < 21; q++) s_Hbar[jq][q] = Hs[q];
      }
    }
  }
  __syncthreads();
  if (blockIdx.x == 0) TL_STAMP(2);
  if (MODE == 2 && tid == 0) {
    double A0[36];
#pragma unroll
    for (int r = 0; r < 6; r++)
#pragma unroll
      for (int cc = r; cc < 6; cc++) {
        double s = 0.0;
        for (int w = 0; w < JQ; w++) s += s_Hbar[w][tri(r, cc)];
        A0[6 * r + cc] = s * (1.0 / (double)P);  // :85 mean over particles
        A0[6 * cc + r] = A0[6 * r + cc];
      }
    // :225 inverse, column by column; the loop stays rolled (six unrolled solves were 1800 instructions of cold code on the
    // critical path of every CTA -- instruction fetch, not arithmetic, is what this single-thread section costs)
#pragma unroll 1
    for (int col = 0; col < 6; col++) {
      double A[36], e[6];
#pragma unroll
      for (int q = 0; q < 36; q++) A[q] = A0[q];
#pragma unroll
      for (int q = 0; q < 6; q++) e[q] = (q == col) ? 1.0 : 0.0;
      ldl_solve6_reg(A, e);
#pragma unroll
      for (int q = 0; q < 6; q++) s_Hinv[6 * q + col] = e[q];
    }
  }
  if (MODE == 2) __syncthreads();

  // ---------------- one thread per particle: solve, pose update, head of the next iteration ----------------
  const double *R0 = ia.sc.R0;
  const double inv_P = 1.0 / (double)P;
  if (warp < TL_WARPS && lane == 0 && (warp % JQ) == 0) {
    const int ii = warp / JQ;
    const int l = blockIdx.x * NI + ii;
    double xfd[12];
#pragma unroll
    for (int k = 0; k < 12; k++) xfd[k] = 0.0;
    if (ii < NI && l < a.P_l) {
      const int p = a.p_lo + l;
      double d[6];
      if constexpr (MODE == 0) {  // SVNICP.cpp:88-89
        double A[36];
        const double *r = rec + (size_t)p * REC;
#pragma unroll
        for (int rr = 0; rr < 6; rr++)
#pragma unroll
          for (int cc = rr; cc < 6; cc++) { A[6 * rr + cc] = __ldcg(r + REC_H + tri(rr, cc)); A[6 * cc + rr] = A[6 * rr + cc]; }
#pragma unroll
        for (int q = 0; q < 6; q++) d[q] = __ldcg(r + REC_B + q);
        ldl_solve6_reg(A, d);
        for (int q = 0; q < 6; q++) d[q] = -d[q];
      } else if constexpr (MODE == 1) {
        double A[36];
#pragma unroll
        for (int rr = 0; rr < 6; rr++)
#pragma unroll
          for (int cc = rr; cc < 6; cc++) {
            double sum = 0.0;
            for (int w = 0; w < JQ; w++) sum += s_part[ii * JQ + w][tri(rr, cc)];
            A[6 * rr + cc] = sum * inv_P;  // x * (1/P): one division instead of 27
            A[6 * cc + rr] = A[6 * rr + cc];
          }
#pragma unroll
        for (int q = 0; q < 6; q++) {
          double sum = 0.0;
          for (int w = 0; w < JQ; w++) sum += s_part[ii * JQ + w][21 + q];
          d[q] = sum * inv_P;
        }
        ldl_solve6_reg(A, d);  // :250 (the reference forms the explicit inverse; H-bar is SPD: tolerance-level difference)
        for (int q = 0; q < 6; q++) d[q] = a.lr * d[q];
      } else {
        double gs[6], kn[6], ks = 0.0;
        for (int q = 0; q < 6; q++) { gs[q] = 0.0; kn[q] = 0.0; }
        for (int w = 0; w < JQ; w++) {
          for (int q = 0; q < 6; q++) { gs[q] += s_part[ii * JQ + w][q]; kn[q] += s_part[ii * JQ + w][6 + q]; }
          ks += s_part[ii * JQ + w][12];
        }
        const double f = 2.0 / h;
        for (int rr = 0; rr < 6; rr++) {
          double s = 0.0;
          for (int cc = 0; cc < 6; cc++) s += s_Hinv[6 * rr + cc] * (f * gs[cc]);
          d[rr] = (kn[rr] + s) / ks;  // no lr (Q5)
        }
      }
#pragma unroll
      for (int q = 0; q < 6; q++) a.delta[(size_t)l * 6 + q] = d[q];
      if (a.stamps && blockIdx.x == 0 && ii == 0) a.stamps[6] = (double)global_timer_ns();  // solve done
      // pose update, SVNICP.cpp:268-279
      double dR[9], Jl[9], R[9], Rn[9], dt[3], t[3], w[3];
      so3_exp(d + 3, dR, Jl);  // :269-271
#pragma unroll
      for (int r = 0; r < 3; r++) dt[r] = Jl[3 * r] * d[0] + Jl[3 * r + 1] * d[1] + Jl[3 * r + 2] * d[2];  // :275
#pragma unroll
      for (int q = 0; q < 9; q++) R[q] = a.R[9 * (size_t)p + q];
#pragma unroll
      for (int r = 0; r < 3; r++)
#pragma unroll
        for (int cc = 0; cc < 3; cc++) Rn[3 * r + cc] = R[3 * r] * dR[cc] + R[3 * r + 1] * dR[3 + cc] + R[3 * r + 2] * dR[6 + cc];  // :277
#pragma unroll
      for (int q = 0; q < 9; q++) a.R[9 * (size_t)p + q] = Rn[q];
#pragma unroll
      for (int r = 0; r < 3; r++) {
        t[r] = (Rn[3 * r] * dt[0] + Rn[3 * r + 1] * dt[1] + Rn[3 * r + 2] * dt[2]) + a.t[3 * (size_t)p + r];  // :278 (Q6)
        a.t[3 * (size_t)p + r] = t[r];
      }
      const double dn = sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2] + d[3] * d[3] + d[4] * d[4] + d[5] * d[5]);  // :96
      a.dnorm[l] = dn;
      // head of the next iteration: x = [t ; Log R] and |delta| into every rank's NEXT record buffer
      so3_log(Rn, w);
      if (a.stamps && blockIdx.x == 0 && ii == 0) a.stamps[7] = (double)global_timer_ns();  // Exp, update, Log done
      for (int r = 0; r < pt.n_ranks; r++) {
        double *o = pt.rec[r] + nxt_off + (size_t)p * REC;
#pragma unroll
        for (int q = 0; q < 3; q++) { o[REC_X + q] = t[q]; o[REC_X + 3 + q] = w[q]; }
        o[REC_DNORM] = dn;
      }
      if (pt.n_ranks > 1) __threadfence_system();
      // fp32 transforms relative to q0 (as k_prep)
      float f[12];
      rel_transform_f32(R0, Rn, t, f);
      float *xf = ia.xf + (size_t)l * 12;
#pragma unroll
      for (int q = 0; q < 12; q++) { xf[q] = f[q]; xfd[q] = (double)f[q]; }
    }
    if (ii < TL_WARPS)
#pragma unroll
      for (int k = 0; k < 12; k++) s_xf[ii][k] = xfd[k];
  }
  __syncthreads();
  if (blockIdx.x == 0) TL_STAMP(3);
  // per-CTA partial of the centre transform, fixed order; then the ticket: the last CTA publishes
  if (tid < 12) {
    double s = 0.0;
    for (int ii = 0; ii < NI; ii++) s += s_xf[ii][tid];
    a.prep_scratch_d[(size_t)blockIdx.x * 12 + tid] = s;
  }
  __threadfence();
  __syncthreads();
  if (tid == 0) s_flag[0] = (atomicAdd(&c->tail_ticket, 1u) == gridDim.x - 1) ? 1 : 0;
  __syncthreads();
  if (!s_flag[0]) return;
  __threadfence();
  TL_STAMP(4);

  // ---------------- last CTA: exact-pruning ball of the local slice for the next iteration (as k_prep) ----------------
  if (tid < 12) {
    double s = 0.0;
    for (int b = 0; b < (int)gridDim.x; b++) s += __ldcg(a.prep_scratch_d + (size_t)b * 12 + tid);
    s_center[tid] = __double2float_rn(s / (double)a.P_l);
  }
  for (int q = tid; q < 4 * PRUNE_BINS; q += blockDim.x) s_envmax[q / PRUNE_BINS][q % PRUNE_BINS] = 0;
  if (tid < 2) { s_ab[tid] = 0; s_flag[1] = 0; }
  __syncthreads();
  {
    float *s_sg = reinterpret_cast<float *>(s_dyn);  // the tile ring is idle now: [TL_ENV_CHUNK] sigma, [TL_ENV_CHUNK] beta
    float *s_bt = s_sg + TL_ENV_CHUNK;
    int emax = 0;  // this thread's bin (tid % 64) over its share (tid / 64) of the chunk
    for (int l0 = 0; l0 < a.P_l; l0 += TL_ENV_CHUNK) {
      const int n = min(TL_ENV_CHUNK, a.P_l - l0);
      for (int u = tid; u < n; u += blockDim.x) {
        const float *xf = ia.xf + (size_t)(l0 + u) * 12;
        double M[9], db = 0;
        for (int q = 0; q < 9; q++) M[q] = (double)__ldcg(xf + q) - (double)s_center[q];
        for (int q = 9; q < 12; q++) { const double dd = (double)__ldcg(xf + q) - (double)s_center[q]; db += dd * dd; }
        const double da = sym3_max_eig_MtM(M);
        float sg = 0.f, bt = 0.f;
        if (da != da || db != db) s_flag[1] = 1;  // NaN state must poison the radius
        else { sg = __double2float_ru(sqrt(da) * (1.0 + 1e-6)); bt = __double2float_ru(sqrt(db) * (1.0 + 1e-6)); }
        s_sg[u] = sg;
        s_bt[u] = bt;
        atomicMax(&s_ab[0], __float_as_int(sg));  // non-negative floats order like their bit patterns
        atomicMax(&s_ab[1], __float_as_int(bt));
      }
      __syncthreads();
      if (tid < 4 * PRUNE_BINS) {
        const int bin = tid % PRUNE_BINS, part = tid / PRUNE_BINS;
        const double r = (double)(bin + 1) * PRUNE_BIN_W;
        for (int u = part; u < n; u += 4) {
          const float vv = __double2float_ru((double)s_sg[u] * r + (double)s_bt[u]);
          emax = max(emax, __float_as_int(vv));
        }
      }
      __syncthreads();
    }
    if (tid < 4 * PRUNE_BINS) s_envmax[tid / PRUNE_BINS][tid % PRUNE_BINS] = emax;
    __syncthreads();
  }
  const bool nan = s_flag[1] != 0;
  for (int q = tid; q < PRUNE_BINS; q += blockDim.x) {
    const int m = max(max(s_envmax[0][q], s_envmax[1][q]), max(s_envmax[2][q], s_envmax[3][q]));
    c->env[q] = nan ? NAN : __int_as_float(m);
  }
  if (tid < 9) c->Abar[tid] = s_center[tid];
  if (tid < 3) c->taubar[tid] = s_center[9 + tid];
  if (tid == 0) {
    c->alpha = nan ? NAN : __int_as_float(s_ab[0]);
    c->beta = nan ? NAN : __int_as_float(s_ab[1]);
    if (a.kept_hist && it <= a.I) a.kept_hist[it] = c->kept_total;  // candidates kept by this iteration's pruning pass
    c->kept_total = 0ull;
    c->tail_ticket = 0u;
    c->iter = it + 1;
  }
  TL_STAMP(5);
#undef TL_STAMP
  // every CTA fenced its peer stores before taking its ticket: the new x of the whole slice is out -> tell the peers
  if (pt.n_ranks > 1 && tid < pt.n_ranks && tid != pt.rank) {
    __threadfence_system();
    st_release_sys(pt.flag[tid] + FLAG_X * MAX_RANKS + pt.rank, seq_x_out);
  }
}

// ---------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------
int head_grid(int P, int sm_count) {
  // the median sweeps P^2/2 pairs: ~4096 per CTA and pass; at most one CTA per SM
  long long pairs = (long long)P * P / 2;
  long long g = (pairs + 4095) / 4096;
  if (g < 4) g = 4;
  if (g > sm_count) g = sm_count;
  if (P < 2) g = 1;
  return (int)g;
}

int launch_head(const SteinArgs &a, const PeerTable &pt, unsigned seq_x, int epilogue, cudaStream_t st) {
  if (a.P <= HD_SMALL_P) {  // one CTA does the whole chain
    k_head_small<<<1, HD_THREADS, 0, st>>>(a, pt, seq_x, epilogue);
    return 1;
  }
  int gp = (6 * a.P + HD_THREADS * 4 - 1) / (HD_THREADS * 4);
  if (gp < 1) gp = 1;
  if (gp > 32) gp = 32;
  k_head_prep<<<epilogue ? 4 : gp, HD_THREADS, 0, st>>>(a, pt, seq_x, epilogue);
  if (epilogue || a.P < 2) return 1;
  const int g = head_grid(a.P, a.sm_count);
  int n = 1;
  if (a.P >= 8) {
    k_head_fast1<<<g, HD_THREADS, 0, st>>>(a);
    k_head_fast2<<<g, HD_THREADS, 0, st>>>(a);
    n += 2;
  }
  for (int s = 0; s < MED_PASSES; s++) k_head_radix<<<g, HD_THREADS, 0, st>>>(a, s);
  return n + MED_PASSES;
}

void tail_shape(int P_l, int sm_count, int *NI, int *JQ, int *stages, size_t *smem) {
  // NI particles x JQ warps per CTA (NI * JQ = 8): the largest NI that still gives ~one CTA per SM -- small slices get more
  // warps per particle (shorter chain over j), large ones share each record tile among more particles (less L2 traffic)
  int ni = 8;
  while (ni > 1 && (P_l + ni - 1) / ni < (sm_count * 4) / 5) ni >>= 1;
  const int jq = TL_WARPS / ni;
  const size_t tile = (size_t)32 * jq * REC * sizeof(double);
  int s = (int)((150 * 1024) / tile);
  if (s > 12) s = 12;
  if (s < 1) s = 1;
  size_t bytes = (size_t)s * tile;
  if (bytes < (size_t)2 * TL_ENV_CHUNK * sizeof(float)) bytes = (size_t)2 * TL_ENV_CHUNK * sizeof(float);
  *NI = ni; *JQ = jq; *stages = s;
  *smem = bytes + 2 * (size_t)s * sizeof(uint64_t) + 128;
}

int launch_tail(const SteinArgs &a, const IterArgs &ia, const PeerTable &pt, unsigned seq_h, unsigned seq_x_out, cudaStream_t st) {
  static unsigned long long attr_set = 0ull;  // per device (the attribute belongs to the device's copy of the function)
  int dev = 0;
  cudaGetDevice(&dev);
  if (!((attr_set >> (dev & 63)) & 1ull)) {
    cudaFuncSetAttribute(k_tail<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    cudaFuncSetAttribute(k_tail<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    cudaFuncSetAttribute(k_tail<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    attr_set |= 1ull << (dev & 63);
  }
  int NI, JQ, stages;
  size_t smem;
  tail_shape(a.P_l, a.sm_count, &NI, &JQ, &stages, &smem);
  const int grid = (a.P_l + NI - 1) / NI;
  if (grid < 1) return 0;
  if (a.P < 2) k_tail<0><<<grid, TL_THREADS, smem, st>>>(a, ia, pt, seq_h, seq_x_out, NI, JQ, stages);
  else if (a.svn_full_grad) k_tail<1><<<grid, TL_THREADS, smem, st>>>(a, ia, pt, seq_h, seq_x_out, NI, JQ, stages);
  else k_tail<2><<<grid, TL_THREADS, smem, st>>>(a, ia, pt, seq_h, seq_x_out, NI, JQ, stages);
  return 1;
}

}  // namespace svn
