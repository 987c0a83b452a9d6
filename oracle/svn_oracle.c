/*
 * svn_oracle.c -- CPU restatement (plain C, fp64) of the SVN-ICP registration inner loop.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under oracle/ is part of the product: only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load this
 * file's shared object, and only as the checker / CPU baseline.  The product path
 * (svn_icp_b200/csrc) never links or calls it.
 *
 * Parity status: the reference ships NO tests, golden vectors or fixtures for this path
 * (SURVEY.md section 4 / 8c).  This restatement is pinned instead against outputs of the
 * reference's own sources compiled in this container (oracle/_ref, see oracle/build_ref.sh and
 * tests/golden/make_golden.py), committed under tests/golden/.
 *
 * Every function cites the reference file:line (relative to /root/reference/svn-icp/) it follows.
 * The second half of the file ("kernel-arithmetic mode", suffix _f32) restates the fp32
 * operation order of the CUDA kernels so correspondence indices can be compared bit-exactly
 * "given identical transformed points" (BASELINE.json north_star).
 *
 * Build: see oracle/Makefile  (gcc -O2 -ffp-contract=off -fopenmp -shared -fPIC).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <stdio.h>
#ifdef _OPENMP
#include <omp.h>
#endif

/* ------------------------------------------------------------------------------------------ */
/* parameters: mirrors SteinICPParam (include/core/SVGDICP.h:41-57), registration fields only  */
/* ------------------------------------------------------------------------------------------ */
typedef struct {
  int iterations;               /* SVGDICP.h:44 */
  double lr;                    /* SVGDICP.h:47 */
  double max_dist;              /* SVGDICP.h:48 */
  int check_early_stop;         /* SVGDICP.h:51 */
  double convergence_threshold; /* SVGDICP.h:53 */
  int knn_count;                /* SVGDICP.h:54 */
  int svn_full_grad;            /* SVGDICP.h:55 */
} oracle_params;

/* optional per-iteration dumps (any pointer may be NULL) */
typedef struct {
  int32_t *corr_idx; /* [I][P][N_s] global map index of the chosen candidate               */
  uint8_t *corr_mask;/* [I][P][N_s] 1 if d2 < max_dist                                      */
  double *H;         /* [I][P][36]                                                          */
  double *b;         /* [I][P][6]                                                           */
  double *delta;     /* [I][P][6]  stein_grad                                               */
  double *x_before;  /* [I][P][6]  [t;Log R] at the head of the iteration                   */
  double *x_after;   /* [I][P][6]  [t;Log R] after pose_update (fp64, unlike the history)   */
  double *bandwidth; /* [I]        h                                                        */
} oracle_dumps;

int oracle_num_threads(void) {
#ifdef _OPENMP
  return omp_get_max_threads();
#else
  return 1;
#endif
}

void oracle_set_num_threads(int n) {
#ifdef _OPENMP
  if (n > 0) omp_set_num_threads(n);
#else
  (void)n;
#endif
}

/* ------------------------------------------------------------------------------------------ */
/* small dense helpers                                                                         */
/* ------------------------------------------------------------------------------------------ */
static void mat3_mul(const double *A, const double *B, double *C) {
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) {
      double s = 0;
      for (int k = 0; k < 3; k++) s += A[3 * i + k] * B[3 * k + j];
      C[3 * i + j] = s;
    }
}
static void mat3_vec(const double *A, const double *v, double *o) {
  for (int i = 0; i < 3; i++) o[i] = A[3 * i] * v[0] + A[3 * i + 1] * v[1] + A[3 * i + 2] * v[2];
}

/* LU with partial pivoting, n<=6, solves A X = B for nrhs columns (LAPACK dgesv order of
 * operations; stands in for torch::linalg::solve / inv at SVNICP.cpp:162,225,250). */
static int lu_solve(int n, const double *A_in, double *B, int nrhs) {
  double A[36];
  int piv[6];
  memcpy(A, A_in, sizeof(double) * n * n);
  for (int k = 0; k < n; k++) {
    int p = k;
    double mx = fabs(A[k * n + k]);
    for (int i = k + 1; i < n; i++)
      if (fabs(A[i * n + k]) > mx) { mx = fabs(A[i * n + k]); p = i; }
    piv[k] = p;
    if (p != k) {
      for (int j = 0; j < n; j++) { double t = A[k * n + j]; A[k * n + j] = A[p * n + j]; A[p * n + j] = t; }
      for (int j = 0; j < nrhs; j++) { double t = B[k * nrhs + j]; B[k * nrhs + j] = B[p * nrhs + j]; B[p * nrhs + j] = t; }
    }
    double d = A[k * n + k];
    for (int i = k + 1; i < n; i++) {
      double l = A[i * n + k] / d;
      A[i * n + k] = l;
      for (int j = k + 1; j < n; j++) A[i * n + j] -= l * A[k * n + j];
      for (int j = 0; j < nrhs; j++) B[i * nrhs + j] -= l * B[k * nrhs + j];
    }
  }
  for (int k = n - 1; k >= 0; k--) {
    for (int j = 0; j < nrhs; j++) {
      double s = B[k * nrhs + j];
      for (int i = k + 1; i < n; i++) s -= A[k * n + i] * B[i * nrhs + j];
      B[k * nrhs + j] = s / A[k * n + k];
    }
  }
  (void)piv;
  return 0;
}

void oracle_solve6(const double *A, const double *b, double *x) {
  memcpy(x, b, 6 * sizeof(double));
  lu_solve(6, A, x, 1);
}

void oracle_inv6(const double *A, double *Ainv) {
  memset(Ainv, 0, 36 * sizeof(double));
  for (int i = 0; i < 6; i++) Ainv[7 * i] = 1.0;
  lu_solve(6, A, Ainv, 6);
}

/* ------------------------------------------------------------------------------------------ */
/* SO(3) maps                                                                                  */
/* ------------------------------------------------------------------------------------------ */

/* SVNICP::to_rotation_tensor, src/core/SVNICP.cpp:166-194.
 * R = cos(a) I + (1-cos a) n n^T + sin(a) [n]x, axis n = r/|r| (0 where |r| < 1e-12);
 * side effect J_l = (sin a / a) I + (1 - sin a / a) n n^T + ((1-cos a)/a) [n]x  (NaN at a == 0:
 * quirk Q7, reproduced literally). */
void oracle_so3_exp(const double r[3], double R[9], double Jl[9]) {
  double a = sqrt(r[0] * r[0] + r[1] * r[1] + r[2] * r[2]); /* :170 */
  double n[3];
  if (a < 1e-12) { n[0] = n[1] = n[2] = 0.0; }            /* :171-173 */
  else { n[0] = r[0] / a; n[1] = r[1] / a; n[2] = r[2] / a; }
  double c = cos(a), s = sin(a);                            /* :174-175 */
  /* a_hat after the .transpose(1,2) at :180 is the usual skew matrix [n]x */
  double ah[9] = {0, -n[2], n[1], n[2], 0, -n[0], -n[1], n[0], 0};
  double sa = s / a;            /* :188 (0/0 = NaN when a == 0) */
  double ca = (1.0 - c) / a;    /* :192 */
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) {
      double id = (i == j) ? 1.0 : 0.0;
      double nn = n[i] * n[j];
      R[3 * i + j] = c * id + (1.0 - c) * nn + s * ah[3 * i + j];          /* :182-186 */
      if (Jl) Jl[3 * i + j] = sa * id + (1.0 - sa) * nn + ca * ah[3 * i + j]; /* :188-192 */
    }
}

/* SVNICP::rotm_to_ypr_tensor, src/core/SVNICP.cpp:196-215 (an SO(3) Log despite the name). */
void oracle_so3_log(const double R[9], double w[3]) {
  double v = 0.5 * (R[0] + R[4] + R[8] - 1.0); /* :199 */
  if (v < -1.0) v = -1.0;
  if (v > 1.0) v = 1.0;                          /* :198-200 clip */
  double a = acos(v);
  double s = sin(a);                             /* :203 */
  if (fabs(s) > 1e-12) {                         /* :205 */
    double f = 0.5 / s * a;                      /* :207 */
    w[0] = f * (R[7] - R[5]);                    /* :209 */
    w[1] = f * (R[2] - R[6]);                    /* :210 */
    w[2] = f * (R[3] - R[1]);                    /* :211 */
  } else {
    w[0] = w[1] = w[2] = 0.0;                    /* :213 */
  }
}

/* ------------------------------------------------------------------------------------------ */
/* per-scan candidate build                                                                    */
/* ------------------------------------------------------------------------------------------ */

/* SVGDICP::knn_source_cloud (src/core/SVGDICP.cpp:201-215) -> KNearestNeighborKernelV1<double,3>
 * (src/core/knn/knn.cu:68-111) with MinK::add (include/core/utils/mink.cuh:62-83).
 * q: [n_q][3] already transformed by (R0,t0); tgt: [n_t][3].
 * idx_out/dist_out: [n_q][K] in MinK slot order, zero padded when n_t < K (knn.cu:343-344).
 * Distance = fma(dz,dz,fma(dy,dy,dx*dx)): nvcc contracts `dist += diff*diff` (knn.cu:101-106). */
void oracle_knn_mink(const double *q, int64_t n_q, const double *tgt, int64_t n_t, int K,
                     int64_t *idx_out, double *dist_out) {
#pragma omp parallel for schedule(dynamic, 64)
  for (int64_t i = 0; i < n_q; i++) {
    double *keys = (double *)calloc((size_t)K, sizeof(double));
    int64_t *vals = (int64_t *)calloc((size_t)K, sizeof(int64_t));
    int size = 0, max_idx = 0;
    double max_key = 0;
    const double qx = q[3 * i], qy = q[3 * i + 1], qz = q[3 * i + 2];
    for (int64_t j = 0; j < n_t; j++) {
      double dx = qx - tgt[3 * j], dy = qy - tgt[3 * j + 1], dz = qz - tgt[3 * j + 2];
      double d = fma(dz, dz, fma(dy, dy, dx * dx));
      if (size < K) {                                   /* mink.cuh:63-70 */
        keys[size] = d; vals[size] = j;
        if (size == 0 || d > max_key) { max_key = d; max_idx = size; }
        size++;
      } else if (d < max_key) {                         /* mink.cuh:71-81 */
        keys[max_idx] = d; vals[max_idx] = j;
        max_key = d;
        for (int k = 0; k < K; k++)
          if (keys[k] > max_key) { max_key = keys[k]; max_idx = k; }
      }
    }
    memcpy(idx_out + i * K, vals, sizeof(int64_t) * K);
    if (dist_out) memcpy(dist_out + i * K, keys, sizeof(double) * K);
    free(keys); free(vals);
  }
}

/* q0_b = R0 s_b + t0 : SVGDICP.cpp:204 (source.matmul(R0^T) + t0). Fixed fma order shared with
 * the CUDA candidate builder so that d0^2 and hence the K-nearest SET agree bit for bit. */
void oracle_transform_q0(const double *src, int64_t n_s, const double R0[9], const double t0[3], double *q0) {
  for (int64_t i = 0; i < n_s; i++) {
    const double x = src[3 * i], y = src[3 * i + 1], z = src[3 * i + 2];
    for (int r = 0; r < 3; r++)
      q0[3 * i + r] = fma(R0[3 * r], x, fma(R0[3 * r + 1], y, fma(R0[3 * r + 2], z, t0[r])));
  }
}

/* ------------------------------------------------------------------------------------------ */
/* per-iteration pieces                                                                        */
/* ------------------------------------------------------------------------------------------ */

/* One particle: transform (SVNICP.cpp:58-64), candidate 1-NN (SVGDICP.cpp:300-329 ->
 * knn.cu:204-251 + RegisterMinK<.,.,1>, mink.cuh:132-153: strict '<', first slot wins),
 * point_filter (SVGDICP.cpp:331-333: SQUARED distance against the UN-squared max_dist, Q1),
 * Newton_grad_right (SVNICP.cpp:116-164).  cand_idx: [n_s][K] MinK-ordered map indices.
 * Returns H (6x6 row-major, includes +1e-6 I), b (6).  corr_out/mask_out optional [n_s]. */
static void particle_gn(const double *Rt /*R_total 3x3*/, const double *tt /*t_total*/,
                        const double *src, int64_t n_s, const double *tgt, const int64_t *cand_idx,
                        int K, double max_dist, double *H, double *b, int32_t *corr_out,
                        uint8_t *mask_out) {
  memset(H, 0, 36 * sizeof(double));
  memset(b, 0, 6 * sizeof(double));
  for (int64_t i = 0; i < n_s; i++) {
    const double *s = src + 3 * i;
    double q[3];
    for (int r = 0; r < 3; r++) q[r] = Rt[3 * r] * s[0] + Rt[3 * r + 1] * s[1] + Rt[3 * r + 2] * s[2] + tt[r];
    /* 1-NN among the K candidates of this source point */
    double best = 0;
    int bestk = -1;
    for (int k = 0; k < K; k++) {
      const double *m = tgt + 3 * cand_idx[i * K + k];
      double dx = q[0] - m[0], dy = q[1] - m[1], dz = q[2] - m[2];
      double d = fma(dz, dz, fma(dy, dy, dx * dx));
      if (bestk < 0 || d < best) { best = d; bestk = k; }
    }
    const int64_t gi = cand_idx[i * K + bestk];
    const double mu = (best < max_dist) ? 1.0 : 0.0;       /* SVGDICP.cpp:332 (Q1) */
    if (corr_out) corr_out[i] = (int32_t)gi;
    if (mask_out) mask_out[i] = (uint8_t)mu;
    double sp[3] = {mu * s[0], mu * s[1], mu * s[2]};     /* source_paired      */
    double e[3];
    for (int r = 0; r < 3; r++) e[r] = mu * q[r] - mu * tgt[3 * gi + r]; /* SVNICP.cpp:119 */
    double en = sqrt(e[0] * e[0] + e[1] * e[1] + e[2] * e[2]);           /* :120 */
    double w = max_dist / (max_dist + 3.0 * en);
    w = w * w;                                                             /* :122 */
    double ew[3] = {w * e[0], w * e[1], w * e[2]};                         /* :123 */
    /* J = [R_c | -R_c s_hat]   :126-146 */
    double sh[9] = {0, -sp[2], sp[1], sp[2], 0, -sp[0], -sp[1], sp[0], 0};
    double Rs[9];
    mat3_mul(Rt, sh, Rs);
    double J[18];
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 3; c++) { J[6 * r + c] = Rt[3 * r + c]; J[6 * r + 3 + c] = -Rs[3 * r + c]; }
    /* H += J^T (w J), b += J^T (w e)  :149-157 */
    for (int k = 0; k < 6; k++) {
      for (int l = 0; l < 6; l++) {
        double acc = 0;
        for (int r = 0; r < 3; r++) acc += J[6 * r + k] * (J[6 * r + l] * w);
        H[6 * k + l] += acc;
      }
      double accb = 0;
      for (int r = 0; r < 3; r++) accb += J[6 * r + k] * ew[r];
      b[k] += accb;
    }
  }
  for (int k = 0; k < 6; k++) H[7 * k] += 1e-6; /* :153 (Q3) */
}

/* element k of the ascending order of n doubles (no NaN).  Quickselect, reorders a. */
static double select_kth(double *a, int64_t n, int64_t k) {
  int64_t lo = 0, hi = n - 1;
  while (lo < hi) {
    double pv = a[lo + (hi - lo) / 2];
    int64_t i = lo, j = hi;
    while (i <= j) {
      while (a[i] < pv) i++;
      while (a[j] > pv) j--;
      if (i <= j) { double t = a[i]; a[i] = a[j]; a[j] = t; i++; j--; }
    }
    if (k <= j) hi = j;
    else if (k >= i) lo = i;
    else break;
  }
  return a[k];
}

/* lower median of n doubles (torch::median over the flattened tensor, SVNICP.cpp:262):
 * element (n-1)/2 of the sorted order.  Quickselect on a scratch copy. */
static double lower_median(double *a, int64_t n) { return select_kth(a, n, (n - 1) / 2); }

/* The bandwidth median as the k_head_* kernels compute it (tail2.cu): pair distances rounded as in hd_sweep,
 * s = fma(df0, df0, df1 * df1), then s = fma(df, df, s) for d = 2..5, once per unordered pair.  x: [P][6].
 * out[0] = lower median of the P^2 entries (P diagonal zeros, every pair twice), out[1] / out[2] = the nearest distinct
 * entry below / above it (-inf / +inf if there is none): a bandwidth check that rejects a neighbouring rank. */
void oracle_pair_median_kernel_order(const double *x, int P, double out[3]) {
  const int64_t n = (int64_t)P * (P - 1) / 2;
  const int64_t rank = ((int64_t)P * P - 1) / 2;
  out[0] = 0.0; out[1] = -INFINITY; out[2] = INFINITY;
  if (n == 0) return;
  double *a = (double *)malloc(sizeof(double) * (size_t)n);
#pragma omp parallel for schedule(dynamic, 16)
  for (int i = 0; i < P; i++) {
    double *row = a + (int64_t)i * (2 * (int64_t)P - i - 1) / 2;  /* pairs (i, j > i) */
    for (int j = i + 1; j < P; j++) {
      double df[6];
      for (int d = 0; d < 6; d++) df[d] = x[6 * i + d] - x[6 * j + d];
      double s = fma(df[0], df[0], df[1] * df[1]);
      for (int d = 2; d < 6; d++) s = fma(df[d], df[d], s);
      row[j - i - 1] = s;
    }
  }
  /* ascending: P zeros, then pair k at entries P + 2k and P + 2k + 1 */
  const double m = rank < P ? 0.0 : select_kth(a, n, (rank - P) / 2);
  double below = m > 0.0 ? 0.0 : -INFINITY, above = INFINITY;
  for (int64_t k = 0; k < n; k++) {
    if (a[k] < m && a[k] > below) below = a[k];
    if (a[k] > m && a[k] < above) above = a[k];
  }
  out[0] = m; out[1] = below; out[2] = above;
  free(a);
}

/* SVNICP::rbf_hessian_kernel, SVNICP.cpp:254-266.  x: [P][6].  Kmat: [P][P]. returns h. */
double oracle_rbf_kernel(const double *x, int P, double *Kmat) {
  double *D = (double *)malloc(sizeof(double) * (size_t)P * P);
#pragma omp parallel for schedule(static)
  for (int i = 0; i < P; i++)
    for (int j = 0; j < P; j++) {
      double s = 0;
      for (int d = 0; d < 6; d++) { double df = x[6 * i + d] - x[6 * j + d]; s += df * df; } /* :257-260 */
      D[(size_t)i * P + j] = s;
    }
  double *scratch = (double *)malloc(sizeof(double) * (size_t)P * P);
  memcpy(scratch, D, sizeof(double) * (size_t)P * P);
  double med = lower_median(scratch, (int64_t)P * P);
  free(scratch);
  double h = med / log((double)(P + 1));        /* :262 (Q4) */
#pragma omp parallel for schedule(static)
  for (int64_t t = 0; t < (int64_t)P * P; t++) Kmat[t] = exp(-D[t] / h); /* :264 */
  free(D);
  return h;
}

/* SVNICP::svn_full_grad, SVNICP.cpp:229-252.  bneg = -b.  out: [P][6] */
static void svn_full_grad(const double *x, const double *H, const double *bneg, int P, double lr,
                          double *out, double *h_out) {
  double *Kmat = (double *)malloc(sizeof(double) * (size_t)P * P);
  double h = oracle_rbf_kernel(x, P, Kmat);
  if (h_out) *h_out = h;
#pragma omp parallel for schedule(static)
  for (int i = 0; i < P; i++) {
    double Hm[36], v[6];
    memset(Hm, 0, sizeof(Hm));
    memset(v, 0, sizeof(v));
    for (int j = 0; j < P; j++) {
      double kij = Kmat[(size_t)i * P + j];
      double g[6];
      for (int d = 0; d < 6; d++) g[d] = 2.0 / h * ((x[6 * i + d] - x[6 * j + d]) * kij); /* :233 */
      double k2 = kij * kij;                                                                /* :238 */
      for (int a = 0; a < 6; a++) {
        for (int c = 0; c < 6; c++) Hm[6 * a + c] += k2 * H[36 * (size_t)j + 6 * a + c] + g[a] * g[c]; /* :236-242 */
        v[a] += kij * bneg[6 * (size_t)j + a] + g[a];                                      /* :244 */
      }
    }
    for (int a = 0; a < 36; a++) Hm[a] /= (double)P;                                       /* :242 */
    for (int a = 0; a < 6; a++) v[a] /= (double)P;                                         /* :244 */
    double Hi[36];
    oracle_inv6(Hm, Hi);                                                                    /* :250 */
    for (int a = 0; a < 6; a++) {
      double s = 0;
      for (int c = 0; c < 6; c++) s += Hi[6 * a + c] * v[c];
      out[6 * i + a] = lr * s;
    }
  }
  free(Kmat);
}

/* SVNICP::svgd_grad, SVNICP.cpp:218-227, called from :85-86 with newton = -H^-1 b and
 * H = mean_p H_p (same matrix for every particle).  No lr (Q5). */
static void svn_svgd_grad(const double *x, const double *newton_neg, const double *Hmean, int P,
                          double *out, double *h_out) {
  double *Kmat = (double *)malloc(sizeof(double) * (size_t)P * P);
  double h = oracle_rbf_kernel(x, P, Kmat);
  if (h_out) *h_out = h;
  double Hi[36];
  oracle_inv6(Hmean, Hi);                                                                   /* :225 */
#pragma omp parallel for schedule(static)
  for (int i = 0; i < P; i++) {
    double g[6] = {0, 0, 0, 0, 0, 0}, kn[6] = {0, 0, 0, 0, 0, 0}, ks = 0;
    for (int j = 0; j < P; j++) {
      double kij = Kmat[(size_t)i * P + j];
      ks += kij;                                                                            /* :226 */
      for (int d = 0; d < 6; d++) {
        g[d] += (x[6 * i + d] - x[6 * j + d]) * kij;                                        /* :221-222 */
        kn[d] += kij * newton_neg[6 * (size_t)j + d];                                       /* :224 */
      }
    }
    for (int d = 0; d < 6; d++) g[d] *= 2.0 / h;
    for (int a = 0; a < 6; a++) {
      double s = 0;
      for (int c = 0; c < 6; c++) s += Hi[6 * a + c] * g[c];
      out[6 * i + a] = (kn[a] + s) / ks;
    }
  }
  free(Kmat);
}

/* SVNICP::pose_update, SVNICP.cpp:268-279: R <- R dR, t <- R_new (J_l dt) + t  (Q6). */
static void pose_update(double *R, double *t, const double *delta) {
  double dR[9], Jl[9], dt[3], Rn[9], Rdt[3];
  oracle_so3_exp(delta + 3, dR, Jl);
  mat3_vec(Jl, delta, dt);
  mat3_mul(R, dR, Rn);
  memcpy(R, Rn, sizeof(Rn));
  mat3_vec(R, dt, Rdt);
  for (int r = 0; r < 3; r++) t[r] = Rdt[r] + t[r];
}

/* ------------------------------------------------------------------------------------------ */
/* whole scan: add_cloud -> set_initial_mean -> stein_align -> getters                         */
/* ------------------------------------------------------------------------------------------ */

/* init_pose: [6][P] component-major (x,y,z,rx,ry,rz rows) as the reference's init_pose tensor
 * [6,P,1] (SVGDICP.cpp:46-61).  R0 row-major = gtsam rotation matrix (SVGDICP.h:102-110).
 * Outputs: particles [6][P] (SVGDICP.cpp:515-520), mean[6] (SVNICP.cpp:286-290),
 * var[6] (:292-297), cov[36] (:299-308), weights[P] (:281-284), history float [I][6][P]
 * (SVGDICP.cpp:172-174,526-534; rows after an early stop stay 0), *iters_done = iterations whose
 * pose update was applied.  cand_idx_out optional [n_s][K] (MinK order). */
int oracle_align(const oracle_params *prm, const double *src, int64_t n_s, const double *tgt,
                 int64_t n_t, const double *init_pose, int P, const double R0[9], const double t0[3],
                 double *particles, double *mean, double *var, double *cov, double *weights,
                 float *history, int *iters_done, int64_t *cand_idx_out, oracle_dumps *dmp) {
  const int K = prm->knn_count, I = prm->iterations;
  double *R = (double *)malloc(sizeof(double) * 9 * P), *t = (double *)malloc(sizeof(double) * 3 * P);
  double *x = (double *)malloc(sizeof(double) * 6 * P);
  double *H = (double *)malloc(sizeof(double) * 36 * P), *b = (double *)malloc(sizeof(double) * 6 * P);
  double *newton = (double *)malloc(sizeof(double) * 6 * P), *delta = (double *)malloc(sizeof(double) * 6 * P);
  double *q0 = (double *)malloc(sizeof(double) * 3 * (n_s > 0 ? n_s : 1));
  int64_t *cand = (int64_t *)calloc((size_t)(n_s > 0 ? n_s : 1) * K, sizeof(int64_t));
  /* add_cloud: SVGDICP.cpp:46-61 */
  for (int p = 0; p < P; p++) {
    double r[3] = {init_pose[3 * P + p], init_pose[4 * P + p], init_pose[5 * P + p]};
    oracle_so3_exp(r, R + 9 * p, NULL);
    for (int c = 0; c < 3; c++) t[3 * p + c] = init_pose[c * P + p];
  }
  /* head of stein_align: SVNICP.cpp:46 weights are float32(1)/P (see get_particle_weight :281-284) */
  const double wgt = (double)(1.0f / (float)P);
  if (history) memset(history, 0, sizeof(float) * (size_t)I * 6 * P); /* SVGDICP.cpp:172-174 */
  /* mini_batch_pair_generator -> knn_source_cloud: SVGDICP.cpp:176-215 */
  oracle_transform_q0(src, n_s, R0, t0, q0);
  oracle_knn_mink(q0, n_s, tgt, n_t, K, cand, NULL);
  if (cand_idx_out) memcpy(cand_idx_out, cand, sizeof(int64_t) * (size_t)n_s * K);

  int done = 0;
  for (int epoch = 0; epoch < I; epoch++) {
#pragma omp parallel for schedule(dynamic, 1)
    for (int p = 0; p < P; p++) {
      double Rt[9], tt[3], R0t[3];
      mat3_mul(R0, R + 9 * p, Rt);                       /* SVNICP.cpp:58 */
      mat3_vec(R0, t + 3 * p, R0t);
      for (int c = 0; c < 3; c++) tt[c] = t0[c] + R0t[c]; /* :59 */
      int32_t *co = (dmp && dmp->corr_idx) ? dmp->corr_idx + ((size_t)epoch * P + p) * n_s : NULL;
      uint8_t *mo = (dmp && dmp->corr_mask) ? dmp->corr_mask + ((size_t)epoch * P + p) * n_s : NULL;
      particle_gn(Rt, tt, src, n_s, tgt, cand, K, prm->max_dist, H + 36 * p, b + 6 * p, co, mo);
      oracle_solve6(H + 36 * p, b + 6 * p, newton + 6 * p); /* :162 */
      for (int c = 0; c < 3; c++) x[6 * p + c] = t[3 * p + c]; /* :74-77 */
      oracle_so3_log(R + 9 * p, x + 6 * p + 3);
    }
    double h = 0;
    if (P > 1) {                                          /* :81 */
      if (prm->svn_full_grad) {
        double *bneg = (double *)malloc(sizeof(double) * 6 * P);
        for (int i = 0; i < 6 * P; i++) bneg[i] = -b[i];
        svn_full_grad(x, H, bneg, P, prm->lr, delta, &h); /* :83 */
        free(bneg);
      } else {
        double Hm[36];
        for (int a = 0; a < 36; a++) {
          double s = 0;
          for (int p = 0; p < P; p++) s += H[36 * p + a];
          Hm[a] = s / (double)P;                          /* :85 */
        }
        double *nn = (double *)malloc(sizeof(double) * 6 * P);
        for (int i = 0; i < 6 * P; i++) nn[i] = -newton[i];
        svn_svgd_grad(x, nn, Hm, P, delta, &h);           /* :86 */
        free(nn);
      }
    } else {
      for (int i = 0; i < 6; i++) delta[i] = -newton[i];  /* :89 */
    }
    if (dmp) {
      if (dmp->H) memcpy(dmp->H + (size_t)epoch * 36 * P, H, sizeof(double) * 36 * P);
      if (dmp->b) memcpy(dmp->b + (size_t)epoch * 6 * P, b, sizeof(double) * 6 * P);
      if (dmp->delta) memcpy(dmp->delta + (size_t)epoch * 6 * P, delta, sizeof(double) * 6 * P);
      if (dmp->x_before) memcpy(dmp->x_before + (size_t)epoch * 6 * P, x, sizeof(double) * 6 * P);
      if (dmp->bandwidth) dmp->bandwidth[epoch] = h;
    }
    for (int p = 0; p < P; p++) pose_update(R + 9 * p, t + 3 * p, delta + 6 * p); /* :92 */
    done = epoch + 1;
    if (dmp && dmp->x_after)
      for (int p = 0; p < P; p++) {
        double *xa = dmp->x_after + ((size_t)epoch * P + p) * 6;
        for (int c = 0; c < 3; c++) xa[c] = t[3 * p + c];
        oracle_so3_log(R + 9 * p, xa + 3);
      }
    if (prm->check_early_stop) {                          /* :95-101 (Q9) */
      double s = 0;
      for (int p = 0; p < P; p++) {
        double n2 = 0;
        for (int c = 0; c < 6; c++) n2 += delta[6 * p + c] * delta[6 * p + c];
        s += sqrt(n2);
      }
      if (s / (double)P < prm->convergence_threshold) break;
    }
    if (history)                                          /* :103-107 */
      for (int p = 0; p < P; p++) {
        double w3[3];
        oracle_so3_log(R + 9 * p, w3);
        for (int c = 0; c < 3; c++) {
          history[((size_t)epoch * 6 + c) * P + p] = (float)t[3 * p + c];
          history[((size_t)epoch * 6 + 3 + c) * P + p] = (float)w3[c];
        }
      }
  }
  if (iters_done) *iters_done = done;
  /* :111 final pose_particles_ [6][P] and getters :281-308 */
  for (int p = 0; p < P; p++) {
    double w3[3];
    oracle_so3_log(R + 9 * p, w3);
    for (int c = 0; c < 3; c++) { particles[c * P + p] = t[3 * p + c]; particles[(3 + c) * P + p] = w3[c]; }
  }
  for (int c = 0; c < 6; c++) {
    double s = 0;
    for (int p = 0; p < P; p++) s += particles[c * P + p] * wgt;
    mean[c] = s;
  }
  for (int c = 0; c < 6; c++) {
    double s = 0;
    for (int p = 0; p < P; p++) { double d = particles[c * P + p] - mean[c]; s += d * d * wgt; }
    var[c] = s;
  }
  for (int a = 0; a < 6; a++)
    for (int c = 0; c < 6; c++) {
      double s = 0;
      for (int p = 0; p < P; p++) s += wgt * ((particles[a * P + p] - mean[a]) * (particles[c * P + p] - mean[c]));
      cov[6 * a + c] = s;
    }
  if (weights) for (int p = 0; p < P; p++) weights[p] = wgt;
  free(R); free(t); free(x); free(H); free(b); free(newton); free(delta); free(q0); free(cand);
  return 1; /* ALIGN_SUCCESS, SVGDICP.h:59-62 */
}

/* Stein step alone (tests of kernel (c)): x [P][6], H [P][36], b [P][6] -> delta [P][6], h. */
void oracle_stein_step(const double *x, const double *H, const double *b, int P, int full, double lr,
                       double *delta, double *h_out) {
  if (P == 1) {
    double g[6];
    oracle_solve6(H, b, g);
    for (int i = 0; i < 6; i++) delta[i] = -g[i];
    if (h_out) *h_out = 0;
    return;
  }
  if (full) {
    double *bneg = (double *)malloc(sizeof(double) * 6 * P);
    for (int i = 0; i < 6 * P; i++) bneg[i] = -b[i];
    svn_full_grad(x, H, bneg, P, lr, delta, h_out);
    free(bneg);
  } else {
    double Hm[36];
    for (int a = 0; a < 36; a++) {
      double s = 0;
      for (int p = 0; p < P; p++) s += H[36 * p + a];
      Hm[a] = s / (double)P;
    }
    double *nn = (double *)malloc(sizeof(double) * 6 * P);
    for (int p = 0; p < P; p++) {
      double g[6];
      oracle_solve6(H + 36 * p, b + 6 * p, g);
      for (int i = 0; i < 6; i++) nn[6 * p + i] = -g[i];
    }
    svn_svgd_grad(x, nn, Hm, P, delta, h_out);
    free(nn);
  }
}

/* pose_update on [R (9), t (3)] arrays for P particles (tests). */
void oracle_pose_update(double *R, double *t, const double *delta, int P) {
  for (int p = 0; p < P; p++) pose_update(R + 9 * p, t + 3 * p, delta + 6 * p);
}

/* GN system for explicit particle poses (tests of kernels (a)+(b)):
 * R,t: per-particle relative pose [P][9],[P][3]; cand_idx [n_s][K]. */
void oracle_gn(const double *R, const double *t, int P, const double R0[9], const double t0[3],
               const double *src, int64_t n_s, const double *tgt, const int64_t *cand_idx, int K,
               double max_dist, double *H, double *b, int32_t *corr_idx, uint8_t *corr_mask) {
#pragma omp parallel for schedule(dynamic, 1)
  for (int p = 0; p < P; p++) {
    double Rt[9], tt[3], R0t[3];
    mat3_mul(R0, R + 9 * p, Rt);
    mat3_vec(R0, t + 3 * p, R0t);
    for (int c = 0; c < 3; c++) tt[c] = t0[c] + R0t[c];
    particle_gn(Rt, tt, src, n_s, tgt, cand_idx, K, max_dist, H + 36 * p, b + 6 * p,
                corr_idx ? corr_idx + (size_t)p * n_s : NULL, corr_mask ? corr_mask + (size_t)p * n_s : NULL);
  }
}

/* ------------------------------------------------------------------------------------------ */
/* SVGDICP-base helpers shared by the drop-in boundary                                         */
/* ------------------------------------------------------------------------------------------ */

/* initialize_particles, src/core/ICPUtils.cpp:45-58: uniform in [lb,ub] per component,
 * P == 1 -> zeros.  u: caller supplied uniforms [6][P] in [0,1) (torch::rand is not
 * reproducible across builds, SURVEY.md App. B). out [6][P]. */
void oracle_initialize_particles(int P, const double ub[6], const double lb[6], const double *u, double *out) {
  for (int c = 0; c < 6; c++)
    for (int p = 0; p < P; p++) out[c * P + p] = (P == 1) ? 0.0 : (ub[c] - lb[c]) * u[c * P + p] + lb[c];
}

/* ========================================================================================== */
/* Kernel-arithmetic mode: restates the fp32 operation order of the CUDA kernels so that       */
/* correspondence indices can be compared BIT-EXACTLY "given identical transformed points"     */
/* (BASELINE.json north_star).  Documented differences to the reference semantics:             */
/*   - candidate slot order is ascending (d0^2, map index) instead of MinK replacement order;  */
/*     the candidate SET is the same K nearest (fp64, same fma order);                         */
/*   - the 1-NN runs in fp32 on coordinates RELATIVE to q0_b (c' = fp32(m - q0_b),            */
/*     q' = A' s' + tau with A' = fp32(R0 (R_p - I) R0^T), tau = fp32(R0 t_p), s' = fp32(R0 s)); */
/*   - tie-break: strict '<' scanning OUR slot order, i.e. among exactly equal fp32 distances  */
/*     the candidate with the smaller (d0^2, index) wins (the reference: lower MinK slot).     */
/* ========================================================================================== */

typedef struct { double d; int64_t idx; } dist_idx;

static int cmp_dist_idx(const void *a, const void *b) {
  const dist_idx *x = (const dist_idx *)a, *y = (const dist_idx *)b;
  if (x->d < y->d) return -1;
  if (x->d > y->d) return 1;
  return (x->idx > y->idx) - (x->idx < y->idx);
}

/* K nearest map points of every q0 (brute force, fp64, fma order of knn.cu:101-106), ascending
 * (d0^2, index); padded with map point 0 when n_t < K (knn.cu:343).  rel: fp32(m - q0) [n_q][K][3]. */
void oracle_cand_sorted(const double *q0, int64_t n_q, const double *tgt, int64_t n_t, int K,
                        int32_t *idx_out, float *rel_out) {
#pragma omp parallel
  {
    dist_idx *a = (dist_idx *)malloc(sizeof(dist_idx) * (size_t)(n_t > 0 ? n_t : 1));
#pragma omp for schedule(dynamic, 16)
    for (int64_t i = 0; i < n_q; i++) {
      const double qx = q0[3 * i], qy = q0[3 * i + 1], qz = q0[3 * i + 2];
      for (int64_t j = 0; j < n_t; j++) {
        double dx = qx - tgt[3 * j], dy = qy - tgt[3 * j + 1], dz = qz - tgt[3 * j + 2];
        a[j].d = fma(dz, dz, fma(dy, dy, dx * dx));
        a[j].idx = j;
      }
      qsort(a, (size_t)n_t, sizeof(dist_idx), cmp_dist_idx);
      for (int k = 0; k < K; k++) {
        const int64_t gi = (k < n_t) ? a[k].idx : 0;
        idx_out[i * K + k] = (int32_t)gi;
        if (rel_out)
          for (int c = 0; c < 3; c++) rel_out[(i * K + k) * 3 + c] = (float)(tgt[3 * gi + c] - q0[3 * i + c]);
      }
    }
    free(a);
  }
}

/* s' = fp32(R0 s) as k_q0 computes it (fma chain without the translation). */
void oracle_source_f32(const double *src, int64_t n_s, const double R0[9], float *sp) {
  for (int64_t i = 0; i < n_s; i++) {
    const double x = src[3 * i], y = src[3 * i + 1], z = src[3 * i + 2];
    for (int r = 0; r < 3; r++) sp[3 * i + r] = (float)fma(R0[3 * r], x, fma(R0[3 * r + 1], y, R0[3 * r + 2] * z));
  }
}

/* fp32 transforms as k_prep computes them from the fp64 particle state: xf [P][12]. */
void oracle_transforms_f32(const double *R, const double *t, int P, const double R0[9], float *xf) {
  for (int p = 0; p < P; p++) {
    double D[9], T[9];
    for (int i = 0; i < 9; i++) D[i] = R[9 * p + i] - ((i % 4 == 0) ? 1.0 : 0.0);
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 3; c++) T[3 * r + c] = R0[3 * r] * D[c] + R0[3 * r + 1] * D[3 + c] + R0[3 * r + 2] * D[6 + c];
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 3; c++)
        xf[12 * p + 3 * r + c] = (float)(T[3 * r] * R0[3 * c] + T[3 * r + 1] * R0[3 * c + 1] + T[3 * r + 2] * R0[3 * c + 2]);
    for (int r = 0; r < 3; r++)
      xf[12 * p + 9 + r] = (float)(R0[3 * r] * t[3 * p] + R0[3 * r + 1] * t[3 * p + 1] + R0[3 * r + 2] * t[3 * p + 2]);
  }
}

/* The index-deciding arithmetic of k_gn (svn_icp_b200/csrc/iter_kernels.cu), operation by operation:
 *   a = fmaf(A0,sx, fmaf(A1,sy, A2*sz)) ; q = a + tau ; d = fmaf(dz,dz, fmaf(dy,dy, dx*dx)) ; strict '<', first wins;
 *   mask = d_best < (float)max_dist.   (gcc: -ffp-contract=off, fmaf() is the correctly rounded fused op)
 * xf [P][12], sp [n_s][3], rel [n_s][K][3], cidx [n_s][K] -> idx [P][n_s], mask [P][n_s]. */
void oracle_corr_f32(const float *xf, int P, const float *sp, int64_t n_s, const float *rel, const int32_t *cidx, int K,
                     double max_dist, int32_t *idx_out, uint8_t *mask_out) {
  const float Dm = (float)max_dist;
#pragma omp parallel for schedule(static)
  for (int p = 0; p < P; p++) {
    const float *A = xf + 12 * p;
    for (int64_t i = 0; i < n_s; i++) {
      const float sx = sp[3 * i], sy = sp[3 * i + 1], sz = sp[3 * i + 2];
      const float ax = fmaf(A[0], sx, fmaf(A[1], sy, A[2] * sz));
      const float ay = fmaf(A[3], sx, fmaf(A[4], sy, A[5] * sz));
      const float az = fmaf(A[6], sx, fmaf(A[7], sy, A[8] * sz));
      const float qx = ax + A[9], qy = ay + A[10], qz = az + A[11];
      float best = INFINITY;
      int bi = 0;
      for (int k = 0; k < K; k++) {
        const float *c = rel + (i * K + k) * 3;
        const float dx = qx - c[0], dy = qy - c[1], dz = qz - c[2];
        const float d = fmaf(dz, dz, fmaf(dy, dy, dx * dx));
        if (d < best) { best = d; bi = k; }
      }
      idx_out[(size_t)p * n_s + i] = cidx[i * K + bi];
      mask_out[(size_t)p * n_s + i] = (best < Dm) ? 1 : 0;
    }
  }
}

/* Newton_grad_right (SVNICP.cpp:116-164) in fp64 for GIVEN correspondences (global map index + mask per
 * (particle, point)), so the Gauss-Newton arithmetic of the CUDA path can be checked independently of the
 * handful of near-tie index differences between fp32 and fp64 geometry.  R,t [P][9],[P][3]. */
void oracle_gn_given_corr(const double *R, const double *t, int P, const double R0[9], const double t0[3],
                          const double *src, int64_t n_s, const double *tgt, const int32_t *corr_idx,
                          const uint8_t *corr_mask, double max_dist, double *H, double *b) {
#pragma omp parallel for schedule(dynamic, 1)
  for (int p = 0; p < P; p++) {
    double Rt[9], tt[3], R0t[3];
    mat3_mul(R0, R + 9 * p, Rt);
    mat3_vec(R0, t + 3 * p, R0t);
    for (int c = 0; c < 3; c++) tt[c] = t0[c] + R0t[c];
    double *Hp = H + 36 * p, *bp = b + 6 * p;
    memset(Hp, 0, 36 * sizeof(double));
    memset(bp, 0, 6 * sizeof(double));
    for (int64_t i = 0; i < n_s; i++) {
      const double *s = src + 3 * i;
      const double mu = corr_mask[(size_t)p * n_s + i] ? 1.0 : 0.0;
      const double *m = tgt + 3 * (int64_t)corr_idx[(size_t)p * n_s + i];
      double q[3], e[3];
      for (int r = 0; r < 3; r++) q[r] = Rt[3 * r] * s[0] + Rt[3 * r + 1] * s[1] + Rt[3 * r + 2] * s[2] + tt[r];
      for (int r = 0; r < 3; r++) e[r] = mu * q[r] - mu * m[r];
      double sp[3] = {mu * s[0], mu * s[1], mu * s[2]};
      double en = sqrt(e[0] * e[0] + e[1] * e[1] + e[2] * e[2]);
      double w = max_dist / (max_dist + 3.0 * en);
      w = w * w;
      double sh[9] = {0, -sp[2], sp[1], sp[2], 0, -sp[0], -sp[1], sp[0], 0};
      double Rs[9], J[18];
      mat3_mul(Rt, sh, Rs);
      for (int r = 0; r < 3; r++)
        for (int c = 0; c < 3; c++) { J[6 * r + c] = Rt[3 * r + c]; J[6 * r + 3 + c] = -Rs[3 * r + c]; }
      for (int k = 0; k < 6; k++) {
        for (int l = 0; l < 6; l++) {
          double acc = 0;
          for (int r = 0; r < 3; r++) acc += J[6 * r + k] * (J[6 * r + l] * w);
          Hp[6 * k + l] += acc;
        }
        double accb = 0;
        for (int r = 0; r < 3; r++) accb += J[6 * r + k] * (w * e[r]);
        bp[k] += accb;
      }
    }
    for (int k = 0; k < 6; k++) Hp[7 * k] += 1e-6;
  }
}
