/*
 * map_refine_oracle.c -- fp64 restatement of svnicp_map_refine.  TEST INFRASTRUCTURE ONLY: tests/test_map_refine_cpu.py compiles
 * it (gcc -O2 -ffp-contract=off -fopenmp -shared) into a temporary directory.
 *
 * Per pose and iteration (svnicp_map_refine's contract, include/svnicp_b200.h):
 *   R~ = R0 Exp(omega), t~ = t0 + R0 t (x = 0: R0, t0 as given); q = R~ s + t~ with fma() in affine_row_fma's order;
 *   the exact nearest map point with d^2 < max_dist (map_nn_oracle.c's rule: fma(dz, dz, fma(dy, dy, dx * dx)), an exact tie to
 *   the lexicographically smallest (x, y, z)), found among the map points of the x-slab |p_x - q_x| <= sqrt(max_dist) (1 + 1e-9)
 *   of a sorted copy, which holds every point with d^2 < max_dist;
 *   Newton_grad_right on those correspondences (oracle_gn_given_corr of oracle/svn_oracle.c: J = [R~, -R~ [s]x], e = q - m,
 *   w = (D / (D + 3 |e|))^2), a point without a correspondence adding I to the translation block (Q2), + 1e-6 I (Q3);
 *   delta = -H^-1 b by LDL^T in ldl_solve6_reg's operation order; the update of tail2.cu:673-690 with J_l = I at delta_w = 0;
 *   x' = [t' ; principal Log(R')]; |delta| in tail2.cu:691's order; an exactly zero delta leaves x unchanged; stop after the
 *   update with |delta| < tol or after `iterations` updates.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

/* SVNICP::to_rotation_tensor (SVNICP.cpp:166-194), as svn::so3_exp: J_l is NaN at a zero angle (Q7); the caller decides */
void oracle_so3_exp(const double r[3], double R[9], double Jl[9]) {
  const double a = sqrt(r[0] * r[0] + r[1] * r[1] + r[2] * r[2]);
  double n[3];
  const double ia = 1.0 / a;
  if (a < 1e-12) { n[0] = n[1] = n[2] = 0.0; }
  else { n[0] = r[0] * ia; n[1] = r[1] * ia; n[2] = r[2] * ia; }
  const double s = sin(a), c = cos(a);
  const double ah[9] = {0, -n[2], n[1], n[2], 0, -n[0], -n[1], n[0], 0};
  const double sa = s * ia, ca = (1.0 - c) * ia;
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) {
      const double id = (i == j) ? 1.0 : 0.0, nn = n[i] * n[j];
      R[3 * i + j] = c * id + (1.0 - c) * nn + s * ah[3 * i + j];
      if (Jl) Jl[3 * i + j] = sa * id + (1.0 - sa) * nn + ca * ah[3 * i + j];
    }
}

/* svn::so3_log_principal (common.cuh) */
void oracle_so3_log_principal(const double R[9], double w[3]) {
  const double v[3] = {R[7] - R[5], R[2] - R[6], R[3] - R[1]};
  const double s = 0.5 * sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
  const double c = 0.5 * (R[0] + R[4] + R[8] - 1.0);
  const double a = atan2(s, c);
  if (c >= 0.0) {
    const double f = s > 0.0 ? 0.5 * a / s : 0.5;
    for (int j = 0; j < 3; j++) w[j] = f * v[j];
    return;
  }
  const double B[9] = {R[0] - c, 0.5 * (R[1] + R[3]), 0.5 * (R[2] + R[6]),
                       0.5 * (R[1] + R[3]), R[4] - c, 0.5 * (R[5] + R[7]),
                       0.5 * (R[2] + R[6]), 0.5 * (R[5] + R[7]), R[8] - c};
  const int k = (B[0] >= B[4] && B[0] >= B[8]) ? 0 : (B[4] >= B[8] ? 1 : 2);
  const double *n = B + 3 * k;
  const double nn = sqrt(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
  const double f = ((n[0] * v[0] + n[1] * v[1] + n[2] * v[2]) < 0.0 ? -a : a) / nn;
  for (int j = 0; j < 3; j++) w[j] = f * n[j];
}

/* svn::ldl_solve6_reg's operation order (upper triangle of A read; A overwritten; b <- A^-1 b) */
static void ldl_solve6(double A[36], double b[6]) {
  double L[36] = {0}, iD[6];
  for (int j = 0; j < 6; j++) {
    double w[6], d = A[j * 6 + j];
    for (int k = 0; k < j; k++) {
      w[k] = L[j * 6 + k] * A[k * 6 + k];
      d -= L[j * 6 + k] * w[k];
    }
    A[j * 6 + j] = d;
    iD[j] = 1.0 / d;
    for (int i = j + 1; i < 6; i++) {
      double sum = A[j * 6 + i];
      for (int k = 0; k < j; k++) sum -= L[i * 6 + k] * w[k];
      L[i * 6 + j] = sum * iD[j];
    }
  }
  for (int i = 1; i < 6; i++)
    for (int k = 0; k < i; k++) b[i] -= L[i * 6 + k] * b[k];
  for (int i = 0; i < 6; i++) b[i] *= iD[i];
  for (int i = 4; i >= 0; i--)
    for (int k = i + 1; k < 6; k++) b[i] -= L[k * 6 + i] * b[k];
}

/* One update from the system at x: x_out (may alias x), returns |delta| */
double oracle_refine_update(const double x[6], const double H[36], const double b[6], double x_out[6]) {
  double A[36], d[6];
  memcpy(A, H, sizeof(A));
  memcpy(d, b, sizeof(d));
  ldl_solve6(A, d);
  for (int i = 0; i < 6; i++) d[i] = -d[i];
  const double dn = sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2] + d[3] * d[3] + d[4] * d[4] + d[5] * d[5]);
  if (d[0] == 0.0 && d[1] == 0.0 && d[2] == 0.0 && d[3] == 0.0 && d[4] == 0.0 && d[5] == 0.0) {
    memmove(x_out, x, 6 * sizeof(double));
    return dn;
  }
  double R[9], dR[9], Jl[9], Rn[9], dt[3], t[3], w[3];
  oracle_so3_exp(x + 3, R, NULL);
  oracle_so3_exp(d + 3, dR, Jl);
  const int rot0 = d[3] == 0.0 && d[4] == 0.0 && d[5] == 0.0;
  for (int r = 0; r < 3; r++) dt[r] = rot0 ? d[r] : Jl[3 * r] * d[0] + Jl[3 * r + 1] * d[1] + Jl[3 * r + 2] * d[2];
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) Rn[3 * r + c] = R[3 * r] * dR[c] + R[3 * r + 1] * dR[3 + c] + R[3 * r + 2] * dR[6 + c];
  for (int r = 0; r < 3; r++) t[r] = (Rn[3 * r] * dt[0] + Rn[3 * r + 1] * dt[1] + Rn[3 * r + 2] * dt[2]) + x[r];
  oracle_so3_log_principal(Rn, w);
  for (int q = 0; q < 3; q++) { x_out[q] = t[q]; x_out[3 + q] = w[q]; }
  return dn;
}

typedef struct {
  const float *map;  /* [n_map][3] */
  int64_t *order;    /* map rows by ascending x */
  int64_t n_map;
} slab_map;

static const slab_map *g_sort_map;
static int cmp_x(const void *a, const void *b) {
  const float xa = g_sort_map->map[3 * *(const int64_t *)a], xb = g_sort_map->map[3 * *(const int64_t *)b];
  return xa < xb ? -1 : (xa > xb ? 1 : 0);
}

/* exact nearest map row of q with d^2 < max_dist (-1 where none), d^2 in *bd */
static int64_t nearest(const slab_map *sm, const double q[3], double max_dist, double *bd_out) {
  const double r = sqrt(max_dist) * (1.0 + 1e-9);
  int64_t lo = 0, hi = sm->n_map;  /* first sorted position with x >= q_x - r */
  while (lo < hi) {
    const int64_t mid = (lo + hi) / 2;
    if ((double)sm->map[3 * sm->order[mid]] < q[0] - r) lo = mid + 1;
    else hi = mid;
  }
  double bd = max_dist;
  int64_t bj = -1;
  for (int64_t k = lo; k < sm->n_map; k++) {
    const float *p = sm->map + 3 * sm->order[k];
    if ((double)p[0] > q[0] + r) break;
    const double dx = q[0] - (double)p[0], dy = q[1] - (double)p[1], dz = q[2] - (double)p[2];
    const double d = fma(dz, dz, fma(dy, dy, dx * dx));
    int take = d < bd;
    if (!take && bj >= 0 && d == bd) {
      const float *b = sm->map + 3 * bj;
      take = p[0] < b[0] || (p[0] == b[0] && (p[1] < b[1] || (p[1] == b[1] && p[2] < b[2])));
    }
    if (take) { bd = d; bj = sm->order[k]; }
  }
  *bd_out = bd;
  return bj;
}

/* Newton_grad_right at x on exact correspondences -> H [36], b [6]; returns the inlier count */
static int64_t system_at(const slab_map *sm, const float *src, int64_t n, const double R0[9], const double t0[3], const double x[6],
                         double max_dist, double H[36], double b[6]) {
  double Rp[9], Rt[9], tt[3];
  oracle_so3_exp(x + 3, Rp, NULL);
  const int zero = x[0] == 0.0 && x[1] == 0.0 && x[2] == 0.0 && x[3] == 0.0 && x[4] == 0.0 && x[5] == 0.0;
  for (int r = 0; r < 3; r++) {
    for (int c = 0; c < 3; c++) Rt[3 * r + c] = zero ? R0[3 * r + c] : R0[3 * r] * Rp[c] + R0[3 * r + 1] * Rp[3 + c] + R0[3 * r + 2] * Rp[6 + c];
    tt[r] = zero ? t0[r] : t0[r] + (R0[3 * r] * x[0] + R0[3 * r + 1] * x[1] + R0[3 * r + 2] * x[2]);
  }
  memset(H, 0, 36 * sizeof(double));
  memset(b, 0, 6 * sizeof(double));
  int64_t cnt = 0;
  for (int64_t i = 0; i < n; i++) {
    const double s[3] = {(double)src[3 * i], (double)src[3 * i + 1], (double)src[3 * i + 2]};
    double q[3];
    for (int a = 0; a < 3; a++) q[a] = fma(Rt[3 * a], s[0], fma(Rt[3 * a + 1], s[1], fma(Rt[3 * a + 2], s[2], tt[a])));
    double bd = 0.0;
    const int64_t j = (isfinite(q[0]) && isfinite(q[1]) && isfinite(q[2])) ? nearest(sm, q, max_dist, &bd) : -1;
    if (j < 0) {
      for (int k = 0; k < 3; k++) H[7 * k] += 1.0;  /* Q2 */
      continue;
    }
    cnt++;
    const float *m = sm->map + 3 * j;
    double e[3];
    for (int r = 0; r < 3; r++) e[r] = q[r] - (double)m[r];
    const double en = sqrt(e[0] * e[0] + e[1] * e[1] + e[2] * e[2]);
    double w = max_dist / (max_dist + 3.0 * en);
    w = w * w;
    const double sh[9] = {0, -s[2], s[1], s[2], 0, -s[0], -s[1], s[0], 0};
    double J[18];
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 3; c++) {
        double rs = 0.0;
        for (int k = 0; k < 3; k++) rs += Rt[3 * r + k] * sh[3 * k + c];
        J[6 * r + c] = Rt[3 * r + c];
        J[6 * r + 3 + c] = -rs;
      }
    for (int k = 0; k < 6; k++) {
      for (int l = 0; l < 6; l++) {
        double acc = 0;
        for (int r = 0; r < 3; r++) acc += J[6 * r + k] * (J[6 * r + l] * w);
        H[6 * k + l] += acc;
      }
      double accb = 0;
      for (int r = 0; r < 3; r++) accb += J[6 * r + k] * (w * e[r]);
      b[k] += accb;
    }
  }
  for (int k = 0; k < 6; k++) H[7 * k] += 1e-6;
  return cnt;
}

/* The whole loop for M poses [6][M]: out_poses [6][M], out_iterations [M], out_step [M], out_count [M] (inliers at the final x) */
void oracle_map_refine(const float *src, int64_t n, const float *map, int64_t n_map, const double R0[9], const double t0[3], int M,
                       const double *poses, double max_dist, int iterations, double tol, double *out_poses, int32_t *out_iterations,
                       double *out_step, int64_t *out_count) {
  slab_map sm = {map, (int64_t *)malloc((size_t)(n_map > 0 ? n_map : 1) * sizeof(int64_t)), n_map};
  for (int64_t k = 0; k < n_map; k++) sm.order[k] = k;
  g_sort_map = &sm;
  qsort(sm.order, (size_t)n_map, sizeof(int64_t), cmp_x);
#pragma omp parallel for schedule(dynamic, 1)
  for (int p = 0; p < M; p++) {
    double x[6], H[36], b[6], dn = 0.0;
    for (int c = 0; c < 6; c++) x[c] = poses[(size_t)c * M + p];
    int it = 0;
    while (it < iterations) {
      system_at(&sm, src, n, R0, t0, x, max_dist, H, b);
      dn = oracle_refine_update(x, H, b, x);
      it++;
      if (dn < tol) break;
    }
    for (int c = 0; c < 6; c++) out_poses[(size_t)c * M + p] = x[c];
    out_iterations[p] = it;
    out_step[p] = dn;
    out_count[p] = system_at(&sm, src, n, R0, t0, x, max_dist, H, b);
  }
  free(sm.order);
}
