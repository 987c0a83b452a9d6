/*
 * map_nn_oracle.c -- brute-force nearest map point, the contract of svnicp_map_evaluate.  TEST INFRASTRUCTURE ONLY:
 * tests/test_map_evaluate_cpu.py compiles it (gcc -O2 -ffp-contract=off -fopenmp -shared) into a temporary directory.
 *
 * For every fp64 query, over all float map points widened to double, d^2 = fma(dz, dz, fma(dy, dy, dx * dx)) (the fma order
 * of the device's dist2); the point with the smallest d^2 < max_dist wins, an exact tie goes to the lexicographically smallest
 * (x, y, z).  A non-finite query has no point.
 * Outputs per query: nearest [3] (zeros where none), d2 (0 where none), mask, idx = map row (-1 where none).
 */
#include <math.h>
#include <stdint.h>

void oracle_map_nn(const double *q, int64_t n, const float *map, int64_t n_map, double max_dist, float *nearest, double *d2,
                   uint8_t *mask, int64_t *idx) {
#pragma omp parallel for schedule(dynamic, 64)
  for (int64_t i = 0; i < n; i++) {
    const double qx = q[3 * i], qy = q[3 * i + 1], qz = q[3 * i + 2];
    double bd = max_dist;
    int64_t bj = -1;
    for (int64_t j = 0; j < n_map; j++) {
      const float *p = map + 3 * j;
      const double dx = qx - (double)p[0], dy = qy - (double)p[1], dz = qz - (double)p[2];
      const double d = fma(dz, dz, fma(dy, dy, dx * dx));
      int take = d < bd;
      if (!take && bj >= 0 && d == bd) {
        const float *b = map + 3 * bj;
        take = p[0] < b[0] || (p[0] == b[0] && (p[1] < b[1] || (p[1] == b[1] && p[2] < b[2])));
      }
      if (take) { bd = d; bj = j; }
    }
    for (int c = 0; c < 3; c++) nearest[3 * i + c] = bj >= 0 ? map[3 * bj + c] : 0.0f;
    d2[i] = bj >= 0 ? bd : 0.0;
    mask[i] = bj >= 0;
    idx[i] = bj;
  }
}
