/*
 * map_snapshot_oracle.c -- the canonical snapshot of the sequential local-map oracle, the contract of svnicp_map_export.
 * TEST INFRASTRUCTURE ONLY: tests/test_map_snapshot_cpu.py compiles it (gcc -O2 -ffp-contract=off, the flags of oracle/Makefile)
 * into a temporary directory.  It includes oracle/voxelmap_oracle.c unchanged, so the library holds the whole oracle map
 * (oracle_vmap_create / add / get / size / clear) plus the export below.
 *
 * The live entries, sorted by (vx, vy, vz) on the host; each voxel's points in the order the oracle keeps them (arrival order).
 */
#include "../oracle/voxelmap_oracle.c"

static int vm_entry_cmp(const void *a, const void *b) {
  const vm_entry *x = *(const vm_entry *const *)a, *y = *(const vm_entry *const *)b;
  for (int c = 0; c < 3; c++)
    if (x->v[c] != y->v[c]) return x->v[c] < y->v[c] ? -1 : 1;
  return 0;
}

/* live voxels and their points (what a snapshot's V and Npts are) */
void oracle_vmap_snapshot_size(vmap *m, int64_t *n_voxels, int64_t *n_points) {
  int64_t V = 0, N = 0;
  for (size_t i = 0; i < m->slots; i++)
    if (m->tab[i].used == 1 && m->tab[i].count > 0) { V++; N += m->tab[i].count; }
  *n_voxels = V;
  *n_points = N;
}

/* voxels [V][3], counts [V], xyz [Npts][3] in the layout of svnicp_map_export; returns 0, or -1 when out of memory */
int oracle_vmap_export(vmap *m, int32_t *voxels, int32_t *counts, float *xyz) {
  int64_t V, N;
  oracle_vmap_snapshot_size(m, &V, &N);
  vm_entry **live = (vm_entry **)malloc(sizeof(vm_entry *) * (size_t)(V > 0 ? V : 1));
  if (!live) return -1;
  int64_t k = 0;
  for (size_t i = 0; i < m->slots; i++)
    if (m->tab[i].used == 1 && m->tab[i].count > 0) live[k++] = &m->tab[i];
  qsort(live, (size_t)V, sizeof(vm_entry *), vm_entry_cmp);
  int64_t p = 0;
  for (int64_t i = 0; i < V; i++) {
    memcpy(voxels + 3 * i, live[i]->v, 3 * sizeof(int32_t));
    counts[i] = live[i]->count;
    memcpy(xyz + 3 * p, live[i]->pts, 3 * sizeof(float) * (size_t)live[i]->count);
    p += live[i]->count;
  }
  free(live);
  return 0;
}
