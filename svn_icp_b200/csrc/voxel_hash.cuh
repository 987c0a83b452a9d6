// voxel_hash.cuh -- the device open-addressing table of voxel keys shared by the local map (voxel_map.cu), the uniform
// sampling of the scan pre-processor (preprocess.cu) and the per-scan K-NN grid (cand_build.cu).
//
// A key packs a voxel index (ix, iy, iz), each in [-2^20, 2^20), as three 21-bit fields of index + 2^20: x in bits 0-20,
// y in 21-41, z in 42-62.  Bit 63 stays clear, so no key equals EMPTY_KEY.  Slots are probed linearly from a murmur-style
// finaliser of the key; an empty slot holds all ones (a table is cleared with a 0xFF memset).  There are no deletions and so
// no tombstones: a lookup may stop at the first empty slot.  How a coordinate becomes a voxel index is each caller's own rule.
#pragma once
#include <cuda_runtime.h>

namespace svn {

constexpr unsigned long long EMPTY_KEY = ~0ull;

__device__ __forceinline__ unsigned long long pack_voxel_key(int ix, int iy, int iz) {
  const unsigned long long B = 1ull << 20;
  return ((unsigned long long)(ix + (long long)B) & 0x1FFFFFull) | (((unsigned long long)(iy + (long long)B) & 0x1FFFFFull) << 21) |
         (((unsigned long long)(iz + (long long)B) & 0x1FFFFFull) << 42);
}

__device__ __forceinline__ unsigned hash_voxel_key(unsigned long long k) {
  k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
  return (unsigned)k;
}

// Find-or-create in keys[0 .. mask] (mask + 1 a power of two): the slot holding key, or -1 when the table is full.  Reads
// first and claims an empty slot with atomicCAS; *created tells whether this call claimed it.
__device__ __forceinline__ int hash_insert(unsigned long long *keys, unsigned mask, unsigned long long key, bool *created) {
  unsigned slot = hash_voxel_key(key) & mask;
  *created = false;
  for (int probe = 0; probe <= (int)mask; probe++) {
    const unsigned long long k = keys[slot];
    if (k == key) return (int)slot;
    if (k == EMPTY_KEY) {
      const unsigned long long old = atomicCAS(&keys[slot], EMPTY_KEY, key);
      if (old == EMPTY_KEY) { *created = true; return (int)slot; }
      if (old == key) return (int)slot;
    }
    slot = (slot + 1) & mask;
  }
  return -1;
}

// Read-only lookup (through the read-only data cache: the table must not change during the kernel): the slot holding key,
// or -1 when it is absent.
__device__ __forceinline__ int hash_find(const unsigned long long *keys, unsigned mask, unsigned long long key) {
  unsigned slot = hash_voxel_key(key) & mask;
  for (int probe = 0; probe <= (int)mask; probe++) {
    const unsigned long long k = __ldg(keys + slot);
    if (k == key) return (int)slot;
    if (k == EMPTY_KEY) return -1;
    slot = (slot + 1) & mask;
  }
  return -1;
}

}  // namespace svn
