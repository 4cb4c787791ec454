// Counter-based dropout mask shared by every kernel that draws or regenerates one (the grouped
// dropout of reduce.cu, the dropout epilogue of the grouped projection GEMM and its backward
// reduction), so that they all draw the same mask for the same (seed, step, element index).
#pragma once
#include <stdint.h>

// splitmix64-style hash of (seed, index) -> 64 well-mixed bits
__device__ __forceinline__ uint64_t hash_bits(uint64_t seed, uint64_t i) {
  uint64_t z = seed + 0x9E3779B97F4A7C15ull * (i + 1);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

// A grouped-dropout seed as the kernels use it: the per-tensor seed plus the device step counter
// (nullable), read when the kernel runs so that a replayed CUDA graph draws new masks.
__device__ __forceinline__ uint64_t drop_seed(uint64_t seed, const unsigned long long* step) {
  return seed + (step ? step[0] * 0xD6E8FEB86659FD93ull : 0ull);
}

// Element i of a contiguous tensor is kept iff its 16-bit field of hash_bits(seed, i >> 2) is at
// least thr = round(p * 65536); h is that hash.
__device__ __forceinline__ bool drop_keep(uint64_t h, uint64_t i, uint32_t thr) {
  return ((uint32_t)(h >> (16 * (i & 3))) & 0xFFFFu) >= thr;
}
