// The mean || max reduction of one pooled feature column, shared by pool_fwd_kernel (pool.cu) and
// the multi-tower pooling of ensemble.cu so that both produce bitwise equal results.
#pragma once
#include "common.cuh"

// Column f = slot * d + k of sample b over the segments of every group (positions in group order).
// ptrs[g * n_slots + slot] is a (B, len[g], d) tensor of T.  Writes the first maximum's flat
// position to *arg when WithArg.
template <typename T, bool WithArg>
__device__ __forceinline__ void pool_column(const void* const* ptrs, const int* len, int n_groups,
                                            int n_slots, int64_t b, int d, int slot, int k,
                                            float& sum, float& mx, int* arg) {
  sum = 0.f;
  mx = -INFINITY;
  int a = 0, pos = 0;
  for (int g = 0; g < n_groups; ++g) {
    const T* __restrict__ p = static_cast<const T*>(ptrs[g * n_slots + slot]) +
                              b * (int64_t)len[g] * d + k;
    // eight independent loads in flight per thread (the positions of one feature are d elements
    // apart: one load at a time left the kernel waiting on memory latency 320 times in a row)
    const int n = len[g];
    int t = 0;
    for (; t + 8 <= n; t += 8) {
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = to_f(p[(int64_t)(t + j) * d]);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        sum += v[j];
        if (v[j] > mx) { mx = v[j]; if (WithArg) a = pos + j; }  // strict '>' keeps the FIRST maximum
      }
      pos += 8;
    }
    for (; t < n; ++t, ++pos) {
      const float v = to_f(p[(int64_t)t * d]);
      sum += v;
      if (v > mx) { mx = v; if (WithArg) a = pos; }
    }
  }
  if (WithArg) *arg = a;
}
