// Uncertainty of a k-fold ensemble's prediction from the folds' logits (inference): per row, the
// softmax of every fold, their mean and unbiased variance per class, the entropy of the mean, the
// mean of the folds' entropies, their difference (mutual information) and the argmax label.
#include <math.h>

#include "common.cuh"

namespace {

constexpr int UQ_NT = 256;               // 8 rows (warps) per CTA
constexpr int UQ_MAX_CHUNKS = 32;        // classes per lane: C <= 32 * 32

// One warp per row n of logits (K, N, C); lane owns classes c = j * 32 + lane, j < J.  The folds
// are walked in order with the next fold's logits loaded before the current one is reduced.
// Per fold: m = max_c x, s = sum_c exp(x - m), p = exp(x - m) / s, H_k = log s - sum_c p (x - m)
// (= -sum_c p log p without evaluating log p of an underflowed p).  Per class mean and sum of
// squared deviations across folds by Welford's update.
template <typename T, int J>
__global__ void __launch_bounds__(UQ_NT)
fold_uncertainty_kernel(const T* __restrict__ x, int K, int64_t N, int C, float* __restrict__ mean_p,
                        float* __restrict__ var_p, float* __restrict__ ent,
                        float* __restrict__ exp_ent, float* __restrict__ mi,
                        int64_t* __restrict__ label) {
  const int lane = threadIdx.x & 31;
  const int64_t n = (int64_t)blockIdx.x * (UQ_NT / 32) + (threadIdx.x >> 5);
  if (n >= N) return;                    // whole warps leave together
  const T* row = x + n * C;
  const int64_t fold_stride = N * (int64_t)C;
  float nxt[J], mu[J], m2[J];
#pragma unroll
  for (int j = 0; j < J; ++j) {
    const int c = j * 32 + lane;
    nxt[j] = c < C ? to_f(row[c]) : -INFINITY;
    mu[j] = 0.f;
    m2[j] = 0.f;
  }
  float h_sum = 0.f;
  for (int k = 0; k < K; ++k) {
    float cur[J];
#pragma unroll
    for (int j = 0; j < J; ++j) cur[j] = nxt[j];
    if (k + 1 < K) {
      const T* r1 = row + (int64_t)(k + 1) * fold_stride;
#pragma unroll
      for (int j = 0; j < J; ++j) {
        const int c = j * 32 + lane;
        nxt[j] = c < C ? to_f(r1[c]) : -INFINITY;
      }
    }
    float m = cur[0];
#pragma unroll
    for (int j = 1; j < J; ++j) m = fmaxf(m, cur[j]);
    m = warp_max(m);
    float e[J], s = 0.f;
#pragma unroll
    for (int j = 0; j < J; ++j) {
      e[j] = j * 32 + lane < C ? expf(cur[j] - m) : 0.f;
      s += e[j];
    }
    s = warp_sum(s);
    float pz = 0.f;
    const float inv_n = 1.0f / (float)(k + 1);
#pragma unroll
    for (int j = 0; j < J; ++j) {
      const float p = e[j] / s;
      if (p > 0.f) pz = fmaf(p, cur[j] - m, pz);
      const float dlt = p - mu[j];
      mu[j] = fmaf(dlt, inv_n, mu[j]);
      m2[j] = fmaf(dlt, p - mu[j], m2[j]);
    }
    h_sum += logf(s) - warp_sum(pz);
  }
  // entropy of the mean and the argmax (first maximum)
  float plogp = 0.f, best = -INFINITY;
  int best_c = 0;
#pragma unroll
  for (int j = 0; j < J; ++j) {
    const int c = j * 32 + lane;
    if (c < C) {
      if (mu[j] > 0.f) plogp = fmaf(mu[j], logf(mu[j]), plogp);
      if (mu[j] > best) { best = mu[j]; best_c = c; }
      mean_p[n * C + c] = mu[j];
      var_p[n * C + c] = K > 1 ? m2[j] / (float)(K - 1) : 0.f;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int oc = __shfl_xor_sync(0xffffffffu, best_c, o);
    if (ob > best || (ob == best && oc < best_c)) { best = ob; best_c = oc; }
  }
  const float h = -warp_sum(plogp);
  if (lane == 0) {
    const float eh = h_sum / (float)K;
    ent[n] = h;
    exp_ent[n] = eh;
    mi[n] = K > 1 ? fmaxf(h - eh, 0.f) : 0.f;   // >= 0 by Jensen; the clamp absorbs rounding
    label[n] = best_c;
  }
}

template <typename T, int J>
void launch_j(const T* x, int K, int64_t N, int C, float* mp, float* vp, float* en, float* ee,
              float* mi, int64_t* lb, cudaStream_t st) {
  const unsigned grid = (unsigned)cdiv(N, UQ_NT / 32);
  fold_uncertainty_kernel<T, J><<<grid, UQ_NT, 0, st>>>(x, K, N, C, mp, vp, en, ee, mi, lb);
}

template <typename T>
int fold_uncertainty(const void* logits, int64_t K, int64_t N, int64_t C, float* mean_p,
                     float* var_p, float* ent, float* exp_ent, float* mi, int64_t* label,
                     cudaStream_t st) {
  MM_REQUIRE(K >= 1 && K <= INT32_MAX && N >= 0 && C >= 1);
  if (C > 32 * UQ_MAX_CHUNKS || cdiv(N, UQ_NT / 32) > INT32_MAX) return MMEMO_ERR_SHAPE;
  if (N == 0) return MMEMO_OK;           // empty buffers may have null pointers
  MM_REQUIRE(logits && mean_p && var_p && ent && exp_ent && mi && label);
  const T* x = static_cast<const T*>(logits);
  const int k = (int)K, c = (int)C;
  if (C <= 32) launch_j<T, 1>(x, k, N, c, mean_p, var_p, ent, exp_ent, mi, label, st);
  else if (C <= 64) launch_j<T, 2>(x, k, N, c, mean_p, var_p, ent, exp_ent, mi, label, st);
  else if (C <= 128) launch_j<T, 4>(x, k, N, c, mean_p, var_p, ent, exp_ent, mi, label, st);
  else if (C <= 256) launch_j<T, 8>(x, k, N, c, mean_p, var_p, ent, exp_ent, mi, label, st);
  else if (C <= 512) launch_j<T, 16>(x, k, N, c, mean_p, var_p, ent, exp_ent, mi, label, st);
  else launch_j<T, 32>(x, k, N, c, mean_p, var_p, ent, exp_ent, mi, label, st);
  MM_LAUNCH_OK();
  return MMEMO_OK;
}

}  // namespace

extern "C" {
int mmemo_fold_uncertainty_f32(const void* logits, int64_t K, int64_t N, int64_t C, float* mean_prob,
                               float* var_prob, float* entropy, float* expected_entropy,
                               float* mutual_info, int64_t* label, mmemo_stream_t s) {
  return fold_uncertainty<float>(logits, K, N, C, mean_prob, var_prob, entropy, expected_entropy,
                                 mutual_info, label, mm_stream(s));
}
int mmemo_fold_uncertainty_bf16(const void* logits, int64_t K, int64_t N, int64_t C,
                                float* mean_prob, float* var_prob, float* entropy,
                                float* expected_entropy, float* mutual_info, int64_t* label,
                                mmemo_stream_t s) {
  return fold_uncertainty<bf16>(logits, K, N, C, mean_prob, var_prob, entropy, expected_entropy,
                                mutual_info, label, mm_stream(s));
}
}
