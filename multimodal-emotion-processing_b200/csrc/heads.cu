// Emotion heads and losses: O(B*C) float32 work, latency-bound.  Each kernel replaces a python
// loop or a dozen tiny ATen launches of the reference.
//   state_transfer : others/realformer.py:274-286 (window recurrence)
//   bilinear_head  : cmu-mosei/run.py:332-339, Ren-MME/run.py:285-292, rencecps/run.py:141-148
//   circle_loss    : others/realformer.py:289-298 (and its copies)
//   rdrop_kl       : Ren-MME/run.py:332-334
#include "heads.cuh"

namespace {

constexpr int CMAX = HEAD_CMAX;

// ---------------------------------------------------------------------------------------------
// One WARP per sample: lane k owns class k; the (C x C) transfer matrix sits in shared memory and
// the previous window's mixed output travels between lanes by shuffles.  (One thread per sample
// with register arrays indexed at run time put those arrays in local memory and left 31 lanes
// idle: 280 us for B = 32 - the step's longest single kernel.)
__global__ void __launch_bounds__(256)
state_transfer_fwd_kernel(const float* __restrict__ feats, const float* __restrict__ trans,
                          float* __restrict__ out, int B, int P, int C) {
  __shared__ float T[CMAX * CMAX];
  for (int i = threadIdx.x; i < C * C; i += blockDim.x) T[i] = trans[i];
  __syncthreads();
  const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (b >= B) return;
  st_fwd_sample(feats, T, out, b, P, C, threadIdx.x & 31);
}

__global__ void __launch_bounds__(256)
state_transfer_bwd_kernel(const float* __restrict__ dout, const float* __restrict__ feats,
                          const float* __restrict__ trans, const float* __restrict__ out,
                          float* __restrict__ dfeats, float* __restrict__ dtrans, int B, int P,
                          int C) {
  __shared__ float T[CMAX * CMAX];
  for (int i = threadIdx.x; i < C * C; i += blockDim.x) T[i] = trans[i];
  __syncthreads();
  const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (b >= B) return;
  st_bwd_sample(dout, feats, T, out, dfeats, dtrans, b, P, C, threadIdx.x & 31);
}

// ---------------------------------------------------------------------------------------------
// One warp per sample; lanes < C own output class k (and lanes < 2C own concat column i).
__global__ void __launch_bounds__(256)
bilinear_fwd_kernel(const float* __restrict__ th, const float* __restrict__ la,
                    const float* __restrict__ T, const float* __restrict__ gamma,
                    const float* __restrict__ beta, const float* __restrict__ W,
                    const float* __restrict__ bias, float* __restrict__ out,
                    float* __restrict__ zsave, int B, int C, float eps) {
  const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (b >= B) return;
  bilinear_fwd_sample(th, la, T, gamma, beta, W, bias, out, zsave, b, C, eps, threadIdx.x & 31);
}

__global__ void __launch_bounds__(256)
bilinear_bwd_kernel(const float* __restrict__ dout, const float* __restrict__ th,
                    const float* __restrict__ la, const float* __restrict__ T,
                    const float* __restrict__ gamma, const float* __restrict__ W,
                    const float* __restrict__ zsave, float* __restrict__ dth,
                    float* __restrict__ dla, float* __restrict__ dT, float* __restrict__ dgamma,
                    float* __restrict__ dbeta, float* __restrict__ dbias, int B, int C, float eps,
                    int copies) {
  extern __shared__ float sm[];
  bilinear_bwd_cta(sm, dout, th, la, T, gamma, W, zsave, dth, dla, dT, dgamma, dbeta, dbias, B, C,
                   eps, copies, blockIdx.x, gridDim.x);
}

// dW[n][i] += sum_b dy[b][n] cat[b][i]: thread per (n, i); blockIdx.y splits the batch into strips
// of 16 samples (one atomic per weight per strip) so that B = 256 is not one serial loop.
__global__ void bilinear_dw_kernel(const float* __restrict__ dout, const float* __restrict__ th,
                                   const float* __restrict__ zsave, const float* __restrict__ gamma,
                                   const float* __restrict__ beta, float* __restrict__ dW, int B,
                                   int C, float eps) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 2 * C * C) return;
  const int b0 = blockIdx.y * 16, b1 = min(B, b0 + 16);
  bilinear_dw_strip(dout, th, zsave, gamma, beta, dW, idx, b0, b1, C, eps);
}

// ---------------------------------------------------------------------------------------------
__global__ void circle_loss_fwd_kernel(const float* __restrict__ s, const float* __restrict__ y,
                                       float* __restrict__ loss, int64_t R, int C) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R) return;
  loss[r] = circle_row_loss(s, y, r, C);
}

__global__ void circle_loss_bwd_kernel(const float* __restrict__ dloss, const float* __restrict__ s,
                                       const float* __restrict__ y, float* __restrict__ ds,
                                       int64_t R, int C) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R) return;
  circle_row_bwd(dloss[r], s, y, ds, r, C);
}

// single CTA: n = B/2 pairs x C classes
__global__ void __launch_bounds__(256)
rdrop_fwd_kernel(const float* __restrict__ s, float* __restrict__ out, int n, int C) {
  rdrop_kl_cta(s, out, n, C);
}

__global__ void rdrop_bwd_kernel(const float* __restrict__ dout, const float* __restrict__ s,
                                 float* __restrict__ ds, int n, int C) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n * C) return;
  rdrop_kl_bwd_elem(dout, s, ds, e, n, C);
}

}  // namespace

extern "C" {
int mmemo_state_transfer_fwd(const float* feats, const float* trans, float* out, int64_t B,
                             int64_t P, int64_t C, mmemo_stream_t s) {
  if (B <= 0 || P <= 0) return MMEMO_OK;
  MM_REQUIRE(feats && trans && out);
  if (C < 1 || C > CMAX) return MMEMO_ERR_SHAPE;
  state_transfer_fwd_kernel<<<(unsigned)cdiv(B, 8), 256, 0, mm_stream(s)>>>(feats, trans, out,
                                                                           (int)B, (int)P, (int)C);
  MM_LAUNCH_OK();
  return MMEMO_OK;
}
int mmemo_state_transfer_bwd(const float* dout, const float* feats, const float* trans,
                             const float* out, float* dfeats, float* dtrans, int64_t B, int64_t P,
                             int64_t C, mmemo_stream_t s) {
  if (B <= 0 || P <= 0) return MMEMO_OK;
  MM_REQUIRE(dout && feats && trans && out && dfeats);
  if (C < 1 || C > CMAX) return MMEMO_ERR_SHAPE;
  state_transfer_bwd_kernel<<<(unsigned)cdiv(B, 8), 256, 0, mm_stream(s)>>>(
      dout, feats, trans, out, dfeats, dtrans, (int)B, (int)P, (int)C);
  MM_LAUNCH_OK();
  return MMEMO_OK;
}
int mmemo_bilinear_head_fwd(const float* this_feat, const float* last_feat, const float* trans,
                            const float* gamma, const float* beta, const float* w,
                            const float* bias, float* out, float* z, int64_t B, int64_t C,
                            float eps, mmemo_stream_t s) {
  if (B <= 0) return MMEMO_OK;
  MM_REQUIRE(this_feat && last_feat && trans && gamma && beta && w && bias && out && z);
  if (C < 1 || C > CMAX) return MMEMO_ERR_SHAPE;
  bilinear_fwd_kernel<<<(unsigned)cdiv(B, 8), 256, 0, mm_stream(s)>>>(
      this_feat, last_feat, trans, gamma, beta, w, bias, out, z, (int)B, (int)C, eps);
  MM_LAUNCH_OK();
  return MMEMO_OK;
}
int mmemo_bilinear_head_bwd(const float* dout, const float* this_feat, const float* last_feat,
                            const float* trans, const float* gamma, const float* beta,
                            const float* w, const float* z, float* dthis, float* dlast,
                            float* dtrans, float* dgamma, float* dbeta, float* dw, float* dbias,
                            int64_t B, int64_t C, float eps, mmemo_stream_t s) {
  if (B <= 0) return MMEMO_OK;
  MM_REQUIRE(dout && this_feat && last_feat && trans && gamma && beta && w && z && dthis && dlast);
  if (C < 1 || C > CMAX) return MMEMO_ERR_SHAPE;
  const int copies = bilinear_bwd_copies(C);
  const size_t smem = bilinear_bwd_smem(C);
  const int64_t blocks = bilinear_bwd_ctas(B);
  bilinear_bwd_kernel<<<(unsigned)blocks, 256, smem, mm_stream(s)>>>(
      dout, this_feat, last_feat, trans, gamma, w, z, dthis, dlast, dtrans, dgamma, dbeta, dbias,
      (int)B, (int)C, eps, copies);
  MM_LAUNCH_OK();
  if (dw) {  // dW needs the full concat value LN(z)+beta: thread per weight, loop over the batch
    bilinear_dw_kernel<<<dim3((unsigned)cdiv(2 * C * C, 128), (unsigned)cdiv(B, 16)), 128, 0,
                         mm_stream(s)>>>(
        dout, this_feat, z, gamma, beta, dw, (int)B, (int)C, eps);
    MM_LAUNCH_OK();
  }
  return MMEMO_OK;
}
int mmemo_circle_loss_fwd(const float* logits, const float* labels, float* loss, int64_t R,
                          int64_t C, mmemo_stream_t s) {
  if (R <= 0) return MMEMO_OK;
  MM_REQUIRE(logits && labels && loss && C > 0);
  circle_loss_fwd_kernel<<<(unsigned)cdiv(R, 128), 128, 0, mm_stream(s)>>>(logits, labels, loss, R,
                                                                          (int)C);
  MM_LAUNCH_OK();
  return MMEMO_OK;
}
int mmemo_circle_loss_bwd(const float* dloss, const float* logits, const float* labels,
                          float* dlogits, int64_t R, int64_t C, mmemo_stream_t s) {
  if (R <= 0) return MMEMO_OK;
  MM_REQUIRE(dloss && logits && labels && dlogits && C > 0);
  circle_loss_bwd_kernel<<<(unsigned)cdiv(R, 128), 128, 0, mm_stream(s)>>>(dloss, logits, labels,
                                                                          dlogits, R, (int)C);
  MM_LAUNCH_OK();
  return MMEMO_OK;
}
int mmemo_rdrop_kl_fwd(const float* logits, float* out, int64_t B, int64_t C, mmemo_stream_t s) {
  MM_REQUIRE(logits && out && C > 0 && B >= 2 && (B % 2) == 0);
  rdrop_fwd_kernel<<<1, 256, 0, mm_stream(s)>>>(logits, out, (int)(B / 2), (int)C);
  MM_LAUNCH_OK();
  return MMEMO_OK;
}
int mmemo_rdrop_kl_bwd(const float* dout, const float* logits, float* dlogits, int64_t B, int64_t C,
                       mmemo_stream_t s) {
  MM_REQUIRE(dout && logits && dlogits && C > 0 && B >= 2 && (B % 2) == 0);
  const int n = (int)(B / 2);
  rdrop_bwd_kernel<<<(unsigned)cdiv((int64_t)n * C, 128), 128, 0, mm_stream(s)>>>(dout, logits,
                                                                                 dlogits, n, (int)C);
  MM_LAUNCH_OK();
  return MMEMO_OK;
}
}
