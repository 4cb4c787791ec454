// The heads and losses of k fold models trained together (folds.py): every kernel of heads.cu for
// many members per launch.  blockIdx.y (loss forwards: blockIdx.x) is the member; each member has
// its own pointers and batch size.  The per-sample bodies are those of heads.cu (heads.cuh), so
// every member's forward is bitwise the per-model kernel's.  Parameter gradients go to each
// member's own buffers: float atomics within a member as in heads.cu, none across members.
//   state_transfer_{fwd,bwd}_multi : others/realformer.py:274-286
//   bilinear_head_{fwd,bwd}_multi  : cmu-mosei/run.py:332-339, Ren-MME/run.py:285-292,
//                                    rencecps/run.py:141-148
//   circle_loss_{fwd,bwd}_multi    : (multi_circle_loss(logits, labels) [* weights]).mean()
//   rdrop_kl_{fwd,bwd}_multi       : Ren-MME/run.py:332-334
#include "heads.cuh"

namespace {

constexpr int FOLD_MAX = 32;           // members per launch

struct StTable {
  const float* dout[FOLD_MAX];
  const float* feats[FOLD_MAX];
  const float* trans[FOLD_MAX];
  const float* out[FOLD_MAX];          // forward output (written by fwd, read by bwd)
  float* dfeats[FOLD_MAX];
  float* dtrans[FOLD_MAX];
  int B[FOLD_MAX];
};

__global__ void __launch_bounds__(256)
state_transfer_fwd_multi_kernel(StTable tb, int P, int C) {
  __shared__ float T[HEAD_CMAX * HEAD_CMAX];
  const int mi = blockIdx.y;
  const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (blockIdx.x * 8 >= tb.B[mi]) return;
  for (int i = threadIdx.x; i < C * C; i += blockDim.x) T[i] = tb.trans[mi][i];
  __syncthreads();
  if (b >= tb.B[mi]) return;
  st_fwd_sample(tb.feats[mi], T, const_cast<float*>(tb.out[mi]), b, P, C, threadIdx.x & 31);
}

__global__ void __launch_bounds__(256)
state_transfer_bwd_multi_kernel(StTable tb, int P, int C) {
  __shared__ float T[HEAD_CMAX * HEAD_CMAX];
  const int mi = blockIdx.y;
  const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (blockIdx.x * 8 >= tb.B[mi]) return;
  for (int i = threadIdx.x; i < C * C; i += blockDim.x) T[i] = tb.trans[mi][i];
  __syncthreads();
  if (b >= tb.B[mi]) return;
  st_bwd_sample(tb.dout[mi], tb.feats[mi], T, tb.out[mi], tb.dfeats[mi], tb.dtrans[mi], b, P, C,
                threadIdx.x & 31);
}

struct BhTable {
  const float* dout[FOLD_MAX];
  const float* th[FOLD_MAX];
  const float* la[FOLD_MAX];
  const float* trans[FOLD_MAX];
  const float* gamma[FOLD_MAX];
  const float* beta[FOLD_MAX];
  const float* w[FOLD_MAX];
  const float* bias[FOLD_MAX];
  float* out[FOLD_MAX];
  float* z[FOLD_MAX];                  // forward: written; backward: read
  float* dth[FOLD_MAX];
  float* dla[FOLD_MAX];
  float* dtrans[FOLD_MAX];
  float* dgamma[FOLD_MAX];
  float* dbeta[FOLD_MAX];
  float* dw[FOLD_MAX];
  float* dbias[FOLD_MAX];
  int B[FOLD_MAX];
};

__global__ void __launch_bounds__(256)
bilinear_fwd_multi_kernel(BhTable tb, int C, float eps) {
  const int mi = blockIdx.y;
  const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (b >= tb.B[mi]) return;
  bilinear_fwd_sample(tb.th[mi], tb.la[mi], tb.trans[mi], tb.gamma[mi], tb.beta[mi], tb.w[mi],
                      tb.bias[mi], tb.out[mi], tb.z[mi], b, C, eps, threadIdx.x & 31);
}

__global__ void __launch_bounds__(256)
bilinear_bwd_multi_kernel(BhTable tb, int C, float eps, int copies) {
  extern __shared__ float sm[];
  const int mi = blockIdx.y;
  const int n_ctas = (int)bilinear_bwd_ctas(tb.B[mi]);
  if ((int)blockIdx.x >= n_ctas) return;
  bilinear_bwd_cta(sm, tb.dout[mi], tb.th[mi], tb.la[mi], tb.trans[mi], tb.gamma[mi], tb.w[mi],
                   tb.z[mi], tb.dth[mi], tb.dla[mi], tb.dtrans[mi], tb.dgamma[mi], tb.dbeta[mi],
                   tb.dbias[mi], tb.B[mi], C, eps, copies, blockIdx.x, n_ctas);
}

__global__ void bilinear_dw_multi_kernel(BhTable tb, int C, float eps) {
  const int mi = blockIdx.z;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int b0 = blockIdx.y * 16, b1 = min(tb.B[mi], b0 + 16);
  if (idx >= 2 * C * C || b0 >= tb.B[mi] || !tb.dw[mi]) return;
  bilinear_dw_strip(tb.dout[mi], tb.th[mi], tb.z[mi], tb.gamma[mi], tb.beta[mi], tb.dw[mi], idx, b0,
                    b1, C, eps);
}

struct LossTable {
  const float* dout[FOLD_MAX];         // circle: d mean; rdrop: d kl (scalars)
  const float* s[FOLD_MAX];
  const float* y[FOLD_MAX];
  const float* wt[FOLD_MAX];           // per-row weights or null
  float* out[FOLD_MAX];                // forward: the member's scalar
  float* ds[FOLD_MAX];
  int64_t R[FOLD_MAX];                 // circle: rows; rdrop: pairs
};

// One CTA of 256 threads per member: mean over rows of (weight *) loss, summed in a fixed order.
__global__ void __launch_bounds__(256) circle_loss_fwd_multi_kernel(LossTable tb, int C) {
  __shared__ float red[8];
  const int mi = blockIdx.x;
  const int64_t R = tb.R[mi];
  float acc = 0.f;
  for (int64_t r = threadIdx.x; r < R; r += 256) {
    const float l = circle_row_loss(tb.s[mi], tb.y[mi], r, C);
    acc += tb.wt[mi] ? l * tb.wt[mi][r] : l;
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += red[w];
    tb.out[mi][0] = t / (float)R;
  }
}

// d loss_r = (d mean / R) (* weight_r): the gradient autograd gives the per-row kernel through
// .mean() (and the product with the weights).
__global__ void circle_loss_bwd_multi_kernel(LossTable tb, int C) {
  const int mi = blockIdx.y;
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t R = tb.R[mi];
  if (r >= R) return;
  float g = tb.dout[mi][0] / (float)R;
  if (tb.wt[mi]) g = g * tb.wt[mi][r];
  circle_row_bwd(g, tb.s[mi], tb.y[mi], tb.ds[mi], r, C);
}

__global__ void __launch_bounds__(256) rdrop_kl_fwd_multi_kernel(LossTable tb, int C) {
  const int mi = blockIdx.x;
  rdrop_kl_cta(tb.s[mi], tb.out[mi], (int)tb.R[mi], C);
}

__global__ void rdrop_kl_bwd_multi_kernel(LossTable tb, int C) {
  const int mi = blockIdx.y;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = (int)tb.R[mi];
  if (e >= n * C) return;
  rdrop_kl_bwd_elem(tb.dout[mi], tb.s[mi], tb.ds[mi], e, n, C);
}

template <typename T>
const T* at(const T* const* a, int i) { return a ? a[i] : nullptr; }
template <typename T>
T* at(T* const* a, int i) { return a ? a[i] : nullptr; }

}  // namespace

extern "C" {
int mmemo_state_transfer_fwd_multi(int n, const float* const* feats, const float* const* trans,
                                   float* const* out, const int64_t* B, int64_t P, int64_t C,
                                   mmemo_stream_t s) {
  MM_REQUIRE(n >= 0 && (n == 0 || (feats && trans && out && B)));
  if (C < 1 || C > HEAD_CMAX) return MMEMO_ERR_SHAPE;
  for (int i = 0; i < n; ++i) MM_REQUIRE(feats[i] && trans[i] && out[i] && B[i] >= 0);
  if (P <= 0) return MMEMO_OK;
  StTable tb = {};
  for (int i0 = 0; i0 < n; i0 += FOLD_MAX) {
    const int m = n - i0 < FOLD_MAX ? n - i0 : FOLD_MAX;
    int64_t bmax = 0;
    for (int j = 0; j < m; ++j) {
      tb.feats[j] = feats[i0 + j]; tb.trans[j] = trans[i0 + j]; tb.out[j] = out[i0 + j];
      tb.B[j] = (int)B[i0 + j];
      bmax = B[i0 + j] > bmax ? B[i0 + j] : bmax;
    }
    if (bmax == 0) continue;
    state_transfer_fwd_multi_kernel<<<dim3((unsigned)cdiv(bmax, 8), (unsigned)m), 256, 0,
                                      mm_stream(s)>>>(tb, (int)P, (int)C);
    MM_LAUNCH_OK();
  }
  return MMEMO_OK;
}
int mmemo_state_transfer_bwd_multi(int n, const float* const* dout, const float* const* feats,
                                   const float* const* trans, const float* const* out,
                                   float* const* dfeats, float* const* dtrans, const int64_t* B,
                                   int64_t P, int64_t C, mmemo_stream_t s) {
  MM_REQUIRE(n >= 0 && (n == 0 || (dout && feats && trans && out && dfeats && B)));
  if (C < 1 || C > HEAD_CMAX) return MMEMO_ERR_SHAPE;
  for (int i = 0; i < n; ++i)
    MM_REQUIRE(dout[i] && feats[i] && trans[i] && out[i] && dfeats[i] && B[i] >= 0);
  if (P <= 0) return MMEMO_OK;
  StTable tb = {};
  for (int i0 = 0; i0 < n; i0 += FOLD_MAX) {
    const int m = n - i0 < FOLD_MAX ? n - i0 : FOLD_MAX;
    int64_t bmax = 0;
    for (int j = 0; j < m; ++j) {
      const int i = i0 + j;
      tb.dout[j] = dout[i]; tb.feats[j] = feats[i]; tb.trans[j] = trans[i]; tb.out[j] = out[i];
      tb.dfeats[j] = dfeats[i]; tb.dtrans[j] = at(dtrans, i);
      tb.B[j] = (int)B[i];
      bmax = B[i] > bmax ? B[i] : bmax;
    }
    if (bmax == 0) continue;
    state_transfer_bwd_multi_kernel<<<dim3((unsigned)cdiv(bmax, 8), (unsigned)m), 256, 0,
                                      mm_stream(s)>>>(tb, (int)P, (int)C);
    MM_LAUNCH_OK();
  }
  return MMEMO_OK;
}

int mmemo_bilinear_head_fwd_multi(int n, const float* const* this_feat,
                                  const float* const* last_feat, const float* const* trans,
                                  const float* const* gamma, const float* const* beta,
                                  const float* const* w, const float* const* bias,
                                  float* const* out, float* const* z, const int64_t* B, int64_t C,
                                  float eps, mmemo_stream_t s) {
  MM_REQUIRE(n >= 0 && (n == 0 || (this_feat && last_feat && trans && gamma && beta && w && bias &&
                                   out && z && B)));
  if (C < 1 || C > HEAD_CMAX) return MMEMO_ERR_SHAPE;
  for (int i = 0; i < n; ++i)
    MM_REQUIRE(this_feat[i] && last_feat[i] && trans[i] && gamma[i] && beta[i] && w[i] &&
               bias[i] && out[i] && z[i] && B[i] >= 0);
  BhTable tb = {};
  for (int i0 = 0; i0 < n; i0 += FOLD_MAX) {
    const int m = n - i0 < FOLD_MAX ? n - i0 : FOLD_MAX;
    int64_t bmax = 0;
    for (int j = 0; j < m; ++j) {
      const int i = i0 + j;
      tb.th[j] = this_feat[i]; tb.la[j] = last_feat[i]; tb.trans[j] = trans[i];
      tb.gamma[j] = gamma[i]; tb.beta[j] = beta[i]; tb.w[j] = w[i]; tb.bias[j] = bias[i];
      tb.out[j] = out[i]; tb.z[j] = z[i];
      tb.B[j] = (int)B[i];
      bmax = B[i] > bmax ? B[i] : bmax;
    }
    if (bmax == 0) continue;
    bilinear_fwd_multi_kernel<<<dim3((unsigned)cdiv(bmax, 8), (unsigned)m), 256, 0,
                                mm_stream(s)>>>(tb, (int)C, eps);
    MM_LAUNCH_OK();
  }
  return MMEMO_OK;
}
int mmemo_bilinear_head_bwd_multi(int n, const float* const* dout, const float* const* this_feat,
                                  const float* const* last_feat, const float* const* trans,
                                  const float* const* gamma, const float* const* beta,
                                  const float* const* w, const float* const* z,
                                  float* const* dthis, float* const* dlast, float* const* dtrans,
                                  float* const* dgamma, float* const* dbeta, float* const* dw,
                                  float* const* dbias, const int64_t* B, int64_t C, float eps,
                                  mmemo_stream_t s) {
  MM_REQUIRE(n >= 0 && (n == 0 || (dout && this_feat && last_feat && trans && gamma && beta && w &&
                                   z && dthis && dlast && B)));
  if (C < 1 || C > HEAD_CMAX) return MMEMO_ERR_SHAPE;
  for (int i = 0; i < n; ++i)
    MM_REQUIRE(dout[i] && this_feat[i] && last_feat[i] && trans[i] && gamma[i] && beta[i] && w[i] &&
               z[i] && dthis[i] && dlast[i] && B[i] >= 0);
  const int copies = bilinear_bwd_copies(C);
  const size_t smem = bilinear_bwd_smem(C);
  BhTable tb = {};
  for (int i0 = 0; i0 < n; i0 += FOLD_MAX) {
    const int m = n - i0 < FOLD_MAX ? n - i0 : FOLD_MAX;
    int64_t bmax = 0;
    bool any_dw = false;
    for (int j = 0; j < m; ++j) {
      const int i = i0 + j;
      tb.dout[j] = dout[i]; tb.th[j] = this_feat[i]; tb.la[j] = last_feat[i];
      tb.trans[j] = trans[i]; tb.gamma[j] = gamma[i]; tb.beta[j] = beta[i]; tb.w[j] = w[i];
      tb.z[j] = const_cast<float*>(z[i]);
      tb.dth[j] = dthis[i]; tb.dla[j] = dlast[i]; tb.dtrans[j] = at(dtrans, i);
      tb.dgamma[j] = at(dgamma, i); tb.dbeta[j] = at(dbeta, i); tb.dw[j] = at(dw, i);
      tb.dbias[j] = at(dbias, i);
      tb.B[j] = (int)B[i];
      bmax = B[i] > bmax ? B[i] : bmax;
      any_dw = any_dw || tb.dw[j];
    }
    if (bmax == 0) continue;
    bilinear_bwd_multi_kernel<<<dim3((unsigned)bilinear_bwd_ctas(bmax), (unsigned)m), 256, smem,
                                mm_stream(s)>>>(tb, (int)C, eps, copies);
    MM_LAUNCH_OK();
    if (any_dw) {
      bilinear_dw_multi_kernel<<<dim3((unsigned)cdiv(2 * C * C, 128), (unsigned)cdiv(bmax, 16),
                                      (unsigned)m), 128, 0, mm_stream(s)>>>(tb, (int)C, eps);
      MM_LAUNCH_OK();
    }
  }
  return MMEMO_OK;
}

int mmemo_circle_loss_fwd_multi(int n, const float* const* logits, const float* const* labels,
                                const float* const* weights, const int64_t* R, int64_t C,
                                float* const* loss, mmemo_stream_t s) {
  MM_REQUIRE(n >= 0 && (n == 0 || (logits && labels && R && loss)) && C > 0);
  for (int i = 0; i < n; ++i) MM_REQUIRE(logits[i] && labels[i] && loss[i] && R[i] > 0);
  LossTable tb = {};
  for (int i0 = 0; i0 < n; i0 += FOLD_MAX) {
    const int m = n - i0 < FOLD_MAX ? n - i0 : FOLD_MAX;
    for (int j = 0; j < m; ++j) {
      const int i = i0 + j;
      tb.s[j] = logits[i]; tb.y[j] = labels[i]; tb.wt[j] = at(weights, i); tb.out[j] = loss[i];
      tb.R[j] = R[i];
    }
    circle_loss_fwd_multi_kernel<<<(unsigned)m, 256, 0, mm_stream(s)>>>(tb, (int)C);
    MM_LAUNCH_OK();
  }
  return MMEMO_OK;
}
int mmemo_circle_loss_bwd_multi(int n, const float* const* dloss, const float* const* logits,
                                const float* const* labels, const float* const* weights,
                                float* const* dlogits, const int64_t* R, int64_t C,
                                mmemo_stream_t s) {
  MM_REQUIRE(n >= 0 && (n == 0 || (dloss && logits && labels && dlogits && R)) && C > 0);
  for (int i = 0; i < n; ++i)
    MM_REQUIRE(dloss[i] && logits[i] && labels[i] && dlogits[i] && R[i] > 0);
  LossTable tb = {};
  for (int i0 = 0; i0 < n; i0 += FOLD_MAX) {
    const int m = n - i0 < FOLD_MAX ? n - i0 : FOLD_MAX;
    int64_t rmax = 0;
    for (int j = 0; j < m; ++j) {
      const int i = i0 + j;
      tb.dout[j] = dloss[i]; tb.s[j] = logits[i]; tb.y[j] = labels[i];
      tb.wt[j] = at(weights, i); tb.ds[j] = dlogits[i]; tb.R[j] = R[i];
      rmax = R[i] > rmax ? R[i] : rmax;
    }
    circle_loss_bwd_multi_kernel<<<dim3((unsigned)cdiv(rmax, 128), (unsigned)m), 128, 0,
                                   mm_stream(s)>>>(tb, (int)C);
    MM_LAUNCH_OK();
  }
  return MMEMO_OK;
}

int mmemo_rdrop_kl_fwd_multi(int n, const float* const* logits, const int64_t* B, int64_t C,
                             float* const* out, mmemo_stream_t s) {
  MM_REQUIRE(n >= 0 && (n == 0 || (logits && B && out)) && C > 0);
  for (int i = 0; i < n; ++i) MM_REQUIRE(logits[i] && out[i] && B[i] >= 2 && B[i] % 2 == 0);
  LossTable tb = {};
  for (int i0 = 0; i0 < n; i0 += FOLD_MAX) {
    const int m = n - i0 < FOLD_MAX ? n - i0 : FOLD_MAX;
    for (int j = 0; j < m; ++j) {
      tb.s[j] = logits[i0 + j]; tb.out[j] = out[i0 + j]; tb.R[j] = B[i0 + j] / 2;
    }
    rdrop_kl_fwd_multi_kernel<<<(unsigned)m, 256, 0, mm_stream(s)>>>(tb, (int)C);
    MM_LAUNCH_OK();
  }
  return MMEMO_OK;
}
int mmemo_rdrop_kl_bwd_multi(int n, const float* const* dout, const float* const* logits,
                             float* const* dlogits, const int64_t* B, int64_t C,
                             mmemo_stream_t s) {
  MM_REQUIRE(n >= 0 && (n == 0 || (dout && logits && dlogits && B)) && C > 0);
  for (int i = 0; i < n; ++i)
    MM_REQUIRE(dout[i] && logits[i] && dlogits[i] && B[i] >= 2 && B[i] % 2 == 0);
  LossTable tb = {};
  for (int i0 = 0; i0 < n; i0 += FOLD_MAX) {
    const int m = n - i0 < FOLD_MAX ? n - i0 : FOLD_MAX;
    int64_t emax = 0;
    for (int j = 0; j < m; ++j) {
      const int i = i0 + j;
      tb.dout[j] = dout[i]; tb.s[j] = logits[i]; tb.ds[j] = dlogits[i]; tb.R[j] = B[i] / 2;
      emax = tb.R[j] * C > emax ? tb.R[j] * C : emax;
    }
    rdrop_kl_bwd_multi_kernel<<<dim3((unsigned)cdiv(emax, 128), (unsigned)m), 128, 0,
                                mm_stream(s)>>>(tb, (int)C);
    MM_LAUNCH_OK();
  }
  return MMEMO_OK;
}
}  // extern "C"
