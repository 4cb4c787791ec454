// Linear / Conv1d(k=1) entry points: map y = x w^T, dx = dy w, dw = dy^T x onto the strided GEMM
// interface and pick the kernel by shape (tcgen05/TMA when the bf16 operands satisfy its tiling
// constraints, the SIMT kernel otherwise).  Both kernels are sm_100a CUDA in this library; this is
// shape routing, not a backend switch, and there is no CPU path.
#include "common.cuh"
#include "gemm.h"

int mmemo_rowsum_dispatch(int bf16_mode, const void* x, int64_t ldx, float* out, int64_t M,
                          int64_t N, cudaStream_t st);

namespace {

int run(const GemmArgs& g, int a_bf16, int b_bf16, int c_bf16, int family, cudaStream_t st) {
  if (a_bf16 && b_bf16 && gemm_tc_supported(g, c_bf16)) return gemm_tc(g, c_bf16, family, st);
  return gemm_simt(g, a_bf16, b_bf16, c_bf16, st);
}

int linear_fwd(int bf, const void* x, int x_is_f32, int64_t ldx, const void* w, int64_t ldw,
               const float* bias, const float* pos, int64_t pos_period, void* y, int64_t ldy,
               int64_t M, int64_t N, int64_t K, int relu, int accumulate, cudaStream_t st) {
  MM_REQUIRE(x && w && y);
  MM_REQUIRE(!pos || pos_period > 0);
  GemmArgs g = {};
  g.A = x; g.sAm = ldx; g.sAk = 1;
  g.B = w; g.sBn = ldw; g.sBk = 1;
  g.C = y; g.ldc = ldy;
  g.M = M; g.N = N; g.K = K;
  g.bias = bias; g.pos = pos; g.pos_period = pos ? pos_period : 1;
  g.relu = relu; g.accumulate = accumulate;
  return run(g, bf && !x_is_f32, bf, bf, 0, st);
}

int linear_bwd_x(int bf, const void* dy, int64_t lddy, const void* w, int64_t ldw, void* dx,
                 int64_t lddx, const void* relu_src, int64_t ldrelu, int64_t M, int64_t N,
                 int64_t K, int accumulate, cudaStream_t st) {
  MM_REQUIRE(dy && w && dx);
  GemmArgs g = {};
  g.A = dy; g.sAm = lddy; g.sAk = 1;      // reduction over n
  g.B = w; g.sBn = 1; g.sBk = ldw;        // B'(k_out, n) = w[n, k_out]
  g.C = dx; g.ldc = lddx;
  g.M = M; g.N = K; g.K = N;
  g.pos_period = 1;
  g.relu_src = relu_src; g.ldrelu = ldrelu; g.relu_src_bf16 = bf;
  g.accumulate = accumulate;
  return run(g, bf, bf, bf, 1, st);
}

int linear_bwd_w(int bf, const void* dy, int64_t lddy, const void* x, int x_is_f32, int64_t ldx,
                 float* dw, int64_t lddw, float* dbias, int64_t M, int64_t N, int64_t K,
                 int accumulate, cudaStream_t st) {
  MM_REQUIRE(dy && x && dw);
  GemmArgs g = {};
  g.A = dy; g.sAm = 1; g.sAk = lddy;      // A'(n, m) = dy[m, n]
  g.B = x; g.sBn = 1; g.sBk = ldx;        // B'(k, m) = x[m, k]
  g.C = dw; g.ldc = lddw;
  g.M = N; g.N = K; g.K = M;
  g.pos_period = 1;
  g.accumulate = accumulate;
  int rc = run(g, bf, bf && !x_is_f32, 0, 2, st);
  if (rc) return rc;
  if (dbias) rc = mmemo_rowsum_dispatch(bf, dy, lddy, dbias, M, N, st);
  return rc;
}

}  // namespace

extern "C" {
int mmemo_gemm_uses_tensor_cores(int64_t M, int64_t N, int64_t K, int64_t lda, int64_t ldb,
                                 int64_t ldc, int mode) {
  GemmArgs g = {};
  static const char dummy[16] = {0};
  g.A = dummy; g.B = dummy; g.C = const_cast<char*>(dummy);
  g.pos_period = 1;
  if (mode == 0) {        // fwd  : y[M,N] = x[M,K] w[N,K]^T
    g.sAm = lda; g.sAk = 1; g.sBn = ldb; g.sBk = 1; g.ldc = ldc; g.M = M; g.N = N; g.K = K;
    return gemm_tc_supported(g, 1) ? 1 : 0;
  } else if (mode == 1) { // bwd_x: dx[M,K] = dy[M,N] w[N,K]
    g.sAm = lda; g.sAk = 1; g.sBn = 1; g.sBk = ldb; g.ldc = ldc; g.M = M; g.N = K; g.K = N;
    return gemm_tc_supported(g, 1) ? 1 : 0;
  } else {                // bwd_w: dw[N,K] = dy[M,N]^T x[M,K]
    g.sAm = 1; g.sAk = lda; g.sBn = 1; g.sBk = ldb; g.ldc = ldc; g.M = N; g.N = K; g.K = M;
    return gemm_tc_supported(g, 0) ? 1 : 0;
  }
}

// ---- grouped variants (bf16): n independent problems, ONE tensor-core launch when all qualify ----
int mmemo_linear_fwd_grouped_bf16(int n, const void* const* x, const int64_t* ldx,
                                  const void* const* w, const int64_t* ldw,
                                  const float* const* bias, void* const* y, const int64_t* ldy,
                                  const int64_t* M, const int64_t* N, const int64_t* K,
                                  const int* relu, const int* accumulate,
                                  const float* const* pos, const int64_t* pos_period,
                                  const int64_t* ldpos, mmemo_stream_t s) {
  if (n < 1 || n > GEMM_TC_MAX_GROUP) return MMEMO_ERR_ARG;
  GemmArgs g[GEMM_TC_MAX_GROUP] = {};
  int cb[GEMM_TC_MAX_GROUP];
  bool tc_ok = true;
  for (int i = 0; i < n; ++i) {
    MM_REQUIRE(x[i] && w[i] && y[i]);
    g[i].A = x[i]; g[i].sAm = ldx[i]; g[i].sAk = 1;
    g[i].B = w[i]; g[i].sBn = ldw[i]; g[i].sBk = 1;
    g[i].C = y[i]; g[i].ldc = ldy[i];
    g[i].M = M[i]; g[i].N = N[i]; g[i].K = K[i];
    g[i].bias = bias ? bias[i] : nullptr; g[i].pos_period = 1;
    g[i].relu = relu ? relu[i] : 0;
    g[i].accumulate = accumulate ? accumulate[i] : 0;
    if (pos && pos[i]) {
      MM_REQUIRE(pos_period && pos_period[i] > 0);
      g[i].pos = pos[i]; g[i].pos_period = pos_period[i];
      if (ldpos && ldpos[i]) {
        MM_REQUIRE(ldpos[i] >= N[i]);
        g[i].ldpos = ldpos[i];
      }
    }
    cb[i] = 1;
    tc_ok = tc_ok && gemm_tc_supported(g[i], 1, n > 1);
  }
  if (tc_ok) return gemm_tc_grouped(g, cb, n, 0, mm_stream(s));
  for (int i = 0; i < n; ++i) {
    const int rc = run(g[i], 1, 1, 1, 0, mm_stream(s));
    if (rc) return rc;
  }
  return MMEMO_OK;
}
int mmemo_linear_fwd_grouped_dropout_bf16(int n, const void* const* x, const int64_t* ldx,
                                          const void* const* w, const int64_t* ldw,
                                          const float* const* bias, void* const* y,
                                          const int64_t* ldy, const int64_t* M, const int64_t* N,
                                          const int64_t* K, const float* const* pos,
                                          const int64_t* pos_period, const int64_t* ldpos,
                                          const uint64_t* seeds, float p, const uint64_t* step,
                                          mmemo_stream_t s) {
  if (n < 1 || n > GEMM_TC_MAX_GROUP) return MMEMO_ERR_ARG;
  MM_REQUIRE(x && ldx && w && ldw && y && ldy && M && N && K && seeds && step);
  MM_REQUIRE(p >= 0.f && p < 1.f);
  GemmArgs g[GEMM_TC_MAX_GROUP] = {};
  int cb[GEMM_TC_MAX_GROUP];
  for (int i = 0; i < n; ++i) {
    MM_REQUIRE(x[i] && w[i] && y[i]);
    g[i].A = x[i]; g[i].sAm = ldx[i]; g[i].sAk = 1;
    g[i].B = w[i]; g[i].sBn = ldw[i]; g[i].sBk = 1;
    g[i].C = y[i]; g[i].ldc = ldy[i];
    g[i].M = M[i]; g[i].N = N[i]; g[i].K = K[i];
    g[i].bias = bias ? bias[i] : nullptr; g[i].pos_period = 1;
    if (pos && pos[i]) {
      MM_REQUIRE(pos_period && pos_period[i] > 0);
      g[i].pos = pos[i]; g[i].pos_period = pos_period[i];
      if (ldpos && ldpos[i]) {
        MM_REQUIRE(ldpos[i] >= N[i]);
        g[i].ldpos = ldpos[i];
      }
    }
    g[i].drop_p = p; g[i].drop_seed = seeds[i]; g[i].drop_step = step;
    cb[i] = 1;
    // the mask exists only in the tensor-core epilogue: a problem it cannot take is an error
    if (!gemm_tc_supported(g[i], 1, true)) return MMEMO_ERR_SHAPE;
  }
  return gemm_tc_grouped(g, cb, n, p > 0.f ? 3 : 0, mm_stream(s));
}
int mmemo_linear_bwd_x_grouped_bf16(int n, const void* const* dy, const int64_t* lddy,
                                    const void* const* w, const int64_t* ldw, void* const* dx,
                                    const int64_t* lddx, const void* const* relu_src,
                                    const int64_t* ldrelu, const int64_t* M, const int64_t* N,
                                    const int64_t* K, const int* accumulate, mmemo_stream_t s) {
  if (n < 1 || n > GEMM_TC_MAX_GROUP) return MMEMO_ERR_ARG;
  GemmArgs g[GEMM_TC_MAX_GROUP] = {};
  int cb[GEMM_TC_MAX_GROUP];
  bool tc_ok = true;
  for (int i = 0; i < n; ++i) {
    MM_REQUIRE(dy[i] && w[i] && dx[i]);
    g[i].A = dy[i]; g[i].sAm = lddy[i]; g[i].sAk = 1;
    g[i].B = w[i]; g[i].sBn = 1; g[i].sBk = ldw[i];
    g[i].C = dx[i]; g[i].ldc = lddx[i];
    g[i].M = M[i]; g[i].N = K[i]; g[i].K = N[i];
    g[i].pos_period = 1;
    g[i].accumulate = accumulate ? accumulate[i] : 0;
    if (relu_src && relu_src[i]) {
      g[i].relu_src = relu_src[i]; g[i].ldrelu = ldrelu[i]; g[i].relu_src_bf16 = 1;
    }
    cb[i] = 1;
    tc_ok = tc_ok && gemm_tc_supported(g[i], 1, n > 1);
  }
  if (tc_ok) return gemm_tc_grouped(g, cb, n, 1, mm_stream(s));
  for (int i = 0; i < n; ++i) {
    const int rc = run(g[i], 1, 1, 1, 1, mm_stream(s));
    if (rc) return rc;
  }
  return MMEMO_OK;
}
int mmemo_linear_bwd_w_grouped_bf16(int n, const void* const* dy, const int64_t* lddy,
                                    const void* const* x, const int64_t* ldx, float* const* dw,
                                    const int64_t* lddw, const int64_t* M, const int64_t* N,
                                    const int64_t* K, int accumulate, mmemo_stream_t s) {
  if (n < 1 || n > GEMM_TC_MAX_GROUP) return MMEMO_ERR_ARG;
  GemmArgs g[GEMM_TC_MAX_GROUP] = {};
  int cb[GEMM_TC_MAX_GROUP];
  bool tc_ok = true;
  for (int i = 0; i < n; ++i) {
    MM_REQUIRE(dy[i] && x[i] && dw[i]);
    g[i].A = dy[i]; g[i].sAm = 1; g[i].sAk = lddy[i];
    g[i].B = x[i]; g[i].sBn = 1; g[i].sBk = ldx[i];
    g[i].C = dw[i]; g[i].ldc = lddw[i];
    g[i].M = N[i]; g[i].N = K[i]; g[i].K = M[i];
    g[i].pos_period = 1;
    g[i].accumulate = accumulate == 1;
    g[i].c_zeroed = accumulate == 2;      // either overwrite or add is correct
    cb[i] = 0;
    tc_ok = tc_ok && gemm_tc_supported(g[i], 0, n > 1);
  }
  if (tc_ok) return gemm_tc_grouped(g, cb, n, 2, mm_stream(s));
  for (int i = 0; i < n; ++i) {
    const int rc = run(g[i], 1, 1, 0, 2, mm_stream(s));
    if (rc) return rc;
  }
  return MMEMO_OK;
}

// ---- grouped float32 variants: n independent problems, one SIMT launch per 48 (the head linears,
// which run in float32 in both precision modes) ----
int mmemo_linear_fwd_grouped_f32(int n, const float* const* x, const int64_t* ldx,
                                 const float* const* w, const int64_t* ldw,
                                 const float* const* bias, float* const* y, const int64_t* ldy,
                                 const int64_t* M, const int64_t* N, const int64_t* K,
                                 mmemo_stream_t s) {
  MM_REQUIRE(n >= 0 && (n == 0 || (x && ldx && w && ldw && y && ldy && M && N && K)));
  GemmArgs g[GEMM_SIMT_MAX_GROUP] = {};
  for (int i0 = 0; i0 < n; i0 += GEMM_SIMT_MAX_GROUP) {
    const int m = n - i0 < GEMM_SIMT_MAX_GROUP ? n - i0 : GEMM_SIMT_MAX_GROUP;
    for (int j = 0; j < m; ++j) {
      const int i = i0 + j;
      MM_REQUIRE(x[i] && w[i] && y[i]);
      g[j] = GemmArgs{};
      g[j].A = x[i]; g[j].sAm = ldx[i]; g[j].sAk = 1;
      g[j].B = w[i]; g[j].sBn = ldw[i]; g[j].sBk = 1;
      g[j].C = y[i]; g[j].ldc = ldy[i];
      g[j].M = M[i]; g[j].N = N[i]; g[j].K = K[i];
      g[j].bias = bias ? bias[i] : nullptr; g[j].pos_period = 1;
    }
    const int rc = gemm_simt_grouped_f32(g, m, mm_stream(s));
    if (rc) return rc;
  }
  return MMEMO_OK;
}
int mmemo_linear_bwd_x_grouped_f32(int n, const float* const* dy, const int64_t* lddy,
                                   const float* const* w, const int64_t* ldw, float* const* dx,
                                   const int64_t* lddx, const int64_t* M, const int64_t* N,
                                   const int64_t* K, mmemo_stream_t s) {
  MM_REQUIRE(n >= 0 && (n == 0 || (dy && lddy && w && ldw && dx && lddx && M && N && K)));
  GemmArgs g[GEMM_SIMT_MAX_GROUP] = {};
  for (int i0 = 0; i0 < n; i0 += GEMM_SIMT_MAX_GROUP) {
    const int m = n - i0 < GEMM_SIMT_MAX_GROUP ? n - i0 : GEMM_SIMT_MAX_GROUP;
    for (int j = 0; j < m; ++j) {
      const int i = i0 + j;
      MM_REQUIRE(dy[i] && w[i] && dx[i]);
      g[j] = GemmArgs{};
      g[j].A = dy[i]; g[j].sAm = lddy[i]; g[j].sAk = 1;
      g[j].B = w[i]; g[j].sBn = 1; g[j].sBk = ldw[i];
      g[j].C = dx[i]; g[j].ldc = lddx[i];
      g[j].M = M[i]; g[j].N = K[i]; g[j].K = N[i];
      g[j].pos_period = 1;
    }
    const int rc = gemm_simt_grouped_f32(g, m, mm_stream(s));
    if (rc) return rc;
  }
  return MMEMO_OK;
}

namespace {
__device__ const float g_one = 1.0f;     // the ones vector (stride 0) of the bias-gradient problems
}

int mmemo_linear_bwd_w_grouped_f32(int n, const float* const* dy, const int64_t* lddy,
                                   const float* const* x, const int64_t* ldx, float* const* dw,
                                   const int64_t* lddw, float* const* dbias, const int64_t* M,
                                   const int64_t* N, const int64_t* K, mmemo_stream_t s) {
  MM_REQUIRE(n >= 0 && (n == 0 || (dy && lddy && x && ldx && dw && lddw && M && N && K)));
  const void* one = nullptr;
  // problem list: every dW, then every dbias as the GEMM dy^T 1 (N x 1, K' = M)
  GemmArgs all[2 * GEMM_SIMT_MAX_GROUP];
  int n_all = 0;
  for (int i0 = 0; i0 < n; i0 += GEMM_SIMT_MAX_GROUP) {
    const int m = n - i0 < GEMM_SIMT_MAX_GROUP ? n - i0 : GEMM_SIMT_MAX_GROUP;
    n_all = 0;
    for (int j = 0; j < m; ++j) {
      const int i = i0 + j;
      MM_REQUIRE(dy[i] && x[i] && dw[i]);
      GemmArgs& g = all[n_all++];
      g = GemmArgs{};
      g.A = dy[i]; g.sAm = 1; g.sAk = lddy[i];
      g.B = x[i]; g.sBn = 1; g.sBk = ldx[i];
      g.C = dw[i]; g.ldc = lddw[i];
      g.M = N[i]; g.N = K[i]; g.K = M[i];
      g.pos_period = 1;
    }
    for (int j = 0; dbias && j < m; ++j) {
      const int i = i0 + j;
      if (!dbias[i]) continue;
      if (!one) MM_CUDA_OK(cudaGetSymbolAddress(const_cast<void**>(&one), g_one));
      GemmArgs& g = all[n_all++];
      g = GemmArgs{};
      g.A = dy[i]; g.sAm = 1; g.sAk = lddy[i];
      g.B = one; g.sBn = 0; g.sBk = 0;
      g.C = dbias[i]; g.ldc = 1;
      g.M = N[i]; g.N = 1; g.K = M[i];
      g.pos_period = 1;
    }
    for (int a = 0; a < n_all; a += GEMM_SIMT_MAX_GROUP) {
      const int rc = gemm_simt_grouped_f32(all + a, n_all - a < GEMM_SIMT_MAX_GROUP ?
                                           n_all - a : GEMM_SIMT_MAX_GROUP, mm_stream(s));
      if (rc) return rc;
    }
  }
  return MMEMO_OK;
}

#define MM_LINEAR(SUF, BF)                                                                        \
  int mmemo_linear_fwd_##SUF(const void* x, int x_is_f32, int64_t ldx, const void* w, int64_t ldw, \
                             const float* bias, const float* pos, int64_t pos_period, void* y,    \
                             int64_t ldy, int64_t M, int64_t N, int64_t K, int relu,              \
                             int accumulate, mmemo_stream_t s) {                                  \
    return linear_fwd(BF, x, (BF) ? x_is_f32 : 1, ldx, w, ldw, bias, pos, pos_period, y, ldy, M,  \
                      N, K, relu, accumulate, mm_stream(s));                                      \
  }                                                                                               \
  int mmemo_linear_bwd_x_##SUF(const void* dy, int64_t lddy, const void* w, int64_t ldw, void* dx, \
                               int64_t lddx, const void* relu_src, int64_t ldrelu, int64_t M,     \
                               int64_t N, int64_t K, int accumulate, mmemo_stream_t s) {          \
    return linear_bwd_x(BF, dy, lddy, w, ldw, dx, lddx, relu_src, ldrelu, M, N, K, accumulate,    \
                        mm_stream(s));                                                            \
  }                                                                                               \
  int mmemo_linear_bwd_w_##SUF(const void* dy, int64_t lddy, const void* x, int x_is_f32,         \
                               int64_t ldx, float* dw, int64_t lddw, float* dbias, int64_t M,     \
                               int64_t N, int64_t K, int accumulate, mmemo_stream_t s) {          \
    return linear_bwd_w(BF, dy, lddy, x, (BF) ? x_is_f32 : 1, ldx, dw, lddw, dbias, M, N, K,      \
                        accumulate, mm_stream(s));                                                \
  }
MM_LINEAR(f32, 0)
MM_LINEAR(bf16, 1)
#undef MM_LINEAR
}
