// Internal GEMM interface shared by the linear-layer entry points, the SIMT kernel and the
// tcgen05 kernel.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

struct GemmArgs {
  const void* A;  // element (m,k) at A[m*sAm + k*sAk]
  const void* B;  // element (n,k) at B[n*sBn + k*sBk]
  void* C;        // element (m,n) at C[m*ldc + n]
  int64_t sAm, sAk, sBn, sBk, ldc;
  int64_t M, N, K;
  const float* bias;       // [N] or null
  const float* pos;        // [pos_period, N] (row stride ldpos, 0 = N) or null
  int64_t pos_period;
  int64_t ldpos;
  const void* relu_src;    // [M, N] (ldrelu) or null: C *= (relu_src > 0)
  int64_t ldrelu;
  int relu_src_bf16;
  int relu;                // C = max(C, 0)
  int accumulate;          // C += result
  int c_zeroed;            // C is known to be all zero: the split-K reduce-add path skips its own fill
  // dropout between bias and position table (forward family 3 only; drop_p = 0: none): the mask
  // of a contiguous (M, N) tensor drawn from drop_seed + step[0] (dropout.cuh)
  float drop_p;
  uint64_t drop_seed;
  const uint64_t* drop_step;
};

// Split-K (float32 C, linear epilogue, small output grid) uses the stream's workspace and sums the
// partial tiles in a fixed order; without a workspace the GEMM does not split.
int gemm_simt(const GemmArgs& g, int a_bf16, int b_bf16, int c_bf16, cudaStream_t st);
// up to 48 independent float32 problems (no ReLU / position / accumulate epilogue) in one SIMT
// launch (or a few, when their split-K scratch does not fit in the workspace at once); the bias
// epilogue is kept.  Each problem gets gemm_simt's split factor: the same bits as gemm_simt.
constexpr int GEMM_SIMT_MAX_GROUP = 48;
int gemm_simt_grouped_f32(const GemmArgs* gs, int n, cudaStream_t st);

// tcgen05/TMA path (bf16 operands, fp32 accumulate in TMEM).  c_bf16=0 -> float32 C.
// Returns 1 if it accepts the shape/layout.
bool gemm_tc_supported(const GemmArgs& g, int c_bf16, bool any_size = false);
// family: 0 forward, 1 dX, 2 dW (only names the kernel instantiation), 3 forward with the dropout
// epilogue (GemmArgs::drop_*)
int gemm_tc(const GemmArgs& g, int c_bf16, int family, cudaStream_t st);
// up to 48 independent problems in one persistent launch (every problem must be gemm_tc_supported)
constexpr int GEMM_TC_MAX_GROUP = 48;
int gemm_tc_grouped(const GemmArgs* gs, const int* c_bf16s, int n, int family, cudaStream_t st);

