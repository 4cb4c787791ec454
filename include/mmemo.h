/*
 * mmemo.h — C ABI of libmmemo.so, the B200 (sm_100a) hot path of
 * youngzhou97qz/Multimodal-emotion-processing.
 *
 * The reference is pure Python/PyTorch and has no FFI of its own; its drop-in boundary is the set
 * of nn.Module forwards listed in SURVEY.md §8(b).  Each entry point below replaces the eager
 * ATen op sequence of one reference code span (cited per function, paths relative to the reference
 * root).  The Python host (multimodal-emotion-processing_b200/ops.py) binds these with ctypes and
 * registers them as torch custom ops; INTEGRATION.md shows the stub.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the comment says "host"; buffers are owned by the
 *     caller; nothing here allocates or synchronises; all work is enqueued on `stream` (a
 *     cudaStream_t passed as void*).  The library keeps NO process-wide mutable state: the three
 *     launch settings of the "library / device info" block (split-K workspace, SM budget,
 *     programmatic dependent launch) are attributes of a STREAM, read by the entry points from the
 *     stream they are given, so host threads driving different streams are independent
 *     (re-entrant); the last-error string is thread-local.
 *   - return 0 on success, <0 on error (MMEMO_ERR_*).  No CPU fallback exists.
 *   - suffix _f32 / _bf16 = dtype of ACTIVATIONS and GEMM weights (T).  Small parameter vectors
 *     (bias, LayerNorm gamma/beta, gates a/b/c, position tables) and ALL parameter gradients are
 *     float32 in both modes; accumulation is always float32.
 *   - "ld*" = leading dimension (row stride, in elements) of a row-major matrix.
 *   - outputs marked "+=" are accumulated into (caller zero-initialises).
 */
#ifndef MMEMO_H_
#define MMEMO_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MMEMO_OK 0
#define MMEMO_ERR_ARG (-1)   /* null / inconsistent argument                         */
#define MMEMO_ERR_SHAPE (-2) /* shape outside what the kernels support (see DESIGN)  */
#define MMEMO_ERR_CUDA (-3)  /* a CUDA runtime / driver call failed                  */

typedef void* mmemo_stream_t; /* cudaStream_t */

/* library / device info */
int mmemo_version(void);
const char* mmemo_last_error(void); /* host string describing the last MMEMO_ERR_CUDA */
/* Per-stream launch settings.  Every entry point below looks them up by the `stream` argument of
 * the call (defaults for a stream that was never configured: no workspace, all SMs, PDL on).
 *  - workspace: scratch for split-K partial tiles of the tcgen05 GEMM when the output is bf16 or
 *    carries a bias (fp32 weight gradients are summed by TMA reduce-add and need none), and of the
 *    SIMT GEMM (float32 outputs: the float32 parity mode and the float32 heads), which sums its
 *    partial tiles in a fixed order, so its results do not depend on CTA scheduling.  The
 *    library never allocates: the host attaches one device buffer to each stream it launches on;
 *    launches of one stream are ordered, so they can share it, and two streams never share one.
 *    A GEMM that would need more than `bytes` simply does not split.
 *  - sm_budget: number of SMs the persistent (one CTA per SM) kernels launched on the stream may
 *    occupy; 0 = all.  Data-parallel training lowers it for the GEMMs that follow a bucket
 *    all-reduce, so that the collective's CTAs have SMs of their own.
 *  - pdl: programmatic dependent launch for the hot kernels (tcgen05 GEMM / attention, vector
 *    LayerNorm, column sums, weight casts): the next kernel's prologue overlaps the previous
 *    kernel's drain.  On by default; 0 launches every kernel of the stream fully serialised.
 *  - reset: forget the stream (call before cudaStreamDestroy; handles can be reused by CUDA). */
int mmemo_stream_set_workspace(mmemo_stream_t stream, void* ptr, int64_t bytes);
int mmemo_stream_set_sm_budget(mmemo_stream_t stream, int n_sms);
int mmemo_stream_set_pdl(mmemo_stream_t stream, int enabled);
int mmemo_stream_reset(mmemo_stream_t stream);
/* 1 if (M,N,K,mode) is served by the tcgen05/TMA tensor-core GEMM, 0 if by the SIMT GEMM */
int mmemo_gemm_uses_tensor_cores(int64_t M, int64_t N, int64_t K, int64_t lda, int64_t ldb,
                                 int64_t ldc, int mode);

/* ---------------------------------------------------------------------------------------------
 * Linear / Conv1d(k=1) layers.  Replaces nn.Linear / nn.Conv1d(kernel_size=1) calls:
 *   others/realformer.py:140-143,188,204,163-168,263,277   cmu-mosei/run.py:213-214,257,261,319
 *   Ren-MME/run.py:165-166,209,213,271   rencecps/run.py:139-140   robot_demo.py:302-311,353,369,441
 * fwd : y[M,N] (+)= act( x[M,K] . w[N,K]^T + bias[N] + pos[m % pos_period, N] )
 *       x may be float32 even in the _bf16 build (x_is_f32=1: raw input features).
 *       pos: learned position table (others/realformer.py:145-152,225-227) fused as a periodic bias.
 * bwd_x: dx[M,K] (+)= ( dy[M,N] . w[N,K] ) * (relu_src[M,K] > 0)
 * bwd_w: dw[N,K] (+)= dy[M,N]^T . x[M,K]  (float32 out);  dbias[N] += colsum(dy) if non-null.
 * ------------------------------------------------------------------------------------------- */
int mmemo_linear_fwd_f32(const void* x, int x_is_f32, int64_t ldx, const void* w, int64_t ldw,
                         const float* bias, const float* pos, int64_t pos_period, void* y,
                         int64_t ldy, int64_t M, int64_t N, int64_t K, int relu, int accumulate,
                         mmemo_stream_t stream);
int mmemo_linear_fwd_bf16(const void* x, int x_is_f32, int64_t ldx, const void* w, int64_t ldw,
                          const float* bias, const float* pos, int64_t pos_period, void* y,
                          int64_t ldy, int64_t M, int64_t N, int64_t K, int relu, int accumulate,
                          mmemo_stream_t stream);
int mmemo_linear_bwd_x_f32(const void* dy, int64_t lddy, const void* w, int64_t ldw, void* dx,
                           int64_t lddx, const void* relu_src, int64_t ldrelu, int64_t M, int64_t N,
                           int64_t K, int accumulate, mmemo_stream_t stream);
int mmemo_linear_bwd_x_bf16(const void* dy, int64_t lddy, const void* w, int64_t ldw, void* dx,
                            int64_t lddx, const void* relu_src, int64_t ldrelu, int64_t M,
                            int64_t N, int64_t K, int accumulate, mmemo_stream_t stream);
int mmemo_linear_bwd_w_f32(const void* dy, int64_t lddy, const void* x, int x_is_f32, int64_t ldx,
                           float* dw, int64_t lddw, float* dbias, int64_t M, int64_t N, int64_t K,
                           int accumulate, mmemo_stream_t stream);
int mmemo_linear_bwd_w_bf16(const void* dy, int64_t lddy, const void* x, int x_is_f32, int64_t ldx,
                            float* dw, int64_t lddw, float* dbias, int64_t M, int64_t N, int64_t K,
                            int accumulate, mmemo_stream_t stream);

/* Grouped variants (bf16): n <= 48 independent problems of the kinds above in ONE persistent
 * tensor-core launch (the Q and K|V projections of a block; its five weight gradients; the same
 * for all nine chains of a fusion-trunk layer at once), so that GEMMs too small to fill 148 SMs
 * share a wave.  All arrays are HOST arrays of length n.  Falls
 * back to n single launches when a problem does not meet the tensor-core kernel's constraints.
 * ldpos (nullable, entries 0 = N): row stride of pos[i], so that a problem can add a COLUMN SLICE
 * of a wider position table (the reference concatenates three visual projections and then adds
 * one table, robot_demo.py:304-311); y[i] / ldy[i] can address the matching slice of the output. */
int mmemo_linear_fwd_grouped_bf16(int n, const void* const* x, const int64_t* ldx,
                                  const void* const* w, const int64_t* ldw,
                                  const float* const* bias, void* const* y, const int64_t* ldy,
                                  const int64_t* M, const int64_t* N, const int64_t* K,
                                  const int* relu, const int* accumulate,
                                  const float* const* pos, const int64_t* pos_period,
                                  const int64_t* ldpos, mmemo_stream_t stream);
/* The grouped forward with a training dropout between the bias and the position table (the
 * modality projections, robot_demo.py:302-311 then :392-394): y[i] = drop_i(x[i] w[i]^T + bias[i])
 * + pos[i], one tensor-core launch.  The mask of problem i is the one mmemo_dropout_multi_* draws
 * for a contiguous (M[i], N[i]) tensor with seeds[i] and the device step counter `step` (read when
 * the kernel runs), whatever ldy[i] is; kept values are scaled by 1 / (1 - p).  p = 0 is the
 * plain grouped forward.  No relu / accumulate; every problem must fit the tensor-core kernel
 * (MMEMO_ERR_SHAPE otherwise: there is no other implementation of the mask). */
int mmemo_linear_fwd_grouped_dropout_bf16(int n, const void* const* x, const int64_t* ldx,
                                          const void* const* w, const int64_t* ldw,
                                          const float* const* bias, void* const* y,
                                          const int64_t* ldy, const int64_t* M, const int64_t* N,
                                          const int64_t* K, const float* const* pos,
                                          const int64_t* pos_period, const int64_t* ldpos,
                                          const uint64_t* seeds, float p, const uint64_t* step,
                                          mmemo_stream_t stream);
int mmemo_linear_bwd_x_grouped_bf16(int n, const void* const* dy, const int64_t* lddy,
                                    const void* const* w, const int64_t* ldw, void* const* dx,
                                    const int64_t* lddx, const void* const* relu_src,
                                    const int64_t* ldrelu, const int64_t* M, const int64_t* N,
                                    const int64_t* K, const int* accumulate, mmemo_stream_t stream);
/* accumulate: 0 = dw is overwritten, 1 = dw += ..., 2 = the caller guarantees that every dw is
 * all zero (both are correct; the split-K reduce-add path then skips its own zero fill). */
int mmemo_linear_bwd_w_grouped_bf16(int n, const void* const* dy, const int64_t* lddy,
                                    const void* const* x, const int64_t* ldx, float* const* dw,
                                    const int64_t* lddw, const int64_t* M, const int64_t* N,
                                    const int64_t* K, int accumulate, mmemo_stream_t stream);
/* Grouped float32 variants: n >= 0 problems (the float32 head linears of k folds), one SIMT launch
 * per 48 problems (more only when their split-K scratch exceeds the stream's workspace).  Each
 * problem splits K exactly as mmemo_linear_*_f32 would split it alone, so y, dx and dw are the
 * same bits as mmemo_linear_*_f32 on that problem.  bias / dbias (nullable arrays and
 * entries): bias[i] (N) added; dbias[i] (N) = column sums of dy[i] (overwritten; the dbias problems
 * are GEMMs of their own, so with n > 24 dbias entries bwd_w takes one launch more). */
int mmemo_linear_fwd_grouped_f32(int n, const float* const* x, const int64_t* ldx,
                                 const float* const* w, const int64_t* ldw,
                                 const float* const* bias, float* const* y, const int64_t* ldy,
                                 const int64_t* M, const int64_t* N, const int64_t* K,
                                 mmemo_stream_t stream);
int mmemo_linear_bwd_x_grouped_f32(int n, const float* const* dy, const int64_t* lddy,
                                   const float* const* w, const int64_t* ldw, float* const* dx,
                                   const int64_t* lddx, const int64_t* M, const int64_t* N,
                                   const int64_t* K, mmemo_stream_t stream);
int mmemo_linear_bwd_w_grouped_f32(int n, const float* const* dy, const int64_t* lddy,
                                   const float* const* x, const int64_t* ldx, float* const* dw,
                                   const int64_t* lddw, float* const* dbias, const int64_t* M,
                                   const int64_t* N, const int64_t* K, mmemo_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Fused residual-attention core (kernel a / a').  Replaces
 *   others/realformer.py:189-203  cmu-mosei/run.py:242-256  Ren-MME/run.py:194-208
 *   robot_demo.py:354-368
 * q (B,Lq,H*hd) row stride ldq; k, v (B,Lk,H*hd); head h lives in columns [h*hd,(h+1)*hd).
 * mask: float 0/1, element (b,i,j) at mask[b*mask_bs + i*mask_rs + j]  ((B,Lk): mask_rs = 0).
 * S = q_h k_h^T / sqrt(hd) + c*S_prev - 1e8*(1-mask)   (fp32 op order of the reference)
 * s_out (B,H,Lq,Lk) receives S (post-mask, pre-softmax; what the reference returns); may be null
 * when no later layer / backward needs it.  o (B,Lq,H*hd) = merge_heads(softmax(S) v_h).
 * lse (B,H,Lq,2) float32 = (row max, row sum of exp(S - max)) saved for backward; kept as a pair
 * because a fully masked row has max = -1e8, where max + log(sum) is absorbed by fp32 rounding.
 * bwd: dS = P*(dP - rowsum(dO*O)) + dS_next; dq = dS k / sqrt(hd); dk = dS^T q / sqrt(hd);
 *      dv = P^T dO; dc += sum(dS*S_prev); ds_prev = c*dS.   s == null -> scores are recomputed
 *      from q, k, mask (and s_prev, c).  dq_ws: float32 (B,Lq,H*hd) scratch, needed for the _bf16
 *      build when Lk > 128 (may be null otherwise).
 * ------------------------------------------------------------------------------------------- */
int mmemo_resattn_fwd_f32(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v,
                          int64_t ldv, const float* mask, int64_t mask_bs, int64_t mask_rs,
                          const void* s_prev, const float* c, void* s_out, void* o, int64_t ldo,
                          float* lse, int64_t B, int64_t H, int64_t Lq, int64_t Lk, int64_t hd,
                          mmemo_stream_t stream);
int mmemo_resattn_fwd_bf16(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v,
                           int64_t ldv, const float* mask, int64_t mask_bs, int64_t mask_rs,
                           const void* s_prev, const float* c, void* s_out, void* o, int64_t ldo,
                           float* lse, int64_t B, int64_t H, int64_t Lq, int64_t Lk, int64_t hd,
                           mmemo_stream_t stream);
int mmemo_resattn_bwd_f32(const void* d_o, int64_t lddo, const void* q, int64_t ldq, const void* k,
                          int64_t ldk, const void* v, int64_t ldv, const float* mask,
                          int64_t mask_bs, int64_t mask_rs, const void* s, const void* s_prev,
                          const float* c, const void* ds_next, const void* o, int64_t ldo,
                          const float* lse, void* dq, int64_t lddq, void* dk, int64_t lddk,
                          void* dv, int64_t lddv, void* ds_prev, float* dc, float* dq_ws, int64_t B,
                          int64_t H, int64_t Lq, int64_t Lk, int64_t hd, mmemo_stream_t stream);
int mmemo_resattn_bwd_bf16(const void* d_o, int64_t lddo, const void* q, int64_t ldq,
                           const void* k, int64_t ldk, const void* v, int64_t ldv,
                           const float* mask, int64_t mask_bs, int64_t mask_rs, const void* s,
                           const void* s_prev, const float* c, const void* ds_next, const void* o,
                           int64_t ldo, const float* lse, void* dq, int64_t lddq, void* dk,
                           int64_t lddk, void* dv, int64_t lddv, void* ds_prev, float* dc,
                           float* dq_ws, int64_t B, int64_t H, int64_t Lq, int64_t Lk, int64_t hd,
                           mmemo_stream_t stream);
/* 1 if the tcgen05/TMA attention kernels serve this shape in the _bf16 build */
int mmemo_resattn_uses_tensor_cores(int64_t Lq, int64_t Lk, int64_t hd, int64_t ld);

/* Grouped residual attention (bf16): n >= 1 independent problems, one launch per 40 (heaviest
 * problems first within each launch; every problem is checked before the first launch) - the nine chains
 * of a fusion-trunk layer (others/realformer.py:232-257, cmu-mosei/run.py:278-313,
 * Ren-MME/run.py:230-265, robot_demo.py:399-434), both towers of Concat_Trans / Base_model
 * (cmu-mosei/run.py:330-331, Ren-MME/run.py:283-284), the members of an ensemble
 * (robot_demo.py:610-614).  Same math and argument meaning as mmemo_resattn_{fwd,bwd}_bf16, one
 * struct per problem (HOST array; pointers inside are device pointers).  (B, Lk) masks only.
 * `lds` is the row stride (elements) of all score-shaped tensors of the problem (s_prev, s_out,
 * s, ds_next, ds_prev: (B, H, Lq, lds) with lds >= Lk; a multiple of 8 enables 16-byte accesses).
 * All problems of a call share hd in {16, 32, 64}.  Runs on the warp-level tensor-core path
 * (mma.sync m16n8k16).  Returns MMEMO_ERR_SHAPE when a problem is outside that kernel's limits
 * (the caller then issues the problems one by one through the ungrouped entry points). */
typedef struct mmemo_attn_problem {
  const void *q, *k, *v;                 /* (B,Lq,H*hd), (B,Lk,H*hd) x2 */
  int64_t ldq, ldk, ldv;
  const float* mask;                     /* (B, Lk) float 0/1 or NULL */
  int64_t mask_bs;
  const void* s_prev;                    /* previous layer's scores or NULL */
  const float* c;
  void* s_out;                           /* fwd: scores out (nullable) */
  int64_t lds;
  void* o;                               /* fwd: out; bwd: the saved forward output */
  int64_t ldo;
  float* lse;                            /* (B,H,Lq,2): fwd out / bwd in */
  int64_t B, H, Lq, Lk, hd;
  /* backward only */
  const void* d_o;
  int64_t lddo;
  const void* s;                         /* stored scores, or NULL -> recomputed */
  const void* ds_next;                   /* gradient arriving at the returned scores or NULL */
  void *dq, *dk, *dv;
  int64_t lddq, lddk, lddv;
  void* ds_prev;                         /* nullable */
  float* dc;                             /* "+=" scalar, nullable */
} mmemo_attn_problem;
int mmemo_resattn_fwd_grouped_bf16(int n, const mmemo_attn_problem* problems, mmemo_stream_t stream);
int mmemo_resattn_bwd_grouped_bf16(int n, const mmemo_attn_problem* problems, mmemo_stream_t stream);
/* 1 if the problem shape (pointers may be dummy non-null, 16-byte aligned) is served by the
 * mma.sync kernels; bwd != 0 asks about the backward */
int mmemo_resattn_uses_mma(int64_t Lq, int64_t Lk, int64_t hd, int64_t ld, int same_kv, int bwd);
/* Which bf16 kernel family a shape runs on: 3 = tcgen05 single tile (L = 128), 2 = tcgen05 tiled
 * (Lk = 256), 1 = mma.sync, 0 = SIMT.  Used by the benchmarks' tables and the routing tests. */
int mmemo_resattn_kernel_path(int64_t Lq, int64_t Lk, int64_t hd, int64_t ld, int bwd);

/* ---------------------------------------------------------------------------------------------
 * Gated residual + LayerNorm (+ReLU).  y = act( LN( res + gate * x ) * gamma + beta ), eps 1e-5.
 * Replaces others/realformer.py:207-208,263  cmu-mosei/run.py:261  Ren-MME/run.py:166,213
 * robot_demo.py:372-373.  res == null -> LN(gate*x); gate == null -> 1.  mean/rstd (M) saved.
 * bwd: dres (nullable) and dx written; dgate, dgamma, dbeta are "+=" float32; dxsum (nullable,
 * "+=" float32 [d]) receives sum_m dx[m,:], the bias gradient of the Linear that produced x.
 * ------------------------------------------------------------------------------------------- */
int mmemo_add_ln_fwd_f32(const void* res, int64_t ldres, const void* x, int64_t ldx,
                         const float* gate, const float* gamma, const float* beta, void* y,
                         int64_t ldy, float* mean, float* rstd, int64_t M, int64_t d, float eps,
                         int relu, mmemo_stream_t stream);
int mmemo_add_ln_fwd_bf16(const void* res, int64_t ldres, const void* x, int64_t ldx,
                          const float* gate, const float* gamma, const float* beta, void* y,
                          int64_t ldy, float* mean, float* rstd, int64_t M, int64_t d, float eps,
                          int relu, mmemo_stream_t stream);
int mmemo_add_ln_bwd_f32(const void* dy, int64_t lddy, const void* res, int64_t ldres,
                         const void* x, int64_t ldx, const float* gate, const float* gamma,
                         const void* y, int64_t ldy, const float* mean, const float* rstd,
                         void* dres, int64_t lddres, void* dx, int64_t lddx, float* dgate,
                         float* dgamma, float* dbeta, float* dxsum, int64_t M, int64_t d,
                         int relu, mmemo_stream_t stream);
int mmemo_add_ln_bwd_bf16(const void* dy, int64_t lddy, const void* res, int64_t ldres,
                          const void* x, int64_t ldx, const float* gate, const float* gamma,
                          const void* y, int64_t ldy, const float* mean, const float* rstd,
                          void* dres, int64_t lddres, void* dx, int64_t lddx, float* dgate,
                          float* dgamma, float* dbeta, float* dxsum, int64_t M, int64_t d,
                          int relu, mmemo_stream_t stream);

/* Grouped variants (n >= 1 problems, one launch per 40; HOST arrays of length n; rows contiguous, i.e.
 * every leading dimension = d): the LayerNorms of the nine chains of a fusion-trunk layer.  The
 * backward serves d <= 512 (its single-pass kernel), no ReLU.  MMEMO_ERR_SHAPE when a problem does
 * not meet the vector kernels' alignment (16-byte pointers, d % 8 == 0 (bf16) / d % 4 == 0). */
int mmemo_add_ln_fwd_grouped_f32(int n, const void* const* res, const void* const* x,
                                 const float* const* gate, const float* const* gamma,
                                 const float* const* beta, void* const* y, float* const* mean,
                                 float* const* rstd, const int64_t* M, int64_t d, float eps,
                                 int relu, mmemo_stream_t stream);
int mmemo_add_ln_fwd_grouped_bf16(int n, const void* const* res, const void* const* x,
                                  const float* const* gate, const float* const* gamma,
                                  const float* const* beta, void* const* y, float* const* mean,
                                  float* const* rstd, const int64_t* M, int64_t d, float eps,
                                  int relu, mmemo_stream_t stream);
int mmemo_add_ln_bwd_grouped_f32(int n, const void* const* dy, const void* const* res,
                                 const void* const* x, const float* const* gate,
                                 const float* const* gamma, const float* const* mean,
                                 const float* const* rstd, void* const* dres, void* const* dx,
                                 float* const* dgate, float* const* dgamma, float* const* dbeta,
                                 float* const* dxsum, const int64_t* M, int64_t d,
                                 mmemo_stream_t stream);
int mmemo_add_ln_bwd_grouped_bf16(int n, const void* const* dy, const void* const* res,
                                  const void* const* x, const float* const* gate,
                                  const float* const* gamma, const float* const* mean,
                                  const float* const* rstd, void* const* dres, void* const* dx,
                                  float* const* dgate, float* const* dgamma, float* const* dbeta,
                                  float* const* dxsum, const int64_t* M, int64_t d,
                                  mmemo_stream_t stream);

/* out[m % period, n] += x[m, n]  (float32 out).  Bias gradients (period 1) and position-table
 * gradients (period L; backward of others/realformer.py:225-227). */
int mmemo_rowsum_f32(const void* x, int64_t ldx, float* out, int64_t M, int64_t N, int64_t period,
                     mmemo_stream_t stream);
int mmemo_rowsum_bf16(const void* x, int64_t ldx, float* out, int64_t M, int64_t N, int64_t period,
                      mmemo_stream_t stream);
/* out[i][c] += sum_m x[i][m, c] for n >= 1 contiguous (M[i], N) bf16 matrices, one launch per 40
 * (the FFN-1 bias gradients of a trunk layer); N % 8 == 0 */
int mmemo_colsum_grouped_bf16(int n, const void* const* x, float* const* out, const int64_t* M,
                              int64_t N, mmemo_stream_t stream);
/* dtype conversion of n contiguous elements (bf16 shadow copies of float32 master weights) */
int mmemo_cast_f32_to_bf16(const float* src, void* dst, int64_t n, mmemo_stream_t stream);
int mmemo_cast_bf16_to_f32(const void* src, float* dst, int64_t n, mmemo_stream_t stream);
/* `count` tensors, one launch per 64 (host arrays): all bf16 weight shadows of a block / of a
 * whole trunk layer */
int mmemo_cast_f32_to_bf16_multi(int count, const float* const* src, void* const* dst,
                                 const int64_t* n, mmemo_stream_t stream);
/* *out (float32 device scalar, zero-initialised by the caller) += mean(x^2) over n contiguous
 * elements; dx = dloss[0] * 2 x / n.  The synthetic loss of the encoder benchmark (BASELINE config 2
 * has no head of its own) as one launch per direction instead of six eager ATen kernels. */
int mmemo_sqmean_fwd_f32(const void* x, int64_t n, float* out, mmemo_stream_t stream);
int mmemo_sqmean_fwd_bf16(const void* x, int64_t n, float* out, mmemo_stream_t stream);
int mmemo_sqmean_bwd_f32(const void* x, const float* dloss, int64_t n, void* dx,
                         mmemo_stream_t stream);
int mmemo_sqmean_bwd_bf16(const void* x, const float* dloss, int64_t n, void* dx,
                          mmemo_stream_t stream);
/* out[i] = sum of n_in[i] (<= 8) equally sized contiguous tensors, for n_out outputs, one launch
 * per 16 (`in` = the inputs of all outputs, concatenated; out[i] may alias its first input): the
 * gradients reaching one modality stream from the chains that read it (others/realformer.py:232-257),
 * which autograd would add pairwise.  16-byte aligned pointers. */
int mmemo_sum_grouped_f32(int n_out, void* const* out, const int* n_in, const void* const* in,
                          const int64_t* numel, mmemo_stream_t stream);
int mmemo_sum_grouped_bf16(int n_out, void* const* out, const int* n_in, const void* const* in,
                           const int64_t* numel, mmemo_stream_t stream);
/* `count` <= 16 float32 (M, K) matrices (row stride lds) -> bf16 (M, ldd) with ldd % 8 == 0 and
 * zero-filled padding columns, in one launch: raw input features (the float tensors built at
 * others/realformer.py:307-309, Ren-MME/run.py:316-327) and their projection weights become
 * 16-byte-strided operands of the tensor-core GEMM. */
int mmemo_cast_pad_f32_to_bf16_multi(int count, const float* const* src, const int64_t* lds,
                                     void* const* dst, const int64_t* ldd, const int64_t* M,
                                     const int64_t* K, mmemo_stream_t stream);
/* y = x * keep/(1-p), keep ~ Bernoulli(1-p) from a counter-based RNG keyed by (seed, element).
 * Forward and backward are the same call (nn.Dropout at others/realformer.py:139,159,167,222). */
int mmemo_dropout_f32(const void* x, void* y, int64_t n, float p, uint64_t seed,
                      mmemo_stream_t stream);
int mmemo_dropout_bf16(const void* x, void* y, int64_t n, float p, uint64_t seed,
                       mmemo_stream_t stream);
/* The same for n >= 1 tensors, one launch per 64 (the dropout sites of a fusion-trunk layer over all
 * of its chains: Ren-MME/run.py:208,212  robot_demo.py:333,368).  x[i] == y[i] is allowed (in
 * place); 16-byte aligned pointers.  x, y, numel, seeds: HOST arrays of length n.  step: nullable
 * DEVICE scalar mixed into every seed when the kernel runs, so that a captured CUDA graph draws
 * new masks on every replay (the caller increments it once per training step). */
int mmemo_dropout_multi_f32(int n, const void* const* x, void* const* y, const int64_t* numel,
                            const uint64_t* seeds, float p, const uint64_t* step,
                            mmemo_stream_t stream);
int mmemo_dropout_multi_bf16(int n, const void* const* x, void* const* y, const int64_t* numel,
                             const uint64_t* seeds, float p, const uint64_t* step,
                             mmemo_stream_t stream);
/* Backward of mmemo_linear_fwd_grouped_dropout_bf16 for n >= 1 problems, one launch per 64: dym[i]
 * (contiguous bf16 (M[i], N[i])) = mask_i * dy[i] / (1 - p), with dy[i] read at row stride
 * lddy[i] (a column slice of a concatenated output) and the mask of that forward (same seeds, p,
 * step); dbias[i] (nullable array and entries, float32 [N[i]]) += column sums of dym[i];
 * dpos[i] (nullable, float32 (period[i], N[i]) at row stride ldpos[i]) += sums of the UNMASKED
 * dy[i] rows m with m % period[i] = r into row r.  N[i] and lddy[i] even. */
int mmemo_proj_dropout_bwd_bf16(int n, const void* const* dy, const int64_t* lddy,
                                void* const* dym, const int64_t* M, const int64_t* N,
                                const uint64_t* seeds, float p, const uint64_t* step,
                                float* const* dbias, float* const* dpos, const int64_t* period,
                                const int64_t* ldpos, mmemo_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Fusion pooling: concat on features, concat on positions (l, a, v), mean || max over ALL
 * positions (mask-unaware).  Replaces others/realformer.py:258-262  cmu-mosei/run.py:314-318
 * Ren-MME/run.py:266-270  robot_demo.py:435-439 without materialising the concatenation.
 * seg_ptrs: HOST array [n_groups*n_slots]; seg[g*n_slots+s] is a (B, group_len[g], d) tensor of T
 * that fills feature slot s for the positions of group g.  out (B, 2*n_slots*d) float32 =
 * [mean | max]; argmax (B, n_slots*d) int32 = flat position of the first maximum.
 * ------------------------------------------------------------------------------------------- */
int mmemo_pool_fwd_f32(const void* const* seg_ptrs, const int64_t* group_len, int n_groups,
                       int n_slots, int64_t B, int64_t d, float* out, int32_t* argmax,
                       mmemo_stream_t stream);
int mmemo_pool_fwd_bf16(const void* const* seg_ptrs, const int64_t* group_len, int n_groups,
                        int n_slots, int64_t B, int64_t d, float* out, int32_t* argmax,
                        mmemo_stream_t stream);
int mmemo_pool_bwd_f32(const float* dout, const int32_t* argmax, void* const* dseg_ptrs,
                       const int64_t* group_len, int n_groups, int n_slots, int64_t B, int64_t d,
                       mmemo_stream_t stream);
int mmemo_pool_bwd_bf16(const float* dout, const int32_t* argmax, void* const* dseg_ptrs,
                        const int64_t* group_len, int n_groups, int n_slots, int64_t B, int64_t d,
                        mmemo_stream_t stream);
/* The same forward for n_towers >= 1 fusion trunks at once (the towers of every member of an
 * ensemble: others/realformer.py:258-262 and cmu-mosei/run.py:314-318 / Ren-MME/run.py:266-270 once
 * per tower and member), without argmax (inference).  seg_ptrs: HOST array [n_towers][n_groups *
 * n_slots]; out: HOST array of n_towers (B, 2*n_slots*d) float32 outputs.  All towers share B, d,
 * n_groups, n_slots and group_len.  Each out[t] is bitwise equal to mmemo_pool_fwd_* on tower t.
 * Every tower is checked before the first launch; one launch per 16 towers (fewer when a tower has
 * more than 16 segments: 256 segment pointers per launch). */
int mmemo_pool_fwd_multi_f32(int n_towers, const void* const* seg_ptrs, const int64_t* group_len,
                             int n_groups, int n_slots, int64_t B, int64_t d, float* const* out,
                             mmemo_stream_t stream);
int mmemo_pool_fwd_multi_bf16(int n_towers, const void* const* seg_ptrs, const int64_t* group_len,
                              int n_groups, int n_slots, int64_t B, int64_t d, float* const* out,
                              mmemo_stream_t stream);

/* Training form for the k folds of folds.py: n_towers towers with their OWN batch sizes B[t] (HOST
 * array), and each tower's argmax (B[t], n_slots*d) int32 in argmax[t] (HOST array).  out[t] and
 * argmax[t] are bitwise what mmemo_pool_fwd_* writes for tower t. */
int mmemo_pool_fwd_multi_arg_f32(int n_towers, const void* const* seg_ptrs,
                                 const int64_t* group_len, int n_groups, int n_slots,
                                 const int64_t* B, int64_t d, float* const* out,
                                 int32_t* const* argmax, mmemo_stream_t stream);
int mmemo_pool_fwd_multi_arg_bf16(int n_towers, const void* const* seg_ptrs,
                                  const int64_t* group_len, int n_groups, int n_slots,
                                  const int64_t* B, int64_t d, float* const* out,
                                  int32_t* const* argmax, mmemo_stream_t stream);
/* mmemo_pool_bwd_* of every tower in one launch per 16 towers: dout[t], argmax[t] and the
 * dseg_ptrs of tower t ([n_towers][n_groups * n_slots], HOST arrays) with batch size B[t].  Each
 * tower's segment gradients are bitwise those of mmemo_pool_bwd_*. */
int mmemo_pool_bwd_multi_f32(int n_towers, const float* const* dout, int32_t* const* argmax,
                             void* const* dseg_ptrs, const int64_t* group_len, int n_groups,
                             int n_slots, const int64_t* B, int64_t d, mmemo_stream_t stream);
int mmemo_pool_bwd_multi_bf16(int n_towers, const float* const* dout, int32_t* const* argmax,
                              void* const* dseg_ptrs, const int64_t* group_len, int n_groups,
                              int n_slots, const int64_t* B, int64_t d, mmemo_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Heads and losses (float32 only; O(B*C) work).
 * state_transfer: others/realformer.py:274-286.  feats (B,P,2C) = [o | g]; out (B,P,C).
 * bilinear_head : cmu-mosei/run.py:332-339  Ren-MME/run.py:285-292  rencecps/run.py:141-148
 *                 z[b,k] = sum_{j,m} this[b,j] last[b,m] T[j,m,k]; out = W [this || LN(z)] + bias.
 * circle_loss   : others/realformer.py:289-298 (per-row loss, literal +-1e12 masking).
 * rdrop_kl      : Ren-MME/run.py:332-334 (scalar; rows 2i / 2i+1; target not detached).
 * ------------------------------------------------------------------------------------------- */
int mmemo_state_transfer_fwd(const float* feats, const float* trans, float* out, int64_t B,
                             int64_t P, int64_t C, mmemo_stream_t stream);
int mmemo_state_transfer_bwd(const float* dout, const float* feats, const float* trans,
                             const float* out, float* dfeats, float* dtrans, int64_t B, int64_t P,
                             int64_t C, mmemo_stream_t stream);
int mmemo_bilinear_head_fwd(const float* this_feat, const float* last_feat, const float* trans,
                            const float* gamma, const float* beta, const float* w,
                            const float* bias, float* out, float* z, int64_t B, int64_t C,
                            float eps, mmemo_stream_t stream);
int mmemo_bilinear_head_bwd(const float* dout, const float* this_feat, const float* last_feat,
                            const float* trans, const float* gamma, const float* beta,
                            const float* w, const float* z, float* dthis, float* dlast,
                            float* dtrans, float* dgamma, float* dbeta, float* dw, float* dbias,
                            int64_t B, int64_t C, float eps, mmemo_stream_t stream);
int mmemo_circle_loss_fwd(const float* logits, const float* labels, float* loss, int64_t R,
                          int64_t C, mmemo_stream_t stream);
int mmemo_circle_loss_bwd(const float* dloss, const float* logits, const float* labels,
                          float* dlogits, int64_t R, int64_t C, mmemo_stream_t stream);
int mmemo_rdrop_kl_fwd(const float* logits, float* out, int64_t B, int64_t C,
                       mmemo_stream_t stream);
int mmemo_rdrop_kl_bwd(const float* dout, const float* logits, float* dlogits, int64_t B, int64_t C,
                       mmemo_stream_t stream);

/* The same heads and losses for n >= 0 members (the k folds trained together by folds.py), one
 * launch per 32 members.  Every pointer argument is a HOST array with one device pointer per member
 * (entries of dtrans / dgamma / dbeta / dw / dbias / weights may be null: not computed / no
 * weights); B[i] / R[i] is member i's batch size / row count; P and C are shared.  Each member's
 * forward output is bitwise that of the per-model entry point; parameter gradients are summed with
 * float atomics within a member (as there) and never across members.
 * circle_loss_fwd_multi: loss[i] (one float) = mean over the R[i] rows of circle_loss (times
 *   weights[i][r] when given): (multi_circle_loss(logits, labels) [* weights]).mean().
 * circle_loss_bwd_multi: its gradient for d loss[i] = dloss[i][0].
 * rdrop_kl_*_multi: mmemo_rdrop_kl_* per member (B[i] even, >= 2). */
int mmemo_state_transfer_fwd_multi(int n, const float* const* feats, const float* const* trans,
                                   float* const* out, const int64_t* B, int64_t P, int64_t C,
                                   mmemo_stream_t stream);
int mmemo_state_transfer_bwd_multi(int n, const float* const* dout, const float* const* feats,
                                   const float* const* trans, const float* const* out,
                                   float* const* dfeats, float* const* dtrans, const int64_t* B,
                                   int64_t P, int64_t C, mmemo_stream_t stream);
int mmemo_bilinear_head_fwd_multi(int n, const float* const* this_feat,
                                  const float* const* last_feat, const float* const* trans,
                                  const float* const* gamma, const float* const* beta,
                                  const float* const* w, const float* const* bias,
                                  float* const* out, float* const* z, const int64_t* B, int64_t C,
                                  float eps, mmemo_stream_t stream);
int mmemo_bilinear_head_bwd_multi(int n, const float* const* dout, const float* const* this_feat,
                                  const float* const* last_feat, const float* const* trans,
                                  const float* const* gamma, const float* const* beta,
                                  const float* const* w, const float* const* z,
                                  float* const* dthis, float* const* dlast, float* const* dtrans,
                                  float* const* dgamma, float* const* dbeta, float* const* dw,
                                  float* const* dbias, const int64_t* B, int64_t C, float eps,
                                  mmemo_stream_t stream);
int mmemo_circle_loss_fwd_multi(int n, const float* const* logits, const float* const* labels,
                                const float* const* weights, const int64_t* R, int64_t C,
                                float* const* loss, mmemo_stream_t stream);
int mmemo_circle_loss_bwd_multi(int n, const float* const* dloss, const float* const* logits,
                                const float* const* labels, const float* const* weights,
                                float* const* dlogits, const int64_t* R, int64_t C,
                                mmemo_stream_t stream);
int mmemo_rdrop_kl_fwd_multi(int n, const float* const* logits, const int64_t* B, int64_t C,
                             float* const* out, mmemo_stream_t stream);
int mmemo_rdrop_kl_bwd_multi(int n, const float* const* dout, const float* const* logits,
                             float* const* dlogits, const int64_t* B, int64_t C,
                             mmemo_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Ensemble head (inference, float32): y = (out_1 + ... + out_K) / K over K >= 1 members, summed as
 * a left fold in member order without atomics (the same bits on every run).  Replaces, per member,
 * the classifier linears and head of others/realformer.py:270-286, cmu-mosei/run.py:330-339,
 * Ren-MME/run.py:283-292 or rencecps/run.py:141-148, and the averaging of
 * others/realformer.py:418-420, Ren-MME/run.py:560, robot_demo.py:610-615.
 *   MMEMO_HEAD_BILINEAR (y (B, C)):  last = w0 x0[b], this = w1 x1[b] (w0, w1: (C, F)),
 *       z = sum_{j,m} this_j last_m trans[j,m,:] (trans (C,C,C)),
 *       out = w_out [this || LN_C(z; ln_gamma, ln_beta)] + b_out   (w_out (C, 2C)).
 *   MMEMO_HEAD_STATE_TRANSFER (y (B, P, C)): for row r = b*P + p of x0 (B*P rows),
 *       h = ReLU(LN_d(w0 x0[r] + b0; ln_gamma, ln_beta))   (w0 (d, F)),
 *       [o | g] = w_out h + b_out   (w_out (2C, d)), then the window recurrence of
 *       mmemo_state_transfer_fwd with trans (C, C).
 * x0 / x1 rows are ld0 / ld1 floats apart (>= F); weights are contiguous.  members: HOST array.
 * C <= 16, d <= 1024, else MMEMO_ERR_SHAPE; a null required pointer is MMEMO_ERR_ARG.  Every member
 * is checked before the first launch; one launch per 8 members (later launches add to y).
 * ------------------------------------------------------------------------------------------- */
#define MMEMO_HEAD_BILINEAR 0
#define MMEMO_HEAD_STATE_TRANSFER 1
typedef struct mmemo_ensemble_member {
  const float* x0;        /* BILINEAR: x_last (B, F);  STATE_TRANSFER: x (B*P, F) */
  int64_t ld0;
  const float* x1;        /* BILINEAR: x_this (B, F);  STATE_TRANSFER: unused */
  int64_t ld1;
  const float* w0;        /* BILINEAR: W_last (C, F);  STATE_TRANSFER: W_fc (d, F) */
  const float* w1;        /* BILINEAR: W_this (C, F);  STATE_TRANSFER: unused */
  const float* b0;        /* BILINEAR: unused;         STATE_TRANSFER: b_fc (d) */
  const float* ln_gamma;  /* LayerNorm over C (BILINEAR) or d (STATE_TRANSFER) */
  const float* ln_beta;
  const float* w_out;     /* BILINEAR: (C, 2C);        STATE_TRANSFER: W_cls (2C, d) */
  const float* b_out;     /* BILINEAR: (C);            STATE_TRANSFER: b_cls (2C) */
  const float* trans;     /* BILINEAR: (C, C, C);      STATE_TRANSFER: (C, C) */
} mmemo_ensemble_member;
int mmemo_ensemble_head_fwd(int kind, int n_members, const mmemo_ensemble_member* members,
                            int64_t B, int64_t P, int64_t F, int64_t d, int64_t C, float eps,
                            float* y, mmemo_stream_t stream);
/* The same, and every member's own output out_k in y_members (K, B, P, C) float32 (P = 1 for
 * BILINEAR); y is bitwise what mmemo_ensemble_head_fwd writes. */
int mmemo_ensemble_head_fwd_members(int kind, int n_members, const mmemo_ensemble_member* members,
                                    int64_t B, int64_t P, int64_t F, int64_t d, int64_t C,
                                    float eps, float* y, float* y_members, mmemo_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Fold-ensemble uncertainty (inference, new: the reference scripts only sum the logits).  logits
 * (K, N, C) contiguous, T = float32 / bf16, K >= 1 folds of N rows; natural log, nats.  Per row n,
 * with p_k = softmax(logits[k, n]) (max subtracted):
 *   mean_prob[n, c]      = (1/K) sum_k p_k[c]                                       (N, C)
 *   var_prob[n, c]       = (1/(K-1)) sum_k (p_k[c] - mean_prob[n, c])^2, 0 if K = 1  (N, C)
 *   entropy[n]           = -sum_c mean_prob log mean_prob                          (N)
 *   expected_entropy[n]  = (1/K) sum_k -sum_c p_k[c] log p_k[c]                     (N)
 *   mutual_info[n]       = max(entropy - expected_entropy, 0), 0 if K = 1          (N)
 *   label[n]             = first argmax_c mean_prob[n, c]                          (N) int64
 * One warp per row, the folds in registers.  C <= 1024, else MMEMO_ERR_SHAPE.
 * ------------------------------------------------------------------------------------------- */
int mmemo_fold_uncertainty_f32(const void* logits, int64_t K, int64_t N, int64_t C,
                               float* mean_prob, float* var_prob, float* entropy,
                               float* expected_entropy, float* mutual_info, int64_t* label,
                               mmemo_stream_t stream);
int mmemo_fold_uncertainty_bf16(const void* logits, int64_t K, int64_t N, int64_t C,
                                float* mean_prob, float* var_prob, float* entropy,
                                float* expected_entropy, float* mutual_info, int64_t* label,
                                mmemo_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Data-parallel gradient exchange (new; the reference is single-GPU, others/realformer.py:16).
 * Two-shot SUM all-reduce, in place, of n_elems float32 starting offset_elems into a buffer that
 * every rank allocated symmetrically (same size; peer mappings exchanged by the host).
 *   multicast_ptr       : NVLS multicast mapping of the buffer, or NULL -> plain peer loads/stores
 *   buffer_ptrs_dev     : device array [world] of the ranks' mappings of the buffer
 *   signal_pad_ptrs_dev : device array [world] of the ranks' uint32 flag pads (zero-initialised);
 *                         slots [signal_slot_base, signal_slot_base + blocks*world) are used
 * n_elems must be a multiple of 4*world, offset_elems of 4.  Every rank must launch the same
 * sequence of calls.  A rank that waits > 20 s for a peer traps instead of hanging.
 * ------------------------------------------------------------------------------------------- */
int mmemo_allreduce_sum_f32(void* multicast_ptr, void* const* buffer_ptrs_dev,
                            void* const* signal_pad_ptrs_dev, int64_t signal_slot_base,
                            int64_t offset_elems, int64_t n_elems, int rank, int world, int blocks,
                            mmemo_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Fused gradient clipping + Adam / AdamW over a list of float32 tensors (host arrays of device
 * pointers and element counts).  Replaces nn.utils.clip_grad_norm_(params, CLIP) +
 * optimizer.step(): others/realformer.py:314-315,342 (Adam), cmu-mosei/run.py:368-369,398,
 * Ren-MME/run.py:336-337,379, rencecps/run.py:175-176,202, robot_demo.py:471-472,502 (AdamW).
 * One call may serve several optimizers (the k folds of a cross-validation, one model each), with
 * one launch per 96 tensors whatever their number; one optimizer is the case of a single slot 0.
 *   grad_sqnorm_multi : sqnorm_out[slot[i]] += |g_i|^2 (float32 device array, zero-initialised by
 *                       the caller): one squared norm per optimizer
 *   clip_grads        : g_i *= min(1, max_norm / (sqrt(*sqnorm) + 1e-6))       [torch's formula]
 *   adam_step_multi   : torch.optim.Adam (decoupled=0: g += wd*p) / AdamW (decoupled=1:
 *                       p *= 1-lr*wd), no amsgrad, with per-tensor lr[i], step[i] (the 1-based step
 *                       count of this update) and weight_decay[i]; betas, eps, decoupled and
 *                       max_norm are shared by the call.  With sqnorm != NULL the clip coefficient
 *                       above, from sqnorm[slot[i]], is applied to the gradients on the fly (grads
 *                       are not modified), so clip + step cost one pass.
 * All arrays of pointers, counts and per-tensor values are HOST arrays of length count.
 * ------------------------------------------------------------------------------------------- */
int mmemo_grad_sqnorm_multi_f32(int count, const float* const* grads, const int64_t* numel,
                                const int* slot, float* sqnorm_out, mmemo_stream_t stream);
int mmemo_clip_grads_f32(int count, float* const* grads, const int64_t* numel, const float* sqnorm,
                         float max_norm, mmemo_stream_t stream);
int mmemo_adam_step_multi_f32(int count, float* const* params, const float* const* grads,
                              float* const* exp_avg, float* const* exp_avg_sq, const int64_t* numel,
                              const float* lr, const int64_t* step, const float* weight_decay,
                              const int* slot, float beta1, float beta2, float eps, int decoupled,
                              const float* sqnorm, float max_norm, mmemo_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Device-side batch assembly: ragged float32 sequences (rows of D features, concatenated in
 * `flat`; sample n owns rows [row_start[n], row_start[n] + n_rows[n])) -> padded batch
 * out (N, m_len, D) + mask (N, m_len; nullable).  mode 0 "tail": the last min(T, m_len) rows
 * (others/realformer.py:72-82,100-102); mode 1 "head": the first ones; mode 2 "stride": T < m_len
 * -> all rows, else rows 0, gap, 2 gap, ... with gap = T / m_len (robot_demo.py:86-99,115-150).
 * Remaining rows are 0 and masked out; do_scrub replaces NaN / +-Inf by scrub_value (-71 in the
 * reference).  n_rows[n] == 0 gives an all-zero, fully masked sample ('no_name' slots).
 * ------------------------------------------------------------------------------------------- */
int mmemo_assemble_batch_f32(const float* flat, const int64_t* row_start, const int64_t* n_rows,
                             float* out, float* mask, int64_t N, int64_t m_len, int64_t D,
                             int mode, int do_scrub, float scrub_value, mmemo_stream_t stream);

/* cmu-mosei/run.py:104-151 (masking, the non-BERT branch used by its data_loader :169-180):
 * out rows 0,1,2 = column-wise max, min, mean over ALL rows of the sample (after the NaN/Inf
 * scrub), rows 3.. = m_len-3 body rows: view 0 = the first ones, view 1 = the last ones (identical
 * to view 0 when the sample has fewer than m_len-3 rows: such samples have ONE view, zero-padded,
 * mask = 1 on their n_rows+3 rows).  n_rows[n] == 0 -> all-zero sample and mask. */
int mmemo_assemble_stats_batch_f32(const float* flat, const int64_t* row_start,
                                   const int64_t* n_rows, float* out, float* mask, int64_t N,
                                   int64_t m_len, int64_t D, int view, int do_scrub,
                                   float scrub_value, mmemo_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* MMEMO_H_ */
