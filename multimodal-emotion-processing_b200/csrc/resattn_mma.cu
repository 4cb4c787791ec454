// Fused residual-attention core on the warp-level tensor-core path (mma.sync.m16n8k16, bf16
// operands, fp32 accumulation) for the head sizes / lengths of the reference's real models:
// hd = 16 (others/realformer.py, cmu-mosei/run.py, Ren-MME/run.py), hd = 32 (robot_demo.py),
// hd = 64 with ragged lengths; any Lq, Lk (20 ... 275 in the reference configs).  tcgen05 tiles
// (128 x N x 16, one head per CTA) do not fit 16-wide heads and 20..275-long sequences, so these
// shapes run as 16-row warp tiles; the tcgen05 kernel (resattn_tc.cu) keeps hd = 64, L = 128.
//
// GROUPED: one launch serves up to MAXP independent problems (the nine chains of a fusion-trunk
// layer, both towers of Concat_Trans / Base_model, the members of an ensemble) - the problem
// table travels as a kernel parameter and blockIdx.x is mapped to (problem, batch, head, tile).
// A call with more problems is split into consecutive chunks of MAXP, one set of launches each.
//
// Forward  (replaces others/realformer.py:189-203 and its twins): CTA = (b, h, 64 query rows),
//   4 warps x 16 rows.  K_h, V_h (and the Q tile) are staged in shared memory by cp.async in an
//   XOR-swizzled layout read back with ldmatrix; keys are walked in blocks of 64:
//   S = Q K^T (mma) -> scale, + c*S_prev, - 1e8*(1-mask) in the reference's fp32 op order, bf16
//   round -> S written -> online softmax (running max / sum, fp32) -> O += P V (mma, P from
//   registers).  The n index of each 8-wide MMA tile is PERMUTED over the keys of a 32-key group
//   (tile i, column n  <->  key 8*(n/2) + 2*i + n%2) so that a lane ends up owning 8 CONTIGUOUS
//   keys of a row: S_prev / S / dS move as 16-byte vectors although the accumulator layout gives a
//   lane only 2 adjacent columns per tile.  The permutation costs nothing: ldmatrix takes one row
//   address per lane.
// Backward (autograd of the above): CTA = (b, h), 8 warps, keys in blocks of KB (64 or 32).
//   phase A (warp = 16 query rows): S (re-read, or recomputed by mma when it was not stored),
//     P = exp(S - max)/sum, dP = dO V^T (mma), dS = P*(dP - D) + dS_next, dc += dS*S_prev,
//     dS_prev = c*dS (16-byte stores), dQ += dS K (mma, fp32 tile in shared memory); P and dS of
//     the block go to shared memory as bf16;
//   phase B (warp = 16 keys x {dV, dK}): dV = P^T dO, dK = dS^T Q over ALL query rows (mma with
//     ldmatrix.trans operands) - complete for the block, written straight to HBM.
#include <math.h>
#include <stdlib.h>

#include "common.cuh"
#include "resattn.h"

namespace {

constexpr int MAXP = 40;          // problems per launch (a call takes any number: chunks of MAXP)
// Kernel instantiations by the role of a layer in its chain.  The flags of a problem (previous
// scores? scores written / stored? score gradients in / out?) are runtime data in M_GEN; the other
// modes fix them at compile time, which removes the per-chunk pointer tests, the scalar fall-back
// of the score-tensor accesses and (M_PLAIN) all score-tensor code from the inner loops.
//            forward                         backward
//  M_PLAIN   no S_prev, S not written        recompute, no S_prev / dS_next / dS_prev   (1-layer chain)
//  M_FIRST   no S_prev, S written            S stored, no S_prev, dS_next, no dS_prev   (first of n)
//  M_MID     S_prev, S written               S stored, S_prev, dS_next, dS_prev
//  M_LAST    S_prev, S not written           recompute, S_prev, no dS_next, dS_prev      (last of n)
// M_FIRST..M_LAST additionally require 16-byte accessible score rows (vec_s).
constexpr int M_GEN = 0, M_PLAIN = 1, M_FIRST = 2, M_MID = 3, M_LAST = 4;
constexpr int FWD_WARPS = 4, FWD_ROWS = 64;
constexpr int BWD_WARPS = 8;
constexpr size_t SMEM_MAX = 226 * 1024;   // dynamic part (227 KB per CTA minus static + reserve)

struct Prob {
  const bf16 *q, *k, *v;
  const float* mask;
  const bf16* s_prev;
  const float* c;
  bf16* s_out;
  bf16* o;
  float* lse;
  // backward
  const bf16 *d_o, *s, *ds_next, *o_in;
  bf16 *dq, *dk, *dv, *ds_prev;
  float* dc;
  int ldq, ldk, ldv, ldo, lds, lddo, lddq, lddk, lddv, mask_bs;
  int B, H, Lq, Lk;
  int vec_s;        // score tensors may be accessed with 16-byte vectors
  int cta_start;
};

struct Table {
  int n, total;
  float inv_sqrt;
  int kv_blocked;   // backward: K / V are staged one key block at a time (long hd = 64 sequences)
  int cta_start[MAXP + 1];   // contiguous: the blockIdx -> problem search reads one or two lines
  Prob p[MAXP];
};

// ---- PTX wrappers ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t s_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void cp16(uint32_t dst, const void* src, bool valid) {
  const int sz = valid ? 16 : 0;     // src-size 0: the 16 bytes are zero-filled
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(sz)
               : "memory");
}
__device__ __forceinline__ void cp_commit_wait() {
  asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory");
}
__device__ __forceinline__ void ldsm4(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ void ldsm4t(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0,
                                         uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, "
      "{%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ float bf_lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf_hi(uint32_t w) { return __uint_as_float(w & 0xFFFF0000u); }
__device__ __forceinline__ float round_bf(float x) {
  return __bfloat162float(__float2bfloat16_rn(x));
}
__device__ __forceinline__ float quad_max(float v) {
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
  return fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
}
__device__ __forceinline__ float quad_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  return v + __shfl_xor_sync(0xffffffffu, v, 2);
}

// Shared-memory tile [rows][HD] of bf16, 16-byte chunks XOR-swizzled so that the 8 row addresses
// of an ldmatrix fall into distinct bank groups for every HD (32 / 64 / 128-byte rows).
template <int HD>
__device__ __forceinline__ uint32_t sw(int row, int chunk) {
  constexpr int RB = HD * 2, CPR = HD / 8, RP = 128 / RB;
  return (uint32_t)(row * RB + ((chunk ^ ((row / RP) % CPR)) << 4));
}
// [rows][64] bf16 tiles (P, dS): 128-byte rows; [rows][32]: 64-byte rows
template <int KB>
__device__ __forceinline__ uint32_t swp(int row, int chunk) {
  return sw<KB>(row, chunk);
}

// key of (tile i of a 32-key group, n index of the MMA tile): lanes end up with 8 contiguous keys
__device__ __forceinline__ int perm_key(int i, int n) { return 8 * (n >> 1) + 2 * i + (n & 1); }

// 8 consecutive bf16 of a score-shaped tensor -> fp32 (vector path when the row stride allows)
__device__ __forceinline__ void load8(const bf16* p, int n_valid, bool vec, float (&v)[8]) {
  if (vec && n_valid >= 8) {
    const uint4 t = *reinterpret_cast<const uint4*>(p);
    const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) { v[2 * i] = bf_lo(w[i]); v[2 * i + 1] = bf_hi(w[i]); }
  } else {
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = (i < n_valid) ? __bfloat162float(p[i]) : 0.f;
  }
}
__device__ __forceinline__ void store8(bf16* p, int n_valid, bool vec, const float (&v)[8]) {
  if (vec && n_valid >= 8) {
    *reinterpret_cast<uint4*>(p) = make_uint4(pack2(v[0], v[1]), pack2(v[2], v[3]),
                                              pack2(v[4], v[5]), pack2(v[6], v[7]));
  } else {
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (i < n_valid) p[i] = __float2bfloat16_rn(v[i]);
  }
}

// Lane-constant shared-memory offsets of the ldmatrix operands.  Key rows are addressed as
// R0 + row with R0 a multiple of 32 and query rows as 16*rt + row: the XOR swizzle term of sw<HD>
// then depends on `row` only, so the offsets are computed once per kernel and the loops add
// R0 * row_bytes (keeps the integer / predicate instruction count - 2/3 of the first version's
// instruction mix - out of the inner loops).
template <int HD>
struct LaneOffs {
  uint32_t a[HD / 16];        // A operand (Q / dO rows 16*rt + ...), per k-tile
  uint32_t n[2][HD / 16];     // B operand, keys as n (K for QK^T, V for dO V^T): [tile pair][k-tile]
  uint32_t t[2][HD / 16];     // B operand, keys as k via .trans (V for PV, K for dS K): [pair][2 n-tiles]
  __device__ __forceinline__ void init(int lane) {
    const int mi = lane >> 3, r = lane & 7;
#pragma unroll
    for (int kt = 0; kt < HD / 16; ++kt) {
      a[kt] = sw<HD>((lane & 7) + ((lane >> 3) & 1) * 8, 2 * kt + (lane >> 4));
#pragma unroll
      for (int ip = 0; ip < 2; ++ip) {
        n[ip][kt] = sw<HD>(perm_key(ip * 2 + (mi >> 1), r), 2 * kt + (mi & 1));
        t[ip][kt] = sw<HD>(perm_key(2 * ip + (mi & 1), r), 2 * kt + (mi >> 1));
      }
    }
  }
};
constexpr float LOG2E = 1.4426950408889634f;
__device__ __forceinline__ float fast_exp2(float x) {          // MUFU.EX2; 2^(-inf) = 0
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// blockIdx.x -> (problem, CTA index inside the problem).  The problem's descriptor is COPIED from
// the kernel-parameter table into shared memory once per CTA: reading it field by field through a
// dynamically indexed constant-bank reference cost an LDCU miss per access (ncu: 36 % of the
// backward kernel's stall samples).
__device__ __forceinline__ const Prob& locate(const Table& T, int& local) {
  __shared__ Prob sp;
  int p = 0;
  while (p + 1 < T.n && (int)blockIdx.x >= T.cta_start[p + 1]) ++p;
  local = (int)blockIdx.x - T.cta_start[p];
  const uint32_t* src = reinterpret_cast<const uint32_t*>(&T.p[p]);
  uint32_t* dst = reinterpret_cast<uint32_t*>(&sp);
  for (int i = threadIdx.x; i < (int)(sizeof(Prob) / 4); i += blockDim.x) dst[i] = src[i];
  __syncthreads();
  return sp;
}

// stage `rows` rows of a (.., ld) bf16 matrix (head slice: HD columns starting at col0) into a
// swizzled tile; rows >= n_rows are zero-filled
template <int HD>
__device__ __forceinline__ void stage(uint32_t dst, const bf16* src, int ld, int n_rows,
                                      int rows_padded) {
  constexpr int CPR = HD / 8;
  const int NT = blockDim.x;
  for (int i = threadIdx.x; i < rows_padded * CPR; i += NT) {
    const int r = i / CPR, ch = i - r * CPR;
    const bool ok = r < n_rows;
    cp16(dst + sw<HD>(r, ch), src + (size_t)(ok ? r : 0) * ld + ch * 8, ok);
  }
}

// =============================================================================================
// forward
// =============================================================================================
// (register caps keep 5 / 4 / 3 CTAs of 4 warps resident per SM for hd = 16 / 32 / 64; the PLAIN
// hd = 16 instantiation fits 72 registers without spills: 7 CTAs)
// PLAIN = no previous scores and no score output: the single layer of a one-layer trunk (Ren-MME's
// default, cmu-mosei with n_layers = 1: any chain of length one).  The scores
// then never leave the registers, so they are not rounded to bf16 (the backward's PLAIN recompute
// does the same), key padding is handled by a +inf entry in the additive-mask row instead of
// per-element selects, and none of the global score-tensor address / predicate code is compiled
// in: 24 -> ~10 instructions per score (ncu source counters, profiles/).
template <int HD, int MODE>
__global__ void __launch_bounds__(FWD_WARPS * 32,
                                  HD == 16 ? (MODE == M_PLAIN ? 7 : 5) : (HD == 32 ? 4 : 3))
resattn_mma_fwd_kernel(const __grid_constant__ Table T) {
  constexpr bool PLAIN = MODE == M_PLAIN, SPEC = MODE >= M_FIRST;
  extern __shared__ __align__(128) uint8_t smem[];
  int local;
  const Prob& P = locate(T, local);
  const int Lq = P.Lq, Lk = P.Lk, H = P.H;
  const int qtiles = (Lq + FWD_ROWS - 1) / FWD_ROWS;
  const int qt = local % qtiles, bh = local / qtiles, h = bh % H, b = bh / H;
  const int q0 = qt * FWD_ROWS;
  const int LkP = (Lk + 63) & ~63;
  const bool same_kv = (P.k == P.v) && (P.ldk == P.ldv);
  const uint32_t sQ = s_u32(smem);
  const uint32_t sK = sQ + FWD_ROWS * HD * 2;
  const uint32_t sV = same_kv ? sK : sK + LkP * HD * 2;
  float* sbias = reinterpret_cast<float*>(smem + FWD_ROWS * HD * 2 + (same_kv ? 1 : 2) * LkP * HD * 2);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;

  pdl_wait();
  pdl_trigger();
  stage<HD>(sQ, P.q + ((size_t)b * Lq + q0) * P.ldq + h * HD, P.ldq,
                            min(FWD_ROWS, Lq - q0), FWD_ROWS);
  stage<HD>(sK, P.k + (size_t)b * Lk * P.ldk + h * HD, P.ldk, Lk, LkP);
  if (!same_kv) stage<HD>(sV, P.v + (size_t)b * Lk * P.ldv + h * HD, P.ldv, Lk, LkP);
  for (int j = threadIdx.x; j < LkP; j += FWD_WARPS * 32) {
    float bias = (P.mask && j < Lk) ? 1.0e8f * (1.0f - P.mask[(size_t)b * P.mask_bs + j]) : 0.f;
    if (PLAIN && j >= Lk) bias = INFINITY;   // padded keys: s = 0 - inf, p = 2^(-inf) = 0
    sbias[j] = bias;
  }
  cp_commit_wait();
  __syncthreads();

  const int r0 = q0 + warp * 16;          // first query row of this warp
  if (r0 >= Lq) return;
  const bool has_prev = SPEC ? (MODE != M_FIRST) : (!PLAIN && P.s_prev != nullptr);
  const bool has_mask = P.mask != nullptr;
  const float cval = (has_prev && P.c) ? P.c[0] : 0.f;
  const float inv_sqrt = T.inv_sqrt;
  const bool vec = SPEC ? true : P.vec_s != 0;
  const int lds = P.lds;
  const int rowA = r0 + g, rowB = r0 + g + 8;
  const bool okA = rowA < Lq, okB = rowB < Lq;
  const size_t sbase = ((size_t)b * H + h) * Lq;
  const size_t soff[2] = {(sbase + (okA ? rowA : 0)) * lds, (sbase + (okB ? rowB : 0)) * lds};
  const bf16* __restrict__ sprev = P.s_prev;
  bf16* __restrict__ sout = P.s_out;
  const bool has_sout = SPEC ? (MODE != M_LAST) : (!PLAIN && sout != nullptr);
  constexpr uint32_t RB = HD * 2;
  LaneOffs<HD> lo;
  lo.init(lane);

  // Q fragments (A operand), all k-tiles
  uint32_t qa[HD / 16][4];
#pragma unroll
  for (int kt = 0; kt < HD / 16; ++kt) ldsm4(sQ + warp * 16 * RB + lo.a[kt], qa[kt]);

  float o[HD / 8][4];
#pragma unroll
  for (int n = 0; n < HD / 8; ++n)
#pragma unroll
    for (int e = 0; e < 4; ++e) o[n][e] = 0.f;
  float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f};

  for (int kb = 0; kb < Lk; kb += 64) {
    float sc[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int e = 0; e < 4; ++e) sc[i][e] = 0.f;
    // ---- S = Q K^T : 2 groups of 32 keys x 4 permuted tiles ------------------------------------
#pragma unroll
    for (int G = 0; G < 2; ++G) {
      const uint32_t kbase = sK + (uint32_t)(kb + 32 * G) * RB;
#pragma unroll
      for (int ip = 0; ip < 2; ++ip)
#pragma unroll
        for (int kt = 0; kt < HD / 16; ++kt) {
          uint32_t kf[4];
          ldsm4(kbase + lo.n[ip][kt], kf);
          mma16816(sc[G * 4 + ip * 2], qa[kt], kf[0], kf[1]);
          mma16816(sc[G * 4 + ip * 2 + 1], qa[kt], kf[2], kf[3]);
        }
    }
    // ---- scale, + c*S_prev, - 1e8*(1-mask), bf16 round, store S; block max ----------------------
    float bmax[2] = {-INFINITY, -INFINITY};
    if constexpr (PLAIN) {
#pragma unroll
      for (int G = 0; G < 2; ++G) {
        const float* bp = sbias + kb + 32 * G + 8 * t;
        const float4 b0 = *reinterpret_cast<const float4*>(bp);
        const float4 b1 = *reinterpret_cast<const float4*>(bp + 4);
        const float bias[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int e = 0; e < 4; ++e) {               // e >> 1 = row half, key = 2 i + (e & 1)
            const float sx = __fsub_rn(__fmul_rn(sc[G * 4 + i][e], inv_sqrt), bias[2 * i + (e & 1)]);
            sc[G * 4 + i][e] = sx;
            bmax[e >> 1] = fmaxf(bmax[e >> 1], sx);
          }
      }
    } else {
#pragma unroll
    for (int G = 0; G < 2; ++G) {
      const int k0 = kb + 32 * G + 8 * t;             // this lane's 8 contiguous keys
      const int nvalid = Lk - k0;                     // >= 8: the whole chunk is inside the keys
      float bias[8];
      if (has_mask) {
        const float4 b0 = *reinterpret_cast<const float4*>(sbias + k0);
        const float4 b1 = *reinterpret_cast<const float4*>(sbias + k0 + 4);
        bias[0] = b0.x; bias[1] = b0.y; bias[2] = b0.z; bias[3] = b0.w;
        bias[4] = b1.x; bias[5] = b1.y; bias[6] = b1.z; bias[7] = b1.w;
      }
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        const bool row_ok = half ? okB : okA;
        const bool use_prev = has_prev && row_ok && nvalid > 0;
        float pv[8];
        if (use_prev) load8(sprev + soff[half] + k0, lds - k0, vec, pv);
        float sv[8];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int j = 2 * i + e;
            float s = sc[G * 4 + i][half * 2 + e] * inv_sqrt;
            if (use_prev) s = __fadd_rn(s, __fmul_rn(cval, pv[j]));
            if (has_mask) s = __fsub_rn(s, bias[j]);
            sv[j] = round_bf(s);
          }
        if (nvalid < 8) {                             // ragged tail of the keys (last block only)
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const bool in = j < nvalid;
            sc[G * 4 + (j >> 1)][half * 2 + (j & 1)] = in ? sv[j] : -INFINITY;
            sv[j] = in ? sv[j] : 0.f;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j) sc[G * 4 + (j >> 1)][half * 2 + (j & 1)] = sv[j];
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
          bmax[half] = fmaxf(bmax[half], fmaxf(sc[G * 4 + i][half * 2], sc[G * 4 + i][half * 2 + 1]));
        if (has_sout && row_ok && k0 < lds) store8(sout + soff[half] + k0, lds - k0, vec, sv);
      }
    }
    }
    // ---- online softmax (base-2 exponentials) ----------------------------------------------------
    // (s - max is formed FIRST: on a fully masked row s = max = bf16(-1e8), where folding max*log2e
    // into an FFMA addend would leave its rounding error - up to +-8 - in the exponent)
    float scale[2];
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      const float m_new = fmaxf(m_run[half], quad_max(bmax[half]));
      scale[half] = fast_exp2((m_run[half] - m_new) * LOG2E);    // first block: 2^(-inf) = 0
      m_run[half] = m_new;
      l_run[half] *= scale[half];
    }
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float p = fast_exp2((sc[i][e] - m_run[e >> 1]) * LOG2E);
        sc[i][e] = p;
        l_run[e >> 1] += p;
      }
#pragma unroll
    for (int n = 0; n < HD / 8; ++n) {
      o[n][0] *= scale[0]; o[n][1] *= scale[0];
      o[n][2] *= scale[1]; o[n][3] *= scale[1];
    }
    // ---- O += P V : P from registers (A operand), V via ldmatrix.trans ---------------------------
#pragma unroll
    for (int G = 0; G < 2; ++G) {
      if (kb + 32 * G >= Lk) continue;                 // whole group beyond the keys (warp-uniform)
      const uint32_t vbase = sV + (uint32_t)(kb + 32 * G) * RB;
#pragma unroll
      for (int pp = 0; pp < 2; ++pp) {
        const int i0 = G * 4 + 2 * pp, i1 = i0 + 1;
        uint32_t pa[4] = {pack2(sc[i0][0], sc[i0][1]), pack2(sc[i0][2], sc[i0][3]),
                          pack2(sc[i1][0], sc[i1][1]), pack2(sc[i1][2], sc[i1][3])};
#pragma unroll
        for (int c2 = 0; c2 < HD / 8; c2 += 2) {
          uint32_t vf[4];
          ldsm4t(vbase + lo.t[pp][c2 >> 1], vf);
          mma16816(o[c2], pa, vf[0], vf[1]);
          mma16816(o[c2 + 1], pa, vf[2], vf[3]);
        }
      }
    }
  }
  // ---- epilogue: normalise, write O (merged-head layout) and the (max, sum) pair ----------------
  const float lA = quad_sum(l_run[0]), lB = quad_sum(l_run[1]);
  const float iA = 1.f / lA, iB = 1.f / lB;
  bf16* oA = P.o + ((size_t)b * Lq + rowA) * P.ldo + h * HD + 2 * t;
  bf16* oB = oA + (size_t)8 * P.ldo;
#pragma unroll
  for (int n = 0; n < HD / 8; ++n) {
    if (okA) *reinterpret_cast<uint32_t*>(oA + 8 * n) = pack2(o[n][0] * iA, o[n][1] * iA);
    if (okB) *reinterpret_cast<uint32_t*>(oB + 8 * n) = pack2(o[n][2] * iB, o[n][3] * iB);
  }
  if (t == 0 && P.lse) {
    if (okA) { P.lse[2 * (sbase + rowA)] = m_run[0]; P.lse[2 * (sbase + rowA) + 1] = lA; }
    if (okB) { P.lse[2 * (sbase + rowB)] = m_run[1]; P.lse[2 * (sbase + rowB) + 1] = lB; }
  }
}

// =============================================================================================
// backward
// =============================================================================================
// (no register cap: forcing three 6-warp CTAs per SM (<= 96 registers) spilled and measured 8 %
// slower on Ren-MME's shapes than two CTAs at 121 registers)
// PLAIN = scores recomputed, no previous scores, no score gradients in or out (the backward of the
// PLAIN forward): unrounded scores, +inf mask entries for the key padding, no per-element selects
// and none of the global score-tensor code.
// DQREG: every warp owns at most three 16-row tiles (Lq <= 384 with the CTA sizing below) and
// keeps their dQ accumulators in registers across the key blocks instead of a read-modify-write
// fp32 tile in shared memory: 18 KB less per CTA at Lq = 275 (87 -> 69 KB: three CTAs per SM).
template <int HD, int KB, int MODE, bool DQREG>
__global__ void __launch_bounds__(BWD_WARPS * 32)
resattn_mma_bwd_kernel(const __grid_constant__ Table T) {
  constexpr bool PLAIN = MODE == M_PLAIN, SPEC = MODE >= M_FIRST;
  constexpr int MAXR = DQREG ? 3 : 1;
  const int NT = blockDim.x, nwarps = blockDim.x >> 5;   // 2..8 warps, chosen per launch (host)
  constexpr int NG = KB / 32;              // 32-key groups per block
  extern __shared__ __align__(128) uint8_t smem[];
  int local;
  const Prob& P = locate(T, local);
  const int Lq = P.Lq, Lk = P.Lk, H = P.H;
  const int h = local % H, b = local / H;
  const int LqP = (Lq + 15) & ~15, LkP = (Lk + KB - 1) / KB * KB;
  const bool same_kv = (P.k == P.v) && (P.ldk == P.ldv);
  const bool kv_blocked = T.kv_blocked != 0;
  const int kv_rows = kv_blocked ? KB : LkP;       // rows of the K / V tiles in shared memory
  // carve-up: Q | dO | K | (V) | P | dS | dQ(fp32) | stat(m, 1/l, D) | bias
  uint32_t off = 0;
  const uint32_t sQ = s_u32(smem) + off;   off += LqP * HD * 2;
  const uint32_t sdO = s_u32(smem) + off;  off += LqP * HD * 2;
  const uint32_t sK = s_u32(smem) + off;   off += kv_rows * HD * 2;
  uint32_t sV = sK;
  if (!same_kv) { sV = s_u32(smem) + off;  off += kv_rows * HD * 2; }
  const uint32_t sP = s_u32(smem) + off;   off += LqP * KB * 2;
  const uint32_t sdS = s_u32(smem) + off;  off += LqP * KB * 2;
  float* sdQ = reinterpret_cast<float*>(smem + off);    off += DQREG ? 0 : LqP * HD * 4;
  float* sstat = reinterpret_cast<float*>(smem + off);  off += LqP * 3 * 4;
  float* sbias = reinterpret_cast<float*>(smem + off);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;

  pdl_wait();
  pdl_trigger();
  stage<HD>(sQ, P.q + (size_t)b * Lq * P.ldq + h * HD, P.ldq, Lq, LqP);
  stage<HD>(sdO, P.d_o + (size_t)b * Lq * P.lddo + h * HD, P.lddo, Lq, LqP);
  if (!kv_blocked) {
    stage<HD>(sK, P.k + (size_t)b * Lk * P.ldk + h * HD, P.ldk, Lk, LkP);
    if (!same_kv) stage<HD>(sV, P.v + (size_t)b * Lk * P.ldv + h * HD, P.ldv, Lk, LkP);
  }
  for (int j = threadIdx.x; j < LkP; j += NT) {
    float bias = (P.mask && j < Lk) ? 1.0e8f * (1.0f - P.mask[(size_t)b * P.mask_bs + j]) : 0.f;
    if (PLAIN && j >= Lk) bias = INFINITY;   // padded keys: s = -inf, p = 0, dS = 0
    sbias[j] = bias;
  }
  if (!DQREG)
    for (int i = threadIdx.x; i < LqP * HD; i += NT) sdQ[i] = 0.f;
  const size_t sbase = ((size_t)b * H + h) * Lq;
  // per-row statistics: max, log2(sum) (saved by the forward), D = rowsum(dO * O)
  for (int r = threadIdx.x; r < LqP; r += NT) {
    float mx = 0.f, inv = 0.f, D = 0.f;
    if (r < Lq) {
      mx = P.lse[2 * (sbase + r)];
      inv = log2f(P.lse[2 * (sbase + r) + 1]);      // P = 2^((s - max) log2e - log2(sum))
      const bf16* dop = P.d_o + ((size_t)b * Lq + r) * P.lddo + h * HD;
      const bf16* op = P.o_in + ((size_t)b * Lq + r) * P.ldo + h * HD;
#pragma unroll
      for (int c8 = 0; c8 < HD / 8; ++c8) {
        const uint4 a = *reinterpret_cast<const uint4*>(dop + c8 * 8);
        const uint4 o4 = *reinterpret_cast<const uint4*>(op + c8 * 8);
        const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, ow[4] = {o4.x, o4.y, o4.z, o4.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
          D = fmaf(bf_lo(aw[i]), bf_lo(ow[i]), fmaf(bf_hi(aw[i]), bf_hi(ow[i]), D));
      }
    }
    sstat[3 * r] = mx; sstat[3 * r + 1] = inv; sstat[3 * r + 2] = D;
  }
  cp_commit_wait();
  __syncthreads();

  const bool has_mask = P.mask != nullptr;
  const bool has_prev = SPEC ? (MODE != M_FIRST) : (!PLAIN && P.s_prev != nullptr);
  const bool recompute = SPEC ? (MODE == M_LAST) : (PLAIN || P.s == nullptr);
  const bool has_next = SPEC ? (MODE != M_LAST) : (!PLAIN && P.ds_next != nullptr);
  const bool has_dsp = SPEC ? (MODE != M_FIRST) : (!PLAIN && P.ds_prev != nullptr);
  const float cval = (has_prev && P.c) ? P.c[0] : 0.f;
  const float inv_sqrt = T.inv_sqrt;
  const bool vec = SPEC ? true : P.vec_s != 0;
  const int lds = P.lds;
  const int n_rt = LqP / 16;
  const bf16* __restrict__ gs = P.s;
  const bf16* __restrict__ gprev = P.s_prev;
  const bf16* __restrict__ gnext = P.ds_next;
  bf16* __restrict__ gdsp = P.ds_prev;
  constexpr uint32_t RB = HD * 2;
  LaneOffs<HD> lo;
  lo.init(lane);
  // shared-memory offsets of this lane's P / dS chunks: row 16*rt + g (+8), chunk 4*G + t
  uint32_t pofs[NG][2];
#pragma unroll
  for (int G = 0; G < NG; ++G) {
    pofs[G][0] = swp<KB>(g, 4 * G + t);
    pofs[G][1] = swp<KB>(g + 8, 4 * G + t);
  }
  float dc_part = 0.f;
  float dqa[MAXR][HD / 8][4];                        // DQREG: dQ of this warp's row tiles
#pragma unroll
  for (int ri = 0; ri < MAXR; ++ri)
#pragma unroll
    for (int n = 0; n < HD / 8; ++n)
#pragma unroll
      for (int e = 0; e < 4; ++e) dqa[ri][n][e] = 0.f;

  for (int kb = 0; kb < Lk; kb += KB) {
    const int kofs = kv_blocked ? kb : 0;            // first key held in the K / V tiles
    if (kv_blocked) {       // (the previous block's readers passed the barrier ending the loop body)
      stage<HD>(sK, P.k + ((size_t)b * Lk + kb) * P.ldk + h * HD, P.ldk, min(KB, Lk - kb), KB);
      if (!same_kv)
        stage<HD>(sV, P.v + ((size_t)b * Lk + kb) * P.ldv + h * HD, P.ldv, min(KB, Lk - kb), KB);
      cp_commit_wait();
      __syncthreads();
    }
    // ================= phase A: one warp per 16-row tile ========================================
    // (DQREG: tile ri of this warp, statically indexed accumulators; else the plain tile loop)
#pragma unroll
    for (int ri = 0; ri < MAXR; ++ri)
    for (int rt = warp + ri * nwarps; rt < n_rt; rt += (DQREG ? n_rt : nwarps)) {
      const int rowA = rt * 16 + g, rowB = rowA + 8;
      const bool ok[2] = {rowA < Lq, rowB < Lq};
      const size_t soff[2] = {(sbase + (ok[0] ? rowA : 0)) * lds, (sbase + (ok[1] ? rowB : 0)) * lds};
      const float st_mx[2] = {sstat[3 * rowA], sstat[3 * rowB]};
      const float st_l2[2] = {sstat[3 * rowA + 1], sstat[3 * rowB + 1]};
      const float st_D[2] = {sstat[3 * rowA + 2], sstat[3 * rowB + 2]};
      const uint32_t abase = (uint32_t)(rt * 16) * RB;
      uint32_t doa[HD / 16][4];
#pragma unroll
      for (int kt = 0; kt < HD / 16; ++kt) ldsm4(sdO + abase + lo.a[kt], doa[kt]);
      float sc[NG * 4][4], dp[NG * 4][4];
#pragma unroll
      for (int i = 0; i < NG * 4; ++i)
#pragma unroll
        for (int e = 0; e < 4; ++e) { sc[i][e] = 0.f; dp[i][e] = 0.f; }
      if (recompute) {
        uint32_t qa[HD / 16][4];
#pragma unroll
        for (int kt = 0; kt < HD / 16; ++kt) ldsm4(sQ + abase + lo.a[kt], qa[kt]);
#pragma unroll
        for (int G = 0; G < NG; ++G) {
          const uint32_t kbase = sK + (uint32_t)(kb - kofs + 32 * G) * RB;
#pragma unroll
          for (int ip = 0; ip < 2; ++ip)
#pragma unroll
            for (int kt = 0; kt < HD / 16; ++kt) {
              uint32_t kf[4];
              ldsm4(kbase + lo.n[ip][kt], kf);
              mma16816(sc[G * 4 + ip * 2], qa[kt], kf[0], kf[1]);
              mma16816(sc[G * 4 + ip * 2 + 1], qa[kt], kf[2], kf[3]);
            }
        }
      }
      // dP = dO V^T
#pragma unroll
      for (int G = 0; G < NG; ++G) {
        const uint32_t vbase = sV + (uint32_t)(kb - kofs + 32 * G) * RB;
#pragma unroll
        for (int ip = 0; ip < 2; ++ip)
#pragma unroll
          for (int kt = 0; kt < HD / 16; ++kt) {
            uint32_t vf[4];
            ldsm4(vbase + lo.n[ip][kt], vf);
            mma16816(dp[G * 4 + ip * 2], doa[kt], vf[0], vf[1]);
            mma16816(dp[G * 4 + ip * 2 + 1], doa[kt], vf[2], vf[3]);
          }
      }
      // elementwise: P, dS, dc, dS_prev; P / dS -> shared memory (bf16, natural key order)
      if constexpr (PLAIN) {
        // rows >= Lq carry zero Q / dO rows and zero statistics, keys >= Lk a +inf mask entry and
        // zero K / V rows: their P / dS come out as finite values times zero operands or exact
        // zeros, so no element needs a guard
#pragma unroll
        for (int G = 0; G < NG; ++G) {
          const float* bp = sbias + kb + 32 * G + 8 * t;
          const float4 b0 = *reinterpret_cast<const float4*>(bp);
          const float4 b1 = *reinterpret_cast<const float4*>(bp + 4);
          const float bias[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            const float mx = st_mx[half], l2 = st_l2[half], D = st_D[half];
            float pb[8], dsb[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int i = G * 4 + (j >> 1), e = half * 2 + (j & 1);
              const float sx = __fsub_rn(__fmul_rn(sc[i][e], inv_sqrt), bias[j]);
              const float pj = fast_exp2(fmaf(sx - mx, LOG2E, -l2));
              pb[j] = pj;
              dsb[j] = pj * (dp[i][e] - D);
              sc[i][e] = dsb[j];                         // A operand of dQ += dS K
            }
            const uint32_t rb = (uint32_t)(rt * 16) * (KB * 2) + pofs[G][half];
            asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(sP + rb),
                         "r"(pack2(pb[0], pb[1])), "r"(pack2(pb[2], pb[3])),
                         "r"(pack2(pb[4], pb[5])), "r"(pack2(pb[6], pb[7])) : "memory");
            asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(sdS + rb),
                         "r"(pack2(dsb[0], dsb[1])), "r"(pack2(dsb[2], dsb[3])),
                         "r"(pack2(dsb[4], dsb[5])), "r"(pack2(dsb[6], dsb[7])) : "memory");
          }
        }
      } else {
#pragma unroll
      for (int G = 0; G < NG; ++G) {
        const int k0 = kb + 32 * G + 8 * t;
        const int nvalid = Lk - k0;                    // >= 8: the whole chunk is inside the keys
        float bias[8];
        if (recompute && has_mask) {
          const float4 b0 = *reinterpret_cast<const float4*>(sbias + k0);
          const float4 b1 = *reinterpret_cast<const float4*>(sbias + k0 + 4);
          bias[0] = b0.x; bias[1] = b0.y; bias[2] = b0.z; bias[3] = b0.w;
          bias[4] = b1.x; bias[5] = b1.y; bias[6] = b1.z; bias[7] = b1.w;
        }
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          const bool in = ok[half] && nvalid > 0;
          const float mx = st_mx[half], l2 = st_l2[half], D = st_D[half];
          float sv[8], pv[8], nv[8], pb[8], dsb[8];
          if (!recompute && in) load8(gs + soff[half] + k0, lds - k0, vec, sv);
          if (has_prev && in) load8(gprev + soff[half] + k0, lds - k0, vec, pv);
          if (has_next && in) load8(gnext + soff[half] + k0, lds - k0, vec, nv);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float s;
            if (recompute) {
              s = sc[G * 4 + (j >> 1)][half * 2 + (j & 1)] * inv_sqrt;
              if (has_prev) s = __fadd_rn(s, __fmul_rn(cval, pv[j]));
              if (has_mask) s = __fsub_rn(s, bias[j]);
              s = round_bf(s);
            } else {
              s = sv[j];
            }
            const float p = fast_exp2(fmaf(s - mx, LOG2E, -l2));
            float ds = p * (dp[G * 4 + (j >> 1)][half * 2 + (j & 1)] - D);
            if (has_next) ds += nv[j];
            pb[j] = p;
            dsb[j] = ds;
          }
          if (!in || nvalid < 8) {                     // rows beyond Lq / ragged tail of the keys
#pragma unroll
            for (int j = 0; j < 8; ++j)
              if (!in || j >= nvalid) { pb[j] = 0.f; dsb[j] = 0.f; pv[j] = 0.f; }   // (padding may hold anything)
          }
          if (has_prev && in) {
            float o8[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              dc_part = fmaf(dsb[j], pv[j], dc_part);
              o8[j] = cval * dsb[j];
            }
            if (has_dsp) store8(gdsp + soff[half] + k0, lds - k0, vec, o8);
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) sc[G * 4 + (j >> 1)][half * 2 + (j & 1)] = dsb[j];   // A of dQ += dS K
          const uint32_t rb = (uint32_t)(rt * 16) * (KB * 2) + pofs[G][half];
          asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(sP + rb),
                       "r"(pack2(pb[0], pb[1])), "r"(pack2(pb[2], pb[3])), "r"(pack2(pb[4], pb[5])),
                       "r"(pack2(pb[6], pb[7])) : "memory");
          asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(sdS + rb),
                       "r"(pack2(dsb[0], dsb[1])), "r"(pack2(dsb[2], dsb[3])),
                       "r"(pack2(dsb[4], dsb[5])), "r"(pack2(dsb[6], dsb[7])) : "memory");
        }
      }
      }
      // dQ tile += dS K  (A = dS from registers, B = K via ldmatrix.trans), fp32 in shared memory
      float dq_blk[HD / 8][4];
      float (&dq)[HD / 8][4] = DQREG ? dqa[ri] : dq_blk;
      if (!DQREG) {
#pragma unroll
        for (int n = 0; n < HD / 8; ++n)
#pragma unroll
          for (int e = 0; e < 4; ++e) dq_blk[n][e] = 0.f;
      }
#pragma unroll
      for (int G = 0; G < NG; ++G) {
        if (kb + 32 * G >= Lk) continue;
        const uint32_t kbase = sK + (uint32_t)(kb - kofs + 32 * G) * RB;
#pragma unroll
        for (int pp = 0; pp < 2; ++pp) {
          const int i0 = G * 4 + 2 * pp, i1 = i0 + 1;
          uint32_t da[4] = {pack2(sc[i0][0], sc[i0][1]), pack2(sc[i0][2], sc[i0][3]),
                            pack2(sc[i1][0], sc[i1][1]), pack2(sc[i1][2], sc[i1][3])};
#pragma unroll
          for (int c2 = 0; c2 < HD / 8; c2 += 2) {
            uint32_t kf[4];
            ldsm4t(kbase + lo.t[pp][c2 >> 1], kf);
            mma16816(dq[c2], da, kf[0], kf[1]);
            mma16816(dq[c2 + 1], da, kf[2], kf[3]);
          }
        }
      }
      if (!DQREG) {
        float* qA = sdQ + rowA * HD + 2 * t;
#pragma unroll
        for (int n = 0; n < HD / 8; ++n) {
          float2* pa = reinterpret_cast<float2*>(qA + 8 * n);
          float2* pb2 = reinterpret_cast<float2*>(qA + 8 * HD + 8 * n);
          float2 a = *pa, b2 = *pb2;
          a.x += dq[n][0]; a.y += dq[n][1]; b2.x += dq[n][2]; b2.y += dq[n][3];
          *pa = a; *pb2 = b2;
        }
      }
    }
    __syncthreads();
    // ================= phase B: dV = P^T dO, dK = dS^T Q for the KB keys of this block ===========
    // When the caller passes ONE buffer for dk and dv (lite blocks: K = V = the source stream) the
    // two are summed here: a task then owns 16 keys and runs both products into one accumulator.
    const bool fuse_kv = (P.dk == P.dv);
    const int n_tasks = fuse_kv ? (KB / 16) : (KB / 16) * 2;
    for (int task = warp; task < n_tasks; task += nwarps) {
      const int ks = fuse_kv ? task : (task >> 1);
      if (kb + 16 * ks >= Lk) continue;
      float acc[HD / 8][4];
#pragma unroll
      for (int n = 0; n < HD / 8; ++n)
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[n][e] = 0.f;
      // pass 0: dK = dS^T Q (scaled by 1/sqrt(hd)); pass 1: dV = P^T dO
      const int p_beg = fuse_kv ? 0 : ((task & 1) ? 0 : 1), p_end = fuse_kv ? 2 : p_beg + 1;
      for (int pass = p_beg; pass < p_end; ++pass) {
        const uint32_t sA = pass == 0 ? sdS : sP, sB = pass == 0 ? sQ : sdO;
        for (int kt = 0; kt < n_rt; ++kt) {
          const int mi = lane >> 3, r = lane & 7;
          uint32_t af[4];
          ldsm4t(sA + swp<KB>(kt * 16 + r + 8 * (mi >> 1), 2 * ks + (mi & 1)), af);
#pragma unroll
          for (int c2 = 0; c2 < HD / 8; c2 += 2) {
            uint32_t bf[4];
            ldsm4t(sB + sw<HD>(kt * 16 + r + 8 * (mi & 1), c2 + (mi >> 1)), bf);
            mma16816(acc[c2], af, bf[0], bf[1]);
            mma16816(acc[c2 + 1], af, bf[2], bf[3]);
          }
        }
        if (pass == 0) {
#pragma unroll
          for (int n = 0; n < HD / 8; ++n)
#pragma unroll
            for (int e = 0; e < 4; ++e) acc[n][e] *= inv_sqrt;
        }
      }
      const bool is_dk = fuse_kv || (task & 1);
      bf16* out = is_dk ? P.dk : P.dv;
      const int ld = is_dk ? P.lddk : P.lddv;
      const int keyA = kb + 16 * ks + g, keyB = keyA + 8;
#pragma unroll
      for (int n = 0; n < HD / 8; ++n) {
        if (keyA < Lk)
          *reinterpret_cast<uint32_t*>(out + ((size_t)b * Lk + keyA) * ld + h * HD + 8 * n + 2 * t) =
              pack2(acc[n][0], acc[n][1]);
        if (keyB < Lk)
          *reinterpret_cast<uint32_t*>(out + ((size_t)b * Lk + keyB) * ld + h * HD + 8 * n + 2 * t) =
              pack2(acc[n][2], acc[n][3]);
      }
    }
    __syncthreads();
  }
  // ---- dQ: registers (DQREG) or the fp32 tile -> bf16 -----------------------------------------
  if (DQREG) {
#pragma unroll
    for (int ri = 0; ri < MAXR; ++ri) {
      const int rt = warp + ri * nwarps;
      if (rt >= n_rt) continue;
      const int rowA = rt * 16 + g, rowB = rowA + 8;
      bf16* qa_ = P.dq + ((size_t)b * Lq + rowA) * P.lddq + h * HD + 2 * t;
      bf16* qb_ = qa_ + (size_t)8 * P.lddq;
#pragma unroll
      for (int n = 0; n < HD / 8; ++n) {
        if (rowA < Lq)
          *reinterpret_cast<uint32_t*>(qa_ + 8 * n) =
              pack2(dqa[ri][n][0] * inv_sqrt, dqa[ri][n][1] * inv_sqrt);
        if (rowB < Lq)
          *reinterpret_cast<uint32_t*>(qb_ + 8 * n) =
              pack2(dqa[ri][n][2] * inv_sqrt, dqa[ri][n][3] * inv_sqrt);
      }
    }
  }
  for (int i = threadIdx.x; !DQREG && i < Lq * (HD / 8); i += NT) {
    const int r = i / (HD / 8), c8 = i - r * (HD / 8);
    const float* s = sdQ + r * HD + c8 * 8;
    *reinterpret_cast<uint4*>(P.dq + ((size_t)b * Lq + r) * P.lddq + h * HD + c8 * 8) =
        make_uint4(pack2(s[0] * inv_sqrt, s[1] * inv_sqrt), pack2(s[2] * inv_sqrt, s[3] * inv_sqrt),
                   pack2(s[4] * inv_sqrt, s[5] * inv_sqrt), pack2(s[6] * inv_sqrt, s[7] * inv_sqrt));
  }
  // ---- dc -------------------------------------------------------------------------------------
  if (P.dc && has_prev) {
    __shared__ float red[BWD_WARPS];
    dc_part = warp_sum(dc_part);
    if (lane == 0) red[warp] = dc_part;
    __syncthreads();
    if (threadIdx.x == 0) {
      float s = 0.f;
      for (int w = 0; w < nwarps; ++w) s += red[w];
      atomicAdd(P.dc, s);
    }
  }
}

// ---- host side --------------------------------------------------------------------------------
inline bool a16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

size_t fwd_smem(int hd, int Lk, bool same_kv) {
  const int LkP = (Lk + 63) & ~63;
  return (size_t)FWD_ROWS * hd * 2 + (size_t)(same_kv ? 1 : 2) * LkP * hd * 2 + (size_t)LkP * 4;
}
size_t bwd_smem(int hd, int kbk, int Lq, int Lk, bool same_kv, bool kv_blocked = false,
                bool dqreg = false) {
  const int LqP = (Lq + 15) & ~15, LkP = (Lk + kbk - 1) / kbk * kbk;
  const int kv_rows = kv_blocked ? kbk : LkP;
  return (size_t)2 * LqP * hd * 2 + (size_t)(same_kv ? 1 : 2) * kv_rows * hd * 2 +
         (size_t)2 * LqP * kbk * 2 + (dqreg ? 0 : (size_t)LqP * hd * 4) + (size_t)LqP * 12 +
         (size_t)LkP * 4;
}

bool operands_ok(const mmemo_attn_problem& a, bool bwd) {
  if (a.hd != 16 && a.hd != 32 && a.hd != 64) return false;
  if (a.B <= 0 || a.H <= 0 || a.Lq <= 0 || a.Lk <= 0) return false;
  if (a.Lq > 4096 || a.Lk > 4096) return false;
  if (!a.q || !a.k || !a.v || !a.o || !a.lse) return false;
  if (!a16(a.q) || !a16(a.k) || !a16(a.v) || a.ldq % 8 || a.ldk % 8 || a.ldv % 8 || a.ldo % 2 ||
      (reinterpret_cast<uintptr_t>(a.o) & 3))
    return false;
  if (a.lds < a.Lk) return false;
  if (bwd) {
    if (!a.d_o || !a.dq || !a.dk || !a.dv) return false;
    if (!a16(a.d_o) || !a16(a.o) || !a16(a.dq) || a.lddo % 8 || a.ldo % 8 || a.lddq % 8 ||
        a.lddk % 2 || a.lddv % 2 || (reinterpret_cast<uintptr_t>(a.dk) & 3) ||
        (reinterpret_cast<uintptr_t>(a.dv) & 3))
      return false;
  }
  return true;
}

void fill(Prob& p, const mmemo_attn_problem& a) {
  p.q = static_cast<const bf16*>(a.q); p.k = static_cast<const bf16*>(a.k);
  p.v = static_cast<const bf16*>(a.v); p.mask = a.mask;
  p.s_prev = static_cast<const bf16*>(a.s_prev); p.c = a.c;
  p.s_out = static_cast<bf16*>(a.s_out); p.o = static_cast<bf16*>(a.o); p.lse = a.lse;
  p.d_o = static_cast<const bf16*>(a.d_o); p.s = static_cast<const bf16*>(a.s);
  p.ds_next = static_cast<const bf16*>(a.ds_next); p.o_in = static_cast<const bf16*>(a.o);
  p.dq = static_cast<bf16*>(a.dq); p.dk = static_cast<bf16*>(a.dk); p.dv = static_cast<bf16*>(a.dv);
  p.ds_prev = static_cast<bf16*>(a.ds_prev); p.dc = a.dc;
  p.ldq = (int)a.ldq; p.ldk = (int)a.ldk; p.ldv = (int)a.ldv; p.ldo = (int)a.ldo;
  p.lds = (int)a.lds; p.lddo = (int)a.lddo; p.lddq = (int)a.lddq; p.lddk = (int)a.lddk;
  p.lddv = (int)a.lddv; p.mask_bs = (int)a.mask_bs;
  p.B = (int)a.B; p.H = (int)a.H; p.Lq = (int)a.Lq; p.Lk = (int)a.Lk;
  const void* sp[5] = {a.s_prev, a.s_out, a.s, a.ds_next, a.ds_prev};
  bool v = a.lds % 8 == 0;
  for (const void* x : sp) v = v && (!x || a16(x));
  p.vec_s = v ? 1 : 0;
}

}  // namespace

bool resattn_mma_supported(const mmemo_attn_problem& a, bool bwd) {
  if (!operands_ok(a, bwd)) return false;
  const bool same = a.k == a.v && a.ldk == a.ldv;
  if (!bwd) return fwd_smem((int)a.hd, (int)a.Lk, same) <= SMEM_MAX;
  return bwd_smem((int)a.hd, 32, (int)a.Lq, (int)a.Lk, same, true) <= SMEM_MAX;
}

namespace {
bool vec_ok(const mmemo_attn_problem& p) {
  auto al = [](const void* x) { return (reinterpret_cast<uintptr_t>(x) & 15) == 0; };
  return p.lds % 8 == 0 && al(p.s_prev) && al(p.s_out) && al(p.s) && al(p.ds_next) && al(p.ds_prev);
}
int fwd_mode(const mmemo_attn_problem& p) {
  if (getenv("MMEMO_ATTN_GENERIC")) return M_GEN;          // A/B switch (tools/prof_attn.py)
  if (!p.s_prev && !p.s_out) return M_PLAIN;
  if (!vec_ok(p)) return M_GEN;
  return p.s_prev ? (p.s_out ? M_MID : M_LAST) : M_FIRST;
}
int bwd_mode(const mmemo_attn_problem& p) {
  if (getenv("MMEMO_ATTN_GENERIC")) return M_GEN;
  if (!p.s && !p.s_prev && !p.ds_next && !p.ds_prev) return M_PLAIN;
  if (!vec_ok(p)) return M_GEN;
  if (p.s && !p.s_prev && p.ds_next && !p.ds_prev) return M_FIRST;
  if (p.s && p.s_prev && p.ds_next && p.ds_prev) return M_MID;
  if (!p.s && p.s_prev && !p.ds_next && p.ds_prev) return M_LAST;
  return M_GEN;
}

// Heaviest problems first: CTAs are dispatched in index order, so the long-sequence CTAs (Ren-MME:
// 275 x 275 scores against 40 x 40) start while the machine is full and the short ones fill the
// tail, instead of a last wave made of the slowest CTAs only.
void heavy_first(const mmemo_attn_problem* ps, int n, int* idx) {
  for (int i = 0; i < n; ++i) idx[i] = i;
  for (int i = 1; i < n; ++i) {          // stable insertion sort (n <= MAXP)
    const int v = idx[i];
    const int64_t w = ps[v].Lq * ps[v].Lk;
    int j = i - 1;
    while (j >= 0 && ps[idx[j]].Lq * ps[idx[j]].Lk < w) { idx[j + 1] = idx[j]; --j; }
    idx[j + 1] = v;
  }
}

// the problems of `ps` that run in `mode`, as one launch of that instantiation
int fwd_launch(const mmemo_attn_problem* ps, int n, int mode, cudaStream_t st) {
  static thread_local Table T;      // host staging (copied by value into the launch)
  const int hd = (int)ps[0].hd;
  size_t smem = 0;
  int ctas = 0, m = 0;
  int order[MAXP];
  heavy_first(ps, n, order);
  for (int oi = 0; oi < n; ++oi) {
    const int i = order[oi];
    if (fwd_mode(ps[i]) != mode) continue;
    fill(T.p[m], ps[i]);
    T.p[m].cta_start = ctas;
    T.cta_start[m] = ctas;
    ctas += (int)(ps[i].B * ps[i].H * cdiv(ps[i].Lq, FWD_ROWS));
    const size_t s = fwd_smem(hd, (int)ps[i].Lk, ps[i].k == ps[i].v && ps[i].ldk == ps[i].ldv);
    smem = s > smem ? s : smem;
    ++m;
  }
  if (m == 0) return MMEMO_OK;
  T.n = m;
  T.total = ctas;
  T.cta_start[m] = ctas;
  T.inv_sqrt = (float)(1.0 / sqrt((double)hd));
#define MM_FWD1(HD, MD)                                                                          \
  {                                                                                              \
    MM_CUDA_OK(cudaFuncSetAttribute(resattn_mma_fwd_kernel<HD, MD>,                              \
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));    \
    MM_CUDA_OK(mm_launch(resattn_mma_fwd_kernel<HD, MD>, dim3((unsigned)ctas),                   \
                         dim3(FWD_WARPS * 32), smem, st, T));                                    \
  }
#define MM_FWD(HD)                                                                               \
  {                                                                                              \
    if (mode == M_PLAIN) MM_FWD1(HD, M_PLAIN)                                                    \
    else if (mode == M_FIRST) MM_FWD1(HD, M_FIRST)                                               \
    else if (mode == M_MID) MM_FWD1(HD, M_MID)                                                   \
    else if (mode == M_LAST) MM_FWD1(HD, M_LAST)                                                 \
    else MM_FWD1(HD, M_GEN)                                                                      \
  }
  if (hd == 16) MM_FWD(16) else if (hd == 32) MM_FWD(32) else MM_FWD(64)
#undef MM_FWD
#undef MM_FWD1
  return MMEMO_OK;
}
}  // namespace

int resattn_mma_fwd(const mmemo_attn_problem* ps, int n, cudaStream_t st) {
  if (n < 1) return MMEMO_ERR_ARG;
  const int hd = (int)ps[0].hd;
  for (int i = 0; i < n; ++i)         // every problem is checked before the first launch
    if (ps[i].hd != hd || !resattn_mma_supported(ps[i], false)) return MMEMO_ERR_SHAPE;
  // chunks of MAXP problems; per chunk one launch per instantiation present (the problems of a
  // trunk layer share their flags: one)
  for (int c0 = 0; c0 < n; c0 += MAXP) {
    const int m = n - c0 < MAXP ? n - c0 : MAXP;
    for (int mode = M_GEN; mode <= M_LAST; ++mode) {
      const int rc = fwd_launch(ps + c0, m, mode, st);
      if (rc) return rc;
    }
  }
  return MMEMO_OK;
}

namespace {
// Warps per backward CTA: phase A hands one 16-row tile to a warp per round, so the CTA is sized
// to the number of tiles split evenly over the rounds (18 tiles -> 3 rounds of 6 warps instead of
// 8 + 8 + 2 on eight; 4 tiles -> 4 warps, twice as many CTAs per SM) - idle warps only add
// barrier stalls (ncu: 7 of 10 issue slots stalled on the barrier with 4 of 8 warps working).
int bwd_warps(int64_t Lq) {
  const int n_rt = (int)cdiv(Lq, 16);
  const int rounds = (int)cdiv(n_rt, BWD_WARPS);
  int w = (int)cdiv(n_rt, rounds);
  return w < 2 ? 2 : w;
}

int bwd_launch(const mmemo_attn_problem* const* ps, int n, int warps, int mode, cudaStream_t st) {
  static thread_local Table T;
  T.n = n;
  const int hd = (int)ps[0]->hd;
  size_t smem64 = 0, smem32 = 0, full32 = 0;
  int ctas = 0;
  for (int i = 0; i < n; ++i) {
    fill(T.p[i], *ps[i]);
    T.p[i].cta_start = ctas;
    T.cta_start[i] = ctas;
    ctas += (int)(ps[i]->B * ps[i]->H);
    const bool same = ps[i]->k == ps[i]->v && ps[i]->ldk == ps[i]->ldv;
    const size_t f32_ = bwd_smem(hd, 32, (int)ps[i]->Lq, (int)ps[i]->Lk, same, false);
    full32 = f32_ > full32 ? f32_ : full32;
  }
  // K and V whole in shared memory when that fits (one load per CTA); otherwise one key block at
  // a time (hd = 64 with L = 256: 64 KB of K, V would not fit next to Q, dO, P, dS and the dQ tile)
  const bool blocked = full32 > SMEM_MAX;
  T.kv_blocked = blocked ? 1 : 0;
  for (int i = 0; i < n; ++i) {
    const bool same = ps[i]->k == ps[i]->v && ps[i]->ldk == ps[i]->ldv;
    const size_t s64 = bwd_smem(hd, 64, (int)ps[i]->Lq, (int)ps[i]->Lk, same, blocked);
    const size_t s32 = bwd_smem(hd, 32, (int)ps[i]->Lq, (int)ps[i]->Lk, same, blocked);
    smem64 = s64 > smem64 ? s64 : smem64;
    smem32 = s32 > smem32 ? s32 : smem32;
  }
  T.total = ctas;
  T.cta_start[n] = ctas;
  T.inv_sqrt = (float)(1.0 / sqrt((double)hd));
  // Key block: the 64-key instantiation needs ~155 registers, the 32-key one ~110: prefer 32
  // whenever two or more CTAs fit (measured 2x faster on cfg 1a and cfg 4), 64 when only one CTA
  // fits either way (fewer block iterations), 32 when 64 does not fit at all.
  // MMEMO_ATTN_KB=32|64 overrides (experiments).
  bool kb64 = smem32 > 110 * 1024 && smem64 <= SMEM_MAX;
  if (const char* e = getenv("MMEMO_ATTN_KB")) {
    if (e[0] == '6' && smem64 <= SMEM_MAX) kb64 = true;
    if (e[0] == '3') kb64 = false;
  }
  // dQ in registers: hd = 16 (8 registers per tile), 32-key blocks, <= 3 row tiles per warp
  // (only where the fp32 tile costs a resident CTA: the register version needs ~30 more registers)
  bool dqreg = hd == 16 && !kb64 && !blocked && smem32 > 70 * 1024 && !getenv("MMEMO_ATTN_DQSMEM");
  for (int i = 0; i < n && dqreg; ++i) dqreg = cdiv(cdiv(ps[i]->Lq, 16), warps) <= 3;
  if (dqreg) {
    smem32 = 0;
    for (int i = 0; i < n; ++i) {
      const bool same = ps[i]->k == ps[i]->v && ps[i]->ldk == ps[i]->ldv;
      const size_t s32 = bwd_smem(hd, 32, (int)ps[i]->Lq, (int)ps[i]->Lk, same, false, true);
      smem32 = s32 > smem32 ? s32 : smem32;
    }
  }
#define MM_BWD2(HD, KBK, PL, DQ, SM)                                                              \
  {                                                                                               \
    MM_CUDA_OK(cudaFuncSetAttribute(resattn_mma_bwd_kernel<HD, KBK, PL, DQ>,                      \
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(SM)));     \
    MM_CUDA_OK(mm_launch(resattn_mma_bwd_kernel<HD, KBK, PL, DQ>, dim3((unsigned)ctas),           \
                         dim3((unsigned)(warps * 32)), SM, st, T));                               \
  }
#define MM_BWD1(HD, KBK, PL, SM)                                                                  \
  {                                                                                               \
    if (HD == 16 && KBK == 32 && dqreg) MM_BWD2(16, 32, PL, true, SM)                             \
    else MM_BWD2(HD, KBK, PL, false, SM)                                                          \
  }
#define MM_BWD(HD, KBK, SM)                                                                       \
  {                                                                                               \
    if (mode == M_PLAIN) MM_BWD1(HD, KBK, M_PLAIN, SM)                                            \
    else if (mode == M_FIRST) MM_BWD1(HD, KBK, M_FIRST, SM)                                       \
    else if (mode == M_MID) MM_BWD1(HD, KBK, M_MID, SM)                                           \
    else if (mode == M_LAST) MM_BWD1(HD, KBK, M_LAST, SM)                                         \
    else MM_BWD1(HD, KBK, M_GEN, SM)                                                              \
  }
  if (kb64) {
    if (hd == 16) MM_BWD(16, 64, smem64) else if (hd == 32) MM_BWD(32, 64, smem64)
    else MM_BWD(64, 64, smem64)
  } else {
    if (hd == 16) MM_BWD(16, 32, smem32) else if (hd == 32) MM_BWD(32, 32, smem32)
    else MM_BWD(64, 32, smem32)
  }
#undef MM_BWD
#undef MM_BWD1
#undef MM_BWD2
  return MMEMO_OK;
}
}  // namespace

namespace {
int bwd_chunk(const mmemo_attn_problem* ps, int n, cudaStream_t st) {
  int fixed = 0;
  if (const char* e = getenv("MMEMO_ATTN_WARPS")) fixed = atoi(e);      // experiments
  // one launch per (CTA size, instantiation): all chains of realformer / robot_demo share one;
  // Ren-MME's three query lengths give three
  const mmemo_attn_problem* sel[MAXP];
  bool done[MAXP] = {};
  int order[MAXP];
  heavy_first(ps, n, order);             // launches and the problems inside them, heaviest first
  for (int oi = 0; oi < n; ++oi) {
    const int i = order[oi];
    if (done[i]) continue;
    const int w = (fixed >= 2 && fixed <= BWD_WARPS) ? fixed : bwd_warps(ps[i].Lq);
    const int mode = bwd_mode(ps[i]);
    int m = 0;
    for (int oj = oi; oj < n; ++oj) {
      const int j = order[oj];
      const int wj = (fixed >= 2 && fixed <= BWD_WARPS) ? fixed : bwd_warps(ps[j].Lq);
      if (!done[j] && wj == w && bwd_mode(ps[j]) == mode) { sel[m++] = &ps[j]; done[j] = true; }
    }
    const int rc = bwd_launch(sel, m, w, mode, st);
    if (rc) return rc;
  }
  return MMEMO_OK;
}
}  // namespace

int resattn_mma_bwd(const mmemo_attn_problem* ps, int n, cudaStream_t st) {
  if (n < 1) return MMEMO_ERR_ARG;
  const int hd = (int)ps[0].hd;
  for (int i = 0; i < n; ++i)         // every problem is checked before the first launch
    if (ps[i].hd != hd || !resattn_mma_supported(ps[i], true)) return MMEMO_ERR_SHAPE;
  for (int c0 = 0; c0 < n; c0 += MAXP) {          // chunks of MAXP problems
    const int rc = bwd_chunk(ps + c0, n - c0 < MAXP ? n - c0 : MAXP, st);
    if (rc) return rc;
  }
  return MMEMO_OK;
}
