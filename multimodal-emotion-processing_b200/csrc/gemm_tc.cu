// Persistent tcgen05 / TMA GEMM for sm_100a:  C[M,N] (+)= epi( A * B^T ), bf16 operands, fp32
// accumulation in TMEM.  Two configurations of one kernel template:
//
//   CTA2 = true  (default when N >= 256): CTA PAIRS (cluster of 2, cta_group::2).  A pair owns a
//       256 x 256 output tile: each CTA stages its own 128 rows of A and its own 128 columns of B
//       (32 KB per k-block per CTA), the leader CTA issues tcgen05.mma.cta_group::2 (M = 256,
//       N = 256) that reads both CTAs' shared memory, and each CTA's TMEM receives its 128 x 256
//       half of the accumulator.  Bytes staged per flop are half those of a 128 x 128 tile — the
//       128 x 128 version was L2-bandwidth-bound (profiles/).
//   CTA2 = false: one CTA per 128 x 128 tile (small N, and the ragged shapes).
//   LITE (CTA2 = false only): the same kernel with a 2-stage ring and one 32 KB bf16 staging tile
//       (98 KB, 256 TMEM columns): TWO CTAs per SM.  The small-K grouped launches of the d <= 192
//       models are bound by the epilogue's dependent chain (TMEM load -> math -> st.shared ->
//       fence -> barrier -> TMA store, ncu: 3/4 of the stall samples) with the loads idle; a
//       second resident CTA runs its loads / MMAs / epilogue in the gaps of the first.
//
//   warp 0   TMA producer : cp.async.bulk.tensor (SWIZZLE_128B) into a 5-stage shared-memory ring
//   warp 1   MMA issuer   : one thread (of the leader CTA) issues the UMMAs into one of TWO TMEM
//                           accumulators; tcgen05.commit frees ring slots (in both CTAs) and hands
//                           the finished accumulator to the epilogue warps (of both CTAs)
//   warps 2-5 epilogue    : tcgen05.ld (thread = row) -> bias / position table / ReLU / ReLU-mask /
//                           accumulate -> bf16 or fp32 tile in swizzled shared memory -> TMA store,
//                           128 columns at a time, overlapped with the MMAs of the next tile.
// All global traffic goes through TMA: operands, the optional "aux" tile (old C for accumulate, or
// the saved activation whose sign masks a ReLU gradient; prefetched one step ahead) and the output.
// Operand "majors" are encoded in the UMMA descriptors, so y = x w^T (K-major A, B), dx = dy w
// (B MN-major) and dw = dy^T x (A and B MN-major) run without transposes in HBM.
// Split-K (weight gradients: tiny output, K = B*L rows): fp32 slices are summed into C by TMA
// reduce-add (C zero-filled here unless the caller says it already is); bf16 outputs use a
// caller-provided workspace + a fixed-order reduce kernel.
// Grouped launches: up to MAXG independent problems (own tensor maps and epilogue flags) share one
// persistent grid; work items are numbered problem by problem.  The kernel is launched with
// programmatic stream serialization: its prologue runs while the previous kernel drains
// (griddepcontrol.wait before the first global access).
#include <stdlib.h>

#include "common.cuh"
#include "dropout.cuh"
#include "gemm.h"
#include "tc_common.cuh"

namespace {

constexpr int BM = 128, BK = 64, STAGES = 5;
constexpr int STAGES_FULL = STAGES;
constexpr uint32_t A_TILE = BM * BK * 2, B_TILE = 128 * BK * 2;   // per CTA per stage: 16 KB + 16 KB
constexpr uint32_t RING = STAGES * (A_TILE + B_TILE);             // 160 KB
constexpr uint32_t OUT_BYTES = 64 * 1024;    // fp32 staging (128x128), or bf16 staging + aux tile
constexpr uint32_t OUT_FULL = OUT_BYTES;
constexpr int NTHREADS = 320;   // TMA warp, MMA warp, two epilogue warpgroups
constexpr uint32_t SMEM_BYTES = RING + OUT_BYTES + 1024 /*align*/ + 256 /*barriers*/ + 512 /*bias*/;
constexpr int LITE_STAGES = 2;
constexpr uint32_t LITE_OUT = 32 * 1024;
constexpr uint32_t SMEM_LITE = LITE_STAGES * (A_TILE + B_TILE) + LITE_OUT + 1024 + 256 + 512;
constexpr int AUX_NONE = 0, AUX_ACC = 1, AUX_RELU = 2;

struct TcArgs {
  int M, N, K;
  int c_bf16;              // output element type of the TMA store (0: fp32)
  const float* bias;
  const float* pos;
  int pos_period, pos_ld;
  int relu, aux;
  int a_mn, b_mn;
  uint32_t idesc;
  int splits, kb_per, kb_total;
  int reduce_add;          // split-K slices are summed into the fp32 C by TMA reduce-add
  int tiles_m, tiles_n;    // in units of the (pair) tile: TM x BN
  uint32_t drop_thr;       // family 3: dropout threshold round(p * 65536) (0: keep all) ...
  float drop_scale;        //   ... and 1 / (1 - p)
  unsigned long long drop_seed;
};

// One launch can serve up to MAXG independent GEMMs ("grouped"): the work items of all problems
// form one list that the persistent CTAs walk, so small GEMMs that would each leave the machine
// half empty (the five weight gradients of a block, the Q and K|V projections) share one wave.
// Two capacities of the same kernel: NG = 6 (the launches of one block: ~3.5 KB of kernel
// parameters) and NG = 48 (the nine chains x five weight gradients of a fusion-trunk layer, both
// towers' projections: ~29 KB, within the 32 764-byte parameter limit of CUDA >= 12.1).
// FAM names the instantiation after the Linear-layer pass it serves (0 fwd, 1 dX, 2 dW), so that
// profiler launch lists can be read per family; FAM 3 is the forward with a dropout between the
// bias and the position table (the training-mode modality projections), the only instantiation
// that carries the mask code.
constexpr int MAXG_SMALL = 6, MAXG = 48;
template <int NG> struct TmapGroup { CUtensorMap a[NG], b[NG], c[NG], aux[NG]; };
template <int NG> struct GroupArgs {
  int n;
  int any_aux;             // some problem of the launch prefetches an aux tile (owns the second 32 KB)
  int streamk;             // 1: item_start counts K-BLOCKS (tiles x kb_total per problem) and every
  int kb_per_unit;         //    unit owns one contiguous range of kb_per_unit of them (see below)
  const unsigned long long* drop_step;   // family 3: device step counter mixed into the seeds
  int item_start[NG + 1];
  TcArgs p[NG];
};

template <bool CTA2, int NG, int FAM, bool LITE = false>
__global__ void __launch_bounds__(NTHREADS, LITE ? 2 : 1)
gemm_tc_kernel(const __grid_constant__ TmapGroup<NG> TMS, const __grid_constant__ GroupArgs<NG> G) {
  static_assert(!(LITE && CTA2), "the two-CTA-per-SM variant is single-CTA tiles only");
  constexpr int STAGES = LITE ? LITE_STAGES : STAGES_FULL;
  constexpr uint32_t RING = STAGES * (A_TILE + B_TILE);
  constexpr uint32_t OUT_BYTES = LITE ? LITE_OUT : OUT_FULL;
  constexpr int BN = CTA2 ? 256 : 128;        // accumulator columns per tile
  constexpr int TM = CTA2 ? 256 : 128;        // output rows per work item (pair or CTA)
  constexpr int NHALF = BN / 128;             // epilogue works on 128 columns at a time
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = tc::smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  const uint32_t sA = base, sB = base + STAGES * A_TILE;
  const uint32_t sOut = base + RING, sAux = sOut + 32 * 1024;
  const uint32_t bars = sOut + OUT_BYTES;
  const uint32_t bar_full = bars, bar_empty = bars + 8 * STAGES;
  const uint32_t bar_accf = bars + 16 * STAGES, bar_acce = bar_accf + 16, bar_aux = bar_acce + 16;
  const uint32_t tmem_slot = bar_aux + 8;
  volatile uint32_t* tmem_slot_ptr =
      reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - raw));
  float* sbias = reinterpret_cast<float*>(smem_raw + (bars + 256 - raw));   // bias of this half tile

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = CTA2 ? tc::cluster_ctarank() : 0u;      // 0 = leader of the pair
  const int unit = CTA2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int units = CTA2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  const int total = G.item_start[G.n];

  // global work item -> (problem, item within the problem).  Every role walks its items in
  // increasing order, so the search resumes from the caller's previous problem (`g` is a cursor
  // the caller keeps): O(1) amortised instead of a scan over up to 48 table entries per tile.
  auto locate = [&](int w, int& g, int& lw) {
    while (g + 1 < G.n && w >= G.item_start[g + 1]) ++g;
    lw = w - G.item_start[g];
  };
  // The work of a unit (CTA or CTA pair) is a sequence of SEGMENTS = (problem, output tile, range
  // of k-blocks); one accumulator pass each.
  //   regular : items (tile, split-K slice) numbered problem by problem; unit u takes items
  //             u, u + units, ...
  //   stream-K: (grouped weight gradients: one or two output tiles per problem, K of very
  //             different lengths, fp32 C summed by TMA reduce-add) the k-blocks of ALL tiles of
  //             all problems form one line, cut into `units` equal ranges; a unit's range covers
  //             the tail of one tile and the head of the next, so every unit gets the same number
  //             of MMAs whatever the tile count and the K of each problem (the host decides when:
  //             gemm_tc_grouped_t).
  struct WorkIter { int pos, end, g; };
  auto iter_init = [&](WorkIter& it) {
    it.g = 0;
    if (G.streamk) {
      it.pos = unit * G.kb_per_unit;
      it.end = min(total, it.pos + G.kb_per_unit);
    } else {
      it.pos = unit;
      it.end = total;
    }
  };
  auto iter_next = [&](WorkIter& it, int& g, int& tile, int& sp, int& kb_beg, int& kb_end) -> bool {
    if (it.pos >= it.end) return false;
    int lw;
    locate(it.pos, it.g, lw);
    g = it.g;
    const TcArgs& a = G.p[g];
    if (G.streamk) {
      tile = lw / a.kb_total;
      kb_beg = lw - tile * a.kb_total;
      kb_end = min(a.kb_total, kb_beg + (it.end - it.pos));
      sp = 0;
      it.pos += kb_end - kb_beg;
    } else {
      if (a.splits == 1) { sp = 0; tile = lw; }          // (no integer division on the common path)
      else { sp = lw % a.splits; tile = lw / a.splits; }
      kb_beg = sp * a.kb_per;
      kb_end = min(a.kb_total, kb_beg + a.kb_per);
      it.pos += units;
    }
    return true;
  };
  auto tile_origin = [&](const TcArgs& a, int tile, int& m0, int& n0) {
    int tm, tn;
    if (a.tiles_n == 1) { tm = tile; tn = 0; }
    else if (a.tiles_n == 2) { tm = tile >> 1; tn = tile & 1; }
    else { tm = tile / a.tiles_n; tn = tile - tm * a.tiles_n; }
    m0 = tm * TM + (int)rank * BM;     // rows owned by this CTA
    n0 = tn * BN;                      // first column of the (pair) tile
  };

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      tc::mbar_init(bar_full + 8 * s, 1);
      tc::mbar_init(bar_empty + 8 * s, 1);
    }
    for (int i = 0; i < 2; ++i) {
      tc::mbar_init(bar_accf + 8 * i, 1);
      tc::mbar_init(bar_acce + 8 * i, CTA2 ? 2 : 1);   // one elected epilogue thread per CTA
    }
    tc::mbar_init(bar_aux, 1);
    tc::fence_barrier_init();
    tc::tma_prefetch_desc(&TMS.a[0]);
    tc::tma_prefetch_desc(&TMS.b[0]);
    tc::tma_prefetch_desc(&TMS.c[0]);
  }
  // The dependents may be scheduled right away; this kernel's own setup (barriers, TMEM, the
  // pair's first cluster barrier) touches no global memory and overlaps the previous kernel's
  // drain.  griddepcontrol.wait comes right before the first global access of each role: the TMA
  // producer (everything the MMA issuer and the epilogue consume derives from its loads) and the
  // epilogue threads (bias / position-table reads, aux loads, stores).
  pdl_trigger();
  if (warp == 1) {
    if (CTA2) { tc::tmem_alloc_2sm(tmem_slot, 2 * BN); tc::tmem_relinquish_2sm(); }
    else      { tc::tmem_alloc(tmem_slot, 2 * BN); tc::tmem_relinquish(); }
  }
  tc::tc_fence_before();
  if (CTA2) tc::cluster_sync(); else __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    // ================= TMA producer (every CTA stages its own rows of A and columns of B) =========
    if (lane == 0) {
      pdl_wait();
      uint32_t it = 0;
      WorkIter wi;
      iter_init(wi);
      int g, tile, sp, kb_beg, kb_end;
      while (iter_next(wi, g, tile, sp, kb_beg, kb_end)) {
        int m0, n0;
        const TcArgs& a = G.p[g];
        const CUtensorMap* tmA = &TMS.a[g];
        const CUtensorMap* tmB = &TMS.b[g];
        tile_origin(a, tile, m0, n0);
        const int nb = n0 + (int)rank * 128;           // this CTA's 128 columns of B
        for (int kb = kb_beg; kb < kb_end; ++kb, ++it) {
          const uint32_t s = it % STAGES, ph = (it / STAGES) & 1;
          tc::mbar_wait(bar_empty + 8 * s, ph ^ 1);
          const uint32_t fb = bar_full + 8 * s;
          if (rank == 0) tc::mbar_expect_tx(fb, (CTA2 ? 2u : 1u) * (A_TILE + B_TILE));
          const int k0 = kb * BK;
          const uint32_t da = sA + s * A_TILE, db = sB + s * B_TILE;
          auto ld = [&](uint32_t dst, const CUtensorMap* tm, int c0, int c1) {
            if (CTA2) tc::tma_load_2d_2sm(dst, tm, c0, c1, fb);   // credits the leader's barrier
            else tc::tma_load_2d(dst, tm, c0, c1, fb);
          };
          if (!a.a_mn) {
            ld(da, tmA, k0, m0);                                 // box {64 k, 128 m}
          } else {
            ld(da, tmA, m0, k0);                                 // box {64 m, 64 k}
            ld(da + A_TILE / 2, tmA, m0 + 64, k0);
          }
          if (!a.b_mn) {
            ld(db, tmB, k0, nb);
          } else {
            ld(db, tmB, nb, k0);
            ld(db + B_TILE / 2, tmB, nb + 64, k0);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer (leader CTA only) =================
    if (lane == 0 && rank == 0) {
      uint32_t it = 0, ti = 0;
      WorkIter wi;
      iter_init(wi);
      int g, tile, sp, kb_beg, kb_end;
      for (; iter_next(wi, g, tile, sp, kb_beg, kb_end); ++ti) {
        const TcArgs& a = G.p[g];
        const uint32_t buf = ti & 1, aph = (ti >> 1) & 1;
        tc::mbar_wait(bar_acce + 8 * buf, aph ^ 1);     // epilogues have drained this accumulator
        tc::tc_fence_after();
        const uint32_t tacc = tmem_base + buf * BN;
        for (int kb = kb_beg; kb < kb_end; ++kb, ++it) {
          const uint32_t s = it % STAGES, ph = (it / STAGES) & 1;
          tc::mbar_wait(bar_full + 8 * s, ph);
          tc::tc_fence_after();
          const uint32_t da = sA + s * A_TILE, db = sB + s * B_TILE;
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            // K-major: +32 B per 16 k inside the 128 B swizzle row; MN-major: +16 rows of 128 B
            const uint64_t ad = a.a_mn ? tc::smem_desc_sw128(da + k * 2048, A_TILE / 2, 1024)
                                       : tc::smem_desc_sw128(da + k * 32, 16, 1024);
            const uint64_t bd = a.b_mn ? tc::smem_desc_sw128(db + k * 2048, B_TILE / 2, 1024)
                                       : tc::smem_desc_sw128(db + k * 32, 16, 1024);
            const uint32_t acc = (kb > kb_beg || k > 0) ? 1u : 0u;
            if (CTA2) tc::umma_bf16_2sm(tacc, ad, bd, a.idesc, acc);
            else tc::umma_bf16(tacc, ad, bd, a.idesc, acc);
          }
          // ring slot reusable (in both CTAs) once these MMAs have read it
          if (CTA2) tc::umma_commit_2sm(bar_empty + 8 * s, 3); else tc::umma_commit(bar_empty + 8 * s);
        }
        // accumulator complete -> epilogue warps of both CTAs
        if (CTA2) tc::umma_commit_2sm(bar_accf + 8 * buf, 3); else tc::umma_commit(bar_accf + 8 * buf);
      }
    }
  } else {
    // ===== epilogue: warps 2..9, TMEM lane quarter = warp % 4; the two warpgroups split every
    // 128-column half (64 columns = one bf16 staging panel each), so thread = (row, column half) =====
    const int quarter = warp & 3;
    const int cgp = (warp - 2) >> 2;
    const int row = quarter * 32 + lane;
    const int te = threadIdx.x - 64;
    // step = (work item, 128-column half); aux tile of a step: old C (accumulate) or the saved
    // activation (ReLU mask), bf16, prefetched one step ahead (issue order == consumption order)
    auto issue_aux = [&](int g, int tile, int half) {
      if (!G.p[g].aux) return;
      int m0, n0;
      tile_origin(G.p[g], tile, m0, n0);
      tc::mbar_expect_tx(bar_aux, 32 * 1024);
      tc::tma_load_2d(sAux, &TMS.aux[g], n0 + half * 128, m0, bar_aux);
      tc::tma_load_2d(sAux + 16384, &TMS.aux[g], n0 + half * 128 + 64, m0, bar_aux);
    };
    pdl_wait();
    WorkIter wi;
    iter_init(wi);
    int g, tile, sp, kb_beg, kb_end;
    if (te == 0 && G.any_aux) {    // aux tile of the first step
      WorkIter first = wi;
      if (iter_next(first, g, tile, sp, kb_beg, kb_end)) issue_aux(g, tile, 0);
    }
    uint32_t ti = 0, aux_ctr = 0, step = 0;
    bool prev_f32 = true;          // the previous step's store may span both staging buffers
    for (; iter_next(wi, g, tile, sp, kb_beg, kb_end); ++ti) {
      int m0, n0;
      const TcArgs& a = G.p[g];
      const CUtensorMap* tmC = &TMS.c[g];
      const bool partial = a.splits > 1 || G.streamk;
      const bool out_f32 = partial || !a.c_bf16;
      tile_origin(a, tile, m0, n0);
      const int64_t m = (int64_t)m0 + row;
      const int pos_row = a.pos ? (int)((uint32_t)(m0 + row) % (uint32_t)a.pos_period) : 0;
      const uint32_t buf = ti & 1, aph = (ti >> 1) & 1;
      tc::mbar_wait(bar_accf + 8 * buf, aph);
      tc::tc_fence_after();
#pragma unroll 1
      for (int half = 0; half < NHALF; ++half, ++step) {
        const int nh = n0 + half * 128;                  // first column of this half
        // bf16 tiles (32 KB) alternate between the two 32 KB staging buffers when no problem of
        // the launch needs the second one for aux tiles: the store of the previous step may then
        // still be reading its buffer while this step fills the other one
        const bool alt = !LITE && !out_f32 && !G.any_aux;
        const uint32_t sO = sOut + ((alt && (step & 1)) ? 32 * 1024 : 0);
        if (te == 0) {
          if (alt && !prev_f32) tc::tma_store_wait_read1();
          else tc::tma_store_wait_read();                // previous store has left the staging tile
        }
        prev_f32 = out_f32;
        if (a.bias && te < 128) sbias[te] = (nh + te < a.N) ? __ldg(a.bias + nh + te) : 0.f;
        asm volatile("bar.sync 1, 256;" ::: "memory");
        if (a.aux) { tc::mbar_wait(bar_aux, aux_ctr & 1); ++aux_ctr; }
        const uint32_t taddr =
            tmem_base + buf * BN + half * 128 + ((uint32_t)(quarter * 32) << 16);
#pragma unroll 1
        for (int c2 = 0; c2 < 2; ++c2) {
          const int ch = cgp * 2 + c2;
          uint32_t r[32];
          tc::tmem_ld32(taddr + ch * 32, r);
          tc::tmem_ld_wait();
          // rows >= M / columns >= N hold zeros or junk that the TMA store clips: no guards needed
          if (a.bias) {
#pragma unroll
            for (int i = 0; i < 32; ++i)
              r[i] = __float_as_uint(__uint_as_float(r[i]) + sbias[ch * 32 + i]);
          }
          if constexpr (FAM == 3) {
            // y = drop(x W^T + b) + pos: the mask of element (m, c) of the contiguous (M, N)
            // tensor, i = m*N + c, one hash per four consecutive i (dropout.cuh)
            if (a.drop_thr) {
              const uint64_t seed = drop_seed(a.drop_seed, G.drop_step);
              const uint64_t i0 = (uint64_t)m * (uint64_t)a.N + (uint64_t)(nh + ch * 32);
              uint64_t h = hash_bits(seed, i0 >> 2);
#pragma unroll
              for (int i = 0; i < 32; ++i) {
                const uint64_t e = i0 + i;
                if (i > 0 && (e & 3) == 0) h = hash_bits(seed, e >> 2);
                r[i] = __float_as_uint(drop_keep(h, e, a.drop_thr)
                                           ? __uint_as_float(r[i]) * a.drop_scale : 0.f);
              }
            }
          }
          if (a.pos && m < a.M) {   // position table row of this output row (period = seq length)
            const float* prow = a.pos + (int64_t)pos_row * a.pos_ld + nh + ch * 32;
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (nh + ch * 32 + i < a.N)
                r[i] = __float_as_uint(__uint_as_float(r[i]) + __ldg(prow + i));
          }
          if (a.relu) {
#pragma unroll
            for (int i = 0; i < 32; ++i) r[i] = __float_as_uint(fmaxf(__uint_as_float(r[i]), 0.f));
          }
          if (a.aux) {
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              uint32_t x[4];
              asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
                           : "=r"(x[0]), "=r"(x[1]), "=r"(x[2]), "=r"(x[3])
                           : "r"(sAux + (ch >> 1) * 16384 +
                                 tc::sw128_offset(row, (ch & 1) * 4 + c)));
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float lo = __uint_as_float(x[e] << 16);
                const float hi = __uint_as_float(x[e] & 0xFFFF0000u);
                float v0 = __uint_as_float(r[8 * c + 2 * e]);
                float v1 = __uint_as_float(r[8 * c + 2 * e + 1]);
                if (a.aux == AUX_ACC) { v0 += lo; v1 += hi; }
                else { if (!(lo > 0.f)) v0 = 0.f; if (!(hi > 0.f)) v1 = 0.f; }
                r[8 * c + 2 * e] = __float_as_uint(v0);
                r[8 * c + 2 * e + 1] = __float_as_uint(v1);
              }
            }
          }
          if (out_f32) {      // 4 panels of 32 fp32 columns: [128 rows][128 B]
#pragma unroll
            for (int c = 0; c < 8; ++c)
              asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(
                               sO + ch * 16384 + tc::sw128_offset(row, c)),
                           "r"(r[4 * c]), "r"(r[4 * c + 1]), "r"(r[4 * c + 2]), "r"(r[4 * c + 3])
                           : "memory");
          } else {            // 2 panels of 64 bf16 columns
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              uint32_t pk[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                __nv_bfloat162 t = __floats2bfloat162_rn(__uint_as_float(r[8 * c + 2 * e]),
                                                         __uint_as_float(r[8 * c + 2 * e + 1]));
                pk[e] = *reinterpret_cast<uint32_t*>(&t);
              }
              asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(
                               sO + (ch >> 1) * 16384 + tc::sw128_offset(row, (ch & 1) * 4 + c)),
                           "r"(pk[0]), "r"(pk[1]), "r"(pk[2]), "r"(pk[3])
                           : "memory");
            }
          }
        }
        tc::tc_fence_before();
        tc::fence_proxy_async();
        asm volatile("bar.sync 1, 256;" ::: "memory");
        if (te == 0) {
          if (half == NHALF - 1) {   // whole accumulator drained by this CTA -> tell the MMA issuer
            if (CTA2) tc::mbar_arrive_cta(bar_acce + 8 * buf, 0); else tc::mbar_arrive(bar_acce + 8 * buf);
          }
          if (partial && a.reduce_add) {   // C += slice, summed by the L2
#pragma unroll
            for (int p = 0; p < 4; ++p)
              if (nh + p * 32 < a.N) tc::tma_reduce_add_2d(tmC, sO + p * 16384, nh + p * 32, m0);
          } else if (partial) {   // workspace: [(tile*splits + split)*TM rows][BN fp32 columns]
            const int prow = (tile * a.splits + sp) * TM + (int)rank * BM;
#pragma unroll
            for (int p = 0; p < 4; ++p)
              tc::tma_store_2d(tmC, sO + p * 16384, half * 128 + p * 32, prow);
          } else if (out_f32) {
#pragma unroll
            for (int p = 0; p < 4; ++p)
              if (nh + p * 32 < a.N) tc::tma_store_2d(tmC, sO + p * 16384, nh + p * 32, m0);
          } else {
            if (nh < a.N) tc::tma_store_2d(tmC, sO, nh, m0);
            if (nh + 64 < a.N) tc::tma_store_2d(tmC, sO + 16384, nh + 64, m0);
          }
          tc::tma_store_commit();
          // prefetch the aux tile of the next step (if that step has one)
          if (G.any_aux) {
            if (half + 1 < NHALF) {
              issue_aux(g, tile, half + 1);
            } else {
              WorkIter nx = wi;      // (wi already points past the current segment)
              int g2, t2, s2, b2, e2;
              if (iter_next(nx, g2, t2, s2, b2, e2)) issue_aux(g2, t2, 0);
            }
          }
        }
      }
    }
    // the staging tiles must outlive the bulk stores' READS only; the writes are complete by the
    // time the grid is (what a dependent launch waits for), like the attention kernels' exits
    if (te == 0) tc::tma_store_wait_read();
  }
  tc::tc_fence_before();
  if (CTA2) tc::cluster_sync(); else __syncthreads();   // the peer may still signal our barriers
  if (warp == 1) {
    tc::tc_fence_after();
    if (CTA2) tc::tmem_dealloc_2sm(tmem_base, 2 * BN); else tc::tmem_dealloc(tmem_base, 2 * BN);
  }
}

struct ReduceArgs {
  const float* partial;
  void* C;
  int64_t ldc;
  int M, N, splits, tiles_n, c_bf16, accumulate, tm_rows, bn_cols;
  const float* bias;
};

// bf16 outputs only: sum the split-K partial tiles in a fixed order, bias / accumulate / convert
__global__ void __launch_bounds__(256) splitk_reduce_kernel(const ReduceArgs a) {
  const int tile = blockIdx.x;
  const int TMr = a.tm_rows, BNc = a.bn_cols;
  const int m0 = (tile / a.tiles_n) * TMr, n0 = (tile % a.tiles_n) * BNc;
  const float* src = a.partial + (size_t)tile * a.splits * TMr * BNc;
  for (int e = threadIdx.x + blockIdx.y * 256; e < TMr * BNc / 4; e += 256 * gridDim.y) {
    const int row = e / (BNc / 4), c4 = (e % (BNc / 4)) * 4;
    const int64_t m = (int64_t)m0 + row;
    const int n = n0 + c4;
    if (m >= a.M || n >= a.N) continue;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int s = 0; s < a.splits; ++s) {
      const float4 v = *reinterpret_cast<const float4*>(src + ((size_t)s * TMr + row) * BNc + c4);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    float x[4] = {acc.x, acc.y, acc.z, acc.w};
    for (int j = 0; j < 4 && n + j < a.N; ++j) {
      if (a.bias) x[j] += __ldg(a.bias + n + j);
      if (a.c_bf16) {
        bf16* c = static_cast<bf16*>(a.C) + m * a.ldc + n + j;
        *c = from_f<bf16>(a.accumulate ? x[j] + to_f(*c) : x[j]);
      } else {
        float* c = static_cast<float*>(a.C) + m * a.ldc + n + j;
        *c = a.accumulate ? x[j] + *c : x[j];
      }
    }
  }
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

int num_sms(int sm_budget) {
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess ||
      cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
    n = 148;
  // a communication kernel running concurrently (all-reduce overlapped with backward) holds some
  // SMs; a persistent grid larger than what is free would serialise its last CTAs
  return (sm_budget > 0 && sm_budget < n) ? sm_budget : n;
}

bool make_tmap(CUtensorMap* out, CUtensorMapDataType dt, const void* base, int rank,
               const uint64_t* dims, const uint64_t* strides_bytes, const uint32_t* box) {
  PFN_encodeTiled enc = mm_get_encode_tiled();
  if (!enc) return false;
  cuuint64_t gd[5], gs[5];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) {
    gd[i] = dims[i];
    bx[i] = box[i];
    es[i] = 1;
    if (i + 1 < rank) gs[i] = strides_bytes[i];
  }
  const CUresult r = enc(out, dt, (cuuint32_t)rank, const_cast<void*>(base), gd, gs, bx, es,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

}  // namespace

PFN_encodeTiled mm_get_encode_tiled() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      return nullptr;
    fn = reinterpret_cast<PFN_encodeTiled>(p);
  }
  return fn;
}

bool mm_make_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims,
                       const uint64_t* strides_bytes, const uint32_t* box) {
  return make_tmap(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, base, rank, dims, strides_bytes, box);
}
bool mm_make_tmap_f32(CUtensorMap* out, const void* base, int rank, const uint64_t* dims,
                      const uint64_t* strides_bytes, const uint32_t* box) {
  return make_tmap(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, base, rank, dims, strides_bytes, box);
}

bool gemm_tc_supported(const GemmArgs& g, int c_bf16, bool any_size) {
  // Size floor: a lone small GEMM is faster on the SIMT kernel than on a 128-row tensor-core tile.
  // Inside a GROUPED launch (any_size) small problems ride along with the others - TMA zero-fills
  // / clips the rows and columns a tile has beyond the matrix - which is what keeps a batch-1
  // inference layer (M = 25 rows) at one launch per kernel kind.
  if (!any_size) {
    if (g.M < 64 || g.N < 64 || g.K < 64) return false;
    if ((double)g.M * (double)g.N * (double)g.K < (double)(1 << 22)) return false;
  }
  if (g.M < 1 || g.N < 8 || g.K < 8) return false;
  if (g.M > (1ll << 31) - 512 || g.N > (1ll << 31) - 512 || g.K > (1ll << 31) - 512) return false;
  const bool a_k = (g.sAk == 1 && g.sAm % 8 == 0), a_mn = (g.sAm == 1 && g.sAk % 8 == 0);
  const bool b_k = (g.sBk == 1 && g.sBn % 8 == 0), b_mn = (g.sBn == 1 && g.sBk % 8 == 0);
  if (!(a_k || a_mn) || !(b_k || b_mn)) return false;
  if (!aligned16(g.A) || !aligned16(g.B) || !aligned16(g.C)) return false;
  if (g.ldc % (c_bf16 ? 8 : 4) != 0) return false;
  if (g.relu_src && (!g.relu_src_bf16 || !aligned16(g.relu_src) || g.ldrelu % 8 != 0)) return false;
  if (g.relu_src && (g.accumulate || !c_bf16)) return false;   // one aux tile at a time
  if (g.accumulate && !c_bf16) return false;                   // fp32 C += ... : SIMT path
  return true;
}

namespace {
template <int NG, int FAM>
int gemm_tc_grouped_t(const GemmArgs* gs, const int* c_bf16s, int n, cudaStream_t st) {
  // (idempotent and cheap: no guard variable, so concurrent callers cannot race on one)
  MM_CUDA_OK(cudaFuncSetAttribute(gemm_tc_kernel<false, NG, FAM>,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
  MM_CUDA_OK(cudaFuncSetAttribute(gemm_tc_kernel<true, NG, FAM>,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
  MM_CUDA_OK(cudaFuncSetAttribute(gemm_tc_kernel<false, NG, FAM, true>,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_LITE));
  const MmStreamCfg scfg = mm_stream_cfg(st);    // this stream's workspace / SM budget / PDL
  float* const ws = scfg.ws;
  const size_t ws_bytes = scfg.ws_bytes;
  // CTA pairs (256 x 256 tiles) when every output is wide and tall enough to fill them
  bool cta2 = true;
  for (int i = 0; i < n; ++i) cta2 = cta2 && gs[i].N >= 256 && gs[i].M >= 256;
  {
    // experiment hook: MMEMO_GEMM_CTA2=0 forces single-CTA 128 x 128 tiles, =N (> 1) uses them
    // when the launch has fewer than N pair tiles per CTA pair
    const char* env = getenv("MMEMO_GEMM_CTA2");
    if (env && cta2) {
      const int v = atoi(env);
      if (v == 0) cta2 = false;
      else if (v > 1) {
        long pt = 0;
        for (int i = 0; i < n; ++i) pt += cdiv(gs[i].M, 256) * cdiv(gs[i].N, 256);
        if (pt * 100 < (long)v * (num_sms(scfg.sm_budget) / 2)) cta2 = false;   // v = percent of one pair wave
      }
    }
  }
  const int TM = cta2 ? 256 : 128, BN = cta2 ? 256 : 128;
  const int sms = num_sms(scfg.sm_budget);
  const int units_max = cta2 ? sms / 2 : sms;      // schedulable work units (pairs or CTAs)
  // split-K when the outputs have too few tiles to occupy the machine and K is long (needs linear
  // epilogues: bias and accumulate are applied after / by the reduction)
  int tiles_sum = 0, kb_min = 1 << 30;
  bool linear = true, all_reduce_add = true;
  for (int i = 0; i < n; ++i) {
    const GemmArgs& g = gs[i];
    tiles_sum += (int)(cdiv(g.M, TM) * cdiv(g.N, BN));
    const int kb = (int)cdiv(g.K, BK);
    kb_min = kb < kb_min ? kb : kb_min;
    linear = linear && !g.relu && !g.relu_src && !g.pos && !(g.drop_p > 0.f);
    all_reduce_add = all_reduce_add && !c_bf16s[i] && !g.bias;   // fp32 C summed by TMA reduce-add
  }
  int splits = 1;
  // Stream-K (see the kernel): fp32 outputs summed by TMA reduce-add.  Each unit gets
  // ceil(total k-blocks / units) consecutive k-blocks, so problems of very different K share the
  // machine evenly (Ren-MME layer, 48 weight gradients with K = 10 240 ... 70 400 rows: 127 ->
  // 104 us).  Only for launches whose problems have at most two output tiles each: tiles of ONE
  // problem share operand strips, and the regular item list keeps them in lockstep along K so
  // that a strip is fetched from HBM once; stream-K ranges start at unrelated k offsets and
  // measured 166 vs 108 us on the 32-tile weight-gradient group of the seq-256 encoder (operand
  // traffic 1.07 GB instead of 0.44 GB) and 32.9 vs 31.7 us at seq 128.
  int64_t kb_sum = 0, operand_bytes = 0;
  int tiles_max = 0;
  for (int i = 0; i < n; ++i) {
    const int t = (int)(cdiv(gs[i].M, TM) * cdiv(gs[i].N, BN));
    tiles_max = t > tiles_max ? t : tiles_max;
    kb_sum += t * cdiv(gs[i].K, BK);
    operand_bytes += 2 * gs[i].K * (gs[i].M + gs[i].N);
  }
  // (... or whose operands are small enough to stay in L2 whatever the order: the modality
  // projections' weight gradients - three problems of 10 / 50 / 100 k-blocks on five tiles - ran
  // 33 us on five CTAs.)  A range is at least 8 k-blocks, so tiny launches use fewer units.
  int kb_per_unit = (int)cdiv(kb_sum, units_max);
  if (kb_per_unit < 8) kb_per_unit = 8;
  bool streamk = linear && all_reduce_add && (tiles_max <= 2 || operand_bytes <= (16ll << 20)) &&
                 tiles_sum <= 4 * units_max && kb_sum >= 16 && kb_sum < (1ll << 30) &&
                 (n > 1 || tiles_sum * 2 <= units_max);
  {
    const char* env = getenv("MMEMO_GEMM_STREAMK");     // A/B knob: 0 = the split-K item list
    if (env && env[0] == '0') streamk = false;
  }
  if (!streamk && tiles_sum * 2 <= units_max && kb_min >= 16 && linear && (all_reduce_add || n == 1)) {
    splits = units_max / tiles_sum;                     // one balanced round of work items
    if (splits > kb_min / 4) splits = kb_min / 4;
    if (splits > 32) splits = 32;
    if (!all_reduce_add) {
      const size_t per_split = (size_t)tiles_sum * TM * BN * sizeof(float);
      if (per_split * (size_t)splits > ws_bytes) splits = (int)(ws_bytes / per_split);
    }
    if (splits < 2) splits = 1;
  }

  static thread_local TmapGroup<NG> tms;     // host staging (copied by value into the launch)
  static thread_local GroupArgs<NG> G;
  G = GroupArgs<NG>{};
  G.n = n;
  G.streamk = streamk ? 1 : 0;
  G.kb_per_unit = kb_per_unit;
  int items = 0;
  bool ok = true;
  for (int i = 0; i < n; ++i) {
    const GemmArgs& g = gs[i];
    const int c_bf16 = c_bf16s[i];
    const bool a_mn = !(g.sAk == 1 && g.sAm % 8 == 0);
    const bool b_mn = !(g.sBk == 1 && g.sBn % 8 == 0);
    const int tiles_n = (int)cdiv(g.N, BN), tiles_m = (int)cdiv(g.M, TM);
    const int tiles = tiles_m * tiles_n;
    const int kb_total = (int)cdiv(g.K, BK);
    const int kb_per = (int)cdiv(kb_total, splits);
    const int sp = (int)cdiv(kb_total, kb_per);        // every slice owns >= 1 k-block
    const bool partial = sp > 1 || streamk;
    const bool reduce_add = partial && all_reduce_add;
    const int aux = partial ? AUX_NONE : (g.relu_src ? AUX_RELU : (g.accumulate ? AUX_ACC : AUX_NONE));
    uint64_t dims[2], str[1];
    uint32_t box[2];
    if (!a_mn) { dims[0] = g.K; dims[1] = g.M; str[0] = g.sAm * 2; box[0] = 64; box[1] = BM; }
    else       { dims[0] = g.M; dims[1] = g.K; str[0] = g.sAk * 2; box[0] = 64; box[1] = BK; }
    ok = ok && mm_make_tmap_bf16(&tms.a[i], g.A, 2, dims, str, box);
    if (!b_mn) { dims[0] = g.K; dims[1] = g.N; str[0] = g.sBn * 2; box[0] = 64; box[1] = 128; }
    else       { dims[0] = g.N; dims[1] = g.K; str[0] = g.sBk * 2; box[0] = 64; box[1] = BK; }
    ok = ok && mm_make_tmap_bf16(&tms.b[i], g.B, 2, dims, str, box);
    if (partial && !reduce_add) {     // n == 1 here
      dims[0] = BN; dims[1] = (uint64_t)tiles * sp * TM; str[0] = (uint64_t)BN * 4;
      box[0] = 32; box[1] = BM;
      ok = ok && mm_make_tmap_f32(&tms.c[i], ws, 2, dims, str, box);
    } else if (!c_bf16) {
      dims[0] = g.N; dims[1] = g.M; str[0] = g.ldc * 4; box[0] = 32; box[1] = BM;
      ok = ok && mm_make_tmap_f32(&tms.c[i], g.C, 2, dims, str, box);
    } else {
      dims[0] = g.N; dims[1] = g.M; str[0] = g.ldc * 2; box[0] = 64; box[1] = BM;
      ok = ok && mm_make_tmap_bf16(&tms.c[i], g.C, 2, dims, str, box);
    }
    if (aux == AUX_RELU) {
      dims[0] = g.N; dims[1] = g.M; str[0] = g.ldrelu * 2; box[0] = 64; box[1] = BM;
      ok = ok && mm_make_tmap_bf16(&tms.aux[i], g.relu_src, 2, dims, str, box);
    } else if (aux == AUX_ACC) {
      dims[0] = g.N; dims[1] = g.M; str[0] = g.ldc * 2; box[0] = 64; box[1] = BM;
      ok = ok && mm_make_tmap_bf16(&tms.aux[i], g.C, 2, dims, str, box);
    } else {
      tms.aux[i] = tms.a[i];
    }
    TcArgs& a = G.p[i];
    a.M = (int)g.M; a.N = (int)g.N; a.K = (int)g.K; a.c_bf16 = c_bf16;
    a.bias = partial ? nullptr : g.bias;
    a.pos = g.pos; a.pos_period = (int)g.pos_period;
    a.pos_ld = (int)(g.ldpos ? g.ldpos : g.N);
    a.relu = g.relu; a.aux = aux;
    if (aux != AUX_NONE) G.any_aux = 1;
    a.a_mn = a_mn; a.b_mn = b_mn;
    a.idesc = tc::idesc_bf16(TM, BN, a_mn, b_mn);
    a.splits = sp; a.kb_per = kb_per; a.kb_total = kb_total;
    a.reduce_add = reduce_add;
    a.tiles_m = tiles_m; a.tiles_n = tiles_n;
    if (g.drop_p > 0.f) {
      a.drop_thr = (uint32_t)(g.drop_p * 65536.0f + 0.5f);
      a.drop_scale = 1.0f / (1.0f - g.drop_p);
      a.drop_seed = g.drop_seed;
      G.drop_step = reinterpret_cast<const unsigned long long*>(g.drop_step);
    }
    G.item_start[i] = items;
    items += streamk ? tiles * kb_total : tiles * sp;
    if (reduce_add && !g.accumulate && !g.c_zeroed)   // the slices accumulate into C: start from zero
      MM_CUDA_OK(cudaMemset2DAsync(g.C, g.ldc * sizeof(float), 0, g.N * sizeof(float), g.M, st));
  }
  G.item_start[n] = items;
  if (!ok) {
    mmemo_set_error("cuTensorMapEncodeTiled failed (gemm_tc)", __FILE__, __LINE__);
    return MMEMO_ERR_CUDA;
  }
  // two CTAs per SM (LITE) for launches of bf16 tiles with no auxiliary tile and more than one
  // tile per SM: one CTA's epilogue chain overlaps the other's loads and MMAs
  bool lite = !cta2 && !streamk && splits == 1 && !G.any_aux && items > units_max;
  for (int i = 0; i < n && lite; ++i) lite = c_bf16s[i] != 0;
  {
    const char* env = getenv("MMEMO_GEMM_LITE");        // A/B knob: 0 = one CTA per SM
    if (env && env[0] == '0') lite = false;
  }
  const int cap = lite ? 2 * units_max : units_max;
  const int units = streamk ? (int)cdiv(items, kb_per_unit) : (items < cap ? items : cap);
  if (lite) {
    MM_CUDA_OK(mm_launch(gemm_tc_kernel<false, NG, FAM, true>, dim3((unsigned)units),
                         dim3(NTHREADS), SMEM_LITE, st, tms, G));
  } else if (cta2) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(2 * units));
    cfg.blockDim = dim3(NTHREADS);
    cfg.dynamicSmemBytes = SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute at[2];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = scfg.pdl ? 2 : 1;
    MM_CUDA_OK(cudaLaunchKernelEx(&cfg, gemm_tc_kernel<true, NG, FAM>, tms, G));
  } else {
    MM_CUDA_OK(mm_launch(gemm_tc_kernel<false, NG, FAM>, dim3((unsigned)units), dim3(NTHREADS),
                         SMEM_BYTES, st, tms, G));
  }
  if (n == 1 && G.p[0].splits > 1 && !G.p[0].reduce_add) {
    const GemmArgs& g = gs[0];
    ReduceArgs r = {};
    r.partial = ws; r.C = g.C; r.ldc = g.ldc; r.M = (int)g.M; r.N = (int)g.N;
    r.splits = G.p[0].splits; r.tiles_n = G.p[0].tiles_n; r.c_bf16 = c_bf16s[0];
    r.accumulate = g.accumulate;
    r.tm_rows = TM; r.bn_cols = BN;
    r.bias = g.bias;
    const int tiles = G.p[0].tiles_m * G.p[0].tiles_n;
    int ysplit = (int)cdiv(2 * sms, tiles);
    if (ysplit > 16) ysplit = 16;
    splitk_reduce_kernel<<<dim3((unsigned)tiles, (unsigned)ysplit), 256, 0, st>>>(r);
    MM_LAUNCH_OK();
  }
  return MMEMO_OK;
}
}  // namespace

int gemm_tc_grouped(const GemmArgs* gs, const int* c_bf16s, int n, int family, cudaStream_t st) {
  if (n < 1 || n > MAXG) return MMEMO_ERR_ARG;
  if (n <= MAXG_SMALL) {
    if (family == 0) return gemm_tc_grouped_t<MAXG_SMALL, 0>(gs, c_bf16s, n, st);
    if (family == 1) return gemm_tc_grouped_t<MAXG_SMALL, 1>(gs, c_bf16s, n, st);
    if (family == 3) return gemm_tc_grouped_t<MAXG_SMALL, 3>(gs, c_bf16s, n, st);
    return gemm_tc_grouped_t<MAXG_SMALL, 2>(gs, c_bf16s, n, st);
  }
  if (family == 0) return gemm_tc_grouped_t<MAXG, 0>(gs, c_bf16s, n, st);
  if (family == 1) return gemm_tc_grouped_t<MAXG, 1>(gs, c_bf16s, n, st);
  if (family == 3) return gemm_tc_grouped_t<MAXG, 3>(gs, c_bf16s, n, st);
  return gemm_tc_grouped_t<MAXG, 2>(gs, c_bf16s, n, st);
}

int gemm_tc(const GemmArgs& g, int c_bf16, int family, cudaStream_t st) {
  return gemm_tc_grouped(&g, &c_bf16, 1, family, st);
}
