// Generic strided SIMT GEMM (fp32 accumulate) used (i) for the float32 parity mode everywhere and
// (ii) in the bf16 mode for shapes the tcgen05 kernel does not take (tiny N, ragged K, fp32 inputs).
//
//   C[m,n] (+)= epi( sum_k A[m*sAm + k*sAk] * B[n*sBn + k*sBk] )
//
// One kernel covers y = x w^T (NT), dx = dy w (NN) and dw = dy^T x (TN) through the strides.
// 64x64x16 tiles, 256 threads, 4x4 register micro-tile; split-K over gridDim.z for the tall-skinny
// weight-gradient shapes (K' = B*L rows, M'xN' = a weight matrix) and the small float32 heads.
//
// Split-K sums in a fixed order: every CTA of a tile writes its float32 partial tile to the
// stream's workspace (slot tile * n_split + split), and the last of them to arrive (a per-tile
// counter, zeroed before the launch) adds the slots in split order and runs the epilogue.  A
// result therefore does not depend on CTA scheduling, and the grouped launch, which gives each
// problem the split factor gemm_simt would give it, reproduces gemm_simt bit for bit.
#include "common.cuh"
#include "gemm.h"

namespace {

constexpr int BM = 64, BN = 64, BK = 16, PAD = 4;
constexpr size_t SLOT_BYTES = BM * BN * sizeof(float);     // one partial tile

// workspace bytes of the per-tile arrival counters (256-byte aligned, so the slots that follow are)
size_t counter_bytes(int64_t tiles) { return (size_t)(tiles * sizeof(unsigned) + 255) / 256 * 256; }

// Split-K factor of one problem (gemm_simt and the grouped launch use the same rule): only when the
// output grid cannot fill the GPU, K is long, C is float32 with no non-linear epilogue, and the
// partial tiles fit in the workspace next to the counters.
int64_t split_of(const GemmArgs& g, bool linear_f32, size_t ws_bytes) {
  const int64_t tiles = cdiv(g.M, BM) * cdiv(g.N, BN);
  // (also the small float32 head GEMMs: (B, 576..2304) x (9..96 outputs) are 3-8 tiles whose serial
  // K loop took 30-76 us on a handful of CTAs)
  if (!linear_f32 || tiles <= 0 || tiles >= 148 || g.K < 128) return 1;
  int64_t split = cdiv(296, tiles);
  if (split > g.K / 64) split = g.K / 64;
  const size_t fixed = counter_bytes(tiles);
  const int64_t fit = ws_bytes > fixed ? (int64_t)((ws_bytes - fixed) / (tiles * SLOT_BYTES)) : 0;
  if (split > fit) split = fit;
  return split < 2 ? 1 : split;
}

size_t split_bytes(const GemmArgs& g, int64_t split) {
  const int64_t tiles = cdiv(g.M, BM) * cdiv(g.N, BN);
  return split > 1 ? counter_bytes(tiles) + (size_t)(tiles * split) * SLOT_BYTES : 0;
}

// One 64x64 output tile (tile_m, tile_n) of g over split-K part `split` of `n_split`; with
// n_split > 1, `part` holds the problem's partial tiles and `count` its per-tile counters.
template <typename TA, typename TB, typename TC>
__device__ __forceinline__ void gemm_simt_tile(const GemmArgs& g, int64_t tile_m, int64_t tile_n,
                                               int split, int n_split, float* part,
                                               unsigned* count) {
  __shared__ __align__(16) float As[BK][BM + PAD];
  __shared__ __align__(16) float Bs[BK][BN + PAD];
  const TA* __restrict__ A = static_cast<const TA*>(g.A);
  const TB* __restrict__ B = static_cast<const TB*>(g.B);
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int64_t m0 = tile_m * BM, n0 = tile_n * BN;
  // split-K range of this CTA
  const int64_t kchunk = ((g.K + n_split - 1) / n_split + BK - 1) / BK * BK;
  const int64_t kbeg = (int64_t)split * kchunk;
  const int64_t kend = min(g.K, kbeg + kchunk);

  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  const bool a_kfast = (g.sAk == 1), b_kfast = (g.sBk == 1);
  for (int64_t k0 = kbeg; k0 < kend; k0 += BK) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int idx = tid + i * 256;
      int mm, kk;
      if (a_kfast) { mm = idx >> 4; kk = idx & 15; } else { kk = idx >> 6; mm = idx & 63; }
      const int64_t m = m0 + mm, k = k0 + kk;
      As[kk][mm] = (m < g.M && k < kend) ? to_f(A[m * g.sAm + k * g.sAk]) : 0.f;
      int nn;
      if (b_kfast) { nn = idx >> 4; kk = idx & 15; } else { kk = idx >> 6; nn = idx & 63; }
      const int64_t n = n0 + nn, kb = k0 + kk;
      Bs[kk][nn] = (n < g.N && kb < kend) ? to_f(B[n * g.sBn + kb * g.sBk]) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      const float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      const float4 b = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }

  if (n_split > 1) {
    // split-K: park the partial tile; the last CTA of the tile sums all of them in split order
    __shared__ int is_last;
    const int64_t tile = tile_m * ((g.N + BN - 1) / BN) + tile_n;
    float* slots = part + (size_t)tile * n_split * (BM * BN);
    const bool cols = n0 + tx * 4 < g.N;
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (cols && m0 + ty * 4 + i < g.M)
        *reinterpret_cast<float4*>(slots + (size_t)split * (BM * BN) + (ty * 4 + i) * BN + tx * 4) =
            make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
    __threadfence();
    __syncthreads();
    if (tid == 0) is_last = atomicAdd(count + tile, 1u) == (unsigned)(n_split - 1);
    __syncthreads();
    if (!is_last) return;
    __threadfence();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (!cols || m0 + ty * 4 + i >= g.M) continue;
      const float* src = slots + (ty * 4 + i) * BN + tx * 4;
      float4 s = __ldcg(reinterpret_cast<const float4*>(src));
#pragma unroll 8
      for (int p = 1; p < n_split; ++p) {
        const float4 t = __ldcg(reinterpret_cast<const float4*>(src + (size_t)p * (BM * BN)));
        s.x += t.x; s.y += t.y; s.z += t.z; s.w += t.w;
      }
      acc[i][0] = s.x; acc[i][1] = s.y; acc[i][2] = s.z; acc[i][3] = s.w;
    }
  }

  TC* __restrict__ C = static_cast<TC*>(g.C);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t m = m0 + ty * 4 + i;
    if (m >= g.M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int64_t n = n0 + tx * 4 + j;
      if (n >= g.N) continue;
      float v = acc[i][j];
      if (g.bias) v += g.bias[n];
      if (g.pos) v += g.pos[(m % g.pos_period) * (g.ldpos ? g.ldpos : g.N) + n];
      if (g.relu) v = fmaxf(v, 0.f);
      if (g.relu_src) {
        const float r = g.relu_src_bf16
                            ? to_f(static_cast<const bf16*>(g.relu_src)[m * g.ldrelu + n])
                            : static_cast<const float*>(g.relu_src)[m * g.ldrelu + n];
        v = r > 0.f ? v : 0.f;
      }
      if (g.accumulate) v += to_f(C[m * g.ldc + n]);
      C[m * g.ldc + n] = from_f<TC>(v);
    }
  }
}

template <typename TA, typename TB, typename TC>
__global__ void __launch_bounds__(256) gemm_simt_kernel(GemmArgs g, float* part, unsigned* count) {
  gemm_simt_tile<TA, TB, TC>(g, blockIdx.y, blockIdx.x, blockIdx.z, gridDim.z, part, count);
}

// Grouped float32 GEMM: a flat list of CTAs over the problems of the table; problem p owns the CTAs
// [first[p], first[p + 1]) = its tiles (n-fastest) times its split-K parts.
struct SimtGroup {
  GemmArgs g[GEMM_SIMT_MAX_GROUP];
  float* part[GEMM_SIMT_MAX_GROUP];       // split problems: partial tiles / tile counters
  unsigned* count[GEMM_SIMT_MAX_GROUP];
  int first[GEMM_SIMT_MAX_GROUP + 1];
  int n_split[GEMM_SIMT_MAX_GROUP];
  int n;
};

__global__ void __launch_bounds__(256) gemm_simt_grouped_kernel(SimtGroup tb) {
  const int cta = blockIdx.x;
  int p = 0;
  while (cta >= tb.first[p + 1]) ++p;
  const GemmArgs& g = tb.g[p];
  const int local = cta - tb.first[p];
  const int64_t tiles_n = (g.N + BN - 1) / BN;
  const int64_t tiles = (g.M + BM - 1) / BM * tiles_n;
  const int split = (int)(local / tiles);
  const int64_t t = local - (int64_t)split * tiles;
  gemm_simt_tile<float, float, float>(g, t / tiles_n, t % tiles_n, split, tb.n_split[p],
                                      tb.part[p], tb.count[p]);
}

template <typename TA, typename TB, typename TC>
int launch(const GemmArgs& g, int splitk, float* ws, cudaStream_t st) {
  dim3 grid((unsigned)cdiv(g.N, BN), (unsigned)cdiv(g.M, BM), (unsigned)splitk);
  const int64_t tiles = (int64_t)grid.x * grid.y;
  float* part = splitk > 1 ? ws + counter_bytes(tiles) / sizeof(float) : nullptr;
  unsigned* count = splitk > 1 ? reinterpret_cast<unsigned*>(ws) : nullptr;
  if (splitk > 1) MM_CUDA_OK(cudaMemsetAsync(count, 0, tiles * sizeof(unsigned), st));
  gemm_simt_kernel<TA, TB, TC><<<grid, 256, 0, st>>>(g, part, count);
  MM_LAUNCH_OK();
  return MMEMO_OK;
}

// one grouped launch of problems whose split-K scratch fits in the workspace together: all tile
// counters first (one fill), then the partial tiles
int launch_group(const GemmArgs* gs, const int64_t* splits, int n, char* ws, cudaStream_t st) {
  SimtGroup tb;
  tb.n = n;
  int64_t cnt_tiles = 0;
  for (int i = 0; i < n; ++i)
    if (splits[i] > 1) cnt_tiles += cdiv(gs[i].M, BM) * cdiv(gs[i].N, BN);
  unsigned* counts = reinterpret_cast<unsigned*>(ws);
  float* slots = cnt_tiles ? reinterpret_cast<float*>(ws + counter_bytes(cnt_tiles)) : nullptr;
  int64_t total = 0, c_off = 0, s_off = 0;
  for (int i = 0; i < n; ++i) {
    const GemmArgs& g = gs[i];
    const int64_t tiles = g.M > 0 && g.N > 0 ? cdiv(g.M, BM) * cdiv(g.N, BN) : 0;
    tb.g[i] = g;
    tb.n_split[i] = (int)splits[i];
    tb.first[i] = (int)total;
    tb.part[i] = nullptr;
    tb.count[i] = nullptr;
    if (splits[i] > 1) {
      tb.count[i] = counts + c_off;
      tb.part[i] = slots + s_off * (BM * BN);
      c_off += tiles;
      s_off += tiles * splits[i];
    }
    total += tiles * splits[i];
  }
  tb.first[n] = (int)total;
  if (total == 0) return MMEMO_OK;
  if (cnt_tiles) MM_CUDA_OK(cudaMemsetAsync(counts, 0, cnt_tiles * sizeof(unsigned), st));
  gemm_simt_grouped_kernel<<<(unsigned)total, 256, 0, st>>>(tb);
  MM_LAUNCH_OK();
  return MMEMO_OK;
}

}  // namespace

int gemm_simt(const GemmArgs& g, int a_bf16, int b_bf16, int c_bf16, cudaStream_t st) {
  if (g.M <= 0 || g.N <= 0) return MMEMO_OK;
  MM_REQUIRE(g.A && g.B && g.C && g.K >= 0);
  const bool linear_f32 = !c_bf16 && !g.relu && !g.relu_src;
  const MmStreamCfg scfg = linear_f32 ? mm_stream_cfg(st) : MmStreamCfg{};
  const int splitk = (int)split_of(g, linear_f32, scfg.ws_bytes);
  if (!a_bf16 && !b_bf16 && !c_bf16) return launch<float, float, float>(g, splitk, scfg.ws, st);
  if (a_bf16 && b_bf16 && c_bf16) return launch<bf16, bf16, bf16>(g, splitk, scfg.ws, st);
  if (!a_bf16 && b_bf16 && c_bf16) return launch<float, bf16, bf16>(g, splitk, scfg.ws, st);
  if (a_bf16 && b_bf16 && !c_bf16) return launch<bf16, bf16, float>(g, splitk, scfg.ws, st);
  if (a_bf16 && !b_bf16 && !c_bf16) return launch<bf16, float, float>(g, splitk, scfg.ws, st);
  return MMEMO_ERR_ARG;
}

int gemm_simt_grouped_f32(const GemmArgs* gs, int n, cudaStream_t st) {
  MM_REQUIRE(n >= 1 && n <= GEMM_SIMT_MAX_GROUP);
  for (int i = 0; i < n; ++i) {
    const GemmArgs& g = gs[i];
    MM_REQUIRE(g.A && g.B && g.C && g.K >= 0 && g.M >= 0 && g.N >= 0);
    MM_REQUIRE(!g.relu && !g.relu_src && !g.accumulate && !g.pos);
  }
  // each problem gets the split factor gemm_simt gives it alone (so the results are the same bits);
  // consecutive problems share a launch while their scratch fits in the workspace together
  const MmStreamCfg scfg = mm_stream_cfg(st);
  char* ws = reinterpret_cast<char*>(scfg.ws);
  int64_t splits[GEMM_SIMT_MAX_GROUP];
  for (int i = 0; i < n; ++i)
    splits[i] = gs[i].M > 0 && gs[i].N > 0 ? split_of(gs[i], true, scfg.ws_bytes) : 1;
  int b = 0;
  size_t used = 0;
  for (int i = 0; i < n; ++i) {
    const size_t need = split_bytes(gs[i], splits[i]);
    if (i > b && used + need > scfg.ws_bytes) {
      const int rc = launch_group(gs + b, splits + b, i - b, ws, st);
      if (rc) return rc;
      b = i;
      used = 0;
    }
    used += need;
  }
  return launch_group(gs + b, splits + b, n - b, ws, st);
}
