// Small bandwidth-bound helpers: periodic row-sum (bias / position-table gradients), dtype casts
// (bf16 shadow weights) and counter-based dropout.
#include "common.cuh"
#include "dropout.cuh"

namespace {

// out[(m % period), n] += x[m, n].  CTA = (64 columns, a strip of rows); lanes own column pairs so the
// global reads are coalesced; rows with equal (m % period) are summed in registers first.
template <typename T>
__global__ void __launch_bounds__(256)
rowsum_kernel(const T* __restrict__ x, int64_t ldx, float* __restrict__ out, int64_t M, int64_t N,
              int64_t period, int64_t rows_per_cta) {
  __shared__ float red[8][2][33];
  const int lane = threadIdx.x & 31, wy = threadIdx.x >> 5;
  pdl_wait();
  pdl_trigger();
  const int64_t n = (int64_t)blockIdx.x * 64 + lane * 2;     // lane owns two adjacent columns
  const int64_t p = blockIdx.z;                       // residue class handled by this CTA
  const int64_t r_beg = (int64_t)blockIdx.y * rows_per_cta;  // in units of periods
  const int64_t n_per = (M - p + period - 1) / period;       // rows m = p + t*period, t < n_per
  float acc0 = 0.f, acc1 = 0.f;
  if (n < N) {
    const bool two = n + 1 < N;
    const int64_t t_end = min(n_per, r_beg + rows_per_cta);
#pragma unroll 4
    for (int64_t t = r_beg + wy; t < t_end; t += 8) {
      const T* px = x + (p + t * period) * ldx + n;
      acc0 += to_f(px[0]);
      if (two) acc1 += to_f(px[1]);
    }
  }
  red[wy][0][lane] = acc0;
  red[wy][1][lane] = acc1;
  __syncthreads();
  if (wy < 2 && n + wy < N) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += red[i][wy][lane];
    atomicAdd(out + p * N + n + wy, t);
  }
}

__global__ void cast_f2b_kernel(const float* __restrict__ s, bf16* __restrict__ d, int64_t n) {
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i + 3 < n) {
    const float4 v = *reinterpret_cast<const float4*>(s + i);
    __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
    uint2 o;
    o.x = *reinterpret_cast<uint32_t*>(&a);
    o.y = *reinterpret_cast<uint32_t*>(&b);
    *reinterpret_cast<uint2*>(d + i) = o;
  } else {
    for (int64_t j = i; j < n; ++j) d[j] = __float2bfloat16_rn(s[j]);
  }
}
__global__ void cast_b2f_kernel(const bf16* __restrict__ s, float* __restrict__ d, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) d[i] = __bfloat162float(s[i]);
}

// a uniform in [0,1) from hash_bits (dropout.cuh)
__device__ __forceinline__ float hash_uniform(uint64_t seed, uint64_t i) {
  return (float)(hash_bits(seed, i) >> 40) * (1.0f / 16777216.0f);
}
template <typename T>
__global__ void dropout_kernel(const T* __restrict__ x, T* __restrict__ y, int64_t n, float p,
                               float scale, uint64_t seed) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) y[i] = from_f<T>(hash_uniform(seed, (uint64_t)i) >= p ? to_f(x[i]) * scale : 0.f);
}

// dropout of several tensors in ONE launch (the two dropout sites of a fusion-trunk layer over all
// of its chains), in place or out of place.  Per-tensor seeds; `step` (device scalar, nullable) is
// mixed into every seed at run time so that a captured CUDA graph draws new masks on every replay.
constexpr int DROP_MAXT = 64;
struct DropTable {
  const void* x[DROP_MAXT];
  void* y[DROP_MAXT];
  long long n[DROP_MAXT];
  unsigned long long seed[DROP_MAXT];
  int count;
};
template <typename T>
__global__ void __launch_bounds__(256)
dropout_multi_kernel(const __grid_constant__ DropTable t, float p, float scale,
                     const unsigned long long* __restrict__ step) {
  const int which = blockIdx.y;
  pdl_wait();
  pdl_trigger();
  if (which >= t.count) return;
  const T* __restrict__ x = static_cast<const T*>(t.x[which]);
  T* __restrict__ y = static_cast<T*>(t.y[which]);
  const long long n = t.n[which];
  const uint64_t seed = t.seed[which] + (step ? step[0] * 0xD6E8FEB86659FD93ull : 0ull);
  // one 64-bit hash per FOUR consecutive elements, 16 bits each (p is resolved to 1/65536): the
  // per-element hash of dropout_kernel made this kernel ALU-bound (0.49 of HBM on cfg 4)
  const uint32_t thr = (uint32_t)(p * 65536.0f + 0.5f);
  constexpr int V = 16 / sizeof(T);            // elements per 16-byte access (4 or 8)
  for (long long i = ((long long)blockIdx.x * 256 + threadIdx.x) * V; i < n;
       i += (long long)gridDim.x * 256 * V) {
    if (i + V <= n) {
      uint4 raw = *reinterpret_cast<const uint4*>(x + i);
      T* e = reinterpret_cast<T*>(&raw);
#pragma unroll
      for (int q = 0; q < V / 4; ++q) {
        const uint64_t h = hash_bits(seed, (uint64_t)(i >> 2) + q);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          e[4 * q + k] = from_f<T>(((uint32_t)(h >> (16 * k)) & 0xFFFFu) >= thr
                                       ? to_f(e[4 * q + k]) * scale : 0.f);
      }
      *reinterpret_cast<uint4*>(y + i) = raw;
    } else {
      for (long long j = i; j < n; ++j) {
        const uint64_t h = hash_bits(seed, (uint64_t)(j >> 2));
        y[j] = from_f<T>(((uint32_t)(h >> (16 * (j & 3))) & 0xFFFFu) >= thr ? to_f(x[j]) * scale
                                                                             : 0.f);
      }
    }
  }
}

// Backward of the grouped projection's dropout epilogue, y_g = drop_g(x_g W_g^T + b_g) + pos_g
// (gemm_tc.cu, family 3), for every problem of a group in ONE launch.  Problem g reads its dY
// (M, N) once (ld = row stride: the column slices of a concatenated output are read in place),
// regenerates the mask of the contiguous (M, N) tensor, writes m∘dY as a contiguous bf16 (M, N)
// copy for the weight-gradient / input-gradient GEMMs and adds colsum(m∘dY) to dbias and the
// period-row-sum of the UNMASKED dY (the table is added after the dropout) to dpos.
// CTA = (problem, 64 columns, residue class r of the row period, strip of periods); lanes own
// column pairs, the 8 warps split the strip's rows, partial sums meet in shared memory and reach
// the zero-filled gradient buffer by one atomic add per column and CTA.
constexpr int PDB_MAXP = 64;
struct ProjDropBwdTable {
  const bf16* dy[PDB_MAXP];
  bf16* dym[PDB_MAXP];
  float* dbias[PDB_MAXP];
  float* dpos[PDB_MAXP];
  long long lddy[PDB_MAXP], M[PDB_MAXP], ldpos[PDB_MAXP];
  unsigned long long seed[PDB_MAXP];
  int N[PDB_MAXP], period[PDB_MAXP], per_strip[PDB_MAXP];
  int block_start[PDB_MAXP + 1];
  int count;
};
__global__ void __launch_bounds__(256)
proj_dropout_bwd_kernel(const __grid_constant__ ProjDropBwdTable t, uint32_t thr, float scale,
                        const unsigned long long* __restrict__ step) {
  __shared__ float red[8][4][33];
  pdl_wait();
  pdl_trigger();
  int g = 0;
  while (g + 1 < t.count && (int)blockIdx.x >= t.block_start[g + 1]) ++g;
  const int lane = threadIdx.x & 31, wy = threadIdx.x >> 5;
  const int N = t.N[g], P = t.period[g];
  const int col_chunks = (N + 63) / 64;
  int b = (int)blockIdx.x - t.block_start[g];
  const int chunk = b % col_chunks;
  b /= col_chunks;
  const int r = b % P;                          // residue class of the row period
  const int strip = b / P;
  const long long M = t.M[g], lddy = t.lddy[g];
  const int n = chunk * 64 + 2 * lane;          // lane owns columns n, n + 1 (N is even)
  const uint64_t seed = drop_seed(t.seed[g], step);
  const bf16* __restrict__ dy = t.dy[g];
  bf16* __restrict__ dym = t.dym[g];
  float db0 = 0.f, db1 = 0.f, dp0 = 0.f, dp1 = 0.f;
  if (n < N) {
    const long long n_per = (M - r + P - 1) / P;               // rows m = r + j*P, j < n_per
    const long long j_end = min(n_per, (long long)(strip + 1) * t.per_strip[g]);
    for (long long j = (long long)strip * t.per_strip[g] + wy; j < j_end; j += 8) {
      const long long m = r + j * P;
      const __nv_bfloat162 v = *reinterpret_cast<const __nv_bfloat162*>(dy + m * lddy + n);
      const float v0 = __low2float(v), v1 = __high2float(v);
      const uint64_t i = (uint64_t)m * (uint64_t)N + (uint64_t)n;   // even: i, i+1 share a hash
      const uint64_t h = hash_bits(seed, i >> 2);
      const float m0 = drop_keep(h, i, thr) ? v0 * scale : 0.f;
      const float m1 = drop_keep(h, i + 1, thr) ? v1 * scale : 0.f;
      *reinterpret_cast<__nv_bfloat162*>(dym + m * N + n) = __floats2bfloat162_rn(m0, m1);
      db0 += m0; db1 += m1;
      dp0 += v0; dp1 += v1;
    }
  }
  red[wy][0][lane] = db0; red[wy][1][lane] = db1;
  red[wy][2][lane] = dp0; red[wy][3][lane] = dp1;
  __syncthreads();
  if (wy < 4) {
    const int c = n + (wy & 1);
    float* out = wy < 2 ? t.dbias[g] : t.dpos[g];
    if (out && c < N) {
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) s += red[w][wy][lane];
      atomicAdd(wy < 2 ? out + c : out + (long long)r * t.ldpos[g] + c, s);
    }
  }
}

// several float32 tensors -> bf16 in ONE launch (all bf16 weight shadows of a block)
constexpr int CAST_MAXT = 64;
struct CastTable {
  const float* src[CAST_MAXT];
  bf16* dst[CAST_MAXT];
  long long n[CAST_MAXT];
  int count;
};
__global__ void __launch_bounds__(256) cast_multi_kernel(const __grid_constant__ CastTable t) {
  const int which = blockIdx.y;
  pdl_wait();
  pdl_trigger();
  if (which >= t.count) return;
  const float* __restrict__ s = t.src[which];
  bf16* __restrict__ d = t.dst[which];
  const long long n = t.n[which];
  for (long long i = ((long long)blockIdx.x * 256 + threadIdx.x) * 4; i < n;
       i += (long long)gridDim.x * 1024) {
    if (i + 3 < n) {
      const float4 v = *reinterpret_cast<const float4*>(s + i);
      __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
      uint2 o;
      o.x = *reinterpret_cast<uint32_t*>(&a);
      o.y = *reinterpret_cast<uint32_t*>(&b);
      *reinterpret_cast<uint2*>(d + i) = o;
    } else {
      for (long long j = i; j < n; ++j) d[j] = __float2bfloat16_rn(s[j]);
    }
  }
}

// period 1, bf16, 16-byte aligned rows: lane owns 8 adjacent columns (one uint4 per row), a warp
// covers 256 columns, the 8 warps of a CTA stride over the rows of its strip
__global__ void __launch_bounds__(256)
colsum_bf16_vec_kernel(const bf16* __restrict__ x, int64_t ldx, float* __restrict__ out, int64_t M,
                       int64_t N, int64_t rows_per_cta) {
  __shared__ float red[8][256 + 8];
  const int lane = threadIdx.x & 31, wy = threadIdx.x >> 5;
  pdl_wait();
  pdl_trigger();
  const int64_t n = (int64_t)blockIdx.x * 256 + lane * 8;
  const int64_t r_beg = (int64_t)blockIdx.y * rows_per_cta;
  const int64_t r_end = min(M, r_beg + rows_per_cta);
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
  if (n < N) {
#pragma unroll 4
    for (int64_t m = r_beg + wy; m < r_end; m += 8) {
      const uint4 t = *reinterpret_cast<const uint4*>(x + m * ldx + n);
      const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        acc[2 * i] += __uint_as_float(w[i] << 16);
        acc[2 * i + 1] += __uint_as_float(w[i] & 0xFFFF0000u);
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) red[wy][lane * 8 + j] = acc[j];
  __syncthreads();
  const int64_t c = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (c < N) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += red[i][threadIdx.x];
    atomicAdd(out + c, t);
  }
}

// grouped column sums (the FFN-1 bias gradients of the nine chains of a trunk layer in one launch):
// blockIdx.z selects the problem; same lane / warp layout as colsum_bf16_vec_kernel
constexpr int CS_MAXP = 40;
struct ColsumTable {
  const bf16* x[CS_MAXP];
  float* out[CS_MAXP];
  long long M[CS_MAXP];
};
__global__ void __launch_bounds__(256)
colsum_bf16_vec_grouped_kernel(const __grid_constant__ ColsumTable tb, int64_t N) {
  __shared__ float red[8][256 + 8];
  const int lane = threadIdx.x & 31, wy = threadIdx.x >> 5;
  pdl_wait();
  pdl_trigger();
  const bf16* __restrict__ x = tb.x[blockIdx.z];
  float* __restrict__ out = tb.out[blockIdx.z];
  const int64_t M = tb.M[blockIdx.z];
  const int64_t rows_per_cta = (M + gridDim.y - 1) / gridDim.y;
  const int64_t n = (int64_t)blockIdx.x * 256 + lane * 8;
  const int64_t r_beg = (int64_t)blockIdx.y * rows_per_cta;
  const int64_t r_end = min(M, r_beg + rows_per_cta);
  if (r_beg >= M) return;
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
  if (n < N) {
#pragma unroll 4
    for (int64_t m = r_beg + wy; m < r_end; m += 8) {
      const uint4 t = *reinterpret_cast<const uint4*>(x + m * N + n);
      const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        acc[2 * i] += __uint_as_float(w[i] << 16);
        acc[2 * i + 1] += __uint_as_float(w[i] & 0xFFFF0000u);
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) red[wy][lane * 8 + j] = acc[j];
  __syncthreads();
  const int64_t c = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (c < N) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += red[i][threadIdx.x];
    atomicAdd(out + c, t);
  }
}

// float32 (M, K) matrices with arbitrary leading dimension -> bf16 (M, ldd) with ldd = K rounded up
// to 8 and zero padding: the raw input features (others/realformer.py:307-309 float tensors of
// width 300 / 35 / 74, Ren-MME 768 / 640 / 205) become TMA-legal operands of the tcgen05 GEMM
// (16-byte row stride).  One launch for all modalities / towers: blockIdx.y = tensor.
constexpr int PC_MAXT = 16;
struct PadCastTable {
  const float* src[PC_MAXT];
  bf16* dst[PC_MAXT];
  long long M[PC_MAXT];
  int K[PC_MAXT], lds[PC_MAXT], ldd[PC_MAXT];
};
__global__ void __launch_bounds__(256) cast_pad_kernel(const __grid_constant__ PadCastTable t) {
  const int w = blockIdx.y;
  pdl_wait();
  pdl_trigger();
  const float* __restrict__ s = t.src[w];
  bf16* __restrict__ d = t.dst[w];
  const int K = t.K[w], lds = t.lds[w], ldd = t.ldd[w];
  const int cpr = ldd >> 3;                                 // 8-column chunks per row
  const long long total = t.M[w] * cpr;
  const bool vec = (lds & 3) == 0 && (reinterpret_cast<uintptr_t>(s) & 15) == 0;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total;
       i += (long long)gridDim.x * 256) {
    const long long r = i / cpr;
    const int c0 = (int)(i - r * cpr) * 8;
    const float* sp = s + r * lds + c0;
    float v[8];
    if (vec && c0 + 8 <= K) {
      const float4 a = *reinterpret_cast<const float4*>(sp);
      const float4 b = *reinterpret_cast<const float4*>(sp + 4);
      v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = (c0 + j < K) ? sp[j] : 0.f;
    }
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
      o[j] = *reinterpret_cast<uint32_t*>(&h);
    }
    *reinterpret_cast<uint4*>(d + r * ldd + c0) = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

// out_i = sum of up to 8 equally shaped tensors, for up to 16 outputs in one launch: the gradients
// that flow into ONE activation from several consumers (a modality stream feeds three chains as
// query and three as key/value source: others/realformer.py:232-257) - autograd would add them
// pairwise, one launch per pair.  out may alias its first input.
constexpr int SG_MAXO = 16, SG_MAXI = 8;
struct SumTable {
  void* out[SG_MAXO];
  const void* in[SG_MAXO][SG_MAXI];
  long long n[SG_MAXO];
  int n_in[SG_MAXO];
};
template <typename T>
__global__ void __launch_bounds__(256) sum_grouped_kernel(const __grid_constant__ SumTable t) {
  constexpr int V = 16 / sizeof(T);
  const int w = blockIdx.y;
  pdl_wait();
  pdl_trigger();
  const long long n = t.n[w];
  const int k = t.n_in[w];
  T* __restrict__ out = static_cast<T*>(t.out[w]);
  for (long long i = ((long long)blockIdx.x * 256 + threadIdx.x) * V; i < n;
       i += (long long)gridDim.x * 256 * V) {
    float acc[V];
#pragma unroll
    for (int j = 0; j < V; ++j) acc[j] = 0.f;
    if (i + V <= n) {
      for (int q = 0; q < k; ++q) {
        const uint4 v = *reinterpret_cast<const uint4*>(static_cast<const T*>(t.in[w][q]) + i);
        const T* e = reinterpret_cast<const T*>(&v);
#pragma unroll
        for (int j = 0; j < V; ++j) acc[j] += to_f(e[j]);
      }
      uint4 o;
      T* e = reinterpret_cast<T*>(&o);
#pragma unroll
      for (int j = 0; j < V; ++j) e[j] = from_f<T>(acc[j]);
      *reinterpret_cast<uint4*>(out + i) = o;
    } else {
      for (long long j = i; j < n; ++j) {
        float a = 0.f;
        for (int q = 0; q < k; ++q) a += to_f(static_cast<const T*>(t.in[w][q])[j]);
        out[j] = from_f<T>(a);
      }
    }
  }
}

// launch == false: check the arguments only (every chunk is checked before the first launch)
template <typename T>
int sum_grouped_chunk(int n_out, void* const* out, const int* n_in, const void* const* in,
                      const int64_t* numel, bool launch, cudaStream_t st) {
  if (n_out > SG_MAXO) return MMEMO_ERR_ARG;
  static thread_local SumTable t;
  long long most = 0;
  int pos = 0;
  for (int i = 0; i < n_out; ++i) {
    MM_REQUIRE(out[i] && n_in[i] >= 1 && n_in[i] <= SG_MAXI && numel[i] >= 0);
    MM_REQUIRE((reinterpret_cast<uintptr_t>(out[i]) & 15) == 0);
    t.out[i] = out[i]; t.n[i] = numel[i]; t.n_in[i] = n_in[i];
    for (int q = 0; q < n_in[i]; ++q) {
      MM_REQUIRE(in[pos] && (reinterpret_cast<uintptr_t>(in[pos]) & 15) == 0);
      t.in[i][q] = in[pos++];
    }
    most = numel[i] > most ? numel[i] : most;
  }
  if (!launch || most == 0) return MMEMO_OK;
  long long bx = cdiv(most, 256 * (16 / (long long)sizeof(T)));
  const long long cap = cdiv(148 * 8, n_out);
  if (bx > cap) bx = cap;
  MM_CUDA_OK(mm_launch(sum_grouped_kernel<T>, dim3((unsigned)bx, (unsigned)n_out), dim3(256), 0, st,
                       t));
  return MMEMO_OK;
}

template <typename T>
int sum_grouped(int n_out, void* const* out, const int* n_in, const void* const* in,
                const int64_t* numel, cudaStream_t st) {
  if (n_out <= 0) return MMEMO_OK;
  for (int pass = 0; pass < 2; ++pass) {
    int pos = 0;                 // first input of the chunk in the concatenated `in`
    for (int c = 0; c < n_out; c += SG_MAXO) {
      const int m = n_out - c < SG_MAXO ? n_out - c : SG_MAXO;
      const int rc = sum_grouped_chunk<T>(m, out + c, n_in + c, in + pos, numel + c, pass == 1, st);
      if (rc) return rc;
      for (int i = c; i < c + m; ++i) pos += n_in[i];
    }
  }
  return MMEMO_OK;
}

// mean(x^2) and its gradient (the loss of the encoder benchmark / a plain L2 activation penalty):
// one launch each instead of a cast, a pow, a reduction and their three autograd kernels.
template <typename T>
__global__ void __launch_bounds__(256) sqmean_fwd_kernel(const T* __restrict__ x, long long n,
                                                         float scale, float* __restrict__ out) {
  constexpr int V = 16 / sizeof(T);
  __shared__ float red[8];
  pdl_wait();
  pdl_trigger();
  float acc = 0.f;
  for (long long i = ((long long)blockIdx.x * 256 + threadIdx.x) * V; i < n;
       i += (long long)gridDim.x * 256 * V) {
    if (i + V <= n) {
      const uint4 v = *reinterpret_cast<const uint4*>(x + i);
      const T* e = reinterpret_cast<const T*>(&v);
#pragma unroll
      for (int j = 0; j < V; ++j) acc = fmaf(to_f(e[j]), to_f(e[j]), acc);
    } else {
      for (long long j = i; j < n; ++j) acc = fmaf(to_f(x[j]), to_f(x[j]), acc);
    }
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += red[w];
    atomicAdd(out, t * scale);
  }
}
template <typename T>
__global__ void __launch_bounds__(256) sqmean_bwd_kernel(const T* __restrict__ x,
                                                         const float* __restrict__ dloss,
                                                         long long n, float scale,
                                                         T* __restrict__ dx) {
  constexpr int V = 16 / sizeof(T);
  pdl_wait();
  pdl_trigger();
  const float g = dloss[0] * scale;
  for (long long i = ((long long)blockIdx.x * 256 + threadIdx.x) * V; i < n;
       i += (long long)gridDim.x * 256 * V) {
    if (i + V <= n) {
      const uint4 v = *reinterpret_cast<const uint4*>(x + i);
      const T* e = reinterpret_cast<const T*>(&v);
      uint4 o;
      T* d = reinterpret_cast<T*>(&o);
#pragma unroll
      for (int j = 0; j < V; ++j) d[j] = from_f<T>(g * to_f(e[j]));
      *reinterpret_cast<uint4*>(dx + i) = o;
    } else {
      for (long long j = i; j < n; ++j) dx[j] = from_f<T>(g * to_f(x[j]));
    }
  }
}

template <typename T>
int rowsum(const void* x, int64_t ldx, float* out, int64_t M, int64_t N, int64_t period,
           cudaStream_t st) {
  if (M <= 0 || N <= 0) return MMEMO_OK;
  MM_REQUIRE(x && out && period >= 1);
  if (period > 65535) return MMEMO_ERR_SHAPE;
  if (sizeof(T) == 2 && period == 1 && N % 8 == 0 && ldx % 8 == 0 &&
      reinterpret_cast<uintptr_t>(x) % 16 == 0) {
    const int64_t groups = cdiv(N, 256);
    int64_t strips = cdiv(148 * 2, groups);
    if (strips > cdiv(M, 32)) strips = cdiv(M, 32);
    if (strips < 1) strips = 1;
    const int64_t rows_per_cta = cdiv(M, strips);
    MM_CUDA_OK(mm_launch(colsum_bf16_vec_kernel, dim3((unsigned)groups, (unsigned)strips), dim3(256),
                         0, st, static_cast<const bf16*>(x), ldx, out, M, N, rows_per_cta));
    return MMEMO_OK;
  }
  const int64_t n_per = cdiv(M, period);
  // enough CTAs to fill the machine, at least 64 rows each
  int64_t strips = cdiv(n_per, 64);
  const int64_t base = cdiv(N, 64) * period;
  if (strips * base > 148 * 16) strips = cdiv(148 * 16, base);
  if (strips < 1) strips = 1;
  if (strips > 65535) strips = 65535;
  const int64_t rows_per_cta = cdiv(n_per, strips);
  dim3 grid((unsigned)cdiv(N, 64), (unsigned)strips, (unsigned)period);
  MM_CUDA_OK(mm_launch(rowsum_kernel<T>, grid, dim3(256), 0, st, static_cast<const T*>(x), ldx, out,
                       M, N, period, rows_per_cta));
  return MMEMO_OK;
}

template <typename T>
int dropout_multi_chunk(int n, const void* const* x, void* const* y, const int64_t* numel,
                        const uint64_t* seeds, float p, const uint64_t* step, bool launch,
                        cudaStream_t st) {
  if (n < 1 || n > DROP_MAXT) return MMEMO_ERR_ARG;
  MM_REQUIRE(x && y && numel && seeds && p >= 0.f && p < 1.f);
  DropTable t = {};
  long long nmax = 0;
  for (int i = 0; i < n; ++i) {
    MM_REQUIRE(x[i] && y[i] && numel[i] >= 0);
    if ((reinterpret_cast<uintptr_t>(x[i]) | reinterpret_cast<uintptr_t>(y[i])) & 15)
      return MMEMO_ERR_ARG;
    t.x[i] = x[i]; t.y[i] = y[i]; t.n[i] = numel[i]; t.seed[i] = seeds[i];
    nmax = numel[i] > nmax ? numel[i] : nmax;
  }
  t.count = n;
  if (!launch || nmax == 0) return MMEMO_OK;
  const long long per_block = 256 * (16 / sizeof(T)) * 4;      // four 16-byte accesses per thread
  long long gx = cdiv(nmax, per_block);
  gx = gx > 1184 ? 1184 : gx;                                  // 8 CTAs per SM at most
  MM_CUDA_OK(mm_launch(dropout_multi_kernel<T>, dim3((unsigned)gx, (unsigned)n), dim3(256), 0, st, t,
                       p, 1.0f / (1.0f - p),
                       reinterpret_cast<const unsigned long long*>(step)));
  return MMEMO_OK;
}

template <typename T>
int dropout_multi(int n, const void* const* x, void* const* y, const int64_t* numel,
                  const uint64_t* seeds, float p, const uint64_t* step, cudaStream_t st) {
  if (n < 1) return MMEMO_ERR_ARG;
  MM_REQUIRE(x && y && numel && seeds);
  for (int pass = 0; pass < 2; ++pass)
    for (int c = 0; c < n; c += DROP_MAXT) {
      const int rc = dropout_multi_chunk<T>(n - c < DROP_MAXT ? n - c : DROP_MAXT, x + c, y + c,
                                            numel + c, seeds + c, p, step, pass == 1, st);
      if (rc) return rc;
    }
  return MMEMO_OK;
}

int proj_dropout_bwd_chunk(int n, const void* const* dy, const int64_t* lddy, void* const* dym,
                           const int64_t* M, const int64_t* N, const uint64_t* seeds, float p,
                           const uint64_t* step, float* const* dbias, float* const* dpos,
                           const int64_t* period, const int64_t* ldpos, bool launch,
                           cudaStream_t st) {
  if (n < 1 || n > PDB_MAXP) return MMEMO_ERR_ARG;
  MM_REQUIRE(dy && lddy && dym && M && N && seeds && p >= 0.f && p < 1.f);
  static thread_local ProjDropBwdTable t;
  t = ProjDropBwdTable{};
  long long blocks = 0;
  for (int i = 0; i < n; ++i) {
    MM_REQUIRE(dy[i] && dym[i] && M[i] >= 0 && N[i] > 0 && N[i] % 2 == 0 && lddy[i] >= N[i]);
    MM_REQUIRE(lddy[i] % 2 == 0 && ((reinterpret_cast<uintptr_t>(dy[i]) |
                                     reinterpret_cast<uintptr_t>(dym[i])) & 3) == 0);
    const float* dp = dpos ? dpos[i] : nullptr;
    if (dp) MM_REQUIRE(period && period[i] >= 1 && period[i] <= 65535 && ldpos &&
                       ldpos[i] >= N[i]);
    const int P = dp ? (int)period[i] : 1;
    const long long n_per = cdiv(M[i], (int64_t)P);
    const int per_strip = 64;                       // rows of one residue class per CTA
    const long long strips = n_per > 0 ? cdiv(n_per, (int64_t)per_strip) : 0;
    t.dy[i] = static_cast<const bf16*>(dy[i]);
    t.dym[i] = static_cast<bf16*>(dym[i]);
    t.dbias[i] = dbias ? dbias[i] : nullptr;
    t.dpos[i] = const_cast<float*>(dp);
    t.lddy[i] = lddy[i]; t.M[i] = M[i]; t.ldpos[i] = dp ? ldpos[i] : 0;
    t.seed[i] = seeds[i];
    t.N[i] = (int)N[i]; t.period[i] = P; t.per_strip[i] = per_strip;
    t.block_start[i] = (int)blocks;
    blocks += cdiv(N[i], (int64_t)64) * P * strips;
    if (blocks > (1ll << 30)) return MMEMO_ERR_SHAPE;
  }
  t.block_start[n] = (int)blocks;
  t.count = n;
  if (!launch || blocks == 0) return MMEMO_OK;
  MM_CUDA_OK(mm_launch(proj_dropout_bwd_kernel, dim3((unsigned)blocks), dim3(256), 0, st, t,
                       (uint32_t)(p * 65536.0f + 0.5f), 1.0f / (1.0f - p),
                       reinterpret_cast<const unsigned long long*>(step)));
  return MMEMO_OK;
}

int cast_multi_chunk(int count, const float* const* src, void* const* dst, const int64_t* n,
                     bool launch, cudaStream_t st) {
  if (count > CAST_MAXT) return MMEMO_ERR_ARG;
  static thread_local CastTable t;
  t = CastTable{};
  t.count = count;
  int64_t nmax = 0;
  for (int i = 0; i < count; ++i) {
    MM_REQUIRE(src[i] && dst[i] && n[i] >= 0);
    // 16-byte aligned sources / 8-byte aligned destinations (vector accesses)
    MM_REQUIRE((reinterpret_cast<uintptr_t>(src[i]) & 15) == 0 &&
               (reinterpret_cast<uintptr_t>(dst[i]) & 7) == 0);
    t.src[i] = src[i];
    t.dst[i] = static_cast<bf16*>(dst[i]);
    t.n[i] = n[i];
    nmax = n[i] > nmax ? n[i] : nmax;
  }
  if (!launch) return MMEMO_OK;
  int64_t bx = cdiv(cdiv(nmax, 4), 256);
  if (bx > 148) bx = 148;
  if (bx < 1) bx = 1;
  MM_CUDA_OK(mm_launch(cast_multi_kernel, dim3((unsigned)bx, (unsigned)count), dim3(256), 0, st, t));
  return MMEMO_OK;
}

int colsum_grouped_chunk(int n, const void* const* x, float* const* out, const int64_t* M,
                         int64_t N, bool launch, cudaStream_t st) {
  if (n < 1 || n > CS_MAXP) return MMEMO_ERR_ARG;
  if (N <= 0 || N % 8) return MMEMO_ERR_SHAPE;
  static thread_local ColsumTable tb;
  int64_t mmax = 0;
  for (int i = 0; i < n; ++i) {
    MM_REQUIRE(x[i] && out[i] && M[i] >= 0);
    if (reinterpret_cast<uintptr_t>(x[i]) % 16) return MMEMO_ERR_SHAPE;
    tb.x[i] = static_cast<const bf16*>(x[i]);
    tb.out[i] = out[i];
    tb.M[i] = M[i];
    mmax = M[i] > mmax ? M[i] : mmax;
  }
  if (!launch || mmax == 0) return MMEMO_OK;
  const int64_t groups = cdiv(N, 256);
  // ~6 CTAs of 8 warps per SM over the whole group: with 2 the launch was latency-bound (the
  // nine chains of a trunk layer, N = 192: 36 rows per warp in turn; cfg 1a step 1.335 -> 1.322 ms)
  int64_t strips = cdiv(148 * 6, groups * n);
  if (strips > cdiv(mmax, 32)) strips = cdiv(mmax, 32);
  if (strips < 1) strips = 1;
  MM_CUDA_OK(mm_launch(colsum_bf16_vec_grouped_kernel,
                       dim3((unsigned)groups, (unsigned)strips, (unsigned)n), dim3(256), 0, st, tb,
                       N));
  return MMEMO_OK;
}

template <typename T>
int dropout(const void* x, void* y, int64_t n, float p, uint64_t seed, cudaStream_t st) {
  if (n <= 0) return MMEMO_OK;
  MM_REQUIRE(x && y && p >= 0.f && p < 1.f);
  dropout_kernel<T><<<(unsigned)cdiv(n, 256), 256, 0, st>>>(
      static_cast<const T*>(x), static_cast<T*>(y), n, p, 1.0f / (1.0f - p), seed);
  MM_LAUNCH_OK();
  return MMEMO_OK;
}

}  // namespace

extern "C" {
int mmemo_rowsum_f32(const void* x, int64_t ldx, float* out, int64_t M, int64_t N, int64_t period,
                     mmemo_stream_t s) {
  return rowsum<float>(x, ldx, out, M, N, period, mm_stream(s));
}
int mmemo_rowsum_bf16(const void* x, int64_t ldx, float* out, int64_t M, int64_t N, int64_t period,
                      mmemo_stream_t s) {
  return rowsum<bf16>(x, ldx, out, M, N, period, mm_stream(s));
}
int mmemo_cast_f32_to_bf16(const float* src, void* dst, int64_t n, mmemo_stream_t s) {
  if (n <= 0) return MMEMO_OK;
  MM_REQUIRE(src && dst);
  cast_f2b_kernel<<<(unsigned)cdiv(cdiv(n, 4), 256), 256, 0, mm_stream(s)>>>(
      src, static_cast<bf16*>(dst), n);
  MM_LAUNCH_OK();
  return MMEMO_OK;
}
int mmemo_cast_f32_to_bf16_multi(int count, const float* const* src, void* const* dst,
                                 const int64_t* n, mmemo_stream_t s) {
  if (count <= 0) return MMEMO_OK;
  for (int pass = 0; pass < 2; ++pass)          // check every chunk, then launch them
    for (int c = 0; c < count; c += CAST_MAXT) {
      const int rc = cast_multi_chunk(count - c < CAST_MAXT ? count - c : CAST_MAXT, src + c,
                                      dst + c, n + c, pass == 1, mm_stream(s));
      if (rc) return rc;
    }
  return MMEMO_OK;
}
/* *out (float32, zero-initialised by the caller) += mean(x^2);  dx = dloss * 2 x / n */
int mmemo_sqmean_fwd_bf16(const void* x, int64_t n, float* out, mmemo_stream_t s) {
  if (n <= 0) return MMEMO_OK;
  MM_REQUIRE(x && out && (reinterpret_cast<uintptr_t>(x) & 15) == 0);
  int64_t bx = cdiv(n, 256 * 8);
  if (bx > 148 * 4) bx = 148 * 4;
  MM_CUDA_OK(mm_launch(sqmean_fwd_kernel<bf16>, dim3((unsigned)bx), dim3(256), 0, mm_stream(s),
                       static_cast<const bf16*>(x), (long long)n, 1.0f / (float)n, out));
  return MMEMO_OK;
}
int mmemo_sqmean_fwd_f32(const void* x, int64_t n, float* out, mmemo_stream_t s) {
  if (n <= 0) return MMEMO_OK;
  MM_REQUIRE(x && out && (reinterpret_cast<uintptr_t>(x) & 15) == 0);
  int64_t bx = cdiv(n, 256 * 4);
  if (bx > 148 * 4) bx = 148 * 4;
  MM_CUDA_OK(mm_launch(sqmean_fwd_kernel<float>, dim3((unsigned)bx), dim3(256), 0, mm_stream(s),
                       static_cast<const float*>(x), (long long)n, 1.0f / (float)n, out));
  return MMEMO_OK;
}
int mmemo_sqmean_bwd_bf16(const void* x, const float* dloss, int64_t n, void* dx, mmemo_stream_t s) {
  if (n <= 0) return MMEMO_OK;
  MM_REQUIRE(x && dloss && dx && (reinterpret_cast<uintptr_t>(x) & 15) == 0 &&
             (reinterpret_cast<uintptr_t>(dx) & 15) == 0);
  int64_t bx = cdiv(n, 256 * 8);
  if (bx > 148 * 8) bx = 148 * 8;
  MM_CUDA_OK(mm_launch(sqmean_bwd_kernel<bf16>, dim3((unsigned)bx), dim3(256), 0, mm_stream(s),
                       static_cast<const bf16*>(x), dloss, (long long)n, 2.0f / (float)n,
                       static_cast<bf16*>(dx)));
  return MMEMO_OK;
}
int mmemo_sqmean_bwd_f32(const void* x, const float* dloss, int64_t n, void* dx, mmemo_stream_t s) {
  if (n <= 0) return MMEMO_OK;
  MM_REQUIRE(x && dloss && dx && (reinterpret_cast<uintptr_t>(x) & 15) == 0 &&
             (reinterpret_cast<uintptr_t>(dx) & 15) == 0);
  int64_t bx = cdiv(n, 256 * 4);
  if (bx > 148 * 8) bx = 148 * 8;
  MM_CUDA_OK(mm_launch(sqmean_bwd_kernel<float>, dim3((unsigned)bx), dim3(256), 0, mm_stream(s),
                       static_cast<const float*>(x), dloss, (long long)n, 2.0f / (float)n,
                       static_cast<float*>(dx)));
  return MMEMO_OK;
}
int mmemo_sum_grouped_f32(int n_out, void* const* out, const int* n_in, const void* const* in,
                          const int64_t* numel, mmemo_stream_t s) {
  return sum_grouped<float>(n_out, out, n_in, in, numel, mm_stream(s));
}
int mmemo_sum_grouped_bf16(int n_out, void* const* out, const int* n_in, const void* const* in,
                           const int64_t* numel, mmemo_stream_t s) {
  return sum_grouped<bf16>(n_out, out, n_in, in, numel, mm_stream(s));
}
int mmemo_cast_pad_f32_to_bf16_multi(int count, const float* const* src, const int64_t* lds,
                                     void* const* dst, const int64_t* ldd, const int64_t* M,
                                     const int64_t* K, mmemo_stream_t s) {
  if (count <= 0) return MMEMO_OK;
  if (count > PC_MAXT) return MMEMO_ERR_ARG;
  static thread_local PadCastTable t;
  long long most = 0;
  for (int i = 0; i < count; ++i) {
    MM_REQUIRE(src[i] && dst[i] && M[i] >= 0 && K[i] > 0 && lds[i] >= K[i] && ldd[i] >= K[i]);
    MM_REQUIRE(ldd[i] % 8 == 0 && (reinterpret_cast<uintptr_t>(dst[i]) & 15) == 0);
    t.src[i] = src[i]; t.dst[i] = static_cast<bf16*>(dst[i]);
    t.M[i] = M[i]; t.K[i] = (int)K[i]; t.lds[i] = (int)lds[i]; t.ldd[i] = (int)ldd[i];
    const long long n = M[i] * (ldd[i] / 8);
    most = n > most ? n : most;
  }
  if (most == 0) return MMEMO_OK;
  long long bx = cdiv(most, 256);
  const long long cap = cdiv(148 * 8, count);
  if (bx > cap) bx = cap;
  MM_CUDA_OK(mm_launch(cast_pad_kernel, dim3((unsigned)bx, (unsigned)count), dim3(256), 0,
                       mm_stream(s), t));
  return MMEMO_OK;
}
/* out[i][c] += sum_m x[i][m, c] for n contiguous (M[i], N) bf16 matrices, one launch per CS_MAXP */
int mmemo_colsum_grouped_bf16(int n, const void* const* x, float* const* out, const int64_t* M,
                              int64_t N, mmemo_stream_t s) {
  if (n < 1) return MMEMO_ERR_ARG;
  for (int pass = 0; pass < 2; ++pass)          // check every chunk, then launch them
    for (int c = 0; c < n; c += CS_MAXP) {
      const int rc = colsum_grouped_chunk(n - c < CS_MAXP ? n - c : CS_MAXP, x + c, out + c, M + c,
                                          N, pass == 1, mm_stream(s));
      if (rc) return rc;
    }
  return MMEMO_OK;
}
int mmemo_cast_bf16_to_f32(const void* src, float* dst, int64_t n, mmemo_stream_t s) {
  if (n <= 0) return MMEMO_OK;
  MM_REQUIRE(src && dst);
  cast_b2f_kernel<<<(unsigned)cdiv(n, 256), 256, 0, mm_stream(s)>>>(
      static_cast<const bf16*>(src), dst, n);
  MM_LAUNCH_OK();
  return MMEMO_OK;
}
int mmemo_dropout_f32(const void* x, void* y, int64_t n, float p, uint64_t seed, mmemo_stream_t s) {
  return dropout<float>(x, y, n, p, seed, mm_stream(s));
}
int mmemo_dropout_bf16(const void* x, void* y, int64_t n, float p, uint64_t seed,
                       mmemo_stream_t s) {
  return dropout<bf16>(x, y, n, p, seed, mm_stream(s));
}
int mmemo_dropout_multi_f32(int n, const void* const* x, void* const* y, const int64_t* numel,
                            const uint64_t* seeds, float p, const uint64_t* step,
                            mmemo_stream_t s) {
  return dropout_multi<float>(n, x, y, numel, seeds, p, step, mm_stream(s));
}
int mmemo_dropout_multi_bf16(int n, const void* const* x, void* const* y, const int64_t* numel,
                             const uint64_t* seeds, float p, const uint64_t* step,
                             mmemo_stream_t s) {
  return dropout_multi<bf16>(n, x, y, numel, seeds, p, step, mm_stream(s));
}
int mmemo_proj_dropout_bwd_bf16(int n, const void* const* dy, const int64_t* lddy,
                                void* const* dym, const int64_t* M, const int64_t* N,
                                const uint64_t* seeds, float p, const uint64_t* step,
                                float* const* dbias, float* const* dpos, const int64_t* period,
                                const int64_t* ldpos, mmemo_stream_t s) {
  if (n < 1) return MMEMO_ERR_ARG;
  for (int pass = 0; pass < 2; ++pass)          // check every chunk, then launch them
    for (int c = 0; c < n; c += PDB_MAXP) {
      const int rc = proj_dropout_bwd_chunk(
          n - c < PDB_MAXP ? n - c : PDB_MAXP, dy + c, lddy + c, dym + c, M + c, N + c, seeds + c,
          p, step, dbias ? dbias + c : nullptr, dpos ? dpos + c : nullptr,
          period ? period + c : nullptr, ldpos ? ldpos + c : nullptr, pass == 1, mm_stream(s));
      if (rc) return rc;
    }
  return MMEMO_OK;
}
}

// internal: bias gradient (column sum) used by linear_bwd_w
int mmemo_rowsum_dispatch(int bf16_mode, const void* x, int64_t ldx, float* out, int64_t M,
                          int64_t N, cudaStream_t st) {
  return bf16_mode ? rowsum<bf16>(x, ldx, out, M, N, 1, st) : rowsum<float>(x, ldx, out, M, N, 1, st);
}
