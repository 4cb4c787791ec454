// Gated residual + LayerNorm (+ReLU), forward and backward:  y = act( LN(res + gate*x)*gamma + beta )
// Replaces others/realformer.py:207-208,263  cmu-mosei/run.py:261  Ren-MME/run.py:166,213.
//
// HBM-bound kernels (fwd: read res,x, write y; bwd: read dy,res,x, write dres,dx).  One warp per
// row, the row lives in registers, 16-byte vector loads/stores (8 bf16 / 4 fp32 per lane per
// access), statistics by warp shuffles with a two-pass variance.  The backward is a single pass
// (ln_bwd_fused_vec) while a lane owns <= 16 columns (d <= 512); wider rows are split in two so
// that neither part needs many registers:
//   * row kernel   : dz -> dres, dx (+ one atomic per CTA for dgate)
//   * column kernel: dgamma[c] = sum_m dy*xhat, dbeta[c] = sum_m dy — lanes own column pairs, warps
//                    stride over rows, one atomic per column per CTA
// A scalar version (any d <= 1024, any alignment) serves shapes the vector path does not take.
#include "common.cuh"

namespace {

constexpr int LN_WARPS = 8;

template <typename T> struct Vec;
template <> struct Vec<float> {
  static constexpr int N = 4;
  __device__ static void unpack(const uint4& t, float* v) {
    v[0] = __uint_as_float(t.x); v[1] = __uint_as_float(t.y);
    v[2] = __uint_as_float(t.z); v[3] = __uint_as_float(t.w);
  }
  __device__ static void load(const float* p, float* v) {
    const float4 t = *reinterpret_cast<const float4*>(p);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  }
  __device__ static void store(float* p, const float* v) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  }
};
template <> struct Vec<bf16> {
  static constexpr int N = 8;
  __device__ static void unpack(const uint4& t, float* v) {
    const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      v[2 * i] = __uint_as_float(w[i] << 16);
      v[2 * i + 1] = __uint_as_float(w[i] & 0xFFFF0000u);
    }
  }
  __device__ static void load(const bf16* p, float* v) {
    const uint4 t = *reinterpret_cast<const uint4*>(p);
    const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      v[2 * i] = __uint_as_float(w[i] << 16);
      v[2 * i + 1] = __uint_as_float(w[i] & 0xFFFF0000u);
    }
  }
  __device__ static void store(bf16* p, const float* v) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __nv_bfloat162 t = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
      w[i] = *reinterpret_cast<uint32_t*>(&t);
    }
    *reinterpret_cast<uint4*>(p) = make_uint4(w[0], w[1], w[2], w[3]);
  }
};

// ---------------------------------------------------------------------------------------------
// vector kernels: lane owns chunks c = lane + 32*i (i < NCH) of V consecutive columns
// ---------------------------------------------------------------------------------------------
// sum over the LPR-lane group a row lives in (LPR = 32: the whole warp)
template <int LPR>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// (bid, nblk): this CTA's index / the number of CTAs that share the rows of this problem.
// LPR = lanes per row: narrow rows (d <= 128 bf16 / 64 fp32) put 2 or 4 rows in a warp so that the
// lanes are not 60 % idle (d = 96: 12 of 32 lanes busy with one row per warp).  LPR < 32 needs
// NCH == 1.
template <typename T, int NCH, int LPR = 32>
__device__ __forceinline__ void
ln_fwd_vec_body(const T* __restrict__ res, int64_t ldres, const T* __restrict__ x, int64_t ldx,
                const float* __restrict__ gate, const float* __restrict__ gamma,
                const float* __restrict__ beta, T* __restrict__ y, int64_t ldy,
                float* __restrict__ mean_out, float* __restrict__ rstd_out, int64_t M, int d,
                float eps, int relu, unsigned bid, unsigned nblk) {
  constexpr int V = Vec<T>::N;
  constexpr int RPW = 32 / LPR;                 // rows per warp
  const int lane = threadIdx.x & 31;
  const int sub = lane / LPR, l = lane % LPR;
  const float g = gate ? gate[0] : 1.f;
  const int nchunk = d / V;
  float gm[NCH][V], bt[NCH][V];
#pragma unroll
  for (int i = 0; i < NCH; ++i)
    if (l + LPR * i < nchunk) {
      Vec<float>::load(gamma + (l + LPR * i) * V, gm[i]);
      Vec<float>::load(beta + (l + LPR * i) * V, bt[i]);
      if (V == 8) {
        Vec<float>::load(gamma + (l + LPR * i) * V + 4, gm[i] + 4);
        Vec<float>::load(beta + (l + LPR * i) * V + 4, bt[i] + 4);
      }
    }
  for (int64_t row0 = ((int64_t)bid * LN_WARPS + (threadIdx.x >> 5)) * RPW; row0 < M;
       row0 += (int64_t)nblk * LN_WARPS * RPW) {
  const int64_t row = row0 + sub;
  const bool live = row < M;
  float z[NCH][V];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < NCH; ++i) {
    const int c = l + LPR * i;
    if (live && c < nchunk) {
      float xv[V];
      Vec<T>::load(x + row * ldx + c * V, xv);
      if (res) {
        float rv[V];
        Vec<T>::load(res + row * ldres + c * V, rv);
#pragma unroll
        for (int j = 0; j < V; ++j) z[i][j] = g * xv[j] + rv[j];
      } else {
#pragma unroll
        for (int j = 0; j < V; ++j) z[i][j] = g * xv[j];
      }
#pragma unroll
      for (int j = 0; j < V; ++j) sum += z[i][j];
    }
  }
  const float mean = group_sum<LPR>(sum) / (float)d;
  float var = 0.f;
#pragma unroll
  for (int i = 0; i < NCH; ++i)
    if (live && l + LPR * i < nchunk) {
#pragma unroll
      for (int j = 0; j < V; ++j) {
        const float t = z[i][j] - mean;
        var = fmaf(t, t, var);
      }
    }
  const float rstd = rsqrtf(group_sum<LPR>(var) / (float)d + eps);
#pragma unroll
  for (int i = 0; i < NCH; ++i) {
    const int c = l + LPR * i;
    if (live && c < nchunk) {
      float o[V];
#pragma unroll
      for (int j = 0; j < V; ++j) {
        float v = (z[i][j] - mean) * rstd * gm[i][j] + bt[i][j];
        o[j] = relu ? fmaxf(v, 0.f) : v;
      }
      Vec<T>::store(y + row * ldy + c * V, o);
    }
  }
  if (l == 0 && live) {
    if (mean_out) mean_out[row] = mean;
    if (rstd_out) rstd_out[row] = rstd;
  }
  }  // row loop
}

template <typename T, int NCH>
__global__ void __launch_bounds__(LN_WARPS * 32)
ln_fwd_vec(const T* __restrict__ res, int64_t ldres, const T* __restrict__ x, int64_t ldx,
           const float* __restrict__ gate, const float* __restrict__ gamma,
           const float* __restrict__ beta, T* __restrict__ y, int64_t ldy,
           float* __restrict__ mean_out, float* __restrict__ rstd_out, int64_t M, int d, float eps,
           int relu) {
  pdl_wait();
  pdl_trigger();
  ln_fwd_vec_body<T, NCH>(res, ldres, x, ldx, gate, gamma, beta, y, ldy, mean_out, rstd_out, M, d,
                          eps, relu, blockIdx.x, gridDim.x);
}

// Grouped launches: up to LN_MAXP independent problems (the nine chains of a fusion-trunk layer,
// both towers, ...) share one grid; blockIdx.y selects the problem, the CTAs of a column of the
// grid stride over its rows.  Rows are contiguous (leading dimension d).  A call with more
// problems checks all of them, then launches consecutive chunks of LN_MAXP.
constexpr int LN_MAXP = 40;
struct LnProb {
  const void *res, *x, *dy;
  const float *gate, *gamma, *beta;
  void *y, *dres, *dx;
  float *mean, *rstd, *dgate, *dgamma, *dbeta, *dxsum;
  long long M;
};
// cta_start: the CTAs [cta_start[i], cta_start[i+1]) of the one-dimensional grid stride over the
// rows of problem i.  The host hands out CTAs in proportion to the problems' row counts (Ren-MME's
// streams have 40 / 76 / 275 positions: with the same number of CTAs per problem the long
// streams ran 2-7x longer than the short ones) and keeps the backward grid within one wave of
// full-register-file CTAs (n x ceil(148 / n) CTAs used to spill a few CTAs into a second wave,
// doubling the launch: 153 CTAs for the nine chains of a trunk layer).
struct LnTable {
  LnProb p[LN_MAXP];
  int n;
  int cta_start[LN_MAXP + 1];
};
__device__ __forceinline__ int ln_locate(const LnTable& tb, unsigned& bid, unsigned& nblk) {
  int g = 0;
  while (g + 1 < tb.n && (int)blockIdx.x >= tb.cta_start[g + 1]) ++g;
  bid = blockIdx.x - (unsigned)tb.cta_start[g];
  nblk = (unsigned)(tb.cta_start[g + 1] - tb.cta_start[g]);
  return g;
}

template <typename T, int NCH, int LPR>
__global__ void __launch_bounds__(LN_WARPS * 32)
ln_fwd_vec_grouped(const __grid_constant__ LnTable tb, int d, float eps, int relu) {
  unsigned bid, nblk;
  const LnProb& a = tb.p[ln_locate(tb, bid, nblk)];
  pdl_wait();
  pdl_trigger();
  ln_fwd_vec_body<T, NCH, LPR>(static_cast<const T*>(a.res), d, static_cast<const T*>(a.x), d,
                               a.gate, a.gamma, a.beta, static_cast<T*>(a.y), d, a.mean, a.rstd,
                               a.M, d, eps, relu, bid, nblk);
}

template <typename T, int NCH>
__global__ void __launch_bounds__(LN_WARPS * 32)
ln_bwd_row_vec(const T* __restrict__ dy, int64_t lddy, const T* __restrict__ res, int64_t ldres,
               const T* __restrict__ x, int64_t ldx, const float* __restrict__ gate,
               const float* __restrict__ gamma, const T* __restrict__ y, int64_t ldy,
               const float* __restrict__ mean_in, const float* __restrict__ rstd_in,
               T* __restrict__ dres, int64_t lddres, T* __restrict__ dx, int64_t lddx,
               float* __restrict__ dgate, int64_t M, int d, int relu) {
  constexpr int V = Vec<T>::N;
  __shared__ float dgs[LN_WARPS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float g = gate ? gate[0] : 1.f;
  const int nchunk = d / V;
  float dg = 0.f;
  float gm[NCH][V];
#pragma unroll
  for (int i = 0; i < NCH; ++i)
    if (lane + 32 * i < nchunk) {
      Vec<float>::load(gamma + (lane + 32 * i) * V, gm[i]);
      if (V == 8) Vec<float>::load(gamma + (lane + 32 * i) * V + 4, gm[i] + 4);
    }
  for (int64_t row = (int64_t)blockIdx.x * LN_WARPS + warp; row < M;
       row += (int64_t)gridDim.x * LN_WARPS) {
    const float mean = mean_in[row], rstd = rstd_in[row];
    float xh[NCH][V], w[NCH][V], xv[NCH][V];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < NCH; ++i) {
      const int c = lane + 32 * i;
      if (c < nchunk) {
        float dv[V], rv[V];
        Vec<T>::load(x + row * ldx + c * V, xv[i]);
        Vec<T>::load(dy + row * lddy + c * V, dv);
        if (res) Vec<T>::load(res + row * ldres + c * V, rv);
        if (relu) {
          float yv[V];
          Vec<T>::load(y + row * ldy + c * V, yv);
#pragma unroll
          for (int j = 0; j < V; ++j)
            if (!(yv[j] > 0.f)) dv[j] = 0.f;
        }
#pragma unroll
        for (int j = 0; j < V; ++j) {
          const float zz = g * xv[i][j] + (res ? rv[j] : 0.f);
          xh[i][j] = (zz - mean) * rstd;
          w[i][j] = dv[j] * gm[i][j];
          s1 += w[i][j];
          s2 = fmaf(w[i][j], xh[i][j], s2);
        }
      }
    }
    s1 = warp_sum(s1) / (float)d;
    s2 = warp_sum(s2) / (float)d;
#pragma unroll
    for (int i = 0; i < NCH; ++i) {
      const int c = lane + 32 * i;
      if (c < nchunk) {
        float dz[V], gx[V];
#pragma unroll
        for (int j = 0; j < V; ++j) {
          dz[j] = rstd * (w[i][j] - s1 - xh[i][j] * s2);
          gx[j] = g * dz[j];
          dg = fmaf(dz[j], xv[i][j], dg);
        }
        if (dres) Vec<T>::store(dres + row * lddres + c * V, dz);
        Vec<T>::store(dx + row * lddx + c * V, gx);
      }
    }
  }
  if (dgate && gate) {
    dg = warp_sum(dg);
    if (lane == 0) dgs[warp] = dg;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = 0.f;
#pragma unroll
      for (int w2 = 0; w2 < LN_WARPS; ++w2) t += dgs[w2];
      atomicAdd(dgate, t);
    }
  }
}

// Single-pass backward (vector path): one read of dy/res/x, dres/dx written once, and the column
// sums (dgamma, dbeta and optionally dxsum = sum_m dx[m,:], the bias gradient of the layer that
// produced x) accumulated per lane in registers over the warp's rows, then reduced through shared
// memory and added to global memory once per CTA.
constexpr int LNB_WARPS = 16;

// LPR = lanes per row (see ln_fwd_vec_body); LPR < 32 needs NCH == 1 and a staging buffer of
// LNB_WARPS * (32 / LPR) rows.
template <typename T, int NCH, bool DXSUM, int LPR = 32>
__device__ __forceinline__ void
ln_bwd_fused_body(const T* __restrict__ dy, int64_t lddy, const T* __restrict__ res, int64_t ldres,
                  const T* __restrict__ x, int64_t ldx, const float* __restrict__ gate,
                  const float* __restrict__ gamma,
                  const float* __restrict__ mean_in, const float* __restrict__ rstd_in,
                  T* __restrict__ dres, int64_t lddres, T* __restrict__ dx, int64_t lddx,
                  float* __restrict__ dgate, float* __restrict__ dgamma, float* __restrict__ dbeta,
                  float* __restrict__ dxsum, int64_t M, int d, unsigned bid, unsigned nblk) {
  constexpr int V = Vec<T>::N;
  extern __shared__ __align__(16) float ln_sm[];   // gamma [d] | staging [LNB_WARPS][d]
  float* sg = ln_sm;
  float* stage = ln_sm + d;
  __shared__ float dgs[LNB_WARPS];
  constexpr int RPW = 32 / LPR;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int sub = lane / LPR, l = lane % LPR;
  for (int i = threadIdx.x; i < d; i += LNB_WARPS * 32) sg[i] = gamma[i];
  __syncthreads();
  const float g = gate ? gate[0] : 1.f;
  const int nchunk = d / V;
  float dg = 0.f;
  float accg[NCH][V], accb[NCH][V], accx[DXSUM ? NCH : 1][V];
#pragma unroll
  for (int i = 0; i < NCH; ++i)
#pragma unroll
    for (int j = 0; j < V; ++j) {
      accg[i][j] = 0.f;
      accb[i][j] = 0.f;
      if (DXSUM) accx[i][j] = 0.f;
    }
  // the row loop is software-pipelined: the 16-byte vectors of the next row are requested (and
  // held packed) before the current row is reduced, so every warp keeps two rows of loads in flight
  const int64_t rstep = (int64_t)nblk * LNB_WARPS * RPW;
  int64_t row = ((int64_t)bid * LNB_WARPS + warp) * RPW + sub;
  uint4 cur[NCH][3], nxt[NCH][3];
  auto fetch = [&](int64_t r, uint4 (&buf)[NCH][3]) {
#pragma unroll
    for (int i = 0; i < NCH; ++i) {
      const int c = l + LPR * i;
      if (c < nchunk) {
        buf[i][0] = *reinterpret_cast<const uint4*>(x + r * ldx + c * V);
        buf[i][1] = *reinterpret_cast<const uint4*>(dy + r * lddy + c * V);
        if (res) buf[i][2] = *reinterpret_cast<const uint4*>(res + r * ldres + c * V);
      }
    }
  };
  if (row < M) fetch(row, cur);
  for (; row - sub < M; row += rstep) {            // (row - sub: the same trip count for the whole warp)
    const bool live = row < M;
    if (row + rstep < M) fetch(row + rstep, nxt);
    const float mean = live ? mean_in[row] : 0.f, rstd = live ? rstd_in[row] : 0.f;
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < NCH; ++i) {
      const int c = l + LPR * i;
      if (live && c < nchunk) {
        float xv[V], dv[V], rv[V];
        Vec<T>::unpack(cur[i][0], xv);
        Vec<T>::unpack(cur[i][1], dv);
        if (res) Vec<T>::unpack(cur[i][2], rv);
#pragma unroll
        for (int j = 0; j < V; ++j) {
          const float xh = (g * xv[j] + (res ? rv[j] : 0.f) - mean) * rstd;
          const float w = dv[j] * sg[c * V + j];
          s1 += w;
          s2 = fmaf(w, xh, s2);
        }
      }
    }
    s1 = group_sum<LPR>(s1) / (float)d;
    s2 = group_sum<LPR>(s2) / (float)d;
#pragma unroll
    for (int i = 0; i < NCH; ++i) {
      const int c = l + LPR * i;
      if (live && c < nchunk) {
        float xv[V], dv[V], rv[V], dz[V], gx[V];
        Vec<T>::unpack(cur[i][0], xv);
        Vec<T>::unpack(cur[i][1], dv);
        if (res) Vec<T>::unpack(cur[i][2], rv);
#pragma unroll
        for (int j = 0; j < V; ++j) {
          const float xh = (g * xv[j] + (res ? rv[j] : 0.f) - mean) * rstd;
          dz[j] = rstd * (dv[j] * sg[c * V + j] - s1 - xh * s2);
          gx[j] = g * dz[j];
          dg = fmaf(dz[j], xv[j], dg);
          accg[i][j] = fmaf(dv[j], xh, accg[i][j]);
          accb[i][j] += dv[j];
          if (DXSUM) accx[i][j] += gx[j];
        }
        if (dres) Vec<T>::store(dres + row * lddres + c * V, dz);
        Vec<T>::store(dx + row * lddx + c * V, gx);
      }
    }
#pragma unroll
    for (int i = 0; i < NCH; ++i)
#pragma unroll
      for (int k = 0; k < 3; ++k) cur[i][k] = nxt[i][k];
  }
  // column partials: registers -> shared [warp][column] -> one sum per column -> one global atomic
  // per column per CTA; the three quantities take turns in the same staging buffer
  if (dgate && gate) {
    dg = warp_sum(dg);
    if (lane == 0) dgs[warp] = dg;
  }
#pragma unroll
  for (int q = 0; q < (DXSUM ? 3 : 2); ++q) {
    float* out = q == 0 ? dgamma : (q == 1 ? dbeta : dxsum);
    if (q) __syncthreads();
#pragma unroll
    for (int i = 0; i < NCH; ++i) {
      const int c = l + LPR * i;
      if (c < nchunk) {
        float* dst = stage + (warp * RPW + sub) * d + c * V;
#pragma unroll
        for (int j = 0; j < V; j += 4) {
          const float* a = q == 0 ? &accg[i][j] : (q == 1 ? &accb[i][j] : &accx[DXSUM ? i : 0][j]);
          *reinterpret_cast<float4*>(dst + j) = make_float4(a[0], a[1], a[2], a[3]);
        }
      }
    }
    __syncthreads();
    if (out)
      for (int c = threadIdx.x; c < d; c += LNB_WARPS * 32) {
        float t = 0.f;
#pragma unroll
        for (int w2 = 0; w2 < LNB_WARPS * RPW; ++w2) t += stage[w2 * d + c];
        atomicAdd(out + c, t);
      }
  }
  if (dgate && gate && threadIdx.x == 0) {
    float t = 0.f;
#pragma unroll
    for (int w2 = 0; w2 < LNB_WARPS; ++w2) t += dgs[w2];
    atomicAdd(dgate, t);
  }
}

template <typename T, int NCH, bool DXSUM>
__global__ void __launch_bounds__(LNB_WARPS * 32, 1)
ln_bwd_fused_vec(const T* __restrict__ dy, int64_t lddy, const T* __restrict__ res, int64_t ldres,
                 const T* __restrict__ x, int64_t ldx, const float* __restrict__ gate,
                 const float* __restrict__ gamma, const T* __restrict__ y, int64_t ldy,
                 const float* __restrict__ mean_in, const float* __restrict__ rstd_in,
                 T* __restrict__ dres, int64_t lddres, T* __restrict__ dx, int64_t lddx,
                 float* __restrict__ dgate, float* __restrict__ dgamma, float* __restrict__ dbeta,
                 float* __restrict__ dxsum, int64_t M, int d, int relu) {
  pdl_wait();
  pdl_trigger();
  ln_bwd_fused_body<T, NCH, DXSUM>(dy, lddy, res, ldres, x, ldx, gate, gamma, mean_in, rstd_in, dres,
                                   lddres, dx, lddx, dgate, dgamma, dbeta, dxsum, M, d, blockIdx.x,
                                   gridDim.x);
}

template <typename T, int NCH, bool DXSUM, int LPR>
__global__ void __launch_bounds__(LNB_WARPS * 32, 1)
ln_bwd_fused_vec_grouped(const __grid_constant__ LnTable tb, int d) {
  unsigned bid, nblk;
  const LnProb& a = tb.p[ln_locate(tb, bid, nblk)];
  pdl_wait();
  pdl_trigger();
  ln_bwd_fused_body<T, NCH, DXSUM, LPR>(static_cast<const T*>(a.dy), d, static_cast<const T*>(a.res), d,
                                   static_cast<const T*>(a.x), d, a.gate, a.gamma, a.mean, a.rstd,
                                   static_cast<T*>(a.dres), d, static_cast<T*>(a.dx), d, a.dgate,
                                   a.dgamma, a.dbeta, DXSUM ? a.dxsum : nullptr, a.M, d, bid, nblk);
}

// dgamma / dbeta: CTA = (64 columns, strip of rows); lane owns 2 adjacent columns
template <typename T>
__global__ void __launch_bounds__(LN_WARPS * 32)
ln_bwd_col(const T* __restrict__ dy, int64_t lddy, const T* __restrict__ res, int64_t ldres,
           const T* __restrict__ x, int64_t ldx, const float* __restrict__ gate,
           const T* __restrict__ y, int64_t ldy, const float* __restrict__ mean_in,
           const float* __restrict__ rstd_in, float* __restrict__ dgamma,
           float* __restrict__ dbeta, int64_t M, int d, int relu, int64_t rows_per_cta) {
  __shared__ float red[LN_WARPS][4][33];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c0 = blockIdx.x * 64 + lane * 2;
  const float g = gate ? gate[0] : 1.f;
  float ga0 = 0.f, ga1 = 0.f, be0 = 0.f, be1 = 0.f;
  if (c0 < d) {
    const int64_t r_beg = (int64_t)blockIdx.y * rows_per_cta;
    const int64_t r_end = min(M, r_beg + rows_per_cta);
    const bool two = (c0 + 1 < d);
#pragma unroll 4
    for (int64_t m = r_beg + warp; m < r_end; m += LN_WARPS) {
      const float mean = mean_in[m], rstd = rstd_in[m];
      float d0 = to_f(dy[m * lddy + c0]), d1 = two ? to_f(dy[m * lddy + c0 + 1]) : 0.f;
      float z0 = g * to_f(x[m * ldx + c0]), z1 = two ? g * to_f(x[m * ldx + c0 + 1]) : 0.f;
      if (res) {
        z0 += to_f(res[m * ldres + c0]);
        if (two) z1 += to_f(res[m * ldres + c0 + 1]);
      }
      if (relu) {
        if (!(to_f(y[m * ldy + c0]) > 0.f)) d0 = 0.f;
        if (two && !(to_f(y[m * ldy + c0 + 1]) > 0.f)) d1 = 0.f;
      }
      ga0 = fmaf(d0, (z0 - mean) * rstd, ga0);
      ga1 = fmaf(d1, (z1 - mean) * rstd, ga1);
      be0 += d0;
      be1 += d1;
    }
  }
  red[warp][0][lane] = ga0; red[warp][1][lane] = ga1;
  red[warp][2][lane] = be0; red[warp][3][lane] = be1;
  __syncthreads();
  if (warp < 4) {   // warp w reduces quantity w over the LN_WARPS partials
    float t = 0.f;
#pragma unroll
    for (int w2 = 0; w2 < LN_WARPS; ++w2) t += red[w2][warp][lane];
    const int c = c0 + (warp & 1);
    if (c < d) {
      if (warp < 2) { if (dgamma) atomicAdd(dgamma + c, t); }
      else { if (dbeta) atomicAdd(dbeta + c, t); }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// scalar fallback (any alignment): lane owns columns lane, lane+32, ...; NPL = columns per lane
// ---------------------------------------------------------------------------------------------
template <typename T, int NPL>
__global__ void __launch_bounds__(LN_WARPS * 32)
ln_fwd_scalar(const T* __restrict__ res, int64_t ldres, const T* __restrict__ x, int64_t ldx,
              const float* __restrict__ gate, const float* __restrict__ gamma,
              const float* __restrict__ beta, T* __restrict__ y, int64_t ldy,
              float* __restrict__ mean_out, float* __restrict__ rstd_out, int64_t M, int d,
              float eps, int relu) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * LN_WARPS + (threadIdx.x >> 5);
  if (row >= M) return;
  const float g = gate ? gate[0] : 1.f;
  float z[NPL];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < NPL; ++i) {
    z[i] = 0.f;
    const int col = lane + 32 * i;
    if (col < d) {
      float v = g * to_f(x[row * ldx + col]);
      if (res) v += to_f(res[row * ldres + col]);
      z[i] = v;
      sum += v;
    }
  }
  const float mean = warp_sum(sum) / (float)d;
  float var = 0.f;
#pragma unroll
  for (int i = 0; i < NPL; ++i)
    if (lane + 32 * i < d) {
      const float t = z[i] - mean;
      var = fmaf(t, t, var);
    }
  const float rstd = rsqrtf(warp_sum(var) / (float)d + eps);
#pragma unroll
  for (int i = 0; i < NPL; ++i) {
    const int col = lane + 32 * i;
    if (col < d) {
      float v = (z[i] - mean) * rstd * gamma[col] + beta[col];
      if (relu) v = fmaxf(v, 0.f);
      y[row * ldy + col] = from_f<T>(v);
    }
  }
  if (lane == 0) {
    if (mean_out) mean_out[row] = mean;
    if (rstd_out) rstd_out[row] = rstd;
  }
}

template <typename T, int NPL>
__global__ void __launch_bounds__(LN_WARPS * 32)
ln_bwd_row_scalar(const T* __restrict__ dy, int64_t lddy, const T* __restrict__ res, int64_t ldres,
                  const T* __restrict__ x, int64_t ldx, const float* __restrict__ gate,
                  const float* __restrict__ gamma, const T* __restrict__ y, int64_t ldy,
                  const float* __restrict__ mean_in, const float* __restrict__ rstd_in,
                  T* __restrict__ dres, int64_t lddres, T* __restrict__ dx, int64_t lddx,
                  float* __restrict__ dgate, int64_t M, int d, int relu) {
  __shared__ float dgs[LN_WARPS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t row = (int64_t)blockIdx.x * LN_WARPS + warp;
  const float g = gate ? gate[0] : 1.f;
  float dg = 0.f;
  if (row < M) {
    const float mean = mean_in[row], rstd = rstd_in[row];
    float xh[NPL], w[NPL], xv[NPL];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      xh[i] = 0.f; w[i] = 0.f; xv[i] = 0.f;
      const int col = lane + 32 * i;
      if (col < d) {
        xv[i] = to_f(x[row * ldx + col]);
        float zz = g * xv[i];
        if (res) zz += to_f(res[row * ldres + col]);
        xh[i] = (zz - mean) * rstd;
        float dyv = to_f(dy[row * lddy + col]);
        if (relu && !(to_f(y[row * ldy + col]) > 0.f)) dyv = 0.f;
        w[i] = dyv * gamma[col];
        s1 += w[i];
        s2 = fmaf(w[i], xh[i], s2);
      }
    }
    s1 = warp_sum(s1) / (float)d;
    s2 = warp_sum(s2) / (float)d;
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int col = lane + 32 * i;
      if (col < d) {
        const float dz = rstd * (w[i] - s1 - xh[i] * s2);
        if (dres) dres[row * lddres + col] = from_f<T>(dz);
        dx[row * lddx + col] = from_f<T>(g * dz);
        dg = fmaf(dz, xv[i], dg);
      }
    }
  }
  if (dgate && gate) {
    dg = warp_sum(dg);
    if (lane == 0) dgs[warp] = dg;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = 0.f;
      for (int w2 = 0; w2 < LN_WARPS; ++w2) t += dgs[w2];
      atomicAdd(dgate, t);
    }
  }
}

inline bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

template <typename T>
int fwd(const void* res, int64_t ldres, const void* x, int64_t ldx, const float* gate,
        const float* gamma, const float* beta, void* y, int64_t ldy, float* mean, float* rstd,
        int64_t M, int64_t d, float eps, int relu, cudaStream_t st) {
  if (M <= 0) return MMEMO_OK;
  MM_REQUIRE(x && gamma && beta && y && d > 0);
  if (d > 1024) return MMEMO_ERR_SHAPE;
  constexpr int V = Vec<T>::N;
  const T* r = static_cast<const T*>(res);
  const T* xx = static_cast<const T*>(x);
  T* yy = static_cast<T*>(y);
  int64_t grid64 = cdiv(M, LN_WARPS);
  if (grid64 > 148 * 6) grid64 = 148 * 6;       // persistent: 6 CTAs (48 warps) per SM, rows strided
  const unsigned grid = (unsigned)grid64;
  const bool vec = d % V == 0 && ldx % V == 0 && ldy % V == 0 && (!res || ldres % V == 0) &&
                   al16(x) && al16(y) && (!res || al16(res)) && al16(gamma) && al16(beta) &&
                   d / V <= 256;
#define MM_ARGS r, ldres, xx, ldx, gate, gamma, beta, yy, ldy, mean, rstd, M, (int)d, eps, relu
  if (vec) {
    const int nch = (int)cdiv(d / V, 32);
    if (nch <= 1) MM_CUDA_OK(mm_launch(ln_fwd_vec<T, 1>, dim3(grid), dim3(LN_WARPS * 32), 0, st, MM_ARGS));
    else if (nch <= 2) MM_CUDA_OK(mm_launch(ln_fwd_vec<T, 2>, dim3(grid), dim3(LN_WARPS * 32), 0, st, MM_ARGS));
    else if (nch <= 4) MM_CUDA_OK(mm_launch(ln_fwd_vec<T, 4>, dim3(grid), dim3(LN_WARPS * 32), 0, st, MM_ARGS));
    else MM_CUDA_OK(mm_launch(ln_fwd_vec<T, 8>, dim3(grid), dim3(LN_WARPS * 32), 0, st, MM_ARGS));
  } else {
    if (d <= 128) ln_fwd_scalar<T, 4><<<grid, LN_WARPS * 32, 0, st>>>(MM_ARGS);
    else if (d <= 512) ln_fwd_scalar<T, 16><<<grid, LN_WARPS * 32, 0, st>>>(MM_ARGS);
    else ln_fwd_scalar<T, 32><<<grid, LN_WARPS * 32, 0, st>>>(MM_ARGS);
  }
#undef MM_ARGS
  MM_LAUNCH_OK();
  return MMEMO_OK;
}

template <typename T>
int bwd(const void* dy, int64_t lddy, const void* res, int64_t ldres, const void* x, int64_t ldx,
        const float* gate, const float* gamma, const void* y, int64_t ldy, const float* mean,
        const float* rstd, void* dres, int64_t lddres, void* dx, int64_t lddx, float* dgate,
        float* dgamma, float* dbeta, float* dxsum, int64_t M, int64_t d, int relu,
        cudaStream_t st) {
  if (M <= 0) return MMEMO_OK;
  MM_REQUIRE(dy && x && gamma && mean && rstd && dx && d > 0 && (!relu || y));
  if (d > 1024) return MMEMO_ERR_SHAPE;
  constexpr int V = Vec<T>::N;
  const T* dyy = static_cast<const T*>(dy);
  const T* r = static_cast<const T*>(res);
  const T* xx = static_cast<const T*>(x);
  const T* yy = static_cast<const T*>(y);
  T* dr = static_cast<T*>(dres);
  T* dxx = static_cast<T*>(dx);
  int64_t grid64 = cdiv(M, LN_WARPS);
  if (grid64 > 148 * 6) grid64 = 148 * 6;       // persistent: 6 CTAs (48 warps) per SM, rows strided
  const unsigned grid = (unsigned)grid64;
  const bool vec = d % V == 0 && ldx % V == 0 && lddy % V == 0 && lddx % V == 0 &&
                   (!res || ldres % V == 0) && (!dres || lddres % V == 0) &&
                   (!relu || ldy % V == 0) && al16(dy) && al16(x) && al16(dx) &&
                   (!res || al16(res)) && (!dres || al16(dres)) && (!relu || al16(y)) &&
                   al16(gamma) && d / V <= 256;
  if (vec && !relu && (dgamma || dbeta || dxsum) && cdiv(d / V, 32) * V <= 16) {
    // single pass (<= 16 columns per lane keep the accumulators in registers): one persistent
    // 16-warp CTA per SM
    // one full-register-file CTA per SM, rows strided: like the persistent GEMM it honours the
    // stream's SM budget, so that a gradient all-reduce in flight keeps SMs of its own instead of
    // making the last CTAs of this grid wait for it
    const int sb = mm_stream_cfg(st).sm_budget;
    const int64_t sms = (sb > 0 && sb < 148) ? sb : 148;
    int64_t g1 = cdiv(M, LNB_WARPS);
    if (g1 > sms) g1 = sms;
    const int nch = (int)cdiv(d / V, 32);
    const size_t sm_bytes = (1 + LNB_WARPS) * (size_t)d * sizeof(float);   // <= 34 KB
#define MM_FUSED(NCH_)                                                                          \
    do {                                                                                        \
      if (dxsum)                                                                                \
        MM_CUDA_OK(mm_launch(ln_bwd_fused_vec<T, NCH_, true>, dim3((unsigned)g1),                \
                             dim3(LNB_WARPS * 32), sm_bytes, st, dyy, lddy, r, ldres, xx, ldx,  \
                             gate, gamma, yy, ldy, mean, rstd, dr, lddres, dxx, lddx, dgate,    \
                             dgamma, dbeta, dxsum, M, (int)d, relu));                           \
      else                                                                                      \
        MM_CUDA_OK(mm_launch(ln_bwd_fused_vec<T, NCH_, false>, dim3((unsigned)g1),               \
                             dim3(LNB_WARPS * 32), sm_bytes, st, dyy, lddy, r, ldres, xx, ldx,  \
                             gate, gamma, yy, ldy, mean, rstd, dr, lddres, dxx, lddx, dgate,    \
                             dgamma, dbeta, (float*)nullptr, M, (int)d, relu));                 \
    } while (0)
    if (nch <= 1) MM_FUSED(1);
    else if (nch <= 2) MM_FUSED(2);
    else if (V == 4) MM_FUSED(4);
#undef MM_FUSED
    MM_LAUNCH_OK();
    return MMEMO_OK;
  }
#define MM_ARGS dyy, lddy, r, ldres, xx, ldx, gate, gamma, yy, ldy, mean, rstd, dr, lddres, dxx, \
                lddx, dgate, M, (int)d, relu
  if (vec) {
    const int nch = (int)cdiv(d / V, 32);
    if (nch <= 1) ln_bwd_row_vec<T, 1><<<grid, LN_WARPS * 32, 0, st>>>(MM_ARGS);
    else if (nch <= 2) ln_bwd_row_vec<T, 2><<<grid, LN_WARPS * 32, 0, st>>>(MM_ARGS);
    else if (nch <= 4) ln_bwd_row_vec<T, 4><<<grid, LN_WARPS * 32, 0, st>>>(MM_ARGS);
    else ln_bwd_row_vec<T, 8><<<grid, LN_WARPS * 32, 0, st>>>(MM_ARGS);
  } else {
    if (d <= 128) ln_bwd_row_scalar<T, 4><<<grid, LN_WARPS * 32, 0, st>>>(MM_ARGS);
    else if (d <= 512) ln_bwd_row_scalar<T, 16><<<grid, LN_WARPS * 32, 0, st>>>(MM_ARGS);
    else ln_bwd_row_scalar<T, 32><<<grid, LN_WARPS * 32, 0, st>>>(MM_ARGS);
  }
#undef MM_ARGS
  MM_LAUNCH_OK();
  if (dgamma || dbeta) {
    const int64_t col_ctas = cdiv(d, 64);
    int64_t strips = cdiv(148 * 4, col_ctas);
    if (strips > cdiv(M, 4 * LN_WARPS)) strips = cdiv(M, 4 * LN_WARPS);
    if (strips < 1) strips = 1;
    const int64_t rows_per_cta = cdiv(M, strips);
    ln_bwd_col<T><<<dim3((unsigned)col_ctas, (unsigned)strips), LN_WARPS * 32, 0, st>>>(
        dyy, lddy, r, ldres, xx, ldx, gate, yy, ldy, mean, rstd, dgamma, dbeta, M, (int)d, relu,
        rows_per_cta);
    MM_LAUNCH_OK();
  }
  if (dxsum)   // shapes the single-pass kernel does not take: separate column sum of dx
    return sizeof(T) == 2 ? mmemo_rowsum_bf16(dx, lddx, dxsum, M, d, 1, st)
                          : mmemo_rowsum_f32(dx, lddx, dxsum, M, d, 1, st);
  return MMEMO_OK;
}

// CTAs per problem: one each plus a share of the rest proportional to the rows, never more than
// a problem has row groups; returns the grid size (<= total whenever total >= n).
unsigned ln_share_ctas(LnTable& tb, int n, const int64_t* M, int64_t rows_per_cta, int64_t total) {
  int64_t msum = 0;
  for (int i = 0; i < n; ++i) msum += M[i];
  const int64_t spare = total > n ? total - n : 0;
  int at = 0;
  tb.n = n;
  for (int i = 0; i < n; ++i) {
    int64_t c = 1 + (msum > 0 ? spare * M[i] / msum : 0);
    const int64_t useful = cdiv(M[i], rows_per_cta) > 1 ? cdiv(M[i], rows_per_cta) : 1;
    if (c > useful) c = useful;
    tb.cta_start[i] = at;
    at += (int)c;
  }
  tb.cta_start[n] = at;
  return (unsigned)at;
}

// launch == false: check the problems only (every chunk is checked before the first launch)
template <typename T>
int fwd_grouped_chunk(int n, const void* const* res, const void* const* x, const float* const* gate,
                      const float* const* gamma, const float* const* beta, void* const* y,
                      float* const* mean, float* const* rstd, const int64_t* M, int64_t d,
                      float eps, int relu, bool launch, cudaStream_t st) {
  if (n < 1 || n > LN_MAXP) return MMEMO_ERR_ARG;
  constexpr int V = Vec<T>::N;
  if (d <= 0 || d % V || d / V > 256) return MMEMO_ERR_SHAPE;
  static thread_local LnTable tb;
  int64_t mmax = 0;
  for (int i = 0; i < n; ++i) {
    MM_REQUIRE(x[i] && gamma[i] && beta[i] && y[i] && M[i] >= 0);
    if (!al16(x[i]) || !al16(y[i]) || (res && res[i] && !al16(res[i])) || !al16(gamma[i]) ||
        !al16(beta[i]))
      return MMEMO_ERR_SHAPE;
    LnProb& a = tb.p[i];
    a = LnProb{};
    a.res = res ? res[i] : nullptr; a.x = x[i]; a.gate = gate ? gate[i] : nullptr;
    a.gamma = gamma[i]; a.beta = beta[i]; a.y = y[i];
    a.mean = mean ? mean[i] : nullptr; a.rstd = rstd ? rstd[i] : nullptr; a.M = M[i];
    mmax = M[i] > mmax ? M[i] : mmax;
  }
  if (!launch || mmax == 0) return MMEMO_OK;
  // narrow rows share a warp (LPR lanes per row)
  const int nchunk = (int)(d / V);
  const int rpw = nchunk <= 8 ? 4 : (nchunk <= 16 ? 2 : 1);
  const int nch = (int)cdiv(nchunk, 32);
  // the grid is ONE wave of resident CTAs (registers allow 3 ... 8 per SM, by instantiation): the
  // rows are shared out evenly, so CTAs of a partial second wave would finish a whole CTA-time late
#define MM_G(NCH_, LPR_)                                                                          \
  do {                                                                                            \
    static thread_local int occ = 0;                                                              \
    if (!occ) {                                                                                   \
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(                                          \
              &occ, ln_fwd_vec_grouped<T, NCH_, LPR_>, LN_WARPS * 32, 0) != cudaSuccess || occ < 1) \
        occ = 4;                                                                                  \
    }                                                                                             \
    const dim3 grid(ln_share_ctas(tb, n, M, LN_WARPS * rpw, 148 * (int64_t)occ));                 \
    MM_CUDA_OK(mm_launch(ln_fwd_vec_grouped<T, NCH_, LPR_>, grid, dim3(LN_WARPS * 32), 0, st, tb, \
                         (int)d, eps, relu));                                                     \
  } while (0)
  if (rpw == 4) MM_G(1, 8); else if (rpw == 2) MM_G(1, 16);
  else if (nch <= 1) MM_G(1, 32); else if (nch <= 2) MM_G(2, 32); else if (nch <= 4) MM_G(4, 32);
  else MM_G(8, 32);
#undef MM_G
  return MMEMO_OK;
}

template <typename T>
int bwd_grouped_chunk(int n, const void* const* dy, const void* const* res, const void* const* x,
                      const float* const* gate, const float* const* gamma, const float* const* mean,
                      const float* const* rstd, void* const* dres, void* const* dx,
                      float* const* dgate, float* const* dgamma, float* const* dbeta,
                      float* const* dxsum, const int64_t* M, int64_t d, bool launch,
                      cudaStream_t st) {
  if (n < 1 || n > LN_MAXP) return MMEMO_ERR_ARG;
  constexpr int V = Vec<T>::N;
  if (d <= 0 || d % V || cdiv(d / V, 32) * V > 16) return MMEMO_ERR_SHAPE;   // single-pass kernel only
  static thread_local LnTable tb;
  int64_t mmax = 0;
  bool any_dxsum = false;
  for (int i = 0; i < n; ++i) {
    MM_REQUIRE(dy[i] && x[i] && gamma[i] && mean[i] && rstd[i] && dx[i] && M[i] >= 0);
    if (!al16(dy[i]) || !al16(x[i]) || !al16(dx[i]) || (res && res[i] && !al16(res[i])) ||
        (dres && dres[i] && !al16(dres[i])) || !al16(gamma[i]))
      return MMEMO_ERR_SHAPE;
    LnProb& a = tb.p[i];
    a = LnProb{};
    a.dy = dy[i]; a.res = res ? res[i] : nullptr; a.x = x[i]; a.gate = gate ? gate[i] : nullptr;
    a.gamma = gamma[i]; a.mean = const_cast<float*>(mean[i]); a.rstd = const_cast<float*>(rstd[i]);
    a.dres = dres ? dres[i] : nullptr; a.dx = dx[i]; a.dgate = dgate ? dgate[i] : nullptr;
    a.dgamma = dgamma ? dgamma[i] : nullptr; a.dbeta = dbeta ? dbeta[i] : nullptr;
    a.dxsum = dxsum ? dxsum[i] : nullptr; a.M = M[i];
    any_dxsum = any_dxsum || a.dxsum;
    mmax = M[i] > mmax ? M[i] : mmax;
  }
  if (!launch || mmax == 0) return MMEMO_OK;
  // one persistent 16-warp CTA per SM over the whole group (at least one per problem); narrow rows
  // share a warp (LPR lanes per row)
  const int nchunk = (int)(d / V);
  const int rpw = nchunk <= 8 ? 4 : (nchunk <= 16 ? 2 : 1);
  const int sb = mm_stream_cfg(st).sm_budget;
  const int64_t sms = (sb > 0 && sb < 148) ? sb : 148;      // (see ln_bwd_fused_vec's launcher)
  const dim3 grid(ln_share_ctas(tb, n, M, LNB_WARPS * rpw, sms));
  const int nch = (int)cdiv(nchunk, 32);
  const size_t sm_bytes = (1 + LNB_WARPS * rpw) * (size_t)d * sizeof(float);
#define MM_G(NCH_, LPR_)                                                                          \
  do {                                                                                            \
    if (any_dxsum)                                                                                \
      MM_CUDA_OK(mm_launch(ln_bwd_fused_vec_grouped<T, NCH_, true, LPR_>, grid,                   \
                           dim3(LNB_WARPS * 32), sm_bytes, st, tb, (int)d));                      \
    else                                                                                          \
      MM_CUDA_OK(mm_launch(ln_bwd_fused_vec_grouped<T, NCH_, false, LPR_>, grid,                  \
                           dim3(LNB_WARPS * 32), sm_bytes, st, tb, (int)d));                      \
  } while (0)
  if (rpw == 4) MM_G(1, 8); else if (rpw == 2) MM_G(1, 16);
  else if (nch <= 1) MM_G(1, 32); else if (nch <= 2) MM_G(2, 32); else if (V == 4) MM_G(4, 32);
#undef MM_G
  return MMEMO_OK;
}

// an offset into a nullable per-problem host array
template <typename P>
P* at(P* a, int i) { return a ? a + i : nullptr; }

template <typename T>
int fwd_grouped(int n, const void* const* res, const void* const* x, const float* const* gate,
                const float* const* gamma, const float* const* beta, void* const* y,
                float* const* mean, float* const* rstd, const int64_t* M, int64_t d, float eps,
                int relu, cudaStream_t st) {
  if (n < 1) return MMEMO_ERR_ARG;
  for (int pass = 0; pass < 2; ++pass)
    for (int c = 0; c < n; c += LN_MAXP) {
      const int rc = fwd_grouped_chunk<T>(n - c < LN_MAXP ? n - c : LN_MAXP, at(res, c), x + c,
                                          at(gate, c), gamma + c, beta + c, y + c, at(mean, c),
                                          at(rstd, c), M + c, d, eps, relu, pass == 1, st);
      if (rc) return rc;
    }
  return MMEMO_OK;
}

template <typename T>
int bwd_grouped(int n, const void* const* dy, const void* const* res, const void* const* x,
                const float* const* gate, const float* const* gamma, const float* const* mean,
                const float* const* rstd, void* const* dres, void* const* dx, float* const* dgate,
                float* const* dgamma, float* const* dbeta, float* const* dxsum, const int64_t* M,
                int64_t d, cudaStream_t st) {
  if (n < 1) return MMEMO_ERR_ARG;
  for (int pass = 0; pass < 2; ++pass)
    for (int c = 0; c < n; c += LN_MAXP) {
      const int rc = bwd_grouped_chunk<T>(n - c < LN_MAXP ? n - c : LN_MAXP, dy + c, at(res, c),
                                          x + c, at(gate, c), gamma + c, mean + c, rstd + c,
                                          at(dres, c), dx + c, at(dgate, c), at(dgamma, c),
                                          at(dbeta, c), at(dxsum, c), M + c, d, pass == 1, st);
      if (rc) return rc;
    }
  return MMEMO_OK;
}

}  // namespace

extern "C" {
int mmemo_add_ln_fwd_grouped_f32(int n, const void* const* res, const void* const* x,
                                 const float* const* gate, const float* const* gamma,
                                 const float* const* beta, void* const* y, float* const* mean,
                                 float* const* rstd, const int64_t* M, int64_t d, float eps,
                                 int relu, mmemo_stream_t s) {
  return fwd_grouped<float>(n, res, x, gate, gamma, beta, y, mean, rstd, M, d, eps, relu, mm_stream(s));
}
int mmemo_add_ln_fwd_grouped_bf16(int n, const void* const* res, const void* const* x,
                                  const float* const* gate, const float* const* gamma,
                                  const float* const* beta, void* const* y, float* const* mean,
                                  float* const* rstd, const int64_t* M, int64_t d, float eps,
                                  int relu, mmemo_stream_t s) {
  return fwd_grouped<bf16>(n, res, x, gate, gamma, beta, y, mean, rstd, M, d, eps, relu, mm_stream(s));
}
int mmemo_add_ln_bwd_grouped_f32(int n, const void* const* dy, const void* const* res,
                                 const void* const* x, const float* const* gate,
                                 const float* const* gamma, const float* const* mean,
                                 const float* const* rstd, void* const* dres, void* const* dx,
                                 float* const* dgate, float* const* dgamma, float* const* dbeta,
                                 float* const* dxsum, const int64_t* M, int64_t d,
                                 mmemo_stream_t s) {
  return bwd_grouped<float>(n, dy, res, x, gate, gamma, mean, rstd, dres, dx, dgate, dgamma, dbeta,
                            dxsum, M, d, mm_stream(s));
}
int mmemo_add_ln_bwd_grouped_bf16(int n, const void* const* dy, const void* const* res,
                                  const void* const* x, const float* const* gate,
                                  const float* const* gamma, const float* const* mean,
                                  const float* const* rstd, void* const* dres, void* const* dx,
                                  float* const* dgate, float* const* dgamma, float* const* dbeta,
                                  float* const* dxsum, const int64_t* M, int64_t d,
                                  mmemo_stream_t s) {
  return bwd_grouped<bf16>(n, dy, res, x, gate, gamma, mean, rstd, dres, dx, dgate, dgamma, dbeta,
                           dxsum, M, d, mm_stream(s));
}
int mmemo_add_ln_fwd_f32(const void* res, int64_t ldres, const void* x, int64_t ldx,
                         const float* gate, const float* gamma, const float* beta, void* y,
                         int64_t ldy, float* mean, float* rstd, int64_t M, int64_t d, float eps,
                         int relu, mmemo_stream_t s) {
  return fwd<float>(res, ldres, x, ldx, gate, gamma, beta, y, ldy, mean, rstd, M, d, eps, relu,
                    mm_stream(s));
}
int mmemo_add_ln_fwd_bf16(const void* res, int64_t ldres, const void* x, int64_t ldx,
                          const float* gate, const float* gamma, const float* beta, void* y,
                          int64_t ldy, float* mean, float* rstd, int64_t M, int64_t d, float eps,
                          int relu, mmemo_stream_t s) {
  return fwd<bf16>(res, ldres, x, ldx, gate, gamma, beta, y, ldy, mean, rstd, M, d, eps, relu,
                   mm_stream(s));
}
int mmemo_add_ln_bwd_f32(const void* dy, int64_t lddy, const void* res, int64_t ldres,
                         const void* x, int64_t ldx, const float* gate, const float* gamma,
                         const void* y, int64_t ldy, const float* mean, const float* rstd,
                         void* dres, int64_t lddres, void* dx, int64_t lddx, float* dgate,
                         float* dgamma, float* dbeta, float* dxsum, int64_t M, int64_t d,
                         int relu, mmemo_stream_t s) {
  return bwd<float>(dy, lddy, res, ldres, x, ldx, gate, gamma, y, ldy, mean, rstd, dres, lddres,
                    dx, lddx, dgate, dgamma, dbeta, dxsum, M, d, relu, mm_stream(s));
}
int mmemo_add_ln_bwd_bf16(const void* dy, int64_t lddy, const void* res, int64_t ldres,
                          const void* x, int64_t ldx, const float* gate, const float* gamma,
                          const void* y, int64_t ldy, const float* mean, const float* rstd,
                          void* dres, int64_t lddres, void* dx, int64_t lddx, float* dgate,
                          float* dgamma, float* dbeta, float* dxsum, int64_t M, int64_t d,
                          int relu, mmemo_stream_t s) {
  return bwd<bf16>(dy, lddy, res, ldres, x, ldx, gate, gamma, y, ldy, mean, rstd, dres, lddres,
                   dx, lddx, dgate, dgamma, dbeta, dxsum, M, d, relu, mm_stream(s));
}
}
