// Inference of an ensemble of k fold models (others/realformer.py:418-420, Ren-MME/run.py:560,
// robot_demo.py:610-615: pred = mean of the members' logits).
//   pool_{fwd,bwd}_multi : the mean || max pooling of many fusion trunks (towers) in one launch,
//                          with argmax and backward for the grouped training of k folds (folds.py)
//   ensemble_head_fwd : every member's classifier linears + head, and the member mean, in one launch
//                       (_members: each member's output as well, for fold_uncertainty)
#include <cooperative_groups.h>
#include <math.h>

#include "pool.cuh"

namespace cg = cooperative_groups;

namespace {

// ---------------------------------------------------------------------------------------------
// Grouped pooling: pool_fwd_kernel / pool_bwd_kernel (pool.cu) for several towers with their own
// batch sizes; blockIdx.z = tower (backward: tower * zsplit + part of the position axis).
constexpr int POOL_MAX_GROUPS = 4;
constexpr int POOL_MAX_SLOTS = 32;
constexpr int POOL_MAX_PTRS = 256;    // segment pointers per launch
constexpr int POOL_MAX_TOWERS = 16;   // towers per launch (fewer when a tower has > 16 segments)

struct PoolMultiTable {
  const void* ptr[POOL_MAX_PTRS];     // [tower][group * n_slots + slot]
  float* out[POOL_MAX_TOWERS];        // forward: pooled output; backward: its gradient
  int32_t* amax[POOL_MAX_TOWERS];     // training forward / backward only
  int B[POOL_MAX_TOWERS];
  int len[POOL_MAX_GROUPS];
  int n_groups, n_slots, total_len;
};

template <typename T, bool WithArg>
__global__ void __launch_bounds__(128)
pool_fwd_multi_kernel(PoolMultiTable tb, int d) {
  const int F = tb.n_slots * d;
  const int f = blockIdx.x * 128 + threadIdx.x;
  const int64_t b = blockIdx.y;
  const int tower = blockIdx.z;
  if (f >= F || b >= tb.B[tower]) return;
  const int slot = f / d, k = f - slot * d;
  float sum, mx;
  int arg;
  pool_column<T, WithArg>(tb.ptr + tower * tb.n_groups * tb.n_slots, tb.len, tb.n_groups,
                          tb.n_slots, b, d, slot, k, sum, mx, &arg);
  float* out = tb.out[tower];
  out[b * 2 * F + f] = sum / (float)tb.total_len;
  out[b * 2 * F + F + f] = mx;
  if (WithArg) tb.amax[tower][b * F + f] = arg;
}

template <typename T>
__global__ void __launch_bounds__(128)
pool_bwd_multi_kernel(PoolMultiTable tb, int d, int zsplit) {
  const int F = tb.n_slots * d;
  const int f = blockIdx.x * 128 + threadIdx.x;
  const int64_t b = blockIdx.y;
  const int tower = blockIdx.z / zsplit, part = blockIdx.z - tower * zsplit;
  if (f >= F || b >= tb.B[tower]) return;
  const int slot = f / d, k = f - slot * d;
  const float* dout = tb.out[tower];
  const float dmean = dout[b * 2 * F + f] / (float)tb.total_len;
  const float dmax = dout[b * 2 * F + F + f];
  const int arg = tb.amax[tower][b * F + f];
  const int per = (tb.total_len + zsplit - 1) / zsplit;
  const int p_beg = part * per, p_end = min(tb.total_len, p_beg + per);
  pool_column_bwd<T>(tb.ptr + tower * tb.n_groups * tb.n_slots, tb.len, tb.n_groups, tb.n_slots,
                     b, d, slot, k, dmean, dmax, arg, p_beg, p_end);
}

// One table per POOL_MAX_TOWERS towers; `bwd` = the backward (out = dout, ptrs = dsegs).
template <typename T>
int pool_multi(bool bwd, int n_towers, const void* const* ptrs, const int64_t* len, int n_groups,
               int n_slots, const int64_t* B, int64_t B_all, int64_t d, float* const* out,
               int32_t* const* amax, cudaStream_t st) {
  MM_REQUIRE(n_towers >= 1 && ptrs && len && out && d > 0);
  if (n_groups < 1 || n_groups > POOL_MAX_GROUPS || n_slots < 1 || n_slots > POOL_MAX_SLOTS)
    return MMEMO_ERR_SHAPE;
  PoolMultiTable tb;
  tb.n_groups = n_groups;
  tb.n_slots = n_slots;
  tb.total_len = 0;
  for (int g = 0; g < n_groups; ++g) {
    MM_REQUIRE(len[g] >= 0);
    tb.len[g] = (int)len[g];
    tb.total_len += (int)len[g];
  }
  MM_REQUIRE(tb.total_len > 0);
  const int segs = n_groups * n_slots;
  for (int t = 0; t < n_towers; ++t) {          // check every tower before the first launch
    MM_REQUIRE(out[t] && (!amax || amax[t]) && (B ? B[t] : B_all) >= 0);
    for (int i = 0; i < segs; ++i) MM_REQUIRE(ptrs[(int64_t)t * segs + i]);
  }
  const int per = POOL_MAX_PTRS / segs < POOL_MAX_TOWERS ? POOL_MAX_PTRS / segs : POOL_MAX_TOWERS;
  const unsigned gx = (unsigned)cdiv((int64_t)n_slots * d, 128);
  for (int t0 = 0; t0 < n_towers; t0 += per) {
    const int n = n_towers - t0 < per ? n_towers - t0 : per;
    int64_t b_max = 0, b_sum = 0;
    for (int t = 0; t < n; ++t) {
      tb.out[t] = out[t0 + t];
      tb.amax[t] = amax ? amax[t0 + t] : nullptr;
      tb.B[t] = (int)(B ? B[t0 + t] : B_all);
      b_max = tb.B[t] > b_max ? tb.B[t] : b_max;
      b_sum += tb.B[t];
      for (int i = 0; i < segs; ++i) tb.ptr[t * segs + i] = ptrs[(int64_t)(t0 + t) * segs + i];
    }
    if (b_max == 0) continue;
    if (!bwd) {
      dim3 grid(gx, (unsigned)b_max, (unsigned)n);
      if (amax) pool_fwd_multi_kernel<T, true><<<grid, 128, 0, st>>>(tb, (int)d);
      else pool_fwd_multi_kernel<T, false><<<grid, 128, 0, st>>>(tb, (int)d);
    } else {
      const int64_t zsplit = pool_bwd_zsplit((int64_t)gx * b_sum, tb.total_len);
      dim3 grid(gx, (unsigned)b_max, (unsigned)(n * zsplit));
      pool_bwd_multi_kernel<T><<<grid, 128, 0, st>>>(tb, (int)d, (int)zsplit);
    }
    MM_LAUNCH_OK();
  }
  return MMEMO_OK;
}

// ---------------------------------------------------------------------------------------------
// Ensemble head.  One cluster of CS CTAs per tile of TS samples; the cluster walks the members of
// the launch in order.  For each member:
//   1. split-K GEMM: CTA `rank` computes, for every row of the tile and every output column,
//      the partial dot product over its F / CS slice of the features (x and weight slices staged
//      through shared memory in chunks of FCH columns) into its own shared buffer;
//   2. cluster barrier;
//   3. the CTA that owns a sample (sample index within the tile % CS == rank) adds the CS
//      partials in rank order through distributed shared memory and runs the head: LN + ReLU +
//      classifier + window recurrence (STATE_TRANSFER) or the bilinear head, and folds the result
//      into y in member order.
// The partial buffers alternate between two halves per member, so one cluster barrier per member
// suffices.  Every sum has a fixed order: no atomics, the same bits on every run.
constexpr int CS = 8;            // CTAs per cluster (split of the feature axis)
constexpr int NT = 256;          // threads per CTA
constexpr int NW = NT / 32;
constexpr int FCH = 32;          // feature columns per staged chunk
constexpr int HEAD_MAX_MEMBERS = 8;
constexpr int HEAD_CMAX = 16;
constexpr int HEAD_DMAX = 1024;
constexpr size_t HEAD_SMEM_MAX = 200 * 1024;

struct HeadTable {
  mmemo_ensemble_member m[HEAD_MAX_MEMBERS];
  int n;
};

struct HeadShape {
  int B, P, F, d, C, TS;
  int R, RX, N;                  // rows of the tile, staged x rows, output columns of the GEMM
  float eps;
};

__host__ __device__ inline size_t head_smem_floats(const HeadShape& s, bool st) {
  size_t n = 2 * (size_t)s.R * s.N + (size_t)(s.RX + s.N) * (FCH + 1);
  if (st) n += (size_t)s.R * 2 * s.C + (size_t)NW * s.d;
  return n;
}

__device__ __forceinline__ float head_sigmoid(float x) { return 1.0f / (1.0f + expf(-x)); }

template <bool ST>
__global__ void __cluster_dims__(CS, 1, 1) __launch_bounds__(NT, 1)
ensemble_head_kernel(HeadTable tb, HeadShape sh, float* __restrict__ y, float* __restrict__ ym,
                     int member0, int n_total) {
  extern __shared__ float sm[];
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int C = sh.C, N = sh.N, R = sh.R, P = sh.P, TS = sh.TS;
  const int s0 = (blockIdx.x / CS) * TS;
  float* part = sm;                                  // [2][R][N]
  float* xs = part + 2 * R * N;                      // [RX][FCH + 1]
  float* ws = xs + sh.RX * (FCH + 1);                // [N][FCH + 1]
  float* og = ws + N * (FCH + 1);                    // ST: [R][2C] classifier outputs
  float* hb = og + R * 2 * C;                        // ST: [NW][d] LayerNorm rows
  const int fs = (sh.F + CS - 1) / CS;
  const int f_beg = rank * fs, f_end = min(sh.F, f_beg + fs);

  for (int mi = 0; mi < tb.n; ++mi) {
    const mmemo_ensemble_member& mb = tb.m[mi];
    float* buf = part + (mi & 1) * R * N;
    for (int p = tid; p < R * N; p += NT) buf[p] = 0.f;
    for (int f0 = f_beg; f0 < f_end; f0 += FCH) {
      const int fl = min(FCH, f_end - f0);
      __syncthreads();                               // previous chunk consumed
      for (int e = tid; e < sh.RX * FCH; e += NT) {
        const int r = e / FCH, c = e - r * FCH;
        float v = 0.f;
        if (c < fl) {
          if (ST) {
            if (s0 + r / P < sh.B) v = mb.x0[((int64_t)s0 * P + r) * mb.ld0 + f0 + c];
          } else if (r < TS) {
            if (s0 + r < sh.B) v = mb.x0[(int64_t)(s0 + r) * mb.ld0 + f0 + c];
          } else if (s0 + r - TS < sh.B) {
            v = mb.x1[(int64_t)(s0 + r - TS) * mb.ld1 + f0 + c];
          }
        }
        xs[r * (FCH + 1) + c] = v;
      }
      for (int e = tid; e < N * FCH; e += NT) {
        const int j = e / FCH, c = e - j * FCH;
        float v = 0.f;
        if (c < fl) v = (ST || j < C) ? mb.w0[(int64_t)j * sh.F + f0 + c]
                                      : mb.w1[(int64_t)(j - C) * sh.F + f0 + c];
        ws[j * (FCH + 1) + c] = v;
      }
      __syncthreads();
      for (int p = tid; p < R * N; p += NT) {
        const int i = p / N, j = p - i * N;
        const float* xr = xs + (ST || j < C ? i : TS + i) * (FCH + 1);
        const float* wr = ws + j * (FCH + 1);
        float acc = buf[p];
#pragma unroll 8
        for (int c = 0; c < FCH; ++c) acc = fmaf(xr[c], wr[c], acc);
        buf[p] = acc;
      }
    }
    cluster.sync();                                  // every rank's partials of this member ready

    const int gm = member0 + mi;                     // member index in the whole ensemble
    const int n_own = rank < TS ? (TS - rank + CS - 1) / CS : 0;   // samples ls = rank + u * CS
    const int off = (mi & 1) * R * N;
    if (ST) {
      const int d = sh.d;
      float* h = hb + warp * d;
      for (int t = warp; t < n_own * P; t += NW) {
        const int u = t / P, p = t - u * P;
        const int ls = rank + u * CS;
        if (s0 + ls >= sh.B) continue;
        const int i = ls * P + p;
        float sum = 0.f;
        for (int j = lane; j < d; j += 32) {
          float v = 0.f;
#pragma unroll
          for (int r = 0; r < CS; ++r) v += cluster.map_shared_rank(part, r)[off + i * N + j];
          v += mb.b0[j];
          h[j] = v;
          sum += v;
        }
        const float mean = warp_sum(sum) / (float)d;
        float var = 0.f;
        for (int j = lane; j < d; j += 32) {
          const float t2 = h[j] - mean;
          var = fmaf(t2, t2, var);
        }
        const float rstd = rsqrtf(warp_sum(var) / (float)d + sh.eps);
        for (int j = lane; j < d; j += 32)
          h[j] = fmaxf((h[j] - mean) * rstd * mb.ln_gamma[j] + mb.ln_beta[j], 0.f);
        __syncwarp();
        if (lane < 2 * C) {
          float o = mb.b_out[lane];
          const float* wq = mb.w_out + (int64_t)lane * d;
          for (int j = 0; j < d; ++j) o = fmaf(wq[j], h[j], o);
          og[t * 2 * C + lane] = o;
        }
        __syncwarp();
      }
      __syncthreads();
      // window recurrence (state_transfer_fwd_kernel, heads.cu): one warp per sample, lane = class
      const bool on = lane < C;
      for (int u = warp; u < n_own; u += NW) {
        const int s = s0 + rank + u * CS;
        if (s >= sh.B) continue;
        float op = 0.f, gp = 0.f;
        for (int p = 0; p < P; ++p) {
          const float* f = og + (u * P + p) * 2 * C;
          float o = on ? f[lane] : 0.f;
          const float g = on ? f[C + lane] : 0.f;
          if (p > 0) {
            float uu = 0.f;
            for (int j = 0; j < C; ++j) {
              const float opj = __shfl_sync(0xffffffffu, op, j);
              if (on) uu = fmaf(opj, mb.trans[j * C + lane], uu);
            }
            const float alpha = head_sigmoid(g + gp);
            o = (1.0f - alpha) * o + alpha * tanhf(uu);
          }
          if (on) {
            const int64_t e = ((int64_t)s * P + p) * C + lane;
            float* yp = y + e;
            float acc = gm == 0 ? o : *yp + o;
            if (gm + 1 == n_total) acc = acc / (float)n_total;
            *yp = acc;
            if (ym) ym[(int64_t)gm * sh.B * P * C + e] = o;
          }
          op = o;
          gp = g;
        }
      }
    } else {
      // bilinear head (bilinear_fwd_kernel, heads.cu): one warp per sample; after the GEMM lane
      // l < C holds last[l] and lane C + l holds this[l]
      for (int u = warp; u < n_own; u += NW) {
        const int ls = rank + u * CS;
        const int s = s0 + ls;
        if (s >= sh.B) continue;
        float v = 0.f;
        if (lane < 2 * C) {
#pragma unroll
          for (int r = 0; r < CS; ++r) v += cluster.map_shared_rank(part, r)[off + ls * N + lane];
        }
        float z = 0.f;
        for (int j = 0; j < C; ++j) {
          const float tj = __shfl_sync(0xffffffffu, v, C + j);
          for (int m = 0; m < C; ++m) {
            const float lm = __shfl_sync(0xffffffffu, v, m);
            if (lane < C) z = fmaf(tj * lm, mb.trans[(j * C + m) * C + lane], z);
          }
        }
        const float mean = warp_sum(lane < C ? z : 0.f) / (float)C;
        const float dlt = lane < C ? z - mean : 0.f;
        const float rstd = rsqrtf(warp_sum(dlt * dlt) / (float)C + sh.eps);
        const float thv = __shfl_sync(0xffffffffu, v, lane < C ? C + lane : 0);
        float cat = lane < C ? thv : 0.f;
        const float ln = lane < C ? dlt * rstd * mb.ln_gamma[lane] + mb.ln_beta[lane] : 0.f;
        const float ln_sh = __shfl_sync(0xffffffffu, ln, lane >= C ? lane - C : 0);
        if (lane >= C && lane < 2 * C) cat = ln_sh;
        float o = lane < C ? mb.b_out[lane] : 0.f;
        for (int i = 0; i < 2 * C; ++i) {
          const float ci = __shfl_sync(0xffffffffu, cat, i);
          if (lane < C) o = fmaf(mb.w_out[lane * 2 * C + i], ci, o);
        }
        if (lane < C) {
          float* yp = y + (int64_t)s * C + lane;
          float acc = gm == 0 ? o : *yp + o;
          if (gm + 1 == n_total) acc = acc / (float)n_total;
          *yp = acc;
          if (ym) ym[((int64_t)gm * sh.B + s) * C + lane] = o;
        }
      }
    }
  }
  cluster.sync();                                    // no CTA leaves while others read its partials
}

bool member_ok(const mmemo_ensemble_member& m, bool st) {
  if (!m.x0 || !m.w0 || !m.ln_gamma || !m.ln_beta || !m.w_out || !m.b_out || !m.trans) return false;
  return st ? m.b0 != nullptr : (m.x1 && m.w1);
}

}  // namespace

extern "C" {
int mmemo_pool_fwd_multi_f32(int n_towers, const void* const* seg_ptrs, const int64_t* group_len,
                             int n_groups, int n_slots, int64_t B, int64_t d, float* const* out,
                             mmemo_stream_t s) {
  return pool_multi<float>(false, n_towers, seg_ptrs, group_len, n_groups, n_slots, nullptr, B, d,
                           out, nullptr, mm_stream(s));
}
int mmemo_pool_fwd_multi_bf16(int n_towers, const void* const* seg_ptrs, const int64_t* group_len,
                              int n_groups, int n_slots, int64_t B, int64_t d, float* const* out,
                              mmemo_stream_t s) {
  return pool_multi<bf16>(false, n_towers, seg_ptrs, group_len, n_groups, n_slots, nullptr, B, d,
                          out, nullptr, mm_stream(s));
}
int mmemo_pool_fwd_multi_arg_f32(int n_towers, const void* const* seg_ptrs,
                                 const int64_t* group_len, int n_groups, int n_slots,
                                 const int64_t* B, int64_t d, float* const* out,
                                 int32_t* const* argmax, mmemo_stream_t s) {
  MM_REQUIRE(B && argmax);
  return pool_multi<float>(false, n_towers, seg_ptrs, group_len, n_groups, n_slots, B, 0, d, out,
                           argmax, mm_stream(s));
}
int mmemo_pool_fwd_multi_arg_bf16(int n_towers, const void* const* seg_ptrs,
                                  const int64_t* group_len, int n_groups, int n_slots,
                                  const int64_t* B, int64_t d, float* const* out,
                                  int32_t* const* argmax, mmemo_stream_t s) {
  MM_REQUIRE(B && argmax);
  return pool_multi<bf16>(false, n_towers, seg_ptrs, group_len, n_groups, n_slots, B, 0, d, out,
                          argmax, mm_stream(s));
}
int mmemo_pool_bwd_multi_f32(int n_towers, const float* const* dout, int32_t* const* argmax,
                             void* const* dseg_ptrs, const int64_t* group_len, int n_groups,
                             int n_slots, const int64_t* B, int64_t d, mmemo_stream_t s) {
  MM_REQUIRE(B && argmax && dout);
  return pool_multi<float>(true, n_towers, const_cast<const void* const*>(dseg_ptrs), group_len,
                           n_groups, n_slots, B, 0, d, const_cast<float* const*>(dout), argmax,
                           mm_stream(s));
}
int mmemo_pool_bwd_multi_bf16(int n_towers, const float* const* dout, int32_t* const* argmax,
                              void* const* dseg_ptrs, const int64_t* group_len, int n_groups,
                              int n_slots, const int64_t* B, int64_t d, mmemo_stream_t s) {
  MM_REQUIRE(B && argmax && dout);
  return pool_multi<bf16>(true, n_towers, const_cast<const void* const*>(dseg_ptrs), group_len,
                          n_groups, n_slots, B, 0, d, const_cast<float* const*>(dout), argmax,
                           mm_stream(s));
}

}  // extern "C"

namespace {
int ensemble_head(int kind, int n_members, const mmemo_ensemble_member* members, int64_t B,
                  int64_t P, int64_t F, int64_t d, int64_t C, float eps, float* y, float* ym,
                  mmemo_stream_t s) {
  MM_REQUIRE(kind == MMEMO_HEAD_BILINEAR || kind == MMEMO_HEAD_STATE_TRANSFER);
  MM_REQUIRE(n_members >= 1 && members && y && B >= 0 && F >= 1);
  const bool st = kind == MMEMO_HEAD_STATE_TRANSFER;
  if (!st) P = 1;
  MM_REQUIRE(P >= 1);
  if (C < 1 || C > HEAD_CMAX || (st && (d < 1 || d > HEAD_DMAX))) return MMEMO_ERR_SHAPE;
  for (int k = 0; k < n_members; ++k) {              // check every member before the first launch
    MM_REQUIRE(member_ok(members[k], st));
    MM_REQUIRE(members[k].ld0 >= F && (st || members[k].ld1 >= F));
  }
  if (B == 0) return MMEMO_OK;
  HeadShape sh;
  sh.B = (int)B; sh.P = (int)P; sh.F = (int)F; sh.d = st ? (int)d : 0; sh.C = (int)C;
  sh.eps = eps;
  sh.N = st ? (int)d : 2 * (int)C;
  // one cluster per TS samples: about 148 / CS clusters, fewer samples per tile when the shared
  // buffers would not fit
  int TS = (int)cdiv(B, 148 / CS);
  size_t smem = 0;
  for (;; TS = (TS + 1) / 2) {
    sh.TS = TS;
    sh.R = st ? TS * (int)P : TS;
    sh.RX = st ? TS * (int)P : 2 * TS;
    smem = head_smem_floats(sh, st) * sizeof(float);
    if (smem <= HEAD_SMEM_MAX) break;
    if (TS == 1) return MMEMO_ERR_SHAPE;
  }
  auto kern = st ? ensemble_head_kernel<true> : ensemble_head_kernel<false>;
  if (smem > 48 * 1024)
    MM_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const unsigned grid = (unsigned)(cdiv(B, TS) * CS);
  HeadTable tb;
  for (int k0 = 0; k0 < n_members; k0 += HEAD_MAX_MEMBERS) {
    tb.n = n_members - k0 < HEAD_MAX_MEMBERS ? n_members - k0 : HEAD_MAX_MEMBERS;
    for (int k = 0; k < tb.n; ++k) tb.m[k] = members[k0 + k];
    kern<<<grid, NT, smem, mm_stream(s)>>>(tb, sh, y, ym, k0, n_members);
    MM_LAUNCH_OK();
  }
  return MMEMO_OK;
}
}  // namespace

extern "C" {
int mmemo_ensemble_head_fwd(int kind, int n_members, const mmemo_ensemble_member* members,
                            int64_t B, int64_t P, int64_t F, int64_t d, int64_t C, float eps,
                            float* y, mmemo_stream_t s) {
  return ensemble_head(kind, n_members, members, B, P, F, d, C, eps, y, nullptr, s);
}
int mmemo_ensemble_head_fwd_members(int kind, int n_members, const mmemo_ensemble_member* members,
                                    int64_t B, int64_t P, int64_t F, int64_t d, int64_t C,
                                    float eps, float* y, float* y_members, mmemo_stream_t s) {
  MM_REQUIRE(y_members);
  return ensemble_head(kind, n_members, members, B, P, F, d, C, eps, y, y_members, s);
}
}
