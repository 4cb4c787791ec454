// Per-sample / per-row bodies of the head and loss kernels, shared by the per-model kernels
// (heads.cu) and the many-fold kernels (folds.cu) so that both produce bitwise equal forwards.
#pragma once
#include <math.h>

#include "common.cuh"

constexpr int HEAD_CMAX = 16;

__device__ __forceinline__ float head_sigmoidf(float x) { return 1.0f / (1.0f + expf(-x)); }
__device__ __forceinline__ float head_logsigmoidf(float x) {
  return fminf(x, 0.f) - log1pf(expf(-fabsf(x)));
}

// ---------------------------------------------------------------------------------------------
// state transfer (others/realformer.py:274-286): one WARP per sample b, lane k owns class k; T is
// the (C x C) transfer matrix in shared memory.
__device__ __forceinline__ void st_fwd_sample(const float* __restrict__ feats, const float* T,
                                              float* __restrict__ out, int b, int P, int C,
                                              int lane) {
  const bool on = lane < C;
  float op = 0.f, gp = 0.f;
  for (int i = 0; i < P; ++i) {
    const float* f = feats + ((int64_t)b * P + i) * 2 * C;
    float o = on ? f[lane] : 0.f;
    const float g = on ? f[C + lane] : 0.f;
    if (i > 0) {
      float u = 0.f;
      for (int j = 0; j < C; ++j) {
        const float opj = __shfl_sync(0xffffffffu, op, j);
        if (on) u = fmaf(opj, T[j * C + lane], u);
      }
      const float alpha = head_sigmoidf(g + gp);
      o = (1.0f - alpha) * o + alpha * tanhf(u);
    }
    if (on) out[((int64_t)b * P + i) * C + lane] = o;
    op = o;
    gp = g;
  }
}

// Backward of one sample; adds the sample's share of dT into dtrans (float atomics, may be null).
__device__ __forceinline__ void st_bwd_sample(const float* __restrict__ dout,
                                              const float* __restrict__ feats, const float* T,
                                              const float* __restrict__ out,
                                              float* __restrict__ dfeats, float* __restrict__ dtrans,
                                              int b, int P, int C, int lane) {
  const bool on = lane < C;
  float cdo = 0.f, cdg = 0.f;          // gradients carried from window i+1 into (o_i, g_i)
  float dTr[HEAD_CMAX];                // column `lane` of dT, rows j
#pragma unroll
  for (int j = 0; j < HEAD_CMAX; ++j) dTr[j] = 0.f;
  for (int i = P - 1; i >= 0; --i) {
    const float* f = feats + ((int64_t)b * P + i) * 2 * C;
    float* df = dfeats + ((int64_t)b * P + i) * 2 * C;
    const float dy = on ? dout[((int64_t)b * P + i) * C + lane] : 0.f;
    const float dtot = dy + cdo;
    if (i > 0) {
      const float fo = on ? f[lane] : 0.f, fg = on ? f[C + lane] : 0.f;
      const float gpv = on ? feats[((int64_t)b * P + i - 1) * 2 * C + C + lane] : 0.f;
      const float op = on ? out[((int64_t)b * P + i - 1) * C + lane] : 0.f;
      float u = 0.f;
      for (int j = 0; j < C; ++j) {
        const float opj = __shfl_sync(0xffffffffu, op, j);
        if (on) u = fmaf(opj, T[j * C + lane], u);
      }
      const float a = head_sigmoidf(fg + gpv);
      const float t0 = tanhf(u);
      const float dgs = dtot * (t0 - fo) * a * (1.0f - a);
      const float du = on ? dtot * a * (1.0f - t0 * t0) : 0.f;
      if (on) {
        df[lane] = dtot * (1.0f - a);
        df[C + lane] = dgs + cdg;
      }
      cdg = dgs;
      // d o_{i-1}[j] = sum_k du[k] T[j][k]  (lane = j);  dT[j][k] += o_{i-1}[j] du[k]  (lane = k)
      float ndo = 0.f;
#pragma unroll
      for (int k = 0; k < HEAD_CMAX; ++k) {
        if (k < C) {
          const float duk = __shfl_sync(0xffffffffu, du, k);
          const float opk = __shfl_sync(0xffffffffu, op, k);
          if (on) ndo = fmaf(duk, T[lane * C + k], ndo);
          dTr[k] = fmaf(opk, du, dTr[k]);
        }
      }
      cdo = ndo;
    } else if (on) {
      df[lane] = dtot;
      df[C + lane] = cdg;
    }
  }
  if (dtrans && on) {
#pragma unroll
    for (int j = 0; j < HEAD_CMAX; ++j)
      if (j < C) atomicAdd(dtrans + j * C + lane, dTr[j]);
  }
}

// ---------------------------------------------------------------------------------------------
// bilinear head (cmu-mosei/run.py:332-339): one warp per sample; lanes < C own output class k (and
// lanes < 2C own concat column i).
__device__ __forceinline__ void bilinear_fwd_sample(
    const float* __restrict__ th, const float* __restrict__ la, const float* __restrict__ T,
    const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ W,
    const float* __restrict__ bias, float* __restrict__ out, float* __restrict__ zsave, int b,
    int C, float eps, int lane) {
  float z = 0.f;
  if (lane < C)
    for (int j = 0; j < C; ++j) {
      const float tj = th[b * C + j];
      for (int m = 0; m < C; ++m) z = fmaf(tj * la[b * C + m], T[(j * C + m) * C + lane], z);
    }
  const float mean = warp_sum(lane < C ? z : 0.f) / (float)C;
  const float dlt = lane < C ? z - mean : 0.f;
  const float rstd = rsqrtf(warp_sum(dlt * dlt) / (float)C + eps);
  // cat[i]: i < C -> this[i]; else LN(z)[i-C]
  float cat = 0.f;
  if (lane < C) cat = th[b * C + lane];
  const float ln = lane < C ? dlt * rstd * gamma[lane] + beta[lane] : 0.f;
  const float ln_sh = __shfl_sync(0xffffffffu, ln, lane >= C ? lane - C : 0);
  if (lane >= C && lane < 2 * C) cat = ln_sh;
  float o = (lane < C) ? bias[lane] : 0.f;
  for (int i = 0; i < 2 * C; ++i) {
    const float ci = __shfl_sync(0xffffffffu, cat, i);
    if (lane < C) o = fmaf(W[lane * 2 * C + i], ci, o);
  }
  if (lane < C) {
    out[b * C + lane] = o;
    zsave[b * C + lane] = z;
  }
}

// The body of one CTA of the bilinear backward (everything except dW).  sm: [copies][C^3] dT |
// [C] dbias | [C] dgamma | [C] dbeta.  copies = 8 (one private dT per warp: plain += by the lane
// that owns class k, no shared-memory atomics - those are CAS loops and made this the longest
// kernel of the rencecps step) when it fits, else 1 (atomics).  The CTA's sums are added to the
// parameter gradients with float atomics.
__device__ __forceinline__ void bilinear_bwd_cta(
    float* sm, const float* __restrict__ dout, const float* __restrict__ th,
    const float* __restrict__ la, const float* __restrict__ T, const float* __restrict__ gamma,
    const float* __restrict__ W, const float* __restrict__ zsave, float* __restrict__ dth,
    float* __restrict__ dla, float* __restrict__ dT, float* __restrict__ dgamma,
    float* __restrict__ dbeta, float* __restrict__ dbias, int B, int C, float eps, int copies,
    int cta, int n_ctas) {
  const int C3 = C * C * C;
  float* sT = sm;
  float* sb = sT + copies * C3;
  float* sg = sb + C;
  float* sbe = sg + C;
  const int nsm = copies * C3 + 3 * C;
  for (int i = threadIdx.x; i < nsm; i += blockDim.x) sm[i] = 0.f;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* myT = sT + (copies > 1 ? warp * C3 : 0);
  for (int b = cta * 8 + warp; b < B; b += n_ctas * 8) {
    const float z = lane < C ? zsave[b * C + lane] : 0.f;
    const float mean = warp_sum(z) / (float)C;
    const float dlt = lane < C ? z - mean : 0.f;
    const float rstd = rsqrtf(warp_sum(dlt * dlt) / (float)C + eps);
    const float zh = dlt * rstd;
    const float dy = lane < C ? dout[b * C + lane] : 0.f;
    const float thv = lane < C ? th[b * C + lane] : 0.f;
    const float lav = lane < C ? la[b * C + lane] : 0.f;
    // dcat[i] = sum_n dy[n] W[n][i]
    float dcat = 0.f;
    for (int n = 0; n < C; ++n) {
      const float dyn = __shfl_sync(0xffffffffu, dy, n);
      if (lane < 2 * C) dcat = fmaf(dyn, W[n * 2 * C + lane], dcat);
    }
    // LN backward on the second half of dcat
    const float dln = __shfl_sync(0xffffffffu, dcat, lane < C ? lane + C : 0);
    const float w = lane < C ? dln * gamma[lane] : 0.f;
    const float m1 = warp_sum(w) / (float)C;
    const float m2 = warp_sum(w * zh) / (float)C;
    const float dz = lane < C ? rstd * (w - m1 - zh * m2) : 0.f;
    if (lane < C) {
      atomicAdd(&sg[lane], dln * zh);
      atomicAdd(&sbe[lane], dln);
      atomicAdd(&sb[lane], dy);
    }
    // d_this[j] = dcat[j] + sum_{m,k} last[m] T[j][m][k] dz[k];  d_last[m] = sum_{j,k} this[j] T dz
    float dthis = (lane < C) ? dcat : 0.f, dlast = 0.f;
    for (int k = 0; k < C; ++k) {
      const float dzk = __shfl_sync(0xffffffffu, dz, k);
      for (int o2 = 0; o2 < C; ++o2) {
        const float l_o = __shfl_sync(0xffffffffu, lav, o2);
        const float t_o = __shfl_sync(0xffffffffu, thv, o2);
        if (lane < C) {
          dthis = fmaf(l_o * dzk, T[(lane * C + o2) * C + k], dthis);  // j = lane, m = o2
          dlast = fmaf(t_o * dzk, T[(o2 * C + lane) * C + k], dlast);  // j = o2, m = lane
        }
      }
    }
    if (lane < C) {
      dth[b * C + lane] = dthis;
      dla[b * C + lane] = dlast;
    }
    // dT[j][m][k] += this[j] last[m] dz[k]   (lane = k)
    for (int j = 0; j < C; ++j) {
      const float tj = __shfl_sync(0xffffffffu, thv, j);
      for (int m = 0; m < C; ++m) {
        const float lm = __shfl_sync(0xffffffffu, lav, m);
        if (lane < C) {
          if (copies > 1) myT[(j * C + m) * C + lane] += tj * lm * dz;
          else atomicAdd(&sT[(j * C + m) * C + lane], tj * lm * dz);
        }
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < C3; i += blockDim.x)
    if (dT) {
      float t = 0.f;
      for (int c = 0; c < copies; ++c) t += sT[c * C3 + i];
      atomicAdd(dT + i, t);
    }
  for (int i = threadIdx.x; i < C; i += blockDim.x) {
    if (dgamma) atomicAdd(dgamma + i, sg[i]);
    if (dbeta) atomicAdd(dbeta + i, sbe[i]);
    if (dbias) atomicAdd(dbias + i, sb[i]);
  }
}

// CTA counts and shared memory of bilinear_bwd_cta for a batch of B samples.
inline int bilinear_bwd_copies(int64_t C) { return C <= 10 ? 8 : 1; }   // 8 x C^3 floats <= 32 KB
inline size_t bilinear_bwd_smem(int64_t C) {
  return sizeof(float) * (bilinear_bwd_copies(C) * C * C * C + 3 * C);
}
__host__ __device__ inline int64_t bilinear_bwd_ctas(int64_t B) {
  const int64_t blocks = (B + 7) / 8;
  return blocks > 32 ? 32 : blocks;
}

// dW[n][i] += sum_{b in [b0, b1)} dy[b][n] cat[b][i] for weight idx = n * 2C + i (one float atomic).
__device__ __forceinline__ void bilinear_dw_strip(const float* __restrict__ dout,
                                                  const float* __restrict__ th,
                                                  const float* __restrict__ zsave,
                                                  const float* __restrict__ gamma,
                                                  const float* __restrict__ beta,
                                                  float* __restrict__ dW, int idx, int b0, int b1,
                                                  int C, float eps) {
  const int n = idx / (2 * C), i = idx - n * 2 * C;
  float acc = 0.f;
  for (int b = b0; b < b1; ++b) {
    float cat;
    if (i < C) {
      cat = th[b * C + i];
    } else {
      float mean = 0.f;
      for (int k = 0; k < C; ++k) mean += zsave[b * C + k];
      mean /= (float)C;
      float var = 0.f;
      for (int k = 0; k < C; ++k) {
        const float t = zsave[b * C + k] - mean;
        var = fmaf(t, t, var);
      }
      const float rstd = rsqrtf(var / (float)C + eps);
      cat = (zsave[b * C + i - C] - mean) * rstd * gamma[i - C] + beta[i - C];
    }
    acc = fmaf(dout[b * C + n], cat, acc);
  }
  atomicAdd(dW + idx, acc);
}

// ---------------------------------------------------------------------------------------------
// circle loss (others/realformer.py:289-298) of row r.
__device__ __forceinline__ void circle_row_stats(const float* __restrict__ s,
                                                 const float* __restrict__ y, int64_t r, int C,
                                                 float& mn, float& mp, float& sn, float& sp) {
  mn = 0.f;
  mp = 0.f;  // the appended zero
  for (int i = 0; i < C; ++i) {
    const float yi = y[r * C + i];
    const float v = (1.0f - 2.0f * yi) * s[r * C + i];
    mn = fmaxf(mn, v - yi * 1e12f);
    mp = fmaxf(mp, v - (1.0f - yi) * 1e12f);
  }
  sn = expf(0.f - mn);
  sp = expf(0.f - mp);
  for (int i = 0; i < C; ++i) {
    const float yi = y[r * C + i];
    const float v = (1.0f - 2.0f * yi) * s[r * C + i];
    sn += expf(v - yi * 1e12f - mn);
    sp += expf(v - (1.0f - yi) * 1e12f - mp);
  }
}

__device__ __forceinline__ float circle_row_loss(const float* __restrict__ s,
                                                 const float* __restrict__ y, int64_t r, int C) {
  float mn, mp, sn, sp;
  circle_row_stats(s, y, r, C, mn, mp, sn, sp);
  return (mn + logf(sn)) + (mp + logf(sp));
}

// ds[r, :] = g * d loss_r / d s[r, :]
__device__ __forceinline__ void circle_row_bwd(float g, const float* __restrict__ s,
                                               const float* __restrict__ y, float* __restrict__ ds,
                                               int64_t r, int C) {
  float mn, mp, sn, sp;
  circle_row_stats(s, y, r, C, mn, mp, sn, sp);
  for (int i = 0; i < C; ++i) {
    const float yi = y[r * C + i];
    const float sg = 1.0f - 2.0f * yi;
    const float v = sg * s[r * C + i];
    const float pn = expf(v - yi * 1e12f - mn) / sn;
    const float pp = expf(v - (1.0f - yi) * 1e12f - mp) / sp;
    ds[r * C + i] = g * sg * (pn + pp);
  }
}

// ---------------------------------------------------------------------------------------------
// R-Drop KL (Ren-MME/run.py:332-334): n = B/2 pairs of rows (2i, 2i+1).  rdrop_kl_cta: one CTA of
// 256 threads writes the scalar; rdrop_kl_bwd_elem: element e = i * C + c of the pairs.
__device__ __forceinline__ void rdrop_kl_cta(const float* __restrict__ s, float* __restrict__ out,
                                             int n, int C) {
  __shared__ float red[8];
  float acc = 0.f;
  for (int e = threadIdx.x; e < n * C; e += 256) {
    const int i = e / C, c = e - i * C;
    const float a = s[(2 * i) * C + c], b = s[(2 * i + 1) * C + c];
    const float la = head_logsigmoidf(a), lb = head_logsigmoidf(b);
    acc += expf(lb) * (lb - la) + expf(la) * (la - lb);
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += red[w];
    out[0] = t / (float)n * 0.5f;
  }
}

__device__ __forceinline__ void rdrop_kl_bwd_elem(const float* __restrict__ dout,
                                                  const float* __restrict__ s,
                                                  float* __restrict__ ds, int e, int n, int C) {
  const int i = e / C, c = e - i * C;
  const float a = s[(2 * i) * C + c], b = s[(2 * i + 1) * C + c];
  const float la = head_logsigmoidf(a), lb = head_logsigmoidf(b);
  const float sa = expf(la), sb = expf(lb);
  const float g = dout[0] * 0.5f / (float)n;
  // d/da [ sb*(lb-la) + sa*(la-lb) ] = -sb*(1-sa) + sa*(1-sa)*(la-lb) + sa*(1-sa)
  ds[(2 * i) * C + c] = g * ((1.0f - sa) * (sa * (la - lb + 1.0f) - sb));
  ds[(2 * i + 1) * C + c] = g * ((1.0f - sb) * (sb * (lb - la + 1.0f) - sa));
}
