// Fused gradient clipping + Adam / AdamW step over a list of tensors (SURVEY.md §8f-1).
// Replaces  nn.utils.clip_grad_norm_(model.parameters(), CLIP); optimizer.step()
//   others/realformer.py:314-315,342 (Adam)   cmu-mosei/run.py:368-369,398   Ren-MME/run.py:336-337,379
//   rencecps/run.py:175-176,202   robot_demo.py:471-472,502 (AdamW)
// which torch runs as ~5 multi-tensor launches for the norm/clip and ~10 for the update over
// 100-280 small tensors.  Here, for one optimizer or for the k fold optimizers of a cross-validation
// at once: one launch for the squared norms (one per optimizer), one for the update (the clip
// coefficient is computed on the device from the norm, so there is no host sync), per chunk of 96
// tensors.  HBM-bound: reads p, g, m, v and writes p, m, v once (28 B per parameter).
#include "common.cuh"

namespace {

constexpr int OPT_MAXT = 96;

struct NormTable {
  const float* g[OPT_MAXT];
  long long n[OPT_MAXT];
  int slot[OPT_MAXT];       // output slot of each tensor (one per fold / member; 0 for one model)
  int count;
};

struct AdamTable {
  float* p[OPT_MAXT];
  float* g[OPT_MAXT];
  float* m[OPT_MAXT];
  float* v[OPT_MAXT];
  long long n[OPT_MAXT];
  int count;
};

__device__ __forceinline__ float clip_coef(const float* sqnorm, float max_norm) {
  // torch.nn.utils.clip_grad_norm_: coef = max_norm / (total_norm + 1e-6), clamped to 1
  if (!sqnorm) return 1.f;
  const float c = max_norm / (sqrtf(sqnorm[0]) + 1e-6f);
  return c < 1.f ? c : 1.f;
}

__global__ void __launch_bounds__(256) sqnorm_multi_kernel(NormTable t, float* __restrict__ out) {
  __shared__ float red[8];
  const int which = blockIdx.y;
  const float* __restrict__ g = t.g[which];
  const long long n = t.n[which];
  float acc = 0.f;
  const bool vec = (reinterpret_cast<uintptr_t>(g) & 15) == 0;
  if (vec) {
    const long long n4 = n / 4;
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n4;
         i += (long long)gridDim.x * 256) {
      const float4 x = reinterpret_cast<const float4*>(g)[i];
      acc = fmaf(x.x, x.x, acc); acc = fmaf(x.y, x.y, acc);
      acc = fmaf(x.z, x.z, acc); acc = fmaf(x.w, x.w, acc);
    }
    if (blockIdx.x == 0 && threadIdx.x < (int)(n - n4 * 4)) {
      const float x = g[n4 * 4 + threadIdx.x];
      acc = fmaf(x, x, acc);
    }
  } else {
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n;
         i += (long long)gridDim.x * 256)
      acc = fmaf(g[i], g[i], acc);
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float s = threadIdx.x < 8 ? red[threadIdx.x] : 0.f;
    s = warp_sum(s);
    if (threadIdx.x == 0 && s != 0.f) atomicAdd(out + t.slot[which], s);
  }
}

__global__ void __launch_bounds__(256)
scale_multi_kernel(AdamTable t, const float* __restrict__ sqnorm, float max_norm) {
  const float coef = clip_coef(sqnorm, max_norm);
  if (coef == 1.f) return;
  const int which = blockIdx.y;
  float* __restrict__ g = t.g[which];
  const long long n = t.n[which];
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n;
       i += (long long)gridDim.x * 256)
    g[i] *= coef;
}

struct AdamHyper {
  float lr, beta1, beta2, eps, weight_decay;
  float step_size;      // lr / (1 - beta1^t)
  float inv_bc2_sqrt;   // 1 / sqrt(1 - beta2^t)
  float max_norm;
  int decoupled;        // 1: AdamW (p *= 1 - lr*wd), 0: Adam (g += wd*p)
};

__device__ __forceinline__ void adam_one(float& p, float g, float& m, float& v, const AdamHyper& h,
                                         float coef) {
  g *= coef;
  if (h.decoupled) p *= 1.f - h.lr * h.weight_decay;
  else if (h.weight_decay != 0.f) g = fmaf(h.weight_decay, p, g);
  m = fmaf(1.f - h.beta1, g - m, m);                    // lerp(m, g, 1-beta1)
  v = fmaf((1.f - h.beta2) * g, g, v * h.beta2);        // v*beta2 + (1-beta2)*g*g
  const float denom = sqrtf(v) * h.inv_bc2_sqrt + h.eps;
  p -= h.step_size * (m / denom);
}

// tensor `which` of the table: grid-stride over its elements
__device__ __forceinline__ void adam_tensor(const AdamTable& t, int which, const AdamHyper& h,
                                            float coef) {
  float* __restrict__ p = t.p[which];
  const float* __restrict__ g = t.g[which];
  float* __restrict__ m = t.m[which];
  float* __restrict__ v = t.v[which];
  const long long n = t.n[which];
  const bool vec = ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) |
                     reinterpret_cast<uintptr_t>(m) | reinterpret_cast<uintptr_t>(v)) & 15) == 0;
  if (vec) {
    const long long n4 = n / 4;
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n4;
         i += (long long)gridDim.x * 256) {
      float4 pp = reinterpret_cast<float4*>(p)[i];
      const float4 gg = reinterpret_cast<const float4*>(g)[i];
      float4 mm = reinterpret_cast<float4*>(m)[i];
      float4 vv = reinterpret_cast<float4*>(v)[i];
      adam_one(pp.x, gg.x, mm.x, vv.x, h, coef);
      adam_one(pp.y, gg.y, mm.y, vv.y, h, coef);
      adam_one(pp.z, gg.z, mm.z, vv.z, h, coef);
      adam_one(pp.w, gg.w, mm.w, vv.w, h, coef);
      reinterpret_cast<float4*>(p)[i] = pp;
      reinterpret_cast<float4*>(m)[i] = mm;
      reinterpret_cast<float4*>(v)[i] = vv;
    }
    if (blockIdx.x == 0 && threadIdx.x < (int)(n - n4 * 4)) {
      const long long i = n4 * 4 + threadIdx.x;
      adam_one(p[i], g[i], m[i], v[i], h, coef);
    }
  } else {
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n;
         i += (long long)gridDim.x * 256)
      adam_one(p[i], g[i], m[i], v[i], h, coef);
  }
}

// Each tensor carries its own lr, weight decay, bias corrections (its own step count) and the norm
// slot of its optimizer, so one launch serves any number of optimizers (e.g. the k folds).
struct MemberHyper {
  float lr[OPT_MAXT], weight_decay[OPT_MAXT], step_size[OPT_MAXT], inv_bc2_sqrt[OPT_MAXT];
  int slot[OPT_MAXT];
};

__global__ void __launch_bounds__(256)
adam_member_kernel(const __grid_constant__ AdamTable t, const __grid_constant__ MemberHyper mh,
                   AdamHyper h, const float* __restrict__ sqnorm) {
  const int which = blockIdx.y;
  h.lr = mh.lr[which];
  h.weight_decay = mh.weight_decay[which];
  h.step_size = mh.step_size[which];
  h.inv_bc2_sqrt = mh.inv_bc2_sqrt[which];
  adam_tensor(t, which, h, clip_coef(sqnorm ? sqnorm + mh.slot[which] : nullptr, h.max_norm));
}

unsigned grid_x(long long nmax) {
  long long bx = cdiv(cdiv(nmax, 4), 256);
  if (bx > 148 * 2) bx = 148 * 2;
  return (unsigned)(bx < 1 ? 1 : bx);
}

}  // namespace

extern "C" {

int mmemo_grad_sqnorm_multi_f32(int count, const float* const* grads, const int64_t* numel,
                                const int* slot, float* sqnorm_out, mmemo_stream_t s) {
  MM_REQUIRE(count >= 0 && sqnorm_out && (count == 0 || (grads && numel && slot)));
  cudaStream_t st = mm_stream(s);
  for (int i = 0; i < count; ++i) MM_REQUIRE(grads[i] && numel[i] >= 0 && slot[i] >= 0);
  for (int base = 0; base < count; base += OPT_MAXT) {
    NormTable t = {};
    long long nmax = 0;
    t.count = count - base < OPT_MAXT ? count - base : OPT_MAXT;
    for (int i = 0; i < t.count; ++i) {
      t.g[i] = grads[base + i];
      t.n[i] = numel[base + i];
      t.slot[i] = slot[base + i];
      nmax = t.n[i] > nmax ? t.n[i] : nmax;
    }
    sqnorm_multi_kernel<<<dim3(grid_x(nmax), (unsigned)t.count), 256, 0, st>>>(t, sqnorm_out);
    MM_LAUNCH_OK();
  }
  return MMEMO_OK;
}

int mmemo_clip_grads_f32(int count, float* const* grads, const int64_t* numel, const float* sqnorm,
                         float max_norm, mmemo_stream_t s) {
  MM_REQUIRE(count >= 0 && sqnorm && max_norm > 0.f && (count == 0 || (grads && numel)));
  cudaStream_t st = mm_stream(s);
  for (int base = 0; base < count; base += OPT_MAXT) {
    AdamTable t = {};
    long long nmax = 0;
    t.count = count - base < OPT_MAXT ? count - base : OPT_MAXT;
    for (int i = 0; i < t.count; ++i) {
      MM_REQUIRE(grads[base + i]);
      t.g[i] = grads[base + i];
      t.n[i] = numel[base + i];
      nmax = t.n[i] > nmax ? t.n[i] : nmax;
    }
    scale_multi_kernel<<<dim3(grid_x(nmax * 4), (unsigned)t.count), 256, 0, st>>>(t, sqnorm, max_norm);
    MM_LAUNCH_OK();
  }
  return MMEMO_OK;
}

int mmemo_adam_step_multi_f32(int count, float* const* params, const float* const* grads,
                              float* const* exp_avg, float* const* exp_avg_sq, const int64_t* numel,
                              const float* lr, const int64_t* step, const float* weight_decay,
                              const int* slot, float beta1, float beta2, float eps, int decoupled,
                              const float* sqnorm, float max_norm, mmemo_stream_t s) {
  MM_REQUIRE(count >= 0 && (count == 0 || (params && grads && exp_avg && exp_avg_sq && numel && lr &&
                                           step && weight_decay && slot)));
  MM_REQUIRE(!sqnorm || max_norm > 0.f);
  for (int j = 0; j < count; ++j)
    MM_REQUIRE(params[j] && grads[j] && exp_avg[j] && exp_avg_sq[j] && numel[j] >= 0 &&
               step[j] >= 1 && slot[j] >= 0);
  cudaStream_t st = mm_stream(s);
  AdamHyper h = {};
  h.beta1 = beta1; h.beta2 = beta2; h.eps = eps;
  h.max_norm = max_norm;
  h.decoupled = decoupled;
  for (int base = 0; base < count; base += OPT_MAXT) {
    static thread_local AdamTable t;
    static thread_local MemberHyper mh;
    t = AdamTable{};
    long long nmax = 0;
    t.count = count - base < OPT_MAXT ? count - base : OPT_MAXT;
    for (int i = 0; i < t.count; ++i) {
      const int j = base + i;
      t.p[i] = params[j];
      t.g[i] = const_cast<float*>(grads[j]);
      t.m[i] = exp_avg[j];
      t.v[i] = exp_avg_sq[j];
      t.n[i] = numel[j];
      nmax = t.n[i] > nmax ? t.n[i] : nmax;
      // bias corrections in double like torch's Python scalars (1 - beta ** step)
      const double bc1 = 1.0 - pow((double)beta1, (double)step[j]);
      const double bc2 = 1.0 - pow((double)beta2, (double)step[j]);
      mh.lr[i] = lr[j];
      mh.weight_decay[i] = weight_decay[j];
      mh.step_size[i] = (float)((double)lr[j] / bc1);
      mh.inv_bc2_sqrt[i] = (float)(1.0 / sqrt(bc2));
      mh.slot[i] = slot[j];
    }
    adam_member_kernel<<<dim3(grid_x(nmax), (unsigned)t.count), 256, 0, st>>>(t, mh, h, sqnorm);
    MM_LAUNCH_OK();
  }
  return MMEMO_OK;
}

}  // extern "C"
