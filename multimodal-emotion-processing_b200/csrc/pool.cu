// Fusion pooling without materialising the concatenation.
//
// The reference builds x = cat([cat(l_list,2), cat(a_list,2), cat(v_list,2)], 1) and then
// cat([x.mean(1), x.max(1)[0]], 1)  (others/realformer.py:258-262, cmu-mosei/run.py:314-318,
// Ren-MME/run.py:266-270, robot_demo.py:435-439): four concat copies + two reductions.  Here every
// chain output stays where its block wrote it; one kernel walks the segment table.
// Pooling is mask-unaware (padded positions are pooled) exactly like the reference.
#include "pool.cuh"

namespace {

constexpr int MAX_GROUPS = 4;
constexpr int MAX_SLOTS = 32;

struct SegTable {
  const void* ptr[MAX_GROUPS * MAX_SLOTS];
  int len[MAX_GROUPS];
  int n_groups, n_slots, total_len;
};

template <typename T>
__global__ void __launch_bounds__(128)
pool_fwd_kernel(SegTable tb, int64_t B, int d, float* __restrict__ out, int32_t* __restrict__ amax) {
  const int F = tb.n_slots * d;
  const int f = blockIdx.x * 128 + threadIdx.x;
  const int64_t b = blockIdx.y;
  if (f >= F) return;
  const int slot = f / d, k = f - slot * d;
  float sum, mx;
  int arg;
  pool_column<T, true>(tb.ptr, tb.len, tb.n_groups, tb.n_slots, b, d, slot, k, sum, mx, &arg);
  out[b * 2 * F + f] = sum / (float)tb.total_len;
  out[b * 2 * F + F + f] = mx;
  amax[b * F + f] = arg;
}

template <typename T>
__global__ void __launch_bounds__(128)
pool_bwd_kernel(SegTable tb, int64_t B, int d, const float* __restrict__ dout,
                const int32_t* __restrict__ amax) {
  const int F = tb.n_slots * d;
  const int f = blockIdx.x * 128 + threadIdx.x;
  const int64_t b = blockIdx.y;
  if (f >= F) return;
  const int slot = f / d, k = f - slot * d;
  const float dmean = dout[b * 2 * F + f] / (float)tb.total_len;
  const float dmax = dout[b * 2 * F + F + f];
  const int arg = amax[b * F + f];
  // gridDim.z splits the position axis
  const int per = (tb.total_len + gridDim.z - 1) / gridDim.z;
  const int p_beg = blockIdx.z * per, p_end = min(tb.total_len, p_beg + per);
  pool_column_bwd<T>(tb.ptr, tb.len, tb.n_groups, tb.n_slots, b, d, slot, k, dmean, dmax, arg,
                     p_beg, p_end);
}

int make_table(SegTable& tb, const void* const* ptrs, const int64_t* len, int n_groups, int n_slots) {
  if (n_groups < 1 || n_groups > MAX_GROUPS || n_slots < 1 || n_slots > MAX_SLOTS || !ptrs || !len)
    return MMEMO_ERR_SHAPE;
  tb.n_groups = n_groups;
  tb.n_slots = n_slots;
  tb.total_len = 0;
  for (int g = 0; g < n_groups; ++g) {
    tb.len[g] = (int)len[g];
    tb.total_len += (int)len[g];
    for (int s = 0; s < n_slots; ++s) {
      tb.ptr[g * n_slots + s] = ptrs[g * n_slots + s];
      if (!tb.ptr[g * n_slots + s]) return MMEMO_ERR_ARG;
    }
  }
  return tb.total_len > 0 ? MMEMO_OK : MMEMO_ERR_ARG;
}

template <typename T>
int pool_fwd(const void* const* ptrs, const int64_t* len, int n_groups, int n_slots, int64_t B,
             int64_t d, float* out, int32_t* amax, cudaStream_t st) {
  if (B <= 0) return MMEMO_OK;
  MM_REQUIRE(out && amax && d > 0);
  SegTable tb;
  const int rc = make_table(tb, ptrs, len, n_groups, n_slots);
  if (rc) return rc;
  dim3 grid((unsigned)cdiv((int64_t)n_slots * d, 128), (unsigned)B);
  pool_fwd_kernel<T><<<grid, 128, 0, st>>>(tb, B, (int)d, out, amax);
  MM_LAUNCH_OK();
  return MMEMO_OK;
}

template <typename T>
int pool_bwd(const float* dout, const int32_t* amax, void* const* ptrs, const int64_t* len,
             int n_groups, int n_slots, int64_t B, int64_t d, cudaStream_t st) {
  if (B <= 0) return MMEMO_OK;
  MM_REQUIRE(dout && amax && d > 0);
  SegTable tb;
  const int rc = make_table(tb, const_cast<const void* const*>(ptrs), len, n_groups, n_slots);
  if (rc) return rc;
  const int64_t base = cdiv((int64_t)n_slots * d, 128) * B;
  const int64_t zsplit = pool_bwd_zsplit(base, tb.total_len);
  dim3 grid((unsigned)cdiv((int64_t)n_slots * d, 128), (unsigned)B, (unsigned)zsplit);
  pool_bwd_kernel<T><<<grid, 128, 0, st>>>(tb, B, (int)d, dout, amax);
  MM_LAUNCH_OK();
  return MMEMO_OK;
}

}  // namespace

extern "C" {
int mmemo_pool_fwd_f32(const void* const* seg_ptrs, const int64_t* group_len, int n_groups,
                       int n_slots, int64_t B, int64_t d, float* out, int32_t* argmax,
                       mmemo_stream_t s) {
  return pool_fwd<float>(seg_ptrs, group_len, n_groups, n_slots, B, d, out, argmax, mm_stream(s));
}
int mmemo_pool_fwd_bf16(const void* const* seg_ptrs, const int64_t* group_len, int n_groups,
                        int n_slots, int64_t B, int64_t d, float* out, int32_t* argmax,
                        mmemo_stream_t s) {
  return pool_fwd<bf16>(seg_ptrs, group_len, n_groups, n_slots, B, d, out, argmax, mm_stream(s));
}
int mmemo_pool_bwd_f32(const float* dout, const int32_t* argmax, void* const* dseg_ptrs,
                       const int64_t* group_len, int n_groups, int n_slots, int64_t B, int64_t d,
                       mmemo_stream_t s) {
  return pool_bwd<float>(dout, argmax, dseg_ptrs, group_len, n_groups, n_slots, B, d, mm_stream(s));
}
int mmemo_pool_bwd_bf16(const float* dout, const int32_t* argmax, void* const* dseg_ptrs,
                        const int64_t* group_len, int n_groups, int n_slots, int64_t B, int64_t d,
                        mmemo_stream_t s) {
  return pool_bwd<bf16>(dout, argmax, dseg_ptrs, group_len, n_groups, n_slots, B, d, mm_stream(s));
}
}
