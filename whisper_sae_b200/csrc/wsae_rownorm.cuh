// wsae_rownorm.cuh — row arithmetic shared by the kernels that must agree bit for bit:
//   * the final-LayerNorm statistics and formula of wsae_layernorm_rows (extraction) and of
//     wsae_splice_pack / wsae_splice_decode (splicing an SAE back into Whisper);
//   * K0's single-term bf16 row packing (wsae_pack_activations*) and wsae_splice_pack.
// A spliced forward therefore sees exactly the activations extraction wrote to the cache, and K1 gets
// exactly the packed operand the train step would build from them.
#pragma once

#include "wsae_common.cuh"

namespace wsae {

constexpr int kLnMaxPerLane = 128;   // d <= 32 * 128 = 4096

template <typename TIn>
__device__ __forceinline__ float ln_load(const TIn* p, size_t i);
template <>
__device__ __forceinline__ float ln_load<float>(const float* p, size_t i) { return p[i]; }
template <>
__device__ __forceinline__ float ln_load<__nv_bfloat16>(const __nv_bfloat16* p, size_t i) {
  return __bfloat162float(p[i]);
}
template <>
__device__ __forceinline__ float ln_load<__half>(const __half* p, size_t i) { return __half2float(p[i]); }

// fp32 result -> output element, rounded to nearest
__device__ __forceinline__ void ln_store(float* p, float v) { *p = v; }
__device__ __forceinline__ void ln_store(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
__device__ __forceinline__ void ln_store(__half* p, float v) { *p = __float2half_rn(v); }

// Lanes per row element: lane l owns columns j * 32 + l, j < PER.  The launchers pick PER from these
// buckets (ln_per_bucket), and the statistics add in that order, so every caller gets the same mean
// and rstd for the same row.
__host__ __device__ constexpr int ln_per_bucket(int d) {
  return ceil_div(d, 32) <= 4 ? 4 : ceil_div(d, 32) <= 12 ? 12 : ceil_div(d, 32) <= 16 ? 16
       : ceil_div(d, 32) <= 24 ? 24 : ceil_div(d, 32) <= 32 ? 32 : ceil_div(d, 32) <= 40 ? 40
       : ceil_div(d, 32) <= 64 ? 64 : kLnMaxPerLane;
}

// Two-pass mean / biased variance of one row held by a warp: get(j) is the element at column
// j * 32 + lane, 0 beyond d.  rstd = rsqrt(var + eps) (torch.nn.LayerNorm).
template <int PER, typename Get>
__device__ __forceinline__ void ln_moments(Get get, int d, int lane, float eps, float& mean, float& rstd) {
  float sum = 0.f;
#pragma unroll
  for (int j = 0; j < PER; ++j) sum += get(j);
  mean = warp_sum(sum) / static_cast<float>(d);
  float sq = 0.f;
#pragma unroll
  for (int j = 0; j < PER; ++j) {
    const int c = j * 32 + lane;
    const float t = c < d ? get(j) - mean : 0.f;
    sq = fmaf(t, t, sq);
  }
  rstd = rsqrtf(warp_sum(sq) / static_cast<float>(d) + eps);
}

// x = LN(h) for one element, fp32
__device__ __forceinline__ float ln_apply(float v, float mean, float rstd, float g, float b) {
  return (v - mean) * rstd * g + b;
}

// K0, one term: 8 consecutive centred activations (x - b_pre) -> 8 bf16, rounded to nearest
__device__ __forceinline__ uint4 k0_pack8(float4 a, float4 b) {
  __nv_bfloat162 p0 = __floats2bfloat162_rn(a.x, a.y), p1 = __floats2bfloat162_rn(a.z, a.w);
  __nv_bfloat162 p2 = __floats2bfloat162_rn(b.x, b.y), p3 = __floats2bfloat162_rn(b.z, b.w);
  uint4 out;
  out.x = *reinterpret_cast<uint32_t*>(&p0);
  out.y = *reinterpret_cast<uint32_t*>(&p1);
  out.z = *reinterpret_cast<uint32_t*>(&p2);
  out.w = *reinterpret_cast<uint32_t*>(&p3);
  return out;
}

// K0, one term: the first 8 columns of an activation row's bias block (ones against the three
// bias pieces of W')
__device__ __forceinline__ uint4 k0_bias_block8() {
  return make_uint4(0x3F803F80u,    // bf16 1.0, 1.0
                    0x00003F80u,    // bf16 1.0, 0
                    0u, 0u);
}

}  // namespace wsae
