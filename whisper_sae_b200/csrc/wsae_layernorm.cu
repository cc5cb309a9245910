// wsae_layernorm.cu — row LayerNorm of captured Whisper hidden states, written straight into the
// activation matrix the SAE trains on.
//
// Producer side of the cache format (reference /root/reference/src/whisper_sae/sae/hooks.py):
//   :85-86, :103-104  activation = encoder.layer_norm(hidden_states)   (the model's FINAL LayerNorm,
//                     applied to every hooked layer: "apply layer norm before SAE")
//   :213-230          flatten_activations: [batch, seq, d] -> [batch * seq, d]
// The reference normalises on whatever device the model runs on, copies every hooked tensor to the
// host (.cpu(), :90,107) and concatenates there.  Here one warp normalises one row (two-pass
// mean / variance in registers for d <= 4096, biased variance, eps inside the sqrt - the
// torch.nn.LayerNorm formula) and writes fp32 row `out_row0 + r` of a caller-owned [N, d] device
// matrix, so flatten + concatenate are just the destination offset.
// HBM bound: d * (in_bytes + 4) bytes per row.
#include "wsae_rownorm.cuh"

namespace wsae {

template <typename TIn, typename TOut, int PER>
__global__ void __launch_bounds__(256)
layernorm_rows_kernel(const TIn* __restrict__ x, long long rows, int d, long long in_pitch,
                      const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                      TOut* __restrict__ out, long long out_pitch) {
  const int lane = threadIdx.x & 31;
  const long long row = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const TIn* xr = x + row * in_pitch;
  float v[PER];
#pragma unroll
  for (int j = 0; j < PER; ++j) {
    const int c = j * 32 + lane;
    v[j] = c < d ? ln_load<TIn>(xr, c) : 0.f;
  }
  float mean, rstd;
  ln_moments<PER>([&](int j) { return v[j]; }, d, lane, eps, mean, rstd);
  TOut* orow = out + row * out_pitch;
#pragma unroll
  for (int j = 0; j < PER; ++j) {
    const int c = j * 32 + lane;
    if (c < d) {
      const float g = gamma != nullptr ? gamma[c] : 1.f;
      const float b = beta != nullptr ? beta[c] : 0.f;
      ln_store(orow + c, ln_apply(v[j], mean, rstd, g, b));
    }
  }
}

template <typename TIn, typename TOut>
static int launch_layernorm(const void* x, long long rows, int d, long long in_pitch, const float* gamma,
                            const float* beta, float eps, void* out_v, long long out_pitch,
                            cudaStream_t stream) {
  TOut* out = static_cast<TOut*>(out_v);
  const int warps = 8;
  const unsigned blocks = static_cast<unsigned>((rows + warps - 1) / warps);
  const TIn* xi = static_cast<const TIn*>(x);
  const int per = ln_per_bucket(d);
#define WSAE_LN_CASE(P)                                                                        \
  layernorm_rows_kernel<TIn, TOut, P><<<blocks, warps * 32, 0, stream>>>(xi, rows, d, in_pitch, gamma, \
                                                                   beta, eps, out, out_pitch)
  if (per == 4) WSAE_LN_CASE(4);
  else if (per == 12) WSAE_LN_CASE(12);
  else if (per == 16) WSAE_LN_CASE(16);
  else if (per == 24) WSAE_LN_CASE(24);
  else if (per == 32) WSAE_LN_CASE(32);
  else if (per == 40) WSAE_LN_CASE(40);
  else if (per == 64) WSAE_LN_CASE(64);
  else WSAE_LN_CASE(kLnMaxPerLane);
#undef WSAE_LN_CASE
  return static_cast<int>(cudaGetLastError());
}

}  // namespace wsae

using namespace wsae;

// See include/wsae.h.  in_dtype / out_dtype: 0 = float32, 1 = bfloat16, 2 = float16.
extern "C" int wsae_layernorm_rows_typed(const void* x, int in_dtype, long long rows, int d,
                                         long long in_pitch_elems, const float* gamma, const float* beta,
                                         float eps, void* out, int out_dtype, long long out_pitch_elems,
                                         cudaStream_t stream) {
  if (!x || !out || rows < 0 || d <= 0) return kBadArg;
  if (in_pitch_elems < d || out_pitch_elems < d) return kBadArg;
  if (d > 32 * kLnMaxPerLane) return kUnsupported;
  if (out_dtype < 0 || out_dtype > 2) return kBadArg;
  if (rows == 0) return kOk;
  if (rows > 0x7fffffffLL * 8) return kUnsupported;
  return with_x_dtype(in_dtype, [&](auto in_tag) {
    using TIn = std::remove_cv_t<std::remove_pointer_t<decltype(in_tag)>>;
    return with_x_dtype(out_dtype, [&](auto out_tag) {
      using TOut = std::remove_cv_t<std::remove_pointer_t<decltype(out_tag)>>;
      return launch_layernorm<TIn, TOut>(x, rows, d, in_pitch_elems, gamma, beta, eps, out, out_pitch_elems, stream);
    });
  });
}

extern "C" int wsae_layernorm_rows(const void* x, int in_dtype, long long rows, int d,
                                   long long in_pitch_elems, const float* gamma, const float* beta,
                                   float eps, float* out, long long out_pitch_elems,
                                   cudaStream_t stream) {
  return wsae_layernorm_rows_typed(x, in_dtype, rows, d, in_pitch_elems, gamma, beta, eps, out, 0, out_pitch_elems,
                                   stream);
}
