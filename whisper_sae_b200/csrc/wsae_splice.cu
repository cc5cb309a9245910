// wsae_splice.cu — splicing a trained TopK SAE into Whisper's forward pass (sae/splice.py).
//
// A site's hook replaces the layer output h [N, d] by h' (include/wsae.h states the formulas):
//   wsae_splice_pack   : x = LN(h) with the component's final LayerNorm, then K0's packed K1 operand
//                        bf16(x - b_pre) | bias block | zero rows up to Bp, plus (mu, rstd) per row.
//                        x itself never reaches HBM.  HBM bound: N*d*sizeof(h) in, Bp*Kp*2 + 8N out.
//   (K1, unchanged)    : (idx, val) = TopK_k of the pre-activations
//   wsae_splice_decode : sparse decode of relu(val) from the bf16 decoder shadow (K2's convention),
//                        the intervention (per-feature gain, steering vector), the inverse LayerNorm
//                        and the store in h's dtype; optional SSE / sum x^2 / L0 / x_sum /
//                        per-feature counts.  L2-gather bound: N * l0 * d * 2 bytes of decoder rows.
#include "wsae_rownorm.cuh"

extern "C" int wsae_packed_k(int d, int terms, int* dp_out, int* used_cols_out, int* kp_out);

namespace wsae {

struct SpliceStats {
  double sse;                     // sum of (recon - x)^2, unmodified reconstruction
  double sumsq;                   // sum of x^2
  unsigned long long l0;          // selected values > 0
};

constexpr int kPackWarps = 4;

// One warp per packed row.  The row is staged in shared memory (fp32, d <= 4096): the statistics are
// read from it in wsae_layernorm_rows' lane order, and the packed row is written from it in K0's
// 8-column groups.
template <typename TIn, int PER>
__global__ void __launch_bounds__(kPackWarps * 32)
splice_pack_kernel(const TIn* __restrict__ h, int N, int Bp, int d, int Kp, const float* __restrict__ gamma,
                   const float* __restrict__ beta, float eps, const float* __restrict__ b_pre,
                   __nv_bfloat16* __restrict__ a_packed, float2* __restrict__ row_stats) {
  extern __shared__ __align__(16) float s_rows[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int row = blockIdx.x * kPackWarps + warp;
  if (row >= Bp) return;
  uint4* dst = reinterpret_cast<uint4*>(a_packed + static_cast<size_t>(row) * Kp);
  const int groups = Kp >> 3;
  if (row >= N) {
    for (int q = lane; q < groups; q += 32) dst[q] = make_uint4(0u, 0u, 0u, 0u);
    return;
  }
  float* s = s_rows + warp * d;
  const TIn* hr = h + static_cast<size_t>(row) * d;
#pragma unroll 4
  for (int c = lane; c < d; c += 32) s[c] = ln_load<TIn>(hr, c);
  __syncwarp();
  float mean, rstd;
  ln_moments<PER>([&](int j) {
    const int c = j * 32 + lane;
    return c < d ? s[c] : 0.f;
  }, d, lane, eps, mean, rstd);
  if (lane == 0) row_stats[row] = make_float2(mean, rstd);
  for (int c = lane; c < d; c += 32) {
    const float g = gamma != nullptr ? gamma[c] : 1.f;
    const float b = beta != nullptr ? beta[c] : 0.f;
    float v = ln_apply(s[c], mean, rstd, g, b);
    if (b_pre != nullptr) v -= b_pre[c];
    s[c] = v;
  }
  __syncwarp();
  for (int q = lane; q < groups; q += 32) {
    const int c0 = q << 3;
    uint4 out = make_uint4(0u, 0u, 0u, 0u);
    if (c0 < d) {
      const float4 a = *reinterpret_cast<const float4*>(s + c0);
      const float4 b = *reinterpret_cast<const float4*>(s + c0 + 4);
      out = k0_pack8(a, b);
    } else if (c0 == d) {
      out = k0_bias_block8();
    }
    dst[q] = out;
  }
}

// ---- decode ------------------------------------------------------------------------------------
// 4 consecutive elements of the hidden state: the raw bits (to write back unchanged) and their fp32
__device__ __forceinline__ float4 h4_raw(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ uint2 h4_raw(const __nv_bfloat16* p) { return *reinterpret_cast<const uint2*>(p); }
__device__ __forceinline__ uint2 h4_raw(const __half* p) { return *reinterpret_cast<const uint2*>(p); }
__device__ __forceinline__ float4 h4_float(float4 r, const float*) { return r; }
template <typename TX>
__device__ __forceinline__ float4 h4_float(uint2 r, const TX*) { return x4_to_float4<TX>(r); }

__device__ __forceinline__ uint32_t to_bits16(float v, const __nv_bfloat16*) {
  return __bfloat16_as_ushort(__float2bfloat16_rn(v));
}
__device__ __forceinline__ uint32_t to_bits16(float v, const __half*) { return __half_as_ushort(__float2half_rn(v)); }

// Store 4 elements rounded to nearest; in error mode (keep_zero) an element whose difference dl is
// exactly 0 is written back as its raw input bits.
__device__ __forceinline__ void h4_store(float* p, float4 v, float4 raw, float4 dl, bool keep_zero) {
  float4 o;
  o.x = keep_zero && dl.x == 0.f ? raw.x : v.x;
  o.y = keep_zero && dl.y == 0.f ? raw.y : v.y;
  o.z = keep_zero && dl.z == 0.f ? raw.z : v.z;
  o.w = keep_zero && dl.w == 0.f ? raw.w : v.w;
  *reinterpret_cast<float4*>(p) = o;
}
template <typename TX>
__device__ __forceinline__ void h4_store(TX* p, float4 v, uint2 raw, float4 dl, bool keep_zero) {
  const TX* tag = nullptr;
  const uint32_t e0 = keep_zero && dl.x == 0.f ? (raw.x & 0xFFFFu) : to_bits16(v.x, tag);
  const uint32_t e1 = keep_zero && dl.y == 0.f ? (raw.x >> 16) : to_bits16(v.y, tag);
  const uint32_t e2 = keep_zero && dl.z == 0.f ? (raw.y & 0xFFFFu) : to_bits16(v.z, tag);
  const uint32_t e3 = keep_zero && dl.w == 0.f ? (raw.y >> 16) : to_bits16(v.w, tag);
  *reinterpret_cast<uint2*>(p) = make_uint2(e0 | (e1 << 16), e2 | (e3 << 16));
}

// Per element: x = LN(h) (or h), the statistics, and h' (formulas in include/wsae.h)
struct SpliceElem {
  bool ln, want_x, want_stats, replace;
  float mu, rs;
  __device__ __forceinline__ float operator()(float hv, float g, float b, float rc, float dl, float* xs,
                                              float& sse, float& sq) const {
    if (want_x) {
      const float x = ln ? ln_apply(hv, mu, rs, g, b) : hv;
      if (want_stats) {
        const float r = rc - x;
        sse = fmaf(r, r, sse);
        sq = fmaf(x, x, sq);
      }
      if (xs != nullptr) *xs += x;
    }
    if (replace) {
      const float rp = rc + dl;
      return ln ? mu + ((rp - b) / g) / rs : rp;
    }
    return ln ? hv + (dl / g) / rs : hv + dl;
  }
};

// One warp per row (persistent grid).  Lane l owns columns chunk*128*NV + 128*c + 4*l .. +3, c < NV:
// rows wider than 128*NV columns are done in column chunks, each walking the row's active entries
// again (the decoder bytes gathered stay the same).  acc = the SAE's reconstruction in K2's order
// (b_dec + b_pre, then fmaf over the active entries in selection order, activations rounded to bf16);
// dacc = recon' - recon = steer + sum (gain - 1) * a * W_dec[i], over the entries whose gain is not 1.
template <typename TX, int NV>
__global__ void __launch_bounds__(256)
splice_decode_kernel(const TX* __restrict__ h, const float2* __restrict__ row_stats,
                     const float* __restrict__ gamma, const float* __restrict__ beta,
                     const __nv_bfloat16* __restrict__ w_decT, const float* __restrict__ b_dec,
                     const float* __restrict__ b_pre, const int32_t* __restrict__ idx,
                     const float* __restrict__ val, const float* __restrict__ gain,
                     const float* __restrict__ steer, int N, int d, int F, int k, int mode,
                     TX* __restrict__ out, SpliceStats* __restrict__ stats, double* __restrict__ x_sum,
                     long long* __restrict__ feature_count) {
  extern __shared__ __align__(16) float s_xsum[];   // [warps][d] when x_sum != nullptr
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int warps_per_block = blockDim.x >> 5;
  const int warp_stride = gridDim.x * warps_per_block;
  const bool want_x = stats != nullptr || x_sum != nullptr;
  // error mode needs the full reconstruction only for the SSE; otherwise it gathers the rows whose
  // gain is not 1
  const bool full = mode == 0 || stats != nullptr;
  float* xs = x_sum != nullptr ? s_xsum + warp * d : nullptr;
  if (xs != nullptr)
    for (int c = lane; c < d; c += 32) xs[c] = 0.f;
  const int chunk_cols = 128 * NV;

  float sse_local = 0.f, sq_local = 0.f;
  unsigned int l0_local = 0;

  for (int row = blockIdx.x * warps_per_block + warp; row < N; row += warp_stride) {
    SpliceElem el{row_stats != nullptr, want_x, stats != nullptr, mode == 0, 0.f, 1.f};
    if (row_stats != nullptr) {
      const float2 st = row_stats[row];
      el.mu = st.x;
      el.rs = st.y;
    }
    const int32_t* irow = idx + static_cast<size_t>(row) * k;
    const float* vrow = val + static_cast<size_t>(row) * k;
    const TX* hrow = h + static_cast<size_t>(row) * d;
    TX* orow = out + static_cast<size_t>(row) * d;
    for (int col0 = 0; col0 < d; col0 += chunk_cols) {
      const bool first = col0 == 0;
      float4 acc[NV], dacc[NV];
#pragma unroll
      for (int c = 0; c < NV; ++c) {
        const int col = col0 + c * 128 + lane * 4;
        acc[c] = make_float4(0.f, 0.f, 0.f, 0.f);
        dacc[c] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (col < d) {
          if (full) {
            float4 a = *reinterpret_cast<const float4*>(b_dec + col);
            if (b_pre != nullptr) {
              const float4 p = *reinterpret_cast<const float4*>(b_pre + col);
              a.x += p.x; a.y += p.y; a.z += p.z; a.w += p.w;
            }
            acc[c] = a;
          }
          if (steer != nullptr) dacc[c] = *reinterpret_cast<const float4*>(steer + col);
        }
      }
      for (int j0 = 0; j0 < k; j0 += 32) {
        const int jj = j0 + lane;
        int32_t my_i = -1;
        float my_v = 0.f;
        if (jj < k) {
          my_i = irow[jj];
          my_v = vrow[jj];
        }
        const bool fired = (my_i >= 0) && (my_i < F) && (my_v > 0.f);
        // K2's convention: the activation is rounded to bf16 before the bf16 x bf16 product
        const float a_bf = __bfloat162float(__float2bfloat16_rn(my_v));
        const float g = (fired && gain != nullptr) ? gain[my_i] : 1.f;
        const bool modified = fired && g != 1.f;
        const float coef = (g - 1.f) * a_bf;
        const uint32_t act_mask = __ballot_sync(0xffffffffu, fired);
        const uint32_t mod_mask = __ballot_sync(0xffffffffu, modified);
        if (first) {
          if (lane == 0) l0_local += __popc(act_mask);
          if (fired && feature_count != nullptr)
            atomicAdd(reinterpret_cast<unsigned long long*>(feature_count + my_i), 1ull);
        }
        uint32_t m = full ? act_mask : mod_mask;
        while (m) {
          const int src = __ffs(m) - 1;
          m &= m - 1;
          const int32_t f = __shfl_sync(0xffffffffu, my_i, src);
          const float a = __shfl_sync(0xffffffffu, a_bf, src);
          const float cf = __shfl_sync(0xffffffffu, coef, src);
          const bool mod = (mod_mask >> src) & 1u;
          const __nv_bfloat16* wrow = w_decT + static_cast<size_t>(f) * d + col0;
#pragma unroll
          for (int c = 0; c < NV; ++c) {
            const int col = c * 128 + lane * 4;
            if (col0 + col < d) {
              const float4 w = bf16x4_to_float4(__ldg(reinterpret_cast<const uint2*>(wrow + col)));
              if (full) {
                acc[c].x = fmaf(a, w.x, acc[c].x);
                acc[c].y = fmaf(a, w.y, acc[c].y);
                acc[c].z = fmaf(a, w.z, acc[c].z);
                acc[c].w = fmaf(a, w.w, acc[c].w);
              }
              if (mod) {
                dacc[c].x = fmaf(cf, w.x, dacc[c].x);
                dacc[c].y = fmaf(cf, w.y, dacc[c].y);
                dacc[c].z = fmaf(cf, w.z, dacc[c].z);
                dacc[c].w = fmaf(cf, w.w, dacc[c].w);
              }
            }
          }
        }
      }
#pragma unroll
      for (int c = 0; c < NV; ++c) {
        const int col = col0 + c * 128 + lane * 4;
        if (col >= d) continue;
        const auto raw = h4_raw(hrow + col);
        const float4 hv = h4_float(raw, hrow);
        float4 gm = make_float4(1.f, 1.f, 1.f, 1.f), bt = make_float4(0.f, 0.f, 0.f, 0.f);
        if (row_stats != nullptr) {
          if (gamma != nullptr) gm = *reinterpret_cast<const float4*>(gamma + col);
          if (beta != nullptr) bt = *reinterpret_cast<const float4*>(beta + col);
        }
        const float4 rc = acc[c], dl = dacc[c];
        float* xc = xs != nullptr ? xs + col : nullptr;
        float4 o;
        o.x = el(hv.x, gm.x, bt.x, rc.x, dl.x, xc, sse_local, sq_local);
        o.y = el(hv.y, gm.y, bt.y, rc.y, dl.y, xc ? xc + 1 : nullptr, sse_local, sq_local);
        o.z = el(hv.z, gm.z, bt.z, rc.z, dl.z, xc ? xc + 2 : nullptr, sse_local, sq_local);
        o.w = el(hv.w, gm.w, bt.w, rc.w, dl.w, xc ? xc + 3 : nullptr, sse_local, sq_local);
        h4_store(orow + col, o, raw, dl, mode == 1);
      }
    }
  }

  // per-block partials: one set of global atomics per block
  __shared__ float s_sse[8], s_sq[8];
  __shared__ unsigned int s_l0[8];
  const float wsse = warp_sum(sse_local), wsq = warp_sum(sq_local);
  if (lane == 0) {
    s_sse[warp] = wsse;
    s_sq[warp] = wsq;
    s_l0[warp] = l0_local;
  }
  __syncthreads();
  if (threadIdx.x == 0 && stats != nullptr) {
    double t = 0.0, q = 0.0;
    unsigned long long c = 0;
    for (int w = 0; w < warps_per_block; ++w) {
      t += static_cast<double>(s_sse[w]);
      q += static_cast<double>(s_sq[w]);
      c += s_l0[w];
    }
    atomicAdd(&stats->sse, t);
    atomicAdd(&stats->sumsq, q);
    atomicAdd(&stats->l0, c);
  }
  if (x_sum != nullptr) {
    for (int c = threadIdx.x; c < d; c += blockDim.x) {
      double t = 0.0;
      for (int w = 0; w < warps_per_block; ++w) t += static_cast<double>(s_xsum[w * d + c]);
      atomicAdd(x_sum + c, t);
    }
  }
}

template <typename TX>
static int launch_splice_decode(const void* h, const float2* row_stats, const float* gamma, const float* beta,
                                const __nv_bfloat16* w_decT, const float* b_dec, const float* b_pre,
                                const int32_t* idx, const float* val, const float* gain, const float* steer,
                                int N, int d, int F, int k, int mode, void* out, SpliceStats* stats,
                                double* x_sum, long long* feature_count, cudaStream_t stream) {
  int dev = 0, sms = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int threads = 256, wpb = threads / 32;
  const size_t smem = x_sum != nullptr ? static_cast<size_t>(wpb) * d * sizeof(float) : 0;
  const TX* hx = static_cast<const TX*>(h);
  TX* ox = static_cast<TX*>(out);
  auto run = [&](auto kern) {
    if (smem > 48 * 1024) {
      const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 static_cast<int>(smem));
      if (e != cudaSuccess) return static_cast<int>(e);
    }
    int per_sm = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem);
    int blocks = ceil_div(N, wpb);
    const int cap = sms * (per_sm > 0 ? per_sm : 1);
    if (blocks > cap) blocks = cap;
    kern<<<blocks, threads, smem, stream>>>(hx, row_stats, gamma, beta, w_decT, b_dec, b_pre, idx, val, gain,
                                            steer, N, d, F, k, mode, ox, stats, x_sum, feature_count);
    return static_cast<int>(cudaGetLastError());
  };
  const int nv = ceil_div(d, 128);
  if (nv <= 3) return run(splice_decode_kernel<TX, 3>);
  if (nv <= 4) return run(splice_decode_kernel<TX, 4>);
  if (nv <= 6) return run(splice_decode_kernel<TX, 6>);
  if (nv <= 8) return run(splice_decode_kernel<TX, 8>);
  if (nv <= 10) return run(splice_decode_kernel<TX, 10>);
  return run(splice_decode_kernel<TX, 8>);       // d > 1280: column chunks of 1024
}

}  // namespace wsae

using namespace wsae;

extern "C" int wsae_splice_pack(const void* h, int h_dtype, int N, int Bp, int d, const float* gamma,
                                const float* beta, float eps, const float* b_pre, void* a_packed, float* row_stats,
                                cudaStream_t stream) {
  if (!h || !a_packed || !row_stats || N <= 0 || Bp < N || Bp % 128 != 0) return kBadArg;
  if (d <= 0 || d % 8 != 0) return kBadArg;
  if (d > 32 * kLnMaxPerLane) return kUnsupported;
  int Kp = 0;
  if (wsae_packed_k(d, 1, nullptr, nullptr, &Kp)) return kBadArg;
  const size_t smem = static_cast<size_t>(kPackWarps) * d * sizeof(float);
  const unsigned blocks = static_cast<unsigned>(ceil_div(Bp, kPackWarps));
  return with_x_dtype(h_dtype, [&](auto tag) {
    using TIn = std::remove_cv_t<std::remove_pointer_t<decltype(tag)>>;
    auto run = [&](auto kern) {
      if (smem > 48 * 1024) {
        const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                   static_cast<int>(smem));
        if (e != cudaSuccess) return static_cast<int>(e);
      }
      kern<<<blocks, kPackWarps * 32, smem, stream>>>(static_cast<const TIn*>(h), N, Bp, d, Kp, gamma, beta, eps,
                                                      b_pre, static_cast<__nv_bfloat16*>(a_packed),
                                                      reinterpret_cast<float2*>(row_stats));
      return static_cast<int>(cudaGetLastError());
    };
    switch (ln_per_bucket(d)) {
      case 4: return run(splice_pack_kernel<TIn, 4>);
      case 12: return run(splice_pack_kernel<TIn, 12>);
      case 16: return run(splice_pack_kernel<TIn, 16>);
      case 24: return run(splice_pack_kernel<TIn, 24>);
      case 32: return run(splice_pack_kernel<TIn, 32>);
      case 40: return run(splice_pack_kernel<TIn, 40>);
      case 64: return run(splice_pack_kernel<TIn, 64>);
      default: return run(splice_pack_kernel<TIn, kLnMaxPerLane>);
    }
  });
}

extern "C" int wsae_splice_decode(const void* h, int h_dtype, const float* row_stats, const float* gamma,
                                  const float* beta, const void* w_decT_bf16, const float* b_dec,
                                  const float* b_pre, const int32_t* idx, const float* val, const float* gain,
                                  const float* steer, int N, int d, int F, int k, int mode, void* out,
                                  void* stats, double* x_sum, long long* feature_count, cudaStream_t stream) {
  if (!h || !w_decT_bf16 || !b_dec || !idx || !val || !out) return kBadArg;
  if (N <= 0 || d <= 0 || d % 8 != 0 || F <= 0 || k <= 0 || (mode != 0 && mode != 1)) return kBadArg;
  if (d > 32 * kLnMaxPerLane) return kUnsupported;
  return with_x_dtype(h_dtype, [&](auto tag) {
    using TX = std::remove_cv_t<std::remove_pointer_t<decltype(tag)>>;
    return launch_splice_decode<TX>(h, reinterpret_cast<const float2*>(row_stats), gamma, beta,
                                    static_cast<const __nv_bfloat16*>(w_decT_bf16), b_dec, b_pre, idx, val, gain,
                                    steer, N, d, F, k, mode, out, static_cast<SpliceStats*>(stats), x_sum,
                                    feature_count, stream);
  });
}
