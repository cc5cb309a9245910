// wsae_pack.cu — K0: build the packed bf16 GEMM operands consumed by wsae_encode_topk.cu.
//
//   A'[r, :] = [ piece_a0(xc_r) | ... | piece_a(T-1)(xc_r) | 1 1 1 0 ... 0 | 0-pad ]   xc = x - b_pre
//   W'[f, :] = [ piece_w0(W_f)  | ... | piece_w(T-1)(W_f)  | b1 b2 b3 0 .. | 0-pad ]   b1+b2+b3 = b_enc[f]
//   W'[f >= F, :] = [ 0 ... 0 | -inf 0 0 .. | 0-pad ]      (padding rows: pre-activation = -inf)
//
// (reference: x - b_pre is model.py:108; the encoder bias add is part of nn.Linear at model.py:111.)
// Each of the T blocks is dp = round_up(d, 8) columns wide.  A split-bf16 "piece" p of a float v is
//   p0 = bf16(v), p1 = bf16(v - p0), p2 = bf16(v - p0 - p1)
// and the per-block piece schedule makes sum_t A'_t . W'_t equal the product expanded to
// T terms:  T=1: a0*w0        T=3: a0*w0 + a1*w0 + a0*w1
//           T=6: a0*w0 + a0*w1 + a1*w0 + a0*w2 + a1*w1 + a2*w0   (error ~2^-24: fp32 grade)
// The bias block is always a 3-piece split, so the bias is exact to fp32 in every mode.
#include "wsae_rownorm.cuh"

namespace wsae {

__device__ __forceinline__ __nv_bfloat16 split_piece(float v, int p) {
  __nv_bfloat16 h0 = __float2bfloat16_rn(v);
  if (p == 0) return h0;
  float r1 = v - __bfloat162float(h0);
  __nv_bfloat16 h1 = __float2bfloat16_rn(r1);
  if (p == 1) return h1;
  float r2 = r1 - __bfloat162float(h1);
  return __float2bfloat16_rn(r2);
}

struct PieceSchedule {
  int8_t p[6];
};

// One thread writes 8 consecutive bf16 (16 bytes) of one packed row.
// kind 0: activations (subtract center, ones in the bias block).
// kind 1: encoder weights (no center, split bias in the bias block).
template <int KIND>
__global__ void __launch_bounds__(256)
pack_rows_kernel(const float* __restrict__ src, const float* __restrict__ center,
                 const float* __restrict__ bias, int rows, int rows_p, int d, int dp, int T,
                 int Kp, PieceSchedule sched, __nv_bfloat16* __restrict__ dst) {
  pdl_prologue();
  const int groups = Kp >> 3;
  const size_t gid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (gid >= static_cast<size_t>(rows_p) * groups) return;
  const int r = static_cast<int>(gid / groups);
  const int c0 = static_cast<int>(gid - static_cast<size_t>(r) * groups) << 3;
  __align__(16) __nv_bfloat16 out[8];
  const __nv_bfloat16 zero = __float2bfloat16_rn(0.f);
#pragma unroll
  for (int j = 0; j < 8; ++j) out[j] = zero;
  if (r < rows) {
    const int body = T * dp;
    if (c0 < body) {
      const int t = c0 / dp;           // dp % 8 == 0, so the 8 columns stay inside one block
      const int j0 = c0 - t * dp;
      const int piece = sched.p[t];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int col = j0 + j;
        if (col < d) {
          float v = src[static_cast<size_t>(r) * d + col];
          if (KIND == 0 && center != nullptr) v -= center[col];
          out[j] = split_piece(v, piece);
        }
      }
    } else if (c0 == body) {
      if (KIND == 0) {
        const __nv_bfloat16 one = __float2bfloat16_rn(1.f);
        out[0] = one;
        out[1] = one;
        out[2] = one;
      } else {
        const float b = bias != nullptr ? bias[r] : 0.f;
        out[0] = split_piece(b, 0);
        out[1] = split_piece(b, 1);
        out[2] = split_piece(b, 2);
      }
    }
  } else if (KIND == 1 && c0 == T * dp) {
    // zero-padded feature rows (F..Fp) get a -inf bias, so the TopK epilogues of K1 can scan whole
    // tiles without a column guard: no threshold admits -inf, even in a row with fewer than k valid
    // (non-NaN) pre-activations.  (Rows >= B of A' are zero: 0 * -inf = NaN there, and those rows
    // are never written.)
    out[0] = __ushort_as_bfloat16(static_cast<unsigned short>(0xFF80u));
  }
  *reinterpret_cast<uint4*>(dst + static_cast<size_t>(r) * Kp + c0) =
      *reinterpret_cast<const uint4*>(out);
}

// 8 consecutive activations (16-byte aligned), streamed: fp32 is two 16-byte loads, a half type one
__device__ __forceinline__ void ldcs_x8(const float* p, float4& a, float4& b) {
  const float4* src = reinterpret_cast<const float4*>(p);
  a = __ldcs(src);
  b = __ldcs(src + 1);
}
template <typename TX>
__device__ __forceinline__ void ldcs_x8(const TX* p, float4& a, float4& b) {
  const uint4 u = __ldcs(reinterpret_cast<const uint4*>(p));
  a = x4_to_float4<TX>(make_uint2(u.x, u.y));
  b = x4_to_float4<TX>(make_uint2(u.z, u.w));
}

// bf16 fast path for activations (T = 1, d % 8 == 0): one thread converts 8 consecutive columns with
// two 16-byte loads (fp32 input; one for bf16 / fp16 input) and one 16-byte store; the bias block and
// the K padding are written by the same grid.  HBM bound: reads B*d*sizeof(TX), writes Bp*Kp*2 bytes.
template <typename TX>
__global__ void __launch_bounds__(256)
pack_activations_bf16_kernel(const TX* __restrict__ x, const TX* const* __restrict__ x_at,
                             const long long* const* __restrict__ rows_at,
                             const float* __restrict__ center, int rows, int rows_p, int d, int Kp,
                             __nv_bfloat16* __restrict__ dst) {
  pdl_prologue();
  // x_at: the matrix's address is read from device memory (a captured graph replays on whichever
  // batch the slot names - no staging copy of the batch into a graph-owned buffer).  rows_at: slot
  // with the address of an int64 row-index array (0 = identity): batch row r is matrix row
  // (*rows_at)[r], so a shuffled batch of a resident activation matrix is never materialised.
  if (x_at != nullptr) x = *x_at;
  const long long* perm = rows_at != nullptr ? *rows_at : nullptr;
  const int groups = Kp >> 3;
  const size_t gid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (gid >= static_cast<size_t>(rows_p) * groups) return;
  const int r = static_cast<int>(gid / groups);
  const int c0 = static_cast<int>(gid - static_cast<size_t>(r) * groups) << 3;
  uint4 out = make_uint4(0u, 0u, 0u, 0u);
  if (r < rows) {
    if (c0 < d) {
      const size_t sr = perm != nullptr ? static_cast<size_t>(__ldg(perm + r)) : static_cast<size_t>(r);
      float4 a, b;
      ldcs_x8(x + sr * d + c0, a, b);                     // streamed once: do not keep in L2/L1
      if (center != nullptr) {
        const float4 ca = __ldg(reinterpret_cast<const float4*>(center + c0));
        const float4 cb = __ldg(reinterpret_cast<const float4*>(center + c0 + 4));
        a.x -= ca.x; a.y -= ca.y; a.z -= ca.z; a.w -= ca.w;
        b.x -= cb.x; b.y -= cb.y; b.z -= cb.z; b.w -= cb.w;
      }
      out = k0_pack8(a, b);
    } else if (c0 == d) {
      out = k0_bias_block8();
    }
  }
  *reinterpret_cast<uint4*>(dst + static_cast<size_t>(r) * Kp + c0) = out;
}

static bool make_schedule(int T, bool weights, PieceSchedule* s) {
  static const int8_t a1[6] = {0, 0, 0, 0, 0, 0}, w1[6] = {0, 0, 0, 0, 0, 0};
  static const int8_t a3[6] = {0, 1, 0, 0, 0, 0}, w3[6] = {0, 0, 1, 0, 0, 0};
  static const int8_t a6[6] = {0, 0, 1, 0, 1, 2}, w6[6] = {0, 1, 0, 2, 1, 0};
  const int8_t* src = nullptr;
  if (T == 1) src = weights ? w1 : a1;
  else if (T == 3) src = weights ? w3 : a3;
  else if (T == 6) src = weights ? w6 : a6;
  else return false;
  for (int i = 0; i < 6; ++i) s->p[i] = src[i];
  return true;
}

}  // namespace wsae

using namespace wsae;

extern "C" int wsae_packed_k(int d, int terms, int* dp_out, int* used_cols_out, int* kp_out) {
  if (d <= 0 || (terms != 1 && terms != 3 && terms != 6)) return kBadArg;
  const int dp = round_up(d, 8);
  const int used = terms * dp + 16;
  if (dp_out) *dp_out = dp;
  if (used_cols_out) *used_cols_out = used;
  if (kp_out) *kp_out = round_up(used, 64);
  return kOk;
}

// x_dtype: element type of the activations (0 = fp32, 1 = bf16, 2 = fp16); half types are read by the
// single-term fast path only (src / src_at then point at that type).
static int pack_common(int kind, const float* src, const float* center, const float* bias,
                       int rows, int rows_p, int d, int terms, void* dst, cudaStream_t stream,
                       const void* const* src_at = nullptr, const long long* const* rows_at = nullptr,
                       int x_dtype = 0) {
  if ((!src && !src_at) || !dst || rows <= 0 || rows_p < rows) return kBadArg;
  if (x_dtype < 0 || x_dtype > 2) return kBadArg;
  int dp, used, Kp;
  if (wsae_packed_k(d, terms, &dp, &used, &Kp)) return kBadArg;
  PieceSchedule s;
  if (!make_schedule(terms, kind == 1, &s)) return kBadArg;
  const size_t total = static_cast<size_t>(rows_p) * (Kp >> 3);
  const int threads = 256;
  const unsigned blocks = static_cast<unsigned>((total + threads - 1) / threads);
  const bool fast = kind == 0 && terms == 1 && d % 8 == 0 &&
                    (reinterpret_cast<uintptr_t>(src) & 15u) == 0 &&
                    (center == nullptr || (reinterpret_cast<uintptr_t>(center) & 15u) == 0);
  // the slot form and half-precision input exist for the bf16 path only
  if ((src_at != nullptr || x_dtype != 0) && !fast) return kUnsupported;
  if (fast)
    return with_x_dtype(x_dtype, [&](auto tag) {
      using TX = std::remove_cv_t<std::remove_pointer_t<decltype(tag)>>;
      launch_pdl(pack_activations_bf16_kernel<TX>, blocks, threads, 0, stream,
                 reinterpret_cast<const TX*>(src), reinterpret_cast<const TX* const*>(src_at), rows_at,
                 center, rows, rows_p, d, Kp, static_cast<__nv_bfloat16*>(dst));
      return static_cast<int>(cudaGetLastError());
    });
  if (kind == 0)
    launch_pdl(pack_rows_kernel<0>, blocks, threads, 0, stream, src, center, bias, rows, rows_p, d,
               dp, terms, Kp, s, static_cast<__nv_bfloat16*>(dst));
  else
    launch_pdl(pack_rows_kernel<1>, blocks, threads, 0, stream, src, center, bias, rows, rows_p, d,
               dp, terms, Kp, s, static_cast<__nv_bfloat16*>(dst));
  return static_cast<int>(cudaGetLastError());
}

extern "C" int wsae_pack_activations(const float* x, const float* b_pre, int B, int Bp, int d,
                                     int terms, void* a_packed, cudaStream_t stream) {
  return pack_common(0, x, b_pre, nullptr, B, Bp, d, terms, a_packed, stream);
}

// Same, with the activation matrix named by a device-resident pointer slot (*x_at must be 16-byte
// aligned and hold B x d fp32 when the kernel runs).  bf16 single-term packing with d % 8 == 0 only.
extern "C" int wsae_pack_activations_at(const float* const* x_at, const float* b_pre, int B, int Bp,
                                        int d, int terms, void* a_packed, cudaStream_t stream) {
  if (!x_at) return kBadArg;
  return pack_common(0, nullptr, b_pre, nullptr, B, Bp, d, terms, a_packed, stream,
                     reinterpret_cast<const void* const*>(x_at));
}

// Slot form with a row-index indirection: batch row r = (*x_at)[(*rows_at)[r], :]; *rows_at == 0 means
// identity.  (reference: the DataLoader's shuffled TensorDataset batch, data/feature_cache.py:169-197.)
extern "C" int wsae_pack_activations_rows_at(const float* const* x_at, const long long* const* rows_at,
                                             const float* b_pre, int B, int Bp, int d, int terms,
                                             void* a_packed, cudaStream_t stream) {
  if (!x_at || !rows_at) return kBadArg;
  return pack_common(0, nullptr, b_pre, nullptr, B, Bp, d, terms, a_packed, stream,
                     reinterpret_cast<const void* const*>(x_at), rows_at);
}

// Slot form for any activation element type (x_dtype 0 = fp32, 1 = bf16, 2 = fp16); rows_at nullable.
extern "C" int wsae_pack_activations_typed(const void* const* x_at, const long long* const* rows_at, int x_dtype,
                                           const float* b_pre, int B, int Bp, int d, int terms, void* a_packed,
                                           cudaStream_t stream) {
  if (!x_at) return kBadArg;
  return pack_common(0, nullptr, b_pre, nullptr, B, Bp, d, terms, a_packed, stream, x_at, rows_at, x_dtype);
}

extern "C" int wsae_pack_encoder(const float* w_enc, const float* b_enc, int F, int Fp, int d,
                                 int terms, void* w_packed, cudaStream_t stream) {
  return pack_common(1, w_enc, nullptr, b_enc, F, Fp, d, terms, w_packed, stream);
}
