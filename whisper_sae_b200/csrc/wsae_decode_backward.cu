// wsae_decode_backward.cu — K23: the k-sparse decode (K2) and the sparse part of the backward (K3)
// fused into ONE pass over the gathered decoder rows, for the train step where grad_output is known
// when the forward runs (the CUDA-graphed SAETrainer step: loss.backward() with grad_output = 1).
//
// Replaces (reference, /root/reference/src/whisper_sae/sae/model.py, and its autograd at
// sae/training.py:184):
//   :115-116,129  recon = sum_j relu(v_j) * W_dec[:, i_j] + b_dec + b_pre
//   :145,148      mse numerator, l0 count                         -> stats
//   :174-181      last_activated[fired] = step_count + 1
//   backward      g = s * (recon - x);  db_dec = sum_b g;  dv_j = [v_j > 0] * (g . W_dec[:, i_j]);
//                 db_enc[i_j] += dv_j      (the two weight gradients are K4's tensor-core GEMMs,
//                                           fed with bf16(recon - x) and dv from here)
//
// Why fused: decode and backward need the same k decoder rows per activation row (k * d * 2 bytes =
// 24 KB at d = 384 with the bf16 shadow).  Unfused they are fetched from L2 twice, each time inside a
// dependent loop that exposes the load latency.  Here one warp owns one activation row and walks it
// in slices of 128 columns: lane l owns 4 consecutive columns, so the slice of one decoder row is one
// coalesced 8-byte load per lane.  The 32 row slices are loaded into REGISTERS with all 32 loads in
// flight at once, used for the reconstruction and - still in registers - for the 32 partial dot
// products with the residual.  Both are FHFMA.BF16 (bf16 x bf16 products, fp32 accumulate, operand
// halves picked by .H0/.H1 selectors: no conversion instructions); activation and residual enter
// in the bf16 rounding that K4's weight-gradient GEMMs consume.
// Every decoder byte is read from L2 exactly once.  (A first version staged the rows in shared
// memory with one cp.async.bulk per row: 32 bulk copies of 768 B per activation row saturate the
// TMA unit at ~45 ns per copy - 0.62 ms against 0.23 ms for this form; DESIGN.md section 4.)
#include "wsae_common.cuh"

namespace wsae {

struct FusedStats {
  double sse;
  unsigned long long l0_count;
};

// acc0 += a.lo*r.lo + a.hi*r.hi ;  acc1 += c.lo*r.lo + c.hi*r.hi   (bf16 x bf16 products, fp32
// accumulate: SASS FHFMA.BF16 with .H0/.H1 operand selectors, no conversion instructions)
__device__ __forceinline__ void fhfma2(float& acc0, float& acc1, uint32_t a, uint32_t r, uint32_t c) {
  asm("{\n\t"
      ".reg .b16 a0, a1, r0, r1, c0, c1;\n\t"
      "mov.b32 {a0, a1}, %2;\n\t"
      "mov.b32 {r0, r1}, %3;\n\t"
      "mov.b32 {c0, c1}, %4;\n\t"
      "fma.rn.f32.bf16 %0, a0, r0, %0;\n\t"
      "fma.rn.f32.bf16 %1, c0, r0, %1;\n\t"
      "fma.rn.f32.bf16 %0, a1, r1, %0;\n\t"
      "fma.rn.f32.bf16 %1, c1, r1, %1;\n\t"
      "}\n"
      : "+f"(acc0), "+f"(acc1)
      : "r"(a), "r"(r), "r"(c));
}

// acc.{x,y,z,w} += bf16(w.x.lo, w.x.hi, w.y.lo, w.y.hi) * bf16(h.lo)   (fp32 accumulate)
__device__ __forceinline__ void fhfma_bcast4(float4& acc, uint2 w, uint32_t h) {
  asm("{\n\t"
      ".reg .b16 a0, a1, c0, c1, h0, h1;\n\t"
      "mov.b32 {a0, a1}, %4;\n\t"
      "mov.b32 {c0, c1}, %5;\n\t"
      "mov.b32 {h0, h1}, %6;\n\t"
      "fma.rn.f32.bf16 %0, a0, h0, %0;\n\t"
      "fma.rn.f32.bf16 %1, a1, h0, %1;\n\t"
      "fma.rn.f32.bf16 %2, c0, h0, %2;\n\t"
      "fma.rn.f32.bf16 %3, c1, h0, %3;\n\t"
      "}\n"
      : "+f"(acc.x), "+f"(acc.y), "+f"(acc.z), "+f"(acc.w)
      : "r"(w.x), "r"(w.y), "r"(h));
}

// D(16x8, fp32) += A(16x16, bf16, row) * B(16x8, bf16, col): the legacy warp-level tensor-core path
// (SASS HMMA.16816.F32.BF16).  Used for the k dot products of the fast path below; the tcgen05 / TMEM
// path is for the dense GEMMs (K1, K4) - here the operands are 32 gathered rows that already sit in
// registers, the math is 2 % of a GEMM tile and the kernel is bound by the L2 gather, not by FLOPs.
__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2,
                                               uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, "
      "{%8, %9}, {%0, %1, %2, %3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

constexpr int kFusedWarps = 4;

// ---- deterministic accumulation (wsae_decode_backward_det) ------------------------------------------
// The three cross-row sums of this kernel - db_enc[f], db_dec[c] and the SSE - are float atomics in
// the default mode, i.e. summed in whatever order the warps arrive: two runs differ in the last bits,
// and early AdamW steps amplify that (profiles/r1_v12_check_dp_2gpu.txt: 1e-2 rel-L2 in the weights
// after 24 steps).  With a workspace `det_ws` (int64 [F + d + 1], caller-zeroed) every addend is
// rounded ONCE to fixed point and added with integer atomics - integer addition is associative, so
// the result does not depend on the order.  The addends are the UNSCALED dot products r . w (|.| <
// 2^10, scale 2^30), residual column sums (scale 2^28) and squared errors (scale 2^20): the common
// factor s = coef * grad_out is applied by wsae_det_finish, which converts the sums back.
constexpr double kDetScaleEnc = 1073741824.0;      // 2^30
constexpr double kDetScaleDec = 268435456.0;       // 2^28
constexpr double kDetScaleSse = 1048576.0;         // 2^20
__device__ __forceinline__ void det_add(long long* slot, double v, double scale) {
  atomicAdd(reinterpret_cast<unsigned long long*>(slot),
            static_cast<unsigned long long>(__double2ll_rn(v * scale)));
}
constexpr int kDotScratch = 32 * 9;   // floats per warp: 32 dot products x 8 partial sums, stride 9 (bank-conflict free)

// bf16 decoder shadow only.  k <= 32, d % 8 == 0.
//
// kFast (d % 128 == 0: every BASELINE width - 384, 768, 1280, 4 x 384): every slice is full, so the
// gather is 32 unpredicated loads whose address is ONE IMAD.WIDE from a 32-bit row offset (the
// general form spent 5 instructions per load on bounds predicates, register zeroing and re-loading
// the base pointer: 25 % of all instructions issued, ncu source page), and the 32 dot products
// r . W_dec[i_j] run on the tensor pipe: mma.m16n8k16 with A = {w[j].x, w[j'].x, w[j].y, w[j'].y}
// reads lane l's register as "row (l >> 2), k-columns (l & 3)": the 8 "rows" of the A tile are the
// eight 16-column blocks of gathered row j (rows 8-15: row j'), and with B = the lane's own bf16
// residual {rb.x, rb.y} column n of B is block n of the residual - so the DIAGONAL D[g][g] is the
// partial dot product over block g.  Sixteen HMMA per slice replace 128 FHFMA, the accumulators
// stay in registers across the slices, and the diagonal is summed through 1.1 KB of shared memory
// per warp instead of a 31-step shuffle transpose.
// TX: element type of the target matrix (float / __nv_bfloat16 / __half, converted at the load).
template <bool kFast, typename TX>
__global__ void __launch_bounds__(kFusedWarps * 32, kFast ? 3 : 4)
decode_backward_kernel(const TX* __restrict__ target, const __nv_bfloat16* __restrict__ w_decT,
                       const float* __restrict__ b_dec, const float* __restrict__ b_pre,
                       const int32_t* __restrict__ idx, const float* __restrict__ val,
                       const float* __restrict__ grad_out, float coef, int B, int d, int F, int k,
                       float* __restrict__ resid, __nv_bfloat16* __restrict__ resid_bf16,
                       FusedStats* __restrict__ stats, long long* __restrict__ last_activated,
                       const long long* __restrict__ step_count, float* __restrict__ d_b_enc,
                       float* __restrict__ d_b_dec, float* __restrict__ dpre_val,
                       const TX* const* __restrict__ target_at,
                       const long long* const* __restrict__ rows_at, int stamp_words,
                       long long* __restrict__ det_ws) {
  extern __shared__ __align__(16) float fsm[];   // [dp] bias (b_dec + b_pre), then one [dp] db_dec accumulator per warp
  pdl_prologue();
  if (target_at != nullptr) target = *target_at;   // address from a device-resident slot (graph replay)
  // batch row r is row (*rows_at)[r] of the target matrix (0 / null = identity): wsae_pack.cu
  const long long* perm = rows_at != nullptr ? *rows_at : nullptr;
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int dp = round_up(d, 128);
  float* s_bias = fsm;
  float* s_g = fsm + dp + warp * dp;       // warp-private: plain read-modify-write, no atomics
  float* s_dot = fsm + (1 + kFusedWarps) * dp;   // fast path: per-warp scratch of the dot-product reduction
  // fired-feature bitmap of this block (stamp_words = ceil(F / 32), 0 = stamp straight to global memory):
  // 2.4 M scattered 8-byte stamp stores per launch, issued next to as many RED.ADDs on d_b_enc, cost the
  // staged kernel 78 us of 301 (tools/k23_dbg.py); one coalesced pass per block writes them instead
  uint32_t* s_fired = reinterpret_cast<uint32_t*>(s_dot + kFusedWarps * kDotScratch);
  for (int i = threadIdx.x; i < stamp_words; i += blockDim.x) s_fired[i] = 0u;
  for (int i = threadIdx.x; i < dp; i += blockDim.x) {
    float b = 0.f;
    if (i < d) b = b_dec[i] + (b_pre != nullptr ? b_pre[i] : 0.f);
    s_bias[i] = b;
#pragma unroll
    for (int w = 0; w < kFusedWarps; ++w) fsm[dp + w * dp + i] = 0.f;
  }
  __syncthreads();

  const float s = coef * (grad_out != nullptr ? *grad_out : 1.f);
  const long long stamp = (last_activated != nullptr && step_count != nullptr) ? (*step_count + 1) : 0;
  const int warp_global = blockIdx.x * kFusedWarps + warp;
  const int warp_stride = gridDim.x * kFusedWarps;
  const uint2* wbase = reinterpret_cast<const uint2*>(w_decT);   // 4 bf16 per element
  const int d4 = d >> 2;

  float sse_local = 0.f;
  unsigned int l0_local = 0;

  for (int row = warp_global; row < B; row += warp_stride) {
    int32_t my_i = -1;
    float my_v = 0.f;
    if (lane < k) {
      my_i = idx[static_cast<size_t>(row) * k + lane];
      my_v = val[static_cast<size_t>(row) * k + lane];
    }
    const bool fired = (my_i >= 0) && (my_i < F) && (my_v > 0.f);
    if (fired && last_activated != nullptr) {
      if (stamp_words > 0) atomicOr(&s_fired[my_i >> 5], 1u << (my_i & 31));
      else last_activated[my_i] = stamp;
    }
    if (!fired) my_v = 0.f;                         // relu; also neutralises invalid entries
    // bf16 mode: the decoder product is bf16 x bf16 with fp32 accumulation - the activation enters
    // in bf16 like the weight shadow (the reference's autocast decoder Linear rounds `hidden` to
    // half precision too; K4's dW_dec GEMM consumes the same bf16(h))
    const uint32_t my_hb = static_cast<uint32_t>(__bfloat16_as_ushort(__float2bfloat16_rn(my_v)));
    const uint32_t mask = __ballot_sync(0xffffffffu, fired);
    l0_local += (lane == 0) ? __popc(mask) : 0;
    // element offset (in uint2 units) of each selected decoder row; inactive entries read row 0
    // with weight 0, so every lane issues the same, fully unrolled load sequence
    const int my_off = fired ? my_i * d4 : 0;

    if (kFast) {
      // ---------------- fast path: full 128-column slices, dots on the tensor pipe ----------------
      float acc[16][4];
#pragma unroll
      for (int p = 0; p < 16; ++p) acc[p][0] = acc[p][1] = acc[p][2] = acc[p][3] = 0.f;
      const uint2* lane_base = wbase + lane;
      const size_t srow = perm != nullptr ? static_cast<size_t>(__ldg(perm + row)) : static_cast<size_t>(row);
      const TX* trow = target + srow * d + lane * 4;
      for (int c0 = 0; c0 < d; c0 += 128) {
        const uint2* sb = lane_base + (c0 >> 2);
        uint2 w[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const uint32_t off = __shfl_sync(0xffffffffu, static_cast<uint32_t>(my_off), j);
          w[j] = __ldg(sb + off);
        }
        const float4 t = ldg_x4(trow + c0);
        float4 a = *reinterpret_cast<const float4*>(s_bias + c0 + lane * 4);
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const uint32_t hb = __shfl_sync(0xffffffffu, my_hb, j);
          fhfma_bcast4(a, w[j], hb);
        }
        float4 r;
        r.x = a.x - t.x; r.y = a.y - t.y; r.z = a.z - t.z; r.w = a.w - t.w;
        sse_local = fmaf(r.x, r.x, sse_local);
        sse_local = fmaf(r.y, r.y, sse_local);
        sse_local = fmaf(r.z, r.z, sse_local);
        sse_local = fmaf(r.w, r.w, sse_local);
        __nv_bfloat162 rlo = __floats2bfloat162_rn(r.x, r.y);
        __nv_bfloat162 rhi = __floats2bfloat162_rn(r.z, r.w);
        uint2 rb;
        rb.x = *reinterpret_cast<uint32_t*>(&rlo);
        rb.y = *reinterpret_cast<uint32_t*>(&rhi);
        const size_t o = static_cast<size_t>(row) * d + c0 + lane * 4;
        if (resid != nullptr) *reinterpret_cast<float4*>(resid + o) = r;
        if (resid_bf16 != nullptr) *reinterpret_cast<uint2*>(resid_bf16 + o) = rb;
        float4 gs = *reinterpret_cast<float4*>(s_g + c0 + lane * 4);
        gs.x += r.x; gs.y += r.y; gs.z += r.z; gs.w += r.w;
        *reinterpret_cast<float4*>(s_g + c0 + lane * 4) = gs;
#pragma unroll
        for (int p = 0; p < 16; ++p)
          mma_bf16_16816(acc[p], w[2 * p].x, w[2 * p + 1].x, w[2 * p].y, w[2 * p + 1].y, rb.x, rb.y);
      }
      // D[g][g] of tile p lives in lane (g, t = g >> 1): register g & 1 for row 2p, 2 + (g & 1) for
      // row 2p + 1.  The 8 holder lanes park their 32 partial sums in shared memory, lane j adds up
      // the 8 partials of dot product j.
      const int g = lane >> 2;
      float* scr = s_dot + warp * kDotScratch;
      if ((lane & 3) == (g >> 1)) {
        const bool odd = (g & 1) != 0;
#pragma unroll
        for (int p = 0; p < 16; ++p) {
          scr[(2 * p) * 9 + g] = odd ? acc[p][1] : acc[p][0];
          scr[(2 * p + 1) * 9 + g] = odd ? acc[p][3] : acc[p][2];
        }
      }
      __syncwarp();
      float dot = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) dot += scr[lane * 9 + i];
      __syncwarp();
      const float my_dv = fired ? s * dot : 0.f;
      if (lane < k) {
        if (dpre_val != nullptr) dpre_val[static_cast<size_t>(row) * k + lane] = my_dv;
        if (fired && d_b_enc != nullptr) {
          if (det_ws != nullptr) det_add(det_ws + my_i, static_cast<double>(dot), kDetScaleEnc);
          else atomicAdd(d_b_enc + my_i, my_dv);
        }
      }
      continue;
    }

    float part[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) part[j] = 0.f;

    for (int c0 = 0; c0 < d; c0 += 128) {
      const int col = c0 + lane * 4;
      const bool ok = col < d;
      // ---- gather: 32 independent 8-byte loads per lane, all in flight together ----
      uint2 w[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const int off = __shfl_sync(0xffffffffu, my_off, j);
        w[j] = make_uint2(0u, 0u);
        if (ok) w[j] = __ldg(wbase + off + (col >> 2));
      }
      float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
      if (ok) {
        const size_t srow = perm != nullptr ? static_cast<size_t>(__ldg(perm + row)) : static_cast<size_t>(row);
        t = ldg_x4(target + srow * d + col);
      }
      float4 acc = *reinterpret_cast<const float4*>(s_bias + col);
      // ---- reconstruction of this slice (fp32) ----
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const uint32_t hb = __shfl_sync(0xffffffffu, my_hb, j);
        fhfma_bcast4(acc, w[j], hb);
      }
      float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
      if (ok) {
        r.x = acc.x - t.x; r.y = acc.y - t.y; r.z = acc.z - t.z; r.w = acc.w - t.w;
      }
      sse_local = fmaf(r.x, r.x, sse_local);
      sse_local = fmaf(r.y, r.y, sse_local);
      sse_local = fmaf(r.z, r.z, sse_local);
      sse_local = fmaf(r.w, r.w, sse_local);
      __nv_bfloat162 rlo = __floats2bfloat162_rn(r.x, r.y);
      __nv_bfloat162 rhi = __floats2bfloat162_rn(r.z, r.w);
      uint2 rb;
      rb.x = *reinterpret_cast<uint32_t*>(&rlo);
      rb.y = *reinterpret_cast<uint32_t*>(&rhi);
      if (ok) {
        if (resid != nullptr) *reinterpret_cast<float4*>(resid + static_cast<size_t>(row) * d + col) = r;
        if (resid_bf16 != nullptr)
          *reinterpret_cast<uint2*>(resid_bf16 + static_cast<size_t>(row) * d + col) = rb;
        // db_dec partial sums (unscaled; s is applied once at the end)
        float4 gs = *reinterpret_cast<float4*>(s_g + col);
        gs.x += r.x; gs.y += r.y; gs.z += r.z; gs.w += r.w;
        *reinterpret_cast<float4*>(s_g + col) = gs;
      }
      // ---- partial dots bf16(r) . W_dec[i_j] over this slice ----
#pragma unroll
      for (int j = 0; j < 32; j += 2) {   // two independent accumulation chains per pair of rows
        fhfma2(part[j], part[j + 1], w[j].x, rb.x, w[j + 1].x);
        fhfma2(part[j], part[j + 1], w[j].y, rb.y, w[j + 1].y);
      }
    }
    // ---- transpose-reduce: lane j ends up with the sum over lanes of part[j] ----
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
      const bool upper = (lane & off) != 0;
#pragma unroll
      for (int i = 0; i < off; ++i) {
        const float send = upper ? part[i] : part[i + off];
        const float keep = upper ? part[i + off] : part[i];
        part[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
      }
    }
    const float my_dv = fired ? s * part[0] : 0.f;
    if (lane < k) {
      if (dpre_val != nullptr) dpre_val[static_cast<size_t>(row) * k + lane] = my_dv;
      if (fired && d_b_enc != nullptr) {
        if (det_ws != nullptr) det_add(det_ws + my_i, static_cast<double>(part[0]), kDetScaleEnc);
        else atomicAdd(d_b_enc + my_i, my_dv);
      }
    }
  }

  // ---- block reductions: db_dec (per column), SSE (double), L0 (integer) ----
  __shared__ float s_sse[kFusedWarps];
  __shared__ unsigned int s_l0[kFusedWarps];
  const float wsum = warp_sum(sse_local);
  if (lane == 0) {
    s_sse[warp] = wsum;
    s_l0[warp] = l0_local;
  }
  __syncthreads();
  if (stamp_words > 0 && last_activated != nullptr)
    for (int f = threadIdx.x; f < F; f += blockDim.x)
      if ((s_fired[f >> 5] >> (f & 31)) & 1u) last_activated[f] = stamp;
  if (d_b_dec != nullptr)
    for (int i = threadIdx.x; i < d; i += blockDim.x) {
      float t = 0.f;
#pragma unroll
      for (int w = 0; w < kFusedWarps; ++w) t += fsm[dp + w * dp + i];
      if (det_ws != nullptr) det_add(det_ws + F + i, static_cast<double>(t), kDetScaleDec);
      else atomicAdd(d_b_dec + i, s * t);
    }
  if (threadIdx.x == 0 && stats != nullptr) {
    double tsum = 0.0;
    unsigned long long c = 0;
    for (int w = 0; w < kFusedWarps; ++w) {
      tsum += static_cast<double>(s_sse[w]);
      c += s_l0[w];
    }
    if (det_ws != nullptr) det_add(det_ws + F + d, tsum, kDetScaleSse);
    else atomicAdd(&stats->sse, tsum);
    atomicAdd(&stats->l0_count, c);
  }
}

// ================================================================================================
// K23, staged form (d % 128 == 0, d >= 128 * (STAGES - 1)): the gather runs AHEAD of the math.
//
// ncu + tools/l2_gather_bench (profiles/r2_l2_gather.json): a pure gather of the same 1.86 GB of
// decoder rows runs at 14-16 TB/s out of L2, the register-staged kernel above at 8.3 TB/s with the
// issue slots 62 % busy - each warp loads a slice (32 rows x 256 B), waits ~2000 cycles for the loaded
// L2 queue to drain, computes, and only then asks for the next slice, so the memory system idles
// while the warps compute and the warps idle while it works.  Here every warp owns a ring of STAGES
// shared-memory slice buffers (8 KB each) filled by cp.async (LDGSTS.128: L2 -> shared memory, no
// registers): while slice q is multiplied out of registers, slices q+1 .. q+STAGES-1 - of this
// activation row or the next - are already in flight.  16 cp.async per slice (lanes 0-15 copy the
// 256-byte slice of one gathered row, lanes 16-31 the next), one LDS.64 per gathered row and lane to
// bring the staged slice into the same register layout the general kernel uses; the arithmetic
// (FHFMA.BF16 reconstruction and dot products, transpose-reduce, stats, stamps) is unchanged, so the
// results are bit-identical to the general kernel.
// ================================================================================================
__device__ __forceinline__ void cp_async_16(uint32_t smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_dst), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

constexpr int kSliceBytes = 32 * 256;   // one staged slice: 32 gathered rows x 128 bf16 columns

template <int STAGES, typename TX>
__global__ void __launch_bounds__(kFusedWarps * 32, STAGES == 2 ? 3 : 2)
decode_backward_staged_kernel(const TX* __restrict__ target, const __nv_bfloat16* __restrict__ w_decT,
                              const float* __restrict__ b_dec, const float* __restrict__ b_pre,
                              const int32_t* __restrict__ idx, const float* __restrict__ val,
                              const float* __restrict__ grad_out, float coef, int B, int d, int F, int k,
                              float* __restrict__ resid, __nv_bfloat16* __restrict__ resid_bf16,
                              FusedStats* __restrict__ stats, long long* __restrict__ last_activated,
                              const long long* __restrict__ step_count, float* __restrict__ d_b_enc,
                              float* __restrict__ d_b_dec, float* __restrict__ dpre_val,
                              const TX* const* __restrict__ target_at,
                              const long long* const* __restrict__ rows_at, int stamp_words,
                              long long* __restrict__ det_ws, int dbg) {
  extern __shared__ __align__(16) float fsm[];   // [d] bias, [warps][d] db_dec partials, the slice rings, the fired bitmap
  pdl_prologue();
  if (target_at != nullptr) target = *target_at;
  const long long* perm = rows_at != nullptr ? *rows_at : nullptr;
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  float* s_bias = fsm;
  float* s_g = fsm + d + warp * d;
  const uint32_t ring = smem_u32(fsm + (1 + kFusedWarps) * d) + warp * (STAGES * kSliceBytes);
  uint32_t* s_fired = reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(fsm + (1 + kFusedWarps) * d) +
                                                  kFusedWarps * STAGES * kSliceBytes);
  for (int i = threadIdx.x; i < stamp_words; i += blockDim.x) s_fired[i] = 0u;
  for (int i = threadIdx.x; i < d; i += blockDim.x) {
    s_bias[i] = b_dec[i] + (b_pre != nullptr ? b_pre[i] : 0.f);
#pragma unroll
    for (int w = 0; w < kFusedWarps; ++w) fsm[d + w * d + i] = 0.f;
  }
  __syncthreads();

  const float s = coef * (grad_out != nullptr ? *grad_out : 1.f);
  const long long stamp = (last_activated != nullptr && step_count != nullptr) ? (*step_count + 1) : 0;
  const int warp_global = blockIdx.x * kFusedWarps + warp;
  const int warp_stride = gridDim.x * kFusedWarps;
  const int nsl = d >> 7;                      // slices per activation row
  const int row_bytes = d * 2;
  const char* wbytes = reinterpret_cast<const char*>(w_decT);
  // copy role of this lane: rows 2i + (lane >> 4), 16-byte chunk (lane & 15) of the slice
  const int cp_half = lane >> 4;
  const uint32_t cp_dst = (lane >> 4) * 256u + (lane & 15) * 16u;
  const int cp_col = (lane & 15) * 16;

  // (index, value) of a row's k entries, one per lane: byte offset of the gathered decoder row and
  // the bf16 activation; invalid / non-positive entries gather row 0 with weight 0
  auto load_meta = [&](int row, int32_t& mi, float& mv) {
    mi = -1;
    mv = 0.f;
    if (row < B && lane < k) {
      mi = __ldg(idx + static_cast<size_t>(row) * k + lane);
      mv = __ldg(val + static_cast<size_t>(row) * k + lane);
    }
  };
  auto issue_slice = [&](uint32_t off_bytes, int sl, int stage) {     // off_bytes: this lane's entry
    const uint32_t dst0 = ring + stage * kSliceBytes + cp_dst;
    const char* src0 = wbytes + sl * 256 + cp_col;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const uint32_t off = __shfl_sync(0xffffffffu, off_bytes, 2 * i + cp_half);
      cp_async_16(dst0 + i * 512, src0 + off);
    }
  };

  float sse_local = 0.f;
  unsigned int l0_local = 0;

  int row = warp_global;
  int32_t cur_i, nxt_i;
  float cur_v, nxt_v;
  load_meta(row, cur_i, cur_v);
  load_meta(row + warp_stride, nxt_i, nxt_v);
  // Entries that did not fire (value <= 0) still gather THEIR row (weight 0); invalid indices gather a
  // row that differs per (activation row, lane).  Sending them all to row 0, as the register-staged
  // kernel does, is harmless there (L1 serves it) but cp.async bypasses L1: with half of the entries
  // inactive every SM hammered the same few L2 sectors and the kernel ran 10x slower (2.7 ms).
  auto row_offset = [&](int32_t mi, int row_) -> uint32_t {
    const uint32_t f = (mi >= 0 && mi < F) ? static_cast<uint32_t>(mi)
                                           : (static_cast<uint32_t>(row_) * 37u + static_cast<uint32_t>(lane)) % static_cast<uint32_t>(F);
    return f * static_cast<uint32_t>(row_bytes);
  };
  bool cur_f = (cur_i >= 0) && (cur_i < F) && (cur_v > 0.f);
  uint32_t cur_off = row_offset(cur_i, row);
  bool nxt_f = (nxt_i >= 0) && (nxt_i < F) && (nxt_v > 0.f);
  uint32_t nxt_off = row_offset(nxt_i, row + warp_stride);

  // prologue: slices 0 .. STAGES-2 of the flattened (row, slice) sequence (nsl >= STAGES - 1: they
  // belong to the first row)
#pragma unroll
  for (int q = 0; q < STAGES - 1; ++q) {
    if (row < B) issue_slice(cur_off, q, q);
    cp_async_commit();
  }
  int stage = 0;                               // stage holding the slice about to be computed

  for (; row < B; row += warp_stride) {
    const bool fired = cur_f;
    const int32_t my_i = cur_i;
    if (fired && last_activated != nullptr && !(dbg & 4)) {
      if (stamp_words > 0) atomicOr(&s_fired[my_i >> 5], 1u << (my_i & 31));
      else last_activated[my_i] = stamp;
    }
    const float my_v = fired ? cur_v : 0.f;
    const uint32_t my_hb = static_cast<uint32_t>(__bfloat16_as_ushort(__float2bfloat16_rn(my_v)));
    const uint32_t mask = __ballot_sync(0xffffffffu, fired);
    l0_local += (lane == 0) ? __popc(mask) : 0;
    const size_t srow = perm != nullptr ? static_cast<size_t>(__ldg(perm + row)) : static_cast<size_t>(row);
    const TX* trow = target + srow * d + lane * 4;
    int32_t nn_i = -1;     // metadata two rows ahead: requested after the first slice's copies are
    float nn_v = 0.f;      // out (not at the top of the row, where ptxas made the target address wait
                           // for it: 11 % of all stall samples), consumed when this row is done

    float part[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) part[j] = 0.f;

    for (int sl = 0; sl < nsl; ++sl) {
      float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
      if (!(dbg & 1)) t = ldg_x4(trow + sl * 128);
      cp_async_wait<STAGES - 2>();             // slice (row, sl) has landed (this lane's copies)
      __syncwarp();                            // ... and every other lane's; the stage consumed last is free
      {   // keep the ring full: slice sl + STAGES - 1 of this row, or of the next one
        const int ps = sl + STAGES - 1;
        int pstage = stage + STAGES - 1;
        if (pstage >= STAGES) pstage -= STAGES;
        if (ps < nsl) issue_slice(cur_off, ps, pstage);
        else if (row + warp_stride < B) issue_slice(nxt_off, ps - nsl, pstage);
        cp_async_commit();
      }
      if (sl == 0) load_meta(row + 2 * warp_stride, nn_i, nn_v);
      const uint32_t sbase = ring + stage * kSliceBytes + lane * 8;
      uint2 w[32];
#pragma unroll
      for (int j = 0; j < 32; ++j)
        asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(w[j].x), "=r"(w[j].y) : "r"(sbase + j * 256));
      float4 acc = *reinterpret_cast<const float4*>(s_bias + sl * 128 + lane * 4);
      if (dbg & 32) {
#pragma unroll
        for (int j = 0; j < 32; ++j) acc.x += __uint_as_float(w[j].x ^ w[j].y);
      } else if (dbg & 128) {
#pragma unroll
        for (int j = 0; j < 32; ++j) fhfma_bcast4(acc, w[j], my_hb);
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const uint32_t hb = __shfl_sync(0xffffffffu, my_hb, j);
          fhfma_bcast4(acc, w[j], hb);
        }
      }
      float4 r;
      r.x = acc.x - t.x; r.y = acc.y - t.y; r.z = acc.z - t.z; r.w = acc.w - t.w;
      sse_local = fmaf(r.x, r.x, sse_local);
      sse_local = fmaf(r.y, r.y, sse_local);
      sse_local = fmaf(r.z, r.z, sse_local);
      sse_local = fmaf(r.w, r.w, sse_local);
      __nv_bfloat162 rlo = __floats2bfloat162_rn(r.x, r.y);
      __nv_bfloat162 rhi = __floats2bfloat162_rn(r.z, r.w);
      uint2 rb;
      rb.x = *reinterpret_cast<uint32_t*>(&rlo);
      rb.y = *reinterpret_cast<uint32_t*>(&rhi);
      const size_t o = static_cast<size_t>(row) * d + sl * 128 + lane * 4;
      if (!(dbg & 2)) {
        if (resid != nullptr) *reinterpret_cast<float4*>(resid + o) = r;
        if (resid_bf16 != nullptr) *reinterpret_cast<uint2*>(resid_bf16 + o) = rb;
      }
      if (!(dbg & 16)) {
        float4 gs = *reinterpret_cast<float4*>(s_g + sl * 128 + lane * 4);
        gs.x += r.x; gs.y += r.y; gs.z += r.z; gs.w += r.w;
        *reinterpret_cast<float4*>(s_g + sl * 128 + lane * 4) = gs;
      }
      if (!(dbg & 64)) {
#pragma unroll
        for (int j = 0; j < 32; j += 2) {
          fhfma2(part[j], part[j + 1], w[j].x, rb.x, w[j + 1].x);
          fhfma2(part[j], part[j + 1], w[j].y, rb.y, w[j + 1].y);
        }
      }
      if (++stage == STAGES) stage = 0;
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
      const bool upper = (lane & off) != 0;
#pragma unroll
      for (int i = 0; i < off; ++i) {
        const float send = upper ? part[i] : part[i + off];
        const float keep = upper ? part[i + off] : part[i];
        part[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
      }
    }
    const float my_dv = fired ? s * part[0] : 0.f;
    if (lane < k && !(dbg & 8)) {
      if (dpre_val != nullptr) dpre_val[static_cast<size_t>(row) * k + lane] = my_dv;
      if (fired && d_b_enc != nullptr) {
        if (det_ws != nullptr) det_add(det_ws + my_i, static_cast<double>(part[0]), kDetScaleEnc);
        else atomicAdd(d_b_enc + my_i, my_dv);
      }
    }
    // rotate the metadata window
    cur_i = nxt_i; cur_v = nxt_v; cur_f = nxt_f; cur_off = nxt_off;
    nxt_i = nn_i; nxt_v = nn_v;
    nxt_f = (nxt_i >= 0) && (nxt_i < F) && (nxt_v > 0.f);
    nxt_off = row_offset(nxt_i, row + 2 * warp_stride);
  }
  cp_async_wait<0>();

  __shared__ float s_sse[kFusedWarps];
  __shared__ unsigned int s_l0[kFusedWarps];
  const float wsum = warp_sum(sse_local);
  if (lane == 0) {
    s_sse[warp] = wsum;
    s_l0[warp] = l0_local;
  }
  __syncthreads();
  if (stamp_words > 0 && last_activated != nullptr)
    for (int f = threadIdx.x; f < F; f += blockDim.x)
      if ((s_fired[f >> 5] >> (f & 31)) & 1u) last_activated[f] = stamp;
  if (d_b_dec != nullptr)
    for (int i = threadIdx.x; i < d; i += blockDim.x) {
      float t = 0.f;
#pragma unroll
      for (int w = 0; w < kFusedWarps; ++w) t += fsm[d + w * d + i];
      if (det_ws != nullptr) det_add(det_ws + F + i, static_cast<double>(t), kDetScaleDec);
      else atomicAdd(d_b_dec + i, s * t);
    }
  if (threadIdx.x == 0 && stats != nullptr) {
    double tsum = 0.0;
    unsigned long long c = 0;
    for (int w = 0; w < kFusedWarps; ++w) {
      tsum += static_cast<double>(s_sse[w]);
      c += s_l0[w];
    }
    if (det_ws != nullptr) det_add(det_ws + F + d, tsum, kDetScaleSse);
    else atomicAdd(&stats->sse, tsum);
    atomicAdd(&stats->l0_count, c);
  }
}

// ================================================================================================
// K23, tensor form (d % 128 == 0): fragment-order gather, dot products on the warp-level tensor pipe,
// the next 64 columns in flight while the current ones are multiplied.
//
// ncu of the staged kernel above (profiles/r2_k23_staged_ncu.txt): 1784 warp instructions per
// activation row at d = 384 and the issue slots 48 % busy with 8 warps per SM - the FHFMA form spends
// one instruction per (gathered row, 4 columns) on the reconstruction, another on the dot products,
// 64 shuffles per slice to broadcast (offset, h_j) and a 31-step shuffle transpose to reduce the 32
// partial sums.  The L2 gather itself (tools/l2_gather_bench: 115 us for the same bytes) is not
// what holds it at 223 us.  A first tensor form that ran BOTH contractions as mma.sync (fragments
// parked in shared memory, ldmatrix.trans for the reconstruction) halved the instruction count but
// moved every gathered byte through the LSU data pipe three times (LDG, STS, LDSM): 353 wavefronts per
// 128 columns, pipe 88 % busy, 341 us (profiles/r2_k23_tc_ldsm_rejected.txt).  This form moves them
// once:
//   * lane (rho = lane / 8, chi = lane % 8) loads, for its 8 entries j = 4 i + rho, the 16-byte
//     chunk chi of a 64-column half slice: one LDG.128 covers 4 rows x 128 contiguous bytes
//     (4 wavefronts per 512 B; the 8-rows-x-64-B pattern a plain A-fragment load needs costs 8).
//   * dot products: the four registers of a load are the A fragments of two mma.m16n8k16 whose 16
//     "rows" are (entry, column half beta = chi / 4) pairs: fragment row lane / 4 = 2 rho + beta reads
//     entry 4 i + rho over the columns 32 beta + 8 q + .., and column n = beta of B carries the bf16
//     residual of that half (lanes 0-3 and 4-7 load different 16-byte pieces of it).  D[2 rho + beta][beta]
//     is the partial dot product over one half; the two halves meet in one shuffle at the end of
//     the activation row.  8 HMMA per 64 columns, accumulators (16 registers) live across the row.
//   * reconstruction: the lane holds 8 entries x 8 columns, so the products h_j * W[j][c] are FHFMA
//     in registers with the activations h_j fetched ONCE per activation row (8 shuffles, not 32 per
//     slice), and the sum over the 4 entry groups rho is a 2-step shuffle transpose (6 exchanges)
//     that leaves every lane with 2 adjacent columns: coalesced 8-byte target loads, 4-byte bf16
//     residual stores.
// ~140 instructions per 64 columns (FHFMA form: 235), 40 LSU wavefronts; registers hold TWO half
// slices so the loads of the next one (of this activation row or the next) are in flight during the
// arithmetic.  Operands are the same bf16 values as in the other forms (bf16 x bf16 products, fp32
// accumulation), only the order of the fp32 sums differs.
// ================================================================================================
constexpr int kTcGBytes = 256;                       // bf16 residual of two half slices (ping-pong), per warp

// L2 eviction policies: the activation stream (B * d * 4 bytes per launch, read once) is marked
// evict_first and the gathered decoder rows (re-read ~B * k / F times each) evict_last, so the stream
// does not push decoder rows out of L2 (ncu at 768 -> 6144: 896 MB of DRAM traffic per launch against
// 350 MB of compulsory bytes without the hints).
__device__ __forceinline__ uint64_t l2_policy(int kind) {   // 0 = normal, 1 = evict_first, 2 = evict_last
  uint64_t pol;
  if (kind == 1)
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  else if (kind == 2)
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  else
    asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}

template <bool kAllocL1>
__device__ __forceinline__ uint4 ldg_nc_v4(const void* p, uint64_t pol) {
  uint4 v;
  if (kAllocL1)
    asm volatile("ld.global.nc.L2::cache_hint.v4.u32 {%0, %1, %2, %3}, [%4], %5;"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                 : "l"(p), "l"(pol));
  else
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.u32 {%0, %1, %2, %3}, [%4], %5;"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                 : "l"(p), "l"(pol));
  return v;
}
__device__ __forceinline__ float2 ldg_stream_v2(const float* p, uint64_t pol) {
  float2 v;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v2.f32 {%0, %1}, [%2], %3;"
               : "=f"(v.x), "=f"(v.y)
               : "l"(p), "l"(pol));
  return v;
}
// The 2 target columns a lane of the tensor / team forms holds in flight, as loaded: fp32 pairs are
// loaded as float2 (8 bytes), half pairs as their raw 4 bytes and converted where they are used, so the
// load never waits on its own conversion.
template <typename TX>
struct XPair {
  using type = uint32_t;
};
template <>
struct XPair<float> {
  using type = float2;
};
__device__ __forceinline__ float2 ldg_stream_x2(const float* p, uint64_t pol) { return ldg_stream_v2(p, pol); }
template <typename TX>
__device__ __forceinline__ uint32_t ldg_stream_x2(const TX* p, uint64_t pol) {
  uint32_t v;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.b32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
  return v;
}
__device__ __forceinline__ float2 xpair_to_float2(float2 v, const float*) { return v; }
template <typename TX>
__device__ __forceinline__ float2 xpair_to_float2(uint32_t v, const TX* tag) { return x2_to_float2(v, tag); }

// acc[0..3] += bf16x2(w0).{lo,hi}, bf16x2(w1).{lo,hi} times bf16(h.lo)
__device__ __forceinline__ void fhfma_row4(float* acc, uint32_t w0, uint32_t w1, uint32_t h) {
  asm("{\n\t"
      ".reg .b16 a0, a1, c0, c1, h0, h1;\n\t"
      "mov.b32 {a0, a1}, %4;\n\t"
      "mov.b32 {c0, c1}, %5;\n\t"
      "mov.b32 {h0, h1}, %6;\n\t"
      "fma.rn.f32.bf16 %0, a0, h0, %0;\n\t"
      "fma.rn.f32.bf16 %1, a1, h0, %1;\n\t"
      "fma.rn.f32.bf16 %2, c0, h0, %2;\n\t"
      "fma.rn.f32.bf16 %3, c1, h0, %3;\n\t"
      "}\n"
      : "+f"(acc[0]), "+f"(acc[1]), "+f"(acc[2]), "+f"(acc[3])
      : "r"(w0), "r"(w1), "r"(h));
}

// acc[0..3] += bf16x2(w0).{lo,hi}, bf16x2(w1).{lo,hi} times the HIGH half of h
__device__ __forceinline__ void fhfma_row4_hi(float* acc, uint32_t w0, uint32_t w1, uint32_t h) {
  asm("{\n\t"
      ".reg .b16 a0, a1, c0, c1, h0, h1;\n\t"
      "mov.b32 {a0, a1}, %4;\n\t"
      "mov.b32 {c0, c1}, %5;\n\t"
      "mov.b32 {h0, h1}, %6;\n\t"
      "fma.rn.f32.bf16 %0, a0, h1, %0;\n\t"
      "fma.rn.f32.bf16 %1, a1, h1, %1;\n\t"
      "fma.rn.f32.bf16 %2, c0, h1, %2;\n\t"
      "fma.rn.f32.bf16 %3, c1, h1, %3;\n\t"
      "}\n"
      : "+f"(acc[0]), "+f"(acc[1]), "+f"(acc[2]), "+f"(acc[3])
      : "r"(w0), "r"(w1), "r"(h));
}

// STAGES half slices live in registers: one being multiplied, STAGES - 1 in flight (d / 64 must be a
// multiple of STAGES).
template <int kMinBlocks, int STAGES, bool PF, typename TX>
__global__ void __launch_bounds__(kFusedWarps * 32, kMinBlocks)
decode_backward_tc_kernel(const TX* __restrict__ target, const __nv_bfloat16* __restrict__ w_decT,
                          const float* __restrict__ b_dec, const float* __restrict__ b_pre,
                          const int32_t* __restrict__ idx, const float* __restrict__ val,
                          const float* __restrict__ grad_out, float coef, int B, int d, int F, int k,
                          float* __restrict__ resid, __nv_bfloat16* __restrict__ resid_bf16,
                          FusedStats* __restrict__ stats, long long* __restrict__ last_activated,
                          const long long* __restrict__ step_count, float* __restrict__ d_b_enc,
                          float* __restrict__ d_b_dec, float* __restrict__ dpre_val,
                          const TX* const* __restrict__ target_at,
                          const long long* const* __restrict__ rows_at, int stamp_words,
                          long long* __restrict__ det_ws, int pf_dist, int l2hint) {
  static_assert(STAGES == 2 || STAGES == 3, "two or three half slices in registers");
  const uint64_t pol_x = l2_policy((l2hint & 1) ? 1 : 0);      // activation stream
  const uint64_t pol_w = l2_policy((l2hint & 2) ? 2 : 0);      // gathered decoder rows
  // [d] bias | [warps][d] db_dec partials | [warps] bf16 residual ping-pong + 16 zero bytes | fired bitmap
  extern __shared__ __align__(16) float fsm[];
  pdl_prologue();
  if (target_at != nullptr) target = *target_at;
  const long long* perm = rows_at != nullptr ? *rows_at : nullptr;
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int rho = lane >> 3;                 // entry group: this lane gathers entries 4 i + rho
  const int chi = lane & 7;                  // 16-byte chunk of the 64-column half slice
  float* s_bias = fsm;
  float* s_g = fsm + d + warp * d;
  char* dyn = reinterpret_cast<char*>(fsm + (1 + kFusedWarps) * d);
  const uint32_t gbuf = smem_u32(dyn) + warp * kTcGBytes;
  const uint32_t zbuf = smem_u32(dyn) + kFusedWarps * kTcGBytes;     // 16 zero bytes
  uint32_t* s_fired = reinterpret_cast<uint32_t*>(dyn + kFusedWarps * kTcGBytes + 16);
  if (threadIdx.x < 4) reinterpret_cast<uint32_t*>(dyn + kFusedWarps * kTcGBytes)[threadIdx.x] = 0u;
  for (int i = threadIdx.x; i < stamp_words; i += blockDim.x) s_fired[i] = 0u;
  for (int i = threadIdx.x; i < d; i += blockDim.x) {
    s_bias[i] = b_dec[i] + (b_pre != nullptr ? b_pre[i] : 0.f);
#pragma unroll
    for (int w = 0; w < kFusedWarps; ++w) fsm[d + w * d + i] = 0.f;
  }
  __syncthreads();

  const float s = coef * (grad_out != nullptr ? *grad_out : 1.f);
  const long long stamp = (last_activated != nullptr && step_count != nullptr) ? (*step_count + 1) : 0;
  const int warp_global = blockIdx.x * kFusedWarps + warp;
  const int warp_stride = gridDim.x * kFusedWarps;
  const int nhs = d >> 6;                    // half slices (64 columns) per activation row
  const char* wbytes = reinterpret_cast<const char*>(w_decT);
  const size_t row_bytes = static_cast<size_t>(d) * 2;
  // after the shuffle transpose this lane owns 2 adjacent columns of every half slice
  const int b4 = (lane >> 4) & 1, b3 = (lane >> 3) & 1;
  const int c0 = 8 * chi + 4 * b4 + 2 * b3;
  // The bf16 residual of a half slice is parked chunk by chunk (16 bytes = 8 columns) with the column
  // pairs in the order (0,1) (4,5) (2,3) (6,7): the HMMA below takes an LDG.128 register quad as its A
  // operand, i.e. fragment row r reads pairs (0,1) | (4,5) and row r + 8 pairs (2,3) | (6,7) of the
  // lane's chunk, so the matching B pieces are 8 adjacent bytes.
  const uint32_t g_st = static_cast<uint32_t>(chi * 16 + (b4 + 2 * b3) * 4);
  // B column n = lane / 4 stands for (column half beta = n & 1, fragment-row half gam = (n >> 1) & 1);
  // columns 0-3 serve the even entry of a pair, 4-7 the odd one: the other set reads zeros
  const int nB = lane >> 2;
  const uint32_t g_ld = static_cast<uint32_t>(((nB & 1) * 4 + (lane & 3)) * 16 + ((nB >> 1) & 1) * 8);
  const bool lowB = nB < 4;

  float sse_local = 0.f;
  unsigned int l0_local = 0;

  auto load_meta = [&](int row, int32_t& mi, float& mv) {
    mi = -1;
    mv = 0.f;
    if (row < B && lane < k) {
      mi = __ldg(idx + static_cast<size_t>(row) * k + lane);
      mv = __ldg(val + static_cast<size_t>(row) * k + lane);
    }
  };
  // entries that did not fire gather their own row with weight 0; invalid ones a row that differs
  // per (activation row, lane) - no L2 hot spot (see the staged kernel)
  auto gather_feature = [&](int32_t mi, int row) -> uint32_t {
    return (mi >= 0 && mi < F) ? static_cast<uint32_t>(mi)
                               : (static_cast<uint32_t>(row) * 37u + static_cast<uint32_t>(lane)) % static_cast<uint32_t>(F);
  };
  const char* wp[8];                         // this lane's 8 gathered rows (+ its chunk), at the current half slice
  auto set_row = [&](uint32_t feat) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const uint32_t f = __shfl_sync(0xffffffffu, feat, 4 * i + rho);
      wp[i] = wbytes + static_cast<size_t>(f) * row_bytes + chi * 16;
    }
  };
  using XP = typename XPair<TX>::type;
  const TX* trow = target;                   // this lane's 2 target columns, at the current half slice
  auto set_target = [&](int row) {
    const size_t srow = perm != nullptr ? static_cast<size_t>(__ldg(perm + row)) : static_cast<size_t>(row);
    trow = target + srow * d + c0;
  };
  auto gather = [&](uint4 (&w)[8], XP& x, int ahead) {     // `ahead` half slices past the current one
#pragma unroll
    for (int i = 0; i < 8; ++i) w[i] = ldg_nc_v4<PF>(wp[i] + ahead * 128, pol_w);
    x = ldg_stream_x2(trow + ahead * 64, pol_x);
  };
  // PF: every lane asks for ONE 128-byte line of ITS entry's row, pf_dist half slices past the one
  // being gathered - a single instruction per half slice brings all 32 lines (4 KB) into L1 without
  // holding registers; the LDG.128 of the gather then hit L1
  const char* pf_cur = wbytes;               // row of this lane's entry, this activation row / the next
  const char* pf_nxt = wbytes;
  auto prefetch = [&](int h, bool more_rows) {
    if (!PF) return;
    const char* p = pf_cur + h * 128;
    if (h >= nhs) {
      if (!more_rows || h - nhs >= nhs) return;
      p = pf_nxt + (h - nhs) * 128;
    }
    asm volatile("prefetch.global.L1 [%0];" ::"l"(p));
  };
  auto advance = [&](int n) {
#pragma unroll
    for (int i = 0; i < 8; ++i) wp[i] += n * 128;
    trow += n * 64;
  };

  int row = warp_global;
  int32_t cur_i, nxt_i;
  float cur_v, nxt_v;
  load_meta(row, cur_i, cur_v);
  load_meta(row + warp_stride, nxt_i, nxt_v);
  uint4 w0[8], w1[8], w2[8];   // w2: three-stage form only (dead otherwise)
  XP x0{}, x1 = x0, x2 = x0;
  if (row < B) {
    set_row(gather_feature(cur_i, row));
    set_target(row);
    gather(w0, x0, 0);
    if (STAGES == 3) gather(w1, x1, 1);
  }
  if (PF) pf_nxt = wbytes + static_cast<size_t>(gather_feature(cur_i, row)) * row_bytes;

  for (; row < B; row += warp_stride) {
    const int32_t my_i = cur_i;
    const bool fired = (my_i >= 0) && (my_i < F) && (cur_v > 0.f);
    if (fired && last_activated != nullptr) {
      if (stamp_words > 0) atomicOr(&s_fired[my_i >> 5], 1u << (my_i & 31));
      else last_activated[my_i] = stamp;
    }
    const float my_v = fired ? cur_v : 0.f;
    const uint32_t my_hb = static_cast<uint32_t>(__bfloat16_as_ushort(__float2bfloat16_rn(my_v)));
    const uint32_t mask = __ballot_sync(0xffffffffu, fired);
    l0_local += (lane == 0) ? __popc(mask) : 0;
    uint32_t hp[4];                          // bf16 activations of entries 8 m + rho (low half) and 8 m + 4 + rho (high)
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      const uint32_t lo = __shfl_sync(0xffffffffu, my_hb, 8 * m + rho);
      const uint32_t hi = __shfl_sync(0xffffffffu, my_hb, 8 * m + 4 + rho);
      hp[m] = lo | (hi << 16);
    }
    const size_t orow = static_cast<size_t>(row) * d + c0;
    int32_t nn_i = -1;                       // entries two rows ahead
    float nn_v = 0.f;
    const bool more = row + warp_stride < B;
    if (PF) {
      pf_cur = pf_nxt;
      pf_nxt = wbytes + static_cast<size_t>(gather_feature(nxt_i, row + warp_stride)) * row_bytes;
    }

    float dacc[4][4];                        // pair p: entries 8 p + rho (B columns 0-3) and 8 p + 4 + rho (4-7)
#pragma unroll
    for (int p = 0; p < 4; ++p) dacc[p][0] = dacc[p][1] = dacc[p][2] = dacc[p][3] = 0.f;

    auto compute = [&](const uint4 (&w)[8], const XP xp, int hs) {
      const float2 x = xpair_to_float2(xp, static_cast<const TX*>(nullptr));
      // ---- reconstruction partials: 8 entries x 8 columns in this lane ----
      float part[8];
#pragma unroll
      for (int c = 0; c < 8; ++c) part[c] = 0.f;
#pragma unroll
      for (int m = 0; m < 4; ++m) {
        fhfma_row4(part, w[2 * m].x, w[2 * m].y, hp[m]);
        fhfma_row4(part + 4, w[2 * m].z, w[2 * m].w, hp[m]);
        fhfma_row4_hi(part, w[2 * m + 1].x, w[2 * m + 1].y, hp[m]);
        fhfma_row4_hi(part + 4, w[2 * m + 1].z, w[2 * m + 1].w, hp[m]);
      }
      // ---- sum over the 4 entry groups (lane bits 4, 3); this lane keeps columns c0, c0 + 1 ----
      {
        const bool up = b4 != 0;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const float send = up ? part[c] : part[c + 4];
          const float keep = up ? part[c + 4] : part[c];
          part[c] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
        }
      }
      {
        const bool up = b3 != 0;
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          const float send = up ? part[c] : part[c + 2];
          const float keep = up ? part[c + 2] : part[c];
          part[c] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
        }
      }
      // ---- residual, SSE, decoder-bias gradient, bf16 residual ----
      const int col = hs * 64 + c0;
      const float2 bias = *reinterpret_cast<const float2*>(s_bias + col);
      const float r0 = part[0] + bias.x - x.x;
      const float r1 = part[1] + bias.y - x.y;
      sse_local = fmaf(r0, r0, sse_local);
      sse_local = fmaf(r1, r1, sse_local);
      float2 gs = *reinterpret_cast<float2*>(s_g + col);
      gs.x += r0;
      gs.y += r1;
      *reinterpret_cast<float2*>(s_g + col) = gs;
      if (resid != nullptr) *reinterpret_cast<float2*>(resid + orow + hs * 64) = make_float2(r0, r1);
      __nv_bfloat162 rb2 = __floats2bfloat162_rn(r0, r1);
      const uint32_t rb = *reinterpret_cast<uint32_t*>(&rb2);
      if (resid_bf16 != nullptr) *reinterpret_cast<uint32_t*>(resid_bf16 + orow + hs * 64) = rb;
      const uint32_t gb = gbuf + (hs & 1) * 128;
      asm volatile("st.shared.u32 [%0], %1;" ::"r"(gb + g_st), "r"(rb) : "memory");
      __syncwarp();
      // ---- dot products: A = one gathered register quad, B = the residual (or zeros) ----
      uint32_t ge0, ge1, go0, go1;
      asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(ge0), "=r"(ge1) : "r"(lowB ? gb + g_ld : zbuf));
      asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(go0), "=r"(go1) : "r"(lowB ? zbuf : gb + g_ld));
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        mma_bf16_16816(dacc[p], w[2 * p].x, w[2 * p].y, w[2 * p].z, w[2 * p].w, ge0, ge1);
        mma_bf16_16816(dacc[p], w[2 * p + 1].x, w[2 * p + 1].y, w[2 * p + 1].z, w[2 * p + 1].w, go0, go1);
      }
    };
    auto next_row = [&]() {                  // all of this row's gathers are out: retarget the pointers
      set_row(gather_feature(nxt_i, row + warp_stride));
      set_target(row + warp_stride);
    };

    if constexpr (STAGES == 2) {
      for (int hs = 0; hs < nhs; hs += 2) {
        gather(w1, x1, 1);
        prefetch(hs + 1 + pf_dist, more);
        if (hs == 0) load_meta(row + 2 * warp_stride, nn_i, nn_v);
        compute(w0, x0, hs);
        const bool last = hs + 2 >= nhs;
        prefetch(hs + 2 + pf_dist, more);
        if (!last) {
          gather(w0, x0, 2);
        } else if (more) {
          next_row();
          gather(w0, x0, 0);
        }
        compute(w1, x1, hs + 1);
        if (!last) advance(2);
      }
    } else {
      for (int hs = 0; hs < nhs; hs += 3) {
        gather(w2, x2, 2);
        if (hs == 0) load_meta(row + 2 * warp_stride, nn_i, nn_v);
        compute(w0, x0, hs);
        const bool last = hs + 3 >= nhs;
        if (!last) {
          gather(w0, x0, 3);
        } else if (more) {
          next_row();
          gather(w0, x0, 0);
        }
        compute(w1, x1, hs + 1);
        if (!last) {
          gather(w1, x1, 4);
        } else if (more) {
          gather(w1, x1, 1);
        }
        compute(w2, x2, hs + 2);
        if (!last) advance(3);
      }
    }

    // Pair p, lane (r = lane / 4, q = lane % 4): the partial dot product of entry 8 p + 4 (q / 2) + rho
    // over the column quarter (beta = r & 1, gam = q & 1) is D[r + 8 gam][2 q + beta]; the four
    // quarters meet through lanes ^ 4 and ^ 1.  Lane j then takes dot[j] from lane 8 (j % 4) + 2 ((j / 4) % 2)
    // of pair j / 8.
    const bool beta = (lane & 4) != 0, gam = (lane & 1) != 0;
    const int src = 8 * (lane & 3) + 2 * ((lane >> 2) & 1);
    float dot = 0.f;
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      float t = gam ? (beta ? dacc[p][3] : dacc[p][2]) : (beta ? dacc[p][1] : dacc[p][0]);
      t += __shfl_xor_sync(0xffffffffu, t, 4);
      t += __shfl_xor_sync(0xffffffffu, t, 1);
      const float v = __shfl_sync(0xffffffffu, t, src);
      if ((lane >> 3) == p) dot = v;
    }
    const float my_dv = fired ? s * dot : 0.f;
    if (lane < k) {
      if (dpre_val != nullptr) dpre_val[static_cast<size_t>(row) * k + lane] = my_dv;
      if (fired && d_b_enc != nullptr) {
        if (det_ws != nullptr) det_add(det_ws + my_i, static_cast<double>(dot), kDetScaleEnc);
        else atomicAdd(d_b_enc + my_i, my_dv);
      }
    }
    cur_i = nxt_i; cur_v = nxt_v;
    nxt_i = nn_i; nxt_v = nn_v;
  }

  __shared__ float s_sse[kFusedWarps];
  __shared__ unsigned int s_l0[kFusedWarps];
  const float wsum = warp_sum(sse_local);
  if (lane == 0) {
    s_sse[warp] = wsum;
    s_l0[warp] = l0_local;
  }
  __syncthreads();
  if (stamp_words > 0 && last_activated != nullptr)
    for (int f = threadIdx.x; f < F; f += blockDim.x)
      if ((s_fired[f >> 5] >> (f & 31)) & 1u) last_activated[f] = stamp;
  if (d_b_dec != nullptr)
    for (int i = threadIdx.x; i < d; i += blockDim.x) {
      float t = 0.f;
#pragma unroll
      for (int w = 0; w < kFusedWarps; ++w) t += fsm[d + w * d + i];
      if (det_ws != nullptr) det_add(det_ws + F + i, static_cast<double>(t), kDetScaleDec);
      else atomicAdd(d_b_dec + i, s * t);
    }
  if (threadIdx.x == 0 && stats != nullptr) {
    double tsum = 0.0;
    unsigned long long c = 0;
    for (int w = 0; w < kFusedWarps; ++w) {
      tsum += static_cast<double>(s_sse[w]);
      c += s_l0[w];
    }
    if (det_ws != nullptr) det_add(det_ws + F + d, tsum, kDetScaleSse);
    else atomicAdd(&stats->sse, tsum);
    atomicAdd(&stats->l0_count, c);
  }
}

// ================================================================================================
// K23, wide form (32 < k <= 256, d % 128 == 0): a TEAM of ceil(k / 32) warps per activation row.
//
// The tensor form above needs every 64-column half slice of all k gathered rows in one warp's
// registers; that is what caps it at k = 32.  Here warp w of a team owns the selected entries
// [32 w, 32 w + 32) of the row and runs the tensor form's slice code on them unchanged (fragment-order
// LDG.128 gather, FHFMA.BF16 partial reconstruction, mma.sync dot products against the bf16
// residual).  Per half slice the warps meet once:
//   1. each warp parks its partial reconstruction of the 64 columns in shared memory (ping-pong by
//      half-slice parity) and the team meets at a named barrier (bar.sync 1 + team, 32 * team size);
//   2. every warp sums the team's partials in warp order - the same fp32 additions in every warp, so
//      every warp holds the same residual - and forms the residual; warp 0 of the team alone writes
//      resid / resid_bf16 and accumulates the SSE and the decoder-bias gradient;
//   3. every warp runs its dot products against the bf16 residual with the decoder registers it holds.
// A warp reads a partial buffer again only two half slices later, after the next barrier, so one
// barrier per half slice is enough.  Each decoder row is still gathered once; the cost over the
// tensor form is one shared-memory exchange and one barrier per half slice.  Entries past k (the tail
// of the last warp) get activation 0 and gather a spread-out row, like the tensor form's invalid
// entries: they add nothing and get no dv.
//
// kDet (deterministic form, det_ws as in wsae_decode_backward_det): the three cross-row sums go to
// det_ws with det_add instead of float atomics - db_enc one unscaled dot product per fired entry,
// db_dec the block's per-team partials summed in team order, the SSE the block's per-warp partials
// summed in warp order.  A feature appears at most once among a row's k entries, so it still gets at
// most one db_enc addend per row whatever k is, and the int64 headroom of kDetScaleEnc holds as at
// k <= 32.  kDet = false is the default form, unchanged (det_ws unused).
// ================================================================================================
constexpr int kWideMaxK = 256;
constexpr int kWideMaxWarps = 8;

__device__ __forceinline__ void team_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

template <bool kDet, typename TX>
__global__ void __maxnreg__(160)   // 156 registers, no spills: the tensor form's budget
decode_backward_wide_kernel(const TX* __restrict__ target, const __nv_bfloat16* __restrict__ w_decT,
                            const float* __restrict__ b_dec, const float* __restrict__ b_pre,
                            const int32_t* __restrict__ idx, const float* __restrict__ val,
                            const float* __restrict__ grad_out, float coef, int B, int d, int F, int k,
                            float* __restrict__ resid, __nv_bfloat16* __restrict__ resid_bf16,
                            FusedStats* __restrict__ stats, long long* __restrict__ last_activated,
                            const long long* __restrict__ step_count, float* __restrict__ d_b_enc,
                            float* __restrict__ d_b_dec, float* __restrict__ dpre_val,
                            const TX* const* __restrict__ target_at,
                            const long long* const* __restrict__ rows_at, int stamp_words, int l2hint,
                            long long* __restrict__ det_ws) {
  const uint64_t pol_x = l2_policy((l2hint & 1) ? 1 : 0);
  const uint64_t pol_w = l2_policy((l2hint & 2) ? 2 : 0);
  // [d] bias | [teams][d] db_dec partials | [2][warps][64] partial reconstructions |
  // [warps] bf16 residual ping-pong + 16 zero bytes | fired bitmap
  extern __shared__ __align__(16) float fsm[];
  pdl_prologue();
  if (target_at != nullptr) target = *target_at;
  const long long* perm = rows_at != nullptr ? *rows_at : nullptr;
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int nwarps = blockDim.x >> 5;
  const int tsize = (k + 31) >> 5;           // warps per team
  const int teams = nwarps / tsize;
  const int team = warp / tsize;
  const int tw = warp - team * tsize;        // rank in the team: owns entries [32 tw, 32 tw + 32)
  const int entry = 32 * tw + lane;
  const int bar_id = 1 + team;
  const int bar_n = 32 * tsize;
  const int rho = lane >> 3;
  const int chi = lane & 7;
  float* s_bias = fsm;
  float* s_g = fsm + d + team * d;
  float* s_part = fsm + (1 + teams) * d;
  char* dyn = reinterpret_cast<char*>(s_part + 2 * nwarps * 64);
  const uint32_t gbuf = smem_u32(dyn) + warp * kTcGBytes;
  const uint32_t zbuf = smem_u32(dyn) + nwarps * kTcGBytes;
  uint32_t* s_fired = reinterpret_cast<uint32_t*>(dyn + nwarps * kTcGBytes + 16);
  if (threadIdx.x < 4) reinterpret_cast<uint32_t*>(dyn + nwarps * kTcGBytes)[threadIdx.x] = 0u;
  for (int i = threadIdx.x; i < stamp_words; i += blockDim.x) s_fired[i] = 0u;
  for (int i = threadIdx.x; i < d; i += blockDim.x) {
    s_bias[i] = b_dec[i] + (b_pre != nullptr ? b_pre[i] : 0.f);
    for (int t = 0; t < teams; ++t) fsm[d + t * d + i] = 0.f;
  }
  __syncthreads();

  const float s = coef * (grad_out != nullptr ? *grad_out : 1.f);
  const long long stamp = (last_activated != nullptr && step_count != nullptr) ? (*step_count + 1) : 0;
  const int team_global = blockIdx.x * teams + team;
  const int team_stride = gridDim.x * teams;
  const int nhs = d >> 6;
  const char* wbytes = reinterpret_cast<const char*>(w_decT);
  const size_t row_bytes = static_cast<size_t>(d) * 2;
  const int b4 = (lane >> 4) & 1, b3 = (lane >> 3) & 1;
  const int c0 = 8 * chi + 4 * b4 + 2 * b3;
  const uint32_t g_st = static_cast<uint32_t>(chi * 16 + (b4 + 2 * b3) * 4);
  const int nB = lane >> 2;
  const uint32_t g_ld = static_cast<uint32_t>(((nB & 1) * 4 + (lane & 3)) * 16 + ((nB >> 1) & 1) * 8);
  const bool lowB = nB < 4;
  const bool lead = tw == 0;                 // writes the row's residual, SSE and db_dec partials

  float sse_local = 0.f;
  unsigned int l0_local = 0;

  auto load_meta = [&](int row, int32_t& mi, float& mv) {
    mi = -1;
    mv = 0.f;
    if (row < B && entry < k) {
      mi = __ldg(idx + static_cast<size_t>(row) * k + entry);
      mv = __ldg(val + static_cast<size_t>(row) * k + entry);
    }
  };
  auto gather_feature = [&](int32_t mi, int row) -> uint32_t {
    return (mi >= 0 && mi < F) ? static_cast<uint32_t>(mi)
                               : (static_cast<uint32_t>(row) * 37u + static_cast<uint32_t>(entry)) % static_cast<uint32_t>(F);
  };
  const char* wp[8];
  auto set_row = [&](uint32_t feat) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const uint32_t f = __shfl_sync(0xffffffffu, feat, 4 * i + rho);
      wp[i] = wbytes + static_cast<size_t>(f) * row_bytes + chi * 16;
    }
  };
  using XP = typename XPair<TX>::type;
  const TX* trow = target;
  auto set_target = [&](int row) {
    const size_t srow = perm != nullptr ? static_cast<size_t>(__ldg(perm + row)) : static_cast<size_t>(row);
    trow = target + srow * d + c0;
  };
  auto gather = [&](uint4 (&w)[8], XP& x, int ahead) {
#pragma unroll
    for (int i = 0; i < 8; ++i) w[i] = ldg_nc_v4<false>(wp[i] + ahead * 128, pol_w);
    x = ldg_stream_x2(trow + ahead * 64, pol_x);
  };
  auto advance = [&](int n) {
#pragma unroll
    for (int i = 0; i < 8; ++i) wp[i] += n * 128;
    trow += n * 64;
  };

  int row = team_global;
  int32_t cur_i, nxt_i;
  float cur_v, nxt_v;
  load_meta(row, cur_i, cur_v);
  load_meta(row + team_stride, nxt_i, nxt_v);
  uint4 w0[8], w1[8];
  XP x0{}, x1 = x0;
  if (row < B) {
    set_row(gather_feature(cur_i, row));
    set_target(row);
    gather(w0, x0, 0);
  }

  for (; row < B; row += team_stride) {
    const int32_t my_i = cur_i;
    const bool fired = (my_i >= 0) && (my_i < F) && (cur_v > 0.f);
    if (fired && last_activated != nullptr) {
      if (stamp_words > 0) atomicOr(&s_fired[my_i >> 5], 1u << (my_i & 31));
      else last_activated[my_i] = stamp;
    }
    const float my_v = fired ? cur_v : 0.f;
    const uint32_t my_hb = static_cast<uint32_t>(__bfloat16_as_ushort(__float2bfloat16_rn(my_v)));
    const uint32_t mask = __ballot_sync(0xffffffffu, fired);
    l0_local += (lane == 0) ? __popc(mask) : 0;
    uint32_t hp[4];
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      const uint32_t lo = __shfl_sync(0xffffffffu, my_hb, 8 * m + rho);
      const uint32_t hi = __shfl_sync(0xffffffffu, my_hb, 8 * m + 4 + rho);
      hp[m] = lo | (hi << 16);
    }
    const size_t orow = static_cast<size_t>(row) * d + c0;
    int32_t nn_i = -1;
    float nn_v = 0.f;
    const bool more = row + team_stride < B;

    float dacc[4][4];
#pragma unroll
    for (int p = 0; p < 4; ++p) dacc[p][0] = dacc[p][1] = dacc[p][2] = dacc[p][3] = 0.f;

    auto compute = [&](const uint4 (&w)[8], const XP xp, int hs) {
      const float2 x = xpair_to_float2(xp, static_cast<const TX*>(nullptr));
      float part[8];
#pragma unroll
      for (int c = 0; c < 8; ++c) part[c] = 0.f;
#pragma unroll
      for (int m = 0; m < 4; ++m) {
        fhfma_row4(part, w[2 * m].x, w[2 * m].y, hp[m]);
        fhfma_row4(part + 4, w[2 * m].z, w[2 * m].w, hp[m]);
        fhfma_row4_hi(part, w[2 * m + 1].x, w[2 * m + 1].y, hp[m]);
        fhfma_row4_hi(part + 4, w[2 * m + 1].z, w[2 * m + 1].w, hp[m]);
      }
      {
        const bool up = b4 != 0;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const float send = up ? part[c] : part[c + 4];
          const float keep = up ? part[c + 4] : part[c];
          part[c] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
        }
      }
      {
        const bool up = b3 != 0;
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          const float send = up ? part[c] : part[c + 2];
          const float keep = up ? part[c + 2] : part[c];
          part[c] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
        }
      }
      // ---- team exchange: this warp's 32 entries -> the row's reconstruction of the 64 columns ----
      float* pbuf = s_part + (hs & 1) * nwarps * 64;
      *reinterpret_cast<float2*>(pbuf + warp * 64 + c0) = make_float2(part[0], part[1]);
      team_sync(bar_id, bar_n);
      float2 rec = make_float2(0.f, 0.f);
      for (int t = 0; t < tsize; ++t) {
        const float2 p = *reinterpret_cast<const float2*>(pbuf + (team * tsize + t) * 64 + c0);
        rec.x += p.x;
        rec.y += p.y;
      }
      const int col = hs * 64 + c0;
      const float2 bias = *reinterpret_cast<const float2*>(s_bias + col);
      const float r0 = rec.x + bias.x - x.x;
      const float r1 = rec.y + bias.y - x.y;
      __nv_bfloat162 rb2 = __floats2bfloat162_rn(r0, r1);
      const uint32_t rb = *reinterpret_cast<uint32_t*>(&rb2);
      if (lead) {
        sse_local = fmaf(r0, r0, sse_local);
        sse_local = fmaf(r1, r1, sse_local);
        float2 gs = *reinterpret_cast<float2*>(s_g + col);
        gs.x += r0;
        gs.y += r1;
        *reinterpret_cast<float2*>(s_g + col) = gs;
        if (resid != nullptr) *reinterpret_cast<float2*>(resid + orow + hs * 64) = make_float2(r0, r1);
        if (resid_bf16 != nullptr) *reinterpret_cast<uint32_t*>(resid_bf16 + orow + hs * 64) = rb;
      }
      const uint32_t gb = gbuf + (hs & 1) * 128;
      asm volatile("st.shared.u32 [%0], %1;" ::"r"(gb + g_st), "r"(rb) : "memory");
      __syncwarp();
      uint32_t ge0, ge1, go0, go1;
      asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(ge0), "=r"(ge1) : "r"(lowB ? gb + g_ld : zbuf));
      asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(go0), "=r"(go1) : "r"(lowB ? zbuf : gb + g_ld));
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        mma_bf16_16816(dacc[p], w[2 * p].x, w[2 * p].y, w[2 * p].z, w[2 * p].w, ge0, ge1);
        mma_bf16_16816(dacc[p], w[2 * p + 1].x, w[2 * p + 1].y, w[2 * p + 1].z, w[2 * p + 1].w, go0, go1);
      }
    };

    for (int hs = 0; hs < nhs; hs += 2) {
      gather(w1, x1, 1);
      if (hs == 0) load_meta(row + 2 * team_stride, nn_i, nn_v);
      compute(w0, x0, hs);
      const bool last = hs + 2 >= nhs;
      if (!last) {
        gather(w0, x0, 2);
      } else if (more) {
        set_row(gather_feature(nxt_i, row + team_stride));
        set_target(row + team_stride);
        gather(w0, x0, 0);
      }
      compute(w1, x1, hs + 1);
      if (!last) advance(2);
    }

    // dot products: the tensor form's reduction (lane j ends with the dot product of its entry)
    const bool beta = (lane & 4) != 0, gam = (lane & 1) != 0;
    const int src = 8 * (lane & 3) + 2 * ((lane >> 2) & 1);
    float dot = 0.f;
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      float t = gam ? (beta ? dacc[p][3] : dacc[p][2]) : (beta ? dacc[p][1] : dacc[p][0]);
      t += __shfl_xor_sync(0xffffffffu, t, 4);
      t += __shfl_xor_sync(0xffffffffu, t, 1);
      const float v = __shfl_sync(0xffffffffu, t, src);
      if ((lane >> 3) == p) dot = v;
    }
    const float my_dv = fired ? s * dot : 0.f;
    if (entry < k) {
      if (dpre_val != nullptr) dpre_val[static_cast<size_t>(row) * k + entry] = my_dv;
      if (fired && d_b_enc != nullptr) {
        if constexpr (kDet) det_add(det_ws + my_i, static_cast<double>(dot), kDetScaleEnc);
        else atomicAdd(d_b_enc + my_i, my_dv);
      }
    }
    cur_i = nxt_i; cur_v = nxt_v;
    nxt_i = nn_i; nxt_v = nn_v;
  }

  __shared__ float s_sse[kWideMaxWarps];
  __shared__ unsigned int s_l0[kWideMaxWarps];
  const float wsum = warp_sum(sse_local);
  if (lane == 0) {
    s_sse[warp] = wsum;
    s_l0[warp] = l0_local;
  }
  __syncthreads();
  if (stamp_words > 0 && last_activated != nullptr)
    for (int f = threadIdx.x; f < F; f += blockDim.x)
      if ((s_fired[f >> 5] >> (f & 31)) & 1u) last_activated[f] = stamp;
  if (d_b_dec != nullptr)
    for (int i = threadIdx.x; i < d; i += blockDim.x) {
      float t = 0.f;
      for (int tm = 0; tm < teams; ++tm) t += fsm[d + tm * d + i];
      if constexpr (kDet) det_add(det_ws + F + i, static_cast<double>(t), kDetScaleDec);
      else atomicAdd(d_b_dec + i, s * t);
    }
  if (threadIdx.x == 0 && stats != nullptr) {
    double tsum = 0.0;
    unsigned long long c = 0;
    for (int w = 0; w < nwarps; ++w) {
      tsum += static_cast<double>(s_sse[w]);
      c += s_l0[w];
    }
    if constexpr (kDet) det_add(det_ws + F + d, tsum, kDetScaleSse);
    else atomicAdd(&stats->sse, tsum);
    atomicAdd(&stats->l0_count, c);
  }
}

// det_ws (see kDetScale*) -> d_b_enc += s * sum, d_b_dec += s * sum, stats->sse += sum
__global__ void __launch_bounds__(256)
det_finish_kernel(const long long* __restrict__ det_ws, int F, int d, const float* __restrict__ grad_out,
                  float coef, float* __restrict__ d_b_enc, float* __restrict__ d_b_dec,
                  FusedStats* __restrict__ stats) {
  const double s = static_cast<double>(coef) * (grad_out != nullptr ? static_cast<double>(*grad_out) : 1.0);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < F) {
    if (d_b_enc != nullptr) d_b_enc[i] += static_cast<float>(s * (static_cast<double>(det_ws[i]) / kDetScaleEnc));
  } else if (i < F + d) {
    if (d_b_dec != nullptr)
      d_b_dec[i - F] += static_cast<float>(s * (static_cast<double>(det_ws[i]) / kDetScaleDec));
  } else if (i == F + d) {
    if (stats != nullptr) stats->sse += static_cast<double>(det_ws[i]) / kDetScaleSse;
  }
}

// experiments only (wsae_debug_decode_backward_general): 1 = always the general kernel (A/B runs)
static int g_decode_backward_general = 0;   // 0 = per-shape choice (see the launcher), 1 = general, 2 = mma, 3 = staged

}  // namespace wsae

using namespace wsae;

extern "C" int wsae_debug_decode_backward_general(int on) { g_decode_backward_general = on; return 0; }

// The wide form (32 < k <= 256, d % 128 == 0; det_ws non-null: its deterministic form).  Teams of
// ceil(k / 32) warps, two teams per block while they fit in 4 warps, else one.
template <typename TX>
static int decode_backward_wide(const TX* target, const TX* const* target_at,
                                const long long* const* rows_at, long long* det_ws, const __nv_bfloat16* w_decT,
                                const float* b_dec, const float* b_pre, const int32_t* idx,
                                const float* val, const float* grad_out, float coef, int B, int d,
                                int F, int k, float* resid, __nv_bfloat16* resid_bf16, FusedStats* stats,
                                long long* last_activated, const long long* step_count, float* d_b_enc,
                                float* d_b_dec, float* dpre_val, cudaStream_t stream) {
  int dev = 0, sms = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int tsize = ceil_div(k, 32);
  const int teams = tsize <= 2 ? 4 / tsize : 1;
  const int nwarps = teams * tsize;
  const int stamp_words = (last_activated != nullptr && F <= 65536) ? ceil_div(F, 32) : 0;
  const size_t smem = ((1 + teams) * static_cast<size_t>(d) + 2 * nwarps * 64) * sizeof(float) +
                      static_cast<size_t>(nwarps) * kTcGBytes + 16 + static_cast<size_t>(stamp_words) * 4;
  if (smem > 200 * 1024) return kUnsupported;
  const auto kern = det_ws != nullptr ? decode_backward_wide_kernel<true, TX> : decode_backward_wide_kernel<false, TX>;
  static bool attr_set[64] = {};
  if (dev >= 64 || !attr_set[dev]) {
    cudaError_t e = cudaSuccess;
    for (auto kf : {decode_backward_wide_kernel<false, TX>, decode_backward_wide_kernel<true, TX>})
      if (e == cudaSuccess) e = cudaFuncSetAttribute(kf, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e != cudaSuccess) return static_cast<int>(e);
    if (dev < 64) attr_set[dev] = true;
  }
  int per = 0;
  cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, kern, nwarps * 32, smem);
  if (e != cudaSuccess) return static_cast<int>(e);
  if (per < 1) per = 1;
  int nblk = ceil_div(B, teams);
  if (nblk > sms * per) nblk = sms * per;
  // L2 hints as in the tensor form: decoder rows evict_last while the bf16 decoder fits in 48 MB
  const int l2hint = static_cast<long long>(F) * d * 2 <= (48LL << 20) ? 3 : 1;
  launch_pdl(kern, nblk, nwarps * 32, smem, stream, target, w_decT, b_dec, b_pre, idx,
             val, grad_out, coef, B, d, F, k, resid, resid_bf16, stats, last_activated, step_count, d_b_enc,
             d_b_dec, dpre_val, target_at, rows_at, stamp_words, l2hint, det_ws);
  return static_cast<int>(cudaGetLastError());
}

// See include/wsae.h.  Returns WSAE_E_UNSUPPORTED for shapes the fused kernels do not cover
// (fp32 decoder, d % 8 != 0, k > 256, 32 < k with d % 128 != 0): callers then use K2 + K3.
// A deterministic workspace is accepted at every covered shape.  TX: element type of the target matrix.
template <typename TX>
static int decode_backward_launch(const TX* target, const TX* const* target_at,
                                  const long long* const* rows_at, long long* det_ws, const void* w_decT, int w_is_bf16, const float* b_dec,
                                  const float* b_pre, const int32_t* idx, const float* val,
                                  const float* grad_out, float coef, int B, int d, int F, int k,
                                  float* resid, void* resid_bf16, void* stats,
                                  long long* last_activated, const long long* step_count,
                                  float* d_b_enc, float* d_b_dec, float* dpre_val,
                                  cudaStream_t stream) {
  if ((!target && !target_at) || !w_decT || !b_dec || !idx || !val) return kBadArg;
  if (B <= 0 || d <= 0 || F <= 0 || k <= 0) return kBadArg;
  if (!w_is_bf16 || d % 8 != 0 || d > 8192) return kUnsupported;
  if (static_cast<long long>(F) * (d / 4) > 0x7fffffffLL) return kUnsupported;
  if (k > 32) {
    if (k > kWideMaxK || d % 128 != 0) return kUnsupported;
    return decode_backward_wide(target, target_at, rows_at, det_ws, static_cast<const __nv_bfloat16*>(w_decT), b_dec,
                                b_pre, idx, val, grad_out, coef, B, d, F, k, resid,
                                static_cast<__nv_bfloat16*>(resid_bf16), static_cast<FusedStats*>(stats),
                                last_activated, step_count, d_b_enc, d_b_dec, dpre_val, stream);
  }
  int dev = 0, sms = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const bool fast_shape = (d % 128 == 0) && ((g_decode_backward_general & 0xff) == 2 || ((g_decode_backward_general & 0xff) == 0 && d <= 1024));
  const int per_sm = fast_shape ? 3 : 4;
  int blocks = ceil_div(B, kFusedWarps);
  if (blocks > sms * per_sm) blocks = sms * per_sm;
  // fired bitmap in shared memory (F <= 65536: 8 KB), else stamps go straight to global memory
  const int stamp_words = (last_activated != nullptr && F <= 65536) ? ceil_div(F, 32) : 0;
  const size_t smem = ((1 + kFusedWarps) * static_cast<size_t>(round_up(d, 128)) + kFusedWarps * kDotScratch) *
                          sizeof(float) + static_cast<size_t>(stamp_words) * 4;
  if (smem > 48 * 1024) {      // d > 2432: opt in to the large dynamic shared-memory carve-out (once per device)
    static bool attr_set[64] = {};
    if (dev >= 64 || !attr_set[dev]) {
      cudaError_t e = cudaFuncSetAttribute(decode_backward_kernel<true, TX>,
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
      if (e == cudaSuccess)
        e = cudaFuncSetAttribute(decode_backward_kernel<false, TX>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
      if (e != cudaSuccess) return static_cast<int>(e);
      if (dev < 64) attr_set[dev] = true;
    }
  }
  const auto wd = static_cast<const __nv_bfloat16*>(w_decT);
  const auto rbf = static_cast<__nv_bfloat16*>(resid_bf16);
  const auto st = static_cast<FusedStats*>(stats);
  // staged kernel: full slices, ring depth 3 (2 when the shared memory of two resident blocks would
  // not fit), byte offsets of the gathered rows in 32 bits
  const int mode = g_decode_backward_general & 0xff;
  const int dbg = g_decode_backward_general >> 8;
  // Kernel choice (tools/bench_k23.py, same box, B = 75776 / 37888, k = 32):
  // every selected value positive, as K1 hands them over in training (profiles/r2_k23_variants.txt):
  //   d = 384:  staged 226 us | mma 256 us | general 259 us   -> staged where THREE blocks fit an SM
  //   d = 768:  staged 541 us | mma 451 us | general 461 us   -> mma (the ring leaves room for 8 warps only)
  //   d = 1280: staged 434 us | mma 451 us | general 444 us   -> general (F = 40960: decoder > L2 share)
  //   d % 128 != 0: general
  // tensor form (profiles/r2_k23_tensor_form.txt, same boxes): 384: 219-227 us (step 0.769 vs 0.776 ms with
  //   staged), 768: 393 us, 1280: 379 us with the L2 prefetch, 1536: 715 us  -> the choice for d % 128 == 0
  // mode (wsae_debug_decode_backward_general): 0 = this choice, 1 = general, 2 = mma, 3 = staged, 4 = tensor form
  // tensor form (mode 4): the choice for every d % 128 == 0 shape (WSAE_K23_TC=0: the older forms below)
  static const int want_tc = [] {
    const char* e = std::getenv("WSAE_K23_TC");
    return (e && e[0] == '0') ? 0 : 1;
  }();
  if ((mode == 4 || (mode == 0 && want_tc)) && d % 128 == 0) {
    const size_t smem_t = (1 + kFusedWarps) * static_cast<size_t>(d) * sizeof(float) +
                          static_cast<size_t>(kFusedWarps) * kTcGBytes + 16 +
                          static_cast<size_t>(stamp_words) * 4;
    // WSAE_K23_TC = "<blocks per SM: 3|4><stages: 2|3>", e.g. 32 (default 3 blocks; 3 stages where d / 64 % 3 == 0)
    static const int tc_cfg = [] {
      const char* e = std::getenv("WSAE_K23_TC_CFG");
      return (e && e[0] && e[1]) ? (e[0] - '0') * 10 + (e[1] - '0') : 0;
    }();
    int per_want = tc_cfg ? tc_cfg / 10 : 3;
    int stages = tc_cfg ? tc_cfg % 10 : 2;
    if ((d / 64) % 3 != 0) stages = 2;
    if (stages == 3) per_want = 3;
    // L2 prefetch distance (half slices): CCTL.PF1 does not fill L1 here, but it does pull decoder rows
    // that miss L2 in from HBM early - 452 -> 379 us at 1280 -> 40960 (105 MB decoder), +4 % where the
    // decoder is L2 resident (profiles/r2_k23_tensor_form.txt).  WSAE_K23_PF overrides.
    static const int pf_env = [] {
      const char* e = std::getenv("WSAE_K23_PF");
      return e ? std::atoi(e) : -1;
    }();
    const int pf_dist = pf_env >= 0 ? pf_env : (static_cast<long long>(F) * d * 2 > (64LL << 20) ? 1 : 0);
    // L2 eviction hints (WSAE_K23_L2HINT: bit 0 = activation stream evict_first, bit 1 = decoder rows
    // evict_last; default 3 where the bf16 decoder fits comfortably in L2, 1 above 48 MB)
    static const int l2_env = [] {
      const char* e = std::getenv("WSAE_K23_L2HINT");
      return e ? std::atoi(e) : -1;
    }();
    const int l2hint = l2_env >= 0 ? l2_env : (static_cast<long long>(F) * d * 2 <= (48LL << 20) ? 3 : 1);
    using KernT = decltype(&decode_backward_tc_kernel<3, 2, false, TX>);
    KernT kern = stages == 3 ? decode_backward_tc_kernel<3, 3, false, TX>
                             : (per_want == 4 ? (pf_dist > 0 ? decode_backward_tc_kernel<4, 2, true, TX> : decode_backward_tc_kernel<4, 2, false, TX>)
                                              : (pf_dist > 0 ? decode_backward_tc_kernel<3, 2, true, TX> : decode_backward_tc_kernel<3, 2, false, TX>));
    static bool attr_tc[64] = {};
    if (dev >= 64 || !attr_tc[dev]) {
      cudaError_t e = cudaSuccess;
      for (KernT kf : {decode_backward_tc_kernel<4, 2, false, TX>, decode_backward_tc_kernel<4, 2, true, TX>,
                       decode_backward_tc_kernel<3, 2, false, TX>, decode_backward_tc_kernel<3, 2, true, TX>,
                       decode_backward_tc_kernel<3, 3, false, TX>})
        if (e == cudaSuccess)
          e = cudaFuncSetAttribute(kf, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);
      if (e != cudaSuccess) return static_cast<int>(e);
      if (dev < 64) attr_tc[dev] = true;
    }
    if (smem_t <= 220 * 1024) {
      int per = static_cast<int>((227 * 1024) / (smem_t + 1024));
      if (per > per_want) per = per_want;
      if (per < 1) per = 1;
      int nblk = ceil_div(B, kFusedWarps);
      if (nblk > sms * per) nblk = sms * per;
      launch_pdl(kern, nblk, kFusedWarps * 32, smem_t, stream, target, wd, b_dec,
                 b_pre, idx, val, grad_out, coef, B, d, F, k, resid, rbf, st, last_activated, step_count,
                 d_b_enc, d_b_dec, dpre_val, target_at, rows_at, stamp_words, det_ws, pf_dist, l2hint);
      return static_cast<int>(cudaGetLastError());
    }
  }
  const bool staged_fits3 =
      3 * ((1 + kFusedWarps) * static_cast<size_t>(d) * sizeof(float) + kFusedWarps * 2 * kSliceBytes +
           static_cast<size_t>(stamp_words) * 4 + 1024) <= 227 * 1024;
  if (((mode == 0 && staged_fits3) || mode == 3) && d % 128 == 0 &&
      static_cast<long long>(F) * d * 2 <= 0xffffffffLL) {
    const size_t base = (1 + kFusedWarps) * static_cast<size_t>(d) * sizeof(float) + static_cast<size_t>(stamp_words) * 4;
    // ring depth 2 leaves room for three resident blocks (12 warps per SM) at d = 384: measured
    // faster than depth 3 with two blocks (tools/bench_k23.py); WSAE_K23_STAGES overrides
    static const int want_stages = [] {
      const char* e = std::getenv("WSAE_K23_STAGES");
      return (e && e[0] == '3') ? 3 : 2;
    }();
    int stages = want_stages;
    if (2 * (base + kFusedWarps * 3 * kSliceBytes + 1024) > 227 * 1024 || d < 256) stages = 2;
    const size_t smem_s = base + static_cast<size_t>(kFusedWarps) * stages * kSliceBytes;
    static bool attr_staged[64] = {};
    if (dev >= 64 || !attr_staged[dev]) {
      cudaError_t e = cudaFuncSetAttribute(decode_backward_staged_kernel<3, TX>,
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);
      if (e == cudaSuccess)
        e = cudaFuncSetAttribute(decode_backward_staged_kernel<2, TX>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);
      if (e != cudaSuccess) return static_cast<int>(e);
      if (dev < 64) attr_staged[dev] = true;
    }
    if (smem_s <= 220 * 1024) {
      int per = static_cast<int>((227 * 1024) / (smem_s + 1024));
      if (per > (stages == 2 ? 3 : 2)) per = stages == 2 ? 3 : 2;
      if (per < 1) per = 1;
      int nblk = ceil_div(B, kFusedWarps);
      if (nblk > sms * per) nblk = sms * per;
      if (stages == 3)
        launch_pdl(decode_backward_staged_kernel<3, TX>, nblk, kFusedWarps * 32, smem_s, stream, target, wd, b_dec,
                   b_pre, idx, val, grad_out, coef, B, d, F, k, resid, rbf, st, last_activated, step_count,
                   d_b_enc, d_b_dec, dpre_val, target_at, rows_at, stamp_words, det_ws, dbg);
      else
        launch_pdl(decode_backward_staged_kernel<2, TX>, nblk, kFusedWarps * 32, smem_s, stream, target, wd, b_dec,
                   b_pre, idx, val, grad_out, coef, B, d, F, k, resid, rbf, st, last_activated, step_count,
                   d_b_enc, d_b_dec, dpre_val, target_at, rows_at, stamp_words, det_ws, dbg);
      return static_cast<int>(cudaGetLastError());
    }
  }
  const bool fast = (d % 128 == 0) && (mode == 2 || (mode == 0 && d <= 1024));
  if (fast)
    launch_pdl(decode_backward_kernel<true, TX>, blocks, kFusedWarps * 32, smem, stream, target,
               static_cast<const __nv_bfloat16*>(w_decT), b_dec, b_pre, idx, val, grad_out, coef, B, d,
               F, k, resid, static_cast<__nv_bfloat16*>(resid_bf16), static_cast<FusedStats*>(stats),
               last_activated, step_count, d_b_enc, d_b_dec, dpre_val, target_at, rows_at, stamp_words, det_ws);
  else
    launch_pdl(decode_backward_kernel<false, TX>, blocks, kFusedWarps * 32, smem, stream, target,
               static_cast<const __nv_bfloat16*>(w_decT), b_dec, b_pre, idx, val, grad_out, coef, B, d,
               F, k, resid, static_cast<__nv_bfloat16*>(resid_bf16), static_cast<FusedStats*>(stats),
               last_activated, step_count, d_b_enc, d_b_dec, dpre_val, target_at, rows_at, stamp_words, det_ws);
  return static_cast<int>(cudaGetLastError());
}

// x_dtype (0 = fp32, 1 = bf16, 2 = fp16) names the element type of the target matrix.
static int decode_backward_impl(const void* target, const void* const* target_at, int x_dtype,
                                const long long* const* rows_at, long long* det_ws, const void* w_decT,
                                int w_is_bf16, const float* b_dec, const float* b_pre, const int32_t* idx,
                                const float* val, const float* grad_out, float coef, int B, int d, int F, int k,
                                float* resid, void* resid_bf16, void* stats, long long* last_activated,
                                const long long* step_count, float* d_b_enc, float* d_b_dec, float* dpre_val,
                                cudaStream_t stream) {
  return with_x_dtype(x_dtype, [&](auto tag) {
    using TX = std::remove_cv_t<std::remove_pointer_t<decltype(tag)>>;
    return decode_backward_launch<TX>(static_cast<const TX*>(target), reinterpret_cast<const TX* const*>(target_at),
                                      rows_at, det_ws, w_decT, w_is_bf16, b_dec, b_pre, idx, val, grad_out, coef,
                                      B, d, F, k, resid, resid_bf16, stats, last_activated, step_count, d_b_enc,
                                      d_b_dec, dpre_val, stream);
  });
}

extern "C" int wsae_decode_backward(const float* target, const void* w_decT, int w_is_bf16,
                                    const float* b_dec, const float* b_pre, const int32_t* idx,
                                    const float* val, const float* grad_out, float coef, int B,
                                    int d, int F, int k, float* resid, void* resid_bf16,
                                    void* stats, long long* last_activated,
                                    const long long* step_count, float* d_b_enc, float* d_b_dec,
                                    float* dpre_val, cudaStream_t stream) {
  if (!target) return kBadArg;
  return decode_backward_impl(target, nullptr, 0, nullptr, nullptr, w_decT, w_is_bf16, b_dec, b_pre, idx, val, grad_out,
                              coef, B, d, F, k, resid, resid_bf16, stats, last_activated, step_count,
                              d_b_enc, d_b_dec, dpre_val, stream);
}

// Same, with the target matrix named by a device-resident pointer slot (*target_at: 16-byte aligned,
// B x d fp32, read when the kernel runs) - lets a captured graph train on batches in place.
extern "C" int wsae_decode_backward_at(const float* const* target_at, const void* w_decT,
                                       int w_is_bf16, const float* b_dec, const float* b_pre,
                                       const int32_t* idx, const float* val, const float* grad_out,
                                       float coef, int B, int d, int F, int k, float* resid,
                                       void* resid_bf16, void* stats, long long* last_activated,
                                       const long long* step_count, float* d_b_enc, float* d_b_dec,
                                       float* dpre_val, cudaStream_t stream) {
  if (!target_at) return kBadArg;
  return decode_backward_impl(nullptr, reinterpret_cast<const void* const*>(target_at), 0, nullptr, nullptr, w_decT, w_is_bf16, b_dec, b_pre, idx, val,
                              grad_out, coef, B, d, F, k, resid, resid_bf16, stats, last_activated,
                              step_count, d_b_enc, d_b_dec, dpre_val, stream);
}

// Slot form with a row-index indirection: target row of batch row r = (*target_at)[(*rows_at)[r], :]
// (*rows_at == 0: identity).  See wsae_pack_activations_rows_at.
extern "C" int wsae_decode_backward_rows_at(const float* const* target_at,
                                            const long long* const* rows_at, const void* w_decT,
                                            int w_is_bf16, const float* b_dec, const float* b_pre,
                                            const int32_t* idx, const float* val,
                                            const float* grad_out, float coef, int B, int d, int F,
                                            int k, float* resid, void* resid_bf16, void* stats,
                                            long long* last_activated, const long long* step_count,
                                            float* d_b_enc, float* d_b_dec, float* dpre_val,
                                            cudaStream_t stream) {
  if (!target_at || !rows_at) return kBadArg;
  return decode_backward_impl(nullptr, reinterpret_cast<const void* const*>(target_at), 0, rows_at, nullptr, w_decT, w_is_bf16, b_dec, b_pre, idx, val,
                              grad_out, coef, B, d, F, k, resid, resid_bf16, stats, last_activated,
                              step_count, d_b_enc, d_b_dec, dpre_val, stream);
}

// Deterministic form (see kDetScale* above): the slot form of wsae_decode_backward_rows_at
// (target_at / rows_at as there; target may be given directly instead of target_at) with the three
// cross-row float sums accumulated order-independently in det_ws (int64 [F + d + 1], caller-zeroed);
// d_b_enc / d_b_dec / stats->sse are NOT touched here - wsae_det_finish adds the converted sums.
extern "C" int wsae_decode_backward_det(const float* target, const float* const* target_at,
                                        const long long* const* rows_at, const void* w_decT,
                                        int w_is_bf16, const float* b_dec, const float* b_pre,
                                        const int32_t* idx, const float* val, const float* grad_out,
                                        float coef, int B, int d, int F, int k, float* resid,
                                        void* resid_bf16, void* stats, long long* last_activated,
                                        const long long* step_count, float* d_b_enc, float* d_b_dec,
                                        float* dpre_val, long long* det_ws, cudaStream_t stream) {
  if ((!target && !target_at) || !det_ws) return kBadArg;
  return decode_backward_impl(target, reinterpret_cast<const void* const*>(target_at), 0, rows_at, det_ws, w_decT, w_is_bf16, b_dec, b_pre, idx,
                              val, grad_out, coef, B, d, F, k, resid, resid_bf16, stats, last_activated,
                              step_count, d_b_enc, d_b_dec, dpre_val, stream);
}

// Slot form for any target element type (x_dtype 0 = fp32, 1 = bf16, 2 = fp16; *target_at then points
// at that type): rows_at nullable, det_ws nullable (non-NULL: the deterministic form above).
extern "C" int wsae_decode_backward_typed(const void* const* target_at, const long long* const* rows_at,
                                          int x_dtype, const void* w_decT, int w_is_bf16, const float* b_dec,
                                          const float* b_pre, const int32_t* idx, const float* val,
                                          const float* grad_out, float coef, int B, int d, int F, int k,
                                          float* resid, void* resid_bf16, void* stats, long long* last_activated,
                                          const long long* step_count, float* d_b_enc, float* d_b_dec,
                                          float* dpre_val, long long* det_ws, cudaStream_t stream) {
  if (!target_at) return kBadArg;
  return decode_backward_impl(nullptr, target_at, x_dtype, rows_at, det_ws, w_decT, w_is_bf16, b_dec, b_pre, idx,
                              val, grad_out, coef, B, d, F, k, resid, resid_bf16, stats, last_activated,
                              step_count, d_b_enc, d_b_dec, dpre_val, stream);
}

extern "C" int wsae_det_finish(const long long* det_ws, int F, int d, const float* grad_out, float coef,
                               float* d_b_enc, float* d_b_dec, void* stats, cudaStream_t stream) {
  if (!det_ws || F <= 0 || d <= 0) return kBadArg;
  const int n = F + d + 1;
  det_finish_kernel<<<ceil_div(n, 256), 256, 0, stream>>>(det_ws, F, d, grad_out, coef, d_b_enc, d_b_dec,
                                                          static_cast<FusedStats*>(stats));
  return static_cast<int>(cudaGetLastError());
}
