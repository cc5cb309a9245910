// wsae_row_step.cu - the SMALL-BATCH form of K1's selection + K23 + K4: one thread block per
// activation row does, for that row,
//   :114      TopK over the row's dense pre-activations (left in an L2-sized scratch by encode_dense_kernel)
//   :115-116  relu of the k selected values
//   :129      recon = sum_j h_j * W_dec[:, i_j] + b_dec + b_pre
//   :145,148  squared error and L0 count
//   :174-181  fired stamps
//   autograd  dv_j = coef * g . W_dec[:, i_j] * [v_j > 0], db_enc, db_dec, and BOTH weight-gradient
//             rows  dW_dec[i_j, :] += coef * g * h_j * resid,  dW_enc[i_j, :] += dv_j * (x - b_pre)
// (line numbers: /root/reference/src/whisper_sae/sae/model.py).
//
// Why: the shipped configs/tiny_default.yaml trains on 128-row batches.  There the large-batch chain
// rowwise top-k -> K23 -> bucket_by_tile -> two K4 GEMMs is five dependent launches of 8-20 us that each
// leave most of the GPU idle (K23 at 128 rows = 32 blocks of 4 warps; a K4 GEMM = 24 feature tiles x 2
// row chunks).  With one 256-thread block per row the whole chain is ONE launch of B blocks: the k
// decoder rows are read twice from L1/L2 (1.5 MB of traffic per launch at 128 rows), and the 2 k
// weight-gradient rows go out as red.global.add.v2.f32 (2 * k * d / 2 vector reductions per row - at
// 128 rows 1.6 M of them, which L2 absorbs in a few microseconds; at 75 776 rows the same sum is a
// tcgen05 GEMM, wsae_wgrad_gemm.cu).  Products follow K23: bf16 activation x bf16 decoder row with fp32
// accumulation, bf16 residual in the dv dot products; the weight-gradient rows are fp32 x fp32 (more
// exact than K4's bf16 operands).  Sums arrive in atomic order (no deterministic form: the trainer's
// deterministic mode keeps the large-batch chain).
#include "wsae_common.cuh"
#include "wsae_rowselect.cuh"

namespace wsae {

constexpr int kRowStepMaxK = 32;

__device__ __forceinline__ void red_add_v2(float* addr, float a, float b) {
  asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(addr), "f"(a), "f"(b) : "memory");
}

__device__ __forceinline__ float bf16_round(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }

// TX: element type of the activation matrix (float / __nv_bfloat16 / __half, converted at the load).
template <typename TX>
__global__ void __launch_bounds__(kRowTopkThreads)
row_step_kernel(const float* __restrict__ pre, const TX* __restrict__ target,
                const TX* const* __restrict__ target_at, const long long* const* __restrict__ rows_at,
                const __nv_bfloat16* __restrict__ w_decT, const float* __restrict__ b_dec,
                const float* __restrict__ b_pre, const float* __restrict__ grad_out, float coef, int B, int d,
                int F, int k, float* __restrict__ out_val, int32_t* __restrict__ out_idx,
                double* __restrict__ stats_sse, unsigned long long* __restrict__ stats_l0,
                long long* __restrict__ last_activated, long long* step_count,
                float* __restrict__ d_b_enc, float* __restrict__ d_b_dec, float* __restrict__ d_w_enc,
                float* __restrict__ d_w_decT, float* __restrict__ resid_out, float* __restrict__ dpre_val,
                const float* __restrict__ w_enc, float* __restrict__ d_b_pre, unsigned int* ticket,
                long long dead_threshold, long long* dead_count, const long long* seq_src,
                long long* mailbox) {
  extern __shared__ __align__(16) uint32_t s_dyn[];          // [F] keys | [d] residual | [d] x - b_pre
  __shared__ RowSelectSmem sel;
  __shared__ float s_val[kRowStepMaxK];                      // selected pre-activations, ascending feature index
  __shared__ int32_t s_idx[kRowStepMaxK];
  __shared__ float s_dv[kRowStepMaxK];
  __shared__ float s_h[kRowStepMaxK];                        // bf16(relu(v)), 0 where the entry did not fire
  __shared__ int32_t s_row[kRowStepMaxK];                    // decoder row to gather (0 where it did not fire)
  __shared__ float s_sse[kRowTopkThreads / 32];
  pdl_prologue();
  const int row = blockIdx.x;
  if (row >= B) return;
  const int tid = threadIdx.x;
  const int lane = tid & 31, warp = tid >> 5;
  uint32_t* s_key = s_dyn;
  float* s_res = reinterpret_cast<float*>(s_dyn + F);
  float* s_xc = s_res + d;

  // ---- TopK of the row (writes the global (idx, val) lists; a copy stays in shared memory) ----
  float* gv = out_val + static_cast<size_t>(row) * k;
  int32_t* gi = out_idx + static_cast<size_t>(row) * k;
  block_row_topk(pre + static_cast<size_t>(row) * F, F, k, s_key, sel, gv, gi);
  if (tid < kRowStepMaxK) {  // block_row_topk ended with a barrier: the global lists are visible to the block
    const float v = tid < k ? gv[tid] : 0.f;
    const int32_t f = tid < k ? gi[tid] : -1;
    const bool fired = v > 0.f && f >= 0 && f < F;
    s_val[tid] = v;
    s_idx[tid] = f;
    s_h[tid] = fired ? bf16_round(v) : 0.f;
    s_row[tid] = fired ? f : 0;
    s_dv[tid] = 0.f;
  }
  __syncthreads();

  if (target_at != nullptr) target = *target_at;
  const long long* perm = rows_at != nullptr ? *rows_at : nullptr;
  const size_t srow = perm != nullptr ? static_cast<size_t>(perm[row]) : static_cast<size_t>(row);
  const TX* trow = target + srow * d;
  const float s = coef * (grad_out != nullptr ? *grad_out : 1.f);
  const long long stamp = (last_activated != nullptr && step_count != nullptr) ? (*step_count + 1) : 0;
  const uint32_t* wrows = reinterpret_cast<const uint32_t*>(w_decT);     // bf16 pairs
  const int dh = d >> 1;

  // fired entries (relu); stamps, L0
  const bool my_fired = tid < k && s_idx[tid] >= 0 && s_idx[tid] < F && s_val[tid] > 0.f;
  if (my_fired && last_activated != nullptr) last_activated[s_idx[tid]] = stamp;
  if (warp == 0) {
    const uint32_t m = __ballot_sync(0xffffffffu, my_fired);
    if (lane == 0 && stats_l0 != nullptr) atomicAdd(stats_l0, static_cast<unsigned long long>(__popc(m)));
  }

  // ---- decode + residual: thread t owns column pairs t, t + 256, ... ----
  float sse_local = 0.f;
  for (int p = tid; p < dh; p += kRowTopkThreads) {
    const int c = 2 * p;
    const float bp0 = b_pre != nullptr ? b_pre[c] : 0.f, bp1 = b_pre != nullptr ? b_pre[c + 1] : 0.f;
    float a0 = b_dec[c] + bp0, a1 = b_dec[c + 1] + bp1;
    // all k loads in flight at once: entries that did not fire read row 0 with weight 0
    uint32_t w[kRowStepMaxK];
#pragma unroll
    for (int j = 0; j < kRowStepMaxK; ++j) w[j] = __ldg(wrows + static_cast<size_t>(s_row[j]) * dh + p);
#pragma unroll
    for (int j = 0; j < kRowStepMaxK; ++j) {
      const float h = s_h[j];                                // bf16(relu(v)); 0 for padding / unfired entries
      a0 = fmaf(h, __uint_as_float(w[j] << 16), a0);
      a1 = fmaf(h, __uint_as_float(w[j] & 0xffff0000u), a1);
    }
    const float2 t = ld_x2(trow + c);
    const float r0 = a0 - t.x, r1 = a1 - t.y;
    s_res[c] = r0;
    s_res[c + 1] = r1;
    s_xc[c] = t.x - bp0;
    s_xc[c + 1] = t.y - bp1;
    sse_local = fmaf(r0, r0, sse_local);
    sse_local = fmaf(r1, r1, sse_local);
    if (resid_out != nullptr) *reinterpret_cast<float2*>(resid_out + static_cast<size_t>(row) * d + c) = make_float2(r0, r1);
    if (d_b_dec != nullptr) {
      atomicAdd(d_b_dec + c, s * r0);
      atomicAdd(d_b_dec + c + 1, s * r1);
    }
  }
  sse_local = warp_sum(sse_local);
  if (lane == 0) s_sse[warp] = sse_local;
  __syncthreads();
  if (tid == 0 && stats_sse != nullptr) {
    double tot = 0.0;
    for (int w = 0; w < kRowTopkThreads / 32; ++w) tot += static_cast<double>(s_sse[w]);
    atomicAdd(stats_sse, tot);
  }

  // ---- dv_j = s * bf16(resid) . W_dec[i_j]: warp w takes entries w, w + 8, w + 16, w + 24 TOGETHER, so the
  //      loads of all four rows are in flight at once (unfired entries read row 0 and are masked) ----
  {
    constexpr int kPerWarp = kRowStepMaxK / (kRowTopkThreads / 32);      // 4
    float dot[kPerWarp];
    const uint32_t* wr[kPerWarp];
#pragma unroll
    for (int e = 0; e < kPerWarp; ++e) {
      dot[e] = 0.f;
      wr[e] = wrows + static_cast<size_t>(s_row[warp + e * (kRowTopkThreads / 32)]) * dh;
    }
    for (int p = lane; p < dh; p += 32) {
      const float2 r = *reinterpret_cast<const float2*>(s_res + 2 * p);
      const float r0 = bf16_round(r.x), r1 = bf16_round(r.y);
      uint32_t w[kPerWarp];
#pragma unroll
      for (int e = 0; e < kPerWarp; ++e) w[e] = __ldg(wr[e] + p);
#pragma unroll
      for (int e = 0; e < kPerWarp; ++e)
        dot[e] = fmaf(r0, __uint_as_float(w[e] << 16), fmaf(r1, __uint_as_float(w[e] & 0xffff0000u), dot[e]));
    }
#pragma unroll
    for (int e = 0; e < kPerWarp; ++e) {
      const int j = warp + e * (kRowTopkThreads / 32);
      const float tot = warp_sum(dot[e]);
      if (lane == 0 && j < k) {
        const bool fired = s_h[j] != 0.f || (s_val[j] > 0.f && s_idx[j] >= 0 && s_idx[j] < F);
        const float dv = fired ? s * tot : 0.f;
        s_dv[j] = dv;
        if (dpre_val != nullptr) dpre_val[static_cast<size_t>(row) * k + j] = dv;
        if (fired && d_b_enc != nullptr) atomicAdd(d_b_enc + s_idx[j], dv);
      }
    }
  }
  __syncthreads();

  // ---- weight-gradient rows: (entry, column pair) space spread over the whole block ----
  const int total = k * dh;
  for (int q = tid; q < total; q += kRowTopkThreads) {
    const int j = q / dh;
    const int p = q - j * dh;
    const float v = s_val[j];
    const int32_t f = s_idx[j];
    if (!(v > 0.f) || f < 0 || f >= F) continue;
    const size_t off = static_cast<size_t>(f) * d + 2 * p;
    if (d_w_decT != nullptr) {
      const float sh = s * v;
      red_add_v2(d_w_decT + off, sh * s_res[2 * p], sh * s_res[2 * p + 1]);
    }
    if (d_w_enc != nullptr) {
      const float dv = s_dv[j];
      red_add_v2(d_w_enc + off, dv * s_xc[2 * p], dv * s_xc[2 * p + 1]);
    }
  }

  // ---- b_pre gradient of this row: s * resid - sum_j dv_j * W_enc[i_j, :]  (db_dec - db_enc . W_enc summed
  //      over the rows: the separate GEMV kernel is a 20 us launch of its own at these sizes) ----
  if (d_b_pre != nullptr && w_enc != nullptr) {
    for (int p = tid; p < dh; p += kRowTopkThreads) {
      const int c = 2 * p;
      float2 we[kRowStepMaxK];
#pragma unroll
      for (int j = 0; j < kRowStepMaxK; ++j)
        we[j] = __ldg(reinterpret_cast<const float2*>(w_enc + static_cast<size_t>(s_row[j]) * d + c));
      float g0 = s * s_res[c], g1 = s * s_res[c + 1];
#pragma unroll
      for (int j = 0; j < kRowStepMaxK; ++j) {
        const float dv = s_dv[j];                            // 0 for entries that did not fire
        g0 = fmaf(-dv, we[j].x, g0);
        g1 = fmaf(-dv, we[j].y, g1);
      }
      atomicAdd(d_b_pre + c, g0);
      atomicAdd(d_b_pre + c + 1, g1);
    }
  }

  // ---- the step's counters and metrics, by the LAST block to finish (ticket != NULL): what
  //      counters_update_kernel does in a launch of its own - bump step_count (model.py:174), count the dead
  //      features against the new step (model.py:183-195), post {sse, l0, dead, seq} to the host mailbox ----
  if (ticket != nullptr) {
    __shared__ int s_last;
    __shared__ int s_part[kRowTopkThreads / 32];
    __syncthreads();
    if (tid == 0) {
      __threadfence();                                       // this block's stamps / sums before its ticket
      s_last = atomicAdd(ticket, 1u) == gridDim.x - 1 ? 1 : 0;
    }
    __syncthreads();
    if (s_last) {
      __threadfence();
      const long long sc = *step_count + 1;                  // every block read the old value long ago
      int c = 0;
      for (int f = tid; f < F; f += kRowTopkThreads) c += ((sc - __ldcg(last_activated + f)) > dead_threshold) ? 1 : 0;
      c = static_cast<int>(warp_sum(static_cast<float>(c)));  // <= F / 8 per warp: exact in fp32
      if (lane == 0) s_part[warp] = c;
      __syncthreads();
      if (tid == 0) {
        long long t = 0;
        for (int w = 0; w < kRowTopkThreads / 32; ++w) t += s_part[w];
        *step_count = sc;
        if (dead_count != nullptr) *dead_count = t;
        if (mailbox != nullptr) {
          volatile long long* mb = mailbox;
          mb[0] = stats_sse != nullptr ? __ldcg(reinterpret_cast<const long long*>(stats_sse)) : 0;
          mb[1] = stats_l0 != nullptr ? static_cast<long long>(__ldcg(stats_l0)) : 0;
          mb[2] = t;
          __threadfence_system();
          mb[3] = *seq_src;
        }
      }
    }
  }
}

}  // namespace wsae

using namespace wsae;

// See include/wsae.h.  stats = { double sse; uint64 l0_count } (caller-zeroed, as for wsae_decode_mse).
// x_dtype (0 = fp32, 1 = bf16, 2 = fp16): element type of target / *target_at.
extern "C" int wsae_row_step_typed(const float* pre, const void* target, const void* const* target_at,
                                   const long long* const* rows_at, int x_dtype, const void* w_decT_bf16,
                                   const float* b_dec, const float* b_pre, const float* grad_out, float coef, int B,
                                   int d, int F, int k, float* out_val, int32_t* out_idx, void* stats,
                                   long long* last_activated, long long* step_count, float* d_b_enc, float* d_b_dec,
                                   float* d_w_enc, float* d_w_decT, float* resid, float* dpre_val, const float* w_enc,
                                   float* d_b_pre, unsigned int* ticket, long long dead_threshold,
                                   long long* dead_count, const long long* seq, long long* mailbox,
                                   cudaStream_t stream) {
  if (!pre || (!target && !target_at) || !w_decT_bf16 || !b_dec || !out_val || !out_idx) return kBadArg;
  if (B <= 0 || d <= 0 || F <= 0 || k <= 0 || k > F) return kBadArg;
  if (k > kRowStepMaxK || d % 2 != 0) return kUnsupported;
  if (ticket != nullptr && (!step_count || !last_activated || (mailbox != nullptr && !seq))) return kBadArg;
  const size_t smem = (static_cast<size_t>(F) + 2 * static_cast<size_t>(d)) * 4;
  if (smem > 200 * 1024) return kUnsupported;
  return with_x_dtype(x_dtype, [&](auto tag) {
    using TX = std::remove_cv_t<std::remove_pointer_t<decltype(tag)>>;
    int dev = 0;
    cudaGetDevice(&dev);
    static bool attr_set[64] = {};
    if (dev >= 64 || !attr_set[dev]) {
      cudaError_t e = cudaFuncSetAttribute(row_step_kernel<TX>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
      if (e != cudaSuccess) return static_cast<int>(e);
      if (dev < 64) attr_set[dev] = true;
    }
    double* sse = stats ? static_cast<double*>(stats) : nullptr;
    unsigned long long* l0 = stats ? reinterpret_cast<unsigned long long*>(static_cast<char*>(stats) + 8) : nullptr;
    cudaError_t e = launch_pdl(row_step_kernel<TX>, B, kRowTopkThreads, smem, stream, pre,
                               static_cast<const TX*>(target), reinterpret_cast<const TX* const*>(target_at), rows_at,
                               static_cast<const __nv_bfloat16*>(w_decT_bf16), b_dec, b_pre, grad_out, coef, B, d, F,
                               k, out_val, out_idx, sse, l0, last_activated, step_count, d_b_enc, d_b_dec, d_w_enc,
                               d_w_decT, resid, dpre_val, w_enc, d_b_pre, ticket, dead_threshold, dead_count, seq,
                               mailbox);
    return static_cast<int>(e != cudaSuccess ? e : cudaGetLastError());
  });
}

extern "C" int wsae_row_step(const float* pre, const float* target, const float* const* target_at,
                             const long long* const* rows_at, const void* w_decT_bf16, const float* b_dec,
                             const float* b_pre, const float* grad_out, float coef, int B, int d, int F, int k,
                             float* out_val, int32_t* out_idx, void* stats, long long* last_activated,
                             long long* step_count, float* d_b_enc, float* d_b_dec, float* d_w_enc,
                             float* d_w_decT, float* resid, float* dpre_val, const float* w_enc, float* d_b_pre,
                             unsigned int* ticket, long long dead_threshold, long long* dead_count,
                             const long long* seq, long long* mailbox, cudaStream_t stream) {
  return wsae_row_step_typed(pre, target, reinterpret_cast<const void* const*>(target_at), rows_at, 0, w_decT_bf16,
                             b_dec, b_pre, grad_out, coef, B, d, F, k, out_val, out_idx, stats, last_activated,
                             step_count, d_b_enc, d_b_dec, d_w_enc, d_w_decT, resid, dpre_val, w_enc, d_b_pre, ticket,
                             dead_threshold, dead_count, seq, mailbox, stream);
}
