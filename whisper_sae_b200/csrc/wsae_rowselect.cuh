// wsae_rowselect.cuh - one thread block selects the k largest of one row of F floats (exact; ties at
// the k-th value keep the lowest feature index; NaN is never selected): the row-wise TopK of
// torch.topk(pre, k, dim=-1) (/root/reference/src/whisper_sae/sae/model.py:114) for the small-batch
// form of K1, shared by rowwise_topk_kernel (wsae_encode_topk.cu) and row_step_kernel (wsae_row_step.cu).
#pragma once
#include "wsae_common.cuh"

namespace wsae {

constexpr int kRowTopkThreads = 256;

struct RowSelectSmem {
  uint32_t hist[256];
  uint32_t pick[2];                            // chosen digit, count above it
  uint32_t scan[kRowTopkThreads / 32];
};

// Keys (order-preserving integer image of the floats; NaN -> 0 = never selected) live in shared memory
// (s_key[F]).  Four passes of an 8-bit most-significant-digit radix select find the key T of the k-th
// largest value and how many keys lie above it; then every thread walks a CONTIGUOUS chunk of
// features, a block scan turns the per-thread counts into output slots, and ties at T are admitted in
// ascending feature index.  Output: k (value, f_base + index) pairs in ascending feature index through
// the generic pointers ov / oi (global or shared); fewer than k valid candidates: padded with (-inf, -1).
// Every thread of the kRowTopkThreads-wide block must call it; it ends with a __syncthreads().
__device__ __forceinline__ void block_row_topk(const float* __restrict__ src, int F, int k, uint32_t* s_key,
                                               RowSelectSmem& sm, float* ov, int32_t* oi,
                                               int f_base = 0) {
  uint32_t* s_hist = sm.hist;
  uint32_t* s_pick = sm.pick;
  uint32_t* s_scan = sm.scan;
  const int tid = threadIdx.x;
  const int lane = tid & 31, warp = tid >> 5;
  for (int f = tid; f < F; f += kRowTopkThreads) {
    const float v = src[f];
    s_key[f] = (v == v) ? f2key(v) : 0u;
  }
  uint32_t prefix = 0, prefix_mask = 0;       // bits decided so far
  uint32_t need = static_cast<uint32_t>(k);   // rank still wanted inside the prefix bucket
  uint32_t above = 0;                         // keys strictly above the prefix bucket
  for (int shift = 24; shift >= 0; shift -= 8) {
    s_hist[tid] = 0u;
    __syncthreads();
    for (int f = tid; f < F; f += kRowTopkThreads) {
      const uint32_t kk = s_key[f];
      if ((kk & prefix_mask) == prefix && kk != 0u) atomicAdd(&s_hist[(kk >> shift) & 255u], 1u);
    }
    __syncthreads();
    if (warp == 0) {
      // lane l owns digits 8 l .. 8 l + 7; suffix sums from the top digit down
      uint32_t loc[8], tot = 0;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        loc[i] = s_hist[8 * lane + i];
        tot += loc[i];
      }
      uint32_t suf = tot;                      // inclusive suffix sum over lanes >= l
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_down_sync(0xffffffffu, suf, o);
        if (lane + o < 32) suf += t;
      }
      const uint32_t higher = suf - tot;       // keys in digits above this lane's 8
      const bool here = higher < need && suf >= need;
      if (here) {
        uint32_t acc = higher;                 // keys above digit i inside the prefix bucket
        int dsel = 0;
        bool found = false;
#pragma unroll
        for (int i = 7; i >= 0; --i) {
          if (!found) {
            if (acc + loc[i] >= need) {
              dsel = i;
              found = true;
            } else {
              acc += loc[i];
            }
          }
        }
        s_pick[0] = static_cast<uint32_t>(8 * lane + dsel);
        s_pick[1] = acc;
      }
      if (lane == 0 && suf < need) {           // fewer than `need` valid keys: keep them all
        s_pick[0] = 0xFFFFFFFFu;
        s_pick[1] = 0u;
      }
    }
    __syncthreads();
    const uint32_t dsel = s_pick[0];
    if (dsel == 0xFFFFFFFFu) {                 // (only possible in the first pass: NaN rows, k > valid keys)
      prefix = 0u;
      prefix_mask = 0u;
      need = 0u;
      break;
    }
    above += s_pick[1];
    need -= s_pick[1];
    prefix |= dsel << shift;
    prefix_mask |= 255u << shift;
    __syncthreads();
  }
  // prefix = key T of the k-th largest value (or 0: keep every valid key); `above` keys exceed it
  const uint32_t T = prefix_mask ? prefix : 0u;
  const uint32_t ties_wanted = prefix_mask ? static_cast<uint32_t>(k) - above : 0u;
  // contiguous chunks: thread t owns features [t * per, (t + 1) * per)
  const int per = ceil_div(F, kRowTopkThreads);
  const int f_lo = tid * per, f_hi = min(F, f_lo + per);
  uint32_t n_gt = 0, n_tie = 0;
  for (int f = f_lo; f < f_hi; ++f) {
    const uint32_t kk = s_key[f];
    n_gt += (kk > T) ? 1u : 0u;
    n_tie += (prefix_mask && kk == T) ? 1u : 0u;
  }
  // block exclusive scan of (n_gt | n_tie << 16)
  uint32_t packed = n_gt | (n_tie << 16);
  uint32_t incl = packed;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) s_scan[warp] = incl;
  __syncthreads();
  uint32_t woff = 0;
  for (int w = 0; w < warp; ++w) woff += s_scan[w];
  const uint32_t excl = incl - packed + woff;
  uint32_t gt_before = excl & 0xFFFFu, tie_before = excl >> 16;
  for (int f = f_lo; f < f_hi; ++f) {
    const uint32_t kk = s_key[f];
    const bool gt = kk > T;
    const bool tie = prefix_mask && kk == T;
    bool keep = gt;
    if (tie) {
      keep = tie_before < ties_wanted;
      ++tie_before;
    }
    if (keep && kk != 0u) {
      // slot = kept entries before f: all greater ones + the admitted ties
      const uint32_t ties_kept_before = min(tie_before - (tie ? 1u : 0u), ties_wanted);
      const uint32_t slot = gt_before + ties_kept_before;
      if (slot < static_cast<uint32_t>(k)) {
        ov[slot] = src[f];
        oi[slot] = f_base + f;
      }
    }
    gt_before += gt ? 1u : 0u;
  }
  // fewer than k valid candidates (NaN rows): pad with (-inf, -1) like the fused epilogue
  if (!prefix_mask) {
    uint32_t total_valid = 0;
    for (int w = 0; w < kRowTopkThreads / 32; ++w) total_valid += s_scan[w] & 0xFFFFu;
    for (int sidx = static_cast<int>(total_valid) + tid; sidx < k; sidx += kRowTopkThreads) {
      ov[sidx] = __uint_as_float(0xff800000u);
      oi[sidx] = -1;
    }
  }
  __syncthreads();
}

}  // namespace wsae
