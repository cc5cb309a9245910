// wsae_encode_topk.cu — K1: dense encoder GEMM on tcgen05/TMEM with the per-row TopK fused
// into the epilogue, so the [B, F] pre-activation tensor never reaches HBM.
//
// Replaces (reference, /root/reference/src/whisper_sae/sae/model.py):
//   :108  x_centered = x - b_pre            (done by the pack kernel, wsae_pack.cu)
//   :111  pre = encoder(x_centered)         (this GEMM; the bias rides in 16 extra K columns)
//   :114  torch.topk(pre, k, dim=-1)        (epilogue below; values kept in fp32)
//
// Operands are *packed* bf16 matrices produced by wsae_pack.cu:
//   A' [Bp, Kp]  rows = activations, K-major, Kp = T*dp + 16 (+ zero pad to a multiple of 64)
//   W' [Fp, Kp]  rows = features,    K-major
// T = 1 is plain bf16; T = 3 / 6 concatenates split-bf16 pieces along K so the same kernel
// produces fp32-grade results (the "fp32 verification mode").
//
// Kernel shape: one CTA per SM, persistent over (row-block, F-split) work items.
//   warp 0      TMA producer   (A' 128x64 + W' 256x64 bf16 tiles, SWIZZLE_128B, 3-stage ring)
//   warp 1      MMA issuer     (tcgen05.mma 128x256x16, fp32 accumulators double-buffered in TMEM)
//   warp 2      TMEM allocator
//   warps 4..7  epilogue       (tcgen05.ld 32x32b: one thread owns one activation row)
//
// Epilogue TopK: each thread streams its row's accumulator columns, appends values above a
// running threshold tau to a thread-private candidate list in shared memory and, whenever a
// list in the warp is nearly full, raises tau by a bisection select over the list (in
// registers).  The final select per work item is exact (ties broken towards the lower index).
#include <cuda.h>
#include <cudaTypedefs.h>

#include <mutex>
#include <unordered_map>

#include "wsae_common.cuh"
#include "wsae_rowselect.cuh"

namespace wsae {

constexpr int kBM = 128;   // rows per CTA tile  (= TMEM lanes)
constexpr int kBN = 256;   // features per MMA tile (= TMEM columns per accumulator stage)
constexpr int kBK = 64;    // bf16 K elements per pipeline stage (= one 128-byte swizzle row)
constexpr int kAStage = kBM * kBK * 2;
constexpr int kBStage = kBN * kBK * 2;
constexpr int kChunk = 16;  // accumulator columns per tcgen05.ld
constexpr int kSlack = 8;   // intermediate selects may keep up to k + kSlack candidates
constexpr int kCheck = 8;   // list-overflow check every kCheck appended-or-not values

template <int CAP, int STAGES>
struct EncodeSmem {
  static constexpr int kPipeBytes = STAGES * (kAStage + kBStage);
  static constexpr int kCandBytes = CAP * kBM * 8;
  static constexpr int kBarBytes = 256;
  static constexpr int kTotal = kPipeBytes + kCandBytes + kBarBytes + 1024;  // +1024 align slack
};

// Thread-private candidate list: slot s of row r lives at base[s * 128 + r] (values), with the
// feature indices CAP * 512 bytes further on.  `wbase` is the shared-space byte address of the
// thread's slot 0, `waddr` the cursor (address of the first free slot).
//
// topk_compact raises tau so that at most k + slack candidates (exactly k when slack == 0) survive
// and compacts the list in place, preserving order (ascending feature index).  Warp-synchronous:
// every lane of the warp must call it.
//
// The candidate values are pulled into registers once.  The k-th largest is bracketed by a
// bisection over the order-preserving integer image of the floats (it terminates on ties and
// needs no assumption about the value distribution); every comparison is done in float space with
// four independent counters (FSET + FADD per element).  The survivors are then re-appended with
// the same branch-free predicated stores as the scan.  -0.0 == +0.0 throughout (float compares).
__device__ __forceinline__ float lds_f32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
  return v;
}

template <int CAP, bool TIES>
__device__ __forceinline__ uint32_t compact_move(const float (&v)[CAP], uint32_t wbase, float thrf,
                                                 int tie_left) {
  uint32_t w = wbase;
#pragma unroll
  for (int s = 0; s < CAP; s += 4) {
    uint32_t wn;
    if (!TIES) {
      asm volatile(
          "{\n\t"
          ".reg .pred p0, p1, p2, p3;\n\t"
          ".reg .u32 a1, a2, a3, t0, t1, t2, t3, i0, i1, i2, i3;\n\t"
          "setp.gt.f32 p0, %3, %7;\n\t"
          "setp.gt.f32 p1, %4, %7;\n\t"
          "setp.gt.f32 p2, %5, %7;\n\t"
          "setp.gt.f32 p3, %6, %7;\n\t"
          "@p0 ld.shared.u32 i0, [%2+%8];\n\t"
          "@p1 ld.shared.u32 i1, [%2+%9];\n\t"
          "@p2 ld.shared.u32 i2, [%2+%10];\n\t"
          "@p3 ld.shared.u32 i3, [%2+%11];\n\t"
          "selp.u32 t0, %13, 0, p0;\n\t"
          "selp.u32 t1, %13, 0, p1;\n\t"
          "selp.u32 t2, %13, 0, p2;\n\t"
          "selp.u32 t3, %13, 0, p3;\n\t"
          "add.u32 a1, %1, t0;\n\t"
          "add.u32 a2, a1, t1;\n\t"
          "add.u32 a3, a2, t2;\n\t"
          "add.u32 %0, a3, t3;\n\t"
          "@p0 st.shared.f32 [%1], %3;\n\t"
          "@p0 st.shared.u32 [%1+%12], i0;\n\t"
          "@p1 st.shared.f32 [a1], %4;\n\t"
          "@p1 st.shared.u32 [a1+%12], i1;\n\t"
          "@p2 st.shared.f32 [a2], %5;\n\t"
          "@p2 st.shared.u32 [a2+%12], i2;\n\t"
          "@p3 st.shared.f32 [a3], %6;\n\t"
          "@p3 st.shared.u32 [a3+%12], i3;\n\t"
          "}\n"
          : "=r"(wn)
          : "r"(w), "r"(wbase), "f"(v[s]), "f"(v[s + 1]), "f"(v[s + 2]), "f"(v[s + 3]), "f"(thrf),
            "n"(CAP * kBM * 4 + 0 * kBM * 4), "n"(CAP * kBM * 4 + 1 * kBM * 4),
            "n"(CAP * kBM * 4 + 2 * kBM * 4), "n"(CAP * kBM * 4 + 3 * kBM * 4),
            "n"(CAP * kBM * 4), "n"(kBM * 4)
          : "memory");
      // the four index loads above address slots s .. s+3: fold the slot offset into the base
      wbase += 4 * kBM * 4;
    } else {
      wn = w;
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float x = v[s + u];
        const bool tie = (x == thrf) && tie_left > 0;
        tie_left -= tie ? 1 : 0;
        if (x > thrf || tie) {
          const uint32_t src = wbase + u * (kBM * 4) + CAP * kBM * 4;
          uint32_t ix;
          asm volatile("ld.shared.u32 %0, [%1];" : "=r"(ix) : "r"(src) : "memory");
          asm volatile("st.shared.f32 [%0], %1;\n\tst.shared.u32 [%0+%3], %2;" ::"r"(wn), "f"(x),
                       "r"(ix), "n"(CAP * kBM * 4)
                       : "memory");
          wn += kBM * 4;
        }
      }
      wbase += 4 * kBM * 4;
    }
    w = wn;
  }
  return w;
}

template <int CAP>
__device__ __noinline__ void topk_compact(uint32_t wbase, uint32_t& waddr, float& tau, int k,
                                          int slack) {
  static_assert(CAP % 4 == 0, "CAP must be a multiple of 4");
  const float ninf = __uint_as_float(0xff800000u);
  const float pinf = __uint_as_float(0x7f800000u);
  const uint32_t used = waddr - wbase;          // bytes: cnt * 512
  const int cnt = static_cast<int>(used / (kBM * 4));
  float v[CAP];
  float vmax = ninf;
#pragma unroll
  for (int s = 0; s < CAP; ++s) {
    const float x = lds_f32(wbase + s * (kBM * 4));
    v[s] = (static_cast<uint32_t>(s * (kBM * 4)) < used) ? x : ninf;
    vmax = fmaxf(vmax, v[s]);
  }
  const bool keep_all = cnt <= k + slack;   // nothing to drop for this lane (it still loops along)
  // invariants (float semantics): count(v > f(lo)) >= k,  count(v > f(hi)) < k
  uint32_t lo;
  if (tau == ninf) {                        // first compaction of a work item (warp-uniform)
    float vmin = pinf;
#pragma unroll
    for (int s = 0; s < CAP; ++s) vmin = fminf(vmin, (v[s] == ninf) ? pinf : v[s]);
    lo = f2key(vmin) - 1u;                  // below every candidate: count == cnt
  } else {
    // every candidate is >= tau (a tie-breaking compaction keeps entries EQUAL to the tau it sets):
    // start just below it, so count == cnt
    lo = f2key(tau) - 1u;
  }
  uint32_t hi = f2key(vmax);                // count == 0
  int c_lo = cnt;
  bool done = keep_all;
  int it = 0;
  while (true) {
    const bool active = !done && (hi - lo > 1u);
    if (!__any_sync(0xffffffffu, active)) break;
    const uint32_t span = hi - lo;
    // the k-th largest sits in the dense lower part of [vmin, vmax]: first probes split 1:3
    const uint32_t step = max(1u, span >> (it < 2 ? 2 : 1));
    ++it;
    const uint32_t mid = lo + step;
    const float midf = key2f(mid);
    float c0 = 0.f, c1 = 0.f, c2 = 0.f, c3 = 0.f;
#pragma unroll
    for (int s = 0; s < CAP; s += 4) {
      c0 += (v[s] > midf) ? 1.f : 0.f;
      c1 += (v[s + 1] > midf) ? 1.f : 0.f;
      c2 += (v[s + 2] > midf) ? 1.f : 0.f;
      c3 += (v[s + 3] > midf) ? 1.f : 0.f;
    }
    const int c = static_cast<int>((c0 + c1) + (c2 + c3));
    if (active) {
      if (c >= k) {
        lo = mid;
        c_lo = c;
        done = (c <= k + slack);
      } else {
        hi = mid;
      }
    }
  }
  // done: keep v > f(lo).  otherwise hi == lo + 1: the values equal to f(hi) tie across the k-th
  // position; keep everything above plus the first (k - m) ties (lowest feature index first).
  const bool ties = !done;
  const float thrf = keep_all ? ninf : key2f(done ? lo : hi);
  uint32_t wnew;
  if (!__any_sync(0xffffffffu, ties)) {
    wnew = compact_move<CAP, false>(v, wbase, thrf, 0);
  } else {
    int tie_left = 0;
    if (ties) {
      int m = 0;
#pragma unroll
      for (int s = 0; s < CAP; ++s) m += (v[s] > thrf) ? 1 : 0;
      tie_left = k - m;
    }
    wnew = compact_move<CAP, true>(v, wbase, thrf, tie_left);
  }
  if (!keep_all) {
    waddr = wnew;
    if (c_lo >= k) tau = thrf;
  }
}

// End of a work item: reduce the list to exactly k entries and write them to global memory.
// After one ordinary compaction (<= k + kSlack survivors) the few surplus entries are removed by
// repeated min-extraction in registers - much cheaper than bisecting down to adjacent float keys.
// Ties at the k-th value keep the lowest feature index: among equal minima the LAST list slot
// (highest index; the list is in ascending index order) is dropped first.  NaN marks a slot that holds
// no candidate (no NaN ever enters the list), so a +inf candidate is kept like any other value.
template <int CAP, int KMAX>
__device__ __noinline__ void topk_finalize(uint32_t wbase, uint32_t waddr, float tau, int k,
                                           float* __restrict__ out_val,
                                           int32_t* __restrict__ out_idx, bool write) {
  constexpr int NB = KMAX + kSlack;
  const float ninf = __uint_as_float(0xff800000u);
  const float pinf = __uint_as_float(0x7f800000u);
  const float none = __uint_as_float(0x7fc00000u);
  if (__any_sync(0xffffffffu, waddr > wbase + static_cast<uint32_t>(k + kSlack) * (kBM * 4)))
    topk_compact<CAP>(wbase, waddr, tau, k, kSlack);
  const uint32_t used = waddr - wbase;
  int surplus = static_cast<int>(used / (kBM * 4)) - k;     // <= kSlack; negative: fewer than k
  float v[NB];
#pragma unroll
  for (int s = 0; s < NB; ++s) {
    const float x = lds_f32(wbase + s * (kBM * 4));
    v[s] = (static_cast<uint32_t>(s * (kBM * 4)) < used) ? x : none;
  }
  while (__any_sync(0xffffffffu, surplus > 0)) {
    float vmin = pinf;
    int pos = -1;
#pragma unroll
    for (int s = 0; s < NB; ++s) {
      const bool le = v[s] <= vmin;    // false for NaN
      vmin = le ? v[s] : vmin;
      pos = le ? s : pos;
    }
    if (surplus <= 0) pos = -1;
#pragma unroll
    for (int s = 0; s < NB; ++s) v[s] = (s == pos) ? none : v[s];
    --surplus;
  }
  if (write) {
    int w = 0;
#pragma unroll
    for (int s = 0; s < NB; ++s) {
      if (v[s] == v[s] && w < k) {
        uint32_t ix;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(ix) : "r"(wbase + s * (kBM * 4) + CAP * kBM * 4) : "memory");
        out_val[w] = v[s];
        out_idx[w] = static_cast<int32_t>(ix);
        ++w;
      }
    }
    for (; w < k; ++w) {   // fewer than k candidates (split narrower than k, NaN rows): pad
      out_val[w] = ninf;
      out_idx[w] = -1;
    }
  }
}

// Work decomposition shared by every role of the GEMM pipeline.
struct EncodeItems {
  int total_items, nsplit, tiles_per_split, num_n_tiles, num_kb, ksteps;
};

// TMA producer (one elected lane): streams A' 128x64 and W' 256x64 boxes through the stage ring.
template <int STAGES, int NS = 0>
__device__ __forceinline__ void encode_producer_loop(const CUtensorMap* tmap_a,
                                                     const CUtensorMap* tmap_w, uint8_t* pipe,
                                                     uint64_t* full_bar, uint64_t* empty_bar,
                                                     const EncodeItems& it) {
  int stage = 0;
  uint32_t phase = 0;
  for (int item = blockIdx.x; item < it.total_items; item += gridDim.x) {
    const int m_blk = item / it.nsplit;
    const int sp = item - m_blk * it.nsplit;
    const int t0 = sp * it.tiles_per_split;
    const int t1 = min(t0 + it.tiles_per_split, it.num_n_tiles);
    for (int nt = t0; nt < t1; ++nt) {
      for (int kb = 0; kb < it.num_kb; ++kb) {
        mbar_wait_sleep<NS>(&empty_bar[stage], phase ^ 1u);
        mbar_arrive_expect_tx(&full_bar[stage], kAStage + kBStage);
        uint8_t* sa = pipe + stage * (kAStage + kBStage);
        tma_load_2d(sa, tmap_a, &full_bar[stage], kb * kBK, m_blk * kBM);
        tma_load_2d(sa + kAStage, tmap_w, &full_bar[stage], kb * kBK, nt * kBN);
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1u;
        }
      }
    }
  }
}

// MMA issuer (whole warp; one elected lane issues): 128x256x16 tcgen05.mma into the double-buffered
// TMEM accumulators.
template <int STAGES, int NS = 0>
__device__ __forceinline__ void encode_mma_loop(uint8_t* pipe, uint64_t* full_bar,
                                                uint64_t* empty_bar, uint64_t* tfull_bar,
                                                uint64_t* tempty_bar, uint32_t tmem_base,
                                                const EncodeItems& it) {
  constexpr uint32_t idesc = umma_idesc_bf16(kBM, kBN);
  int stage = 0;
  uint32_t phase = 0;
  uint32_t tile = 0;
  for (int item = blockIdx.x; item < it.total_items; item += gridDim.x) {
    const int m_blk = item / it.nsplit;
    const int sp = item - m_blk * it.nsplit;
    const int t0 = sp * it.tiles_per_split;
    const int t1 = min(t0 + it.tiles_per_split, it.num_n_tiles);
    for (int nt = t0; nt < t1; ++nt, ++tile) {
      const uint32_t as = tile & 1u;
      const uint32_t aphase = (tile >> 1) & 1u;
      mbar_wait_sleep<NS>(&tempty_bar[as], aphase ^ 1u);
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + as * kBN;
      for (int kb = 0; kb < it.num_kb; ++kb) {
        mbar_wait_sleep<NS>(&full_bar[stage], phase);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t sa = smem_u32(pipe + stage * (kAStage + kBStage));
          const uint64_t da = umma_desc_sw128_kmajor(sa);
          const uint64_t db = umma_desc_sw128_kmajor(sa + kAStage);
          const int nks = min(kBK / 16, it.ksteps - kb * (kBK / 16));
          for (int ks = 0; ks < nks; ++ks) {
            // advance 16 bf16 = 32 bytes inside the 128-byte swizzle row: +2 in 16-byte units
            umma_bf16(tmem_d, da + static_cast<uint64_t>(2 * ks), db + static_cast<uint64_t>(2 * ks),
                      idesc, (kb | ks) != 0 ? 1u : 0u);
          }
          umma_commit(&empty_bar[stage]);
          if (kb == it.num_kb - 1) umma_commit(&tfull_bar[as]);
        }
        __syncwarp();
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1u;
        }
      }
    }
  }
}

template <int CAP, int STAGES>
__global__ void __launch_bounds__(256, 1)
encode_topk_kernel(const __grid_constant__ CUtensorMap tmap_a,
                   const __grid_constant__ CUtensorMap tmap_w, int B, int F, int k, int ksteps,
                   int num_m_blocks, int num_n_tiles, int nsplit, int tiles_per_split,
                   float* __restrict__ out_val, int32_t* __restrict__ out_idx, int dbg) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // 1024-byte alignment for SWIZZLE_128B tiles, computed as an OFFSET so that the pointers keep
  // their shared address space (a uintptr_t round-trip would demote every access to generic LD/ST)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* pipe = smem;
  float* cand_val = reinterpret_cast<float*>(smem + EncodeSmem<CAP, STAGES>::kPipeBytes);
  uint32_t* cand_idx = reinterpret_cast<uint32_t*>(cand_val + CAP * kBM);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + EncodeSmem<CAP, STAGES>::kPipeBytes +
                                               EncodeSmem<CAP, STAGES>::kCandBytes);
  uint64_t* full_bar = bars;                  // [STAGES]
  uint64_t* empty_bar = bars + STAGES;        // [STAGES]
  uint64_t* tfull_bar = bars + 2 * STAGES;    // [2]
  uint64_t* tempty_bar = bars + 2 * STAGES + 2;  // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_kb = ceil_div(ksteps, kBK / 16);
  const int total_items = num_m_blocks * nsplit;
  const EncodeItems items{total_items, nsplit, tiles_per_split, num_n_tiles, num_kb, ksteps};

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_w);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull_bar[s], 1);
      mbar_init(&tempty_bar[s], kBM);
    }
    mbar_fence_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (elect_one()) encode_producer_loop<STAGES>(&tmap_a, &tmap_w, pipe, full_bar, empty_bar, items);
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    encode_mma_loop<STAGES>(pipe, full_bar, empty_bar, tfull_bar, tempty_bar, tmem_base, items);
  } else if (warp >= 4) {
    // ===================== epilogue: streaming TopK =====================
    const int q = warp - 4;               // TMEM lane quarter this warp may read
    const int row_in_blk = q * 32 + lane;
    float* cv = cand_val + row_in_blk;
    uint32_t* ci = cand_idx + row_in_blk;
    const float neg_inf = __uint_as_float(0xff800000u);
    const uint32_t wbase = smem_u32(cv);                           // list cursor = byte address
    // the overflow check runs every kCheck values: kCheck more must always fit
    const uint32_t wlimit = wbase + (CAP - kCheck) * (kBM * 4);
    uint32_t tile = 0;
    for (int item = blockIdx.x; item < total_items; item += gridDim.x) {
      const int m_blk = item / nsplit;
      const int sp = item - m_blk * nsplit;
      const int t0 = sp * tiles_per_split;
      const int t1 = min(t0 + tiles_per_split, num_n_tiles);
      uint32_t waddr = wbase;
      float tau = neg_inf;
      for (int nt = t0; nt < t1; ++nt, ++tile) {
        const uint32_t as = tile & 1u;
        const uint32_t aphase = (tile >> 1) & 1u;
        mbar_wait(&tfull_bar[as], aphase);
        tc_fence_after();
        const int col0 = nt * kBN;
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * kBN;

        // Branch-free append, four values per block: a value above tau is stored at the list
        // cursor and the cursor advances.  No warp-level branch (some lane would take it for
        // nearly every value: ~k*ln(F/k) values pass per row), and the cursor chain is kept in
        // fresh registers (a0 -> a1 -> a2 -> a3 -> a0') so that no address register is rewritten
        // while a store that reads it is still in flight (the read-after-write scoreboard wait
        // on an in-place `@p add` costs ~20 cycles per value).
        // Zero-padded feature rows of W' carry a -inf bias (wsae_pack.cu), so they never pass.
        auto process = [&](uint32_t (&r)[16], int cbase) {
#pragma unroll
          for (int j = 0; j < kChunk; j += 4) {
            uint32_t wnext;
            asm volatile(
                "{\n\t"
                ".reg .pred p0, p1, p2, p3;\n\t"
                ".reg .u32 a1, a2, a3, t0, t1, t2, t3, i1, i2, i3;\n\t"
                "setp.gt.f32 p0, %2, %6;\n\t"
                "setp.gt.f32 p1, %3, %6;\n\t"
                "setp.gt.f32 p2, %4, %6;\n\t"
                "setp.gt.f32 p3, %5, %6;\n\t"
                "selp.u32 t0, %9, 0, p0;\n\t"
                "selp.u32 t1, %9, 0, p1;\n\t"
                "selp.u32 t2, %9, 0, p2;\n\t"
                "selp.u32 t3, %9, 0, p3;\n\t"
                "add.u32 a1, %1, t0;\n\t"
                "add.u32 a2, a1, t1;\n\t"
                "add.u32 a3, a2, t2;\n\t"
                "add.u32 %0, a3, t3;\n\t"
                "add.u32 i1, %7, 1;\n\t"
                "add.u32 i2, %7, 2;\n\t"
                "add.u32 i3, %7, 3;\n\t"
                "@p0 st.shared.f32 [%1], %2;\n\t"
                "@p0 st.shared.u32 [%1+%8], %7;\n\t"
                "@p1 st.shared.f32 [a1], %3;\n\t"
                "@p1 st.shared.u32 [a1+%8], i1;\n\t"
                "@p2 st.shared.f32 [a2], %4;\n\t"
                "@p2 st.shared.u32 [a2+%8], i2;\n\t"
                "@p3 st.shared.f32 [a3], %5;\n\t"
                "@p3 st.shared.u32 [a3+%8], i3;\n\t"
                "}\n"
                : "=r"(wnext)
                : "r"(waddr), "f"(__uint_as_float(r[j])), "f"(__uint_as_float(r[j + 1])),
                  "f"(__uint_as_float(r[j + 2])), "f"(__uint_as_float(r[j + 3])), "f"(tau),
                  "r"(static_cast<uint32_t>(cbase + j)), "n"(CAP * kBM * 4), "n"(kBM * 4)
                : "memory");
            waddr = wnext;
            if ((j + 4) % kCheck == 0) {
              if (dbg == 2) {
                if (waddr > wlimit) waddr = wbase;
              } else if (__any_sync(0xffffffffu, waddr > wlimit)) {
                topk_compact<CAP>(wbase, waddr, tau, k, kSlack);
              }
            }
          }
        };

        // Every tile is scanned in full: columns >= F are padding rows of W' (never selected).
        uint32_t ra[16], rb[16];
        if (dbg == 1) { tc_fence_before(); mbar_arrive(&tempty_bar[as]); continue; }
        tmem_ld16(taddr, ra);
#pragma unroll 1
        for (int c4 = 0; c4 < kBN / 64; ++c4) {
          const uint32_t ta = taddr + c4 * 64;
          const int cb = col0 + c4 * 64;
          tmem_ld_wait16(ra);
          tmem_ld16(ta + 16, rb);
          process(ra, cb);
          tmem_ld_wait16(rb);
          tmem_ld16(ta + 32, ra);
          process(rb, cb + 16);
          tmem_ld_wait16(ra);
          tmem_ld16(ta + 48, rb);
          process(ra, cb + 32);
          tmem_ld_wait16(rb);
          if (c4 + 1 < kBN / 64) tmem_ld16(ta + 64, ra);
          process(rb, cb + 48);
        }
        // accumulator stage fully read: hand it back to the MMA warp
        tc_fence_before();
        mbar_arrive(&tempty_bar[as]);
      }
      // ---- end of work item: exact select, write k (val, idx) pairs for this row/split ----
      const int row = m_blk * kBM + row_in_blk;
      const size_t obase = (static_cast<size_t>(row < B ? row : 0) * nsplit + sp) * k;
      topk_finalize<CAP, (CAP >= 128 ? 64 : 32)>(wbase, waddr, tau, k, out_val + obase,
                                                 out_idx + obase, row < B);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ================================================================================================
// K1, second epilogue organisation: SCANNER + SELECTOR warps (used for k <= 32).
//
// In the kernel above one epilogue warp per SM sub-partition does everything and issues only
// ~0.4 instructions per cycle (fixed-latency dependency stalls; profiles/r1_v3_k1_*.txt), while
// its list compactions cost as much as the scan itself.  Here each 32-row TMEM lane quarter is
// served by TWO warps on the same sub-partition that run concurrently:
//   * the scanner (warps 4-7) reads the accumulators from TMEM and appends every value above its
//     row threshold tau to a 40-slot FIFO in shared memory - nothing else;
//   * the selector (warps 8-11) keeps the row's current <= k+8 survivors in REGISTERS, merges
//     each handed-over FIFO batch into them (bisection select, repack through the FIFO it just
//     drained), publishes the raised tau back to the scanner, and at the end of the work item
//     reduces to exactly k and writes the result.
// Two FIFO buffers per quarter ping-pong between the two warps on mbarriers (full / empty), so
// scanning batch n+1 overlaps selecting batch n.  A stale (lower) tau in the scanner only lets a
// few more candidates through: the result is unchanged and exact.
// Registers: 384 threads; setmaxnreg moves registers from the producer/MMA warpgroup to the
// selector warpgroup (which holds 80 values + 80 indices per thread).
// ================================================================================================
#ifndef WSAE_ROLE_SLEEP_NS
#define WSAE_ROLE_SLEEP_NS 64
#endif
constexpr int kRoleSleepNs = WSAE_ROLE_SLEEP_NS;   // poll interval of the TMA / MMA roles (see mbar_wait_sleep)
constexpr int kFifo = 40;                          // slots per FIFO buffer (>= k + kSlack)
constexpr int kFifoBytes = kFifo * kBM * 4;        // one buffer of one array: 20480 B
constexpr int kFifoIdxOff = 2 * kFifoBytes;        // idx array sits behind both value buffers

template <int STAGES>
struct Encode2Smem {
  static constexpr int kPipeBytes = STAGES * (kAStage + kBStage);
  static constexpr int kFifoTotal = 4 * kFifoBytes;             // 2 buffers x (val + idx)
  static constexpr int kTauBytes = kBM * 8;                     // {tau, item seq} per row
  static constexpr int kCntBytes = 2 * kBM * 2;                 // entries per row per buffer (u16)
  static constexpr int kBarBytes = 256;
  static_assert((2 * STAGES + 20) * 8 + 8 + 32 <= kBarBytes, "barrier block too small");
  static constexpr int kTotal = kPipeBytes + kFifoTotal + kTauBytes + kCntBytes + kBarBytes + 1024;
  static_assert(kTotal <= 232448, "exceeds the 227 KB shared-memory limit");
};

template <int REGS>
__device__ __forceinline__ void reg_alloc_inc() {
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS));
}
template <int REGS>
__device__ __forceinline__ void reg_alloc_dec() {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS));
}

// Predicated append of four (value, index) pairs at cursor w; IOFF = byte offset of the index array.
// `slot` is the slot stride (kBM * 4 bytes) passed in a REGISTER that ptxas cannot constant-fold (it
// comes from a kernel parameter): with an immediate, ptxas rewrites `selp t, 512, 0, p; add a1, a0, t`
// into `VIADD a1 = a0 + 512; @!p MOV a1 = a0` - two dependent instructions per value on the
// loop-carried cursor chain, which bounded the scanner at ~15 cycles per value (ncu: `wait` stalls on
// exactly those pairs).  SEL + IADD keeps one dependent instruction per value.
// (A variant whose four slot addresses are w + prefix sums of the pass flags measured slower, 277 vs
// 260 us: ptxas built the prefix sums from the same VIADD/MOV pairs.)
template <int IOFF>
__device__ __forceinline__ uint32_t append4(uint32_t w, float thr, float v0, float v1, float v2,
                                            float v3, uint32_t i0, uint32_t i1, uint32_t i2,
                                            uint32_t i3, uint32_t slot) {
  uint32_t wn;
  asm volatile(
      "{\n\t"
      ".reg .pred p0, p1, p2, p3;\n\t"
      ".reg .u32 a1, a2, a3, t0, t1, t2, t3;\n\t"
      "setp.gt.f32 p0, %2, %6;\n\t"
      "setp.gt.f32 p1, %3, %6;\n\t"
      "setp.gt.f32 p2, %4, %6;\n\t"
      "setp.gt.f32 p3, %5, %6;\n\t"
      "selp.u32 t0, %12, 0, p0;\n\t"
      "selp.u32 t1, %12, 0, p1;\n\t"
      "selp.u32 t2, %12, 0, p2;\n\t"
      "selp.u32 t3, %12, 0, p3;\n\t"
      "add.u32 a1, %1, t0;\n\t"
      "add.u32 a2, a1, t1;\n\t"
      "add.u32 a3, a2, t2;\n\t"
      "add.u32 %0, a3, t3;\n\t"
      "@p0 st.shared.f32 [%1], %2;\n\t"
      "@p0 st.shared.u32 [%1+%11], %7;\n\t"
      "@p1 st.shared.f32 [a1], %3;\n\t"
      "@p1 st.shared.u32 [a1+%11], %8;\n\t"
      "@p2 st.shared.f32 [a2], %4;\n\t"
      "@p2 st.shared.u32 [a2+%11], %9;\n\t"
      "@p3 st.shared.f32 [a3], %5;\n\t"
      "@p3 st.shared.u32 [a3+%11], %10;\n\t"
      "}\n"
      : "=r"(wn)
      : "r"(w), "f"(v0), "f"(v1), "f"(v2), "f"(v3), "f"(thr), "r"(i0), "r"(i1), "r"(i2), "r"(i3),
        "n"(IOFF), "r"(slot)
      : "memory");
  return wn;
}

// min.NaN.f32: unlike fminf, a NaN operand makes the result NaN
__device__ __forceinline__ float fmin_nan(float a, float b) {
  float r;
  asm("min.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}

// Scanner threshold from the floor of a work item's first tile (the smallest of its 32 group maxima,
// taken with fmin_nan).  Candidates must be strictly above the threshold, so it steps to the next float
// below the floor, and below -0.0 when the floor is +0.0 or -0.0: every value equal to the floor still
// passes.  A floor that is NaN (a group of 8 NaN columns has no maximum) or -inf (padding columns)
// bounds nothing: tau stays where it is.
__device__ __forceinline__ float floor_threshold(float floor_v, float tau) {
  if (!(floor_v > __uint_as_float(0xff800000u))) return tau;
  return fmaxf(tau, key2f(f2key(floor_v == 0.f ? -0.f : floor_v) - 1u));
}

__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void sts_u32(uint32_t addr, uint32_t v) {
  asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

// Threshold such that k <= count(v > thr) <= k + slack over the N register-resident candidates
// (-inf entries are padding).  Same bisection as topk_compact.  If the candidates tie across the
// k-th position beyond the slack, `ties` is set and thr is the tie value: keep everything above it
// plus the first `tie_left` ties in list order.
template <int N>
__device__ __forceinline__ float select_threshold(const float (&v)[N], int total, int k, int slack,
                                                  float tau, bool& ties, int& tie_left) {
  const float ninf = __uint_as_float(0xff800000u);
  const float pinf = __uint_as_float(0x7f800000u);
  const bool keep_all = total <= k + slack;
  float m0 = ninf, m1 = ninf, m2 = ninf, m3 = ninf;     // four independent chains (latency)
#pragma unroll
  for (int s = 0; s < N; s += 4) {
    m0 = fmaxf(m0, v[s]);
    m1 = fmaxf(m1, v[s + 1]);
    m2 = fmaxf(m2, v[s + 2]);
    m3 = fmaxf(m3, v[s + 3]);
  }
  const float vmax = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
  uint32_t lo;
  if (tau == ninf) {
    float n0 = pinf, n1 = pinf, n2 = pinf, n3 = pinf;
#pragma unroll
    for (int s = 0; s < N; s += 4) {
      n0 = fminf(n0, (v[s] == ninf) ? pinf : v[s]);
      n1 = fminf(n1, (v[s + 1] == ninf) ? pinf : v[s + 1]);
      n2 = fminf(n2, (v[s + 2] == ninf) ? pinf : v[s + 2]);
      n3 = fminf(n3, (v[s + 3] == ninf) ? pinf : v[s + 3]);
    }
    const float vmin = fminf(fminf(n0, n1), fminf(n2, n3));
    lo = f2key(vmin) - 1u;
  } else {
    lo = f2key(tau) - 1u;   // survivors of a tie-breaking select equal tau: start just below it
  }
  uint32_t hi = f2key(vmax);
  bool done = keep_all;
  int it = 0;
  while (true) {
    const bool active = !done && (hi - lo > 1u);
    if (!__any_sync(0xffffffffu, active)) break;
    const uint32_t span = hi - lo;
    const uint32_t step = max(1u, span >> (it < 2 ? 2 : 1));
    ++it;
    const uint32_t mid = lo + step;
    const float midf = key2f(mid);
    float c0 = 0.f, c1 = 0.f, c2 = 0.f, c3 = 0.f;
#pragma unroll
    for (int s = 0; s < N; s += 4) {
      c0 += (v[s] > midf) ? 1.f : 0.f;
      c1 += (v[s + 1] > midf) ? 1.f : 0.f;
      c2 += (v[s + 2] > midf) ? 1.f : 0.f;
      c3 += (v[s + 3] > midf) ? 1.f : 0.f;
    }
    const int c = static_cast<int>((c0 + c1) + (c2 + c3));
    if (active) {
      if (c >= k) {
        lo = mid;
        done = (c <= k + slack);
      } else {
        hi = mid;
      }
    }
  }
  ties = !done;
  tie_left = 0;
  const float thrf = keep_all ? ninf : key2f(done ? lo : hi);
  if (ties) {
    int m = 0;
#pragma unroll
    for (int s = 0; s < N; ++s) m += (v[s] > thrf) ? 1 : 0;
    tie_left = k - m;
  }
  return thrf;
}

// Scanner -> selector hand-over of the FIFO buffer in use (out of line: ~13 calls per work item;
// inlined at every check site it made the scan loop twice the size of the L0 instruction cache).
// st: bit 0 = buffer in use, bits 1 / 2 = parity of the number of fills of buffer 0 / 1.
// Publishes the row's entry count and the `last` flag, arrives on the buffer's full barrier,
// switches to the other buffer and (unless this was the item's last hand-over) waits until the
// selector has drained it.  *_q pointers are this lane quarter's entry of the [2][4] arrays.
template <bool DBG>
__device__ __noinline__ uint32_t scanner_handoff(uint32_t st, uint32_t nslots, uint32_t last,
                                                 uint32_t cnt_addr, uint32_t* meta_q,
                                                 uint64_t* ffull_q, uint64_t* fempty_q, int lane,
                                                 unsigned long long* waited) {
  const uint32_t b = st & 1u;
  asm volatile("st.shared.u16 [%0], %1;" ::"r"(cnt_addr + b * (kBM * 2)),
               "h"(static_cast<unsigned short>(nslots))
               : "memory");
  if (lane == 0) meta_q[b * 4] = last;
  mbar_arrive(&ffull_q[b * 4]);
  st ^= (2u << b) | 1u;                 // one more fill of buffer b; continue on the other buffer
  if (!last) {
    const uint32_t nb = st & 1u;
    const long long t = DBG ? clock64() : 0;
    mbar_wait_backoff(&fempty_q[nb * 4], ((st >> (1u + nb)) & 1u) ^ 1u);
    if (DBG) *waited += clock64() - t;
  }
  return st;
}

template <int STAGES, bool DBG>
__global__ void __launch_bounds__(384, 1)
encode_topk2_kernel(const __grid_constant__ CUtensorMap tmap_a,
                    const __grid_constant__ CUtensorMap tmap_w, int B, int F, int k, int ksteps,
                    int num_m_blocks, int num_n_tiles, int nsplit, int tiles_per_split,
                    float* __restrict__ out_val, int32_t* __restrict__ out_idx,
                    unsigned long long* __restrict__ dbg, int mode, uint32_t slot) {
  using SM = Encode2Smem<STAGES>;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* pipe = smem;
  uint8_t* fifo = smem + SM::kPipeBytes;
  uint8_t* tau_s = fifo + SM::kFifoTotal;
  uint8_t* cnt_s = tau_s + SM::kTauBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(cnt_s + SM::kCntBytes);
  uint64_t* full_bar = bars;                        // [STAGES]
  uint64_t* empty_bar = bars + STAGES;              // [STAGES]
  uint64_t* tfull_bar = bars + 2 * STAGES;          // [2]
  uint64_t* tempty_bar = bars + 2 * STAGES + 2;     // [2]
  uint64_t* ffull_bar = bars + 2 * STAGES + 4;      // [2 buffers][4 quarters]
  uint64_t* fempty_bar = bars + 2 * STAGES + 12;    // [2][4]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 20);
  uint32_t* meta = tmem_slot + 2;                   // [2][4]: 1 = last hand-over of the work item

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_kb = ceil_div(ksteps, kBK / 16);
  const int total_items = num_m_blocks * nsplit;
  const EncodeItems items{total_items, nsplit, tiles_per_split, num_n_tiles, num_kb, ksteps};
  const float neg_inf = __uint_as_float(0xff800000u);

  pdl_launch_dependents();
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_w);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull_bar[s], 1);
      mbar_init(&tempty_bar[s], kBM);
    }
    for (int s = 0; s < 8; ++s) {
      mbar_init(&ffull_bar[s], 32);
      mbar_init(&fempty_bar[s], 32);
    }
    mbar_fence_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  for (int i = threadIdx.x; i < kBM * 2; i += blockDim.x) reinterpret_cast<uint32_t*>(tau_s)[i] = 0u;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();   // set-up done under the predecessor's tail; global memory (TMA, results) from here on

  if (warp < 4) {
    reg_alloc_dec<56>();
    if (warp == 0) {
      if (elect_one())
        encode_producer_loop<STAGES, kRoleSleepNs>(&tmap_a, &tmap_w, pipe, full_bar, empty_bar, items);
    } else if (warp == 1) {
      encode_mma_loop<STAGES, kRoleSleepNs>(pipe, full_bar, empty_bar, tfull_bar, tempty_bar, tmem_base,
                                            items);
    }
  } else if (warp < 8) {
    // ===================== scanner =====================
    reg_alloc_dec<152>();
    const int q = warp - 4;
    const int row_in_blk = q * 32 + lane;
    const uint32_t fv0 = smem_u32(fifo) + row_in_blk * 4;          // buffer 0, slot 0 of this row
    const uint32_t tau_addr = smem_u32(tau_s) + row_in_blk * 8;
    const uint32_t cnt_addr = smem_u32(cnt_s) + row_in_blk * 2;
    uint32_t st = 0, seq = 0, tile = 0;      // st: bit 0 = FIFO buffer in use, bits 1/2 = fill parities
    unsigned long long d_hand = 0, d_wait_e = 0, d_wait_t = 0;
    const long long d_t0 = clock64();
    for (int item = blockIdx.x; item < total_items; item += gridDim.x) {
      const int sp = item - (item / nsplit) * nsplit;
      const int t0 = sp * tiles_per_split;
      const int t1 = min(t0 + tiles_per_split, num_n_tiles);
      ++seq;
      // mode 3 (experiments): nothing passes the filter - times the GEMM pipeline + bare scan
      float tau = (DBG && mode >= 3) ? __uint_as_float(0x7f800000u) : neg_inf;
      mbar_wait_backoff(&fempty_bar[(st & 1u) * 4 + q], ((st >> (1u + (st & 1u))) & 1u) ^ 1u);
      uint32_t wbase = fv0 + (st & 1u) * kFifoBytes;
      uint32_t waddr = wbase;
      uint32_t wlimit = wbase + (kFifo - kCheck) * (kBM * 4);

      for (int nt = t0; nt < t1; ++nt, ++tile) {
        const uint32_t as = tile & 1u;
        const uint32_t aphase = (tile >> 1) & 1u;
        {
          const long long t = DBG ? clock64() : 0;
          mbar_wait(&tfull_bar[as], aphase);
          if (DBG) d_wait_t += clock64() - t;
        }
        tc_fence_after();
        const int col0 = nt * kBN;
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * kBN;

        // ---- first tile of a work item: a floor for the row's threshold before anything is scanned ----
        // The tile's 256 columns form 32 groups of 8; the smallest of the 32 group maxima has at
        // least 32 >= k values at or above it, so the row's k-th largest value cannot be below it.
        // Starting from (just under) that floor instead of -inf, the first tile passes ~40 % of
        // its values instead of all of the first ~120 columns: about two hand-overs fewer per item,
        // in the part of the item where the selector is the bottleneck.  Costs one extra read of
        // the tile (16 tcgen05.ld) and ~0.6 instructions per value while the selector is idle.
        // A group of 8 NaN columns has no maximum: fmin_nan turns the floor into NaN, and padding
        // columns (-inf) turn it into -inf; either leaves tau at -inf.  (k <= 32 here.)
        if (nt == t0 && !(DBG && mode >= 3)) {
          float floor_v = __uint_as_float(0x7f800000u);
          uint32_t rp[16];
#pragma unroll 1
          for (int c = 0; c < kBN; c += 16) {
            tmem_ld16(taddr + c, rp);
            tmem_ld_wait16(rp);
            const float m0 = fmaxf(fmaxf(fmaxf(__uint_as_float(rp[0]), __uint_as_float(rp[1])),
                                         fmaxf(__uint_as_float(rp[2]), __uint_as_float(rp[3]))),
                                   fmaxf(fmaxf(__uint_as_float(rp[4]), __uint_as_float(rp[5])),
                                         fmaxf(__uint_as_float(rp[6]), __uint_as_float(rp[7]))));
            const float m1 = fmaxf(fmaxf(fmaxf(__uint_as_float(rp[8]), __uint_as_float(rp[9])),
                                         fmaxf(__uint_as_float(rp[10]), __uint_as_float(rp[11]))),
                                   fmaxf(fmaxf(__uint_as_float(rp[12]), __uint_as_float(rp[13])),
                                         fmaxf(__uint_as_float(rp[14]), __uint_as_float(rp[15]))));
            floor_v = fmin_nan(floor_v, fmin_nan(m0, m1));
          }
          tau = floor_threshold(floor_v, tau);
        }

        // ---- scan of one 128x256 accumulator tile, 32 columns (two tcgen05.ld.x16) per trip ----
        // A taken branch costs a lone warp ~45-60 cycles (instruction-fetch bubble) and ptxas lays a
        // rare `if (overflow) handoff();` block inline, i.e. the COMMON path takes a skip-branch at
        // every overflow check - four per trip, a third of the scan time.  So the hot trip has no
        // branch at all: an overflow check only folds its vote into `need`, and from then on the
        // filter is closed (threshold +inf) for the rest of the trip.  The single branch per trip is
        // the loop back-edge, which also tests `need`; when it falls through, the cold code below
        // hands the FIFO over and re-scans the groups of that trip that ran with the filter closed.
        auto scan8 = [&](const uint32_t (&r)[16], int j0, int cbase, float thr) {
          const uint32_t c = static_cast<uint32_t>(cbase + j0);
          waddr = append4<kFifoIdxOff>(waddr, thr, __uint_as_float(r[j0]), __uint_as_float(r[j0 + 1]),
                                       __uint_as_float(r[j0 + 2]), __uint_as_float(r[j0 + 3]), c, c + 1,
                                       c + 2, c + 3, slot);
          waddr = append4<kFifoIdxOff>(waddr, thr, __uint_as_float(r[j0 + 4]), __uint_as_float(r[j0 + 5]),
                                       __uint_as_float(r[j0 + 6]), __uint_as_float(r[j0 + 7]), c + 4,
                                       c + 5, c + 6, c + 7, slot);
        };
        auto handoff = [&]() {
          st = scanner_handoff<DBG>(st, (waddr - wbase) / (kBM * 4), 0u, cnt_addr, meta + q,
                                    ffull_bar + q, fempty_bar + q, lane, &d_wait_e);
          ++d_hand;
          wbase = fv0 + (st & 1u) * kFifoBytes;
          waddr = wbase;
          wlimit = wbase + (kFifo - kCheck) * (kBM * 4);
        };
        const float pos_inf = __uint_as_float(0x7f800000u);
        uint32_t ra[16], rb[16];
        tmem_ld16(taddr, ra);
        int c2 = 0;
        while (true) {
          bool need = false;
          int done = 0;            // groups of 8 columns of the current trip scanned with the filter open
#pragma unroll 1
          do {
            const uint32_t ta = taddr + c2 * 32;
            const int cb = col0 + c2 * 32;
            uint32_t tb, tq;   // the selector's latest threshold for this row (valid for this item only)
            asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(tb), "=r"(tq) : "r"(tau_addr) : "memory");
            tmem_ld_wait16(ra);
            tmem_ld16(ta + 16, rb);
            if (tq == seq) tau = fmaxf(tau, __uint_as_float(tb));
            float thr = tau;
            done = 0;
            if (DBG && mode == 4) {        // experiments: TMEM reads only (one compare keeps the loads live)
              if (__uint_as_float(ra[0]) == tau) waddr += 4;
              tmem_ld_wait16(rb);
              if (c2 + 1 < kBN / 32) tmem_ld16(ta + 32, ra);
              if (__uint_as_float(rb[0]) == tau) waddr += 4;
            } else {
              scan8(ra, 0, cb, thr);
              done += need ? 0 : 1;
              need = need | __any_sync(0xffffffffu, waddr > wlimit);
              thr = need ? pos_inf : thr;
              scan8(ra, 8, cb, thr);
              done += need ? 0 : 1;
              need = need | __any_sync(0xffffffffu, waddr > wlimit);
              thr = need ? pos_inf : thr;
              tmem_ld_wait16(rb);
              if (c2 + 1 < kBN / 32) tmem_ld16(ta + 32, ra);
              scan8(rb, 0, cb + 16, thr);
              done += need ? 0 : 1;
              need = need | __any_sync(0xffffffffu, waddr > wlimit);
              thr = need ? pos_inf : thr;
              scan8(rb, 8, cb + 16, thr);
              done += need ? 0 : 1;
              need = need | __any_sync(0xffffffffu, waddr > wlimit);
            }
            ++c2;
          } while (!need && c2 < kBN / 32);
          if (!need) break;                                  // tile scanned
          // ---- cold path: hand the FIFO over, re-scan groups [done, 4) of trip c2 - 1 ----
          // One hand-over call site, in a loop (a second call site after a re-scan made ptxas fail
          // register allocation).  Every group re-reads its 16-column chunk into rb and ra (the
          // prefetched first chunk of the next trip) is fetched again afterwards, so no tcgen05.ld
          // result is live across the call.
          {
            const uint32_t ta = taddr + (c2 - 1) * 32;
            const int cb = col0 + (c2 - 1) * 32;
            int g = done;
            bool over = true;
            while (over) {
              handoff();
              over = false;
#pragma unroll 1
              while (g < 4 && !over) {
                tmem_ld16(ta + (g >> 1) * 16, rb);
                tmem_ld_wait16(rb);
                if (g & 1) scan8(rb, 8, cb + (g >> 1) * 16, tau);
                else scan8(rb, 0, cb + (g >> 1) * 16, tau);
                over = __any_sync(0xffffffffu, waddr > wlimit);
                ++g;
              }
            }
          }
          if (c2 >= kBN / 32) break;
          tmem_ld16(taddr + c2 * 32, ra);      // (again) the first chunk of the next trip
          continue;
          if (c2 >= kBN / 32) break;
        }
        tc_fence_before();
        mbar_arrive(&tempty_bar[as]);
      }
      st = scanner_handoff<DBG>(st, (waddr - wbase) / (kBM * 4), 1u, cnt_addr, meta + q, ffull_bar + q,
                                fempty_bar + q, lane, &d_wait_e);
      ++d_hand;
    }
    if (DBG && dbg && lane == 0) {
      unsigned long long* o = dbg + (static_cast<size_t>(blockIdx.x) * 8 + (warp - 4)) * 8;
      o[0] = d_hand; o[1] = d_wait_e; o[2] = d_wait_t; o[3] = clock64() - d_t0;
    }
  } else {
    // ===================== selector =====================
    reg_alloc_inc<232>();
    const int q = warp - 8;
    const int row_in_blk = q * 32 + lane;
    const uint32_t fv0 = smem_u32(fifo) + row_in_blk * 4;
    const uint32_t tau_addr = smem_u32(tau_s) + row_in_blk * 8;
    const uint32_t cnt_addr = smem_u32(cnt_s) + row_in_blk * 2;
    constexpr int N = 2 * kFifo;
    float v[N];          // [0, kFifo): survivors, [kFifo, N): the batch being merged
    uint32_t ix[N];
    uint32_t uses0 = 0, uses1 = 0, b = 0, seq = 0;
    unsigned long long d_wait_f = 0, d_sel = 0, d_t_load = 0, d_t_select = 0, d_t_repack = 0, d_t_reload = 0, d_t_final = 0;
    const long long d_t0 = clock64();
    for (int item = blockIdx.x; item < total_items; item += gridDim.x) {
      const int m_blk = item / nsplit;
      const int sp = item - m_blk * nsplit;
      ++seq;
      float tau = neg_inf;
      int scnt = 0;
#pragma unroll
      for (int s = 0; s < kFifo; ++s) {
        v[s] = neg_inf;
        ix[s] = 0u;
      }
      while (true) {
        {
          const long long t = DBG ? clock64() : 0;
          mbar_wait_backoff(&ffull_bar[b * 4 + q], (b ? uses1 : uses0) & 1u);
          if (DBG) d_wait_f += clock64() - t;
        }
        const uint32_t base = fv0 + b * kFifoBytes;
        unsigned short n16;
        asm volatile("ld.shared.u16 %0, [%1];" : "=h"(n16) : "r"(cnt_addr + b * (kBM * 2)) : "memory");
        const int n = static_cast<int>(n16);
        const uint32_t last = meta[b * 4 + q];
        long long tt0 = DBG ? clock64() : 0;
#pragma unroll
        for (int s = 0; s < kFifo; ++s) {
          const float x = lds_f32(base + s * (kBM * 4));
          v[kFifo + s] = (s < n) ? x : neg_inf;
          ix[kFifo + s] = lds_u32(base + s * (kBM * 4) + kFifoIdxOff);
        }
        if (DBG) { const long long t = clock64(); d_t_load += t - tt0; tt0 = t; }
        const int total = scnt + n;
        float thr = neg_inf;
        bool ties = false;
        int tie_left = 0;
        // the item's last batch is reduced to EXACTLY k (slack 0; ties keep the lowest feature
        // index), so the survivors re-read below are the result - no separate finalisation pass
        const int slack = last ? 0 : kSlack;
        if (__any_sync(0xffffffffu, total > k + slack)) {
          thr = select_threshold<N>(v, total, k, slack, tau, ties, tie_left);
          ++d_sel;
        }
        if (DBG) { const long long t = clock64(); d_t_select += t - tt0; tt0 = t; }
        // repack the survivors (old ones first: ascending feature index) through the drained FIFO
        uint32_t w = base;
        if (!__any_sync(0xffffffffu, ties)) {
#pragma unroll
          for (int s = 0; s < N; s += 4)
            w = append4<kFifoIdxOff>(w, thr, v[s], v[s + 1], v[s + 2], v[s + 3], ix[s], ix[s + 1],
                                     ix[s + 2], ix[s + 3], slot);
        } else {
#pragma unroll
          for (int s = 0; s < N; ++s) {
            const bool tie = ties && (v[s] == thr) && tie_left > 0;
            tie_left -= tie ? 1 : 0;
            if (v[s] > thr || tie) {
              asm volatile("st.shared.f32 [%0], %1;\n\tst.shared.u32 [%0+%3], %2;" ::"r"(w), "f"(v[s]),
                           "r"(ix[s]), "n"(kFifoIdxOff)
                           : "memory");
              w += kBM * 4;
            }
          }
        }
        scnt = static_cast<int>((w - base) / (kBM * 4));
        if (DBG) { const long long t = clock64(); d_t_repack += t - tt0; tt0 = t; }
#pragma unroll
        for (int s = 0; s < kFifo; ++s) {
          const float x = lds_f32(base + s * (kBM * 4));
          v[s] = (s < scnt) ? x : neg_inf;
          ix[s] = lds_u32(base + s * (kBM * 4) + kFifoIdxOff);
        }
        if (DBG) { const long long t = clock64(); d_t_reload += t - tt0; tt0 = t; }
        if (thr > tau) {
          tau = thr;
          asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(tau_addr), "r"(__float_as_uint(tau)),
                       "r"(seq)
                       : "memory");
        }
        mbar_arrive(&fempty_bar[b * 4 + q]);
        if (b) ++uses1; else ++uses0;
        b ^= 1u;
        if (last) break;
      }
      // ---- write the row's k (value, index) pairs: v[0 .. scnt) in ascending feature index ----
      const long long tf0 = DBG ? clock64() : 0;
      const int row = m_blk * kBM + row_in_blk;
      if (row < B) {
        float* ov = out_val + (static_cast<size_t>(row) * nsplit + sp) * k;
        int32_t* oi = out_idx + (static_cast<size_t>(row) * nsplit + sp) * k;
        if ((k & 3) == 0) {          // 16-byte stores (rows of k * 4 bytes stay 16-byte aligned)
#pragma unroll
          for (int s = 0; s < 32; s += 4) {
            if (s < k) {
              // fewer than k candidates (split narrower than k, NaN rows): pad with (-inf, -1)
              const int4 iv = make_int4(s < scnt ? static_cast<int>(ix[s]) : -1,
                                        s + 1 < scnt ? static_cast<int>(ix[s + 1]) : -1,
                                        s + 2 < scnt ? static_cast<int>(ix[s + 2]) : -1,
                                        s + 3 < scnt ? static_cast<int>(ix[s + 3]) : -1);
              *reinterpret_cast<float4*>(ov + s) = make_float4(v[s], v[s + 1], v[s + 2], v[s + 3]);
              *reinterpret_cast<int4*>(oi + s) = iv;
            }
          }
        } else {
#pragma unroll
          for (int s = 0; s < 32; ++s) {
            if (s < k) {
              ov[s] = v[s];
              oi[s] = s < scnt ? static_cast<int32_t>(ix[s]) : -1;
            }
          }
        }
      }
      if (DBG) d_t_final += clock64() - tf0;
    }
    if (DBG && dbg && lane == 0) {
      unsigned long long* o = dbg + (static_cast<size_t>(blockIdx.x) * 8 + (warp - 4)) * 8;
      o[0] = d_sel; o[1] = d_wait_f; o[3] = clock64() - d_t0;
      o[2] = d_t_load; o[4] = d_t_select; o[5] = d_t_repack; o[6] = d_t_reload; o[7] = d_t_final;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ================================================================================================
// K1, CTA-PAIR form (cta_group::2): the same scanner / selector epilogue, but the two CTAs of a
// 2-CTA cluster (two SMs of one TPC) run ONE 256 x 256 x 16 tcgen05.mma per K step over 256
// activation rows.  Each CTA stages its own 128 A' rows and only HALF of the W' tile (128 of the 256
// feature rows); the tensor cores read the other half out of the peer's shared memory.  The
// single-CTA main loop moves 48 KB in and 48 KB out of shared memory per 64-wide K block against 512
// cycles of MMA (96 KB at 128 B/cycle = 768 cycles: shared-memory bound, 86 % of it measured); here a
// CTA moves 32 KB in and reads 32 KB - 512 cycles, level with the MMA.  A stage shrinks from 48 to
// 32 KB.  Protocol (CUTLASS sm100 2-SM pipeline): both CTAs' TMA copies complete on the LEADER's
// (rank 0) full barrier (.cta_group::2, peer bit of the barrier address cleared); the leader's MMA
// warp issues tcgen05.mma.cta_group::2 and multicasts its commits to both CTAs' empty / tfull
// barriers; the scanner threads of both CTAs arrive on the leader's tempty barrier (256 arrivals).
// ================================================================================================
constexpr int kBHalfStage = (kBN / 2) * kBK * 2;     // 16 KB: this CTA's half of a W' tile
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;       // shared::cluster address -> same offset in the even CTA

constexpr int kPairFifoBufs = 2;                     // scanner -> selector FIFO ring depth of the pair kernel (3 buffers + 3 stages measured slower: 240 vs 221 us at 384->3072, 3374 vs 2610 us at 1280->40960)

template <int STAGES>
struct Encode3Smem {
  static constexpr int kPipeBytes = STAGES * (kAStage + kBHalfStage);
  static constexpr int kFifoTotal = 2 * kPairFifoBufs * kFifoBytes;     // NB buffers x (val + idx)
  static constexpr int kTauBytes = kBM * 8;
  static constexpr int kCntBytes = kPairFifoBufs * kBM * 2;
  static constexpr int kBarBytes = 512;
  static_assert((2 * STAGES + 20) * 8 + 8 + 32 <= kBarBytes, "barrier block too small");
  static constexpr int kTotal = kPipeBytes + kFifoTotal + kTauBytes + kCntBytes + kBarBytes + 1024;
  static_assert(kTotal <= 232448, "exceeds the 227 KB shared-memory limit");
};

// scanner_handoff for a ring of NB FIFO buffers.  st: bits 0-1 = buffer in use, bit 2 + i = parity of
// the number of fills of buffer i.
template <bool DBG, int NB>
__device__ __noinline__ uint32_t scanner_handoff_ring(uint32_t st, uint32_t nslots, uint32_t last,
                                                      uint32_t cnt_addr, uint32_t* meta_q,
                                                      uint64_t* ffull_q, uint64_t* fempty_q, int lane,
                                                      unsigned long long* waited) {
  const uint32_t b = st & 3u;
  asm volatile("st.shared.u16 [%0], %1;" ::"r"(cnt_addr + b * (kBM * 2)),
               "h"(static_cast<unsigned short>(nslots))
               : "memory");
  if (lane == 0) meta_q[b * 4] = last;
  mbar_arrive(&ffull_q[b * 4]);
  const uint32_t nb = (b + 1 == NB) ? 0u : b + 1;
  st = ((st ^ (4u << b)) & ~3u) | nb;      // one more fill of buffer b; continue on the next buffer
  if (!last) {
    const long long t = DBG ? clock64() : 0;
    mbar_wait_backoff(&fempty_q[nb * 4], ((st >> (2u + nb)) & 1u) ^ 1u);
    if (DBG) *waited += clock64() - t;
  }
  return st;
}

__device__ __forceinline__ void tma_load_2d_2sm(void* smem_dst, const void* tmap, uint64_t* bar,
                                                int32_t c_inner, int32_t c_outer) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c_inner), "r"(c_outer)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                              uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// completion of all MMAs issued so far -> the barrier at this offset in BOTH CTAs of the pair
__device__ __forceinline__ void umma_commit_2sm(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(static_cast<uint16_t>(3))
      : "memory");
}
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & kPeerBitMask) : "memory");
}
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t* smem_slot, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_2sm() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

template <int STAGES, bool DBG>
__global__ void __launch_bounds__(384, 1)
encode_topk3_kernel(const __grid_constant__ CUtensorMap tmap_a,
                    const __grid_constant__ CUtensorMap tmap_w, int B, int F, int k, int ksteps,
                    int num_m_blocks, int num_n_tiles, int nsplit, int tiles_per_split,
                    float* __restrict__ out_val, int32_t* __restrict__ out_idx,
                    unsigned long long* __restrict__ dbg, int mode, uint32_t slot) {
  using SM = Encode3Smem<STAGES>;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* pipe = smem;
  uint8_t* fifo = smem + SM::kPipeBytes;
  uint8_t* tau_s = fifo + SM::kFifoTotal;
  uint8_t* cnt_s = tau_s + SM::kTauBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(cnt_s + SM::kCntBytes);
  uint64_t* full_bar = bars;                        // [STAGES]
  uint64_t* empty_bar = bars + STAGES;              // [STAGES]
  uint64_t* tfull_bar = bars + 2 * STAGES;          // [2]
  uint64_t* tempty_bar = bars + 2 * STAGES + 2;     // [2]
  constexpr int NB = kPairFifoBufs;                 // FIFO ring depth (3: the W' half-stages free the room)
  constexpr int kIdxOff = NB * kFifoBytes;          // the index arrays sit behind all value buffers
  uint64_t* ffull_bar = bars + 2 * STAGES + 4;             // [NB buffers][4 quarters]
  uint64_t* fempty_bar = bars + 2 * STAGES + 4 + 4 * NB;   // [NB][4]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4 + 8 * NB);
  uint32_t* meta = tmem_slot + 2;                   // [NB][4]: 1 = last hand-over of the work item

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_kb = ceil_div(ksteps, kBK / 16);
  // work items are PAIRS of 128-row blocks: CTA rank r of the cluster owns block 2 * pair + r; the
  // persistent loop strides over pair-items by the number of clusters
  const uint32_t crank = cluster_ctarank();
  const int cluster_id = blockIdx.x >> 1;
  const int n_clusters = gridDim.x >> 1;
  const int total_items = ((num_m_blocks + 1) >> 1) * nsplit;
  const float neg_inf = __uint_as_float(0xff800000u);

  pdl_launch_dependents();
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_w);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull_bar[s], 1);
      mbar_init(&tempty_bar[s], 2 * kBM);     // leader's: the scanner threads of BOTH CTAs arrive
    }
    for (int s = 0; s < 4 * NB; ++s) {
      mbar_init(&ffull_bar[s], 32);
      mbar_init(&fempty_bar[s], 32);
    }
    mbar_fence_init();
  }
  if (warp == 2) {
    tmem_alloc_2sm(tmem_slot, 512);
    tmem_relinquish_2sm();
  }
  for (int i = threadIdx.x; i < kBM * 2; i += blockDim.x) reinterpret_cast<uint32_t*>(tau_s)[i] = 0u;
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();      // the peer's barriers are initialised before anything signals them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();   // set-up done under the predecessor's tail; global memory (TMA, results) from here on

  if (warp < 4) {
    reg_alloc_dec<56>();
    if (warp == 0) {
      // ===================== TMA producer (both CTAs): own A rows + own half of the W' tile =====================
      if (elect_one()) {
        int stage = 0;
        uint32_t phase = 0;
        for (int item = cluster_id; item < total_items; item += n_clusters) {
          const int pair = item / nsplit;
          const int sp = item - pair * nsplit;
          const int m_blk = 2 * pair + static_cast<int>(crank);
          const int t0 = sp * tiles_per_split;
          const int t1 = min(t0 + tiles_per_split, num_n_tiles);
          for (int nt = t0; nt < t1; ++nt) {
            for (int kb = 0; kb < num_kb; ++kb) {
              mbar_wait_sleep<kRoleSleepNs>(&empty_bar[stage], phase ^ 1u);
              // the leader's full barrier collects the bytes of both CTAs' copies
              if (crank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * (kAStage + kBHalfStage));
              uint8_t* sa = pipe + stage * (kAStage + kBHalfStage);
              tma_load_2d_2sm(sa, &tmap_a, &full_bar[stage], kb * kBK, m_blk * kBM);
              tma_load_2d_2sm(sa + kAStage, &tmap_w, &full_bar[stage], kb * kBK,
                              nt * kBN + static_cast<int>(crank) * (kBN / 2));
              if (++stage == STAGES) {
                stage = 0;
                phase ^= 1u;
              }
            }
          }
        }
      }
    } else if (warp == 1 && crank == 0) {
      // ===================== MMA issuer (leader CTA only): 256 x 256 x 16 across the CTA pair =====================
      constexpr uint32_t idesc = umma_idesc_bf16(2 * kBM, kBN);
      int stage = 0;
      uint32_t phase = 0, tile = 0;
      for (int item = cluster_id; item < total_items; item += n_clusters) {
        const int sp = item - (item / nsplit) * nsplit;
        const int t0 = sp * tiles_per_split;
        const int t1 = min(t0 + tiles_per_split, num_n_tiles);
        for (int nt = t0; nt < t1; ++nt, ++tile) {
          const uint32_t as = tile & 1u;
          const uint32_t aphase = (tile >> 1) & 1u;
          mbar_wait_sleep<kRoleSleepNs>(&tempty_bar[as], aphase ^ 1u);
          tc_fence_after();
          const uint32_t tmem_d = tmem_base + as * kBN;
          for (int kb = 0; kb < num_kb; ++kb) {
            mbar_wait_sleep<kRoleSleepNs>(&full_bar[stage], phase);
            tc_fence_after();
            if (elect_one()) {
              const uint32_t sa = smem_u32(pipe + stage * (kAStage + kBHalfStage));
              const uint64_t da = umma_desc_sw128_kmajor(sa);
              const uint64_t db = umma_desc_sw128_kmajor(sa + kAStage);
              const int nks = min(kBK / 16, ksteps - kb * (kBK / 16));
              for (int ks = 0; ks < nks; ++ks)
                umma_bf16_2sm(tmem_d, da + static_cast<uint64_t>(2 * ks), db + static_cast<uint64_t>(2 * ks),
                              idesc, (kb | ks) != 0 ? 1u : 0u);
              umma_commit_2sm(&empty_bar[stage]);                      // both CTAs' producers
              if (kb == num_kb - 1) umma_commit_2sm(&tfull_bar[as]);   // both CTAs' scanners
            }
            __syncwarp();
            if (++stage == STAGES) {
              stage = 0;
              phase ^= 1u;
            }
          }
        }
      }
    }
  } else if (warp < 8) {
    // ===================== scanner =====================
    reg_alloc_dec<152>();
    const int q = warp - 4;
    const int row_in_blk = q * 32 + lane;
    const uint32_t fv0 = smem_u32(fifo) + row_in_blk * 4;          // buffer 0, slot 0 of this row
    const uint32_t tau_addr = smem_u32(tau_s) + row_in_blk * 8;
    const uint32_t cnt_addr = smem_u32(cnt_s) + row_in_blk * 2;
    uint32_t st = 0, seq = 0, tile = 0;      // st: bit 0 = FIFO buffer in use, bits 1/2 = fill parities
    unsigned long long d_hand = 0, d_wait_e = 0, d_wait_t = 0;
    const long long d_t0 = clock64();
    for (int item = cluster_id; item < total_items; item += n_clusters) {
      const int sp = item - (item / nsplit) * nsplit;
      const int t0 = sp * tiles_per_split;
      const int t1 = min(t0 + tiles_per_split, num_n_tiles);
      ++seq;
      // mode 3 (experiments): nothing passes the filter - times the GEMM pipeline + bare scan
      float tau = (DBG && mode >= 3) ? __uint_as_float(0x7f800000u) : neg_inf;
      mbar_wait_backoff(&fempty_bar[(st & 3u) * 4 + q], ((st >> (2u + (st & 3u))) & 1u) ^ 1u);
      uint32_t wbase = fv0 + (st & 3u) * kFifoBytes;
      uint32_t waddr = wbase;
      uint32_t wlimit = wbase + (kFifo - kCheck) * (kBM * 4);

      for (int nt = t0; nt < t1; ++nt, ++tile) {
        const uint32_t as = tile & 1u;
        const uint32_t aphase = (tile >> 1) & 1u;
        {
          const long long t = DBG ? clock64() : 0;
          mbar_wait(&tfull_bar[as], aphase);
          if (DBG) d_wait_t += clock64() - t;
        }
        tc_fence_after();
        const int col0 = nt * kBN;
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * kBN;

        // ---- first tile of a work item: a floor for the row's threshold before anything is scanned ----
        // The tile's 256 columns form 32 groups of 8; the smallest of the 32 group maxima has at
        // least 32 >= k values at or above it, so the row's k-th largest value cannot be below it.
        // Starting from (just under) that floor instead of -inf, the first tile passes ~40 % of
        // its values instead of all of the first ~120 columns: about two hand-overs fewer per item,
        // in the part of the item where the selector is the bottleneck.  Costs one extra read of
        // the tile (16 tcgen05.ld) and ~0.6 instructions per value while the selector is idle.
        // A group of 8 NaN columns has no maximum: fmin_nan turns the floor into NaN, and padding
        // columns (-inf) turn it into -inf; either leaves tau at -inf.  (k <= 32 here.)
        if (nt == t0 && !(DBG && mode >= 3)) {
          float floor_v = __uint_as_float(0x7f800000u);
          uint32_t rp[16];
#pragma unroll 1
          for (int c = 0; c < kBN; c += 16) {
            tmem_ld16(taddr + c, rp);
            tmem_ld_wait16(rp);
            const float m0 = fmaxf(fmaxf(fmaxf(__uint_as_float(rp[0]), __uint_as_float(rp[1])),
                                         fmaxf(__uint_as_float(rp[2]), __uint_as_float(rp[3]))),
                                   fmaxf(fmaxf(__uint_as_float(rp[4]), __uint_as_float(rp[5])),
                                         fmaxf(__uint_as_float(rp[6]), __uint_as_float(rp[7]))));
            const float m1 = fmaxf(fmaxf(fmaxf(__uint_as_float(rp[8]), __uint_as_float(rp[9])),
                                         fmaxf(__uint_as_float(rp[10]), __uint_as_float(rp[11]))),
                                   fmaxf(fmaxf(__uint_as_float(rp[12]), __uint_as_float(rp[13])),
                                         fmaxf(__uint_as_float(rp[14]), __uint_as_float(rp[15]))));
            floor_v = fmin_nan(floor_v, fmin_nan(m0, m1));
          }
          tau = floor_threshold(floor_v, tau);
        }

        // ---- scan of one 128x256 accumulator tile, 32 columns (two tcgen05.ld.x16) per trip ----
        // A taken branch costs a lone warp ~45-60 cycles (instruction-fetch bubble) and ptxas lays a
        // rare `if (overflow) handoff();` block inline, i.e. the COMMON path takes a skip-branch at
        // every overflow check - four per trip, a third of the scan time.  So the hot trip has no
        // branch at all: an overflow check only folds its vote into `need`, and from then on the
        // filter is closed (threshold +inf) for the rest of the trip.  The single branch per trip is
        // the loop back-edge, which also tests `need`; when it falls through, the cold code below
        // hands the FIFO over and re-scans the groups of that trip that ran with the filter closed.
        auto scan8 = [&](const uint32_t (&r)[16], int j0, int cbase, float thr) {
          const uint32_t c = static_cast<uint32_t>(cbase + j0);
          waddr = append4<kIdxOff>(waddr, thr, __uint_as_float(r[j0]), __uint_as_float(r[j0 + 1]),
                                       __uint_as_float(r[j0 + 2]), __uint_as_float(r[j0 + 3]), c, c + 1,
                                       c + 2, c + 3, slot);
          waddr = append4<kIdxOff>(waddr, thr, __uint_as_float(r[j0 + 4]), __uint_as_float(r[j0 + 5]),
                                       __uint_as_float(r[j0 + 6]), __uint_as_float(r[j0 + 7]), c + 4,
                                       c + 5, c + 6, c + 7, slot);
        };
        auto handoff = [&]() {
          st = scanner_handoff_ring<DBG, NB>(st, (waddr - wbase) / (kBM * 4), 0u, cnt_addr, meta + q,
                                             ffull_bar + q, fempty_bar + q, lane, &d_wait_e);
          ++d_hand;
          wbase = fv0 + (st & 3u) * kFifoBytes;
          waddr = wbase;
          wlimit = wbase + (kFifo - kCheck) * (kBM * 4);
        };
        const float pos_inf = __uint_as_float(0x7f800000u);
        uint32_t ra[16], rb[16];
        tmem_ld16(taddr, ra);
        int c2 = 0;
        while (true) {
          bool need = false;
          int done = 0;            // groups of 8 columns of the current trip scanned with the filter open
#pragma unroll 1
          do {
            const uint32_t ta = taddr + c2 * 32;
            const int cb = col0 + c2 * 32;
            uint32_t tb, tq;   // the selector's latest threshold for this row (valid for this item only)
            asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(tb), "=r"(tq) : "r"(tau_addr) : "memory");
            tmem_ld_wait16(ra);
            tmem_ld16(ta + 16, rb);
            if (tq == seq) tau = fmaxf(tau, __uint_as_float(tb));
            float thr = tau;
            done = 0;
            if (DBG && mode == 4) {        // experiments: TMEM reads only (one compare keeps the loads live)
              if (__uint_as_float(ra[0]) == tau) waddr += 4;
              tmem_ld_wait16(rb);
              if (c2 + 1 < kBN / 32) tmem_ld16(ta + 32, ra);
              if (__uint_as_float(rb[0]) == tau) waddr += 4;
            } else {
              scan8(ra, 0, cb, thr);
              done += need ? 0 : 1;
              need = need | __any_sync(0xffffffffu, waddr > wlimit);
              thr = need ? pos_inf : thr;
              scan8(ra, 8, cb, thr);
              done += need ? 0 : 1;
              need = need | __any_sync(0xffffffffu, waddr > wlimit);
              thr = need ? pos_inf : thr;
              tmem_ld_wait16(rb);
              if (c2 + 1 < kBN / 32) tmem_ld16(ta + 32, ra);
              scan8(rb, 0, cb + 16, thr);
              done += need ? 0 : 1;
              need = need | __any_sync(0xffffffffu, waddr > wlimit);
              thr = need ? pos_inf : thr;
              scan8(rb, 8, cb + 16, thr);
              done += need ? 0 : 1;
              need = need | __any_sync(0xffffffffu, waddr > wlimit);
            }
            ++c2;
          } while (!need && c2 < kBN / 32);
          if (!need) break;                                  // tile scanned
          // ---- cold path: hand the FIFO over, re-scan groups [done, 4) of trip c2 - 1 ----
          // One hand-over call site, in a loop (a second call site after a re-scan made ptxas fail
          // register allocation).  Every group re-reads its 16-column chunk into rb and ra (the
          // prefetched first chunk of the next trip) is fetched again afterwards, so no tcgen05.ld
          // result is live across the call.
          {
            const uint32_t ta = taddr + (c2 - 1) * 32;
            const int cb = col0 + (c2 - 1) * 32;
            int g = done;
            bool over = true;
            while (over) {
              handoff();
              over = false;
#pragma unroll 1
              while (g < 4 && !over) {
                tmem_ld16(ta + (g >> 1) * 16, rb);
                tmem_ld_wait16(rb);
                if (g & 1) scan8(rb, 8, cb + (g >> 1) * 16, tau);
                else scan8(rb, 0, cb + (g >> 1) * 16, tau);
                over = __any_sync(0xffffffffu, waddr > wlimit);
                ++g;
              }
            }
          }
          if (c2 >= kBN / 32) break;
          tmem_ld16(taddr + c2 * 32, ra);      // (again) the first chunk of the next trip
          continue;
          if (c2 >= kBN / 32) break;
        }
        tc_fence_before();
        mbar_arrive_leader(&tempty_bar[as]);     // the leader CTA's MMA warp owns the accumulators of both
      }
      st = scanner_handoff_ring<DBG, NB>(st, (waddr - wbase) / (kBM * 4), 1u, cnt_addr, meta + q, ffull_bar + q,
                                         fempty_bar + q, lane, &d_wait_e);
      ++d_hand;
    }
    if (DBG && dbg && lane == 0) {
      unsigned long long* o = dbg + (static_cast<size_t>(blockIdx.x) * 8 + (warp - 4)) * 8;
      o[0] = d_hand; o[1] = d_wait_e; o[2] = d_wait_t; o[3] = clock64() - d_t0;
    }
  } else {
    // ===================== selector =====================
    reg_alloc_inc<232>();
    const int q = warp - 8;
    const int row_in_blk = q * 32 + lane;
    const uint32_t fv0 = smem_u32(fifo) + row_in_blk * 4;
    const uint32_t tau_addr = smem_u32(tau_s) + row_in_blk * 8;
    const uint32_t cnt_addr = smem_u32(cnt_s) + row_in_blk * 2;
    constexpr int N = 2 * kFifo;
    float v[N];          // [0, kFifo): survivors, [kFifo, N): the batch being merged
    uint32_t ix[N];
    uint32_t uses = 0, b = 0, seq = 0;      // uses: bit i = parity of the number of drains of buffer i
    unsigned long long d_wait_f = 0, d_sel = 0, d_t_load = 0, d_t_select = 0, d_t_repack = 0, d_t_reload = 0, d_t_final = 0;
    const long long d_t0 = clock64();
    for (int item = cluster_id; item < total_items; item += n_clusters) {
      const int m_blk = 2 * (item / nsplit) + static_cast<int>(crank);
      const int sp = item - (item / nsplit) * nsplit;
      ++seq;
      float tau = neg_inf;
      int scnt = 0;
#pragma unroll
      for (int s = 0; s < kFifo; ++s) {
        v[s] = neg_inf;
        ix[s] = 0u;
      }
      while (true) {
        {
          const long long t = DBG ? clock64() : 0;
          mbar_wait_backoff(&ffull_bar[b * 4 + q], (uses >> b) & 1u);
          if (DBG) d_wait_f += clock64() - t;
        }
        const uint32_t base = fv0 + b * kFifoBytes;
        unsigned short n16;
        asm volatile("ld.shared.u16 %0, [%1];" : "=h"(n16) : "r"(cnt_addr + b * (kBM * 2)) : "memory");
        const int n = static_cast<int>(n16);
        const uint32_t last = meta[b * 4 + q];
        long long tt0 = DBG ? clock64() : 0;
#pragma unroll
        for (int s = 0; s < kFifo; ++s) {
          const float x = lds_f32(base + s * (kBM * 4));
          v[kFifo + s] = (s < n) ? x : neg_inf;
          ix[kFifo + s] = lds_u32(base + s * (kBM * 4) + kIdxOff);
        }
        if (DBG) { const long long t = clock64(); d_t_load += t - tt0; tt0 = t; }
        const int total = scnt + n;
        float thr = neg_inf;
        bool ties = false;
        int tie_left = 0;
        // the item's last batch is reduced to EXACTLY k (slack 0; ties keep the lowest feature
        // index), so the survivors re-read below are the result - no separate finalisation pass
        const int slack = last ? 0 : kSlack;
        if (__any_sync(0xffffffffu, total > k + slack)) {
          thr = select_threshold<N>(v, total, k, slack, tau, ties, tie_left);
          ++d_sel;
        }
        if (DBG) { const long long t = clock64(); d_t_select += t - tt0; tt0 = t; }
        // repack the survivors (old ones first: ascending feature index) through the drained FIFO
        uint32_t w = base;
        if (!__any_sync(0xffffffffu, ties)) {
#pragma unroll
          for (int s = 0; s < N; s += 4)
            w = append4<kIdxOff>(w, thr, v[s], v[s + 1], v[s + 2], v[s + 3], ix[s], ix[s + 1],
                                     ix[s + 2], ix[s + 3], slot);
        } else {
#pragma unroll
          for (int s = 0; s < N; ++s) {
            const bool tie = ties && (v[s] == thr) && tie_left > 0;
            tie_left -= tie ? 1 : 0;
            if (v[s] > thr || tie) {
              asm volatile("st.shared.f32 [%0], %1;\n\tst.shared.u32 [%0+%3], %2;" ::"r"(w), "f"(v[s]),
                           "r"(ix[s]), "n"(kIdxOff)
                           : "memory");
              w += kBM * 4;
            }
          }
        }
        scnt = static_cast<int>((w - base) / (kBM * 4));
        if (DBG) { const long long t = clock64(); d_t_repack += t - tt0; tt0 = t; }
#pragma unroll
        for (int s = 0; s < kFifo; ++s) {
          const float x = lds_f32(base + s * (kBM * 4));
          v[s] = (s < scnt) ? x : neg_inf;
          ix[s] = lds_u32(base + s * (kBM * 4) + kIdxOff);
        }
        if (DBG) { const long long t = clock64(); d_t_reload += t - tt0; tt0 = t; }
        if (thr > tau) {
          tau = thr;
          asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(tau_addr), "r"(__float_as_uint(tau)),
                       "r"(seq)
                       : "memory");
        }
        mbar_arrive(&fempty_bar[b * 4 + q]);
        uses ^= 1u << b;
        b = (b + 1 == NB) ? 0u : b + 1;
        if (last) break;
      }
      // ---- write the row's k (value, index) pairs: v[0 .. scnt) in ascending feature index ----
      const long long tf0 = DBG ? clock64() : 0;
      const int row = m_blk * kBM + row_in_blk;
      if (row < B) {
        float* ov = out_val + (static_cast<size_t>(row) * nsplit + sp) * k;
        int32_t* oi = out_idx + (static_cast<size_t>(row) * nsplit + sp) * k;
        if ((k & 3) == 0) {          // 16-byte stores (rows of k * 4 bytes stay 16-byte aligned)
#pragma unroll
          for (int s = 0; s < 32; s += 4) {
            if (s < k) {
              // fewer than k candidates (split narrower than k, NaN rows): pad with (-inf, -1)
              const int4 iv = make_int4(s < scnt ? static_cast<int>(ix[s]) : -1,
                                        s + 1 < scnt ? static_cast<int>(ix[s + 1]) : -1,
                                        s + 2 < scnt ? static_cast<int>(ix[s + 2]) : -1,
                                        s + 3 < scnt ? static_cast<int>(ix[s + 3]) : -1);
              *reinterpret_cast<float4*>(ov + s) = make_float4(v[s], v[s + 1], v[s + 2], v[s + 3]);
              *reinterpret_cast<int4*>(oi + s) = iv;
            }
          }
        } else {
#pragma unroll
          for (int s = 0; s < 32; ++s) {
            if (s < k) {
              ov[s] = v[s];
              oi[s] = s < scnt ? static_cast<int32_t>(ix[s]) : -1;
            }
          }
        }
      }
      if (DBG) d_t_final += clock64() - tf0;
    }
    if (DBG && dbg && lane == 0) {
      unsigned long long* o = dbg + (static_cast<size_t>(blockIdx.x) * 8 + (warp - 4)) * 8;
      o[0] = d_sel; o[1] = d_wait_f; o[3] = clock64() - d_t0;
      o[2] = d_t_load; o[4] = d_t_select; o[5] = d_t_repack; o[6] = d_t_reload; o[7] = d_t_final;
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();      // no CTA leaves (or frees TMEM) while its peer may still signal / use it
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc_2sm(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------------------------
// Merge of per-split partial top-k lists: part_[B, nsplit*k] -> out_[B, k].  One warp per row.
// Candidate order (split, slot) is ascending feature index, so "first tie wins" = lowest index.
// ------------------------------------------------------------------------------------------------
constexpr int kMergeMaxPerLane = 64;

// PER = candidates per lane (ceil(n / 32) rounded up to an instantiated size): the loops are fully
// unrolled over registers, so a small merge (12 splits x 32) does not pay for the 64-wide worst case.
template <int PER>
__global__ void __launch_bounds__(256)
topk_merge_kernel(const float* __restrict__ part_val, const int32_t* __restrict__ part_idx, int B,
                  int n, int k, float* __restrict__ out_val, int32_t* __restrict__ out_idx) {
  pdl_prologue();
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= B) return;
  const float* pv = part_val + static_cast<size_t>(row) * n;
  const int32_t* pi = part_idx + static_cast<size_t>(row) * n;
  const int per = ceil_div(n, 32);  // <= kMergeMaxPerLane (checked on the host)
  uint32_t key[PER];
  uint32_t hi = 0, kmin = 0xFFFFFFFFu;
#pragma unroll
  for (int t = 0; t < PER; ++t) {
    const int p = t * 32 + lane;
    uint32_t kk = 0;
    if (t < per && p < n && pi[p] >= 0) kk = f2key(pv[p]);
    key[t] = kk;
    hi = max(hi, kk);
    kmin = min(kmin, kk ? kk : 0xFFFFFFFFu);
  }
  hi = __reduce_max_sync(0xffffffffu, hi);
  kmin = __reduce_min_sync(0xffffffffu, kmin);
  // bracket: count(key > lo) >= k, count(key > hi) < k.  lo starts just below the smallest valid key
  // (the keys of one row cluster in a narrow band: starting at 1 wasted ~8 halvings) unless fewer
  // than k candidates exist, in which case everything is kept.
  uint32_t lo = (kmin != 0xFFFFFFFFu && kmin > 1u) ? kmin - 1u : 1u;
  bool exact = false;
  while (hi - lo > 1u) {
    const uint32_t mid = lo + ((hi - lo) >> 1);
    int c0 = 0, c1 = 0, c2 = 0, c3 = 0;       // four independent counters, one warp-wide REDUX
#pragma unroll
    for (int t = 0; t < PER; t += 4) {
      c0 += (key[t] > mid) ? 1 : 0;
      if (t + 1 < PER) c1 += (key[t + 1] > mid) ? 1 : 0;
      if (t + 2 < PER) c2 += (key[t + 2] > mid) ? 1 : 0;
      if (t + 3 < PER) c3 += (key[t + 3] > mid) ? 1 : 0;
    }
    const int c = __reduce_add_sync(0xffffffffu, (c0 + c1) + (c2 + c3));
    const bool ge = c >= k;
    lo = ge ? mid : lo;
    hi = ge ? hi : mid;
    if (c == k) {
      exact = true;
      break;
    }
  }
  uint32_t thr = lo, tie_key = 0xFFFFFFFFu;
  int tie_left = 0;
  if (!exact) {
    int m = 0;
#pragma unroll
    for (int t = 0; t < PER; ++t) m += (key[t] > hi) ? 1 : 0;
    m = __reduce_add_sync(0xffffffffu, m);
    thr = hi;
    tie_key = hi;
    tie_left = k - m;
  }
  int base = 0;
  const uint32_t below = (1u << lane) - 1u;
#pragma unroll
  for (int t = 0; t < PER; ++t) {
    if (t >= per) break;
    const uint32_t kk = key[t];
    const bool gt = kk > thr;
    const bool tie = (kk == tie_key);
    const uint32_t tie_mask = __ballot_sync(0xffffffffu, tie);
    const bool keep = gt || (tie && (__popc(tie_mask & below) < tie_left));
    tie_left -= __popc(tie_mask);
    const uint32_t keep_mask = __ballot_sync(0xffffffffu, keep);
    if (keep) {
      const int slot = base + __popc(keep_mask & below);
      if (slot < k) {
        const int p = t * 32 + lane;
        out_val[static_cast<size_t>(row) * k + slot] = pv[p];
        out_idx[static_cast<size_t>(row) * k + slot] = pi[p];
      }
    }
    base += __popc(keep_mask);
  }
  // fewer than k valid candidates (NaN rows): pad with (-inf, -1) as the unmerged lists are
  for (int slot = base + lane; slot < k; slot += 32) {
    out_val[static_cast<size_t>(row) * k + slot] = __uint_as_float(0xff800000u);
    out_idx[static_cast<size_t>(row) * k + slot] = -1;
  }
}

// ================================================================================================
// K1 for SMALL batches (the shipped configs/tiny_default.yaml trains on 128 rows): dense
// pre-activations + one block per row.
//
// With fewer 128-row blocks than SMs the fused epilogue is pure latency: one work item at B = 128 is
// TMA -> 7 k-blocks of MMA -> scan of 256 columns with ~3 hand-overs/selections (the row starts at
// threshold -inf) -> write, and the 12 partial lists per row then go through topk_merge_kernel:
// 38-41 us for K1 + merge from 128 to 4096 rows (tools/bench_k1_small.py), 40 % of the 105 us step.
// At these sizes the [B, F] pre-activations are tiny (1.5 MB at 128 x 3072: they stay in L2), so
// here the GEMM simply stores its accumulators (encode_dense_kernel: same TMA / tcgen05 pipeline,
// one 128 x 256 tile per work item, epilogue = tcgen05.ld -> st.global) and rowwise_topk_kernel
// selects each row's k largest with a 4-pass most-significant-digit radix select over the
// order-preserving integer keys in shared memory: exact, ties at the k-th value keep the lowest
// feature index (as the fused epilogue does), output in ascending feature index.
// ================================================================================================
template <int STAGES>
__global__ void __launch_bounds__(256, 1)
encode_dense_kernel(const __grid_constant__ CUtensorMap tmap_a,
                    const __grid_constant__ CUtensorMap tmap_w, int B, int F, int ld, int ksteps,
                    int num_m_blocks, int num_n_tiles, float* __restrict__ pre) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* pipe = smem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * (kAStage + kBStage));
  uint64_t* full_bar = bars;                  // [STAGES]
  uint64_t* empty_bar = bars + STAGES;        // [STAGES]
  uint64_t* tfull_bar = bars + 2 * STAGES;    // [2]
  uint64_t* tempty_bar = bars + 2 * STAGES + 2;  // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_kb = ceil_div(ksteps, kBK / 16);
  const int total_items = num_m_blocks * num_n_tiles;      // one 128 x 256 tile per item
  const EncodeItems items{total_items, num_n_tiles, 1, num_n_tiles, num_kb, ksteps};

  pdl_launch_dependents();
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_w);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull_bar[s], 1);
      mbar_init(&tempty_bar[s], kBM);
    }
    mbar_fence_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();

  if (warp == 0) {
    if (elect_one()) encode_producer_loop<STAGES>(&tmap_a, &tmap_w, pipe, full_bar, empty_bar, items);
  } else if (warp == 1) {
    encode_mma_loop<STAGES>(pipe, full_bar, empty_bar, tfull_bar, tempty_bar, tmem_base, items);
  } else if (warp >= 4) {
    const int q = warp - 4;               // TMEM lane quarter this warp may read
    const int row_in_blk = q * 32 + lane;
    uint32_t tile = 0;
    for (int item = blockIdx.x; item < total_items; item += gridDim.x, ++tile) {
      const int m_blk = item / num_n_tiles;
      const int nt = item - m_blk * num_n_tiles;
      const uint32_t as = tile & 1u;
      const uint32_t aphase = (tile >> 1) & 1u;
      mbar_wait(&tfull_bar[as], aphase);
      tc_fence_after();
      const int row = m_blk * kBM + row_in_blk;
      const int col0 = nt * kBN;
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * kBN;
      float* out = pre + static_cast<size_t>(row < B ? row : 0) * ld + col0;
      uint32_t ra[16], rb[16];
      tmem_ld16(taddr, ra);
#pragma unroll 1
      for (int c = 0; c < kBN; c += 32) {
        tmem_ld_wait16(ra);
        tmem_ld16(taddr + c + 16, rb);
        if (row < B) {
#pragma unroll
          for (int j = 0; j < 16; j += 4)
            if (col0 + c + j + 3 < F) {
              *reinterpret_cast<uint4*>(out + c + j) = make_uint4(ra[j], ra[j + 1], ra[j + 2], ra[j + 3]);
            } else {
#pragma unroll
              for (int e = 0; e < 4; ++e)
                if (col0 + c + j + e < F) out[c + j + e] = __uint_as_float(ra[j + e]);
            }
        }
        tmem_ld_wait16(rb);
        if (c + 32 < kBN) tmem_ld16(taddr + c + 32, ra);
        if (row < B) {
#pragma unroll
          for (int j = 0; j < 16; j += 4)
            if (col0 + c + 16 + j + 3 < F) {
              *reinterpret_cast<uint4*>(out + c + 16 + j) = make_uint4(rb[j], rb[j + 1], rb[j + 2], rb[j + 3]);
            } else {
#pragma unroll
              for (int e = 0; e < 4; ++e)
                if (col0 + c + 16 + j + e < F) out[c + 16 + j + e] = __uint_as_float(rb[j + e]);
            }
        }
      }
      tc_fence_before();
      mbar_arrive(&tempty_bar[as]);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// One block (256 threads) per (row, column slice): the k largest of pre[row, c0 : c0 + S] with
// c0 = blockIdx.y * S (block_row_topk, wsae_rowselect.cuh), written with their feature indices to the
// slice's k slots of the row's gridDim.y * k list.  One slice (S >= F) is the whole row.
__global__ void __launch_bounds__(kRowTopkThreads)
rowwise_topk_kernel(const float* __restrict__ pre, int B, int F, int ld, int S, int k,
                    float* __restrict__ out_val, int32_t* __restrict__ out_idx) {
  extern __shared__ __align__(16) uint32_t s_key[];          // [S]
  __shared__ RowSelectSmem sm;
  pdl_prologue();
  const int row = blockIdx.x;
  if (row >= B) return;
  const int c0 = blockIdx.y * S;
  const size_t o = (static_cast<size_t>(row) * gridDim.y + blockIdx.y) * k;
  block_row_topk(pre + static_cast<size_t>(row) * ld + c0, min(S, F - c0), k, s_key, sm, out_val + o,
                 out_idx + o, c0);
}

// ------------------------------------------------------------------------------------------------
// host side: tensor maps + launch
// ------------------------------------------------------------------------------------------------
static PFN_cuTensorMapEncodeTiled_v12000 get_encode_fn() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess)
      return static_cast<PFN_cuTensorMapEncodeTiled_v12000>(nullptr);
    if (q != cudaDriverEntryPointSuccess) return static_cast<PFN_cuTensorMapEncodeTiled_v12000>(nullptr);
    return reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  }();
  return fn;
}

// [rows, cols] bf16 row-major (row pitch = cols * 2 bytes), box = box_rows x 64, 128B swizzle.
static int make_tmap_bf16(CUtensorMap* out, const void* ptr, uint64_t rows, uint64_t cols,
                          uint32_t box_rows) {
  auto fn = get_encode_fn();
  if (!fn) return kNoDriver;
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {cols * 2};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(kBK), box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), gdim, gstride,
                  box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? kOk : static_cast<int>(1000 + r);
}

// experiments only (wsae_debug_encode_mode): 1 = skip epilogue, 2 = no compaction (both: one-warp
// epilogue kernel), 3 = scanner filter closed (scanner + selector kernel with the counters buffer set)
static int g_encode_dbg = 0;

template <int CAP, int STAGES>
static int launch_encode(const CUtensorMap& ta, const CUtensorMap& tw, int B, int F, int k,
                         int ksteps, int num_m_blocks, int num_n_tiles, int nsplit,
                         int tiles_per_split, float* out_val, int32_t* out_idx, int num_sms,
                         cudaStream_t stream) {
  auto kern = encode_topk_kernel<CAP, STAGES>;
  constexpr int smem = EncodeSmem<CAP, STAGES>::kTotal;
  static bool attr_set[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 64 && !attr_set[dev]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return static_cast<int>(e);
    attr_set[dev] = true;
  }
  const int total = num_m_blocks * nsplit;
  const int grid = total < num_sms ? total : num_sms;
  kern<<<grid, 256, smem, stream>>>(ta, tw, B, F, k, ksteps, num_m_blocks, num_n_tiles, nsplit,
                                    tiles_per_split, out_val, out_idx, g_encode_dbg);
  return static_cast<int>(cudaGetLastError());
}

static unsigned long long* g_encode_dbg_buf = nullptr;   // experiments only: [grid][8 warps][8] counters

template <int STAGES>
static int launch_encode2(const CUtensorMap& ta, const CUtensorMap& tw, int B, int F, int k,
                          int ksteps, int num_m_blocks, int num_n_tiles, int nsplit,
                          int tiles_per_split, float* out_val, int32_t* out_idx, int num_sms,
                          cudaStream_t stream) {
  constexpr int smem = Encode2Smem<STAGES>::kTotal;
  static bool attr_set[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 64 && !attr_set[dev]) {
    cudaError_t e = cudaFuncSetAttribute(encode_topk2_kernel<STAGES, false>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(encode_topk2_kernel<STAGES, true>,
                               cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return static_cast<int>(e);
    attr_set[dev] = true;
  }
  const int total = num_m_blocks * nsplit;
  const int grid = total < num_sms ? total : num_sms;
  if (g_encode_dbg_buf != nullptr)
    launch_pdl(encode_topk2_kernel<STAGES, true>, grid, 384, smem, stream, ta, tw, B, F, k, ksteps,
               num_m_blocks, num_n_tiles, nsplit, tiles_per_split, out_val, out_idx, g_encode_dbg_buf,
               g_encode_dbg, static_cast<uint32_t>(kBM * 4));
  else
    launch_pdl(encode_topk2_kernel<STAGES, false>, grid, 384, smem, stream, ta, tw, B, F, k, ksteps,
               num_m_blocks, num_n_tiles, nsplit, tiles_per_split, out_val, out_idx, nullptr, 0,
               static_cast<uint32_t>(kBM * 4));
  return static_cast<int>(cudaGetLastError());
}

// CTA-pair launch: 2-CTA clusters, one cluster per pair of SMs.
template <int STAGES>
static int launch_encode3(const CUtensorMap& ta, const CUtensorMap& tw_half, int B, int F, int k,
                          int ksteps, int num_m_blocks, int num_n_tiles, int nsplit,
                          int tiles_per_split, float* out_val, int32_t* out_idx, int num_sms,
                          cudaStream_t stream) {
  constexpr int smem = Encode3Smem<STAGES>::kTotal;
  static bool attr_set[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 64 && !attr_set[dev]) {
    cudaError_t e = cudaFuncSetAttribute(encode_topk3_kernel<STAGES, false>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(encode_topk3_kernel<STAGES, true>,
                               cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return static_cast<int>(e);
    attr_set[dev] = true;
  }
  const int total = ((num_m_blocks + 1) / 2) * nsplit;
  int clusters = num_sms / 2;
  if (total < clusters) clusters = total;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(static_cast<unsigned>(2 * clusters));
  cfg.blockDim = dim3(384);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute at[2];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 2;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[1].val.programmaticStreamSerializationAllowed = pdl_enabled();
  cfg.attrs = at;
  cfg.numAttrs = 2;
  cudaError_t e;
  if (g_encode_dbg_buf != nullptr)
    e = cudaLaunchKernelEx(&cfg, encode_topk3_kernel<STAGES, true>, ta, tw_half, B, F, k, ksteps, num_m_blocks,
                           num_n_tiles, nsplit, tiles_per_split, out_val, out_idx, g_encode_dbg_buf,
                           g_encode_dbg, static_cast<uint32_t>(kBM * 4));
  else
    e = cudaLaunchKernelEx(&cfg, encode_topk3_kernel<STAGES, false>, ta, tw_half, B, F, k, ksteps, num_m_blocks,
                           num_n_tiles, nsplit, tiles_per_split, out_val, out_idx,
                           static_cast<unsigned long long*>(nullptr), 0, static_cast<uint32_t>(kBM * 4));
  if (e != cudaSuccess) return static_cast<int>(e);
  return static_cast<int>(cudaGetLastError());
}

static int g_encode_variant = 0;   // 0 = per-batch choice (default), 1 = single epilogue warp per quarter, 2 = scanner + selector, 3 = 2 + CTA pairs (cta_group::2)

}  // namespace wsae

using namespace wsae;

extern "C" int wsae_debug_encode_variant(int v) { g_encode_variant = v; return 0; }
extern "C" int wsae_debug_encode_counters(void* buf) {
  g_encode_dbg_buf = static_cast<unsigned long long*>(buf);
  return 0;
}

// See include/wsae.h for the contract.
extern "C" int wsae_encode_topk(const void* a_packed, const void* w_packed, int B, int Bp, int F,
                                int Fp, int Kp, int k_used_cols, int k, int nsplit,
                                float* part_val, int32_t* part_idx, float* out_val,
                                int32_t* out_idx, cudaStream_t stream) {
  if (!a_packed || !w_packed || !out_val || !out_idx) return kBadArg;
  if (B <= 0 || F <= 0 || k <= 0 || k > F) return kBadArg;
  if (Bp % kBM != 0 || Fp % kBN != 0 || Kp % kBK != 0 || Bp < B || Fp < F) return kBadArg;
  if (k_used_cols <= 0 || k_used_cols % 16 != 0 || k_used_cols > Kp) return kBadArg;
  if (k > 64) return kUnsupported;
  if (nsplit < 1) return kBadArg;
  const int num_m_blocks = Bp / kBM;
  const int num_n_tiles = ceil_div(F, kBN);
  if (nsplit > num_n_tiles) nsplit = num_n_tiles;
  int tiles_per_split = ceil_div(num_n_tiles, nsplit);
  nsplit = ceil_div(num_n_tiles, tiles_per_split);
  if (nsplit > 1 && (!part_val || !part_idx)) return kBadArg;
  if (nsplit > 1 && ceil_div(nsplit * k, 32) > kMergeMaxPerLane) return kUnsupported;

  CUtensorMap ta, tw;
  int rc = make_tmap_bf16(&ta, a_packed, static_cast<uint64_t>(Bp), static_cast<uint64_t>(Kp), kBM);
  if (rc) return rc;
  rc = make_tmap_bf16(&tw, w_packed, static_cast<uint64_t>(Fp), static_cast<uint64_t>(Kp), kBN);
  if (rc) return rc;

  int dev = 0, num_sms = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
  float* kv = nsplit > 1 ? part_val : out_val;
  int32_t* ki = nsplit > 1 ? part_idx : out_idx;
  const int ksteps = k_used_cols / 16;
#ifndef WSAE_K1_STAGES
#define WSAE_K1_STAGES 3
#endif
#ifndef WSAE_K1_PAIR_STAGES
#define WSAE_K1_PAIR_STAGES 4
#endif
  // CTA-pair kernel (cta_group::2) by default once the batch fills the pairs (>= 1024 rows): 221 vs 231 us
  // at 384 -> 3072, 527 vs 564 us at 768 -> 6144, 2610 vs 3145 us at 1280 -> 40960 (B = 75776 / 37888;
  // tools/check_k1_pair.py, results bit-identical); tiny batches keep the single-CTA kernel (no cluster
  // set-up cost).  wsae_debug_encode_variant: 2 = always single-CTA, 3 = always pairs, 0 = this choice.
  const bool use_pair = g_encode_variant == 3 || (g_encode_variant == 0 && B >= 1024);
  if (k + kSlack <= kFifo && use_pair) {
    CUtensorMap tw_half;    // this CTA's half of a W' tile: 128 feature rows per box
    rc = make_tmap_bf16(&tw_half, w_packed, static_cast<uint64_t>(Fp), static_cast<uint64_t>(Kp), kBN / 2);
    if (rc) return rc;
    rc = launch_encode3<WSAE_K1_PAIR_STAGES>(ta, tw_half, B, F, k, ksteps, num_m_blocks, num_n_tiles, nsplit,
                                             tiles_per_split, kv, ki, num_sms, stream);
  } else if (k + kSlack <= kFifo && (g_encode_variant == 2 || g_encode_variant == 0))
    rc = launch_encode2<WSAE_K1_STAGES>(ta, tw, B, F, k, ksteps, num_m_blocks, num_n_tiles, nsplit,
                           tiles_per_split, kv, ki, num_sms, stream);
  else if (k <= 32)
    rc = launch_encode<80, WSAE_K1_STAGES>(ta, tw, B, F, k, ksteps, num_m_blocks, num_n_tiles, nsplit,
                              tiles_per_split, kv, ki, num_sms, stream);
  else
    rc = launch_encode<128, 2>(ta, tw, B, F, k, ksteps, num_m_blocks, num_n_tiles, nsplit,
                               tiles_per_split, kv, ki, num_sms, stream);
  if (rc) return rc;
  if (nsplit > 1) {
    const int warps = 8;
    const int per = ceil_div(nsplit * k, 32);
    const dim3 grid(ceil_div(B, warps)), block(warps * 32);
#define WSAE_MERGE_CASE(P)                                                                   \
  launch_pdl(topk_merge_kernel<P>, grid, block, 0, stream, part_val, part_idx, B, nsplit * k, k, out_val, \
             out_idx)
    if (per <= 2) WSAE_MERGE_CASE(2);
    else if (per <= 4) WSAE_MERGE_CASE(4);
    else if (per <= 8) WSAE_MERGE_CASE(8);
    else if (per <= 12) WSAE_MERGE_CASE(12);
    else if (per <= 16) WSAE_MERGE_CASE(16);
    else if (per <= 32) WSAE_MERGE_CASE(32);
    else WSAE_MERGE_CASE(64);
#undef WSAE_MERGE_CASE
    rc = static_cast<int>(cudaGetLastError());
  }
  return rc;
}


// The GEMM half of the small-batch form: pre[B, F] = A' x W'^T (bias included) with row pitch ld
// (a multiple of 4: the epilogue stores 16-byte vectors), nothing else.
static int encode_dense_ld(const void* a_packed, const void* w_packed, int B, int Bp, int F, int Fp, int Kp,
                           int k_used_cols, int ld, float* pre, cudaStream_t stream) {
  if (!a_packed || !w_packed || !pre) return kBadArg;
  if (B <= 0 || F <= 0) return kBadArg;
  if (Bp % kBM != 0 || Fp % kBN != 0 || Kp % kBK != 0 || Bp < B || Fp < F) return kBadArg;
  if (k_used_cols <= 0 || k_used_cols % 16 != 0 || k_used_cols > Kp) return kBadArg;
  if (ld < F || ld % 4 != 0) return kBadArg;
  CUtensorMap ta, tw;
  int rc = make_tmap_bf16(&ta, a_packed, static_cast<uint64_t>(Bp), static_cast<uint64_t>(Kp), kBM);
  if (rc) return rc;
  rc = make_tmap_bf16(&tw, w_packed, static_cast<uint64_t>(Fp), static_cast<uint64_t>(Kp), kBN);
  if (rc) return rc;
  int dev = 0, num_sms = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
  constexpr int kStages = 3;
  constexpr int smem_g = kStages * (kAStage + kBStage) + 256 + 1024;
  static bool attr_set[64] = {};
  if (dev >= 64 || !attr_set[dev]) {
    cudaError_t e = cudaFuncSetAttribute(encode_dense_kernel<kStages>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, smem_g);
    if (e != cudaSuccess) return static_cast<int>(e);
    if (dev < 64) attr_set[dev] = true;
  }
  const int num_m_blocks = Bp / kBM;
  const int num_n_tiles = ceil_div(F, kBN);
  const int total = num_m_blocks * num_n_tiles;
  const int grid = total < num_sms ? total : num_sms;
  cudaError_t e = launch_pdl(encode_dense_kernel<kStages>, grid, 256, smem_g, stream, ta, tw, B, F, ld,
                             k_used_cols / 16, num_m_blocks, num_n_tiles, pre);
  return static_cast<int>(e != cudaSuccess ? e : cudaGetLastError());
}

extern "C" int wsae_encode_dense(const void* a_packed, const void* w_packed, int B, int Bp, int F, int Fp,
                                 int Kp, int k_used_cols, float* pre_ws, cudaStream_t stream) {
  if (F > 0 && F % 4 != 0) return kUnsupported;
  return encode_dense_ld(a_packed, w_packed, B, Bp, F, Fp, Kp, k_used_cols, F, pre_ws, stream);
}

// Column slices of the row select: the keys of one slice fill at most 192 KB of shared memory.
constexpr int kSelectMaxCols = 49152;
static int select_slices(int F) { return ceil_div(F, kSelectMaxCols); }
static int select_slice_cols(int F) { return round_up(ceil_div(F, select_slices(F)), 4); }

// The select half: per row of pre (pitch ld), the k largest of pre[row, 0:F] in ascending feature index.
// One slice: one block per row, straight into out_*.  Several: one block per (row, slice) writes k
// candidates per slice to part_* ([B, nslices * k], ascending feature index, short slices padded with
// (-inf, -1)), and topk_merge_kernel keeps the k largest, ties to the earlier candidate, i.e. to the
// lowest feature index, as one unsliced select does.
static int rowwise_select(const float* pre, int B, int F, int ld, int k, float* part_val, int32_t* part_idx,
                          float* out_val, int32_t* out_idx, cudaStream_t stream) {
  const int ns = select_slices(F);
  const int S = select_slice_cols(F);
  int dev = 0;
  cudaGetDevice(&dev);
  static bool attr_set[64] = {};
  if (dev >= 64 || !attr_set[dev]) {
    cudaError_t e = cudaFuncSetAttribute(rowwise_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e != cudaSuccess) return static_cast<int>(e);
    if (dev < 64) attr_set[dev] = true;
  }
  const size_t smem_t = static_cast<size_t>(S) * 4;
  cudaError_t e = launch_pdl(rowwise_topk_kernel, dim3(B, ns), kRowTopkThreads, smem_t, stream, pre, B, F, ld, S,
                             k, ns > 1 ? part_val : out_val, ns > 1 ? part_idx : out_idx);
  if (e != cudaSuccess) return static_cast<int>(e);
  if (ns > 1) {
    const int warps = 8;
    const int n = ns * k;
    const dim3 grid(ceil_div(B, warps)), block(warps * 32);
    const int per = ceil_div(n, 32);
    if (per <= 8) e = launch_pdl(topk_merge_kernel<8>, grid, block, 0, stream, part_val, part_idx, B, n, k, out_val, out_idx);
    else if (per <= 16) e = launch_pdl(topk_merge_kernel<16>, grid, block, 0, stream, part_val, part_idx, B, n, k, out_val, out_idx);
    else if (per <= 32) e = launch_pdl(topk_merge_kernel<32>, grid, block, 0, stream, part_val, part_idx, B, n, k, out_val, out_idx);
    else e = launch_pdl(topk_merge_kernel<64>, grid, block, 0, stream, part_val, part_idx, B, n, k, out_val, out_idx);
    if (e != cudaSuccess) return static_cast<int>(e);
  }
  return static_cast<int>(cudaGetLastError());
}

// Small-batch form of wsae_encode_topk (see encode_dense_kernel): `pre_ws` is B * F floats of scratch.
// Same results as wsae_encode_topk (values bit-identical: the same MMA sequence; ties to the lowest
// feature index), output in ascending feature index.  F * 4 bytes of shared memory per row block:
// F <= 49152.
extern "C" int wsae_encode_topk_dense(const void* a_packed, const void* w_packed, int B, int Bp, int F,
                                      int Fp, int Kp, int k_used_cols, int k, float* pre_ws,
                                      float* out_val, int32_t* out_idx, cudaStream_t stream) {
  if (!out_val || !out_idx) return kBadArg;
  if (k <= 0 || k > F) return kBadArg;
  if (F > kSelectMaxCols || k > 0xFFFF) return kUnsupported;
  int rc = wsae_encode_dense(a_packed, w_packed, B, Bp, F, Fp, Kp, k_used_cols, pre_ws, stream);
  if (rc) return rc;
  return rowwise_select(pre_ws, B, F, F, k, nullptr, nullptr, out_val, out_idx, stream);
}

// K1 for k > 64 at any batch: the dense GEMM and the row select over row chunks of chunk_rows (a multiple
// of 128) with one scratch: [chunk_rows, round_up(F, 4)] fp32 pre-activations, then, when F > 49152, the
// [chunk_rows, nslices * k] candidate values and indices of the sliced select.  The fused epilogues hold a row's candidates in
// registers and stop at k = 64; the radix select does not.  Per chunk the GEMM reads the packed rows from
// a tensor map based at the chunk's first row, so every 128 x 256 tile runs the same MMA sequence as in
// one unchunked call: the values are bit-identical to it, and the selection is exact on them.  Chunks the
// size of a few tens of MB keep the scratch in L2 between the GEMM that writes it and the select that
// reads it.
extern "C" int wsae_encode_topk_chunked(const void* a_packed, const void* w_packed, int B, int Bp, int F,
                                        int Fp, int Kp, int k_used_cols, int k, int chunk_rows,
                                        float* pre_ws, float* out_val, int32_t* out_idx,
                                        cudaStream_t stream) {
  if (!a_packed || !out_val || !out_idx || !pre_ws) return kBadArg;
  if (B <= 0 || Bp < B || Bp % kBM != 0 || Kp % kBK != 0) return kBadArg;
  if (chunk_rows <= 0 || chunk_rows % kBM != 0) return kBadArg;
  if (F <= 0 || k <= 0 || k > F) return kBadArg;
  const int ns = select_slices(F);
  if (k > 0xFFFF || (ns > 1 && (static_cast<long long>(ns) * k + 31) / 32 > kMergeMaxPerLane)) return kUnsupported;
  const int ld = round_up(F, 4);
  const size_t part_n = static_cast<size_t>(chunk_rows) * ns * k;
  float* part_val = pre_ws + static_cast<size_t>(chunk_rows) * ld;
  int32_t* part_idx = reinterpret_cast<int32_t*>(part_val + part_n);
  const size_t row_bytes = static_cast<size_t>(Kp) * 2;
  for (int r0 = 0; r0 < B; r0 += chunk_rows) {
    const int rows = B - r0 < chunk_rows ? B - r0 : chunk_rows;
    const int rows_p = Bp - r0 < chunk_rows ? Bp - r0 : chunk_rows;
    int rc = encode_dense_ld(static_cast<const char*>(a_packed) + r0 * row_bytes, w_packed, rows, rows_p, F,
                             Fp, Kp, k_used_cols, ld, pre_ws, stream);
    if (rc) return rc;
    rc = rowwise_select(pre_ws, rows, F, ld, k, part_val, part_idx, out_val + static_cast<size_t>(r0) * k,
                        out_idx + static_cast<size_t>(r0) * k, stream);
    if (rc) return rc;
  }
  return kOk;
}

extern "C" int wsae_debug_encode_mode(int mode) { g_encode_dbg = mode; return 0; }

// Number of F-splits wsae_encode_topk will actually use for a requested nsplit (so callers can
// size part_val / part_idx = B * nsplit_eff * k entries).
extern "C" int wsae_encode_effective_splits(int F, int nsplit) {
  const int num_n_tiles = ceil_div(F, kBN);
  if (nsplit < 1) nsplit = 1;
  if (nsplit > num_n_tiles) nsplit = num_n_tiles;
  const int tps = ceil_div(num_n_tiles, nsplit);
  return ceil_div(num_n_tiles, tps);
}
