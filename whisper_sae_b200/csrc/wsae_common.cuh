// wsae_common.cuh — sm_100a device helpers shared by the TopK-SAE train-step kernels.
//
// Thin inline-PTX wrappers (mbarrier, TMA, tcgen05/TMEM) plus small numeric utilities.
// Everything here targets Blackwell B200 (compute_100a) only; there is no other code path.
#pragma once

#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <cstdlib>
#include <type_traits>

#ifndef WSAE_SPIN_LIMIT
// Bounded spin on mbarrier waits: a broken pipeline traps (CUDA error) instead of hanging the GPU.
#define WSAE_SPIN_LIMIT (1u << 22)
#endif

namespace wsae {

// ----------------------------------------------------------------------------------------------
// status codes (mirrors include/wsae.h)
// ----------------------------------------------------------------------------------------------
constexpr int kOk = 0;
constexpr int kBadArg = -1;
constexpr int kUnsupported = -2;
constexpr int kNoDriver = -3;

__host__ __device__ constexpr int ceil_div(int a, int b) { return (a + b - 1) / b; }
__host__ __device__ constexpr int round_up(int a, int b) { return ceil_div(a, b) * b; }

// ----------------------------------------------------------------------------------------------
// programmatic dependent launch (PDL): the kernels of the train step form one dependent chain on a
// stream (and in the captured graph).  Launched with the programmatic-serialization attribute, a
// kernel's CTAs may be scheduled while the previous kernel is still draining, so launch latency,
// shared-memory carve-up and barrier / TMEM set-up overlap the predecessor's tail.  Contract for
// every kernel launched through launch_pdl(): pdl_wait() comes before the FIRST global-memory
// access (reads and writes alike: the predecessor may still be reading what this kernel writes);
// griddepcontrol.wait returns when all prerequisite grids have completed and flushed.  Both
// instructions are no-ops in a kernel launched without the attribute.
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_launch_dependents() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
// the usual kernel prologue: let the successor in, then wait for the predecessor
__device__ __forceinline__ void pdl_prologue() {
  pdl_launch_dependents();
  pdl_wait();
}

// OFF by default: measured on the B200 (tools/ab_pdl.sh, same box, 3 x A/B) the graph replay of the
// train step is 0.916 ms without and 0.926 ms with the attribute at B = 75 776, and 0.224 vs 0.223 ms
// at B = 128 - inside a CUDA graph the kernel->kernel edges are already cheap, and CTAs of the
// successor that become resident early only take slots.  WSAE_PDL=1 switches it on (read once).
inline int pdl_enabled() {
  static const int on = [] {
    const char* e = std::getenv("WSAE_PDL");
    return (e && e[0] == '1') ? 1 : 0;
  }();
  return on;
}
// kernel<<<grid, block, smem, stream>>>(args...) with the PDL attribute.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem,
                              cudaStream_t stream, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = pdl_enabled();
  cfg.attrs = at;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// ----------------------------------------------------------------------------------------------
// warp helpers
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t lane_id() {
  uint32_t l;
  asm volatile("mov.u32 %0, %%laneid;" : "=r"(l));
  return l;
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "elect.sync _|P1, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P1;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ----------------------------------------------------------------------------------------------
// order-preserving float <-> uint32 keys (larger float <=> larger key)
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t f2key(float v) {
  uint32_t b = __float_as_uint(v);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float key2f(uint32_t k) {
  uint32_t b = (k & 0x80000000u) ? (k ^ 0x80000000u) : ~k;
  return __uint_as_float(b);
}

// ----------------------------------------------------------------------------------------------
// mbarrier
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P1;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > WSAE_SPIN_LIMIT) __trap();
  }
}

// Wait with back-off: for hand-shakes between two warps that share an SM sub-partition, where a
// tight try_wait loop would steal issue slots from the very warp it is waiting for.
__device__ __forceinline__ void mbar_wait_backoff(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    __nanosleep(100);
    if (++spins > WSAE_SPIN_LIMIT) __trap();
  }
}

// 2D tiled load multicast to every CTA of `cta_mask` in the cluster: the box lands at the same
// shared-memory offset in each destination CTA and completes bytes on each one's own mbarrier.
__device__ __forceinline__ void tma_load_2d_multicast(void* smem_dst, const void* tmap, uint64_t* bar,
                                                      int32_t c_inner, int32_t c_outer,
                                                      uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster"
      " [%0], [%1, {%4, %5}], [%2], %3;"
      ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "h"(cta_mask), "r"(c_inner),
      "r"(c_outer)
      : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_nctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
  return r;
}
// Cluster-wide barrier (every thread of every CTA of the cluster).
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// Wait with a short sleep between polls (NS nanoseconds; 0 = tight loop): for the TMA / MMA roles,
// whose polling would otherwise take issue slots from the epilogue warps on their sub-partition.
template <int NS>
__device__ __forceinline__ void mbar_wait_sleep(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (NS > 0) __nanosleep(NS);
    if (++spins > WSAE_SPIN_LIMIT) __trap();
  }
}

// ----------------------------------------------------------------------------------------------
// TMA (cp.async.bulk.tensor) — 2D tiled load, completion on an mbarrier
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const void* tmap, uint64_t* bar,
                                            int32_t c_inner, int32_t c_outer) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c_inner), "r"(c_outer)
      : "memory");
}

// ----------------------------------------------------------------------------------------------
// tcgen05 / TMEM
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_slot)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// D[tmem] (+)= A[smem desc] * B[smem desc], bf16 x bf16 -> fp32, issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Same, delivered to the barrier at the same shared-memory offset in every CTA of `cta_mask`
// (thread-block cluster): one arrival per destination.
__device__ __forceinline__ void umma_commit_multicast(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(cta_mask)
      : "memory");
}
// Make the mbarrier observe completion of all MMAs issued so far by this thread.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}

// 32 lanes x 16 consecutive fp32 columns: thread t of the warp gets lane (base_lane + t).
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32"
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}

// Wait for the tcgen05.ld that filled r[]; the "+r" operands pin the uses after the wait.
__device__ __forceinline__ void tmem_ld_wait16(uint32_t (&r)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]),
                 "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]),
                 "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
               :
               : "memory");
}

// Shared-memory matrix descriptor for a K-major bf16 operand tile stored with the 128-byte
// swizzle exactly as TMA (CU_TENSOR_MAP_SWIZZLE_128B) writes it: rows of 64 bf16 = 128 B,
// 8-row groups 1024 B apart (SBO), descriptor version 1 (Blackwell), layout type 2 (SW128).
__device__ __forceinline__ uint64_t umma_desc_sw128_kmajor(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);  // start address  [0,14)
  d |= static_cast<uint64_t>(1) << 16;                      // LBO (unused for SW128 K-major)
  d |= static_cast<uint64_t>(1024 >> 4) << 32;              // SBO = 1024 B
  d |= static_cast<uint64_t>(1) << 46;                      // descriptor version
  d |= static_cast<uint64_t>(2) << 61;                      // SWIZZLE_128B
  return d;
}

// Instruction descriptor: kind::f16, A=B=bf16 (K-major), D=fp32, shape M x N.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(N >> 3) << 17) |
         (static_cast<uint32_t>(M >> 4) << 24);
}

// ----------------------------------------------------------------------------------------------
// vectorised global helpers
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void red_add_f32x4(float* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c),
               "f"(d)
               : "memory");
}

__device__ __forceinline__ float4 bf16x4_to_float4(uint2 u) {
  float4 f;
  f.x = __uint_as_float(u.x << 16);
  f.y = __uint_as_float(u.x & 0xFFFF0000u);
  f.z = __uint_as_float(u.y << 16);
  f.w = __uint_as_float(u.y & 0xFFFF0000u);
  return f;
}

// ----------------------------------------------------------------------------------------------
// activation element types: the kernels that read the activation matrix (K0, K23, the row step) are
// templated on its element type TX = float / __nv_bfloat16 / __half (dtype code 0 / 1 / 2, as in
// wsae_layernorm_rows).  A half value converts to fp32 exactly, and the conversion happens at the
// load: the arithmetic after it is the fp32 kernel's, so a half matrix trains bit for bit like its
// fp32 copy.  The loads below are the fp32 kernels' loads for TX = float.
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ float2 x2_to_float2(uint32_t u, const __nv_bfloat16*) {
  return make_float2(__uint_as_float(u << 16), __uint_as_float(u & 0xFFFF0000u));
}
__device__ __forceinline__ float2 x2_to_float2(uint32_t u, const __half*) {
  return __half22float2(*reinterpret_cast<const __half2*>(&u));
}
template <typename TX>
__device__ __forceinline__ float4 x4_to_float4(uint2 u) {
  const float2 lo = x2_to_float2(u.x, static_cast<const TX*>(nullptr));
  const float2 hi = x2_to_float2(u.y, static_cast<const TX*>(nullptr));
  return make_float4(lo.x, lo.y, hi.x, hi.y);
}

// 4 consecutive elements (16-byte aligned for fp32, 8-byte for half types), read-only path
__device__ __forceinline__ float4 ldg_x4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
template <typename TX>
__device__ __forceinline__ float4 ldg_x4(const TX* p) {
  return x4_to_float4<TX>(__ldg(reinterpret_cast<const uint2*>(p)));
}
// 2 consecutive elements, plain load
__device__ __forceinline__ float2 ld_x2(const float* p) { return *reinterpret_cast<const float2*>(p); }
template <typename TX>
__device__ __forceinline__ float2 ld_x2(const TX* p) {
  return x2_to_float2(*reinterpret_cast<const uint32_t*>(p), p);
}

// Host side: fn(static_cast<const TX*>(nullptr)) for the element type of dtype code x_dtype;
// kBadArg for a code that names none.
template <typename Fn>
inline int with_x_dtype(int x_dtype, Fn&& fn) {
  switch (x_dtype) {
    case 0: return fn(static_cast<const float*>(nullptr));
    case 1: return fn(static_cast<const __nv_bfloat16*>(nullptr));
    case 2: return fn(static_cast<const __half*>(nullptr));
    default: return kBadArg;
  }
}

}  // namespace wsae
