// sm_100a building blocks: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (UMMA + TMEM).
// Everything here is inline PTX; nothing in this file links against libcuda.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace vfp {

// ------------------------------------------------------------------------------------------
// misc
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// Device-visible error word: kernels write a nonzero code and trap instead of spinning forever.
// (a hung kernel on a shared box costs a strike; a trapped one only costs the call.)
__device__ unsigned int g_vfp_device_error = 0;

enum DeviceError : unsigned int {
  kErrNone = 0,
  kErrMbarTimeout = 0xBA440001u,
};

// ------------------------------------------------------------------------------------------
// mbarrier
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: ~ several seconds worth of polls, then flag + trap.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) {  // ~2 s at 2 GHz
      atomicExch(&g_vfp_device_error, (unsigned int)kErrMbarTimeout);
      __threadfence_system();
      asm volatile("trap;");
    }
  }
}

// Hang diagnosis (vfp_set_tuning(2, 1)): instead of trapping, a timed-out wait records (barrier smem address, parity,
// thread, block) in g_vfp_hang_log and RETURNS, so the kernel drains (with garbage results) and the host can read
// which barrier never completed. Off by default.
__device__ int g_vfp_hang_mode = 0;
__device__ unsigned int g_vfp_hang_count = 0;
__device__ unsigned int g_vfp_hang_log[64 * 4];

// try_wait with an explicit suspend-time hint: the hardware parks the thread until the phase completes or `ns` nanoseconds
// have passed, whichever comes first, so a waiting warp neither burns issue slots nor adds polling latency to the hand-off.
__device__ __forceinline__ bool mbar_try_wait_hint(uint64_t* bar, uint32_t parity, uint32_t ns) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(ns)
      : "memory");
  return ok != 0;
}

// Wait used by whole warps (epilogue / producer / loader roles) and by the single-lane issuers of the stem kernels.
// History: a tight try_wait loop cost ~60 % of all executed instructions of the fused stem kernel (the default suspend
// time is short); backing off with __nanosleep fixed that but put up to 128 ns of polling latency on EVERY hand-off,
// which made the stem kernels latency-bound (2.5 us per frame with all work knocked out, scripts/dev_knockout.py).
// The suspend-time hint gives both: no spinning, wake-up when the phase completes.
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  uint32_t spins = 0;
  long long t0 = 0;
  while (!mbar_try_wait_hint(bar, parity, 20000u)) {   // <= 20 us per attempt
    if ((++spins & 0x3FF) == 0) {
      if (t0 == 0) t0 = clock64();
      else {
        const int mode = *reinterpret_cast<volatile int*>(&g_vfp_hang_mode);
        if (clock64() - t0 > (mode ? 400000000LL : 4000000000LL)) {
          atomicExch(&g_vfp_device_error, (unsigned int)kErrMbarTimeout);
          if (mode) {
            const unsigned int i = atomicAdd(&g_vfp_hang_count, 1u);
            if (i < 64) {
              g_vfp_hang_log[4 * i] = smem_u32(bar);
              g_vfp_hang_log[4 * i + 1] = parity;
              g_vfp_hang_log[4 * i + 2] = threadIdx.x;
              g_vfp_hang_log[4 * i + 3] = blockIdx.x;
            }
            return;
          }
          __threadfence_system();
          asm volatile("trap;");
        }
      }
    }
  }
}

// Wait for roles that are far from the critical path (frame copy issuer, transposers): sleeping between polls keeps their
// retries out of the issue slots and the shared-memory port the critical roles need.
__device__ __forceinline__ void mbar_wait_lazy(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    __nanosleep(100);
    if (++spins > 40000000u) {   // several seconds
      atomicExch(&g_vfp_device_error, (unsigned int)kErrMbarTimeout);
      if (*reinterpret_cast<volatile int*>(&g_vfp_hang_mode)) return;
      __threadfence_system();
      asm volatile("trap;");
    }
  }
}

// ------------------------------------------------------------------------------------------
// TMA tiled loads (global -> shared), completion on an mbarrier
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* m, uint64_t* bar, void* dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(const CUtensorMap* m, uint64_t* bar, void* dst, int c0, int c1,
                                            int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
      "[%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2),
      "r"(c3)
      : "memory");
}

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.aligned;\n\tbarrier.cluster.wait.aligned;" ::: "memory");
}

// ---- CTA pairs (tcgen05 cta_group::2): two CTAs of a cluster drive ONE UMMA of M = 256; each SM computes 128 rows, reads its own
// A rows and HALF of the B rows from its own shared memory and gets the other half from its peer. Only the leader CTA
// (cluster rank 0) issues the instruction, so both CTAs' loads report to the LEADER's mbarrier. ----
// shared::cluster address of `p` in the CTA with cluster rank `rank`
__device__ __forceinline__ uint32_t mapa_u32(const void* p, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(p)), "r"(rank));
  return r;
}
// Default semantics (.release at CTA scope), as CUTLASS's ClusterBarrier::arrive(cta_id) uses for consumer -> leader signals.
// What the leader's issuer must be able to rely on was ordered before the arrive by the caller: tcgen05.wait::ld +
// tcgen05.fence::before_thread_sync for accumulators that were read, fence.proxy.async for shared-memory operands that were
// written (both act inside the arriving CTA, which is where the tensor core will read them). Spelling the arrive
// .release.cluster makes ptxas emit MEMBAR.ALL.GPU / MEMBAR.SC.SYS + ERRBAR in front of it: ncu attributed 24 % of all warp
// samples of the fused MLP kernel to that stall.
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// local destination, completion bytes counted on the mbarrier at shared::cluster address `bar_cluster_addr` (the leader's)
__device__ __forceinline__ void tma_load_2d_2cta(const CUtensorMap* m, uint32_t bar_cluster_addr, void* dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_2cta(const CUtensorMap* m, uint32_t bar_cluster_addr, void* dst, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_2cta(uint32_t* slot_in_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot_in_smem)), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish_2cta() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2cta(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem of both CTAs] (+)= A[256 rows: 128 in each CTA's smem] * B[N rows: N/2 in each CTA's smem]^T
__device__ __forceinline__ void umma_bf16_2cta(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives (once all earlier UMMAs of the pair have completed) at the mbarrier at this offset in every CTA of `cta_mask`
__device__ __forceinline__ void umma_commit_2cta(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"(cta_mask)
               : "memory");
}

// TMA tiled store (shared -> global), bulk-group completion
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}

// ------------------------------------------------------------------------------------------
// tcgen05: TMEM allocation, UMMA issue, commit, TMEM loads
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* slot_in_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot_in_smem)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]; kind::f16 covers bf16 inputs with fp32 accumulate.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier once all previously issued UMMAs of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 32 lanes x 32 consecutive fp32 columns: thread t of the warp gets lane (base_lane + t), columns c..c+31.
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}

// 32 lanes x 16 consecutive fp32 columns (half the registers of the x32 form)
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}

// 32 lanes x 8 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld_32x8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr)
               : "memory");
}

// ------------------------------------------------------------------------------------------
// packed fp32 pairs (FADD2 / FFMA2 on sm_100)
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) {
  unsigned long long ra, rb, rd;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a.x), "f"(a.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
  float2 d;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(rd));
  return d;
}
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
  unsigned long long ra, rb, rd;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a.x), "f"(a.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
  float2 d;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(rd));
  return d;
}
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  unsigned long long ra, rb, rc, rd;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a.x), "f"(a.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rc) : "f"(c.x), "f"(c.y));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
  float2 d;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(rd));
  return d;
}

// ------------------------------------------------------------------------------------------
// UMMA descriptors
// ------------------------------------------------------------------------------------------
// Shared-memory operand descriptor for a K-major tile whose rows are `row_bytes` wide
// (32, 64 or 128 B = the TMA swizzle span) and stored densely, 8-row groups `8*row_bytes` apart.
// Bit layout (sm_100 "version 1" descriptor):
//   [0,14)  start address >> 4      [16,30) leading byte offset >> 4 (unused for swizzled K-major)
//   [32,46) stride byte offset >> 4 [46,48) version = 1      [61,64) layout: 2=SW128, 4=SW64, 6=SW32
template <int ROW_BYTES>
__device__ __forceinline__ uint64_t umma_smem_desc_kmajor(uint32_t smem_addr) {
  static_assert(ROW_BYTES == 128 || ROW_BYTES == 64 || ROW_BYTES == 32, "swizzle span");
  constexpr uint64_t layout = ROW_BYTES == 128 ? 2ull : (ROW_BYTES == 64 ? 4ull : 6ull);
  constexpr uint64_t sbo = (8ull * ROW_BYTES) >> 4;
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;  // LBO (ignored for swizzled K-major; canonical value 1)
  d |= sbo << 32;
  d |= 1ull << 46;  // descriptor version for Blackwell
  d |= layout << 61;
  return d;
}

// Instruction descriptor, kind::f16: bf16 x bf16 -> fp32, both operands K-major.
//   [4,6) D fmt (1=f32)  [7,10) A fmt (1=bf16)  [10,13) B fmt (1=bf16)  [15] A major  [16] B major
//   [17,23) N>>3  [24,29) M>>4
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(N >> 3) << 17) |
         (static_cast<uint32_t>(M >> 4) << 24);
}

}  // namespace vfp
