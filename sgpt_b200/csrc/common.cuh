// sm_100a building blocks shared by every kernel in this library: mbarrier, TMA, tcgen05 (UMMA / TMEM)
// PTX wrappers, UMMA descriptor encoders, and small numeric helpers.
//
// Everything here is hand-written inline PTX for sm_100a (no CUTLASS/CuTe).  Descriptor bit layouts follow the
// PTX ISA "tcgen05 matrix descriptor" / "instruction descriptor" tables.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace sgpt {

// ---------------------------------------------------------------------------------------------------------------
// misc
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}\n"
      : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float bf16_lo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t v) { return __uint_as_float(v & 0xffff0000u); }

// ---------------------------------------------------------------------------------------------------------------
// Programmatic dependent launch.  Every kernel of the library is launched with
// cudaLaunchAttributeProgrammaticStreamSerialization (host_utils.h: launch_kernel): its CTAs may become resident while the
// previous kernel of the stream is still draining.  pdl_wait() blocks until every prerequisite grid has completed and
// its memory is visible — it must precede the FIRST global-memory access of the kernel; what sits before it (barrier
// init, TMEM allocation, descriptor prefetch, index arithmetic) overlaps the predecessor's tail.
// pdl_launch_dependents() lets the NEXT kernel of the stream start the same way once all CTAs of this grid have
// executed it (or exited).  Both are no-ops when the launch carried no such attribute.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_sync() {
  pdl_wait();
  pdl_launch_dependents();
}

// ---------------------------------------------------------------------------------------------------------------
// mbarrier
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Non-blocking probe: mbarrier.try_wait may SUSPEND the thread for an implementation-defined time when the phase is not
// complete — fine for a thread that waits for one barrier, poison for a thread that polls several (the attention kernel's
// producer and MMA issuer serve 2-4 slots); test_wait returns at once.
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Spin with a bounded poll count: a protocol bug traps (launch error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t polls = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++polls > (1u << 24)) {
      printf("sgpt: mbarrier wait timed out (block %d thread %d bar %p parity %u)\n", blockIdx.x, threadIdx.x,
             (void*)bar, parity);
      __trap();
    }
  }
}

// generic-proxy writes to smem -> visible to the async proxy (TMA / tcgen05 operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ---------------------------------------------------------------------------------------------------------------
// TMA (cp.async.bulk.tensor)
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* desc) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(desc)) : "memory");
}
// 2D tile load: coordinates are (c0 = innermost/contiguous dim, c1 = row).
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* desc, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(desc)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// L2 cache-hinted variant (createpolicy-encoded 64-bit hints as used by the driver's canonical policies).
constexpr uint64_t kCacheEvictFirst = 0x12F0000000000000ull;
constexpr uint64_t kCacheEvictLast = 0x14F0000000000000ull;
__device__ __forceinline__ void tma_load_2d_hint(void* smem_dst, const CUtensorMap* desc, uint64_t* bar, int c0,
                                                 int c1, uint64_t hint) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(desc)), "r"(smem_u32(bar)), "r"(c0), "r"(c1),
        "l"(hint)
      : "memory");
}

// Tile prefetch into L2 only (no smem, no barrier): turns the DRAM latency of a later tma_load_2d into an L2 hit.
__device__ __forceinline__ void tma_prefetch_l2_2d(const CUtensorMap* desc, int c0, int c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];" ::"l"(reinterpret_cast<uint64_t>(desc)),
               "r"(c0), "r"(c1)
               : "memory");
}

// Multicast tile load: the tile lands at the same smem offset in every CTA of the cluster whose bit is set in
// cta_mask, and each destination CTA's mbarrier (same offset) receives the complete_tx.  One L2 read feeds all of them.
__device__ __forceinline__ void tma_load_2d_multicast(void* smem_dst, const CUtensorMap* desc, uint64_t* bar, int c0,
                                                      int c1, uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(desc)), "r"(smem_u32(bar)), "r"(c0), "r"(c1),
        "h"(cta_mask)
      : "memory");
}

// 1-D bulk copy global -> shared (contiguous bytes; size and both addresses multiples of 16), completion on an mbarrier
__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// thread-block cluster helpers
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// smem tile -> global (bulk async-group completion).  Coordinates as for loads; out-of-range rows/columns are clipped.
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* desc, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               :
               : "l"(reinterpret_cast<uint64_t>(desc)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
// global[tile] += smem tile (element-wise fp32 add performed by the L2; each element must be added once per launch
// for a deterministic result)
__device__ __forceinline__ void tma_reduce_add_2d(const CUtensorMap* desc, const void* smem_src, int c0, int c1) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];"
               :
               : "l"(reinterpret_cast<uint64_t>(desc)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// wait until at most N of this thread's bulk groups are still reading their smem source
template <int N>
__device__ __forceinline__ void bulk_wait_group_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
// wait until at most N of this thread's bulk groups are still in flight at all
template <int N>
__device__ __forceinline__ void bulk_wait_group() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// explicit shared-window accesses (32-bit addresses; avoids generic-address LD/ST in hot loops)
__device__ __forceinline__ void sts_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void sts_v2(uint32_t addr, uint32_t a, uint32_t b) {
  asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(addr), "r"(a), "r"(b) : "memory");
}
__device__ __forceinline__ float4 lds_v4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ float2 lds_v2(uint32_t addr) {
  float2 v;
  asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr) : "memory");
  return v;
}

// ---------------------------------------------------------------------------------------------------------------
// tcgen05: TMEM allocation, MMA, commit, load
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_holder, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_holder)),
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
// Arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// Same, arriving on the barrier at this smem offset in every CTA of the cluster selected by cta_mask.
__device__ __forceinline__ void umma_commit_multicast(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(cta_mask)
      : "memory");
}

// D[tmem] (+)= A[smem desc] * B[smem desc], bf16 inputs, fp32 accumulate.
__device__ __forceinline__ void umma_bf16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
      :
      : "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// A operand read from TMEM (packed bf16 pairs per 32-bit column), B from smem.
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n"
      :
      : "r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}

// ---- CTA-pair (cta_group::2) variants: the two CTAs of a 2-CTA cluster (one TPC) execute ONE M=256 MMA.  Each CTA holds
// its own 128 rows of A, HALF of the B tile (N/2 rows) and its own 128 accumulator rows in TMEM; the leader CTA (rank 0)
// issues the MMAs for both.  Compared with two independent M=128 MMAs the per-SM smem footprint, TMA write traffic and
// operand read traffic of B halve, which is what leaves smem bandwidth for the epilogue.
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_holder, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_holder)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_pair() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_bf16_ss_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                                  uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
      :
      : "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// int8 operands (signed x signed), s32 accumulate: K = 32 per instruction, i.e. the same 32 bytes of a 128-byte swizzle
// row as a K = 16 bf16 MMA, so the smem descriptors and their +2 advance are shared with the bf16 forms.
__device__ __forceinline__ void umma_s8_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}\n"
      :
      : "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_s8_ss_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                                uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n\t}\n"
      :
      : "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive (once all previously issued pair MMAs completed) on the barrier at this smem offset in the CTAs of cta_mask.
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(cta_mask)
      : "memory");
}
// shared::cluster address of `local` (a shared::cta address of this CTA) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_shared(uint32_t local, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local), "r"(rank));
  return r;
}
// arrive on an mbarrier that may live in another CTA of the cluster (address from mapa_shared)
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// Tile load into THIS CTA's smem whose complete_tx is delivered to a barrier in the pair's leader CTA
// (bar_cluster_addr from mapa_shared(.., 0)); .cta_group::2 is what permits the barrier to live in the peer.
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* desc, uint32_t bar_cluster_addr,
                                                 int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(desc)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}

// The same, MULTICAST: the tile lands at this smem offset in every CTA of `cta_mask`; each destination CTA's complete_tx is
// delivered to the mbarrier at `bar_addr`'s CTA-relative offset in the LEADER (even-ranked CTA) of the destination's own
// pair — bar_addr is the shared::cluster address of the barrier in the ISSUING CTA's pair leader (mapa).  Used by the
// 4-CTA cluster GEMM: two CTA pairs share every weight tile, fetched from L2 once.
__device__ __forceinline__ void tma_load_2d_pair_multicast(void* smem_dst, const CUtensorMap* desc, uint32_t bar_addr,
                                                           int c0, int c1, uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(desc)), "r"(bar_addr), "r"(c0), "r"(c1), "h"(cta_mask)
      : "memory");
}

// Instruction descriptor for kind::f16 with bf16 A/B and fp32 D.
//   [4,6) D format (1 = f32)   [7,10) A format (1 = bf16)   [10,13) B format (1 = bf16)
//   [15] A major (0 = K)       [16] B major (0 = K, 1 = MN) [17,23) N >> 3            [24,29) M >> 4
__host__ __device__ constexpr uint32_t make_idesc_bf16(int m, int n, bool b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (0u << 15) | ((b_mn_major ? 1u : 0u) << 16) |
         (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}

// Instruction descriptor for kind::i8 with signed 8-bit A/B, s32 D, both operands K-major.
//   [4,6) D format (2 = s32)   [7,10) A format (1 = signed 8-bit)   [10,13) B format (1 = signed 8-bit)
//   [13,15) negate A/B (must be 0 for kind::i8)   [17,23) N >> 3   [24,29) M >> 4
__host__ __device__ constexpr uint32_t make_idesc_s8(int m, int n) {
  return (2u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(n >> 3) << 17) |
         (static_cast<uint32_t>(m >> 4) << 24);
}

// Shared-memory matrix descriptor, SWIZZLE_128B, for tiles written by TMA with a 128-byte inner box.
//   [0,14) start >> 4   [16,30) LBO >> 4   [32,46) SBO >> 4   [46,48) version = 1   [61,64) layout (2 = SW128)
// K-major operand (rows of 64 bf16 = 128 B, 8-row swizzle atoms): SBO = 1024 B, LBO unused (encoded 1).
// MN-major operand (each K index is one 128-B row of 64 MN elements): SBO = 1024 B (8 K rows),
//   LBO = byte distance between consecutive 64-element MN groups.
__device__ __forceinline__ uint64_t make_smem_desc_sw128(uint32_t smem_addr, uint32_t lbo_bytes,
                                                         uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFFu);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= 1ull << 46;
  d |= 2ull << 61;
  return d;
}

// TMEM -> registers: 32 lanes x 32 consecutive fp32 columns (thread i of the warp receives lane base+i).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// registers -> TMEM (same shape as tmem_ld_32x32)
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      :
      : "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]),
        "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]),
        "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------------------------------------------------------
// numerics
// ---------------------------------------------------------------------------------------------------------------
// LayerNorm statistics of a residual-stream row from its partial sums.  The kernels that WRITE the residual stream (token
// embedding, out-proj / c_proj epilogues) leave, per row and per group of 128 columns, (sum x, sum x^2) in
// stats[row * P + group] (P = ceil(d / 128)); the kernels that consume LN(row) — the QKV / c_fc GEMM epilogues with the
// LayerNorm folded into the weights, and the ln_f + pooling kernel — rebuild mean and 1/sqrt(var + eps) from them in a
// fixed summation order (deterministic).  rm = rstd * mean.
struct LnRow {
  float r, rm;
};
__device__ __forceinline__ LnRow ln_row_from_partials(const float2* __restrict__ stats, int P, float inv_d, float eps,
                                                      int row, int M) {
  float s1 = 0.f, s2 = 0.f;
  if (row < M) {
    const float2* s = stats + static_cast<size_t>(row) * P;
    for (int g = 0; g < P; ++g) {
      const float2 t = __ldg(s + g);
      s1 += t.x;
      s2 += t.y;
    }
  }
  const float mean = s1 * inv_d;
  const float var = fmaxf(s2 * inv_d - mean * mean, 0.f);
  LnRow o;
  o.r = rsqrtf(var + eps);
  o.rm = o.r * mean;
  return o;
}

// gelu_new(x) = 0.5 x (1 + tanh(sqrt(2/pi) (x + 0.044715 x^3)))   (HF activations.py NewGELUActivation)
__device__ __forceinline__ float gelu_new(float x) {
  const float k0 = 0.7978845608028654f, k1 = 0.044715f;
  float u = k0 * (x + k1 * x * x * x);
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(u));
  return 0.5f * x * (1.0f + t);
}

}  // namespace sgpt
