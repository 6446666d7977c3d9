// Thin inline-PTX wrappers for the sm_100a features the kernels use: mbarrier, TMA
// (cp.async.bulk.tensor), tcgen05 (MMA into TMEM, TMEM alloc/ld, commit) and the fences
// between the generic, async and tensor proxies.  sm_100a only -- no fallbacks.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace vqa {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "elect.sync _|p, 0xffffffff;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
// generic-proxy writes to smem -> visible to the async proxy (TMA / tcgen05 operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
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
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a pipeline bug must surface as a launch error (trap), never as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 8000000000LL) __trap();   // ~4 s at 2 GHz
  }
}

// ------------------------------------------------------------------ TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
// 2-D tiled load: c0 = coordinate along the contiguous (inner) dimension, c1 = outer.
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

// 3-D tiled load multicast to the CTAs of the cluster in `cta_mask`: ONE read of the box lands at the same shared-memory
// offset in every one of them and completes the transaction bytes on the barrier at the same offset in each.
__device__ __forceinline__ void tma_load_3d_multicast(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0,
                                                      int c1, int c2, uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, "
      "%4, %5}], [%2], %6;" ::"r"(smem_u32(smem_dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "h"(cta_mask)
      : "memory");
}

// 3-D tiled load (c2 = batch index); every operand of the GEMM kernel is described as [batch, outer, inner].
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1,
                                            int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// ------------------------------------------------------------------ tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {   // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {     // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc]; one thread issues for the CTA.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on an mbarrier when every previously issued tcgen05.mma of this thread has completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// TMEM -> registers, 32 lanes x 32 bit, 16 consecutive columns (thread t of the warp gets lane t)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ------------------------------------------------------------------ CTA pairs (cta_group::2)
// Two CTAs of a cluster (same TPC) execute ONE tcgen05.mma over a 256-row tile: each CTA holds its own 128 rows of
// A and HALF of the B tile in shared memory and its own 128 accumulator rows in TMEM; only the leader (rank 0)
// issues the MMA.  The B operand is then read once per pair instead of once per SM.
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_alloc_2cta(uint32_t* smem_dst, uint32_t ncols) {   // warp 1 of BOTH CTAs
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2cta(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_bf16_2cta(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// commit of the pair's MMAs: arrives on the barrier at the same smem offset in BOTH CTAs
__device__ __forceinline__ void umma_commit_2cta(uint64_t* bar) {
  const uint16_t mask = 0x3;
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(mask)
      : "memory");
}
// TMA load issued by either CTA of the pair; the transaction bytes are credited to the LEADER's barrier
// (bit 24 of a shared::cluster address selects the CTA of the pair).
__device__ __forceinline__ void tma_load_3d_2cta(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1,
                                                 int c2) {
  const uint32_t bar_leader = smem_u32(bar) & 0xFEFFFFFFu;
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, "
      "%5}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(map), "r"(bar_leader), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// arrive on the barrier at the same smem offset in CTA `cta` of the cluster
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t cta) {
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(bar)), "r"(cta));
  // default (.release.cta) semantics as CUTLASS' ClusterBarrier::arrive(cta): an explicit .release.cluster costs a
  // cluster-scope fence (~1400 cycles per k-block in the producer loop, measured)
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}

// ------------------------------------------------------------------ descriptors
// Shared-memory matrix descriptor (tcgen05): start>>4 [0,14), LBO>>4 [16,30), SBO>>4 [32,46),
// version=1 [46,48), layout type [61,64) (2 = SWIZZLE_128B).
__host__ __device__ __forceinline__ uint64_t umma_desc_hi(uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// Instruction descriptor for kind::f16 with bf16 operands and an fp32 accumulator.
__host__ __device__ __forceinline__ uint32_t umma_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
  uint32_t d = 0;
  d |= 1u << 4;                       // D format: f32
  d |= 1u << 7;                       // A format: bf16
  d |= 1u << 10;                      // B format: bf16
  d |= (uint32_t)(a_mn_major & 1) << 15;
  d |= (uint32_t)(b_mn_major & 1) << 16;
  d |= (uint32_t)(N >> 3) << 17;
  d |= (uint32_t)(M >> 4) << 24;
  return d;
}

// ------------------------------------------------------------------ small math helpers
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
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ float bf16_lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t u) { return __uint_as_float(u & 0xFFFF0000u); }

// Counter-based dropout mask (the fused-epilogue stand-in for nn.Dropout, mhb_coAtt.py:101):
// one 32-bit hash per PAIR of adjacent columns, 16 bits per element.  keep <=> bits >= thresh16.
__device__ __forceinline__ uint32_t dropout_bits(uint32_t seed, uint32_t row, uint32_t col_pair) {
  uint32_t x = seed ^ (row * 0x9E3779B1u);
  x += col_pair * 0x85EBCA77u;
  x ^= x >> 16; x *= 0x85EBCA6Bu;
  x ^= x >> 13; x *= 0xC2B2AE35u;
  x ^= x >> 16;
  return x;
}
// Device-side salt of a dropout seed.  Under CUDA-graph replay the host seed is baked into the captured launch; the
// per-step variation then comes from a device counter the graph itself increments (low 32 bits of the step count).
// salt == NULL: the host seed as it is (eager launches draw a fresh host seed per call).
__device__ __forceinline__ uint32_t effective_seed(uint32_t seed, const uint32_t* __restrict__ salt) {
  if (salt == nullptr) return seed;
  uint32_t x = seed + __ldg(salt) * 0x9E3779B9u;
  x ^= x >> 16; x *= 0x85EBCA6Bu;
  x ^= x >> 13; x *= 0xC2B2AE35u;
  x ^= x >> 16;
  return x;
}
__device__ __forceinline__ bool dropout_keep(uint32_t seed, uint32_t row, uint32_t col, uint32_t thresh16) {
  uint32_t b = dropout_bits(seed, row, col >> 1);
  uint32_t h = (col & 1) ? (b >> 16) : (b & 0xFFFFu);
  return h >= thresh16;
}

}  // namespace vqa
