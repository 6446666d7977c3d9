// Persistent single-layer LSTM recurrence (forward and backward) for the question encoder that feeds
// the question-attention stage (reference mhb_coAtt.py:69-75: nn.LSTM(batch_first=True) fed the
// [T, N, E] permutation of the embedded question, i.e. a recurrence of N steps over T "batch" rows).
//
// The recurrence is latency-bound: 2*Bt*4H*H flops per step (0.2 GFLOP at Bt=26, H=1024) behind a
// grid-wide dependency per step.  The stock path pays two kernel launches per step (a tf32 GEMM and
// an elementwise cell); here ONE persistent kernel per direction runs the whole sequence.  Each direction has a cluster
// form and a cluster-free form (forward: clusters of 4 CTAs sharing each fetch of h_{t-1} by TMA multicast, or every CTA
// sweeping it; backward: clusters of 4 CTAs splitting the contraction, each half of the grid running half of the batch
// rows, or single CTAs).  The cluster forms run unless cudaOccupancyMaxActiveClusters says their clusters cannot all be
// co-resident, or VQA_B200_LSTM_CLUSTERS=0 asks for the cluster-free pair:
//   * H/8 CTAs (128 at H=1024, one per SM), each owning 8 hidden units = 32 rows of W_hh (forward and single-CTA
//     backward), or, in the row-split backward, a share of the contraction for the 64 units of its cluster over half of
//     the rows (see lstm_bwd_rows_kernel);
//   * the CTA's slice of W_hh lives in REGISTERS for the whole sequence, already laid out as
//     mma.sync.m16n8k16 operand fragments (8 warps split the contraction; 64 registers per thread);
//   * the step-to-step exchange (h_t forward, dgates_t backward; bf16, through L2) carries its own
//     readiness: the buffers are pre-filled with the bf16 pattern 0xFFFF (a NaN no result is ever
//     stored as), producers write plain values with relaxed gpu-scope stores and every consumer warp
//     polls exactly the 16-byte pieces of ITS slice of the contraction until no lane holds the
//     sentinel.  No flags, no fences, no atomics (a first version with per-CTA step flags,
//     membar + st.release / ld.acquire, spent 1.7 us per step in the fences alone).  A consumer warp
//     spins on ONE 16-byte piece per producer CTA (the last batch row), then pulls its whole slice
//     with cp.async.cg and checks the operand fragments it feeds to the tensor cores for sentinels;
//     in the rare case a row had not landed yet it repeats the sweep;
//   * each warp runs the MMAs of its slice, the eight partial tiles meet in shared memory, and
//     thread (batch row, unit) applies the gate non-linearities, keeps c_t in a register and
//     publishes h_t; its x-projection / saved activations are fetched one step ahead;
//   * tensor cores through mma.sync (not tcgen05): a 32x32x1024 tile per CTA per step is far below
//     the 128-row tcgen05 tile and the TMA -> mbarrier -> MMA -> commit -> tcgen05.ld chain would
//     sit on the critical path of every step.
// The x-projection (x W_ih^T + b) and the weight gradients are plain large GEMMs and run on the
// tcgen05 kernel (gemm.cu) before / after these kernels.
#include <cuda_bf16.h>

#include <stdlib.h>
#include <string.h>

#include "common.h"
#include "ptx.cuh"

namespace vqa {
namespace {

constexpr int kU = 8;          // hidden units per CTA
constexpr int kThreads = 256;  // 8 warps, the contraction axis is split 8 ways
constexpr int kWarps = 8;
constexpr int kRows = 32;      // batch rows held per tile (Bt <= 32)

__device__ __forceinline__ uint32_t s_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];\n"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(s_u32(p))
               : "memory");
}
__device__ __forceinline__ void mma16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory");
}
__device__ __forceinline__ uint4 ld_relaxed_v4(const void* p) {
  uint4 v;
  asm volatile("ld.relaxed.gpu.global.v4.u32 {%0,%1,%2,%3}, [%4];\n"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(p)
               : "memory");
  return v;
}
// Publication of eight adjacent bf16 results as ONE 16-byte store.  The eight lanes eu = 0..7 of a row (tid = 8*row + eu)
// hold the eight units of their CTA: the values are gathered with four shuffles and lane eu == 0 stores them.  (Eight
// 2-byte stores into the same 16-byte piece were eight partial-sector writes for L2 to merge and up to eight chances for a
// consumer to sweep a half-written piece: 1.24 -> 1.19 ms per forward pass.)  Call with all 32 lanes converged.
__device__ __forceinline__ void publish8_bf16(__nv_bfloat16* dst, float x, bool store) {
  unsigned short u = __bfloat16_as_ushort(__float2bfloat16_rn(x));
  if (u == 0xFFFFu) u = 0x7FFFu;          // never store the sentinel itself
  const uint32_t v0 = u;
  const uint32_t pr = v0 | (__shfl_down_sync(0xFFFFFFFFu, v0, 1) << 16);       // units (eu, eu+1), valid on even eu
  const uint32_t p1 = __shfl_down_sync(0xFFFFFFFFu, pr, 2);
  const uint32_t q0 = __shfl_down_sync(0xFFFFFFFFu, pr, 4);
  const uint32_t q1 = __shfl_down_sync(0xFFFFFFFFu, p1, 4);
  if (store)
    asm volatile("st.relaxed.gpu.global.v4.u32 [%0], {%1,%2,%3,%4};\n" ::"l"(dst), "r"(pr), "r"(p1), "r"(q0), "r"(q1)
                 : "memory");
}
// bf16 lanes of a 32-bit word that still hold the sentinel (non-zero if any)
__device__ __forceinline__ uint32_t sentinel_lanes(uint32_t x) { return __vcmpeq2(x, 0xFFFFFFFFu); }
__device__ __forceinline__ bool has_sentinel(const uint4& v) {
  return (sentinel_lanes(v.x) | sentinel_lanes(v.y) | sentinel_lanes(v.z) | sentinel_lanes(v.w)) != 0u;
}
// Spin until the 16-byte piece at p holds no sentinel.  Bounded: a scheduling / indexing bug surfaces as a launch
// error, not as a hung GPU.
// (Backing off between polls with __nanosleep(10..160) was measured: 7 % slower -- the polls are not what the
// publications wait behind.)
__device__ __forceinline__ void spin_piece(const void* p) {
  const long long t0 = clock64();
  while (has_sentinel(ld_relaxed_v4(p))) {
    if (clock64() - t0 > 6000000000LL) __trap();
  }
}
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];\n" ::"l"(p)); }
__device__ __forceinline__ float sigmoidf_(float x) { return __fdividef(1.f, 1.f + __expf(-x)); }
__device__ __forceinline__ float tanhf_(float x) { return 1.f - __fdividef(2.f, 1.f + __expf(2.f * x)); }

// Debug hooks (tools/lstm_phase_probe.py): per-phase cycle counters of thread 0 of the first g_dbg_ctas CTAs (16 per
// CTA: [0..7] forward, [8..15] backward) and experiment switches.
unsigned long long* g_dbg = nullptr;
int g_dbg_ctas = 1;
int g_mode = 0;
enum { MODE_NOMMA = 2 };   // experiment switch: skip the MMAs (results are wrong; timing only)

__device__ __forceinline__ uint32_t cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;\n" : "=r"(r));
  return r;
}
// Cluster-wide barrier, full form (release/acquire): used once at start-up and once before exit.  It compiles to
// MEMBAR.ALL.GPU + CCTL.IVALL -- a fence that waits for every outstanding GLOBAL store of the SM and flushes L1 --
// which costs ~1 us when it sits inside the recurrence (measured), so the per-step exchange uses step_barrier below.
__device__ __forceinline__ void cluster_barrier() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}
// Per-step cluster barrier: bar.sync + RELAXED arrive + wait.  After bar.sync has ordered the CTA's st.shared, a
// peer's ld.shared::cluster issued after its wait reads the written values (shared memory has no cache in front of
// it), so the release fence is not needed.  (An mbarrier with remote arrives was measured too: 6 % slower.)
// The PTX memory model only PROMISES visibility of the peers' shared-memory writes with release / acquire on the cluster
// barrier (ADVICE r1); the relaxed form is what the hardware needs today and is 0.16 ms per backward pass faster.
// -DVQA_B200_LSTM_STRICT_BARRIER (VQA_B200_LSTM_STRICT_BARRIER=1 at build time) selects the guaranteed form, and
// tests/test_gpu_lstm.py::test_lstm_backward_variants_agree compares the row-split backward against the single-CTA kernel
// (no cluster exchange at all; VQA_B200_LSTM_CLUSTERS=0) at every supported hidden size, so a silent loss of
// visibility would show as a mismatch.
__device__ __forceinline__ void step_barrier() {
  __syncthreads();
#ifdef VQA_B200_LSTM_STRICT_BARRIER
  asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
#else
  asm volatile("barrier.cluster.arrive.relaxed.aligned;\n" ::: "memory");
  asm volatile("barrier.cluster.wait.aligned;\n" ::: "memory");
#endif
}
__device__ __forceinline__ float ld_dsmem_f32(const float* local_ptr, uint32_t rank) {
  uint32_t ra;
  float v;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;\n" : "=r"(ra) : "r"(s_u32(local_ptr)), "r"(rank));
  asm volatile("ld.shared::cluster.f32 %0, [%1];\n" : "=f"(v) : "r"(ra) : "memory");
  return v;
}

#ifdef VQA_B200_DEBUG
#define LSTM_PROF(a) ((a).dbg != nullptr && (int)blockIdx.x < (a).dbg_ctas && tid == 0)
#else
#define LSTM_PROF(a) false      /* release kernels carry no phase counters: every `if (prof)` is dead code */
#endif
#define LSTM_TICK(i) if (prof) { const long long n_ = clock64(); pc[i] += n_ - tk; tk = n_; }

// Dropout on the OUTPUT of the recurrence (`self.dropout_l(lstm_o)`, mhb_coAtt.py:74 / mfb.py:70), fused into the
// kernels: the forward stores h_t * mask / (1 - p) as its result (the recurrence itself and the saved bf16 states keep the
// clean h_t), the backward multiplies the incoming dL/d(output) by the same regenerated mask.  Mask element = counter
// hash of (seed', time-major row t * Bt + b, column j), as everywhere else (ptx.cuh); thresh16 == 0: no dropout.
struct LstmDrop {
  uint32_t thresh16;
  float scale;
  uint32_t seed;
  const uint32_t* seed_dev;
};
__device__ __forceinline__ float drop_out(float v, const LstmDrop& d, uint32_t dseed, uint32_t row, uint32_t col) {
  if (d.thresh16 == 0u) return v;
  return dropout_keep(dseed, row, col, d.thresh16) ? v * d.scale : 0.f;
}
LstmDrop make_drop(float p, uint32_t seed, const uint32_t* seed_dev) {
  LstmDrop d;
  d.thresh16 = (uint32_t)(p * 65536.0f + 0.5f);
  d.scale = d.thresh16 ? 65536.0f / (65536.0f - (float)d.thresh16) : 1.0f;
  d.seed = seed;
  d.seed_dev = seed_dev;
  return d;
}

// One warp's share of a recurrence step: acc[b, n] = sum_k X[b, k] Wslice[k, n] for the warp's contraction slice.
//   X      : rows of the exchange buffer (bf16, `src` = first column of the slice, `src_pitch` elements between rows);
//            pulled out of L2 with cp.async.cg in (up to) two column halves so that the tensor cores start on the
//            first half while the second is still in flight; staged in the warp's private shared-memory tile
//   Wslice : mma.m16n8k16 B fragments, n-tiles [0, NTR) resident in registers (wfr), n-tiles [NTR, NT) in shared
//            memory (wsm, [ks][nt - NTR][lane] as uint2: one conflict-free 8-byte load per lane)
// MT m-tiles of 16 rows (Bt <= 16 * MT).  The A fragments ldmatrix returns are checked for the 0xFFFF "not written yet"
// mark; returns the number of repeated sweeps (0 in the common case).
template <int KSTEPS, int NT, int MT, int NTR>
__device__ __forceinline__ int sweep_mma(float (&acc)[MT][NT][4], const uint32_t (&wfr)[KSTEPS][NTR][2],
                                         __nv_bfloat16* stage, const __nv_bfloat16* src, size_t src_pitch, int Bt,
                                         int lane, bool skip_mma, const uint2* wsm = nullptr) {
  constexpr int PITCH = KSTEPS * 16 + 8;
  constexpr int NH = KSTEPS >= 2 ? 2 : 1;
  constexpr int KH = KSTEPS / NH;
  constexpr int PR = KH * 2;             // 16-byte pieces per row and half (a power of two <= 32)
  constexpr int RPI = 32 / PR;           // rows covered by one warp-wide cp.async
  // ldmatrix.x4 = one 16x16 A tile: (rows 0-7, k 0-7), (rows 8-15, k 0-7), (rows 0-7, k 8-15), (rows 8-15, k 8-15)
  const int lm_row = (lane & 7) + (((lane >> 3) & 1) << 3);
  const int lm_k = (lane >> 4) * 8;
  const int prow = lane / PR, pcol = lane % PR;
  const __nv_bfloat16* gsrc = src + (size_t)prow * src_pitch + pcol * 8;
  __nv_bfloat16* sdst = stage + prow * PITCH + pcol * 8;
  int tries = 0;
  for (;;) {
#pragma unroll
    for (int hf = 0; hf < NH; ++hf) {
#pragma unroll
      for (int j = 0; j < PR; ++j)
        if (j * RPI < MT * 16 && prow + j * RPI < Bt)
          cp_async16(sdst + j * RPI * PITCH + hf * KH * 16, gsrc + (size_t)(j * RPI) * src_pitch + hf * KH * 16);
      cp_async_commit();
    }
#pragma unroll
    for (int mt = 0; mt < MT; ++mt)
#pragma unroll
      for (int nt = 0; nt < NT; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[mt][nt][e] = 0.f;
    uint32_t top = 0u;                   // per-halfword unsigned maximum of every operand word: 0xFFFF <=> sentinel seen
#pragma unroll
    for (int hf = 0; hf < NH; ++hf) {
      if (hf == 0 && NH == 2) cp_async_wait<1>(); else cp_async_wait<0>();
      __syncwarp();
      uint32_t afr[KH][MT][4];
#pragma unroll
      for (int ks = 0; ks < KH; ++ks)
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
          if (mt * 16 < Bt) {
            ldmatrix_x4(afr[ks][mt], stage + (mt * 16 + lm_row) * PITCH + (hf * KH + ks) * 16 + lm_k);
            top = __vimax3_u16x2(top, afr[ks][mt][0], afr[ks][mt][1]);
            top = __vimax3_u16x2(top, afr[ks][mt][2], afr[ks][mt][3]);
          }
      if (!skip_mma)
#pragma unroll
      for (int ks = 0; ks < KH; ++ks)
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
          if (mt * 16 < Bt)
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
              if (nt < NTR) {
                mma16816(acc[mt][nt], afr[ks][mt], wfr[hf * KH + ks][nt < NTR ? nt : 0][0],
                         wfr[hf * KH + ks][nt < NTR ? nt : 0][1]);
              } else {
                const uint2 b = wsm[((hf * KH + ks) * (NT - NTR) + (nt - NTR)) * 32 + lane];
                mma16816(acc[mt][nt], afr[ks][mt], b.x, b.y);
              }
            }
    }
    if (!__any_sync(0xFFFFFFFFu, sentinel_lanes(top) != 0u)) return tries;
    if (++tries > (1 << 22)) __trap();
  }
}

// Byte offset of 16-byte chunk c of row r in a TMA box of RB-byte rows written with SWIZZLE_<RB>B (box base 1024-byte
// aligned): bits [4, 4 + log2(RB/16)) of the offset are XORed with the bits above bit 7.
template <int RB>
__device__ __forceinline__ uint32_t swz(int r, int c) {
  const uint32_t o = (uint32_t)(r * RB + c * 16);
  return o ^ (((o >> 7) & (uint32_t)(RB / 16 - 1)) << 4);
}

// The multicast counterpart of sweep_mma: the warp's slice arrives by TMA in NH boxes (column halves, RB bytes per row,
// 32-row tiles) that complete `full[hf]`; the MMAs run in exactly sweep_mma's order on exactly its operands, so the
// accumulators are bit-identical.  Returns whether any operand still held the 0xFFFF sentinel.
template <int KSTEPS, int NT>
__device__ __forceinline__ bool mcast_mma(float (&acc)[2][NT][4], const uint32_t (&wfr)[KSTEPS][NT][2],
                                          const unsigned char* stage, uint64_t* full, uint32_t phase, int Bt, int lane,
                                          bool skip_mma) {
  constexpr int NH = KSTEPS >= 2 ? 2 : 1;
  constexpr int KH = KSTEPS / NH;
  constexpr int RB = KH * 32;
  const int lm_row = (lane & 7) + (((lane >> 3) & 1) << 3);
  const int lm_c = lane >> 4;
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[mt][nt][e] = 0.f;
  uint32_t top = 0u;
#pragma unroll
  for (int hf = 0; hf < NH; ++hf) {
    mbar_wait(full + hf, phase);
    const unsigned char* tile = stage + hf * 32 * RB;
    uint32_t afr[KH][2][4];
#pragma unroll
    for (int ks = 0; ks < KH; ++ks)
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
        if (mt * 16 < Bt) {
          ldmatrix_x4(afr[ks][mt], tile + swz<RB>(mt * 16 + lm_row, ks * 2 + lm_c));
          top = __vimax3_u16x2(top, afr[ks][mt][0], afr[ks][mt][1]);
          top = __vimax3_u16x2(top, afr[ks][mt][2], afr[ks][mt][3]);
        }
    if (!skip_mma)
#pragma unroll
    for (int ks = 0; ks < KH; ++ks)
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
        if (mt * 16 < Bt)
#pragma unroll
          for (int nt = 0; nt < NT; ++nt)
            mma16816(acc[mt][nt], afr[ks][mt], wfr[hf * KH + ks][nt][0], wfr[hf * KH + ks][nt][1]);
  }
  return __any_sync(0xFFFFFFFFu, sentinel_lanes(top) != 0u);
}

struct LstmFwdArgs {
  float* gates;                // in: x W_ih^T + b_ih + b_hh  [S, Bt, 4H]; out (training): activated gates i,f,g,o
  const __nv_bfloat16* whh;    // [4H, H]
  float* out;                  // h_t  [S, Bt, H]
  __nv_bfloat16* hb;           // exchange buffer [S+1, Bt, H]: hb[0] = h_{-1} = 0, hb[1..] = 0xFFFF sentinels on entry
  float* c_all;                // [S, Bt, H] cell states (training) or nullptr
  int S, Bt, H;
  unsigned long long* dbg;     // optional phase counters (debug): 16 per CTA, [0..7] forward, [8..15] backward
  int dbg_ctas;                // CTAs whose thread 0 records them (the rows dbg holds)
  int mode;
  LstmDrop drop;               // dropout applied to `out` only
};

// Shared memory of the forward kernel.  CL == 1 (sweep): one padded tile per warp, then the partial tiles.  CL > 1
// (multicast): 1024-byte aligned TMA tiles [step parity][warp][column half] of 32 rows x RB bytes, the partial tiles,
// the `full` barriers [parity][warp][half] and the `empty` barriers [warp].
template <int KS, int CL>
struct FwdSmem {
  static constexpr int NH = KS >= 2 ? 2 : 1;
  static constexpr int RB = KS / NH * 32;                  // bytes per row of one TMA box
  static constexpr int TILE = 32 * RB;                     // bytes of one box tile
  static constexpr size_t STAGE = CL == 1 ? (size_t)kWarps * kRows * (KS * 16 + 8) * 2 : (size_t)2 * kWarps * NH * TILE;
  static constexpr size_t RED = STAGE;
  static constexpr size_t BARS = RED + (size_t)kWarps * 32 * 40 * 4;
  static constexpr size_t BYTES = CL == 1 ? BARS : BARS + (size_t)(2 * kWarps * NH + kWarps) * 8 + 1024;
};

// KS = k-steps (of 16) of one warp's contraction slice: H = 128 * KS.
// Tile orientation: M = batch rows (2 m-tiles), N = the CTA's 32 gate rows in the order n = 4*unit + gate, so that the
// four gate pre-activations of one (row, unit) are adjacent in the partial tiles (one 128-bit read per warp-partial).
//
// CL > 1: multicast exchange.  The grid runs in clusters of CL CTAs, and warp w's slice of h_{t-1} (the same bytes for
// every CTA) is fetched ONCE per cluster: warp w of the cluster's rank w % CL CTA (the slice's owner) polls the slice's
// producers exactly as the sweep does, then issues the slice's TMA boxes multicast to the whole cluster; warp w of every
// CTA waits on its own `full` barrier.  L2 reads and polls per step drop by the factor CL.  Every CTA receives the same
// bytes, so all of them reach the same verdict on the sentinel check: on a hit each CTA re-arms its barrier and tells the
// owner (remote arrive on the owner's `empty` barrier) that it is done reading the buffer, and the owner re-issues the
// load once all CL have done so.
// Buffers alternate by step parity.  The multicast of step t + 2 into a peer's parity-(t & 1) tile cannot overtake that
// peer's reads of step t: the owner issues it only after it has seen h_{t+1} of the slice's producers, those needed the
// peer's h_t, and the peer publishes h_t after the __syncthreads that follows every one of its warps' reads of step t.
template <int KS, int CL>
__global__ void __launch_bounds__(kThreads, 1) lstm_fwd_kernel(const LstmFwdArgs a, const __grid_constant__ CUtensorMap hmap) {
  using SM = FwdSmem<KS, CL>;
  constexpr int PITCH = KS * 16 + 8;     // bf16 elements; (PITCH/2) % 8 == 4 -> conflict-free ldmatrix
  constexpr int RP = 40;                 // floats per batch row of a partial tile: 8*b + n is conflict-free
  constexpr int NPROD = 2 * KS;          // CTAs that produce one warp's slice of h
  constexpr int NH = SM::NH;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned char* smem = CL == 1 ? smem_raw : smem_raw + ((1024u - (s_u32(smem_raw) & 1023u)) & 1023u);
  __nv_bfloat16* hs = reinterpret_cast<__nv_bfloat16*>(smem);
  float* red = reinterpret_cast<float*>(smem + SM::RED);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + SM::BARS);
  uint64_t* empty = full + 2 * kWarps * NH;

  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, g = lane >> 2, tg = lane & 3;
  const int H = a.H, Bt = a.Bt;
  const int j0 = blockIdx.x * kU;
  const int kw = w * KS * 16;            // first contraction index of this warp
  const uint32_t owner = (uint32_t)(w % CL);
  const bool own = CL > 1 && cluster_rank() == owner;

  // rows >= Bt of the tiles are never written and must read as zero
  for (int i = tid; i < (int)(SM::STAGE / 4); i += kThreads) reinterpret_cast<uint32_t*>(hs)[i] = 0u;
  if constexpr (CL > 1) {
    if (tid == 0) {
      for (int i = 0; i < 2 * kWarps * NH; ++i) mbar_init(full + i, 1);
      for (int i = 0; i < kWarps; ++i) mbar_init(empty + i, CL);
      fence_mbar_init();
    }
    fence_proxy_async_smem();
    __syncthreads();
    if (lane == 0)
      for (int i = 0; i < 2 * NH; ++i) mbar_expect_tx(full + ((i / NH) * kWarps + w) * NH + i % NH, (uint32_t)(Bt * SM::RB));
    if (own && lane == 0) tma_prefetch_desc(&hmap);
    cluster_barrier();                   // every barrier of the cluster is armed before the first multicast lands
  }

  // W_hh slice as B fragments: column n = nt*8 + g of the tile is gate (n & 3) of unit (n >> 2)
  uint32_t wfr[KS][4][2];
#pragma unroll
  for (int ks = 0; ks < KS; ++ks)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      const int n = nt * 8 + g;
      const __nv_bfloat16* p = a.whh + (size_t)((n & 3) * H + j0 + (n >> 2)) * H + kw + ks * 16 + 2 * tg;
      wfr[ks][nt][0] = *reinterpret_cast<const uint32_t*>(p);
      wfr[ks][nt][1] = *reinterpret_cast<const uint32_t*>(p + 8);
    }
  __syncthreads();

  __nv_bfloat16* hw = hs + (size_t)w * kRows * PITCH;
  float* redw = red + w * 32 * RP;
  const int eb = tid >> 3, eu = tid & 7;            // epilogue role: (batch row, unit)
  const bool active = eb < Bt;
  float c = 0.f;
  const bool prof = LSTM_PROF(a);
  long long pc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tk = 0;
  const uint32_t dseed = a.drop.thresh16 ? effective_seed(a.drop.seed, a.drop.seed_dev) : 0u;

  // x-projection of the thread's (row, unit), fetched one step ahead of its use
  float xq[4] = {0.f, 0.f, 0.f, 0.f};
  if (active) {
    const float* gp0 = a.gates + (size_t)eb * 4 * H + j0 + eu;
#pragma unroll
    for (int q = 0; q < 4; ++q) xq[q] = __ldcs(gp0 + (size_t)q * H);
  }

  uint32_t ph = 0u, eph = 0u;           // multicast: phase bits of the warp's `full` barriers (bit = parity), `empty`
  for (int t = 0; t < a.S; ++t) {
    if (prof) tk = clock64();
    const __nv_bfloat16* src = a.hb + (size_t)t * Bt * H + kw;
    // ---- wait for h_{t-1}: each lane watches the LAST row's piece of one producer CTA of this warp's slice
    if (t > 0 && (CL == 1 || own)) {
      if (lane < NPROD) spin_piece(src + (size_t)(Bt - 1) * H + lane * 8);
      __syncwarp();
    }
    LSTM_TICK(0)
    float acc[2][4][4];
    int tries = 0;
    if constexpr (CL == 1) {
      tries = sweep_mma<KS, 4>(acc, wfr, hw, src, (size_t)H, Bt, lane, (a.mode & MODE_NOMMA) != 0);
    } else {
      const int p = t & 1;
      unsigned char* tiles = smem + (size_t)(p * kWarps + w) * NH * SM::TILE;
      uint64_t* fb = full + (p * kWarps + w) * NH;
      auto issue = [&]() {
        if (own && lane == 0)
#pragma unroll
          for (int hf = 0; hf < NH; ++hf)
            tma_load_3d_multicast(tiles + hf * SM::TILE, &hmap, fb + hf, kw + hf * (KS / NH) * 16, t * Bt, 0,
                                  (uint16_t)((1u << CL) - 1u));
      };
      issue();
      for (;;) {
        const bool bad = mcast_mma<KS, 4>(acc, wfr, tiles, fb, (ph >> p) & 1u, Bt, lane, (a.mode & MODE_NOMMA) != 0);
        ph ^= 1u << p;
        if (lane == 0)                   // arm the next delivery into this buffer: the retry, or step t + 2
          for (int hf = 0; hf < NH; ++hf) mbar_expect_tx(fb + hf, (uint32_t)(Bt * SM::RB));
        if (!bad) break;
        if (++tries > (1 << 22)) __trap();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(empty + w, owner);
        if (own) {
          mbar_wait(empty + w, eph);
          eph ^= 1u;
          issue();
        }
      }
    }
    if (prof) pc[7] += tries;
    LSTM_TICK(1)
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        const int r = mt * 16 + g, nc = nt * 8 + 2 * tg;
        *reinterpret_cast<float2*>(redw + r * RP + nc) = make_float2(acc[mt][nt][0], acc[mt][nt][1]);
        *reinterpret_cast<float2*>(redw + (r + 8) * RP + nc) = make_float2(acc[mt][nt][2], acc[mt][nt][3]);
      }
    LSTM_TICK(2)
    __syncthreads();
    LSTM_TICK(3)
    float gi = 0.f, gf = 0.f, gg = 0.f, go = 0.f, h = 0.f;
    if (active) {
      float4 pre = make_float4(xq[0], xq[1], xq[2], xq[3]);
#pragma unroll
      for (int ww = 0; ww < kWarps; ++ww) {
        const float4 v = *reinterpret_cast<const float4*>(red + (ww * 32 + eb) * RP + 4 * eu);
        pre.x += v.x; pre.y += v.y; pre.z += v.z; pre.w += v.w;
      }
      gi = sigmoidf_(pre.x); gf = sigmoidf_(pre.y); gg = tanhf_(pre.z); go = sigmoidf_(pre.w);
      c = gf * c + gi * gg;
      h = go * tanhf_(c);
    }
    // publish first: this is what the other CTAs wait for
    publish8_bf16(a.hb + ((size_t)(t + 1) * Bt + eb) * H + j0, h, active && eu == 0);
    if (active) {
      LSTM_TICK(4)
      const size_t o = ((size_t)t * Bt + eb) * H + j0 + eu;
      a.out[o] = drop_out(h, a.drop, dseed, (uint32_t)(t * Bt + eb), (uint32_t)(j0 + eu));
      float* gp = a.gates + ((size_t)t * Bt + eb) * 4 * H + j0 + eu;
      if (a.c_all != nullptr) {
        gp[0] = gi;
        gp[(size_t)H] = gf;
        gp[(size_t)2 * H] = gg;
        gp[(size_t)3 * H] = go;
        a.c_all[o] = c;
      }
      if (t + 1 < a.S) {
        gp += (size_t)Bt * 4 * H;
#pragma unroll
        for (int q = 0; q < 4; ++q) xq[q] = __ldcs(gp + (size_t)q * H);
      }
      LSTM_TICK(5)
    }
    __syncthreads();               // the partial tiles are re-written by the next step's MMAs
    LSTM_TICK(6)
  }
  if constexpr (CL > 1) cluster_barrier();   // no CTA exits while its multicasts or a peer's arrives may be in flight
  if (prof)
    for (int i = 0; i < 8; ++i) a.dbg[(size_t)blockIdx.x * 16 + i] = (unsigned long long)pc[i];
}

struct LstmBwdArgs {
  const float* gates;            // activated gates i,f,g,o  [S, Bt, 4H]
  const float* c_all;            // [S, Bt, H]
  const float* dout;             // dL/dh_t from above: element (t, b, j) at dout[t * dout_st + b * dout_sb + j]
  const __nv_bfloat16* whhT;     // w_layout 0: W_hh^T [H, 4H];  w_layout 1: W_hh itself [4H, H] (the parameter's layout)
  __nv_bfloat16* dg;             // exchange buffer + result: dL/d(pre-activation gates) [S, Bt, 4H], 0xFFFF on entry
  int S, Bt, H;
  unsigned long long* dbg;
  int dbg_ctas;
  int mode;
  long long dout_st, dout_sb;    // strides of dout in elements (the gradient arrives in the caller's [Bt, S, H] order)
  int w_layout;
  LstmDrop drop;                 // the forward's output dropout: dout is multiplied by the same mask
};

// Two consecutive contraction elements (gate columns k, k+1) of unit `unit` as one B-fragment word, from either layout of
// the recurrent weight.  Loaded once per kernel: reading the parameter's own [4H, H] layout saves the per-step transposed
// copy (8 MB, 22 us) the [H, 4H] form needed.
__device__ __forceinline__ uint32_t ld_w_pair(const __nv_bfloat16* w, int layout, size_t unit, size_t k, int H) {
  if (layout == 0) return *reinterpret_cast<const uint32_t*>(w + unit * 4 * H + k);
  const uint32_t lo = *reinterpret_cast<const uint16_t*>(w + k * H + unit);
  const uint32_t hi = *reinterpret_cast<const uint16_t*>(w + (k + 1) * H + unit);
  return lo | (hi << 16);
}

template <int KS>
__global__ void __launch_bounds__(kThreads, 1) lstm_bwd_kernel(const LstmBwdArgs a) {
  constexpr int PITCH = KS * 16 + 8;
  constexpr int NSUB = 4;                // a warp's slice (H/2 gate columns) is streamed in 4 pieces of KS k-steps
  constexpr int NPROD = 8 * KS;          // CTAs that produce one warp's slice of dgates
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __nv_bfloat16* ds = reinterpret_cast<__nv_bfloat16*>(smem_raw);
  float* red = reinterpret_cast<float*>(smem_raw + (size_t)kWarps * 2 * kRows * PITCH * 2);

  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, g = lane >> 2, tg = lane & 3;
  const int H = a.H, Bt = a.Bt, S = a.S;
  const int j0 = blockIdx.x * kU;
  const int kw = w * (H / 2);            // first gate column of this warp's contraction slice

  for (int i = tid; i < kWarps * 2 * kRows * PITCH / 2; i += kThreads) reinterpret_cast<uint32_t*>(ds)[i] = 0u;

  // W_hh[k, j0+g] for the warp's k-slice as B fragments (n = unit, k = gate column)
  uint32_t bfr[NSUB * KS][2];
#pragma unroll
  for (int kk = 0; kk < NSUB * KS; ++kk) {
    const size_t kq = (size_t)kw + kk * 16 + 2 * tg;
    bfr[kk][0] = ld_w_pair(a.whhT, a.w_layout, (size_t)(j0 + g), kq, H);
    bfr[kk][1] = ld_w_pair(a.whhT, a.w_layout, (size_t)(j0 + g), kq + 8, H);
  }
  __syncthreads();

  __nv_bfloat16* dw = ds + (size_t)w * 2 * kRows * PITCH;
  const int eb = tid >> 3, eu = tid & 7;
  const bool active = eb < Bt;
  const int nchunk = Bt * KS * 2;
  // ldmatrix.x4 = one 16x16 A tile: (rows 0-7, k 0-7), (rows 8-15, k 0-7), (rows 0-7, k 8-15), (rows 8-15, k 8-15)
  const int lm_row = (lane & 7) + (((lane >> 3) & 1) << 3);
  const int lm_k = (lane >> 4) * 8;
  float dc = 0.f;
  const bool prof = LSTM_PROF(a);
  long long pc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tk = 0;
  const uint32_t dseed = a.drop.thresh16 ? effective_seed(a.drop.seed, a.drop.seed_dev) : 0u;

  // saved activations of the thread's (row, unit) for step t, fetched one step ahead of their use
  float gi = 0.f, gf = 0.f, gg = 0.f, go = 0.f, ct = 0.f, cprev = 0.f, dh = 0.f;
  auto fetch = [&](int t) {
    const size_t row = (size_t)t * Bt + eb;
    const size_t o = row * H + j0 + eu;
    const float* gp = a.gates + row * 4 * H + j0 + eu;
    gi = __ldcs(gp);
    gf = __ldcs(gp + (size_t)H);
    gg = __ldcs(gp + (size_t)2 * H);
    go = __ldcs(gp + (size_t)3 * H);
    ct = __ldcs(a.c_all + o);
    cprev = t > 0 ? __ldcs(a.c_all + o - (size_t)Bt * H) : 0.f;
    dh = drop_out(__ldcs(a.dout + (size_t)t * a.dout_st + (size_t)eb * a.dout_sb + j0 + eu), a.drop, dseed,
                  (uint32_t)row, (uint32_t)(j0 + eu));
  };
  if (active) fetch(S - 1);

  for (int t = S - 1; t >= 0; --t) {
    if (prof) tk = clock64();
    if (t < S - 1) {
      // ---- dh_t += dgates_{t+1} W_hh: wait for the producers of this warp's slice (last row's pieces), then stream it
      const __nv_bfloat16* src = a.dg + (size_t)(t + 1) * Bt * 4 * H + kw;
#pragma unroll 1
      for (int i = lane; i < NPROD; i += 32) spin_piece(src + (size_t)(Bt - 1) * 4 * H + i * 8);
      __syncwarp();
      LSTM_TICK(0)
      auto issue = [&](int sub) {
        __nv_bfloat16* buf = dw + (sub & 1) * kRows * PITCH;
        const __nv_bfloat16* ssrc = src + sub * KS * 16;
#pragma unroll 1
        for (int i = lane; i < nchunk; i += 32) {
          const int r = i / (KS * 2), col = i % (KS * 2);
          cp_async16(buf + r * PITCH + col * 8, ssrc + (size_t)r * 4 * H + col * 8);
        }
        cp_async_commit();
      };
      float acc[2][4];
      int tries = 0;
      for (;;) {
        issue(0);
        issue(1);
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
          for (int e = 0; e < 4; ++e) acc[mt][e] = 0.f;
        uint32_t bad = 0u;
#pragma unroll
        for (int sub = 0; sub < NSUB; ++sub) {
          if (sub < NSUB - 1) cp_async_wait<1>(); else cp_async_wait<0>();
          __syncwarp();
          const __nv_bfloat16* buf = dw + (sub & 1) * kRows * PITCH;
          if (!(a.mode & MODE_NOMMA))
#pragma unroll
          for (int ks = 0; ks < KS; ++ks) {
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) {
              if (mt * 16 < Bt) {
                uint32_t afr[4];
                ldmatrix_x4(afr, buf + (mt * 16 + lm_row) * PITCH + ks * 16 + lm_k);
                bad |= sentinel_lanes(afr[0]) | sentinel_lanes(afr[1]) | sentinel_lanes(afr[2]) | sentinel_lanes(afr[3]);
                mma16816(acc[mt], afr, bfr[sub * KS + ks][0], bfr[sub * KS + ks][1]);
              }
            }
          }
          __syncwarp();
          if (sub + 2 < NSUB) issue(sub + 2);
        }
        if (!__any_sync(0xFFFFFFFFu, bad != 0u)) break;
        if (++tries > (1 << 22)) __trap();
      }
      if (prof) pc[7] += tries;
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) {
        const int r = mt * 16 + g;
        *reinterpret_cast<float2*>(red + (w * 32 + r) * 8 + 2 * tg) = make_float2(acc[mt][0], acc[mt][1]);
        *reinterpret_cast<float2*>(red + (w * 32 + r + 8) * 8 + 2 * tg) = make_float2(acc[mt][2], acc[mt][3]);
      }
      LSTM_TICK(2)
      __syncthreads();
      LSTM_TICK(3)
      if (active) {
#pragma unroll
        for (int ww = 0; ww < kWarps; ++ww) dh += red[(ww * 32 + eb) * 8 + eu];
      }
    }
    float d_i = 0.f, d_f = 0.f, d_g = 0.f, d_o = 0.f;
    if (active) {
      const float tc = tanhf_(ct);
      d_o = dh * tc * go * (1.f - go);
      const float dct = dc + dh * go * (1.f - tc * tc);
      d_i = dct * gg * gi * (1.f - gi);
      d_g = dct * gi * (1.f - gg * gg);
      d_f = dct * cprev * gf * (1.f - gf);
      dc = dct * gf;
    }
    {
      // one 16-byte publication per gate plane and row (see publish8_bf16)
      __nv_bfloat16* dp = a.dg + ((size_t)t * Bt + (active ? eb : 0)) * 4 * H + j0;
      const bool st_ = active && eu == 0;
      publish8_bf16(dp, d_i, st_);
      publish8_bf16(dp + (size_t)H, d_f, st_);
      publish8_bf16(dp + (size_t)2 * H, d_g, st_);
      publish8_bf16(dp + (size_t)3 * H, d_o, st_);
    }
    if (active) {
      LSTM_TICK(4)
      if (t > 0) fetch(t - 1);
      LSTM_TICK(5)
    }
    __syncthreads();
    LSTM_TICK(6)
  }
  if (prof)
    for (int i = 0; i < 8; ++i) a.dbg[(size_t)blockIdx.x * 16 + 8 + i] = (unsigned long long)pc[i];
}

// ---------------------------------------------------------------------------------------------------------------
// Backward recurrence, row-split cluster version.  dh_{t-1}[b, j] = sum_k dgates_t[b, k] W_hh[k, j] contracts over 4H
// gate columns for only H outputs: with one CTA per 8 units (lstm_bwd_kernel) every CTA has to pull ALL of dgates_t out
// of L2 per step.  Here a cluster of 4 CTAs splits the contraction (CTA rank r takes gate plane r), every CTA computes
// partial sums for all the cluster's units, and the 4 partial tiles meet through distributed shared memory: one
// barrier.cluster per step.  A cluster reads Bt * 4H * 2 bytes of dgates_t per step whatever it does inside, so total
// L2 traffic per step is that times the number of clusters, i.e. inversely proportional to the units a cluster owns.
// The Bt batch rows are independent recurrences, so the grid is split into two halves that each run half of the rows:
// cluster (G, h) owns the 64 units [64G, 64G + 64) for row half h (rows [0, ceil(Bt/2)) or [ceil(Bt/2), Bt)).  At
// Bt = 1 the grid is the first half only.  Each CTA computes partial sums for the 64 units over one 16-row m-tile, and
// owns 16 units for the gate math and publication (two 16-byte pieces per gate plane and row).  A row's element is
// computed the same way whichever m-tile row or half it sits in, so a row's dgates do not depend on the rows run beside
// it.
// Each warp holds B fragments for 8 n-tiles; where they do not all fit in registers (KS = 8) n-tiles 4..7 live in
// shared memory in lane order.
// ---------------------------------------------------------------------------------------------------------------
template <int KS>
struct BwdRowsSmem {
  static constexpr int NTR = KS <= 4 ? 8 : 4;       // n-tiles whose B fragments stay in registers
  static constexpr int PITCH = KS * 16 + 8;         // bf16 elements per operand tile row (conflict-free ldmatrix)
  static constexpr int RP = 64 + 8;                 // floats per row of the partial tiles (conflict-free, see below)
  static constexpr size_t RED = (size_t)kWarps * 16 * PITCH * 2;          // after the operand tiles [warp][16][PITCH]
  static constexpr size_t PART = RED + (size_t)kWarps * 16 * RP * 4;      // after the warp partials [warp][16][RP]
  static constexpr size_t WSM = PART + (size_t)2 * 16 * RP * 4;           // after the CTA partials [parity][16][RP]
  static constexpr size_t BYTES = WSM + (size_t)kWarps * KS * (8 - NTR) * 32 * 8;   // B fragments [warp][ks][nt][lane]
};

template <int KS>
__global__ void __launch_bounds__(kThreads, 1) lstm_bwd_rows_kernel(const LstmBwdArgs a) {
  using SM = BwdRowsSmem<KS>;
  constexpr int NTR = SM::NTR, PITCH = SM::PITCH, RP = SM::RP;
  constexpr int NPROD = 2 * KS;          // 16-byte pieces of one row of a warp's slice (two per producer CTA)
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __nv_bfloat16* ds = reinterpret_cast<__nv_bfloat16*>(smem_raw);
  float* red = reinterpret_cast<float*>(smem_raw + SM::RED);
  float* part = reinterpret_cast<float*>(smem_raw + SM::PART);

  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, g = lane >> 2, tg = lane & 3;
  const int H = a.H, Bt = a.Bt, S = a.S;
  const uint32_t rank = cluster_rank();
  const int ng = H / 64;                             // unit groups per row half
  const int cid = blockIdx.x / 4;
  const int u0 = (cid % ng) * 64;                    // first unit of the cluster
  const int j0 = u0 + (int)rank * 16;                // own units (gate math, dgates output)
  const int rh = (Bt + 1) / 2;
  const int r0 = cid < ng ? 0 : rh, nr = cid < ng ? rh : Bt - rh;   // the cluster's rows
  const int kw = (int)rank * H + w * KS * 16;        // first gate column of this warp's contraction slice

  for (int i = tid; i < (int)(SM::RED / 4); i += kThreads) reinterpret_cast<uint32_t*>(ds)[i] = 0u;

  // W_hh[k, u0 + nt*8 + g] for the warp's k-slice as B fragments (n = unit, k = gate column)
  uint32_t bfr[KS][NTR][2];
  uint2* wsm = reinterpret_cast<uint2*>(smem_raw + SM::WSM) + (size_t)w * KS * (8 - NTR) * 32;
#pragma unroll
  for (int ks = 0; ks < KS; ++ks) {
    const size_t kq = (size_t)kw + ks * 16 + 2 * tg;
#pragma unroll
    for (int nt = 0; nt < NTR; ++nt) {
      bfr[ks][nt][0] = ld_w_pair(a.whhT, a.w_layout, (size_t)(u0 + nt * 8 + g), kq, H);
      bfr[ks][nt][1] = ld_w_pair(a.whhT, a.w_layout, (size_t)(u0 + nt * 8 + g), kq + 8, H);
    }
#pragma unroll
    for (int nt = NTR; nt < 8; ++nt)
      wsm[(ks * (8 - NTR) + nt - NTR) * 32 + lane] =
          make_uint2(ld_w_pair(a.whhT, a.w_layout, (size_t)(u0 + nt * 8 + g), kq, H),
                     ld_w_pair(a.whhT, a.w_layout, (size_t)(u0 + nt * 8 + g), kq + 8, H));
  }
  __syncthreads();

  __nv_bfloat16* dw = ds + (size_t)w * 16 * PITCH;
  float* redw = red + w * 16 * RP;
  const int eb = tid >> 4, eu = tid & 15;            // gate-math role: (row of the half, unit)
  const int b = r0 + eb;
  const bool active = eb < nr;
  // CTA-reduction role: row (tid >> 3) & 15, units (2 jj + (tid >> 7)) * 8 + (tid & 7): a warp reads 4 rows x 8 units,
  // banks 8 * row + unit (RP % 32 == 8), conflict-free
  const int qr = (tid >> 3) & 15, qu = ((tid >> 7) << 3) + (tid & 7);
  float dc = 0.f;
  const bool prof = LSTM_PROF(a);
  long long pc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tk = 0;
  const uint32_t dseed = a.drop.thresh16 ? effective_seed(a.drop.seed, a.drop.seed_dev) : 0u;

  // The saved activations of the thread's (row, unit) are pulled into L2 one step ahead (prefetch.global.L2) and read
  // at the top of their step, long before the gate math needs them.  (Loading them into registers a step ahead made
  // the compiler park each value with a MOV right behind its load: a full DRAM latency, 15 % of the kernel.)
  auto prefetch = [&](int t) {
    const size_t row = (size_t)t * Bt + b;
    const size_t o = row * H + j0 + eu;
    const float* gp = a.gates + row * 4 * H + j0 + eu;
    prefetch_l2(gp);
    prefetch_l2(gp + (size_t)H);
    prefetch_l2(gp + (size_t)2 * H);
    prefetch_l2(gp + (size_t)3 * H);
    prefetch_l2(a.c_all + o);
    prefetch_l2(a.dout + (size_t)t * a.dout_st + (size_t)b * a.dout_sb + j0 + eu);
  };
  if (active && (eu & 7) == 0) prefetch(S - 1);
  cluster_barrier();                     // every CTA of the cluster is resident before anyone touches remote smem

  for (int t = S - 1; t >= 0; --t) {
    if (prof) tk = clock64();
    float gi = 0.f, gf = 0.f, gg = 0.f, go = 0.f, ct = 0.f, cprev = 0.f, dh = 0.f;
    if (active) {
      const size_t row = (size_t)t * Bt + b;
      const size_t o = row * H + j0 + eu;
      const float* gp = a.gates + row * 4 * H + j0 + eu;
      gi = __ldcs(gp);
      gf = __ldcs(gp + (size_t)H);
      gg = __ldcs(gp + (size_t)2 * H);
      go = __ldcs(gp + (size_t)3 * H);
      ct = __ldcs(a.c_all + o);
      cprev = t > 0 ? __ldcs(a.c_all + o - (size_t)Bt * H) : 0.f;
      dh = drop_out(__ldcs(a.dout + (size_t)t * a.dout_st + (size_t)b * a.dout_sb + j0 + eu), a.drop, dseed,
                    (uint32_t)row, (uint32_t)(j0 + eu));
      if (t > 0 && (eu & 7) == 0) prefetch(t - 1);   // one lane per 32-byte sector
    }
    if (t < S - 1) {                     // uniform over the cluster
      // the half's rows of dgates_{t+1}; canaries: the half's last row
      const __nv_bfloat16* src = a.dg + ((size_t)(t + 1) * Bt + r0) * 4 * H + kw;
#pragma unroll 1
      for (int i = lane; i < NPROD; i += 32) spin_piece(src + (size_t)(nr - 1) * 4 * H + i * 8);
      __syncwarp();
      LSTM_TICK(0)
      float acc[1][8][4];
      const int tries =
          sweep_mma<KS, 8>(acc, bfr, dw, src, (size_t)4 * H, nr, lane, (a.mode & MODE_NOMMA) != 0, wsm);
      LSTM_TICK(1)
      if (prof) pc[7] += tries;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        const int uc = nt * 8 + 2 * tg;
        *reinterpret_cast<float2*>(redw + g * RP + uc) = make_float2(acc[0][nt][0], acc[0][nt][1]);
        *reinterpret_cast<float2*>(redw + (g + 8) * RP + uc) = make_float2(acc[0][nt][2], acc[0][nt][3]);
      }
      LSTM_TICK(2)
      __syncthreads();
      // this CTA's partial sums for all 64 units of the cluster (double-buffered by step parity: a remote reader of
      // step t is done before it arrives at the barrier of step t-1, which precedes our next write to this buffer)
      float* pbuf = part + (t & 1) * 16 * RP;
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) {
        float sum = 0.f;
#pragma unroll
        for (int ww = 0; ww < kWarps; ++ww) sum += red[(ww * 16 + qr) * RP + jj * 16 + qu];
        pbuf[qr * RP + jj * 16 + qu] = sum;
      }
      LSTM_TICK(3)
      step_barrier();
      if (active) {
#pragma unroll
        for (int rr = 0; rr < 4; ++rr) dh += ld_dsmem_f32(pbuf + eb * RP + (int)rank * 16 + eu, (uint32_t)rr);
      }
    }
    float d_i = 0.f, d_f = 0.f, d_g = 0.f, d_o = 0.f;
    if (active) {
      const float tc = tanhf_(ct);
      d_o = dh * tc * go * (1.f - go);
      const float dct = dc + dh * go * (1.f - tc * tc);
      d_i = dct * gg * gi * (1.f - gi);
      d_g = dct * gi * (1.f - gg * gg);
      d_f = dct * cprev * gf * (1.f - gf);
      dc = dct * gf;
    }
    {
      // two 16-byte publications per gate plane and row: lanes eu = 0 and 8 each store eight units (publish8_bf16)
      __nv_bfloat16* dp = a.dg + ((size_t)t * Bt + (active ? b : r0)) * 4 * H + j0 + (eu & 8);
      const bool st_ = active && (eu & 7) == 0;
      publish8_bf16(dp, d_i, st_);
      publish8_bf16(dp + (size_t)H, d_f, st_);
      publish8_bf16(dp + (size_t)2 * H, d_g, st_);
      publish8_bf16(dp + (size_t)3 * H, d_o, st_);
    }
    if (active) {
      LSTM_TICK(4)
      LSTM_TICK(5)
    }
  }
  __syncthreads();
  cluster_barrier();                     // nobody exits while a peer may still read its shared memory
  if (prof)
    for (int i = 0; i < 8; ++i) a.dbg[(size_t)blockIdx.x * 16 + 8 + i] = (unsigned long long)pc[i];
}

#undef LSTM_TICK

// Whether cluster launches of the recurrence are also cooperative.  ncu's kernel replay refuses cooperative cluster
// launches (LaunchFailed): VQA_B200_LSTM_COOP=0 drops the attribute for profiling runs on an otherwise idle GPU.
bool coop_launch() {
  static int coop = -1;
  if (coop < 0) {
    const char* e = getenv("VQA_B200_LSTM_COOP");
    coop = (e && e[0] == '0') ? 0 : 1;
  }
  return coop != 0;
}

// VQA_B200_LSTM_CLUSTERS, read at every launch (tests and A/B probes compare the forms in one process): 1, the default,
// runs the cluster forms; 0 runs the cluster-free pair, the forms a device gets when the clusters cannot all be
// co-resident.  Returns 1 or 0, or the library error for any other value.
int clusters_enabled() {
  const char* e = getenv("VQA_B200_LSTM_CLUSTERS");
  if (e == nullptr || strcmp(e, "1") == 0) return 1;
  if (strcmp(e, "0") == 0) return 0;
  return set_error(VQA_B200_EINVAL, "VQA_B200_LSTM_CLUSTERS must be 0 or 1 (got '%s')", e);
}

constexpr int kNotCoResident = -1000;   // launch_clusters4 launched nothing: the caller runs its cluster-free form

// Launches `grid` CTAs of `kern` in clusters of 4.  The CTAs wait on each other, so the whole grid must be co-resident:
// returns kNotCoResident, launching nothing, when cudaOccupancyMaxActiveClusters says the clusters cannot all be.  That
// query answers for an idle GPU only; under data-parallel training the gradient all-reduce may already hold SMs when
// this kernel is enqueued, so the launch is COOPERATIVE as well: the grid is only started once all of it fits, instead
// of resident CTAs spinning on peers that cannot be scheduled.
template <typename... Params, typename... Args>
int launch_clusters4(void (*kern)(Params...), int grid, size_t smem, cudaStream_t st, const char* who, Args... args) {
  VQA_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attrs[2];
  attrs[0].id = cudaLaunchAttributeClusterDimension;
  attrs[0].val.clusterDim.x = 4;
  attrs[0].val.clusterDim.y = 1;
  attrs[0].val.clusterDim.z = 1;
  attrs[1].id = cudaLaunchAttributeCooperative;
  attrs[1].val.cooperative = 1;
  cfg.attrs = attrs;
  cfg.numAttrs = 1;
  int nclusters = 0;
  if (cudaOccupancyMaxActiveClusters(&nclusters, kern, &cfg) != cudaSuccess) {
    (void)cudaGetLastError();
    return kNotCoResident;
  }
  if (nclusters * 4 < grid) return kNotCoResident;
  cfg.numAttrs = coop_launch() ? 2 : 1;
  const cudaError_t e = cudaLaunchKernelEx(&cfg, kern, args...);
  if (e != cudaSuccess) return set_error((int)e, "%s cluster launch: %s", who, cudaGetErrorString(e));
  return 0;
}

// The forward: the multicast form in clusters of 4, else the sweep form (a cooperative launch without clusters).
template <int KS>
int launch_fwd(const LstmFwdArgs& a, cudaStream_t st) {
  const int clusters = clusters_enabled();
  if (clusters < 0) return clusters;
  CUtensorMap hmap;
  memset(&hmap, 0, sizeof(hmap));
  if (clusters) {
    using SM = FwdSmem<KS, 4>;
    // hb as a [(S+1) * Bt, H] matrix (a batch of one); one box = one column half of a warp's slice over the Bt rows of
    // a step
    constexpr CUtensorMapSwizzle swz_mode = SM::RB == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                            : SM::RB == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
    if (int rc = make_tmap(&hmap, a.hb, (uint64_t)a.H, (uint64_t)(a.S + 1) * a.Bt, (uint64_t)a.H, (uint32_t)(SM::RB / 2),
                           (uint32_t)a.Bt, 1, 0, swz_mode))
      return rc;
    const int rc = launch_clusters4(lstm_fwd_kernel<KS, 4>, a.H / kU, SM::BYTES, st, "lstm_fwd", a, hmap);
    if (rc != kNotCoResident) return rc;
  }
  using SM = FwdSmem<KS, 1>;
  auto kern = lstm_fwd_kernel<KS, 1>;
  VQA_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SM::BYTES));
  LstmFwdArgs args = a;
  void* params[] = {&args, &hmap};
  VQA_CUDA_CHECK(cudaLaunchCooperativeKernel((const void*)kern, dim3(a.H / kU), dim3(kThreads), params, SM::BYTES, st));
  return 0;
}

// The backward: the row-split form in clusters of 4, else the single-CTA form (a cooperative launch without clusters).
template <int KS>
int launch_bwd(const LstmBwdArgs& a, cudaStream_t st) {
  const int clusters = clusters_enabled();
  if (clusters < 0) return clusters;
  if (clusters) {
    // two row halves of H/16 CTAs; at Bt = 1 the first only, since the second would hold no rows
    const int rc = launch_clusters4(lstm_bwd_rows_kernel<KS>, (a.Bt >= 2 ? 2 : 1) * a.H / 16, BwdRowsSmem<KS>::BYTES,
                                    st, "lstm_bwd", a);
    if (rc != kNotCoResident) return rc;
  }
  constexpr int PITCH = KS * 16 + 8;
  const size_t smem = (size_t)kWarps * 2 * kRows * PITCH * 2 + (size_t)kWarps * 32 * 8 * 4;
  VQA_CUDA_CHECK(cudaFuncSetAttribute(lstm_bwd_kernel<KS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  LstmBwdArgs args = a;
  void* params[] = {&args};
  VQA_CUDA_CHECK(cudaLaunchCooperativeKernel((const void*)lstm_bwd_kernel<KS>, dim3(a.H / kU), dim3(kThreads), params,
                                             smem, st));
  return 0;
}

int check_shape(const char* who, int S, int Bt, int H) {
  if (S <= 0 || Bt <= 0 || Bt > kRows)
    return set_error(VQA_B200_EINVAL, "%s: need S >= 1 and 1 <= Bt <= %d (S=%d Bt=%d)", who, kRows, S, Bt);
  if (!(H == 128 || H == 256 || H == 512 || H == 1024))
    return set_error(VQA_B200_EINVAL, "%s: hidden size must be 128, 256, 512 or 1024 (got %d)", who, H);
  if (H / kU > sm_count())
    return set_error(VQA_B200_EINVAL, "%s: needs %d co-resident CTAs, device has %d SMs", who, H / kU, sm_count());
  return 0;
}

}  // namespace
}  // namespace vqa

using namespace vqa;

#ifdef VQA_B200_DEBUG
extern "C" void vqa_b200_debug_set_lstm(void* device_u64x16, int mode) {
  g_dbg = (unsigned long long*)device_u64x16;
  g_mode = mode & 0xFF;
  g_dbg_ctas = (mode >> 16) & 0xFFFF;  // bits 16..31: CTAs (rows of 16 counters) the buffer holds; 0 = CTA 0 only
  if (g_dbg_ctas < 1) g_dbg_ctas = 1;
}
#endif

// ---------------------------------------------------------------------------------------------------------------
// Wide-batch regime (mfb.py:68-70: a proper batch_first LSTM, S = T = 26 steps over Bt = N = 64..512 rows).  With
// hundreds of rows per step the recurrent product is a real GEMM ([Bt, H] x [H, 4H] = 4.3 GFLOP at Bt = 512): it runs on
// the tcgen05 kernel, accumulated onto the x-projection already sitting in `gates`, and the gate math is one
// elementwise pass per step.  A thread owns four adjacent hidden units of one row (128-bit accesses per gate plane).
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) lstm_cell_fwd_kernel(float* __restrict__ gates, const float* __restrict__ c_prev,
                                                            float* __restrict__ c_out, float* __restrict__ out,
                                                            long long ld_out, __nv_bfloat16* __restrict__ hb_next,
                                                            int Bt, int H, int save, long long row0, LstmDrop drop) {
  const uint32_t dseed = drop.thresh16 ? effective_seed(drop.seed, drop.seed_dev) : 0u;
  const int q = H >> 2;
  const long long n = (long long)Bt * q;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int b = (int)(i / q), j = (int)(i % q) * 4;
    float* gp = gates + (long long)b * 4 * H + j;
    const float4 pi = *reinterpret_cast<const float4*>(gp);
    const float4 pf = *reinterpret_cast<const float4*>(gp + H);
    const float4 pg = *reinterpret_cast<const float4*>(gp + 2 * (long long)H);
    const float4 po = *reinterpret_cast<const float4*>(gp + 3 * (long long)H);
    float4 c = c_prev ? *reinterpret_cast<const float4*>(c_prev + (long long)b * H + j) : make_float4(0.f, 0.f, 0.f, 0.f);
    float4 gi, gf, gg, go, h;
#define VQA_CELL(X)                                           \
    gi.X = sigmoidf_(pi.X); gf.X = sigmoidf_(pf.X);           \
    gg.X = tanhf_(pg.X);    go.X = sigmoidf_(po.X);           \
    c.X = gf.X * c.X + gi.X * gg.X;                           \
    h.X = go.X * tanhf_(c.X);
    VQA_CELL(x) VQA_CELL(y) VQA_CELL(z) VQA_CELL(w)
#undef VQA_CELL
    *reinterpret_cast<float4*>(c_out + (long long)b * H + j) = c;
    {
      const uint32_t r = (uint32_t)(row0 + b);
      *reinterpret_cast<float4*>(out + (long long)b * ld_out + j) =
          make_float4(drop_out(h.x, drop, dseed, r, j), drop_out(h.y, drop, dseed, r, j + 1),
                      drop_out(h.z, drop, dseed, r, j + 2), drop_out(h.w, drop, dseed, r, j + 3));
    }
    const __nv_bfloat162 lo = __floats2bfloat162_rn(h.x, h.y), hi = __floats2bfloat162_rn(h.z, h.w);
    uint2 u;
    u.x = *reinterpret_cast<const uint32_t*>(&lo);
    u.y = *reinterpret_cast<const uint32_t*>(&hi);
    *reinterpret_cast<uint2*>(hb_next + (long long)b * H + j) = u;
    if (save) {
      *reinterpret_cast<float4*>(gp) = gi;
      *reinterpret_cast<float4*>(gp + H) = gf;
      *reinterpret_cast<float4*>(gp + 2 * (long long)H) = gg;
      *reinterpret_cast<float4*>(gp + 3 * (long long)H) = go;
    }
  }
}

// dh holds the recurrent part of dL/dh_t (accumulated by the tcgen05 GEMM of step t+1; zero at t = S-1) and is reset to
// zero here for the GEMM of this step; dc carries dL/dc across the steps.
__global__ void __launch_bounds__(256) lstm_cell_bwd_kernel(const float* __restrict__ gates,
                                                            const float* __restrict__ c_prev,
                                                            const float* __restrict__ c_t, const float* __restrict__ dout,
                                                            long long ld_dout, float* __restrict__ dh,
                                                            float* __restrict__ dc, __nv_bfloat16* __restrict__ dg,
                                                            int Bt, int H, long long row0, LstmDrop drop) {
  const uint32_t dseed = drop.thresh16 ? effective_seed(drop.seed, drop.seed_dev) : 0u;
  const int q = H >> 2;
  const long long n = (long long)Bt * q;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int b = (int)(i / q), j = (int)(i % q) * 4;
    const float* gp = gates + (long long)b * 4 * H + j;
    const float4 gi = *reinterpret_cast<const float4*>(gp);
    const float4 gf = *reinterpret_cast<const float4*>(gp + H);
    const float4 gg = *reinterpret_cast<const float4*>(gp + 2 * (long long)H);
    const float4 go = *reinterpret_cast<const float4*>(gp + 3 * (long long)H);
    const float4 ct = *reinterpret_cast<const float4*>(c_t + (long long)b * H + j);
    const float4 cp = c_prev ? *reinterpret_cast<const float4*>(c_prev + (long long)b * H + j) : make_float4(0.f, 0.f, 0.f, 0.f);
    float4 d0 = *reinterpret_cast<const float4*>(dout + (long long)b * ld_dout + j);
    {
      const uint32_t r = (uint32_t)(row0 + b);
      d0 = make_float4(drop_out(d0.x, drop, dseed, r, j), drop_out(d0.y, drop, dseed, r, j + 1),
                       drop_out(d0.z, drop, dseed, r, j + 2), drop_out(d0.w, drop, dseed, r, j + 3));
    }
    float4* dhp = reinterpret_cast<float4*>(dh + (long long)b * H + j);
    float4* dcp = reinterpret_cast<float4*>(dc + (long long)b * H + j);
    const float4 dr = *dhp;
    float4 dcv = *dcp;
    float4 di, df, dgg, dO;
#define VQA_CELL(X)                                                     \
    {                                                                   \
      const float dhx = d0.X + dr.X;                                    \
      const float tc = tanhf_(ct.X);                                    \
      dO.X = dhx * tc * go.X * (1.f - go.X);                            \
      const float dct = dcv.X + dhx * go.X * (1.f - tc * tc);           \
      di.X = dct * gg.X * gi.X * (1.f - gi.X);                          \
      dgg.X = dct * gi.X * (1.f - gg.X * gg.X);                         \
      df.X = dct * cp.X * gf.X * (1.f - gf.X);                          \
      dcv.X = dct * gf.X;                                               \
    }
    VQA_CELL(x) VQA_CELL(y) VQA_CELL(z) VQA_CELL(w)
#undef VQA_CELL
    *dcp = dcv;
    *dhp = make_float4(0.f, 0.f, 0.f, 0.f);
    __nv_bfloat16* dp = dg + (long long)b * 4 * H + j;
    auto st4b = [](__nv_bfloat16* p_, const float4& v) {
      const __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
      uint2 u;
      u.x = *reinterpret_cast<const uint32_t*>(&lo);
      u.y = *reinterpret_cast<const uint32_t*>(&hi);
      *reinterpret_cast<uint2*>(p_) = u;
    };
    st4b(dp, di);
    st4b(dp + H, df);
    st4b(dp + 2 * (long long)H, dgg);
    st4b(dp + 3 * (long long)H, dO);
  }
}

static int cell_grid(int Bt, int H) {
  long long blocks = ((long long)Bt * (H / 4) + 255) / 256;
  const long long cap = (long long)sm_count() * 8;
  return (int)(blocks < cap ? blocks : cap);
}

extern "C" int vqa_b200_lstm_supported(int Bt, int H) {
  return (Bt >= 1 && Bt <= kRows && (H == 128 || H == 256 || H == 512 || H == 1024)) ? 1 : 0;
}

extern "C" int vqa_b200_lstm_fwd(float* gates, const void* whh, float* out, void* hb, float* c_all, int S, int Bt, int H,
                                 float drop_p, uint32_t seed, const uint32_t* seed_dev, void* stream) {
  if (!(drop_p >= 0.f && drop_p < 1.f)) return set_error(VQA_B200_EINVAL, "lstm_fwd: bad dropout p");
  if (int rc = check_shape("lstm_fwd", S, Bt, H)) return rc;
  if (!gates || !whh || !out || !hb) return set_error(VQA_B200_EINVAL, "lstm_fwd: null pointer");
  if (!aligned16(whh) || !aligned16(hb)) return set_error(VQA_B200_EALIGN, "lstm_fwd: whh / hb must be 16-byte aligned");
  LstmFwdArgs a{gates, (const __nv_bfloat16*)whh, out, (__nv_bfloat16*)hb, c_all, S, Bt, H, g_dbg, g_dbg_ctas, g_mode,
                make_drop(drop_p, seed, seed_dev)};
  cudaStream_t st = (cudaStream_t)stream;
  switch (H / 128) {
    case 1: return launch_fwd<1>(a, st);
    case 2: return launch_fwd<2>(a, st);
    case 4: return launch_fwd<4>(a, st);
    default: return launch_fwd<8>(a, st);
  }
}

extern "C" int vqa_b200_lstm_bwd(const float* gates, const float* c_all, const float* dout, int64_t dout_st,
                                 int64_t dout_sb, const void* whh, int w_layout, void* dg, int S, int Bt, int H,
                                 float drop_p, uint32_t seed, const uint32_t* seed_dev, void* stream) {
  if (!(drop_p >= 0.f && drop_p < 1.f)) return set_error(VQA_B200_EINVAL, "lstm_bwd: bad dropout p");
  if (int rc = check_shape("lstm_bwd", S, Bt, H)) return rc;
  if (!gates || !c_all || !dout || !whh || !dg) return set_error(VQA_B200_EINVAL, "lstm_bwd: null pointer");
  if (!aligned16(whh) || !aligned16(dg)) return set_error(VQA_B200_EALIGN, "lstm_bwd: whh / dg must be 16-byte aligned");
  if (w_layout != 0 && w_layout != 1) return set_error(VQA_B200_EINVAL, "lstm_bwd: w_layout must be 0 ([H,4H]) or 1 ([4H,H])");
  if (dout_st <= 0 && S > 1) return set_error(VQA_B200_EINVAL, "lstm_bwd: bad dout strides");
  LstmBwdArgs a{gates, c_all, dout, (const __nv_bfloat16*)whh, (__nv_bfloat16*)dg, S, Bt, H, g_dbg, g_dbg_ctas, g_mode,
                (long long)dout_st, (long long)dout_sb, w_layout, make_drop(drop_p, seed, seed_dev)};
  cudaStream_t st = (cudaStream_t)stream;
  switch (H / 128) {
    case 1: return launch_bwd<1>(a, st);
    case 2: return launch_bwd<2>(a, st);
    case 4: return launch_bwd<4>(a, st);
    default: return launch_bwd<8>(a, st);
  }
}

extern "C" int vqa_b200_lstm_cell_fwd(float* gates, const float* c_prev, float* c_out, float* out, int64_t ld_out,
                                      void* hb_next, int Bt, int H, int save_gates, int64_t row0, float drop_p,
                                      uint32_t seed, const uint32_t* seed_dev, void* stream) {
  if (!(drop_p >= 0.f && drop_p < 1.f)) return set_error(VQA_B200_EINVAL, "lstm_cell_fwd: bad dropout p");
  if (!gates || !c_out || !out || !hb_next || Bt <= 0 || H <= 0 || H % 4 != 0 || ld_out < H)
    return set_error(VQA_B200_EINVAL, "lstm_cell_fwd: bad arguments (Bt=%d H=%d, H %% 4 == 0 required)", Bt, H);
  if (!aligned16(gates) || !aligned16(c_out) || !aligned16(out) || (ld_out % 4) != 0 || (c_prev && !aligned16(c_prev)) ||
      (reinterpret_cast<uintptr_t>(hb_next) & 7) != 0)
    return set_error(VQA_B200_EALIGN, "lstm_cell_fwd: operands must be 16-byte aligned (hb_next: 8)");
  lstm_cell_fwd_kernel<<<cell_grid(Bt, H), 256, 0, (cudaStream_t)stream>>>(gates, c_prev, c_out, out, (long long)ld_out,
                                                                         (__nv_bfloat16*)hb_next, Bt, H, save_gates,
                                                                         (long long)row0, make_drop(drop_p, seed, seed_dev));
  VQA_LAUNCH_CHECK("lstm_cell_fwd");
  return 0;
}

extern "C" int vqa_b200_lstm_cell_bwd(const float* gates, const float* c_prev, const float* c_t, const float* dout,
                                      int64_t ld_dout, float* dh, float* dc, void* dg, int Bt, int H, int64_t row0,
                                      float drop_p, uint32_t seed, const uint32_t* seed_dev, void* stream) {
  if (!(drop_p >= 0.f && drop_p < 1.f)) return set_error(VQA_B200_EINVAL, "lstm_cell_bwd: bad dropout p");
  if (!gates || !c_t || !dout || !dh || !dc || !dg || Bt <= 0 || H <= 0 || H % 4 != 0 || ld_dout < H)
    return set_error(VQA_B200_EINVAL, "lstm_cell_bwd: bad arguments (Bt=%d H=%d, H %% 4 == 0 required)", Bt, H);
  if (!aligned16(gates) || !aligned16(c_t) || !aligned16(dout) || (ld_dout % 4) != 0 || !aligned16(dh) || !aligned16(dc) ||
      (c_prev && !aligned16(c_prev)) || (reinterpret_cast<uintptr_t>(dg) & 7) != 0)
    return set_error(VQA_B200_EALIGN, "lstm_cell_bwd: operands must be 16-byte aligned (dg: 8)");
  lstm_cell_bwd_kernel<<<cell_grid(Bt, H), 256, 0, (cudaStream_t)stream>>>(gates, c_prev, c_t, dout, (long long)ld_dout, dh,
                                                                         dc, (__nv_bfloat16*)dg, Bt, H, (long long)row0,
                                                                         make_drop(drop_p, seed, seed_dev));
  VQA_LAUNCH_CHECK("lstm_cell_bwd");
  return 0;
}
