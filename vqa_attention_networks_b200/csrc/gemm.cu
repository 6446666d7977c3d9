// Host side of the tcgen05 GEMM: tensor-map construction, tile-shape selection, launch.
#include <stdlib.h>

#include <mutex>

#include "common.h"
#include "gemm_sm100.cuh"

namespace vqa {

// ------------------------------------------------------------------ error / device helpers
static thread_local char g_err[512] = "";

int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
const char* last_error() { return g_err; }

int sm_count() {
  static int cache[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cache[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cache[dev] = n;
  }
  return cache[dev];
}

// ------------------------------------------------------------------ TMA descriptors
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

// bf16 matrix with `inner` contiguous elements per row, `outer` rows, row pitch ld (elements)
int make_tmap(CUtensorMap* map, const void* base, uint64_t inner, uint64_t outer, uint64_t ld, uint32_t box_inner,
              uint32_t box_outer, uint64_t batch, uint64_t bstride, CUtensorMapSwizzle swizzle) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return set_error(VQA_B200_EDRIVER, "cuTensorMapEncodeTiled entry point not available");
  if (!aligned16(base) || (ld * 2) % 16 != 0)
    return set_error(VQA_B200_EALIGN, "TMA operand needs a 16-byte aligned base and pitch (ld=%llu)",
                     (unsigned long long)ld);
  if (batch < 1) batch = 1;
  if (batch == 1) bstride = ((outer * ld * 2 + 15) / 16) * 8;       // unused dimension: any legal pitch
  if ((bstride * 2) % 16 != 0)
    return set_error(VQA_B200_EALIGN, "TMA operand needs a 16-byte aligned batch stride (%llu elements)",
                     (unsigned long long)bstride);
  cuuint64_t dims[3] = {inner, outer, batch};
  cuuint64_t strides[2] = {ld * 2, bstride * 2};
  cuuint32_t box[3] = {box_inner, box_outer, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(VQA_B200_EDRIVER, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  return 0;
}

static unsigned long long* g_dbg = nullptr;
void debug_set_counters(unsigned long long* p) { g_dbg = p; }

// Debug override of the MN-major descriptor strides (selftest sweeps); 0 = defaults.
static uint32_t g_mn_lbo = 0, g_mn_sbo = 0, g_mn_kadv = 0;
void debug_set_mn_desc(uint32_t lbo, uint32_t sbo, uint32_t kadv_bytes) {
  g_mn_lbo = lbo; g_mn_sbo = sbo; g_mn_kadv = kadv_bytes;
}

static void fill_operand_desc(int mn_major, uint64_t* hi, uint32_t* kadv) {
  if (mn_major) {
    // canonical SW128 MN-major tile: 64 contiguous elements (128 B) per k-row, 8 k-rows per 1024-B
    // swizzle atom (SBO), next 64-element group one TMA box further (LBO = 64 k-rows * 128 B).
    const uint32_t lbo = g_mn_lbo ? g_mn_lbo : (uint32_t)BLOCK_K * 128u;
    const uint32_t sbo = g_mn_sbo ? g_mn_sbo : 1024u;
    const uint32_t adv = g_mn_kadv ? g_mn_kadv : (uint32_t)UMMA_K * 128u;
    *hi = umma_desc_hi(lbo, sbo);
    *kadv = adv >> 4;
  } else {
    // canonical SW128 K-major tile: 128-B rows, 8-row groups 1024 B apart; LBO unused for swizzled K-major
    *hi = umma_desc_hi(16, 1024);
    *kadv = (UMMA_K * 2) >> 4;
  }
}

template <int BN, int EPI, bool CTA2 = false, bool MFBX = false>
static int launch(const CUtensorMap& ta, const CUtensorMap& tb, const GemmArgs& args, cudaStream_t stream) {
  using Cfg = GemmCfg<BN, CTA2>;
  auto kern = gemm_tcgen05_kernel<BN, EPI, CTA2, MFBX>;
  VQA_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
  const long long all_tiles = (long long)args.batch * args.m_blocks * args.n_blocks;
  const long long tiles = args.full_units + (all_tiles - args.full_units) * args.k_split;
  if (CTA2) {
    // one CTA pair (cluster of 2, same TPC) per work unit
    long long pairs = sm_count() / 2;
    if (pairs > tiles) pairs = tiles;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(2 * pairs));
    cfg.blockDim = dim3(GEMM_THREADS);
    cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    VQA_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kern, ta, tb, args));
    return 0;
  }
  int grid = sm_count();
  if (grid > tiles) grid = (int)tiles;
  kern<<<grid, GEMM_THREADS, Cfg::SMEM_BYTES, stream>>>(ta, tb, args);
  VQA_LAUNCH_CHECK("gemm_tcgen05_kernel");
  return 0;
}

// CTA pairs pay off on large tensor-bound problems; VQA_B200_CTA2=0/1 forces the choice (A/B measurements)
static bool use_cta2(long long M, long long N, long long K, int batch) {
  static int forced = -2;
  if (forced == -2) {
    const char* e = getenv("VQA_B200_CTA2");
    forced = e ? atoi(e) : -1;
  }
  if (forced == 0) return false;
  if (forced == 1) return batch == 1 && M >= 256;
  return batch == 1 && M >= 2048 && N >= 240 && (double)M * N * K >= 1e10;
}

static int setup_operands(GemmArgs& g, CUtensorMap* ta, CUtensorMap* tb, const void* A, int a_layout, int64_t lda,
                          const void* B, int b_layout, int64_t ldb, int BN, int64_t a_bstride = 0,
                          int64_t b_bstride = 0, bool cta2 = false) {
  if (g.batch < 1) g.batch = 1;
  const int TILE_M = cta2 ? 2 * BLOCK_M : BLOCK_M;     // a CTA pair covers 256 rows
  const int BN_CTA = cta2 ? BN / 2 : BN;               // ... and each CTA loads half of the B tile
  g.a_mn = a_layout == VQA_B200_MN_MAJOR;
  g.b_mn = b_layout == VQA_B200_MN_MAJOR;
  g.m_blocks = (g.M + TILE_M - 1) / TILE_M;
  g.n_blocks = (g.N + BN - 1) / BN;
  g.k_blocks = (g.K + BLOCK_K - 1) / BLOCK_K;
  fill_operand_desc(g.a_mn, &g.a_desc_hi, &g.a_kadv);
  fill_operand_desc(g.b_mn, &g.b_desc_hi, &g.b_kadv);
  g.idesc = umma_idesc_bf16(TILE_M, BN, g.a_mn, g.b_mn);
  int rc;
  if (g.a_mn) rc = make_tmap(ta, A, (uint64_t)g.M, (uint64_t)g.K, (uint64_t)lda, 64, BLOCK_K, g.batch, a_bstride);
  else        rc = make_tmap(ta, A, (uint64_t)g.K, (uint64_t)g.M, (uint64_t)lda, BLOCK_K, BLOCK_M, g.batch, a_bstride);
  if (rc) return rc;
  if (g.b_mn) rc = make_tmap(tb, B, (uint64_t)g.N, (uint64_t)g.K, (uint64_t)ldb, 64, BLOCK_K, g.batch, b_bstride);
  else        rc = make_tmap(tb, B, (uint64_t)g.K, (uint64_t)g.N, (uint64_t)ldb, BLOCK_K, (uint32_t)BN_CTA, g.batch, b_bstride);
  return rc;
}

}  // namespace vqa

using namespace vqa;

extern "C" int vqa_b200_abi_version(void) { return VQA_B200_ABI_VERSION; }
extern "C" const char* vqa_b200_last_error(void) { return vqa::last_error(); }
#ifdef VQA_B200_DEBUG
extern "C" void vqa_b200_debug_set_counters(void* device_u64x16) {
  vqa::debug_set_counters(reinterpret_cast<unsigned long long*>(device_u64x16));
}
extern "C" void vqa_b200_debug_set_mn_desc(uint32_t lbo, uint32_t sbo, uint32_t kadv_bytes) {
  vqa::debug_set_mn_desc(lbo, sbo, kadv_bytes);
}
#endif

static int gemm_impl(const void* A, int a_layout, int64_t lda, int64_t a_bstride, const void* B, int b_layout,
                     int64_t ldb, int64_t b_bstride, void* C, int c_dtype, int64_t ldc, int64_t c_bstride, int batch,
                     int M, int N, int K, const float* bias, const float* row_scale, int rows_per_group, int act,
                     const void* add, int add_dtype, float drop_p, uint32_t seed, const uint32_t* seed_dev,
                     int accumulate, int k_split, const void* dot_with, int64_t ld_dot, float* dot_out, void* stream) {
  if (!A || !B || !C || M <= 0 || N <= 0 || K <= 0 || batch <= 0)
    return set_error(VQA_B200_EINVAL, "gemm: null operand or empty shape (M=%d N=%d K=%d batch=%d)", M, N, K, batch);
  if (accumulate && c_dtype != VQA_B200_F32)
    return set_error(VQA_B200_EINVAL, "gemm: accumulate mode needs an fp32 C");
  if (!(drop_p >= 0.f && drop_p < 1.f)) return set_error(VQA_B200_EINVAL, "gemm: bad dropout p");
  if (rows_per_group <= 0) rows_per_group = 1;
  GemmArgs g = {};
  g.M = M; g.N = N; g.K = K; g.batch = batch;
  g.dbg = g_dbg;
  g.C = C; g.ldc = ldc; g.c_bstride = c_bstride; g.c_bf16 = (c_dtype == VQA_B200_BF16);
  const int esz = g.c_bf16 ? 2 : 4;
  g.vec_ok = aligned16(C) && ((ldc * esz) % 16 == 0) && ((c_bstride * esz) % 16 == 0) &&
             (dot_with == nullptr || (aligned16(dot_with) && (ld_dot * 2) % 16 == 0 && (c_bstride * 2) % 16 == 0));
  g.bias = bias; g.row_scale = row_scale; g.rows_per_group = rows_per_group; g.act = act;
  g.add = add; g.add_bf16 = (add_dtype == VQA_B200_BF16);
  g.st_drop_seed = seed;
  g.seed_dev = seed_dev;
  g.st_drop_thresh16 = (uint32_t)(drop_p * 65536.0f + 0.5f);
  g.st_drop_scale = g.st_drop_thresh16 ? 65536.0f / (65536.0f - (float)g.st_drop_thresh16) : 1.0f;
  g.dot_with = reinterpret_cast<const __nv_bfloat16*>(dot_with); g.ld_dot = ld_dot; g.dot_out = dot_out;

  // tile width: 256 for wide outputs (halves the smem operand traffic per flop), else 128
  const int sms = sm_count();
  int BN = 128;
  {
    const long long t256 = (long long)batch * ((M + 127) / 128) * ((N + 255) / 256);
    if (N >= 256 && t256 >= sms) BN = 256;
  }
  const bool cta2 = (BN == 256) && use_cta2(M, N, K, batch);
  CUtensorMap ta, tb;
  int rc = setup_operands(g, &ta, &tb, A, a_layout, lda, B, b_layout, ldb, BN, a_bstride, b_bstride, cta2);
  if (rc) return rc;
  const int workers = cta2 ? sms / 2 : sms;           // persistent CTAs or CTA pairs
  g.k_split = 1;
  if (accumulate) {
    int ks = k_split;
    if (ks <= 0) {
      const long long tiles = (long long)batch * g.m_blocks * g.n_blocks;
      const int max_ks = g.k_blocks / 4 > 0 ? g.k_blocks / 4 : 1;       // >= 4 k-blocks per unit
      if (tiles < workers) {
        // fewer tiles than SMs: uniform split; choose the split with the least wave quantisation
        double best = -1.0;
        ks = 1;
        for (int c = 1; c <= (max_ks < 32 ? max_ks : 32); ++c) {
          const long long units = tiles * c;
          const long long waves = (units + workers - 1) / workers;
          const double score = (double)units / (double)(waves * workers) - 0.004 * (c - 1);
          if (score > best + 1e-9) { best = score; ks = c; }
        }
      } else {
        // whole waves run unsplit (K-lockstep keeps the operand panels in L2); only the ragged tail wave is split
        const long long tail = tiles % workers;
        ks = 1;
        if (tail > 0) {
          g.full_units = (int)(tiles - tail);
          ks = (int)(workers / tail);
          if (ks > max_ks) ks = max_ks;
          if (ks < 1) ks = 1;
        }
      }
    }
    if (ks > g.k_blocks) ks = g.k_blocks;
    g.k_split = ks;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (cta2) return accumulate ? launch<256, EPI_ATOMIC, true>(ta, tb, g, st) : launch<256, EPI_STORE, true>(ta, tb, g, st);
  if (accumulate) return BN == 256 ? launch<256, EPI_ATOMIC>(ta, tb, g, st) : launch<128, EPI_ATOMIC>(ta, tb, g, st);
  return BN == 256 ? launch<256, EPI_STORE>(ta, tb, g, st) : launch<128, EPI_STORE>(ta, tb, g, st);
}

extern "C" int vqa_b200_gemm(const void* A, int a_layout, int64_t lda, const void* B, int b_layout, int64_t ldb,
                             void* C, int c_dtype, int64_t ldc, int M, int N, int K, const float* bias,
                             const float* row_scale, int rows_per_group, int relu, int accumulate, int k_split,
                             const void* dot_with, int64_t ld_dot, float* dot_out, void* stream) {
  return gemm_impl(A, a_layout, lda, 0, B, b_layout, ldb, 0, C, c_dtype, ldc, 0, 1, M, N, K, bias, row_scale,
                   rows_per_group, relu ? 1 : 0, nullptr, 0, 0.f, 0, nullptr, accumulate, k_split, dot_with, ld_dot,
                   dot_out, stream);
}

extern "C" int vqa_b200_gemm_batched(const void* A, int a_layout, int64_t lda, int64_t a_bstride, const void* B,
                                     int b_layout, int64_t ldb, int64_t b_bstride, void* C, int c_dtype, int64_t ldc,
                                     int64_t c_bstride, int batch, int M, int N, int K, const float* bias, int act,
                                     const void* add, int add_dtype, float drop_p, uint32_t seed,
                                     const uint32_t* seed_dev, int accumulate, void* stream) {
  return gemm_impl(A, a_layout, lda, a_bstride, B, b_layout, ldb, b_bstride, C, c_dtype, ldc, c_bstride, batch, M, N, K,
                   bias, nullptr, 1, act, add, add_dtype, drop_p, seed, seed_dev, accumulate, 0, nullptr, 0,
                   nullptr, stream);
}

extern "C" int vqa_b200_mfb_fused(const void* X, int64_t ldx, const void* W, int64_t ldw, const float* bias,
                                  const float* Q, int64_t ldq, int rows_per_group, void* Y, int y_dtype,
                                  int64_t ldy, float* ssq, void* keep, int keep_dtype, int M, int N, int K,
                                  int seg_cols, const float* extra, float* prod, float drop_p, uint32_t seed,
                                  const uint32_t* seed_dev, void* stream) {
  if (!X || !W || !bias || !Q || !Y || !ssq || M <= 0 || N <= 0 || K <= 0)
    return set_error(VQA_B200_EINVAL, "mfb_fused: null operand or empty shape");
  if (N % 20 != 0) return set_error(VQA_B200_EINVAL, "mfb_fused: N (=k*o) must be a multiple of 20, got %d", N);
  if (seg_cols <= 0) seg_cols = N;
  if (N % seg_cols != 0 || (seg_cols != N && seg_cols % 40 != 0))
    return set_error(VQA_B200_EINVAL, "mfb_fused: seg_cols (%d) must divide N (%d) and be a multiple of 40", seg_cols, N);
  if (rows_per_group <= 0) rows_per_group = 1;
  if (!aligned16(bias) || !aligned16(Q) || (ldq * 4) % 16 != 0)
    return set_error(VQA_B200_EALIGN, "mfb_fused: bias / Q must be 16-byte aligned (ldq=%lld)", (long long)ldq);
  if (keep && !aligned16(keep)) return set_error(VQA_B200_EALIGN, "mfb_fused: keep must be 16-byte aligned");
  if ((extra && !aligned16(extra)) || (prod && !aligned16(prod)))
    return set_error(VQA_B200_EALIGN, "mfb_fused: extra / prod must be 16-byte aligned");
  if (!(drop_p >= 0.f && drop_p < 1.f)) return set_error(VQA_B200_EINVAL, "mfb_fused: bad dropout p");
  GemmArgs g = {};
  g.M = M; g.N = N; g.K = K;
  g.bias = bias; g.rows_per_group = rows_per_group;
  g.mfb_q = Q; g.mfb_ldq = ldq;
  g.mfb_extra = extra; g.mfb_prod = prod;
  g.mfb_y = Y; g.mfb_ldy = ldy; g.mfb_y_bf16 = (y_dtype == VQA_B200_BF16);
  g.vec_ok = aligned16(Y) && ((ldy * (g.mfb_y_bf16 ? 2 : 4)) % 16 == 0);
  g.mfb_ssq = ssq; g.mfb_seg_cols = seg_cols; g.mfb_keep = keep; g.mfb_keep_f32 = (keep_dtype == VQA_B200_F32);
  g.drop_seed = seed;
  g.seed_dev = seed_dev;
  g.drop_thresh16 = (uint32_t)(drop_p * 65536.0f + 0.5f);
  g.drop_scale = g.drop_thresh16 ? 65536.0f / (65536.0f - (float)g.drop_thresh16) : 1.0f;
  g.k_split = 1; g.batch = 1;
  // segments / cascade operands belong to the vector blocks (M = batch rows): that instance runs single CTAs
  const bool extras = seg_cols != N || extra != nullptr || prod != nullptr;
  const bool cta2 = !extras && use_cta2(M, N, K, 1);
  CUtensorMap ta, tb;
  int rc = setup_operands(g, &ta, &tb, X, VQA_B200_K_MAJOR, ldx, W, VQA_B200_K_MAJOR, ldw, 240, 0, 0, cta2);
  if (rc) return rc;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (extras) return launch<240, EPI_MFB, false, true>(ta, tb, g, st);
  if (cta2) return launch<240, EPI_MFB, true>(ta, tb, g, st);
  return launch<240, EPI_MFB>(ta, tb, g, st);
}
