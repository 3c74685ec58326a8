// Host side of the tcgen05 GEMM: TMA tensor-map encoding, tile/split-K selection, kernel table and launch.
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <mutex>
#include <vector>

#include "common.h"

namespace rvae {

// ------------------------------------------------------------------------------------------------
// error state (thread local; read through rvae_last_error())
// ------------------------------------------------------------------------------------------------
static thread_local char g_last_error[512] = "";

int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_last_error, sizeof(g_last_error), fmt, ap);
  va_end(ap);
  return code;
}
int cuda_error(cudaError_t err, const char* what) {
  snprintf(g_last_error, sizeof(g_last_error), "CUDA error %d (%s) in %s", (int)err, cudaGetErrorString(err), what);
  return RVAE_ERR_CUDA_BASE + (int)err;
}
const char* last_error() { return g_last_error; }

// ------------------------------------------------------------------------------------------------
// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda)
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
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

// 2-D tensor map: dim0 (contiguous) x dim1 rows with pitch `ld` elements; 128-byte swizzle; OOB reads zero, OOB
// writes are dropped.
static int encode_2d(CUtensorMap* tm, const void* base, bool f32, uint64_t dim0, uint64_t dim1, uint64_t ld,
                     uint32_t box0, uint32_t box1) {
  EncodeTiledFn fn = get_encode_fn();
  const uint64_t esz = f32 ? 4 : 2;
  RVAE_REQUIRE(fn != nullptr, RVAE_ERR_DRIVER, "cuTensorMapEncodeTiled entry point unavailable");
  RVAE_REQUIRE((reinterpret_cast<uintptr_t>(base) & 15) == 0, RVAE_ERR_INVALID, "tensor base %p not 16-byte aligned",
               base);
  RVAE_REQUIRE((ld * esz) % 16 == 0, RVAE_ERR_UNSUPPORTED, "row pitch %llu elements is not a multiple of 16 bytes",
               (unsigned long long)ld);
  cuuint64_t gdim[2] = {dim0, dim1};
  cuuint64_t gstride[1] = {ld * esz};
  cuuint32_t box[2] = {box0, box1};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(tm, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2,
                  const_cast<void*>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  RVAE_REQUIRE(r == CUDA_SUCCESS, RVAE_ERR_DRIVER,
               "cuTensorMapEncodeTiled failed (%d): dims %llu x %llu ld %llu box %u x %u", (int)r,
               (unsigned long long)dim0, (unsigned long long)dim1, (unsigned long long)ld, box0, box1);
  return RVAE_OK;
}
static int encode_bf16_2d(CUtensorMap* tm, const void* base, uint64_t dim0, uint64_t dim1, uint64_t ld,
                          uint32_t box0, uint32_t box1) {
  return encode_2d(tm, base, false, dim0, dim1, ld, box0, box1);
}

// Tensor maps of a prepared GEMM's epilogue (TMA stores and side-input loads): bf16 planes in boxes of 64 columns,
// fp32 in boxes of 32 columns, 128 rows each. Re-encodes only the maps whose base pointer changed.
int gemm_bind_outputs(PreparedGemm* g, const EpiArgs& a, bool force) {
  GemmParams& p = g->params;
  const EpiArgs old = p.epi;
  p.epi = a;
  if (a.out_hi && (force || a.out_hi != old.out_hi))
    RVAE_CHECK(encode_2d(&p.tmOutHi, a.out_hi, false, g->out_cols_bf16, g->out_rows, g->out_ld_bf16, 64, 128));
  if (a.out_lo && (force || a.out_lo != old.out_lo))
    RVAE_CHECK(encode_2d(&p.tmOutLo, a.out_lo, false, g->out_cols_bf16, g->out_rows, g->out_ld_bf16, 64, 128));
  if (a.out_f32 && (force || a.out_f32 != old.out_f32))
    RVAE_CHECK(encode_2d(&p.tmOutF32, a.out_f32, true, g->out_cols_f32, g->out_rows, g->out_ld_f32, 32, 128));
  if (a.out_f32_b && g->epi == EPI_HEAD && (force || a.out_f32_b != old.out_f32_b))
    RVAE_CHECK(encode_2d(&p.tmOutF32b, a.out_f32_b, true, g->out_cols_f32, g->out_rows, g->out_ld_f32, 32, 128));
  if (a.in0 && (force || a.in0 != old.in0 || a.ldi != old.ldi)) {
    if (g->epi == EPI_HEAD)  // eps, fp32 [M, L]
      RVAE_CHECK(encode_2d(&p.tmSide, a.in0, true, g->out_cols_f32, g->out_rows, g->out_ld_f32, 32, 128));
    else if (g->epi == EPI_OUT || g->epi == EPI_DRELU)  // x / ReLU mask, bf16 [M, N]
      RVAE_CHECK(encode_2d(&p.tmSide, a.in0, false, g->side_cols > 0 ? g->side_cols : g->out_cols_bf16, g->out_rows,
                           (g->epi == EPI_OUT && a.ldi > 0) ? a.ldi : g->out_ld_bf16, 64, 128));
  }
  return RVAE_OK;
}

// ------------------------------------------------------------------------------------------------
// kernel table
// ------------------------------------------------------------------------------------------------
typedef void (*GemmKernel)(const GemmParams);

struct Variant {
  int block_n, a_major, b_major, epi, cg;
  GemmKernel fn;
  int smem;
};

#define RVAE_VARIANT(BN, AM, BM, EP)                                                          \
  { BN, AM, BM, EP, 1, gemm_kernel<BN, AM, BM, EP>, GemmCfg<BN, 1>::kSmemBytes },             \
  { BN, AM, BM, EP, 2, gemm_kernel_2cta<BN, AM, BM, EP>, GemmCfg<BN, 2>::kSmemBytes }

static const Variant kVariants[] = {
    RVAE_VARIANT(256, MAJOR_K, MAJOR_K, EPI_LINEAR),  RVAE_VARIANT(128, MAJOR_K, MAJOR_K, EPI_LINEAR),
    RVAE_VARIANT(256, MAJOR_K, MAJOR_K, EPI_HEAD),    RVAE_VARIANT(128, MAJOR_K, MAJOR_K, EPI_HEAD),
    RVAE_VARIANT(256, MAJOR_K, MAJOR_K, EPI_OUT),     RVAE_VARIANT(128, MAJOR_K, MAJOR_K, EPI_OUT),
    RVAE_VARIANT(256, MAJOR_K, MAJOR_MN, EPI_DRELU),  RVAE_VARIANT(128, MAJOR_K, MAJOR_MN, EPI_DRELU),
    RVAE_VARIANT(256, MAJOR_K, MAJOR_MN, EPI_REDUCE),  RVAE_VARIANT(128, MAJOR_K, MAJOR_MN, EPI_REDUCE),
    RVAE_VARIANT(256, MAJOR_MN, MAJOR_MN, EPI_REDUCE), RVAE_VARIANT(128, MAJOR_MN, MAJOR_MN, EPI_REDUCE),
#if RVAE_EXPERIMENTS
    // latent dgrad with the reparameterisation / KL backward fused: pair tiles only
    {256, MAJOR_K, MAJOR_MN, EPI_DLATENT, 2, gemm_kernel_2cta<256, MAJOR_K, MAJOR_MN, EPI_DLATENT>,
     GemmCfg<256, 2>::kSmemBytes},
#endif
};
static const int kNumVariants = sizeof(kVariants) / sizeof(kVariants[0]);

static int find_variant(int block_n, int a_major, int b_major, int epi, int cg) {
  for (int i = 0; i < kNumVariants; ++i)
    if (kVariants[i].block_n == block_n && kVariants[i].a_major == a_major && kVariants[i].b_major == b_major &&
        kVariants[i].epi == epi && kVariants[i].cg == cg)
      return i;
  return -1;
}

static int configure_variants() {
  static int rc = -1;
  static std::once_flag once;
  std::call_once(once, [] {
    rc = RVAE_OK;
    for (int i = 0; i < kNumVariants; ++i) {
      cudaError_t e = cudaFuncSetAttribute(reinterpret_cast<const void*>(kVariants[i].fn),
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, kVariants[i].smem);
      if (e != cudaSuccess) {
        rc = cuda_error(e, "cudaFuncSetAttribute(MaxDynamicSharedMemorySize)");
        break;
      }
    }
  });
  return rc;
}

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// Pick the tile: cta_group 2 (256-row pair tiles) whenever there are at least two 128-row blocks; for N, fewer and
// fatter tiles are more efficient per FLOP, but whole waves over the SMs (or SM pairs) matter more.
static void choose_tile(const Ctx* ctx, int M, int N, bool allow128, bool allow256, int* block_n, int* cg) {
  int g = (M > kBlockM) ? 2 : 1;
  if (ctx->force_cta_group == 1 || ctx->force_cta_group == 2) g = ctx->force_cta_group;
  *cg = g;
  const int slots = ctx->num_sms / g;
  const int mb = ceil_div(M, kBlockM * g);
  if (ctx->force_block_n == 128 && allow128) { *block_n = 128; return; }
  if (ctx->force_block_n == 256 && allow256) { *block_n = 256; return; }
  if (!allow256) { *block_n = 128; return; }
  if (!allow128) { *block_n = 256; return; }
  if (N % 256 != 0) { *block_n = 128; return; }
  const double c256 = 1.0 * ceil_div(mb * ceil_div(N, 256), slots);
  const double c128 = 0.6 * ceil_div(mb * ceil_div(N, 128), slots);
  *block_n = (c128 < c256) ? 128 : 256;
}

int gemm_prepare(const Ctx* ctx, const GemmDesc& d, PreparedGemm* out) {
  RVAE_REQUIRE(d.M > 0 && d.N > 0 && d.K > 0, RVAE_ERR_INVALID, "gemm: empty problem %d x %d x %d", d.M, d.N, d.K);
  RVAE_REQUIRE(d.A.hi && d.B.hi, RVAE_ERR_INVALID, "gemm: null operand");
  RVAE_REQUIRE(d.N % 64 == 0, RVAE_ERR_UNSUPPORTED, "gemm: N=%d must be a multiple of 64", d.N);
  RVAE_CHECK(configure_variants());

  PreparedGemm& g = *out;
  memset(&g, 0, sizeof(g));
  GemmParams& p = g.params;
  p.M = d.M; p.N = d.N; p.K = d.K;
  p.epi = d.args;
  p.debug = ctx->debug;
  p.trace = nullptr;

  int block_n, cg;
  if (d.epi == EPI_HEAD) {
    const int L = d.head_L;
    RVAE_REQUIRE(d.N == 2 * L && L % 64 == 0, RVAE_ERR_UNSUPPORTED, "head gemm: N=%d must be 2*L, L=%d %% 64 == 0",
                 d.N, L);
    choose_tile(ctx, d.M, d.N, true, L % 128 == 0, &block_n, &cg);
    p.n_blocks = L / (block_n / 2);
    p.b_tile_stride = block_n / 2;
    p.b_half_stride = L;
    p.epi.L = L;
  } else {
    // reduce-add GEMMs (weight gradients, latent dgrad): 256-wide tiles, split-K fills the machine; others: by
    // wave count
    choose_tile(ctx, d.M, d.N, d.epi != EPI_DLATENT && (d.epi != EPI_REDUCE || d.N % 256 != 0), true, &block_n, &cg);
    if (d.epi == EPI_DLATENT)
      RVAE_REQUIRE(d.args.in0 && d.args.in1 && d.args.in2 && d.args.out_hi && !d.args.out_lo && !d.A.lo && !d.B.lo &&
                       d.args.L == d.N && d.args.ldo == 2 * d.N,
                   RVAE_ERR_UNSUPPORTED, "latent dgrad gemm: bf16 mode with eps, logvar, mu and d_ml [M, 2L] only");
    p.n_blocks = ceil_div(d.N, block_n);
    p.b_tile_stride = block_n;
    p.b_half_stride = block_n / 2;
  }
  p.m_blocks = ceil_div(d.M, kBlockM * cg);
  const int slots = ctx->num_sms / cg;
  p.kb_total = ceil_div(d.K, kBlockK);

  // split-K only where the epilogue is a linear accumulation
  int splits = 1;
  if (d.epi == EPI_REDUCE) {
    const int tiles = p.m_blocks * p.n_blocks;
    static const int env_splits = getenv("RVAE_WGRAD_SPLITS") ? atoi(getenv("RVAE_WGRAD_SPLITS")) : 0;
    if (d.k_splits > 0) {
      splits = d.k_splits;
    } else if (env_splits > 0 && d.A.major == MAJOR_MN) {   // experiments: finer weight-gradient units
      splits = env_splits;
    } else {
      // smallest split (<= 8, >= 8 k-blocks each) whose last wave is >= 90% full; else the best seen
      double best = 0.0;
      for (int s = 1; s <= 8 && p.kb_total / s >= 8; ++s) {
        const int units = tiles * s;
        const double eff = (double)units / (ceil_div(units, slots) * (double)slots);
        if (eff > best + 1e-9) { best = eff; splits = s; }
        if (eff >= 0.90) break;
      }
    }
    if (splits > p.kb_total) splits = p.kb_total;
    RVAE_REQUIRE(splits == 1 || d.args.accumulate, RVAE_ERR_INVALID, "reduce gemm: split-K needs accumulate=1");
  }
  p.kb_per_split = ceil_div(p.kb_total, splits);
  p.k_splits = ceil_div(p.kb_total, p.kb_per_split);  // every split owns >= 1 k-block

  // passes: hi*hi (+ hi*lo + lo*hi when both operands carry a residual plane)
  const Operand* pa[kMaxPasses];
  const void* a_ptr[kMaxPasses];
  const void* b_ptr[kMaxPasses];
  (void)pa;
  int np = 0;
  if (d.A.lo && d.B.lo) {
    a_ptr[np] = d.A.lo; b_ptr[np] = d.B.hi; ++np;
    a_ptr[np] = d.A.hi; b_ptr[np] = d.B.lo; ++np;
  } else if (d.A.lo) {
    a_ptr[np] = d.A.lo; b_ptr[np] = d.B.hi; ++np;
  } else if (d.B.lo) {
    a_ptr[np] = d.A.hi; b_ptr[np] = d.B.lo; ++np;
  }
  a_ptr[np] = d.A.hi; b_ptr[np] = d.B.hi; ++np;
  p.num_passes = np;

  const int b_rows = (d.epi == EPI_HEAD) ? d.N : d.N;
  // extent of an operand's contiguous dimension in its tensor map: columns past Operand::cols read as zeros
  auto dim0 = [](const Operand& o, int extent) { return (uint64_t)(o.cols > 0 && o.cols < extent ? o.cols : extent); };
  for (int i = 0; i < np; ++i) {
    if (d.A.major == MAJOR_K)
      RVAE_CHECK(encode_bf16_2d(&p.tmA[i], a_ptr[i], dim0(d.A, d.K), d.M, d.A.ld, kBlockK, kBlockM));
    else
      RVAE_CHECK(encode_bf16_2d(&p.tmA[i], a_ptr[i], dim0(d.A, d.M), d.K, d.A.ld, 64, kBlockK));
    if (d.B.major == MAJOR_K)
      RVAE_CHECK(encode_bf16_2d(&p.tmB[i], b_ptr[i], dim0(d.B, d.K), b_rows, d.B.ld, kBlockK, block_n / 2));
    else
      RVAE_CHECK(encode_bf16_2d(&p.tmB[i], b_ptr[i], dim0(d.B, d.N), d.K, d.B.ld, 64, kBlockK));
  }

  // epilogue tensors (what the TMA stores write and the side-input loads read)
  g.epi = d.epi;
  g.out_rows = d.M;
  g.side_cols = d.epi == EPI_OUT ? d.side_cols : 0;
  if (d.epi == EPI_HEAD) {            // z [M, L] bf16; mu, logvar, eps [M, L] fp32
    g.out_cols_bf16 = d.head_L; g.out_ld_bf16 = d.head_L;
    g.out_cols_f32 = d.head_L; g.out_ld_f32 = d.head_L;
  } else if (d.epi == EPI_DLATENT) {  // d_ml = [d_mu | d_logvar], [M, 2L] bf16
    g.out_cols_bf16 = 2 * d.N; g.out_ld_bf16 = d.args.ldo;
    g.out_cols_f32 = d.N; g.out_ld_f32 = d.N;
  } else {
    g.out_cols_bf16 = d.N; g.out_ld_bf16 = d.args.ldo;
    g.out_cols_f32 = d.N; g.out_ld_f32 = d.args.ldo;
  }
  RVAE_CHECK(gemm_bind_outputs(&g, p.epi, true));

  g.block_n = block_n;
  g.a_major = d.A.major; g.b_major = d.B.major; g.cg = cg;
  g.variant = find_variant(block_n, d.A.major, d.B.major, d.epi, cg);
  RVAE_REQUIRE(g.variant >= 0, RVAE_ERR_UNSUPPORTED, "gemm: no kernel for block_n=%d majors (%d,%d) epilogue %d",
               block_n, d.A.major, d.B.major, d.epi);
  // Persistent grid: the fewest CTAs (pairs) that still finish in the same number of waves. What wave quantisation
  // would leave idle in the last wave is left idle for the whole kernel instead - those SMs run the concurrent
  // HBM-bound work of the step (noise, Adam, all-reduce) without taking anything from this GEMM.
  const int units = p.m_blocks * p.n_blocks * p.k_splits;
  const int waves = ceil_div(units, slots);
  const int slots_eff = ceil_div(units, waves);
  g.grid = cg * (units < slots_eff ? units : slots_eff);
  g.smem_bytes = kVariants[g.variant].smem;
  return RVAE_OK;
}

int gemm_run(Ctx* ctx, const PreparedGemm& g, cudaStream_t stream) {
  if (ctx->trace != nullptr) {  // debug: successive launches write successive slabs of the trace buffer
    GemmParams p = g.params;
    const uint64_t slab = ctx->trace_launches > 1 ? ctx->trace_seq % (uint64_t)ctx->trace_launches : 0;
    p.trace = ctx->trace + slab * (uint64_t)ctx->num_sms_total * kTraceCtaWords;
    ctx->trace_seq++;
    RVAE_CUDA(launch_kernel(ctx, kVariants[g.variant].fn, dim3(g.grid), dim3(kGemmThreads), (size_t)g.smem_bytes,
                            stream, p));
    ctx->launches++;
    return RVAE_OK;
  }
  RVAE_CUDA(launch_kernel(ctx, kVariants[g.variant].fn, dim3(g.grid), dim3(kGemmThreads), (size_t)g.smem_bytes, stream,
                          g.params));
  ctx->launches++;
  return RVAE_OK;
}

// ------------------------------------------------------------------------------------------------
// fused launches of several GEMMs
// ------------------------------------------------------------------------------------------------
typedef void (*ChainKernel)(const ChainParams);
struct KindId {
  int a, b, e;
};
struct ChainVariant {
  int count;
  KindId k[kMaxChain];
  ChainKernel fn;
};
using KDrelu = Kind<MAJOR_K, MAJOR_MN, EPI_DRELU>;
using KWgrad = Kind<MAJOR_MN, MAJOR_MN, EPI_REDUCE>;
using KDz = Kind<MAJOR_K, MAJOR_MN, EPI_REDUCE>;
using KDlat = Kind<MAJOR_K, MAJOR_MN, EPI_DLATENT>;
using KLinear = Kind<MAJOR_K, MAJOR_K, EPI_LINEAR>;
using KHead = Kind<MAJOR_K, MAJOR_K, EPI_HEAD>;
using KOut = Kind<MAJOR_K, MAJOR_K, EPI_OUT>;
#define RVAE_KID(K) {K::A, K::B, K::EPI}
static const ChainVariant kChainVariants[] = {
    // dgrad + ReLU mask | weight gradient            (backward stages 0 and 2)
    {2, {RVAE_KID(KDrelu), RVAE_KID(KWgrad)}, gemm_chain_kernel_2cta<256, KDrelu, KWgrad, NoKind, NoKind>},
    // split-K latent dgrad | weight gradient         (backward stage 1)
    {2, {RVAE_KID(KDz), RVAE_KID(KWgrad)}, gemm_chain_kernel_2cta<256, KDz, KWgrad, NoKind, NoKind>},

#if RVAE_EXPERIMENTS
    // dgrad + ReLU mask | weight gradient | the previous stage's weight gradient   (stage 2 with B3w riding along:
    // measured equal at N = 1 and 1.2 % slower at N = 2 than the split stage 1, profiles/README.md)
    {3, {RVAE_KID(KDrelu), RVAE_KID(KWgrad), RVAE_KID(KWgrad)}, gemm_chain_kernel_2cta<256, KDrelu, KWgrad, KWgrad, NoKind>},
    // latent dgrad with fused reparameterisation / KL backward | weight gradient   (backward stage 1, bf16 mode)
    {2, {RVAE_KID(KDlat), RVAE_KID(KWgrad)}, gemm_chain_kernel_2cta<256, KDlat, KWgrad, NoKind, NoKind>},
    // layers chained by tile-level dependencies: fc1 -> head, fc3 -> fc4 + loss, and the whole forward pass
    {2, {RVAE_KID(KLinear), RVAE_KID(KHead)}, gemm_chain_kernel_2cta<256, KLinear, KHead, NoKind, NoKind>},
    {2, {RVAE_KID(KLinear), RVAE_KID(KOut)}, gemm_chain_kernel_2cta<256, KLinear, KOut, NoKind, NoKind>},
    {4, {RVAE_KID(KLinear), RVAE_KID(KHead), RVAE_KID(KLinear), RVAE_KID(KOut)},
     gemm_chain_kernel_2cta<256, KLinear, KHead, KLinear, KOut>},
#endif
};
static const int kNumChainVariants = sizeof(kChainVariants) / sizeof(kChainVariants[0]);

static int configure_chain_variants() {
  static int rc = -1;
  static std::once_flag once;
  std::call_once(once, [] {
    rc = RVAE_OK;
    for (int i = 0; i < kNumChainVariants; ++i) {
      cudaError_t e = cudaFuncSetAttribute(reinterpret_cast<const void*>(kChainVariants[i].fn),
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, GemmCfg<256, 2>::kSmemBytes);
      if (e != cudaSuccess) {
        rc = cuda_error(e, "cudaFuncSetAttribute(MaxDynamicSharedMemorySize)");
        break;
      }
    }
  });
  return rc;
}

// Estimated cost of one unit in k-block times: the MMA main loop, or the epilogue when that is longer (it overlaps
// the next unit's main loop), plus a fixed hand-over cost.
static double unit_cost(const PreparedGemm& g) {
  const double mma = (double)g.params.kb_per_split * g.params.num_passes;
  const double epi = (g.epi == EPI_DRELU || g.epi == EPI_OUT) ? 11.0 : 8.0;
  // the fused latent epilogue is long and such a unit is the only one of its pair: nothing overlaps it
  if (g.epi == EPI_DLATENT) return mma + 22.0 + 2.0;
  return (mma > epi ? mma : epi) + 2.0;
}

int gemm_prepare_chain(const Ctx* ctx, const PreparedGemm* const* g, int count, int pairs, int* sched_dev,
                       PreparedChain* out, unsigned int* dep_flags) {
  RVAE_REQUIRE(count >= 2 && count <= kMaxChain, RVAE_ERR_INVALID, "chain gemm: %d problems", count);
  for (int i = 0; i < count; ++i)
    RVAE_REQUIRE(g[i]->block_n == 256 && g[i]->cg == 2, RVAE_ERR_UNSUPPORTED,
                 "chain gemm: every problem must use 256-wide pair tiles");
  RVAE_REQUIRE(sched_dev != nullptr && pairs >= 1 && 2 * pairs <= ctx->num_sms_total, RVAE_ERR_INVALID,
               "chain gemm: bad schedule buffer / pair count %d", pairs);
  RVAE_CHECK(configure_chain_variants());
  int variant = -1;
  for (int v = 0; v < kNumChainVariants && variant < 0; ++v) {
    const ChainVariant& cv = kChainVariants[v];
    if (cv.count != count) continue;
    bool match = true;
    for (int i = 0; i < count; ++i)
      match = match && cv.k[i].a == g[i]->a_major && cv.k[i].b == g[i]->b_major && cv.k[i].e == g[i]->epi;
    if (match) variant = v;
  }
  RVAE_REQUIRE(variant >= 0, RVAE_ERR_UNSUPPORTED, "chain gemm: no fused kernel for this combination of problems");
  int nunits[kMaxChain], base[kMaxChain + 1];
  base[0] = 0;
  for (int i = 0; i < kMaxChain; ++i) {
    nunits[i] = i < count ? g[i]->params.m_blocks * g[i]->params.n_blocks * g[i]->params.k_splits : 0;
    base[i + 1] = base[i] + nunits[i];
  }
  RVAE_REQUIRE(base[kMaxChain] <= pairs * kSchedMax, RVAE_ERR_UNSUPPORTED, "chain gemm: %d units exceed the schedule",
               base[kMaxChain]);
  struct U { int id; double cost; };
  std::vector<U> units;
  units.reserve(base[kMaxChain]);
  if (dep_flags == nullptr) {
    // independent problems: longest-processing-time-first
    for (int i = 0; i < count; ++i)
      for (int u = 0; u < nunits[i]; ++u) units.push_back({base[i] + u, unit_cost(*g[i])});
    std::stable_sort(units.begin(), units.end(), [](const U& a, const U& b) { return a.cost > b.cost; });
  } else {
    // chained: layer by layer, row-block-major within a layer (unit = n_blk * m_blocks + m_blk), so that row blocks
    // complete one after the other and tiles that run at the same time share their A rows and B columns in L2
    for (int i = 0; i < count; ++i) {
      const int mb = g[i]->params.m_blocks, nb = g[i]->params.n_blocks;
      RVAE_REQUIRE(g[i]->params.k_splits == 1 && mb == g[0]->params.m_blocks && g[i]->params.M == g[0]->params.M &&
                       mb <= 256,
                   RVAE_ERR_UNSUPPORTED, "chain gemm: chained problems must share the row blocking");
      for (int m = 0; m < mb; ++m)
        for (int n = 0; n < nb; ++n) units.push_back({base[i] + n * mb + m, unit_cost(*g[i])});
    }
  }
  // each unit, in that order, to the least loaded pair: every pair runs a subsequence of the global order
  std::vector<double> load(pairs, 0.0);
  std::vector<int> cnt(pairs, 0);
  std::vector<int> sched((size_t)pairs * kSchedMax, -1);
  for (const U& u : units) {
    int best = -1;
    for (int pidx = 0; pidx < pairs; ++pidx)
      if (cnt[pidx] < kSchedMax && (best < 0 || load[pidx] < load[best] - 1e-9)) best = pidx;
    RVAE_REQUIRE(best >= 0, RVAE_ERR_UNSUPPORTED, "chain gemm: schedule overflow");
    sched[(size_t)best * kSchedMax + cnt[best]++] = u.id;
    load[best] += u.cost;
  }
  if (dep_flags == nullptr) {
    // Order WITHIN a pair (independent problems only). A unit's epilogue overlaps the next unit's MMAs, so a pair is
    // fastest when long-MMA units (split-K weight gradients: light epilogue) sit BETWEEN short-MMA, epilogue-heavy
    // units (dgrad tiles) instead of in front of them, where nothing overlaps their main loop: the heavy units are
    // spread evenly through the light ones, never first (measured on the role traces, profiles/README.md).
    static const int order_mode = getenv("RVAE_CHAIN_ORDER") ? atoi(getenv("RVAE_CHAIN_ORDER")) : 1;
    auto prob_of = [&](int id) { int q = 0; while (q + 1 < count && id >= base[q + 1]) ++q; return q; };
    for (int pidx = 0; pidx < pairs && order_mode == 1; ++pidx) {
      int* row = &sched[(size_t)pidx * kSchedMax];
      std::vector<int> heavy, light;
      double min_mma = 1e30;
      for (int k = 0; k < cnt[pidx]; ++k) {
        const PreparedGemm& gq = *g[prob_of(row[k])];
        min_mma = std::min(min_mma, (double)gq.params.kb_per_split * gq.params.num_passes);
      }
      for (int k = 0; k < cnt[pidx]; ++k) {
        const PreparedGemm& gq = *g[prob_of(row[k])];
        const double mma = (double)gq.params.kb_per_split * gq.params.num_passes;
        (mma > 1.5 * min_mma ? heavy : light).push_back(row[k]);
      }
      if (heavy.empty() || light.size() < 2) continue;
      std::vector<int> merged;
      const size_t nh = heavy.size(), nl = light.size();
      size_t li = 0;
      for (size_t h = 0; h < nh; ++h) {
        // light units before heavy unit h: an even share, at least one (two before the first when there are enough)
        size_t upto = (h + 1) * nl / (nh + 1);
        if (h == 0 && upto < 2 && nl >= 3) upto = 2;
        if (upto < li + (h == 0 ? 1 : 0)) upto = li + (h == 0 ? 1 : 0);
        if (upto > nl) upto = nl;
        while (li < upto) merged.push_back(light[li++]);
        merged.push_back(heavy[h]);
      }
      while (li < nl) merged.push_back(light[li++]);
      for (size_t k = 0; k < merged.size(); ++k) row[k] = merged[k];
    }
  }
  RVAE_CUDA(cudaMemcpy(sched_dev, sched.data(), sched.size() * sizeof(int), cudaMemcpyHostToDevice));
  PreparedChain& d = *out;
  memset(&d, 0, sizeof(d));
  for (int i = 0; i < kMaxChain; ++i) d.params.p[i] = g[i < count ? i : 0]->params;
  for (int i = 0; i <= kMaxChain; ++i) d.params.base[i] = base[i];
  d.params.sched = sched_dev;
  RVAE_REQUIRE(dep_flags == nullptr || RVAE_EXPERIMENTS, RVAE_ERR_UNSUPPORTED,
               "chain gemm: dependent problems need a build with RVAE_EXPERIMENTS=1");
  if (dep_flags != nullptr) {
    for (int i = 0; i + 1 < count; ++i) {
      unsigned int* flags = dep_flags + 256 * i;
      d.params.p[i].dep_signal = flags;
      d.params.p[i + 1].dep_wait = flags;
      d.params.p[i + 1].dep_target = (unsigned)(g[i]->params.n_blocks * 2 * kEpiTeams);  // tiles x CTAs x teams
    }
  }
  d.count = count;
  d.variant = variant;
  d.grid = 2 * pairs;
  d.smem_bytes = GemmCfg<256, 2>::kSmemBytes;
  return RVAE_OK;
}

int gemm_run_chain(Ctx* ctx, const PreparedChain& g, cudaStream_t stream) {
  if (ctx->trace != nullptr) {
    ChainParams p = g.params;
    const uint64_t slab = ctx->trace_launches > 1 ? ctx->trace_seq % (uint64_t)ctx->trace_launches : 0;
    for (int i = 0; i < kMaxChain; ++i) p.p[i].trace = ctx->trace + slab * (uint64_t)ctx->num_sms_total * kTraceCtaWords;
    ctx->trace_seq++;
    RVAE_CUDA(launch_kernel(ctx, kChainVariants[g.variant].fn, dim3(g.grid), dim3(kGemmThreads), (size_t)g.smem_bytes,
                            stream, p));
    ctx->launches++;
    return RVAE_OK;
  }
  RVAE_CUDA(launch_kernel(ctx, kChainVariants[g.variant].fn, dim3(g.grid), dim3(kGemmThreads), (size_t)g.smem_bytes,
                          stream, g.params));
  ctx->launches++;
  return RVAE_OK;
}

int gemm_launch(Ctx* ctx, const GemmDesc& d, cudaStream_t stream) {
  PreparedGemm g;
  RVAE_CHECK(gemm_prepare(ctx, d, &g));
  return gemm_run(ctx, g, stream);
}

}  // namespace rvae
