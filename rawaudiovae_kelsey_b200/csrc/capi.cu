// C ABI (include/rvae_b200.h): context, op-level entry points and the plan that issues a whole training or
// inference step from C. No torch types cross this boundary.
#include <cmath>
#include <cstdlib>
#include <dlfcn.h>
#include <cstring>
#include <map>
#include <new>
#include <utility>
#include <vector>

#include "../../include/rvae_b200.h"
#include "common.h"

namespace rvae {
const char* last_error();
}

using namespace rvae;

// NCCL entry points, resolved at run time from the libnccl the process already uses (torch's): no link-time
// dependency, and the communicator is created from an id the host side exchanges over torch.distributed.
struct NcclId {
  char internal[128];  // ncclUniqueId
};
struct NcclApi {
  void* handle;
  int (*GetUniqueId)(NcclId*);
  int (*CommInitRank)(void** comm, int nranks, NcclId id, int rank);
  int (*AllReduce)(const void* send, void* recv, size_t count, int dtype, int op, void* comm, cudaStream_t stream);
  int (*CommDestroy)(void* comm);
  const char* (*GetErrorString)(int);
};

struct rvae_ctx {
  Ctx c;
  NcclApi nccl;
  void* comm;      // ncclComm_t of the data-parallel group (nullptr = single process)
  int dp_rank, dp_world;
  // peer-memory all-reduce: this rank's symmetric allocation ([flags | gradient data]) and the peers' mappings
  uint8_t* sym_base;
  bool sym_owned;      // rvae_dp_sym_alloc made the allocation (else adopted from the caller: rvae_dp_sym_adopt)
  size_t sym_data_bytes;
  void* peer_base[kP2PMaxWorld];
  P2PArgs p2p;
  bool p2p_ready;
  int p2p_ctas;        // CTAs of an all-reduce that runs under the GEMMs (they live on the spare SMs)
  int p2p_ctas_last;   // CTAs of the step's last, exposed all-reduce
};

static inline cudaStream_t S_(void* s) { return reinterpret_cast<cudaStream_t>(s); }
static inline const __nv_bfloat16* BF(const void* p) { return reinterpret_cast<const __nv_bfloat16*>(p); }
static inline __nv_bfloat16* BF(void* p) { return reinterpret_cast<__nv_bfloat16*>(p); }

extern "C" {

int rvae_abi_version(void) { return RVAE_ABI_VERSION; }
int rvae_build_experiments(void) { return RVAE_EXPERIMENTS; }
const char* rvae_last_error(void) { return rvae::last_error(); }

int rvae_ctx_create(int device, rvae_ctx** out) {
  RVAE_REQUIRE(out != nullptr, RVAE_ERR_INVALID, "ctx_create: null out");
  int count = 0;
  RVAE_CUDA(cudaGetDeviceCount(&count));
  RVAE_REQUIRE(device >= 0 && device < count, RVAE_ERR_INVALID, "ctx_create: device %d of %d", device, count);
  cudaDeviceProp prop;
  RVAE_CUDA(cudaGetDeviceProperties(&prop, device));
  RVAE_REQUIRE(prop.major == 10, RVAE_ERR_UNSUPPORTED,
               "device %d is sm_%d%d; librvae_b200 contains sm_100a code only (no fallback path)", device, prop.major,
               prop.minor);
  rvae_ctx* ctx = new (std::nothrow) rvae_ctx();
  RVAE_REQUIRE(ctx != nullptr, RVAE_ERR_INVALID, "ctx_create: out of host memory");
  ctx->c.device = device;
  ctx->c.num_sms = prop.multiProcessorCount;
  ctx->c.num_sms_total = prop.multiProcessorCount;
  // RVAE_NUM_SMS caps the SMs the persistent GEMM grids occupy (leaves the rest to concurrent kernels, e.g. NCCL)
  if (const char* e = getenv("RVAE_NUM_SMS")) {
    const int v = atoi(e);
    if (v >= 2 && v <= prop.multiProcessorCount) ctx->c.num_sms = v & ~1;
  }
  ctx->c.launches = 0;
  ctx->c.aux_grid_cap = 0;
  memset(&ctx->nccl, 0, sizeof(ctx->nccl));
  ctx->comm = nullptr; ctx->dp_rank = 0; ctx->dp_world = 1;
  ctx->sym_base = nullptr; ctx->sym_owned = true; ctx->sym_data_bytes = 0; ctx->p2p_ready = false; ctx->p2p_ctas = 20; ctx->p2p_ctas_last = 48;
  memset(ctx->peer_base, 0, sizeof(ctx->peer_base));
  memset(&ctx->p2p, 0, sizeof(ctx->p2p));
  if (const char* e = getenv("RVAE_P2P_CTAS")) {
    const int v = atoi(e);
    if (v >= 1 && v <= kP2PMaxCtas) ctx->p2p_ctas = v;
  }
  if (const char* e = getenv("RVAE_P2P_CTAS_LAST")) {
    const int v = atoi(e);
    if (v >= 1 && v <= kP2PMaxCtas) ctx->p2p_ctas_last = v;
  }
  ctx->c.trace = nullptr;
  ctx->c.trace_launches = 1;
  ctx->c.trace_seq = 0;
  ctx->c.aux_trace = nullptr; ctx->c.aux_cap = 0; ctx->c.aux_seq = 0;
  ctx->c.force_block_n = 0;
  if (const char* e = getenv("RVAE_BLOCK_N")) ctx->c.force_block_n = atoi(e);
  ctx->c.force_cta_group = 0;
  if (const char* e = getenv("RVAE_CTA_GROUP")) ctx->c.force_cta_group = atoi(e);
  ctx->c.debug = 0;
  if (const char* e = getenv("RVAE_DEBUG")) ctx->c.debug = atoi(e);
  ctx->c.use_pdl = 1;
  if (const char* e = getenv("RVAE_PDL")) ctx->c.use_pdl = atoi(e);
  *out = ctx;
  return RVAE_OK;
}
void rvae_ctx_destroy(rvae_ctx* ctx) {
  if (!ctx) return;
  if (ctx->comm && ctx->nccl.CommDestroy) ctx->nccl.CommDestroy(ctx->comm);
  if (ctx->sym_owned) {
    for (int p = 0; p < kP2PMaxWorld; ++p)
      if (ctx->peer_base[p] && p != ctx->dp_rank) cudaIpcCloseMemHandle(ctx->peer_base[p]);
    if (ctx->sym_base) cudaFree(ctx->sym_base);
  }
  delete ctx;
}

static int nccl_load(rvae_ctx* ctx, const char* path) {
  if (ctx->nccl.handle) return RVAE_OK;
  void* h = dlopen(path && path[0] ? path : "libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  RVAE_REQUIRE(h != nullptr, RVAE_ERR_DRIVER, "dlopen(%s) failed: %s", path && path[0] ? path : "libnccl.so.2", dlerror());
  NcclApi a;
  a.handle = h;
  a.GetUniqueId = reinterpret_cast<int (*)(NcclId*)>(dlsym(h, "ncclGetUniqueId"));
  a.CommInitRank = reinterpret_cast<int (*)(void**, int, NcclId, int)>(dlsym(h, "ncclCommInitRank"));
  a.AllReduce = reinterpret_cast<int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t)>(dlsym(h, "ncclAllReduce"));
  a.CommDestroy = reinterpret_cast<int (*)(void*)>(dlsym(h, "ncclCommDestroy"));
  a.GetErrorString = reinterpret_cast<const char* (*)(int)>(dlsym(h, "ncclGetErrorString"));
  RVAE_REQUIRE(a.GetUniqueId && a.CommInitRank && a.AllReduce && a.CommDestroy && a.GetErrorString, RVAE_ERR_DRIVER,
               "libnccl lacks a required symbol");
  ctx->nccl = a;
  return RVAE_OK;
}
#define RVAE_NCCL(ctx, expr)                                                                             \
  do {                                                                                                   \
    const int _r = (expr);                                                                               \
    if (_r != 0) return set_error(RVAE_ERR_DRIVER, "NCCL error %d (%s) in %s", _r, (ctx)->nccl.GetErrorString(_r), #expr); \
  } while (0)

int rvae_dp_unique_id(rvae_ctx* ctx, const char* libnccl_path, void* out128) {
  RVAE_REQUIRE(ctx != nullptr && out128 != nullptr, RVAE_ERR_INVALID, "dp_unique_id: null argument");
  RVAE_CHECK(nccl_load(ctx, libnccl_path));
  NcclId id;
  RVAE_NCCL(ctx, ctx->nccl.GetUniqueId(&id));
  memcpy(out128, &id, sizeof(id));
  return RVAE_OK;
}

int rvae_dp_init(rvae_ctx* ctx, const char* libnccl_path, const void* id128, int rank, int world) {
  RVAE_REQUIRE(ctx != nullptr && id128 != nullptr, RVAE_ERR_INVALID, "dp_init: null argument");
  RVAE_REQUIRE(world >= 1 && rank >= 0 && rank < world, RVAE_ERR_INVALID, "dp_init: rank %d of %d", rank, world);
  RVAE_REQUIRE(ctx->comm == nullptr, RVAE_ERR_STATE, "dp_init: communicator already created");
  RVAE_CHECK(nccl_load(ctx, libnccl_path));
  NcclId id;
  memcpy(&id, id128, sizeof(id));
  RVAE_CUDA(cudaSetDevice(ctx->c.device));
  RVAE_NCCL(ctx, ctx->nccl.CommInitRank(&ctx->comm, world, id, rank));
  ctx->dp_rank = rank;
  ctx->dp_world = world;
  return RVAE_OK;
}

int rvae_dp_world(const rvae_ctx* ctx) { return ctx && ctx->comm ? ctx->dp_world : 1; }

int rvae_dp_allreduce(rvae_ctx* ctx, float* ptr, int64_t count, int bucket, void* stream) {
  RVAE_REQUIRE(ctx && ptr && count > 0, RVAE_ERR_INVALID, "dp_allreduce: bad argument");
  const uint8_t* g0 = reinterpret_cast<const uint8_t*>(ptr);
  if (ctx->p2p_ready && g0 >= ctx->sym_base + kP2PFlagBytes &&
      g0 + sizeof(float) * (size_t)count <= ctx->sym_base + kP2PFlagBytes + ctx->sym_data_bytes) {
    P2PSegs sg;
    memset(&sg, 0, sizeof(sg));
    sg.off[0] = ptr - ctx->p2p.data[ctx->p2p.rank];
    sg.n[0] = count;
    return launch_allreduce_p2p(&ctx->c, ctx->p2p, sg, bucket, ctx->p2p_ctas, S_(stream));
  }
  RVAE_REQUIRE(ctx->comm != nullptr, RVAE_ERR_STATE, "dp_allreduce: no communicator (rvae_dp_init / rvae_dp_sym_open)");
  RVAE_NCCL(ctx, ctx->nccl.AllReduce(ptr, ptr, (size_t)count, /*ncclFloat32*/ 7, /*ncclSum*/ 0, ctx->comm, S_(stream)));
  return RVAE_OK;
}

int rvae_dp_sym_alloc(rvae_ctx* ctx, size_t data_bytes, void** data_ptr, void* ipc_handle64) {
  RVAE_REQUIRE(ctx && data_ptr && ipc_handle64 && data_bytes > 0, RVAE_ERR_INVALID, "dp_sym_alloc: bad argument");
  RVAE_REQUIRE(ctx->sym_base == nullptr, RVAE_ERR_STATE, "dp_sym_alloc: already allocated");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  RVAE_CUDA(cudaSetDevice(ctx->c.device));
  const size_t bytes = kP2PFlagBytes + ((data_bytes + 255) / 256) * 256;
  void* base = nullptr;
  RVAE_CUDA(cudaMalloc(&base, bytes));
  RVAE_CUDA(cudaMemset(base, 0, bytes));
  cudaIpcMemHandle_t h;
  RVAE_CUDA(cudaIpcGetMemHandle(&h, base));
  memcpy(ipc_handle64, &h, sizeof(h));
  ctx->sym_base = reinterpret_cast<uint8_t*>(base);
  ctx->sym_data_bytes = data_bytes;
  *data_ptr = ctx->sym_base + kP2PFlagBytes;
  return RVAE_OK;
}

// shared tail of rvae_dp_sym_open / rvae_dp_sym_adopt: ctx->peer_base[0..world) are mapped
static int finish_p2p_setup(rvae_ctx* ctx, int rank, int world);

size_t rvae_dp_sym_flag_bytes(void) { return kP2PFlagBytes; }

int rvae_dp_sym_adopt(rvae_ctx* ctx, const void* const* peer_bases, void* multicast_base, size_t data_bytes, int rank,
                      int world) {
  RVAE_REQUIRE(ctx && peer_bases && data_bytes > 0, RVAE_ERR_INVALID, "dp_sym_adopt: bad argument");
  RVAE_REQUIRE(ctx->sym_base == nullptr, RVAE_ERR_STATE, "dp_sym_adopt: a symmetric buffer is already set up");
  RVAE_REQUIRE(world >= 2 && world <= kP2PMaxWorld && rank >= 0 && rank < world, RVAE_ERR_INVALID,
               "dp_sym_adopt: rank %d of %d (at most %d ranks)", rank, world, kP2PMaxWorld);
  for (int p = 0; p < world; ++p)
    RVAE_REQUIRE(peer_bases[p] != nullptr && (reinterpret_cast<uintptr_t>(peer_bases[p]) & 255) == 0, RVAE_ERR_INVALID,
                 "dp_sym_adopt: peer %d base %p (need 256-byte alignment)", p, peer_bases[p]);
  RVAE_REQUIRE((reinterpret_cast<uintptr_t>(multicast_base) & 255) == 0, RVAE_ERR_INVALID, "dp_sym_adopt: multicast base");
  RVAE_CUDA(cudaSetDevice(ctx->c.device));
  for (int p = 0; p < world; ++p) ctx->peer_base[p] = const_cast<void*>(peer_bases[p]);
  ctx->sym_base = reinterpret_cast<uint8_t*>(ctx->peer_base[rank]);
  ctx->sym_data_bytes = data_bytes;
  ctx->sym_owned = false;   // the caller owns the allocation and the peer mappings
  RVAE_CHECK(finish_p2p_setup(ctx, rank, world));
  ctx->p2p.mc_data = multicast_base ? reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(multicast_base) + kP2PFlagBytes)
                                    : nullptr;
  if (const char* e = getenv("RVAE_NVLS")) if (atoi(e) == 0) ctx->p2p.mc_data = nullptr;
  return RVAE_OK;
}

int rvae_dp_uses_multicast(const rvae_ctx* ctx) { return ctx && ctx->p2p_ready && ctx->p2p.mc_data != nullptr; }

int rvae_dp_sym_open(rvae_ctx* ctx, const void* handles, int rank, int world) {
  RVAE_REQUIRE(ctx && handles && ctx->sym_base, RVAE_ERR_STATE, "dp_sym_open: call rvae_dp_sym_alloc first");
  RVAE_REQUIRE(world >= 2 && world <= kP2PMaxWorld && rank >= 0 && rank < world, RVAE_ERR_INVALID,
               "dp_sym_open: rank %d of %d (at most %d ranks)", rank, world, kP2PMaxWorld);
  RVAE_CUDA(cudaSetDevice(ctx->c.device));
  for (int p = 0; p < world; ++p) {
    void* base = ctx->sym_base;
    if (p != rank) {
      cudaIpcMemHandle_t h;
      memcpy(&h, reinterpret_cast<const uint8_t*>(handles) + 64 * p, sizeof(h));
      RVAE_CUDA(cudaIpcOpenMemHandle(&base, h, cudaIpcMemLazyEnablePeerAccess));
    }
    ctx->peer_base[p] = base;
  }
  return finish_p2p_setup(ctx, rank, world);
}

static int finish_p2p_setup(rvae_ctx* ctx, int rank, int world) {
  for (int p = 0; p < world; ++p) {
    void* base = ctx->peer_base[p];
    ctx->p2p.flags[p] = reinterpret_cast<uint32_t*>(base);
    ctx->p2p.data[p] = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(base) + kP2PFlagBytes);
  }
  ctx->p2p.mc_data = nullptr;
  // local: epochs and tickets behind the flag table
  static_assert(kP2PMaxBuckets * kP2PMaxCtas * kP2PMaxWorld * kP2PFlagStride * 4 + 2 * kP2PMaxBuckets * 4 + 4 <= kP2PFlagBytes,
                "flag area");
  ctx->p2p.epoch = reinterpret_cast<uint32_t*>(ctx->sym_base) + kP2PMaxBuckets * kP2PMaxCtas * kP2PMaxWorld * kP2PFlagStride;
  ctx->p2p.ticket = ctx->p2p.epoch + kP2PMaxBuckets;
  ctx->p2p.status = ctx->p2p.ticket + kP2PMaxBuckets;
  {  // how long a barrier waits for a peer before it records a failure (never a trap): minutes, in SM clocks
    double seconds = 600.0;
    if (const char* e = getenv("RVAE_P2P_TIMEOUT_S")) seconds = atof(e) > 0 ? atof(e) : seconds;
    int khz = 0;
    if (cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, ctx->c.device) != cudaSuccess || khz <= 0) khz = 1965000;
    ctx->p2p.timeout_cycles = static_cast<long long>(seconds * 1e3 * khz);
  }
  ctx->p2p.rank = rank;
  ctx->p2p.world = world;
  ctx->p2p.mode = 1;
  if (const char* e = getenv("RVAE_P2P_MODE")) ctx->p2p.mode = atoi(e);
  ctx->dp_rank = rank;
  ctx->dp_world = world;
  ctx->p2p_ready = true;
  return RVAE_OK;
}
int rvae_dp_status(rvae_ctx* ctx, unsigned int* status) {
  RVAE_REQUIRE(ctx && status, RVAE_ERR_INVALID, "dp_status: null argument");
  *status = 0;
  if (!ctx->p2p_ready) return RVAE_OK;
  // (synchronous 4-byte read on the legacy stream: call it where the host synchronises anyway - a loss read-back)
  RVAE_CUDA(cudaMemcpy(status, ctx->p2p.status, sizeof(unsigned int), cudaMemcpyDeviceToHost));
  return RVAE_OK;
}
int rvae_ctx_num_sms(const rvae_ctx* ctx) { return ctx ? ctx->c.num_sms : 0; }
uint64_t rvae_ctx_launch_count(const rvae_ctx* ctx) { return ctx ? ctx->c.launches : 0; }

#define CTX_OR_FAIL(ctx) RVAE_REQUIRE((ctx) != nullptr, RVAE_ERR_INVALID, "null rvae_ctx")

int rvae_debug_set_aux_trace(rvae_ctx* ctx, void* buf, int launches) {
  CTX_OR_FAIL(ctx);
  ctx->c.aux_trace = reinterpret_cast<unsigned long long*>(buf);
  ctx->c.aux_cap = buf ? launches : 0;
  ctx->c.aux_seq = 0;
  return RVAE_OK;
}

int rvae_debug_set_trace(rvae_ctx* ctx, void* buf, int launches) {
  CTX_OR_FAIL(ctx);
  RVAE_REQUIRE(launches >= 1, RVAE_ERR_INVALID, "debug_set_trace: launches=%d", launches);
  ctx->c.trace_launches = launches;
  ctx->c.trace_seq = 0;
  static_assert(RVAE_TRACE_WORDS_PER_CTA == kTraceCtaWords && RVAE_TRACE_HEADER_WORDS == kTraceHeader &&
                    RVAE_TRACE_TILES == kTraceTiles && RVAE_TRACE_EVENTS == kTraceEvents,
                "trace layout");
  ctx->c.trace = reinterpret_cast<unsigned long long*>(buf);
  return RVAE_OK;
}

int rvae_frame_gather(rvae_ctx* ctx, const void* audio, int audio_is_i16, int64_t n_samples,
                      const int64_t* frame_idx, int64_t first_frame, int64_t n_frames, int hop, int S, void* out_hi,
                      void* out_lo, float* out_f32, void* stream) {
  CTX_OR_FAIL(ctx);
  return launch_frame_gather(&ctx->c, audio, audio_is_i16, n_samples, frame_idx, first_frame, n_frames, hop, S, S,
                             BF(out_hi), BF(out_lo), out_f32, S_(stream));
}
int rvae_overlap_add(rvae_ctx* ctx, const float* frames, int64_t n_frames, int S, int hop, float* out, int64_t t_begin,
                     int64_t n_out, void* stream) {
  CTX_OR_FAIL(ctx);
  return launch_overlap_add(&ctx->c, frames, n_frames, S, hop, out, t_begin, n_out, S_(stream));
}
int rvae_randn(rvae_ctx* ctx, float* out, int64_t n, uint64_t seed, uint64_t offset, int64_t elem_base,
               void* stream) {
  CTX_OR_FAIL(ctx);
  RVAE_REQUIRE(elem_base >= 0, RVAE_ERR_INVALID, "randn: elem_base %lld", (long long)elem_base);
  // a base that is not a multiple of 4 starts inside a Philox block (a shard of a [B, L] draw with odd L): one row
  // of the element-wise kernel
  if (elem_base % 4 != 0) return launch_randn_rows(&ctx->c, out, 1, n, n, seed, offset, nullptr, elem_base, S_(stream));
  return launch_randn(&ctx->c, out, n, seed, offset, nullptr, elem_base, S_(stream));
}
int rvae_lerp_reparameterize(rvae_ctx* ctx, const float* mu_a, const float* logvar_a, const float* mu_b,
                             const float* logvar_b, const void* alpha, int alpha_is_f64, const float* eps,
                             int64_t rows, int L, float* z, float* mu_out, float* logvar_out, void* stream) {
  CTX_OR_FAIL(ctx);
  return launch_lerp_reparam(&ctx->c, mu_a, logvar_a, mu_b, logvar_b, alpha, alpha_is_f64, eps, rows, L, L, z, nullptr,
                             nullptr, mu_out, logvar_out, S_(stream));
}
int rvae_split_bf16(rvae_ctx* ctx, const float* src, int64_t n, void* hi, void* lo, void* stream) {
  CTX_OR_FAIL(ctx);
  return launch_split_bf16(&ctx->c, src, n, BF(hi), BF(lo), S_(stream));
}
int rvae_reparameterize(rvae_ctx* ctx, const float* mu, const float* logvar, const float* eps, int64_t n, float* z,
                        void* stream) {
  CTX_OR_FAIL(ctx);
  return launch_reparam(&ctx->c, mu, logvar, eps, n, z, S_(stream));
}
int rvae_loss_fwd(rvae_ctx* ctx, const float* xhat, const float* x, const float* mu, const float* logvar, int64_t B,
                  int S, int L, float beta, double* acc, float* loss_out, void* stream) {
  CTX_OR_FAIL(ctx);
  return launch_loss_fwd(&ctx->c, xhat, x, mu, logvar, B, S, L, beta, acc, loss_out, S_(stream));
}
int rvae_frame_loss(rvae_ctx* ctx, const float* xhat, int ld_xhat, const float* mu, const float* logvar, int ld_lat,
                    int64_t rows, int S, int L, const void* audio, int audio_is_i16, int64_t n_samples,
                    int64_t first_frame, int hop, float* rec_out, float* kl_out, void* stream) {
  // arguments first: a malformed call is reported the same way with or without a device
  RVAE_REQUIRE(xhat && mu && logvar && audio && rec_out && kl_out, RVAE_ERR_INVALID, "frame_loss: null buffer");
  RVAE_REQUIRE(rows > 0 && S > 0 && L > 0, RVAE_ERR_INVALID, "frame_loss: rows %lld, S %d, L %d (need > 0)",
               (long long)rows, S, L);
  RVAE_REQUIRE(ld_xhat >= S && ld_lat >= L, RVAE_ERR_INVALID, "frame_loss: row pitch ld_xhat %d < S %d or ld_lat %d < L %d",
               ld_xhat, S, ld_lat, L);
  RVAE_REQUIRE(hop > 0 && n_samples >= 0 && first_frame >= 0, RVAE_ERR_INVALID,
               "frame_loss: hop %d, n_samples %lld, first_frame %lld (need hop > 0, n_samples >= 0, first_frame >= 0)",
               hop, (long long)n_samples, (long long)first_frame);
  CTX_OR_FAIL(ctx);
  return launch_frame_loss(&ctx->c, xhat, ld_xhat, mu, logvar, ld_lat, rows, S, L, audio, audio_is_i16, n_samples,
                           first_frame, hop, rec_out, kl_out, S_(stream));
}
int rvae_loss_bwd(rvae_ctx* ctx, const float* xhat, const float* x, const float* mu, const float* logvar, int64_t B,
                  int S, int L, float beta, const float* grad_out, float* g_xhat, float* g_mu, float* g_logvar,
                  void* stream) {
  CTX_OR_FAIL(ctx);
  return launch_loss_bwd(&ctx->c, xhat, x, mu, logvar, B, S, L, beta, grad_out, g_xhat, g_mu, g_logvar, S_(stream));
}
int rvae_tanh_bwd(rvae_ctx* ctx, const float* g_xhat, const float* xhat, int64_t n, void* da_hi, void* da_lo,
                  void* stream) {
  CTX_OR_FAIL(ctx);
  return launch_tanh_bwd(&ctx->c, g_xhat, xhat, n, BF(da_hi), BF(da_lo), S_(stream));
}
int rvae_colsum(rvae_ctx* ctx, const void* hi, const void* lo, int64_t M, int N, int ld, float* out, int accumulate,
                void* stream) {
  CTX_OR_FAIL(ctx);
  return launch_colsum(&ctx->c, BF(hi), BF(lo), M, N, ld, out, accumulate, S_(stream));
}
int rvae_step_inc(rvae_ctx* ctx, float* step, void* stream) {
  CTX_OR_FAIL(ctx);
  return launch_step_inc(&ctx->c, step, S_(stream));
}
int rvae_adam_step(rvae_ctx* ctx, float* p, const float* g, float* m, float* v, int64_t n, double lr, double beta1,
                   double beta2, double eps, double weight_decay, float grad_scale, const float* step, void* shadow_hi,
                   void* shadow_lo, void* stream) {
  CTX_OR_FAIL(ctx);
  return launch_adam(&ctx->c, p, const_cast<float*>(g), m, v, n, lr, beta1, beta2, eps, weight_decay, grad_scale, step,
                     BF(shadow_hi), BF(shadow_lo), 0, S_(stream));
}
size_t rvae_param_histogram_bytes(int n_segs, int n_edges) { return param_histogram_bytes(n_segs, n_edges); }
int rvae_param_histogram(rvae_ctx* ctx, const float* params, const int64_t* seg_offsets_host,
                         const int64_t* seg_lengths_host, int n_segs, const double* edges_host, int n_edges,
                         void* record, void* stream) {
  CTX_OR_FAIL(ctx);
  return launch_param_histogram(&ctx->c, params, seg_offsets_host, seg_lengths_host, n_segs, edges_host, n_edges,
                                record, S_(stream));
}
int rvae_param_histogram_rows(rvae_ctx* ctx, const float* params, const int64_t* seg_offsets_host,
                              const int64_t* seg_rows_host, const int64_t* seg_cols_host, const int64_t* seg_pitch_host,
                              int n_segs, const double* edges_host, int n_edges, void* record, void* stream) {
  CTX_OR_FAIL(ctx);
  return launch_param_histogram_rows(&ctx->c, params, seg_offsets_host, seg_rows_host, seg_cols_host, seg_pitch_host,
                                     n_segs, edges_host, n_edges, record, S_(stream));
}

// ---------------------------------------------------------------------------------------------------------
// GEMM-level ops
// ---------------------------------------------------------------------------------------------------------
static GemmDesc desc_base(int epi, int M, int N, int K) {
  GemmDesc d;
  memset(&d, 0, sizeof(d));
  d.epi = epi; d.M = M; d.N = N; d.K = K;
  return d;
}
static Operand op(const void* hi, const void* lo, int major, int ld) {
  Operand o;
  o.hi = BF(hi); o.lo = BF(lo); o.major = major; o.ld = ld; o.cols = 0;
  return o;
}

int rvae_linear_act_fwd(rvae_ctx* ctx, const void* x_hi, const void* x_lo, const void* w_hi, const void* w_lo,
                        const float* bias, int M, int N, int K, int act, void* y_hi, void* y_lo, float* y_f32,
                        void* stream) {
  CTX_OR_FAIL(ctx);
  RVAE_REQUIRE(y_hi || y_f32, RVAE_ERR_INVALID, "linear_act_fwd: no output buffer");
  GemmDesc d = desc_base(EPI_LINEAR, M, N, K);
  d.A = op(x_hi, x_lo, MAJOR_K, K);
  d.B = op(w_hi, w_lo, MAJOR_K, K);
  d.args.bias = bias; d.args.act = act; d.args.ldo = N;
  d.args.out_hi = BF(y_hi); d.args.out_lo = BF(y_lo); d.args.out_f32 = y_f32;
  return gemm_launch(&ctx->c, d, S_(stream));
}

int rvae_encode_head_fwd(rvae_ctx* ctx, const void* h_hi, const void* h_lo, const void* w2_hi, const void* w2_lo,
                         const float* b2, int M, int L, int K, const float* eps, float* mu, float* logvar, void* z_hi,
                         void* z_lo, double* kl_acc, void* stream) {
  CTX_OR_FAIL(ctx);
  RVAE_REQUIRE(b2 && mu && logvar, RVAE_ERR_INVALID, "encode_head_fwd: null buffer");
  GemmDesc d = desc_base(EPI_HEAD, M, 2 * L, K);
  d.head_L = L;
  d.A = op(h_hi, h_lo, MAJOR_K, K);
  d.B = op(w2_hi, w2_lo, MAJOR_K, K);
  d.args.bias = b2; d.args.in0 = eps; d.args.out_f32 = mu; d.args.out_f32_b = logvar;
  d.args.out_hi = BF(z_hi); d.args.out_lo = BF(z_lo);
  d.args.loss_acc = kl_acc; d.args.L = L; d.args.ldo = L;
  return gemm_launch(&ctx->c, d, S_(stream));
}

int rvae_out_tanh_mse_fwd(rvae_ctx* ctx, const void* h_hi, const void* h_lo, const void* w4_hi, const void* w4_lo,
                          const float* b4, int M, int S, int K, const void* x_hi, const void* x_lo, int tanh_approx,
                          float* xhat, void* da_hi, void* da_lo, float grad_scale, double* mse_acc, float* bias_grad,
                          void* stream) {
  CTX_OR_FAIL(ctx);
  RVAE_REQUIRE(b4 && x_hi, RVAE_ERR_INVALID, "out_tanh_mse_fwd: null buffer");
  GemmDesc d = desc_base(EPI_OUT, M, S, K);
  d.A = op(h_hi, h_lo, MAJOR_K, K);
  d.B = op(w4_hi, w4_lo, MAJOR_K, K);
  d.args.bias = b4; d.args.in0 = x_hi; d.args.in1 = x_lo; d.args.out_f32 = xhat;
  d.args.out_hi = BF(da_hi); d.args.out_lo = BF(da_lo);
  d.args.act = tanh_approx ? ACT_TANH_APPROX : ACT_TANH;
  d.args.c0 = grad_scale; d.args.loss_acc = mse_acc; d.args.ldo = S; d.args.colsum = bias_grad;
  return gemm_launch(&ctx->c, d, S_(stream));
}

int rvae_dgrad_relu(rvae_ctx* ctx, const void* dy_hi, const void* dy_lo, const void* w_hi, const void* w_lo, int M,
                    int N, int Kd, const void* mask, void* dx_hi, void* dx_lo, float* bias_grad, void* stream) {
  CTX_OR_FAIL(ctx);
  RVAE_REQUIRE(dx_hi, RVAE_ERR_INVALID, "dgrad_relu: null output");
  GemmDesc d = desc_base(EPI_DRELU, M, N, Kd);
  d.A = op(dy_hi, dy_lo, MAJOR_K, Kd);
  d.B = op(w_hi, w_lo, MAJOR_MN, N);
  d.args.in0 = mask; d.args.out_hi = BF(dx_hi); d.args.out_lo = BF(dx_lo); d.args.ldo = N;
  d.args.colsum = bias_grad;
  return gemm_launch(&ctx->c, d, S_(stream));
}

int rvae_dgrad_latent(rvae_ctx* ctx, const void* da3_hi, const void* da3_lo, const void* w3_hi, const void* w3_lo,
                      int M, int L, int H, const float* eps, const float* logvar, const float* mu,
                      const float* g_mu_ext, const float* g_logvar_ext, float kl_grad_scale, float* dz_scratch,
                      void* dml_hi, void* dml_lo, float* bias_grad, void* stream) {
  CTX_OR_FAIL(ctx);
  RVAE_REQUIRE(eps && logvar && dz_scratch && dml_hi, RVAE_ERR_INVALID, "dgrad_latent: null buffer");
  RVAE_CUDA(cudaMemsetAsync(dz_scratch, 0, sizeof(float) * (size_t)M * L, S_(stream)));
  GemmDesc d = desc_base(EPI_REDUCE, M, L, H);
  d.A = op(da3_hi, da3_lo, MAJOR_K, H);
  d.B = op(w3_hi, w3_lo, MAJOR_MN, L);
  d.args.out_f32 = dz_scratch; d.args.ldo = L; d.args.accumulate = 1;
  RVAE_CHECK(gemm_launch(&ctx->c, d, S_(stream)));
  return launch_latent_bwd(&ctx->c, dz_scratch, eps, logvar, mu, g_mu_ext, g_logvar_ext, kl_grad_value(kl_grad_scale), M, L,
                           BF(dml_hi), BF(dml_lo), bias_grad, 0, nullptr, S_(stream));
}

int rvae_wgrad(rvae_ctx* ctx, const void* dy_hi, const void* dy_lo, const void* x_hi, const void* x_lo, int B, int M,
               int N, float* dW, int accumulate, int k_splits, void* stream) {
  CTX_OR_FAIL(ctx);
  RVAE_REQUIRE(dW, RVAE_ERR_INVALID, "wgrad: null output");
  RVAE_REQUIRE(M % 64 == 0, RVAE_ERR_UNSUPPORTED, "wgrad: M=%d must be a multiple of 64", M);
  GemmDesc d = desc_base(EPI_REDUCE, M, N, B);
  d.A = op(dy_hi, dy_lo, MAJOR_MN, M);
  d.B = op(x_hi, x_lo, MAJOR_MN, N);
  d.args.out_f32 = dW; d.args.ldo = N; d.args.accumulate = accumulate;
  d.k_splits = accumulate ? k_splits : 1;
  return gemm_launch(&ctx->c, d, S_(stream));
}

// ---------------------------------------------------------------------------------------------------------
// parameter layout
// ---------------------------------------------------------------------------------------------------------
int rvae_param_layout(int S, int H, int L, rvae_layout* out) {
  RVAE_REQUIRE(out, RVAE_ERR_INVALID, "param_layout: null out");
  RVAE_REQUIRE(S > 0 && H > 0 && L > 0 && S % 64 == 0 && H % 64 == 0 && L % 64 == 0, RVAE_ERR_UNSUPPORTED,
               "segment_length=%d, n_units=%d, latent_dim=%d must be positive multiples of 64", S, H, L);
  int64_t o = 0;
  out->w1 = o; o += (int64_t)H * S;
  out->w2 = o; o += (int64_t)2 * L * H;
  out->w3 = o; o += (int64_t)H * L;
  out->w4 = o; o += (int64_t)S * H;
  out->b1 = o; o += H;
  out->b2 = o; o += 2 * L;
  out->b3 = o; o += H;
  out->b4 = o; o += S;
  out->total = o;
  return RVAE_OK;
}

int rvae_param_layout_padded(int S, int H, int L, rvae_layout* out, int* Sp, int* Hp, int* Lp) {
  RVAE_REQUIRE(out && Sp && Hp && Lp, RVAE_ERR_INVALID, "param_layout_padded: null out");
  RVAE_REQUIRE(S > 0 && H > 0 && L > 0 && S <= (1 << 24) && H <= (1 << 24) && L <= (1 << 24), RVAE_ERR_UNSUPPORTED,
               "segment_length=%d, n_units=%d, latent_dim=%d must be in 1..%d", S, H, L, 1 << 24);
  const int sp = (S + 63) / 64 * 64, hp = (H + 63) / 64 * 64, lp = (L + 63) / 64 * 64;
  RVAE_CHECK(rvae_param_layout(sp, hp, lp, out));
  *Sp = sp; *Hp = hp; *Lp = lp;
  return RVAE_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------
// plan
// ---------------------------------------------------------------------------------------------------------
namespace {

struct Planes {
  __nv_bfloat16* hi = nullptr;
  __nv_bfloat16* lo = nullptr;
};

// gradient-norm launches: W4 | W3 | W2 + biases | W1, in the order the backward stages complete them
constexpr int kNormGroups = 4;
constexpr int kNormMaxBlocks = 1024;

enum GemmId { G_F1, G_F2, G_F3, G_F4_OUT, G_F4_LIN, G_B4W, G_B4D, G_B3W, G_B3D, G_B2W, G_B2D, G_B1W, G_COUNT };
// timing slots of the non-GEMM kernels follow the GEMM slots
enum AuxSlot { T_LOAD = G_COUNT, T_EPS, T_FINALIZE, T_COLSUM, T_ADAM, T_TANHBWD, T_LATENT, T_COUNT };

// internal slot past the public ones: the latent dgrad with the reparameterisation / KL backward fused into its
// epilogue (timed and reported as G_B3D)
constexpr int G_B3D_LAT = G_COUNT;
constexpr int kGemmSlots = G_COUNT + 1;

struct GemmSet {
  PreparedGemm g[kGemmSlots];
  bool ready[kGemmSlots];
  PreparedChain dual[3];  // backward stage s: dgrad + weight gradient in one launch
  int dual_state[3];      // 0 = not tried, 1 = ready, -1 = unsupported for these shapes (separate launches)
  PreparedChain dual_lat; // stage 1 with the fused latent epilogue (G_B3D_LAT + G_B3W)
  int dual_lat_state;
  PreparedChain tri;      // stage 2 with stage 1's weight gradient riding along: B2d + B2w + B3w in one launch
  int tri_state;
  PreparedChain fwd;      // forward: fc1 -> encoder head -> fc3 -> fc4/loss chained by tile-level dependencies
  int fwd_state;
};

}  // namespace

struct rvae_plan {
  rvae_ctx* ctx;
  // S, H, L: the dims the plan computes at - the model's dims rounded up to multiples of 64 (rvae_param_layout_padded):
  // workspace, GEMM shapes, tensor maps, parameter blocks. The padding holds exact zeros through every step.
  // s_true, h_true, l_true: the model's dims - loss normalisation and the shapes of every caller tensor.
  int S, H, L, max_batch, precision;
  int s_true, h_true, l_true;
  rvae_layout lay;
  rvae_plan_buffers bufs;
  bool bound;
  size_t ws_bytes;
  // workspace sections
  Planes x, h1, z, h3, da4, da3, dml, da1;
  float *mu, *lv, *eps, *dz, *xhat;
  // padded plans only: the external upstream gradients of rvae_plan_backward_external at the padded row pitch
  float *ext_gx, *ext_gmu, *ext_glv, *ext_lv;
  // second input set (frames + noise) the background stream fills for the NEXT step while this one runs
  Planes x_alt;
  float* eps_alt;
  int cur;                 // which input set is current (GEMM tensor maps are prepared per set)
  // Frames read IN PLACE (rvae_plan_load_span / rvae_plan_prefetch_span): the x planes hold the batch's contiguous
  // sample span [(count - 1) * hop + S samples] instead of count materialised rows, and fc1's A operand, the MSE
  // side input and the fc1 weight gradient's B operand read frame i at row pitch hop through overlapping-row tensor
  // maps. 0 = the planes hold dense [count, S] rows (gather / tensor input).
  int x_pitch, x_pitch_alt;
  int* sched_dev;          // schedules of the fused launches: [2 input sets][6 launches][128 pairs][kSchedMax]
  int sched_batch;         // the batch size those schedules were built for (0 = none yet): the buffer holds ONE set of
                           // schedules, so other batch sizes of this plan (a ragged last batch) run separate launches
  unsigned int* dep_flags; // row-block counters of the chained forward launch: [3 layer transitions][256]
  bool fuse_forward;       // env RVAE_FUSE_FORWARD=1: forward pass as one chained launch (default off)
  bool fuse_latent;        // env RVAE_FUSE_LATENT: backward of reparameterize + KL inside the latent dgrad's epilogue
  int dual_pairs;          // CTA pairs a fused launch uses (0 = fused launches off)
  unsigned int* ticket;    // last-block ticket of the step's final Adam launch (advances the step counter); ticket[1]:
                           // the gradient-norm finalisation's
  bool ticket_zeroed;
  bool norm_ticket_zeroed;
  // gradient-norm clipping (rvae_plan_set_grad_clip): clip_max != nullptr makes every training step clip
  const double* clip_max;  // device max_norm
  float* clip_norm_out;    // pre-clip norm ring (may be nullptr)
  int clip_ring;
  double* norm_parts;      // workspace: fp64 partials of the norm launches, [kNormGroups][kNormMaxBlocks]
  float* clip_coef;        // workspace: the step's clipping factor, read by the Adam launch
  struct Prefetch {
    bool registered;       // rvae_plan_prefetch_frames called; consumed by the next rvae_plan_train_step
    int ready_batch;       // > 0: the alternate set holds this many frames (+ their noise), enqueued by a train step
    const void* audio; int audio_is_i16; int64_t n_samples; const int64_t* frame_idx; int64_t first_frame;
    int count, hop; uint64_t seed, offset; int add_step;
    bool span;             // frames are the run first_frame (or frame_idx[0]) .. + count: read in place (x_pitch)
    int64_t noise_row0;    // plan->noise_row0 at registration time (the shard of the NEXT global batch)
  } pf;
  double* loss_acc;
  // redirected outputs
  float *out_mu, *out_lv, *out_xhat;
  int batch;        // current batch
  int64_t global_batch;  // loss normalisation under data parallelism (0 = local batch)
  int64_t noise_row0;    // first row of this rank's shard in the global batch: Philox counters start at row0 * L, so
                         // the ranks draw disjoint pieces of the single-process noise tensor (0 = single process)
  bool dp_enabled;       // rvae_plan_enable_dp: this plan's train steps all-reduce their gradients
  float kl_c0;           // kl_beta / (B L) of the last fused-loss forward (KL gradient scale of the latent backward)
  double kl_bl;          // B L of that forward (global batch under data parallelism)
  const rvae_hparams* hp_dev;   // during rvae_plan_train_step_hp: the device record the kernels read kl_beta from
  int hp_early;                 // ... and the latent backward may read it before griddepcontrol.wait (two streams)
  bool dz_zeroed;        // the split-K latent dgrad accumulator holds zeros (left so by the latent backward kernel)
  bool grads_zeroed[5];  // gradient bucket s (0..3 weights, 4 biases) already holds zeros (left so by the fused Adam)
  // internal streams (created on first use): see rvae_plan_train_step
  bool streams_ready;
  cudaEvent_t ev_fork;
  bool two_streams;      // env RVAE_TWO_STREAMS=0: everything on the caller's stream (debugging / attribution)
  bool have_eps;
  // eps is generated on the side stream, concurrently with the batch load and fc1; F2 waits for ev_eps
  cudaEvent_t ev_eps;
  bool eps_pending;
  // per-bucket Adam launches of rvae_plan_train_step run on their own stream, under the remaining backward GEMMs
  cudaStream_t adam_stream;   // lowest priority: background work never takes an SM a pending GEMM CTA could use
  cudaEvent_t ev_adam_fork, ev_adam_join;
  // rvae_plan_train_step runs its critical chain on a highest-priority stream forked from the caller's stream
  cudaStream_t hp;
  cudaEvent_t ev_hp_fork, ev_hp_join;
  // backward stage 1 split over two streams: latent dgrad -> {latent backward kernel || fc3 weight gradient}. The
  // HBM-bound latent kernel and the weight-gradient GEMM (held to s1_wgrad_ctas CTAs) share the machine instead of
  // running one after the other (nothing can co-reside with a GEMM CTA: it owns the SM's shared memory)
  cudaStream_t hp2;
  cudaEvent_t ev_s1_fork, ev_s1_join;
  bool split_stage1;
  int s1_wgrad_ctas, s1_order;
  // The fc3 weight gradient (B3w) needs only da3 and z, so it does not have to run in stage 1: when all four stages of a
  // backward pass are issued together (rvae_plan_train_step, rvae_plan_backward(-1), the autograd backward), stage 1 is
  // just latent dgrad -> latent kernel on the whole machine, and B3w's MMA-heavy units ride in stage 2's fused launch,
  // whose dgrad tiles are epilogue-bound and leave the tensor pipe idle (B2d + B2w + B3w). Gradient bucket 1 (fc3) is
  // then complete after stage 2 instead of stage 1.
  bool merge_b3w;        // env RVAE_MERGE_B3W in RVAE_EXPERIMENTS builds; default off: measured, not a win (profiles/README.md)
  bool allow_defer;      // set by the callers that issue all stages of a pass
  bool b3w_deferred;     // stage 1 of the current pass left B3w to stage 2
  int adam_bg_blocks;    // grid cap of the single-process background Adam launch (0 = none)
  // data parallelism: gradient all-reduces run on their own stream, bucket by bucket as backward completes them
  cudaStream_t comm_stream;
  cudaStream_t comm_stream2;  // the step's last exchange: must not queue behind the previous one
  cudaEvent_t ev_comm_fork, ev_comm_done[5];
  // loss finalisation deferred into the latent backward kernel (rvae_plan_finish_loss_deferred)
  LossFinalize fin;
  bool fin_pending;
  std::map<int64_t, GemmSet> sets;  // prepared GEMMs per (batch size, input set, frame pitch)
  // optional per-GEMM timing
  bool timing;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev_pool;
  std::vector<std::pair<int, int>> ev_used;  // (gemm id, pool index)
  double t_ms[T_COUNT];
  int64_t t_n[T_COUNT];
  double t_flops[T_COUNT];
};

namespace {

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Walks the workspace layout; with base == nullptr only sizes are computed.
size_t carve(rvae_plan* p, uint8_t* base) {
  const size_t B = p->max_batch, S = p->S, H = p->H, L = p->L;
  const bool lo = p->precision == RVAE_PRECISION_FP32;
  size_t off = 0;
  auto take = [&](size_t bytes) -> uint8_t* {
    uint8_t* r = base ? base + off : nullptr;
    off += align_up(bytes, 256);
    return r;
  };
  auto planes = [&](Planes& pl, size_t elems) {
    pl.hi = reinterpret_cast<__nv_bfloat16*>(take(elems * 2));
    pl.lo = lo ? reinterpret_cast<__nv_bfloat16*>(take(elems * 2)) : nullptr;
  };
  planes(p->x, B * S);
  planes(p->x_alt, B * S);
  planes(p->h1, B * H);
  planes(p->z, B * L);
  planes(p->h3, B * H);
  planes(p->da4, B * S);
  planes(p->da3, B * H);
  planes(p->dml, B * 2 * L);
  planes(p->da1, B * H);
  p->mu = reinterpret_cast<float*>(take(B * L * 4));
  p->lv = reinterpret_cast<float*>(take(B * L * 4));
  p->eps = reinterpret_cast<float*>(take(B * L * 4));
  p->eps_alt = reinterpret_cast<float*>(take(B * L * 4));
  p->ticket = reinterpret_cast<unsigned int*>(take(256));
  p->sched_dev = reinterpret_cast<int*>(take(sizeof(int) * 2 * 6 * 128 * kSchedMax));
  p->dep_flags = reinterpret_cast<unsigned int*>(take(sizeof(unsigned int) * 3 * 256));
  p->norm_parts = reinterpret_cast<double*>(take(sizeof(double) * kNormGroups * kNormMaxBlocks));
  p->clip_coef = reinterpret_cast<float*>(take(sizeof(float)));
  p->dz = reinterpret_cast<float*>(take(B * L * 4));
  p->xhat = reinterpret_cast<float*>(take(B * S * 4));
  p->loss_acc = reinterpret_cast<double*>(take(2 * sizeof(double)));
  p->ext_gx = p->ext_gmu = p->ext_glv = p->ext_lv = nullptr;
  if (p->S != (size_t)p->s_true) p->ext_gx = reinterpret_cast<float*>(take(B * S * 4));
  if (p->L != (size_t)p->l_true) {
    p->ext_gmu = reinterpret_cast<float*>(take(B * L * 4));
    p->ext_glv = reinterpret_cast<float*>(take(B * L * 4));
    p->ext_lv = reinterpret_cast<float*>(take(B * L * 4));
  }
  return off;
}

Operand opnd(const Planes& pl, int major, int ld) {
  Operand o;
  o.hi = pl.hi; o.lo = pl.lo; o.major = major; o.ld = ld; o.cols = 0;
  return o;
}
Operand wopnd(const rvae_plan* p, int64_t off, int major, int ld) {
  Operand o;
  o.hi = BF(p->bufs.shadow_hi) + off;
  o.lo = p->bufs.shadow_lo ? BF(p->bufs.shadow_lo) + off : nullptr;
  o.major = major; o.ld = ld; o.cols = 0;
  return o;
}

int prepare(rvae_plan* p, GemmSet& gs, int id) {
  if (gs.ready[id]) return RVAE_OK;
  const int B = p->batch, S = p->S, H = p->H, L = p->L;
  const int ldx = p->x_pitch > 0 ? p->x_pitch : S;   // row pitch of the frames in the x planes
  const rvae_layout& ly = p->lay;
  float* params = p->bufs.params;
  float* grads = p->bufs.grads;
  GemmDesc d;
  memset(&d, 0, sizeof(d));
  const bool bf16_mode = p->precision == RVAE_PRECISION_BF16;
  switch (id) {
    case G_F1:
      d.epi = EPI_LINEAR; d.M = B; d.N = H; d.K = S;
      d.A = opnd(p->x, MAJOR_K, ldx); d.B = wopnd(p, ly.w1, MAJOR_K, S);
      d.A.cols = p->s_true;   // frames read in place: the columns past segment_length are padding (zeros)
      d.args.bias = params + ly.b1; d.args.act = ACT_RELU; d.args.ldo = H;
      d.args.out_hi = p->h1.hi; d.args.out_lo = p->h1.lo;
      break;
    case G_F2:
      d.epi = EPI_HEAD; d.M = B; d.N = 2 * L; d.K = H; d.head_L = L;
      d.A = opnd(p->h1, MAJOR_K, H); d.B = wopnd(p, ly.w2, MAJOR_K, H);
      d.args.bias = params + ly.b2; d.args.in0 = p->eps; d.args.out_f32 = p->mu; d.args.out_f32_b = p->lv;
      d.args.out_hi = p->z.hi; d.args.out_lo = p->z.lo;
      d.args.loss_acc = p->loss_acc + 1; d.args.L = L; d.args.ldo = L;
      break;
    case G_F3:
      d.epi = EPI_LINEAR; d.M = B; d.N = H; d.K = L;
      d.A = opnd(p->z, MAJOR_K, L); d.B = wopnd(p, ly.w3, MAJOR_K, L);
      d.args.bias = params + ly.b3; d.args.act = ACT_RELU; d.args.ldo = H;
      d.args.out_hi = p->h3.hi; d.args.out_lo = p->h3.lo;
      break;
    case G_F4_OUT:
      d.epi = EPI_OUT; d.M = B; d.N = S; d.K = H;
      d.A = opnd(p->h3, MAJOR_K, H); d.B = wopnd(p, ly.w4, MAJOR_K, H);
      d.args.bias = params + ly.b4; d.args.in0 = p->x.hi; d.args.in1 = p->x.lo; d.args.out_f32 = p->xhat;
      d.args.out_hi = p->da4.hi; d.args.out_lo = p->da4.lo;
      d.args.act = bf16_mode ? ACT_TANH_APPROX : ACT_TANH;
      d.args.loss_acc = p->loss_acc; d.args.ldo = S; d.args.ldi = ldx; d.side_cols = p->s_true;
      d.args.colsum = grads ? grads + ly.b4 : nullptr;   // db4 = column sums of da4
      break;
    case G_F4_LIN:
      d.epi = EPI_LINEAR; d.M = B; d.N = S; d.K = H;
      d.A = opnd(p->h3, MAJOR_K, H); d.B = wopnd(p, ly.w4, MAJOR_K, H);
      d.args.bias = params + ly.b4; d.args.act = bf16_mode ? ACT_TANH_APPROX : ACT_TANH; d.args.ldo = S;
      d.args.out_f32 = p->xhat;
      break;
    case G_B4W:
      d.epi = EPI_REDUCE; d.M = S; d.N = H; d.K = B;
      d.A = opnd(p->da4, MAJOR_MN, S); d.B = opnd(p->h3, MAJOR_MN, H);
      d.args.out_f32 = grads + ly.w4; d.args.ldo = H; d.args.accumulate = 1;
      break;
    case G_B4D:
      d.epi = EPI_DRELU; d.M = B; d.N = H; d.K = S;
      d.A = opnd(p->da4, MAJOR_K, S); d.B = wopnd(p, ly.w4, MAJOR_MN, H);
      d.args.in0 = p->h3.hi; d.args.out_hi = p->da3.hi; d.args.out_lo = p->da3.lo; d.args.ldo = H;
      d.args.colsum = grads + ly.b3;                     // db3 = column sums of da3
      break;
    case G_B3W:
      d.epi = EPI_REDUCE; d.M = H; d.N = L; d.K = B;
      d.A = opnd(p->da3, MAJOR_MN, H); d.B = opnd(p->z, MAJOR_MN, L);
      d.args.out_f32 = grads + ly.w3; d.args.ldo = L; d.args.accumulate = 1;
      break;
    case G_B3D:
      // dz = da3 W3 as a split-K reduce-add GEMM into fp32; the latent backward kernel turns dz into d_ml and db2
      d.epi = EPI_REDUCE; d.M = B; d.N = L; d.K = H;
      d.A = opnd(p->da3, MAJOR_K, H); d.B = wopnd(p, ly.w3, MAJOR_MN, L);
      d.args.out_f32 = p->dz; d.args.ldo = L; d.args.accumulate = 1;
      break;
    case G_B3D_LAT:
      // d_ml = [dz + c mu | dz eps sigma / 2 + c (sigma^2 - 1) / 2] and db2 straight from the accumulator (bf16 mode):
      // no split-K, no dz round trip, no separate latent backward kernel
      d.epi = EPI_DLATENT; d.M = B; d.N = L; d.K = H;
      d.A = opnd(p->da3, MAJOR_K, H); d.B = wopnd(p, ly.w3, MAJOR_MN, L);
      d.args.in0 = p->eps; d.args.in1 = p->lv; d.args.in2 = p->mu;
      d.args.out_hi = p->dml.hi; d.args.ldo = 2 * L; d.args.L = L;
      d.args.colsum = grads + ly.b2;                     // [db21; db22] = column sums of d_ml
      break;
    case G_B2W:
      d.epi = EPI_REDUCE; d.M = 2 * L; d.N = H; d.K = B;
      d.A = opnd(p->dml, MAJOR_MN, 2 * L); d.B = opnd(p->h1, MAJOR_MN, H);
      d.args.out_f32 = grads + ly.w2; d.args.ldo = H; d.args.accumulate = 1;
      break;
    case G_B2D:
      d.epi = EPI_DRELU; d.M = B; d.N = H; d.K = 2 * L;
      d.A = opnd(p->dml, MAJOR_K, 2 * L); d.B = wopnd(p, ly.w2, MAJOR_MN, H);
      d.args.in0 = p->h1.hi; d.args.out_hi = p->da1.hi; d.args.out_lo = p->da1.lo; d.args.ldo = H;
      d.args.colsum = grads + ly.b1;                     // db1 = column sums of da1
      break;
    case G_B1W:
      d.epi = EPI_REDUCE; d.M = H; d.N = S; d.K = B;
      d.A = opnd(p->da1, MAJOR_MN, H); d.B = opnd(p->x, MAJOR_MN, ldx); d.B.cols = p->s_true;
      d.args.out_f32 = grads + ly.w1; d.args.ldo = S; d.args.accumulate = 1;
      break;
    default:
      return set_error(RVAE_ERR_INVALID, "plan: bad gemm id %d", id);
  }
  RVAE_CHECK(gemm_prepare(&p->ctx->c, d, &gs.g[id]));
  gs.ready[id] = true;
  return RVAE_OK;
}

int get_set(rvae_plan* p, GemmSet** out) {
  // tensor maps bake in the addresses of the current input set and the row pitch of its frames
  const int64_t key = ((int64_t)p->batch * 2 + p->cur) * 65536 + p->x_pitch;
  auto it = p->sets.find(key);
  if (it == p->sets.end()) {
    GemmSet gs;
    memset(&gs, 0, sizeof(gs));
    it = p->sets.emplace(key, gs).first;
  }
  *out = &it->second;
  return RVAE_OK;
}

int run_untimed(rvae_plan* p, GemmSet* gs, int id, cudaStream_t st, const EpiArgs* override_args) {
  if (override_args) {
    PreparedGemm g = gs->g[id];
    EpiArgs a = *override_args;
    if (a.L == 0) a.L = g.params.epi.L;
    RVAE_CHECK(gemm_bind_outputs(&g, a, false));  // re-encodes the TMA store maps of redirected outputs
    return gemm_run(&p->ctx->c, g, st);
  }
  return gemm_run(&p->ctx->c, gs->g[id], st);
}

// Bracket a non-GEMM launch with timing events when timing is enabled.
struct TimedScope {
  rvae_plan* p; int slot; cudaStream_t st; int idx;
  TimedScope(rvae_plan* p_, int slot_, cudaStream_t st_) : p(p_), slot(slot_), st(st_), idx(-1) {
    if (!p->timing) return;
    const size_t k = p->ev_used.size();
    if (k >= p->ev_pool.size()) {
      cudaEvent_t a, b;
      if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) return;
      p->ev_pool.emplace_back(a, b);
    }
    idx = (int)k;
    cudaEventRecord(p->ev_pool[k].first, st);
  }
  ~TimedScope() {
    if (idx < 0) return;
    cudaEventRecord(p->ev_pool[idx].second, st);
    p->ev_used.emplace_back(slot, idx);
  }
};

int run(rvae_plan* p, int id, cudaStream_t st, const EpiArgs* override_args = nullptr) {
  GemmSet* gs;
  RVAE_CHECK(get_set(p, &gs));
  RVAE_CHECK(prepare(p, *gs, id));
  if (!p->timing) return run_untimed(p, gs, id, st, override_args);
  const size_t slot = p->ev_used.size();
  if (slot >= p->ev_pool.size()) {
    cudaEvent_t a, b;
    RVAE_CUDA(cudaEventCreate(&a));
    RVAE_CUDA(cudaEventCreate(&b));
    p->ev_pool.emplace_back(a, b);
  }
  RVAE_CUDA(cudaEventRecord(p->ev_pool[slot].first, st));
  RVAE_CHECK(run_untimed(p, gs, id, st, override_args));
  RVAE_CUDA(cudaEventRecord(p->ev_pool[slot].second, st));
  const int tid = id == G_B3D_LAT ? G_B3D : id;
  p->ev_used.emplace_back(tid, (int)slot);
  const GemmParams& gp = gs->g[id].params;
  p->t_flops[tid] = 2.0 * gp.M * gp.N * gp.K;
  return RVAE_OK;
}

// Caller tensors of a padded plan cross the API at their true width `cols`; the plan's buffers have row pitch `ld`.
// dst [rows, ld] <- src [rows, cols] with zeros in columns cols..ld
int pad_rows(float* dst, const float* src, int rows, int cols, int ld, cudaStream_t st) {
  RVAE_CUDA(cudaMemcpy2DAsync(dst, sizeof(float) * ld, src, sizeof(float) * cols, sizeof(float) * cols, rows,
                              cudaMemcpyDeviceToDevice, st));
  RVAE_CUDA(cudaMemset2DAsync(dst + cols, sizeof(float) * ld, 0, sizeof(float) * (ld - cols), rows, st));
  return RVAE_OK;
}
// dst [rows, cols] <- the first cols columns of src [rows, ld]
int strip_rows(float* dst, const float* src, int rows, int cols, int ld, cudaStream_t st) {
  RVAE_CUDA(cudaMemcpy2DAsync(dst, sizeof(float) * cols, src, sizeof(float) * ld, sizeof(float) * cols, rows,
                              cudaMemcpyDeviceToDevice, st));
  return RVAE_OK;
}
// redirected mu / logvar of a plan with a padded latent_dim: copied out of the workspace
int copy_latents_out(rvae_plan* p, cudaStream_t st) {
  if (p->out_mu) RVAE_CHECK(strip_rows(p->out_mu, p->mu, p->batch, p->l_true, p->L, st));
  if (p->out_lv) RVAE_CHECK(strip_rows(p->out_lv, p->lv, p->batch, p->l_true, p->L, st));
  return RVAE_OK;
}

// Philox noise for `rows` rows of the batch starting at global row `row0`: element (r, c) is element
// (row0 + r) * L + c of the unpadded [global batch, L] draw, whatever the padding of the plan's eps buffer
int draw_eps(rvae_plan* p, float* out, int rows, uint64_t seed, uint64_t offset, const float* offset_src, int64_t row0,
             cudaStream_t st) {
  if (p->l_true == p->L)
    return launch_randn(&p->ctx->c, out, (int64_t)rows * p->L, seed, offset, offset_src, row0 * p->L, st);
  return launch_randn_rows(&p->ctx->c, out, rows, p->l_true, p->L, seed, offset, offset_src, row0 * p->l_true, st);
}

// decoder of rvae_plan_decode / rvae_plan_decode_lerp once z is in fc3's operand: fc3, fc4 + tanh -> xhat_out
int decode_tail(rvae_plan* p, float* xhat_out, cudaStream_t st) {
  RVAE_CHECK(run(p, G_F3, st));
  GemmSet* gs;
  RVAE_CHECK(get_set(p, &gs));
  RVAE_CHECK(prepare(p, *gs, G_F4_LIN));
  EpiArgs a = gs->g[G_F4_LIN].params.epi;
  const bool rec_direct = p->S == p->s_true;
  a.out_f32 = rec_direct ? xhat_out : p->xhat;
  RVAE_CHECK(run(p, G_F4_LIN, st, &a));
  return rec_direct ? RVAE_OK : strip_rows(xhat_out, p->xhat, p->batch, p->s_true, p->S, st);
}

int check_ready(const rvae_plan* p, bool need_batch) {
  RVAE_REQUIRE(p != nullptr, RVAE_ERR_INVALID, "null rvae_plan");
  RVAE_REQUIRE(p->bound, RVAE_ERR_STATE, "plan: rvae_plan_bind has not been called");
  if (need_batch) RVAE_REQUIRE(p->batch > 0, RVAE_ERR_STATE, "plan: no batch loaded");
  return RVAE_OK;
}

// Bias gradients accumulate (atomicAdd) into the bias block from the epilogues that produce the pre-activation
// gradients; make sure the block starts from zero.
int ensure_bias_zeroed(rvae_plan* p, cudaStream_t st) {
  if (p->grads_zeroed[4]) return RVAE_OK;
  const rvae_layout& ly = p->lay;
  RVAE_CUDA(cudaMemsetAsync(p->bufs.grads + ly.b1, 0, sizeof(float) * (size_t)(ly.total - ly.b1), st));
  p->grads_zeroed[4] = true;
  return RVAE_OK;
}

int ensure_side_stream(rvae_plan* p) {
  if (p->streams_ready) return RVAE_OK;
  int least = 0, greatest = 0;
  RVAE_CUDA(cudaDeviceGetStreamPriorityRange(&least, &greatest));
  RVAE_CUDA(cudaStreamCreateWithPriority(&p->hp, cudaStreamNonBlocking, greatest));
  RVAE_CUDA(cudaStreamCreateWithPriority(&p->adam_stream, cudaStreamNonBlocking, least));
  RVAE_CUDA(cudaStreamCreateWithPriority(&p->hp2, cudaStreamNonBlocking, greatest));
  RVAE_CUDA(cudaEventCreateWithFlags(&p->ev_s1_fork, cudaEventDisableTiming));
  RVAE_CUDA(cudaEventCreateWithFlags(&p->ev_s1_join, cudaEventDisableTiming));
  RVAE_CUDA(cudaEventCreateWithFlags(&p->ev_hp_fork, cudaEventDisableTiming));
  RVAE_CUDA(cudaEventCreateWithFlags(&p->ev_hp_join, cudaEventDisableTiming));
  RVAE_CUDA(cudaStreamCreateWithPriority(&p->comm_stream, cudaStreamNonBlocking, greatest));
  RVAE_CUDA(cudaStreamCreateWithPriority(&p->comm_stream2, cudaStreamNonBlocking, greatest));
  RVAE_CUDA(cudaEventCreateWithFlags(&p->ev_comm_fork, cudaEventDisableTiming));
  for (int i = 0; i < 5; ++i) RVAE_CUDA(cudaEventCreateWithFlags(&p->ev_comm_done[i], cudaEventDisableTiming));
  RVAE_CUDA(cudaEventCreateWithFlags(&p->ev_fork, cudaEventDisableTiming));
  RVAE_CUDA(cudaEventCreateWithFlags(&p->ev_eps, cudaEventDisableTiming));
  RVAE_CUDA(cudaEventCreateWithFlags(&p->ev_adam_fork, cudaEventDisableTiming));
  RVAE_CUDA(cudaEventCreateWithFlags(&p->ev_adam_join, cudaEventDisableTiming));
  p->streams_ready = true;
  return RVAE_OK;
}

// Adam over the gradient buckets selected by `mask` (bit s = bucket s of rvae_plan_bucket): the selected buckets are
// merged into contiguous segments of the flat buffer and updated with one launch per pair of segments.
int adam_buckets(rvae_plan* p, unsigned mask, const HpArg& hp, float grad_scale, int zero_grads, int step_bias,
                 bool advance_step, cudaStream_t st, const float* coef = nullptr) {
  const rvae_layout& ly = p->lay;
  const rvae_plan_buffers& b = p->bufs;
  // flat order: W1 (bucket 3) | W2 (2) | W3 (1) | W4 (0) | biases (4)
  const int order[5] = {3, 2, 1, 0, 4};
  const int64_t begin[6] = {ly.w1, ly.w2, ly.w3, ly.w4, ly.b1, ly.total};
  int64_t seg_off[5], seg_n[5];
  int nseg = 0;
  for (int i = 0; i < 5; ++i) {
    if (!(mask & (1u << order[i]))) continue;
    if (nseg > 0 && seg_off[nseg - 1] + seg_n[nseg - 1] == begin[i]) seg_n[nseg - 1] += begin[i + 1] - begin[i];
    else { seg_off[nseg] = begin[i]; seg_n[nseg] = begin[i + 1] - begin[i]; ++nseg; }
  }
  if (advance_step && !p->ticket_zeroed) {
    RVAE_CUDA(cudaMemsetAsync(p->ticket, 0, sizeof(unsigned int), st));
    p->ticket_zeroed = true;
  }
  for (int i = 0; i < nseg; i += 2) {
    const int64_t o = seg_off[i];
    const bool pair = i + 1 < nseg;
    const bool last = i + 2 >= nseg;
    RVAE_CHECK(launch_adam2(&p->ctx->c, b.params + o, b.grads + o, b.exp_avg + o, b.exp_avg_sq + o, seg_n[i],
                            pair ? seg_off[i + 1] - o : 0, pair ? seg_n[i + 1] : 0, hp, grad_scale, coef, b.step, step_bias, (advance_step && last) ? p->ticket : nullptr,
                            BF(b.shadow_hi) + o, b.shadow_lo ? BF(b.shadow_lo) + o : nullptr, zero_grads, st));
  }
  for (int s = 0; s < 5; ++s)
    if (mask & (1u << s)) p->grads_zeroed[s] = zero_grads != 0;
  return RVAE_OK;
}

// Sum of squares of norm group k (0: W4, 1: W3, 2: W2 + biases, 3: W1) into its partial slots. The partition and the
// grids are fixed, so the norm of a gradient buffer has the same bits on every path (two streams, one stream, data
// parallel, rvae_plan_grad_norm). fin != nullptr: this is the last launch of the reduction; it finalises into *fin.
int grad_norm_group(rvae_plan* p, int k, NormFinalize* fin, cudaStream_t st) {
  const rvae_layout& ly = p->lay;
  const int64_t off[kNormGroups][2] = {{ly.w4, 0}, {ly.w3, 0}, {ly.w2, ly.b1}, {ly.w1, 0}};
  const int64_t len[kNormGroups][2] = {{ly.b1 - ly.w4, 0}, {ly.w4 - ly.w3, 0}, {ly.w3 - ly.w2, ly.total - ly.b1},
                                       {ly.w2 - ly.w1, 0}};
  // the groups' partials are packed in group order: group k starts after the blocks of groups 0..k-1
  int base[kNormGroups + 1] = {0};
  for (int j = 0; j < kNormGroups; ++j) base[j + 1] = base[j] + grad_norm_blocks(&p->ctx->c, len[j][0] + len[j][1]);
  RVAE_REQUIRE(base[kNormGroups] <= kNormGroups * kNormMaxBlocks, RVAE_ERR_UNSUPPORTED, "grad_norm: %d blocks",
               base[kNormGroups]);
  if (fin != nullptr) {
    if (!p->norm_ticket_zeroed) {
      RVAE_CUDA(cudaMemsetAsync(p->ticket + 1, 0, sizeof(unsigned int), st));
      p->norm_ticket_zeroed = true;
    }
    fin->parts = p->norm_parts;
    fin->n_parts = base[kNormGroups];
    fin->ticket = p->ticket + 1;
  }
  NormFinalize none;
  memset(&none, 0, sizeof(none));
  return launch_grad_norm(&p->ctx->c, p->bufs.grads + off[k][0], len[k][0], off[k][1] - off[k][0], len[k][1],
                          p->norm_parts + base[k], fin ? *fin : none, st);
}

// The finalisation of a clipping training step: the pre-clip norm into the ring slot of the step, the factor into
// the workspace slot the Adam launch reads
NormFinalize clip_finalize(rvae_plan* p) {
  NormFinalize f;
  memset(&f, 0, sizeof(f));
  f.step = p->bufs.step;
  f.norm_out = p->clip_norm_out;
  f.ring_size = p->clip_ring;
  f.max_norm = p->clip_max;
  f.coef_out = p->clip_coef;
  return f;
}

// Backward stage s, in one stream: the dgrad GEMM that produces the next layer's pre-activation gradient (and, in its
// epilogue, that layer's bias gradient) first - it is the critical dependency chain - then the weight gradient of
// layer (4 - s). After stage s gradient bucket s is complete on `st`.
//   s=0: da3 = (da4 W4) * [h3>0], db3                                   ; dW4 = da4^T h3
//   s=1: dz = da3 W3 (split-K, fp32) -> latent backward kernel: d_ml, db2 ; dW3 = da3^T z
//   s=2: da1 = (d_ml W2) * [h1>0], db1                                  ; dW2 = d_ml^T h1
//   s=3:                                                                  dW1 = da1^T x
// The GEMMs are persistent on the fewest SMs that keep their wave count (gemm_prepare); running the two GEMMs of a
// stage concurrently only makes them share those SMs, so they are not forked - the SMs left over belong to the
// background stream (noise, Adam per bucket, all-reduce).
// External upstream gradients of (mu, logvar) for the autograd path, with the logvar tensor of that forward.
struct LatentExt {
  const float* g_mu;
  const float* g_lv;
  const float* lv;
};

// KL gradient scale of the latent backward: the host's kl_c0, or beta(k) / (B L) from the record of a scheduled step
KlGrad plan_kl(const rvae_plan* p) { return KlGrad{p->hp_dev, p->bufs.step, p->kl_bl, p->kl_c0, p->hp_early}; }

// Fused launches read their tile schedule from the plan's one schedule buffer: usable by the batch size that owns it.
bool sched_usable(const rvae_plan* p) { return p->sched_batch == 0 || p->sched_batch == p->batch; }

// Stage 1 runs the reparameterisation / KL backward inside the latent dgrad's epilogue (bf16 mode, fused loss)
bool latent_fused(const rvae_plan* p) {
  return p->fuse_latent && p->precision == RVAE_PRECISION_BF16 && p->batch > kBlockM;
}

// Stage 1 with G_B3D_LAT: [d_ml, db2 = latent dgrad + fused epilogue | dW3] as one fused launch (or two GEMMs when
// fused launches are off / timed). The weight-gradient bucket has been cleared by the caller.
int backward_stage_latent_fused(rvae_plan* p, cudaStream_t st) {
  GemmSet* gs;
  RVAE_CHECK(get_set(p, &gs));
  if (p->fin_pending) {
    // no latent backward kernel to carry the deferred loss finalisation (rvae_plan_train_step moves it to the
    // background stream before it gets here)
    RVAE_CHECK(launch_loss_finalize_prepared(&p->ctx->c, p->fin, st));
    p->fin_pending = false;
  }
  if (p->dual_pairs > 0 && !p->timing && sched_usable(p)) {
    int pairs = p->dual_pairs > 64 ? 64 : p->dual_pairs;
    if (const char* e = getenv("RVAE_DUAL_PAIRS_S1")) {
      const int v = atoi(e);
      if (v >= 1 && 2 * v <= p->ctx->c.num_sms_total) pairs = v;
    }
    if (gs->dual_lat_state == 0) {
      RVAE_CHECK(prepare(p, *gs, G_B3D_LAT));
      RVAE_CHECK(prepare(p, *gs, G_B3W));
      int* sched = p->sched_dev + ((size_t)p->cur * 6 + 4) * 128 * kSchedMax;
      const PreparedGemm* both[2] = {&gs->g[G_B3D_LAT], &gs->g[G_B3W]};
      const int rc = gemm_prepare_chain(&p->ctx->c, both, 2, pairs, sched, &gs->dual_lat);
      gs->dual_lat_state = rc == RVAE_OK ? 1 : -1;
      if (rc != RVAE_OK && rc != RVAE_ERR_UNSUPPORTED) return rc;
      if (rc == RVAE_OK) p->sched_batch = p->batch;
    }
    if (gs->dual_lat_state == 1) {
      PreparedChain d = gs->dual_lat;
      d.params.p[0].epi.c0 = p->kl_c0;
      return gemm_run_chain(&p->ctx->c, d, st);
    }
  }
  RVAE_CHECK(prepare(p, *gs, G_B3D_LAT));
  EpiArgs a = gs->g[G_B3D_LAT].params.epi;
  a.c0 = p->kl_c0;
  RVAE_CHECK(run(p, G_B3D_LAT, st, &a));
  return run(p, G_B3W, st);
}

int backward_stage(rvae_plan* p, int stage, const LatentExt* ext, cudaStream_t st) {
  const int S = p->S, H = p->H, L = p->L;
  const rvae_layout& ly = p->lay;
  float* grads = p->bufs.grads;
  static const int kWgrad[4] = {G_B4W, G_B3W, G_B2W, G_B1W};
  static const int kDgrad[4] = {G_B4D, G_B3D, G_B2D, -1};
  RVAE_REQUIRE(stage >= 0 && stage < 4, RVAE_ERR_INVALID, "plan_backward: stage %d not in -1..3", stage);
  float* wptr[4] = {grads + ly.w4, grads + ly.w3, grads + ly.w2, grads + ly.w1};
  const size_t wcount[4] = {(size_t)S * H, (size_t)H * L, (size_t)2 * L * H, (size_t)H * S};
  if (!p->grads_zeroed[stage]) RVAE_CUDA(cudaMemsetAsync(wptr[stage], 0, sizeof(float) * wcount[stage], st));
  p->grads_zeroed[stage] = false;
  // stage 1, bf16 mode, fused loss: the reparameterisation / KL backward runs inside the latent dgrad's epilogue
  if (stage == 1 && ext == nullptr && latent_fused(p)) return backward_stage_latent_fused(p, st);
  if (stage == 1 && !p->dz_zeroed)
    RVAE_CUDA(cudaMemsetAsync(p->dz, 0, sizeof(float) * (size_t)p->max_batch * L, st));
  auto stage_pairs = [&](int st_idx) {
    // under data parallelism the fused launches leave the same spare SMs as the single GEMMs do: the exchange kernels
    // run there
    int pairs = (p->dp_enabled && p->ctx->dp_world > 1 && p->dual_pairs > 64) ? 64 : p->dual_pairs;
    const char* names[3] = {"RVAE_DUAL_PAIRS_S0", "RVAE_DUAL_PAIRS_S1", "RVAE_DUAL_PAIRS_S2"};
    if (const char* e = getenv(names[st_idx])) {   // experiments
      const int v = atoi(e);
      if (v >= 1 && 2 * v <= p->ctx->c.num_sms_total) pairs = v;
    }
    return pairs;
  };
  if (stage == 1 && p->allow_defer && p->merge_b3w && p->dual_pairs > 0 && sched_usable(p) && p->batch > kBlockM) {
    // leave B3w to stage 2 - if the three-problem launch exists for these shapes
    GemmSet* gs;
    RVAE_CHECK(get_set(p, &gs));
    if (gs->tri_state == 0) {
      RVAE_CHECK(prepare(p, *gs, G_B2D));
      RVAE_CHECK(prepare(p, *gs, G_B2W));
      RVAE_CHECK(prepare(p, *gs, G_B3W));
      int* sched = p->sched_dev + ((size_t)p->cur * 6 + 5) * 128 * kSchedMax;
      const PreparedGemm* three[3] = {&gs->g[G_B2D], &gs->g[G_B2W], &gs->g[G_B3W]};
      const int rc = gemm_prepare_chain(&p->ctx->c, three, 3, stage_pairs(2), sched, &gs->tri);
      gs->tri_state = rc == RVAE_OK ? 1 : -1;
      if (rc != RVAE_OK && rc != RVAE_ERR_UNSUPPORTED) return rc;
      if (rc == RVAE_OK) p->sched_batch = p->batch;
    }
    if (gs->tri_state == 1) {
      RVAE_CHECK(run(p, G_B3D, st));
      {
        TimedScope ts(p, T_LATENT, st);
        RVAE_CHECK(launch_latent_bwd(&p->ctx->c, p->dz, p->eps, ext ? ext->lv : p->lv, p->mu, ext ? ext->g_mu : nullptr,
                                     ext ? ext->g_lv : nullptr, plan_kl(p), p->batch, L, p->dml.hi, p->dml.lo, grads + ly.b2,
                                     1, p->fin_pending ? &p->fin : nullptr, st));
      }
      p->fin_pending = false;
      p->dz_zeroed = true;
      p->b3w_deferred = true;
      return RVAE_OK;
    }
  }
  if (stage == 2 && p->b3w_deferred) {
    GemmSet* gs;
    RVAE_CHECK(get_set(p, &gs));
    RVAE_REQUIRE(gs->tri_state == 1, RVAE_ERR_STATE, "plan_backward: stage 1 deferred the fc3 weight gradient but the "
                 "three-problem launch is not prepared (batch or input set changed between the stages)");
    p->b3w_deferred = false;
    TimedScope ts(p, G_B2D, st);   // per-kernel timing: one kernel, the flops of all three problems
    if (p->timing) {
      double f = 0.0;
      for (int id : {G_B2D, G_B2W, G_B3W}) { const GemmParams& q = gs->g[id].params; f += 2.0 * q.M * q.N * q.K; }
      p->t_flops[G_B2D] = f;
    }
    return gemm_run_chain(&p->ctx->c, gs->tri, st);
  }
  if (stage == 1 && p->split_stage1 && p->timing && p->batch > kBlockM) {
    // per-kernel timing of the split stage: the same three kernels, one after the other on `st`
    GemmSet* gs;
    RVAE_CHECK(get_set(p, &gs));
    RVAE_CHECK(run(p, G_B3D, st));
    RVAE_CHECK(prepare(p, *gs, G_B3W));
    {
      TimedScope ts(p, G_B3W, st);
      PreparedGemm w = gs->g[G_B3W];
      p->t_flops[G_B3W] = 2.0 * w.params.M * w.params.N * w.params.K;
      if (w.grid > p->s1_wgrad_ctas) w.grid = p->s1_wgrad_ctas;
      RVAE_CHECK(gemm_run(&p->ctx->c, w, st));
    }
    TimedScope ts(p, T_LATENT, st);
    RVAE_CHECK(launch_latent_bwd(&p->ctx->c, p->dz, p->eps, ext ? ext->lv : p->lv, p->mu, ext ? ext->g_mu : nullptr,
                                 ext ? ext->g_lv : nullptr, plan_kl(p), p->batch, L, p->dml.hi, p->dml.lo, grads + ly.b2, 1,
                                 p->fin_pending ? &p->fin : nullptr, st));
    p->fin_pending = false;
    p->dz_zeroed = true;
    return RVAE_OK;
  }
  if (stage == 1 && p->split_stage1 && p->two_streams && !p->timing && p->batch > kBlockM) {
    // latent dgrad, then the latent backward kernel (HBM-bound, feeds stage 2: the critical chain) on `st` while the fc3
    // weight gradient runs beside it on a second stream, held to a part of the machine
    RVAE_CHECK(ensure_side_stream(p));
    GemmSet* gs;
    RVAE_CHECK(get_set(p, &gs));
    RVAE_CHECK(prepare(p, *gs, G_B3D));
    RVAE_CHECK(prepare(p, *gs, G_B3W));
    RVAE_CHECK(gemm_run(&p->ctx->c, gs->g[G_B3D], st));
    RVAE_CUDA(cudaEventRecord(p->ev_s1_fork, st));
    RVAE_CUDA(cudaStreamWaitEvent(p->hp2, p->ev_s1_fork, 0));
    // Order matters: nothing co-resides with a GEMM CTA (it owns the SM's shared memory), so whichever kernel gets its
    // blocks resident first takes the SMs. s1_order = 0: the weight gradient follows the dgrad on `st` (its CTAs take
    // the first SMs the dgrad frees), the latent kernel fills the rest from the second stream; 1: the other way round.
    cudaStream_t s_w = p->s1_order == 0 ? st : p->hp2;
    cudaStream_t s_l = p->s1_order == 0 ? p->hp2 : st;
    auto run_wgrad = [&]() -> int {
      PreparedGemm w = gs->g[G_B3W];
      // persistent: the pairs stride over the units. Under data parallelism the all-reduce kernels live on the spare
      // SMs too: 64 CTAs there (measured at N = 2: 96 costs 3 %), 96 in a single process
      const int cap = (p->dp_enabled && p->ctx->dp_world > 1 && p->s1_wgrad_ctas > 64) ? 64 : p->s1_wgrad_ctas;
      if (w.grid > cap) w.grid = cap;
      return gemm_run(&p->ctx->c, w, s_w);
    };
    auto run_latent = [&]() -> int {
      return launch_latent_bwd(&p->ctx->c, p->dz, p->eps, ext ? ext->lv : p->lv, p->mu, ext ? ext->g_mu : nullptr,
                               ext ? ext->g_lv : nullptr, plan_kl(p), p->batch, L, p->dml.hi, p->dml.lo, grads + ly.b2, 1,
                               p->fin_pending ? &p->fin : nullptr, s_l);
    };
    if (p->s1_order == 0) { RVAE_CHECK(run_wgrad()); RVAE_CHECK(run_latent()); }
    else { RVAE_CHECK(run_latent()); RVAE_CHECK(run_wgrad()); }
    RVAE_CUDA(cudaEventRecord(p->ev_s1_join, p->hp2));
    p->fin_pending = false;
    p->dz_zeroed = true;
    RVAE_CUDA(cudaStreamWaitEvent(st, p->ev_s1_join, 0));
    return RVAE_OK;
  }
  // dgrad and weight gradient of the stage as ONE persistent launch over a mixed, load-balanced tile list
  bool fused = false;
  if (kDgrad[stage] >= 0 && p->dual_pairs > 0 && sched_usable(p)) {
    int pairs = stage_pairs(stage);
    if (stage == 1 && pairs > 64 && !getenv("RVAE_DUAL_PAIRS_S1")) pairs = 64;   // the small stage gains nothing from 10 more pairs
    GemmSet* gs;
    RVAE_CHECK(get_set(p, &gs));
    if (gs->dual_state[stage] == 0) {
      RVAE_CHECK(prepare(p, *gs, kDgrad[stage]));
      RVAE_CHECK(prepare(p, *gs, kWgrad[stage]));
      int* sched = p->sched_dev + ((size_t)p->cur * 6 + stage) * 128 * kSchedMax;
      const PreparedGemm* both[2] = {&gs->g[kDgrad[stage]], &gs->g[kWgrad[stage]]};
      const int rc = gemm_prepare_chain(&p->ctx->c, both, 2, pairs, sched, &gs->dual[stage]);
      gs->dual_state[stage] = rc == RVAE_OK ? 1 : -1;
      if (rc != RVAE_OK && rc != RVAE_ERR_UNSUPPORTED) return rc;
      if (rc == RVAE_OK) p->sched_batch = p->batch;
    }
    if (gs->dual_state[stage] == 1) {
      // per-kernel timing: the fused launch IS the kernel of this stage - its time and the flops of both problems are
      // booked on the dgrad's slot (the weight gradient's slot stays empty)
      TimedScope ts(p, kDgrad[stage], st);
      if (p->timing) {
        const GemmParams& a = gs->g[kDgrad[stage]].params;
        const GemmParams& b = gs->g[kWgrad[stage]].params;
        p->t_flops[kDgrad[stage]] = 2.0 * a.M * a.N * a.K + 2.0 * b.M * b.N * b.K;
      }
      RVAE_CHECK(gemm_run_chain(&p->ctx->c, gs->dual[stage], st));
      fused = true;
    }
  }
  if (!fused && kDgrad[stage] >= 0) RVAE_CHECK(run(p, kDgrad[stage], st));
  if (stage == 1) {
    TimedScope ts(p, T_LATENT, st);
    RVAE_CHECK(launch_latent_bwd(&p->ctx->c, p->dz, p->eps, ext ? ext->lv : p->lv, p->mu, ext ? ext->g_mu : nullptr,
                                 ext ? ext->g_lv : nullptr, plan_kl(p), p->batch, L, p->dml.hi, p->dml.lo, grads + ly.b2, 1,
                                 p->fin_pending ? &p->fin : nullptr, st));
    p->fin_pending = false;
    p->dz_zeroed = true;
  }
  return fused ? RVAE_OK : run(p, kWgrad[stage], st);
}

}  // namespace

extern "C" {

int rvae_plan_create(rvae_ctx* ctx, int S, int H, int L, int max_batch, int precision, rvae_plan** out) {
  CTX_OR_FAIL(ctx);
  RVAE_REQUIRE(out, RVAE_ERR_INVALID, "plan_create: null out");
  RVAE_REQUIRE(max_batch > 0, RVAE_ERR_INVALID, "plan_create: max_batch=%d", max_batch);
  RVAE_REQUIRE(precision == RVAE_PRECISION_BF16 || precision == RVAE_PRECISION_FP32, RVAE_ERR_INVALID,
               "plan_create: precision %d", precision);
  rvae_layout lay;
  int Sp, Hp, Lp;
  RVAE_CHECK(rvae_param_layout_padded(S, H, L, &lay, &Sp, &Hp, &Lp));
  rvae_plan* p = new (std::nothrow) rvae_plan();
  RVAE_REQUIRE(p, RVAE_ERR_INVALID, "plan_create: out of host memory");
  p->ctx = ctx; p->S = Sp; p->H = Hp; p->L = Lp; p->max_batch = max_batch; p->precision = precision;
  p->s_true = S; p->h_true = H; p->l_true = L;
  p->lay = lay; p->bound = false; p->batch = 0; p->have_eps = false; p->global_batch = 0; p->noise_row0 = 0;
  p->timing = false;
  p->kl_c0 = 0.f; p->kl_bl = 0.0; p->hp_dev = nullptr; p->hp_early = 0; p->dz_zeroed = false; p->dp_enabled = false;
  p->cur = 0; p->ticket_zeroed = false; p->ticket = nullptr; p->norm_ticket_zeroed = false;
  p->clip_max = nullptr; p->clip_norm_out = nullptr; p->clip_ring = 1;
  p->x_pitch = 0; p->x_pitch_alt = 0;
  p->fuse_latent = false;
  p->sched_batch = 0;
  memset(&p->pf, 0, sizeof(p->pf));
  for (int i = 0; i < 5; ++i) p->grads_zeroed[i] = false;
  p->streams_ready = false; p->ev_fork = nullptr;
  p->hp = nullptr; p->ev_hp_fork = nullptr; p->ev_hp_join = nullptr;
  p->comm_stream = nullptr; p->comm_stream2 = nullptr; p->ev_comm_fork = nullptr;
  for (int i = 0; i < 5; ++i) p->ev_comm_done[i] = nullptr;
  p->adam_stream = nullptr; p->ev_eps = nullptr; p->ev_adam_fork = nullptr; p->ev_adam_join = nullptr;
  p->eps_pending = false; p->fin_pending = false;
  p->two_streams = true;
  p->hp2 = nullptr; p->ev_s1_fork = nullptr; p->ev_s1_join = nullptr;
  p->split_stage1 = true;
  p->s1_wgrad_ctas = 96;   // measured (profiles/README.md): 96 CTAs, weight gradient first
  p->s1_order = 0;
  p->merge_b3w = false; p->allow_defer = false; p->b3w_deferred = false;
#if RVAE_EXPERIMENTS
  if (const char* e = getenv("RVAE_MERGE_B3W")) p->merge_b3w = atoi(e) != 0;
#endif
  p->adam_bg_blocks = 0;
  if (const char* e = getenv("RVAE_ADAM_BG_BLOCKS")) p->adam_bg_blocks = atoi(e) > 0 ? atoi(e) : 0;
  if (const char* e = getenv("RVAE_S1_ORDER")) p->s1_order = atoi(e) != 0;
  if (const char* e = getenv("RVAE_SPLIT_STAGE1")) p->split_stage1 = atoi(e) != 0;
  if (const char* e = getenv("RVAE_S1_WGRAD_CTAS")) {
    const int v = atoi(e);
    if (v >= 2 && v <= ctx->c.num_sms_total) p->s1_wgrad_ctas = v & ~1;
  }
  p->fuse_forward = false;  // measured: no faster than the four separate launches (profiles/README.md); opt-in
#if RVAE_EXPERIMENTS
  if (const char* e = getenv("RVAE_FUSE_LATENT")) p->fuse_latent = atoi(e) != 0;
  if (const char* e = getenv("RVAE_FUSE_FORWARD")) p->fuse_forward = atoi(e) != 0;
#endif
  p->dual_pairs = ctx->c.num_sms / 2;
  if (const char* e = getenv("RVAE_DUAL_PAIRS")) {
    const int v = atoi(e);
    if (v >= 0 && 2 * v <= ctx->c.num_sms_total) p->dual_pairs = v;
  }
  if (const char* e = getenv("RVAE_TWO_STREAMS")) p->two_streams = atoi(e) != 0;
  for (int i = 0; i < T_COUNT; ++i) { p->t_ms[i] = 0; p->t_n[i] = 0; p->t_flops[i] = 0; }
  p->out_mu = p->out_lv = p->out_xhat = nullptr;
  memset(&p->bufs, 0, sizeof(p->bufs));
  p->ws_bytes = carve(p, nullptr);
  *out = p;
  return RVAE_OK;
}

void rvae_plan_destroy(rvae_plan* plan) {
  if (!plan) return;
  for (auto& e : plan->ev_pool) {
    cudaEventDestroy(e.first);
    cudaEventDestroy(e.second);
  }
  if (plan->streams_ready) {
    cudaStreamSynchronize(plan->adam_stream);
    cudaStreamSynchronize(plan->hp);
    cudaStreamSynchronize(plan->comm_stream);
    cudaStreamSynchronize(plan->comm_stream2);
    cudaStreamDestroy(plan->comm_stream2);
    cudaEventDestroy(plan->ev_comm_fork);
    for (int i = 0; i < 5; ++i) cudaEventDestroy(plan->ev_comm_done[i]);
    cudaStreamDestroy(plan->comm_stream);
    cudaEventDestroy(plan->ev_hp_fork);
    cudaEventDestroy(plan->ev_hp_join);
    cudaStreamDestroy(plan->hp);
    cudaStreamSynchronize(plan->hp2);
    cudaStreamDestroy(plan->hp2);
    cudaEventDestroy(plan->ev_s1_fork);
    cudaEventDestroy(plan->ev_s1_join);
    cudaEventDestroy(plan->ev_fork);
    cudaEventDestroy(plan->ev_eps);
    cudaEventDestroy(plan->ev_adam_fork);
    cudaEventDestroy(plan->ev_adam_join);
    cudaStreamDestroy(plan->adam_stream);
  }
  delete plan;
}

int rvae_plan_enable_timing(rvae_plan* plan, int enable) {
  RVAE_REQUIRE(plan, RVAE_ERR_INVALID, "null rvae_plan");
  plan->timing = enable != 0;
  return RVAE_OK;
}

int rvae_plan_read_timing(rvae_plan* plan, float* ms, int64_t* launches, double* flops_per_launch) {
  RVAE_REQUIRE(plan && ms && launches && flops_per_launch, RVAE_ERR_INVALID, "plan_read_timing: null argument");
  static_assert(G_COUNT == RVAE_NUM_GEMM_SLOTS && T_COUNT == RVAE_NUM_TIMING_SLOTS, "slot count");
  for (auto& u : plan->ev_used) {
    auto& e = plan->ev_pool[u.second];
    RVAE_CUDA(cudaEventSynchronize(e.second));
    float t = 0.f;
    RVAE_CUDA(cudaEventElapsedTime(&t, e.first, e.second));
    plan->t_ms[u.first] += t;
    plan->t_n[u.first] += 1;
  }
  plan->ev_used.clear();
  for (int i = 0; i < T_COUNT; ++i) {
    ms[i] = (float)plan->t_ms[i];
    launches[i] = plan->t_n[i];
    flops_per_launch[i] = plan->t_flops[i];
    plan->t_ms[i] = 0; plan->t_n[i] = 0;
  }
  return RVAE_OK;
}

size_t rvae_plan_workspace_bytes(const rvae_plan* plan) { return plan ? plan->ws_bytes : 0; }

int rvae_plan_bind(rvae_plan* plan, const rvae_plan_buffers* b) {
  RVAE_REQUIRE(plan && b, RVAE_ERR_INVALID, "plan_bind: null argument");
  RVAE_REQUIRE(b->params && b->shadow_hi && b->workspace, RVAE_ERR_INVALID,
               "plan_bind: params, shadow_hi and workspace are required");
  RVAE_REQUIRE(plan->precision == RVAE_PRECISION_BF16 || b->shadow_lo, RVAE_ERR_INVALID,
               "plan_bind: fp32 mode needs shadow_lo");
  RVAE_REQUIRE((reinterpret_cast<uintptr_t>(b->workspace) & 255) == 0, RVAE_ERR_INVALID,
               "plan_bind: workspace must be 256-byte aligned");
  plan->bufs = *b;
  if (plan->precision == RVAE_PRECISION_BF16) plan->bufs.shadow_lo = nullptr;
  carve(plan, reinterpret_cast<uint8_t*>(b->workspace));
  plan->sets.clear();
  plan->sched_batch = 0;
  for (int i = 0; i < 5; ++i) plan->grads_zeroed[i] = false;
  plan->dz_zeroed = false;
  plan->cur = 0; plan->ticket_zeroed = false; plan->norm_ticket_zeroed = false;
  memset(&plan->pf, 0, sizeof(plan->pf));
  if (plan->two_streams) RVAE_CHECK(ensure_side_stream(plan));
  plan->bound = true;
  plan->batch = 0;
  return RVAE_OK;
}

int rvae_plan_sync_shadow(rvae_plan* plan, void* stream) {
  RVAE_CHECK(check_ready(plan, false));
  return launch_split_bf16(&plan->ctx->c, plan->bufs.params, plan->lay.total, BF(plan->bufs.shadow_hi),
                           BF(plan->bufs.shadow_lo), S_(stream));
}

int rvae_plan_load_frames(rvae_plan* plan, const void* audio, int audio_is_i16, int64_t n_samples,
                          const int64_t* frame_idx, int64_t first_frame, int count, int hop, int row_offset,
                          void* stream) {
  RVAE_CHECK(check_ready(plan, false));
  RVAE_REQUIRE(count > 0 && row_offset >= 0 && row_offset + count <= plan->max_batch, RVAE_ERR_INVALID,
               "plan_load_frames: rows %d..%d outside 0..%d", row_offset, row_offset + count, plan->max_batch);
  RVAE_REQUIRE(row_offset == 0 || row_offset == plan->batch, RVAE_ERR_STATE,
               "plan_load_frames: row_offset %d does not continue the loaded batch (%d rows)", row_offset,
               plan->batch);
  RVAE_REQUIRE(row_offset == 0 || plan->x_pitch == 0, RVAE_ERR_STATE,
               "plan_load_frames: cannot append rows to a batch that was loaded as a sample span");
  plan->batch = row_offset + count;
  plan->x_pitch = 0;
  plan->have_eps = false;
  const size_t off = (size_t)row_offset * plan->S;
  TimedScope ts(plan, T_LOAD, S_(stream));
  return launch_frame_gather(&plan->ctx->c, audio, audio_is_i16, n_samples, frame_idx, first_frame, count, hop,
                             plan->s_true, plan->S, plan->x.hi + off, plan->x.lo ? plan->x.lo + off : nullptr, nullptr,
                             S_(stream));
}

int rvae_plan_load_batch(rvae_plan* plan, const float* x, int batch, void* stream) {
  RVAE_CHECK(check_ready(plan, false));
  RVAE_REQUIRE(x, RVAE_ERR_INVALID, "plan_load_batch: null x");
  RVAE_REQUIRE(batch > 0 && batch <= plan->max_batch, RVAE_ERR_INVALID, "plan_load_batch: batch %d not in 1..%d",
               batch, plan->max_batch);
  plan->batch = batch;
  plan->x_pitch = 0;
  plan->have_eps = false;
  TimedScope ts(plan, T_LOAD, S_(stream));
  if (plan->s_true != plan->S)
    return launch_split_bf16_rows(&plan->ctx->c, x, batch, plan->s_true, plan->s_true, plan->S, plan->x.hi, plan->x.lo,
                                  S_(stream));
  return launch_split_bf16(&plan->ctx->c, x, (int64_t)batch * plan->S, plan->x.hi, plan->x.lo, S_(stream));
}

// A run of `count` frames at stride hop is one contiguous span of (count - 1) * hop + S samples: convert the span once
// (fp32 / PCM16 -> bf16 [+ residual plane]) into the x planes - the framing kernel with ONE "frame" of span length -
// and let the GEMMs read frame i at row pitch hop. Every sample is touched once instead of S / hop times and the
// [count, S] operand is never materialised (rawvae/dataset.py:61-69: sequential frames of a stream).
static int span_eligible(const rvae_plan* p, int count, int hop) {
  // 16-byte row pitch for the tensor maps; the span must fit the planes (hop <= S). A padded segment_length reads
  // zeros past S through the tensor maps; the fp32 mode's residual plane of x is read by the fc4 epilogue straight
  // from memory, where a frame's columns past S are the next frame's samples, so that mode gathers padded rows.
  const int S = p->s_true;
  return hop > 0 && hop % 8 == 0 && hop <= S && S % 8 == 0 && count > 0 && count <= p->max_batch &&
         (S == p->S || p->precision == RVAE_PRECISION_BF16);
}
static int convert_span(rvae_plan* p, const void* audio, int audio_is_i16, int64_t n_samples,
                        const int64_t* first_frame_dev, int64_t first_frame, int count, int hop, Planes& dst,
                        cudaStream_t st) {
  const int64_t span = (int64_t)(count - 1) * hop + p->s_true;
  RVAE_REQUIRE(span <= (int64_t)INT32_MAX, RVAE_ERR_UNSUPPORTED, "plan span: %lld samples", (long long)span);
  return launch_frame_gather(&p->ctx->c, audio, audio_is_i16, n_samples, first_frame_dev, first_frame, 1, hop,
                             (int)span, (int)span, dst.hi, dst.lo, nullptr, st);
}

int rvae_plan_span_supported(const rvae_plan* plan, int count, int hop) {
  return plan ? span_eligible(plan, count, hop) : 0;
}

int rvae_plan_load_span(rvae_plan* plan, const void* audio, int audio_is_i16, int64_t n_samples,
                        const int64_t* first_frame_dev, int64_t first_frame, int count, int hop, void* stream) {
  RVAE_CHECK(check_ready(plan, false));
  RVAE_REQUIRE(audio && span_eligible(plan, count, hop), RVAE_ERR_UNSUPPORTED,
               "plan_load_span: count %d (max %d), hop %d (needs hop %% 8 == 0 and hop <= S = %d; S %% 8 == 0; bf16 "
               "mode if S %% 64 != 0)", count, plan->max_batch, hop, plan->s_true);
  // (samples past n_samples read as zeros, exactly as in the gather: the zero-padded tail of a file)
  RVAE_REQUIRE(first_frame_dev || first_frame >= 0, RVAE_ERR_INVALID, "plan_load_span: first_frame %lld",
               (long long)first_frame);
  plan->batch = count;
  plan->x_pitch = hop;
  plan->have_eps = false;
  TimedScope ts(plan, T_LOAD, S_(stream));
  return convert_span(plan, audio, audio_is_i16, n_samples, first_frame_dev, first_frame, count, hop, plan->x,
                      S_(stream));
}

int rvae_plan_set_eps(rvae_plan* plan, const float* eps, void* stream) {
  RVAE_CHECK(check_ready(plan, true));
  RVAE_REQUIRE(eps, RVAE_ERR_INVALID, "plan_set_eps: null eps");
  if (plan->l_true != plan->L)
    RVAE_CHECK(pad_rows(plan->eps, eps, plan->batch, plan->l_true, plan->L, S_(stream)));
  else
    RVAE_CUDA(cudaMemcpyAsync(plan->eps, eps, sizeof(float) * (size_t)plan->batch * plan->L, cudaMemcpyDeviceToDevice,
                              S_(stream)));
  plan->have_eps = true;
  return RVAE_OK;
}

int rvae_plan_gen_eps(rvae_plan* plan, uint64_t seed, uint64_t offset, int add_step, void* stream) {
  RVAE_CHECK(check_ready(plan, true));
  RVAE_REQUIRE(!add_step || plan->bufs.step, RVAE_ERR_STATE, "plan_gen_eps(add_step): no step counter bound");
  plan->have_eps = true;
  cudaStream_t st = S_(stream);
  if (plan->two_streams && !plan->timing) {
    // fork: the noise does not depend on the batch load or fc1, so it is drawn on the background stream meanwhile;
    // rvae_plan_forward joins before the encoder head
    RVAE_CHECK(ensure_side_stream(plan));
    RVAE_CUDA(cudaEventRecord(plan->ev_fork, st));
    RVAE_CUDA(cudaStreamWaitEvent(plan->adam_stream, plan->ev_fork, 0));
    RVAE_CHECK(draw_eps(plan, plan->eps, plan->batch, seed, offset, add_step ? plan->bufs.step : nullptr,
                        plan->noise_row0, plan->adam_stream));
    RVAE_CUDA(cudaEventRecord(plan->ev_eps, plan->adam_stream));
    plan->eps_pending = true;
    return RVAE_OK;
  }
  TimedScope ts(plan, T_EPS, st);
  return draw_eps(plan, plan->eps, plan->batch, seed, offset, add_step ? plan->bufs.step : nullptr, plan->noise_row0,
                  st);
}

int rvae_plan_set_outputs(rvae_plan* plan, float* mu, float* logvar, float* xhat) {
  RVAE_REQUIRE(plan, RVAE_ERR_INVALID, "null rvae_plan");
  plan->out_mu = mu; plan->out_lv = logvar; plan->out_xhat = xhat;
  return RVAE_OK;
}

int rvae_plan_enable_dp(rvae_plan* plan, int on) {
  RVAE_REQUIRE(plan, RVAE_ERR_INVALID, "null rvae_plan");
  RVAE_REQUIRE(!on || plan->ctx->comm != nullptr || plan->ctx->p2p_ready, RVAE_ERR_STATE,
               "plan_enable_dp: call rvae_dp_init / rvae_dp_sym_open first");
  if (plan->dp_enabled != (on != 0) && !plan->sets.empty()) {
    // fused-launch schedules depend on the SM budget: rebuild them - once nothing in flight reads the old ones
    RVAE_CUDA(cudaDeviceSynchronize());
    plan->sets.clear();
    plan->sched_batch = 0;
  }
  plan->dp_enabled = on != 0;
  return RVAE_OK;
}

int rvae_plan_set_noise_rows(rvae_plan* plan, int64_t first_global_row) {
  RVAE_REQUIRE(plan && first_global_row >= 0, RVAE_ERR_INVALID, "plan_set_noise_rows: bad argument");
  plan->noise_row0 = first_global_row;
  return RVAE_OK;
}

int rvae_plan_set_global_batch(rvae_plan* plan, int64_t global_batch) {
  RVAE_REQUIRE(plan && global_batch >= 0, RVAE_ERR_INVALID, "plan_set_global_batch: bad argument");
  plan->global_batch = global_batch;
  return RVAE_OK;
}

int rvae_plan_forward(rvae_plan* plan, float kl_beta, int fused_loss, int want_xhat, void* stream) {
  RVAE_CHECK(check_ready(plan, true));
  RVAE_REQUIRE(plan->have_eps, RVAE_ERR_STATE, "plan_forward: call rvae_plan_set_eps / rvae_plan_gen_eps first");
  cudaStream_t st = S_(stream);
  rvae_plan* p = plan;
  const double nb = p->global_batch > 0 ? (double)p->global_batch : (double)p->batch;
  const double BL = nb * p->l_true, BS = nb * p->s_true;
  // caller tensors of a padded plan: the epilogues write the workspace, the true columns are copied out afterwards
  const bool lat_direct = p->L == p->l_true, rec_direct = p->S == p->s_true;
  GemmSet* gs;
  RVAE_CHECK(get_set(p, &gs));

  // Training step: the whole forward pass (fc1 -> encoder head -> fc3 -> fc4 + loss) as ONE persistent launch whose
  // tiles are chained by row-block dependencies (a tile of the next layer starts as soon as the tiles of its row
  // block are stored) - instead of four kernels with their fill, drain and half-empty last waves.
  const bool chain = fused_loss && !want_xhat && p->fuse_forward && p->dual_pairs > 0 && !p->timing && sched_usable(p) && !p->out_mu &&
                     !p->out_lv && !p->out_xhat && p->bufs.grads != nullptr;
  if (chain) {
    if (gs->fwd_state == 0) {
      static const int kLayers[4] = {G_F1, G_F2, G_F3, G_F4_OUT};
      const PreparedGemm* layers[4];
      for (int k = 0; k < 4; ++k) {
        RVAE_CHECK(prepare(p, *gs, kLayers[k]));
        layers[k] = &gs->g[kLayers[k]];
      }
      int* sched = p->sched_dev + ((size_t)p->cur * 6 + 3) * 128 * kSchedMax;
      int fpairs = p->dual_pairs;
      if (const char* e = getenv("RVAE_DUAL_PAIRS_F")) {
        const int v = atoi(e);
        if (v >= 1 && 2 * v <= p->ctx->c.num_sms_total) fpairs = v;
      }
      const int rc = gemm_prepare_chain(&p->ctx->c, layers, 4, fpairs, sched, &gs->fwd, p->dep_flags);
      gs->fwd_state = rc == RVAE_OK ? 1 : -1;
      if (rc != RVAE_OK && rc != RVAE_ERR_UNSUPPORTED) return rc;
      if (rc == RVAE_OK) p->sched_batch = p->batch;
    }
    if (gs->fwd_state == 1) {
      p->kl_c0 = (float)((double)kl_beta / BL);
      p->kl_bl = BL;
      RVAE_CHECK(ensure_bias_zeroed(p, st));   // F4's epilogue accumulates db4, the backward epilogues db3, db2, db1
      p->grads_zeroed[4] = false;
      RVAE_CUDA(cudaMemsetAsync(p->dep_flags, 0, sizeof(unsigned int) * 3 * 256, st));
      if (p->eps_pending) {
        RVAE_CUDA(cudaStreamWaitEvent(st, p->ev_eps, 0));
        p->eps_pending = false;
      }
      PreparedChain d = gs->fwd;
      d.params.p[3].epi.c0 = (float)(2.0 / BS);
      d.params.p[3].epi.out_f32 = nullptr;
      return gemm_run_chain(&p->ctx->c, d, st);
    }
  }
  RVAE_CHECK(run(p, G_F1, st));
  if (p->eps_pending) {
    RVAE_CUDA(cudaStreamWaitEvent(st, p->ev_eps, 0));
    p->eps_pending = false;
  }
  {
    RVAE_CHECK(prepare(p, *gs, G_F2));
    EpiArgs a = gs->g[G_F2].params.epi;
    if (p->out_mu && lat_direct) a.out_f32 = p->out_mu;
    if (p->out_lv && lat_direct) a.out_f32_b = p->out_lv;
    if (fused_loss) { p->kl_c0 = (float)((double)kl_beta / BL); p->kl_bl = BL; }
    else a.loss_acc = nullptr;
    RVAE_CHECK(run(p, G_F2, st, &a));
    if (!lat_direct) RVAE_CHECK(copy_latents_out(p, st));
  }
  RVAE_CHECK(run(p, G_F3, st));
  if (fused_loss) {
    RVAE_REQUIRE(p->bufs.grads, RVAE_ERR_STATE, "plan_forward(fused_loss): no grads buffer bound");
    RVAE_REQUIRE(!p->out_mu && !p->out_lv, RVAE_ERR_STATE,
                 "plan_forward(fused_loss): mu / logvar must stay in the workspace (the fused backward reads them)");
    RVAE_CHECK(ensure_bias_zeroed(p, st));   // F4's epilogue accumulates db4, the backward epilogues db3, db2, db1
    p->grads_zeroed[4] = false;              // ... so after this step the block is dirty again
    RVAE_CHECK(prepare(p, *gs, G_F4_OUT));
    EpiArgs a = gs->g[G_F4_OUT].params.epi;
    a.c0 = (float)(2.0 / BS);
    a.out_f32 = want_xhat ? (p->out_xhat && rec_direct ? p->out_xhat : p->xhat) : nullptr;
    RVAE_CHECK(run(p, G_F4_OUT, st, &a));
    if (want_xhat && p->out_xhat && !rec_direct) RVAE_CHECK(strip_rows(p->out_xhat, p->xhat, p->batch, p->s_true, p->S, st));
  } else {
    RVAE_CHECK(prepare(p, *gs, G_F4_LIN));
    EpiArgs a = gs->g[G_F4_LIN].params.epi;
    a.out_f32 = p->out_xhat && rec_direct ? p->out_xhat : p->xhat;
    RVAE_CHECK(run(p, G_F4_LIN, st, &a));
    if (p->out_xhat && !rec_direct) RVAE_CHECK(strip_rows(p->out_xhat, p->xhat, p->batch, p->s_true, p->S, st));
  }
  return RVAE_OK;
}

int rvae_plan_backward(rvae_plan* plan, int stage, void* stream) {
  RVAE_CHECK(check_ready(plan, true));
  RVAE_REQUIRE(plan->bufs.grads, RVAE_ERR_STATE, "plan_backward: no grads buffer bound");
  if (stage == -1) {
    plan->allow_defer = true;   // all four stages follow each other
    int rc = RVAE_OK;
    for (int s = 0; s < 4 && rc == RVAE_OK; ++s) rc = backward_stage(plan, s, nullptr, S_(stream));
    plan->allow_defer = false;
    return rc;
  }
  return backward_stage(plan, stage, nullptr, S_(stream));
}

int rvae_plan_backward_external(rvae_plan* plan, const float* g_xhat, const float* xhat, const float* g_mu,
                                const float* g_logvar, const float* logvar, void* stream) {
  RVAE_CHECK(check_ready(plan, true));
  RVAE_REQUIRE(plan->bufs.grads, RVAE_ERR_STATE, "plan_backward_external: no grads buffer bound");
  RVAE_REQUIRE(g_xhat && xhat && g_mu && g_logvar && logvar, RVAE_ERR_INVALID,
               "plan_backward_external: null argument");
  rvae_plan* p = plan;
  cudaStream_t st = S_(stream);
  if (p->S != p->s_true) {   // padded plan: the caller's [batch, S] tensors at the padded row pitch, zero padding
    RVAE_CHECK(pad_rows(p->ext_gx, g_xhat, p->batch, p->s_true, p->S, st));
    RVAE_CHECK(pad_rows(p->xhat, xhat, p->batch, p->s_true, p->S, st));
    g_xhat = p->ext_gx;
    xhat = p->xhat;
  }
  if (p->L != p->l_true) {
    RVAE_CHECK(pad_rows(p->ext_gmu, g_mu, p->batch, p->l_true, p->L, st));
    RVAE_CHECK(pad_rows(p->ext_glv, g_logvar, p->batch, p->l_true, p->L, st));
    RVAE_CHECK(pad_rows(p->ext_lv, logvar, p->batch, p->l_true, p->L, st));
    g_mu = p->ext_gmu;
    g_logvar = p->ext_glv;
    logvar = p->ext_lv;
  }
  RVAE_CHECK(ensure_bias_zeroed(p, st));
  p->grads_zeroed[4] = false;
  { TimedScope ts(p, T_TANHBWD, st); RVAE_CHECK(launch_tanh_bwd(&p->ctx->c, g_xhat, xhat, (int64_t)p->batch * p->S, p->da4.hi, p->da4.lo, st)); }
  { TimedScope ts(p, T_COLSUM, st);
    RVAE_CHECK(launch_colsum(&p->ctx->c, p->da4.hi, p->da4.lo, p->batch, p->S, p->S, p->bufs.grads + p->lay.b4, 1, st)); }
  const LatentExt ext = {g_mu, g_logvar, logvar};
  p->allow_defer = true;   // all four stages follow each other
  int rc = RVAE_OK;
  for (int s = 0; s < 4 && rc == RVAE_OK; ++s) rc = backward_stage(p, s, &ext, st);
  p->allow_defer = false;
  return rc;
}

int rvae_plan_finish_loss(rvae_plan* plan, float kl_beta, float* loss_out, int ring_size, void* stream) {
  RVAE_CHECK(check_ready(plan, true));
  RVAE_REQUIRE(ring_size >= 1, RVAE_ERR_INVALID, "plan_finish_loss: ring_size %d", ring_size);
  // The reported loss is the mean over THIS rank's frames (under data parallelism: an unbiased estimate of the
  // global mean that needs no collective); the gradients use the global-batch normalisation set on the plan.
  TimedScope ts(plan, T_FINALIZE, S_(stream));
  return launch_loss_finalize(&plan->ctx->c, plan->loss_acc, plan->batch, plan->s_true, plan->l_true, kl_beta, loss_out,
                              ring_size, plan->bufs.step, S_(stream));
}

int rvae_plan_finish_loss_deferred(rvae_plan* plan, float kl_beta, float* loss_out, int ring_size) {
  RVAE_CHECK(check_ready(plan, true));
  RVAE_REQUIRE(ring_size >= 1, RVAE_ERR_INVALID, "plan_finish_loss_deferred: ring_size %d", ring_size);
  plan->fin = make_loss_finalize(plan->loss_acc, plan->batch, plan->s_true, plan->l_true, kl_beta, loss_out, ring_size,
                                 plan->bufs.step);
  plan->fin_pending = true;
  return RVAE_OK;
}

int rvae_plan_prefetch_frames(rvae_plan* plan, const void* audio, int audio_is_i16, int64_t n_samples,
                              const int64_t* frame_idx, int64_t first_frame, int count, int hop, uint64_t seed,
                              uint64_t offset, int add_step) {
  RVAE_CHECK(check_ready(plan, false));
  RVAE_REQUIRE(audio && count > 0 && count <= plan->max_batch && hop > 0, RVAE_ERR_INVALID,
               "plan_prefetch_frames: bad arguments (count %d of max %d)", count, plan->max_batch);
  rvae_plan::Prefetch& f = plan->pf;
  f.audio = audio; f.audio_is_i16 = audio_is_i16; f.n_samples = n_samples; f.frame_idx = frame_idx;
  f.first_frame = first_frame; f.count = count; f.hop = hop; f.seed = seed; f.offset = offset; f.add_step = add_step;
  f.noise_row0 = plan->noise_row0;
  f.span = false;
  f.registered = true;
  return RVAE_OK;
}

int rvae_plan_prefetch_span(rvae_plan* plan, const void* audio, int audio_is_i16, int64_t n_samples,
                            const int64_t* first_frame_dev, int64_t first_frame, int count, int hop, uint64_t seed,
                            uint64_t offset, int add_step) {
  RVAE_CHECK(check_ready(plan, false));
  RVAE_REQUIRE(audio && span_eligible(plan, count, hop), RVAE_ERR_UNSUPPORTED,
               "plan_prefetch_span: count %d (max %d), hop %d (needs hop %% 8 == 0 and hop <= S = %d; S %% 8 == 0; "
               "bf16 mode if S %% 64 != 0)", count, plan->max_batch, hop, plan->s_true);
  RVAE_REQUIRE(first_frame_dev || first_frame >= 0, RVAE_ERR_INVALID, "plan_prefetch_span: first_frame %lld",
               (long long)first_frame);
  RVAE_CHECK(rvae_plan_prefetch_frames(plan, audio, audio_is_i16, n_samples, first_frame_dev, first_frame, count, hop,
                                       seed, offset, add_step));
  plan->pf.span = true;
  return RVAE_OK;
}

int rvae_plan_swap_prefetched(rvae_plan* plan) {
  RVAE_CHECK(check_ready(plan, false));
  RVAE_REQUIRE(plan->pf.ready_batch > 0, RVAE_ERR_STATE, "plan_swap_prefetched: no prefetched batch");
  std::swap(plan->x, plan->x_alt);
  std::swap(plan->x_pitch, plan->x_pitch_alt);
  std::swap(plan->eps, plan->eps_alt);
  plan->cur ^= 1;
  plan->batch = plan->pf.ready_batch;
  plan->pf.ready_batch = 0;
  plan->have_eps = true;
  plan->eps_pending = false;
  return RVAE_OK;
}

int rvae_plan_prefetched_batch(const rvae_plan* plan) { return plan ? plan->pf.ready_batch : 0; }

int rvae_plan_join_background(rvae_plan* plan, void* stream) {
  RVAE_CHECK(check_ready(plan, false));
  if (plan->eps_pending) {
    RVAE_CUDA(cudaStreamWaitEvent(S_(stream), plan->ev_eps, 0));
    plan->eps_pending = false;
  }
  return RVAE_OK;
}

int rvae_plan_note_prefetched(rvae_plan* plan, int count, int span_hop) {
  RVAE_CHECK(check_ready(plan, false));
  RVAE_REQUIRE(count > 0 && count <= plan->max_batch && span_hop >= 0, RVAE_ERR_INVALID,
               "plan_note_prefetched: count %d span_hop %d", count, span_hop);
  plan->pf.ready_batch = count;
  plan->x_pitch_alt = span_hop;
  return RVAE_OK;
}

int rvae_plan_adam(rvae_plan* plan, double lr, double beta1, double beta2, double eps, double weight_decay,
                   float grad_scale, int zero_grads, void* stream) {
  return rvae_plan_adam_buckets(plan, 0x1f, lr, beta1, beta2, eps, weight_decay, grad_scale, zero_grads, stream);
}

int rvae_plan_adam_buckets(rvae_plan* plan, unsigned bucket_mask, double lr, double beta1, double beta2, double eps,
                           double weight_decay, float grad_scale, int zero_grads, void* stream) {
  RVAE_CHECK(check_ready(plan, false));
  const rvae_plan_buffers& b = plan->bufs;
  RVAE_REQUIRE(b.grads && b.exp_avg && b.exp_avg_sq && b.step, RVAE_ERR_STATE,
               "plan_adam: grads / exp_avg / exp_avg_sq / step not bound");
  RVAE_REQUIRE(bucket_mask != 0 && bucket_mask <= 0x1f, RVAE_ERR_INVALID, "plan_adam_buckets: mask %#x", bucket_mask);
  // zero_grads: the kernel clears the gradient buffer after consuming it (what optimizer.zero_grad() does at the top
  // of the reference loop, train.py:184), so the next step's split-K weight gradients can reduce-add without memsets
  TimedScope ts(plan, T_ADAM, S_(stream));
  return adam_buckets(plan, bucket_mask, hp_value(lr, beta1, beta2, eps, weight_decay), grad_scale, zero_grads, 0,
                      false, S_(stream));
}

// The training step behind rvae_plan_train_step (hp by value, KL weight kl_beta) and rvae_plan_train_step_hp (hp.dev
// = the device record, which the Adam launches, the latent backward and the loss finalisation read instead)
static int train_step(rvae_plan* plan, float kl_beta, const HpArg& hp, int zero_grads, float* loss_out, int ring_size,
               void* stream) {
  RVAE_CHECK(check_ready(plan, true));
  const rvae_plan_buffers& b = plan->bufs;
  RVAE_REQUIRE(b.grads && b.exp_avg && b.exp_avg_sq && b.step, RVAE_ERR_STATE,
               "plan_train_step: grads / exp_avg / exp_avg_sq / step not bound");
  rvae_plan* p = plan;
  // The step counter t (Adam's bias correction, the loss-ring slot, the Philox offset) stays at its old value for
  // the whole step: every Adam launch uses t + 1, and the last block of the final launch advances it.
  const bool fork = plan->two_streams && !plan->timing;
  // Gradient clipping: the global norm depends on every bucket and Adam is nonlinear in g, so no bucket is updated
  // before the norm is known. Each bucket's norm partial takes the place of its background Adam launch; the last one
  // finalises the clipping factor, and one Adam launch over all buckets reads it.
  const bool clip = plan->clip_max != nullptr;
  // With a record bound, the latent backward evaluates it before griddepcontrol.wait, overlapping the GEMM before it,
  // when the step runs on the internal streams. That is safe: (1) the record is written by a copy the caller orders
  // before this call on `stream`, and every kernel of the step runs on `st` after cudaStreamWaitEvent(ev_hp_fork),
  // which is recorded on `stream` after the copy; (2) the step counter was last written by the previous step's final
  // Adam launch, an earlier operation of `st`; the wait on ev_hp_fork lies between it and this step's kernels, and a
  // stream operation other than a kernel starts only when every earlier operation of its stream is complete, so that
  // launch has completed before any kernel of this step starts (replays of a captured graph run one after the other:
  // the same holds); (3) no kernel of this step writes the counter before its final Adam launch. On one stream
  // (per-kernel timing, RVAE_TWO_STREAMS=0) only kernels separate the steps, and a chain of early starts could reach
  // back to the previous step's last kernel, so the kernel reads the record after griddepcontrol.wait.
  plan->hp_early = fork && plan->hp_dev != nullptr;
  if (!fork) {
    // (per-kernel timing / RVAE_TWO_STREAMS=0: a LOCAL step - no collectives are issued even when the context has a
    // communicator; bench.py's attribution pass runs this on rank 0 only)
    RVAE_CHECK(rvae_plan_forward(plan, kl_beta, 1, 0, stream));
    RVAE_CHECK(rvae_plan_finish_loss_deferred(plan, kl_beta, loss_out, ring_size));  // runs inside stage 1
    plan->fin.inc_step = 0;
    plan->fin.hp = hp.dev;
    RVAE_CHECK(rvae_plan_backward(plan, -1, stream));
    TimedScope ts(plan, T_ADAM, S_(stream));   // (gradient-norm launches are booked with Adam)
    if (clip) {
      NormFinalize fin = clip_finalize(plan);
      for (int k = 0; k < kNormGroups; ++k)
        RVAE_CHECK(grad_norm_group(plan, k, k == kNormGroups - 1 ? &fin : nullptr, S_(stream)));
    }
    return adam_buckets(plan, 0x1f, hp, 1.0f, zero_grads, 1, true, S_(stream), clip ? plan->clip_coef : nullptr);
  }
  // The critical chain (GEMMs) runs on a highest-priority stream; the HBM-bound side work (next batch + its noise,
  // Adam per bucket) on a lowest-priority background stream. The persistent GEMM grids leave the SMs that wave
  // quantisation would idle anyway to that background work (gemm_prepare), and at kernel boundaries a pending GEMM
  // CTA always wins the SM.
  RVAE_CHECK(ensure_side_stream(plan));
  cudaStream_t st = plan->hp, bg = plan->adam_stream;
  RVAE_CUDA(cudaEventRecord(plan->ev_hp_fork, S_(stream)));
  RVAE_CUDA(cudaStreamWaitEvent(st, plan->ev_hp_fork, 0));
  auto enqueue_prefetch = [&]() -> int {
    if (!p->pf.registered) return RVAE_OK;
    // next step's inputs: frames gathered into the alternate x planes, noise drawn into the alternate eps buffer
    const rvae_plan::Prefetch& f = p->pf;
    RVAE_CUDA(cudaStreamWaitEvent(bg, plan->ev_hp_fork, 0));
    if (f.span) {
      RVAE_CHECK(convert_span(p, f.audio, f.audio_is_i16, f.n_samples, f.frame_idx, f.first_frame, f.count, f.hop,
                              p->x_alt, bg));
      p->x_pitch_alt = f.hop;
    } else {
      RVAE_CHECK(launch_frame_gather(&p->ctx->c, f.audio, f.audio_is_i16, f.n_samples, f.frame_idx, f.first_frame,
                                     f.count, f.hop, p->s_true, p->S, p->x_alt.hi, p->x_alt.lo, nullptr, bg));
      p->x_pitch_alt = 0;
    }
    // the consumer sees a step counter advanced by one
    RVAE_CHECK(draw_eps(p, p->eps_alt, f.count, f.seed, f.offset + (f.add_step ? 1 : 0), f.add_step ? b.step : nullptr,
                        f.noise_row0, bg));
    p->pf.ready_batch = f.count;
    p->pf.registered = false;
    return RVAE_OK;
  };
  static const bool pf_late = getenv("RVAE_PF_LATE") ? atoi(getenv("RVAE_PF_LATE")) != 0 : false;
  if (!pf_late) RVAE_CHECK(enqueue_prefetch());
  RVAE_CHECK(rvae_plan_forward(plan, kl_beta, 1, 0, st));
  if (pf_late) {   // experiment: the GEMMs of the forward pass are in the hardware queues first
    RVAE_CUDA(cudaEventRecord(plan->ev_hp_fork, st));
    RVAE_CHECK(enqueue_prefetch());
  }
  RVAE_CHECK(rvae_plan_finish_loss_deferred(plan, kl_beta, loss_out, ring_size));  // runs inside stage 1
  plan->fin.inc_step = 0;
  plan->fin.hp = hp.dev;
  // Adam per bucket as soon as the bucket's gradient is complete; the dgrad GEMM that reads the bucket's bf16
  // shadow weights runs before the weight-gradient GEMM of the same stage, so nothing of this step reads them again.
  // Data parallelism: bucket s is SUM all-reduced (NCCL over NVLink / NVSwitch) on the communication stream as soon
  // as stage s completes it, under the GEMMs of the later stages; its Adam launch waits for the reduced gradient.
  // The loss was normalised by the global batch (rvae_plan_set_global_batch), so the sum IS the gradient.
  rvae_ctx* cx = plan->ctx;
  const bool dp = plan->dp_enabled && (cx->comm != nullptr || cx->p2p_ready) && cx->dp_world > 1;
  cudaStream_t cs = plan->comm_stream;
  // gradients that live in the symmetric allocation are reduced by our own peer-memory kernel; anything else by NCCL
  const uint8_t* g0 = reinterpret_cast<const uint8_t*>(b.grads);
  const bool use_p2p = cx->p2p_ready && cx->sym_base != nullptr && g0 >= cx->sym_base + kP2PFlagBytes &&
                       g0 + sizeof(float) * (size_t)plan->lay.total <= cx->sym_base + kP2PFlagBytes + cx->sym_data_bytes;
  RVAE_REQUIRE(!dp || use_p2p || cx->comm != nullptr, RVAE_ERR_STATE, "plan_train_step: no communicator for these gradients");
  // all-reduce of the gradient buckets in `mask` as ONE operation (a flag hop between two GPUs costs ~5 us, so
  // small buckets are merged): our kernel takes them as segments, NCCL gets one call per bucket
  auto allreduce_buckets = [&](unsigned mask, int flag_set, int ctas, cudaStream_t cs) -> int {
    P2PSegs sg;
    memset(&sg, 0, sizeof(sg));
    int ns = 0;
    for (int bucket = 0; bucket < 5; ++bucket) {
      if (!(mask & (1u << bucket))) continue;
      float* ptr; int64_t cnt;
      RVAE_CHECK(rvae_plan_bucket(plan, bucket, &ptr, &cnt));
      if (use_p2p) {
        RVAE_REQUIRE(ns < 3, RVAE_ERR_INVALID, "plan_train_step: too many segments in one all-reduce");
        sg.off[ns] = ptr - cx->p2p.data[cx->p2p.rank];
        sg.n[ns] = cnt;
        ++ns;
      } else {
        RVAE_NCCL(cx, cx->nccl.AllReduce(ptr, ptr, (size_t)cnt, /*ncclFloat32*/ 7, /*ncclSum*/ 0, cx->comm, cs));
      }
    }
    if (use_p2p) return launch_allreduce_p2p(&cx->c, cx->p2p, sg, flag_set, ctas, cs);
    return RVAE_OK;
  };
  static const unsigned kBucketMask[3] = {0x1, 0x2, 0x4};
  // with the latent backward fused into a GEMM epilogue no elementwise kernel of the critical chain is left to carry
  // the deferred loss finalisation: it rides on the background stream once the forward pass is known complete
  auto finalize_on_bg = [&]() -> int {
    if (!(plan->fin_pending && latent_fused(plan))) return RVAE_OK;
    RVAE_CHECK(launch_loss_finalize_prepared(&cx->c, plan->fin, bg));
    plan->fin_pending = false;
    return RVAE_OK;
  };
  // all stages of this pass are issued here: stage 1 may leave the fc3 weight gradient to stage 2's fused launch
  struct DeferGuard {
    rvae_plan* p;
    explicit DeferGuard(rvae_plan* p_) : p(p_) { p->allow_defer = true; }
    ~DeferGuard() { p->allow_defer = false; p->b3w_deferred = false; }
  } defer_guard(plan);
  bool w3_with_stage2 = false;
  for (int s = 0; s < 3; ++s) {
    RVAE_CHECK(rvae_plan_backward(plan, s, st));
    if (s == 1) w3_with_stage2 = plan->b3w_deferred;
    if (dp) {
      // exchanges per step: W4 after stage 0, W3 after stage 1 (or, when stage 1 left its weight gradient to stage 2,
      // together with the next one), W2 + all biases after stage 2 (kept small: it must be out of the way when stage
      // 3 ends), W1 after stage 3
      static const unsigned kExchange[3] = {0x1u, 0x2u, 0x14u};
      if (s == 1 && w3_with_stage2) continue;   // bucket 1 is not complete yet
      const unsigned extra = (s == 2 && w3_with_stage2) ? 0x2u : 0u;
      RVAE_CUDA(cudaEventRecord(plan->ev_comm_fork, st));
      RVAE_CUDA(cudaStreamWaitEvent(cs, plan->ev_comm_fork, 0));
      RVAE_CHECK(allreduce_buckets(kExchange[s] | extra, s, cx->p2p_ctas, cs));
      RVAE_CUDA(cudaEventRecord(plan->ev_comm_done[s], cs));
      RVAE_CUDA(cudaStreamWaitEvent(bg, plan->ev_comm_done[s], 0));
      if (s == 0) RVAE_CHECK(finalize_on_bg());
      if (clip) {
        if (extra) RVAE_CHECK(grad_norm_group(plan, 1, nullptr, bg));
        RVAE_CHECK(grad_norm_group(plan, s, nullptr, bg));   // norm group s = the buckets of exchange s
      } else {
        RVAE_CHECK(adam_buckets(plan, kBucketMask[s] | extra, hp, 1.0f, zero_grads, 1, false, bg));
      }
      continue;
    }
    if (clip) {
      // single process: the norm partial of each bucket on the background stream as soon as its stage completes it
      if (s == 1 && w3_with_stage2) continue;   // W3's gradient is complete after stage 2
      RVAE_CUDA(cudaEventRecord(plan->ev_adam_fork, st));
      RVAE_CUDA(cudaStreamWaitEvent(bg, plan->ev_adam_fork, 0));
      if (s == 0) RVAE_CHECK(finalize_on_bg());
      if (s == 2 && w3_with_stage2) RVAE_CHECK(grad_norm_group(plan, 1, nullptr, bg));
      RVAE_CHECK(grad_norm_group(plan, s, nullptr, bg));
      continue;
    }
    // single process: only W4 (the first bucket to complete, with the most GEMM time left to hide under) is updated
    // in the background; W3 and W2 would queue behind it and end up as two more exposed launches after stage 3, so
    // they join W1 and the biases in the final launch (W1|W2|W3 are contiguous in the flat buffer)
    if (s == 0) {
      RVAE_CUDA(cudaEventRecord(plan->ev_adam_fork, st));
      RVAE_CUDA(cudaStreamWaitEvent(bg, plan->ev_adam_fork, 0));
      RVAE_CHECK(finalize_on_bg());
      // (single process) held to adam_bg_blocks blocks: it then lives on the SMs the 128-CTA GEMM grids leave free
      // instead of taking every SM a finishing GEMM releases before the latent kernel of stage 1 gets there
      cx->c.aux_grid_cap = plan->adam_bg_blocks;
      const int rc_bg = adam_buckets(plan, kBucketMask[0], hp, 1.0f, zero_grads, 1, false, bg);
      cx->c.aux_grid_cap = 0;
      RVAE_CHECK(rc_bg);
    }
  }
  RVAE_CUDA(cudaEventRecord(plan->ev_adam_join, bg));
  RVAE_CHECK(rvae_plan_backward(plan, 3, st));
  if (dp) {
    // The last exchange is exposed and has the machine to itself: more CTAs, more NVLink bytes in flight. With our
    // own kernel it runs on a second communication stream, so it starts when stage 3 ends even if the previous
    // exchange is still waiting for a slower rank (different flag sets; the earlier kernel is already resident).
    cudaStream_t cs3 = use_p2p ? plan->comm_stream2 : cs;
    RVAE_CUDA(cudaEventRecord(plan->ev_comm_fork, st));
    RVAE_CUDA(cudaStreamWaitEvent(cs3, plan->ev_comm_fork, 0));
    RVAE_CHECK(allreduce_buckets(0x8u, 3, cx->p2p_ctas_last, cs3));
    RVAE_CUDA(cudaEventRecord(plan->ev_comm_done[3], cs3));
    RVAE_CUDA(cudaStreamWaitEvent(st, plan->ev_comm_done[3], 0));
    RVAE_CUDA(cudaStreamWaitEvent(st, plan->ev_comm_done[2], 0));   // the bias bucket travelled with exchange 2
  }
  RVAE_CUDA(cudaStreamWaitEvent(st, plan->ev_adam_join, 0));  // every earlier Adam launch has read the step counter
  if (clip) {
    // (the background norm partials are complete: the wait above)
    NormFinalize fin = clip_finalize(plan);
    RVAE_CHECK(grad_norm_group(plan, 3, &fin, st));
    RVAE_CHECK(adam_buckets(plan, 0x1fu, hp, 1.0f, zero_grads, 1, true, st, plan->clip_coef));
  } else {
    RVAE_CHECK(adam_buckets(plan, dp ? 0x18u : 0x1eu, hp, 1.0f, zero_grads, 1, true, st));
  }
  RVAE_CUDA(cudaEventRecord(plan->ev_hp_join, st));
  RVAE_CUDA(cudaStreamWaitEvent(S_(stream), plan->ev_hp_join, 0));
  return RVAE_OK;
}

int rvae_plan_train_step(rvae_plan* plan, float kl_beta, double lr, double beta1, double beta2, double eps,
                         double weight_decay, int zero_grads, float* loss_out, int ring_size, void* stream) {
  return train_step(plan, kl_beta, hp_value(lr, beta1, beta2, eps, weight_decay), zero_grads, loss_out, ring_size,
                    stream);
}

int rvae_plan_train_step_hp(rvae_plan* plan, const rvae_hparams* hp_dev, int zero_grads, float* loss_out,
                            int ring_size, void* stream) {
  RVAE_REQUIRE(hp_dev != nullptr && ring_size >= 1, RVAE_ERR_INVALID, "plan_train_step_hp: null record or ring_size %d",
               ring_size);
  RVAE_CHECK(check_ready(plan, true));
  // the experiments-only fused latent epilogue takes its KL scale from the host (EpiArgs::c0)
  RVAE_REQUIRE(!latent_fused(plan), RVAE_ERR_UNSUPPORTED,
               "plan_train_step_hp: the fused latent epilogue (RVAE_FUSE_LATENT) does not read the record");
  struct HpGuard {   // the record is bound for the kernels of this call only
    rvae_plan* p;
    HpGuard(rvae_plan* p_, const rvae_hparams* hp) : p(p_) { p->hp_dev = hp; }
    ~HpGuard() { p->hp_dev = nullptr; p->hp_early = 0; }
  } guard(plan, hp_dev);
  return train_step(plan, 0.0f, hp_device(hp_dev), zero_grads, loss_out, ring_size, stream);
}

int rvae_plan_set_grad_clip(rvae_plan* plan, const double* max_norm_dev, float* norm_out, int ring_size) {
  RVAE_REQUIRE(norm_out == nullptr || ring_size >= 1, RVAE_ERR_INVALID, "plan_set_grad_clip: ring_size %d", ring_size);
  RVAE_REQUIRE(plan, RVAE_ERR_INVALID, "null rvae_plan");
  // the experiments-only fused latent epilogue runs its own stage-1 path, which this step layout does not cover
  RVAE_REQUIRE(max_norm_dev == nullptr || !(plan->fuse_latent && plan->precision == RVAE_PRECISION_BF16),
               RVAE_ERR_UNSUPPORTED,
               "plan_set_grad_clip: the fused latent epilogue (RVAE_FUSE_LATENT) is not supported");
  plan->clip_max = max_norm_dev;
  plan->clip_norm_out = max_norm_dev ? norm_out : nullptr;
  plan->clip_ring = norm_out ? ring_size : 1;
  return RVAE_OK;
}

int rvae_plan_grad_norm(rvae_plan* plan, float* norm_out, void* stream) {
  RVAE_REQUIRE(norm_out, RVAE_ERR_INVALID, "plan_grad_norm: null norm_out");
  RVAE_CHECK(check_ready(plan, false));
  RVAE_REQUIRE(plan->bufs.grads, RVAE_ERR_STATE, "plan_grad_norm: grads not bound");
  NormFinalize fin;
  memset(&fin, 0, sizeof(fin));
  fin.norm_out = norm_out;
  fin.ring_size = 1;
  for (int k = 0; k < kNormGroups; ++k)
    RVAE_CHECK(grad_norm_group(plan, k, k == kNormGroups - 1 ? &fin : nullptr, S_(stream)));
  return RVAE_OK;
}

int rvae_hparams_check(const rvae_hparams* h) {
  RVAE_REQUIRE(h, RVAE_ERR_INVALID, "hparams_check: null record");
  const double vals[9] = {h->lr, h->beta1, h->beta2, h->eps, h->weight_decay, h->kl_beta, h->lr_min, h->kl_beta_start,
                          h->kl_cycle_ratio};
  for (double v : vals) RVAE_REQUIRE(std::isfinite(v), RVAE_ERR_INVALID, "hparams_check: non-finite value");
  RVAE_REQUIRE(h->lr_schedule >= RVAE_LR_CONSTANT && h->lr_schedule <= RVAE_LR_COSINE, RVAE_ERR_INVALID,
               "hparams_check: lr_schedule %d", h->lr_schedule);
  RVAE_REQUIRE(h->kl_anneal >= RVAE_KL_CONSTANT && h->kl_anneal <= RVAE_KL_CYCLICAL, RVAE_ERR_INVALID,
               "hparams_check: kl_anneal %d", h->kl_anneal);
  RVAE_REQUIRE(h->warmup_steps >= 0, RVAE_ERR_INVALID, "hparams_check: warmup_steps %lld", (long long)h->warmup_steps);
  RVAE_REQUIRE(h->total_steps >= 1 || (h->lr_schedule == RVAE_LR_CONSTANT && h->kl_anneal != RVAE_KL_CYCLICAL),
               RVAE_ERR_INVALID, "hparams_check: total_steps %lld", (long long)h->total_steps);
  RVAE_REQUIRE(h->kl_anneal_steps >= 1 || h->kl_anneal != RVAE_KL_LINEAR, RVAE_ERR_INVALID,
               "hparams_check: kl_anneal_steps %lld", (long long)h->kl_anneal_steps);
  RVAE_REQUIRE(h->kl_cycles >= 1 || h->kl_anneal != RVAE_KL_CYCLICAL, RVAE_ERR_INVALID, "hparams_check: kl_cycles %lld",
               (long long)h->kl_cycles);
  RVAE_REQUIRE(h->kl_cycle_ratio > 0.0 && h->kl_cycle_ratio <= 1.0, RVAE_ERR_INVALID, "hparams_check: kl_cycle_ratio %g",
               h->kl_cycle_ratio);
  return RVAE_OK;
}

int rvae_hparams_eval(rvae_ctx* ctx, const rvae_hparams* hp_dev, const int64_t* k_dev, int n, double* lr_out,
                      float* beta_out, void* stream) {
  // arguments first: a malformed call is reported the same way with or without a device
  RVAE_REQUIRE(hp_dev && k_dev && lr_out && beta_out && n > 0, RVAE_ERR_INVALID,
               "hparams_eval: null buffer or n %d (need n > 0)", n);
  CTX_OR_FAIL(ctx);
  return launch_hparams_eval(&ctx->c, hp_dev, k_dev, n, lr_out, beta_out, S_(stream));
}

const float* rvae_plan_mu(const rvae_plan* plan) { return plan ? plan->mu : nullptr; }
const float* rvae_plan_logvar(const rvae_plan* plan) { return plan ? plan->lv : nullptr; }
const float* rvae_plan_xhat(const rvae_plan* plan) { return plan ? plan->xhat : nullptr; }
const float* rvae_plan_eps(const rvae_plan* plan) { return plan ? plan->eps : nullptr; }

int rvae_plan_activation(const rvae_plan* plan, int which, void** hi, void** lo, int* cols) {
  RVAE_REQUIRE(plan && hi && lo && cols, RVAE_ERR_INVALID, "plan_activation: null argument");
  RVAE_REQUIRE(plan->bound, RVAE_ERR_STATE, "plan_activation: plan not bound");
  const Planes* t[8] = {&plan->x, &plan->h1, &plan->z, &plan->h3, &plan->da4, &plan->da3, &plan->dml, &plan->da1};
  const int c[8] = {plan->S, plan->H, plan->L, plan->H, plan->S, plan->H, 2 * plan->L, plan->H};
  RVAE_REQUIRE(which >= 0 && which < 8, RVAE_ERR_INVALID, "plan_activation: which=%d not in 0..7", which);
  *hi = t[which]->hi; *lo = t[which]->lo; *cols = c[which];
  return RVAE_OK;
}

int rvae_plan_bucket(const rvae_plan* plan, int s, float** ptr, int64_t* count) {
  RVAE_REQUIRE(plan && ptr && count, RVAE_ERR_INVALID, "plan_bucket: null argument");
  RVAE_REQUIRE(plan->bound && plan->bufs.grads, RVAE_ERR_STATE, "plan_bucket: grads not bound");
  const rvae_layout& ly = plan->lay;
  float* g = plan->bufs.grads;
  const int64_t S = plan->S, H = plan->H, L = plan->L;
  switch (s) {
    case 0: *ptr = g + ly.w4; *count = S * H; break;
    case 1: *ptr = g + ly.w3; *count = H * L; break;
    case 2: *ptr = g + ly.w2; *count = 2 * L * H; break;
    case 3: *ptr = g + ly.w1; *count = H * S; break;
    case 4: *ptr = g + ly.b1; *count = ly.total - ly.b1; break;
    default: return set_error(RVAE_ERR_INVALID, "plan_bucket: bucket %d not in 0..4", s);
  }
  return RVAE_OK;
}

int rvae_plan_decode(rvae_plan* plan, const float* z, int batch, float* xhat_out, void* stream) {
  RVAE_CHECK(check_ready(plan, false));
  RVAE_REQUIRE(z && xhat_out, RVAE_ERR_INVALID, "plan_decode: null buffer");
  RVAE_REQUIRE(batch > 0 && batch <= plan->max_batch, RVAE_ERR_INVALID, "plan_decode: batch %d not in 1..%d", batch,
               plan->max_batch);
  rvae_plan* p = plan;
  cudaStream_t st = S_(stream);
  p->batch = batch;
  p->have_eps = false;
  if (p->l_true != p->L)
    RVAE_CHECK(launch_split_bf16_rows(&p->ctx->c, z, batch, p->l_true, p->l_true, p->L, p->z.hi, p->z.lo, st));
  else
    RVAE_CHECK(launch_split_bf16(&p->ctx->c, z, (int64_t)batch * p->L, p->z.hi, p->z.lo, st));
  return decode_tail(p, xhat_out, st);
}

int rvae_plan_decode_lerp(rvae_plan* plan, const float* mu_a, const float* logvar_a, const float* mu_b,
                          const float* logvar_b, const void* alpha, int alpha_is_f64, const float* eps, int batch,
                          float* xhat_out, void* stream) {
  RVAE_CHECK(check_ready(plan, false));
  RVAE_REQUIRE(mu_a && logvar_a && mu_b && logvar_b && alpha && xhat_out, RVAE_ERR_INVALID, "plan_decode_lerp: null buffer");
  RVAE_REQUIRE(batch > 0 && batch <= plan->max_batch, RVAE_ERR_INVALID, "plan_decode_lerp: batch %d not in 1..%d", batch,
               plan->max_batch);
  rvae_plan* p = plan;
  cudaStream_t st = S_(stream);
  p->batch = batch;
  p->have_eps = false;
  // interpolated latents -> z written straight into fc3's bf16 operand planes (no fp32 z, no split pass)
  RVAE_CHECK(launch_lerp_reparam(&p->ctx->c, mu_a, logvar_a, mu_b, logvar_b, alpha, alpha_is_f64, eps, batch, p->l_true,
                                 p->L, nullptr, p->z.hi, p->z.lo, nullptr, nullptr, st));
  return decode_tail(p, xhat_out, st);
}

int rvae_plan_encode(rvae_plan* plan, void* stream) {
  RVAE_CHECK(check_ready(plan, true));
  rvae_plan* p = plan;
  cudaStream_t st = S_(stream);
  RVAE_CHECK(run(p, G_F1, st));
  GemmSet* gs;
  RVAE_CHECK(get_set(p, &gs));
  RVAE_CHECK(prepare(p, *gs, G_F2));
  EpiArgs a = gs->g[G_F2].params.epi;
  const bool lat_direct = p->L == p->l_true;
  if (p->out_mu && lat_direct) a.out_f32 = p->out_mu;
  if (p->out_lv && lat_direct) a.out_f32_b = p->out_lv;
  a.in0 = nullptr; a.out_hi = nullptr; a.out_lo = nullptr;
  a.loss_acc = nullptr;
  RVAE_CHECK(run(p, G_F2, st, &a));
  return lat_direct ? RVAE_OK : copy_latents_out(p, st);
}

}  // extern "C"
