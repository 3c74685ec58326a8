// Internal (non-ABI) declarations shared by the translation units of librvae_b200.so.
#pragma once
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "../../include/rvae_b200.h"
#include "gemm.cuh"

namespace rvae {

// Error codes returned across the C ABI (0 = ok). CUDA runtime errors are returned as 1000 + cudaError_t.
enum : int {
  RVAE_OK = 0,
  RVAE_ERR_INVALID = 1,      // bad argument (null pointer, misaligned buffer, negative size)
  RVAE_ERR_UNSUPPORTED = 2,  // shape not supported by the sm_100a kernels (see DESIGN.md constraints)
  RVAE_ERR_DRIVER = 3,       // cuTensorMapEncodeTiled or driver entry point failure
  RVAE_ERR_STATE = 4,        // plan not bound / wrong call order
  RVAE_ERR_CUDA_BASE = 1000,
};

int set_error(int code, const char* fmt, ...);
int cuda_error(cudaError_t err, const char* what);

#define RVAE_CUDA(expr)                                       \
  do {                                                        \
    cudaError_t _e = (expr);                                  \
    if (_e != cudaSuccess) return ::rvae::cuda_error(_e, #expr); \
  } while (0)

#define RVAE_CHECK(expr)           \
  do {                             \
    int _rc = (expr);              \
    if (_rc != RVAE_OK) return _rc; \
  } while (0)

#define RVAE_REQUIRE(cond, code, ...)                        \
  do {                                                       \
    if (!(cond)) return ::rvae::set_error(code, __VA_ARGS__); \
  } while (0)

struct Ctx {
  int device;
  int num_sms;
  int num_sms_total;  // SMs of the device (num_sms may be capped by RVAE_NUM_SMS)
  int force_block_n;  // 0 = heuristic, 128 / 256 = forced (env RVAE_BLOCK_N, for experiments)
  int force_cta_group;  // 0 = heuristic, 1 / 2 = forced (env RVAE_CTA_GROUP, for experiments)
  int debug;            // env RVAE_DEBUG, experiments only (see GemmParams::debug)
  int use_pdl;          // programmatic dependent launch between consecutive kernels (env RVAE_PDL=0 disables)
  unsigned long long* trace;  // GEMM timeline trace buffer (rvae_debug_set_trace), nullptr = off
  int trace_launches;         // capacity of the trace buffer in launches (successive launches use successive slabs)
  uint64_t trace_seq;         // GEMM launches since the trace was set
  unsigned long long* aux_trace;  // elementwise-kernel trace: [aux_cap][8] = {first start, last end, kind, blocks, 4 x detail}
  int aux_cap;
  uint64_t aux_seq;
  uint64_t launches;  // number of kernels launched through this context (bench.py reports it)
  int aux_grid_cap;   // > 0: upper bound for the grid of the next Adam launch (background launches of a training step
                      // are held to the SMs the GEMM grids leave free, so they do not squat on SMs a waiting
                      // high-priority kernel wants: resident blocks are never preempted)
};

// Launch with programmatic stream serialization: the kernel may start (and run its prologue) while the previous
// kernel of the stream drains; every kernel of this library executes griddepcontrol.wait before touching memory.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_kernel(const Ctx* ctx, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                                 cudaStream_t stream, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = ctx->use_pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// Debug trace of an elementwise launch (rvae_debug_set_aux_trace): globaltimer of the first block start / last block
// end. kind: 1 gather, 2 randn, 3 latent_bwd, 4 adam.
struct AuxTrace {
  unsigned long long* slot;  // nullptr = off
};
inline AuxTrace next_aux(Ctx* ctx, int kind) {
  AuxTrace t;
  t.slot = nullptr;
  if (ctx->aux_trace != nullptr && ctx->aux_cap > 0) {
    t.slot = ctx->aux_trace + (ctx->aux_seq % (uint64_t)ctx->aux_cap) * 8;
    ctx->aux_seq++;
    (void)kind;
  }
  return t;
}

// A bf16 GEMM operand. K-major: storage [mn][k] (k contiguous, row pitch ld). MN-major: storage [k][mn].
struct Operand {
  const __nv_bfloat16* hi;
  const __nv_bfloat16* lo;  // optional residual plane (fp32 emulation)
  int major;
  int ld;    // elements
  int cols;  // > 0: only the first `cols` elements of each row are data, the rest read as zeros through the tensor
             // map (frames read in place whose segment_length is padded up to the GEMM's extent); 0 = the full extent
};

struct GemmDesc {
  int epi;
  int M, N, K;
  Operand A, B;
  EpiArgs args;
  int head_L;    // EPI_HEAD: latent width L (B holds 2L stacked rows, N must equal 2L)
  int k_splits;  // EPI_WGRAD: requested split-K (0 = choose)
  int side_cols; // EPI_OUT: > 0 = columns of the side input x that are data (as Operand::cols); 0 = N
};

struct PreparedGemm {
  GemmParams params;
  int block_n;
  int variant;  // index into the kernel table
  int grid;
  int smem_bytes;
  // geometry of the epilogue's output tensors (for re-binding output pointers)
  int epi;
  int a_major, b_major, cg;
  int out_rows, out_cols_bf16, out_ld_bf16, out_cols_f32, out_ld_f32;
  int side_cols;  // GemmDesc::side_cols
};

int gemm_bind_outputs(PreparedGemm* g, const EpiArgs& args, bool force);

// Up to four prepared GEMMs fused into one persistent launch (gemm_chain_kernel_2cta): units are assigned to CTA pairs
// by a host-built schedule stored in device memory.
struct PreparedChain {
  ChainParams params;
  int count;    // problems
  int variant;  // index into the chain kernel table
  int grid;
  int smem_bytes;
};
// g[0..count): the problems. sched_dev: device buffer of at least pairs * kSchedMax ints (written here with a
// synchronous copy). dep_flags == nullptr: independent problems, longest-processing-time-first schedule.
// dep_flags != nullptr: problem i + 1 consumes problem i's output row block by row block; dep_flags points to
// (count - 1) x 256 device counters the caller zeroes before every launch, and the schedule lists the problems
// layer by layer (every pair runs a subsequence of one global order in which producers precede consumers, which
// makes the in-kernel dependency waits deadlock-free).
int gemm_prepare_chain(const Ctx* ctx, const PreparedGemm* const* g, int count, int pairs, int* sched_dev,
                       PreparedChain* out, unsigned int* dep_flags = nullptr);
int gemm_run_chain(Ctx* ctx, const PreparedChain& g, cudaStream_t stream);

int gemm_prepare(const Ctx* ctx, const GemmDesc& d, PreparedGemm* out);
int gemm_run(Ctx* ctx, const PreparedGemm& g, cudaStream_t stream);
int gemm_launch(Ctx* ctx, const GemmDesc& d, cudaStream_t stream);  // prepare + run

// Elementwise launchers (elementwise.cu)
int launch_frame_gather(Ctx* ctx, const void* audio, int audio_is_i16, int64_t n_samples, const int64_t* frame_idx,
                        int64_t first_frame, int64_t n_frames, int hop, int S, int W, __nv_bfloat16* out_hi,
                        __nv_bfloat16* out_lo, float* out_f32, cudaStream_t stream);
int launch_overlap_add(Ctx* ctx, const float* frames, int64_t n_frames, int S, int hop, float* out, int64_t t_begin,
                       int64_t n_out, cudaStream_t stream);
int launch_randn(Ctx* ctx, float* out, int64_t n, uint64_t seed, uint64_t offset, const float* offset_src,
                 int64_t elem_base, cudaStream_t stream);
int launch_randn_rows(Ctx* ctx, float* out, int64_t rows, int64_t cols, int64_t ld, uint64_t seed, uint64_t offset,
                      const float* offset_src, int64_t elem_base, cudaStream_t stream);
int launch_split_bf16_rows(Ctx* ctx, const float* src, int64_t rows, int cols, int ld_src, int ld_dst,
                           __nv_bfloat16* hi, __nv_bfloat16* lo, cudaStream_t stream);
int launch_split_bf16(Ctx* ctx, const float* src, int64_t n, __nv_bfloat16* hi, __nv_bfloat16* lo,
                      cudaStream_t stream);
int launch_colsum(Ctx* ctx, const __nv_bfloat16* hi, const __nv_bfloat16* lo, int64_t M, int N, int ld, float* out,
                  int accumulate, cudaStream_t stream);
int launch_loss_fwd(Ctx* ctx, const float* xhat, const float* x, const float* mu, const float* lv, int64_t B, int S,
                    int L, float beta, double* acc, float* loss_out, cudaStream_t stream);
int launch_frame_loss(Ctx* ctx, const float* xhat, int ld_xhat, const float* mu, const float* lv, int ld_lat,
                      int64_t rows, int S, int L, const void* audio, int audio_is_i16, int64_t n_samples,
                      int64_t first_frame, int hop, float* rec_out, float* kl_out, cudaStream_t stream);
int launch_loss_bwd(Ctx* ctx, const float* xhat, const float* x, const float* mu, const float* lv, int64_t B, int S,
                    int L, float beta, const float* grad_out, float* g_xhat, float* g_mu, float* g_lv,
                    cudaStream_t stream);
int launch_tanh_bwd(Ctx* ctx, const float* g_xhat, const float* xhat, int64_t n, __nv_bfloat16* da_hi,
                    __nv_bfloat16* da_lo, cudaStream_t stream);
int launch_reparam(Ctx* ctx, const float* mu, const float* lv, const float* eps, int64_t n, float* z,
                   cudaStream_t stream);
int launch_lerp_reparam(Ctx* ctx, const float* mu_a, const float* lv_a, const float* mu_b, const float* lv_b,
                        const void* alpha, int alpha_is_f64, const float* eps, int64_t rows, int L, int ld_z,
                        float* z_f32, __nv_bfloat16* z_hi, __nv_bfloat16* z_lo, float* mu_out, float* lv_out,
                        cudaStream_t stream);
int launch_loss_finalize(Ctx* ctx, double* acc, int64_t B, int S, int L, float beta, float* loss_out, int ring_size,
                         float* step, cudaStream_t stream);
// The hyper-parameters of an Adam launch: the device record `dev` (read when the kernel runs), or the record `val`
// passed by value when dev == nullptr
struct HpArg {
  const rvae_hparams* dev;
  rvae_hparams val;
};
HpArg hp_value(double lr, double beta1, double beta2, double eps, double weight_decay);   // a constant record
inline HpArg hp_device(const rvae_hparams* dev) { HpArg a = hp_value(0.0, 0.0, 0.0, 0.0, 0.0); a.dev = dev; return a; }
int launch_adam(Ctx* ctx, float* p, float* g, float* m, float* v, int64_t n, double lr, double beta1, double beta2,
                double eps, double weight_decay, float grad_scale, const float* step, __nv_bfloat16* shadow_hi,
                __nv_bfloat16* shadow_lo, int zero_grads, cudaStream_t stream);
int launch_adam2(Ctx* ctx, float* p, float* g, float* m, float* v, int64_t n, int64_t off_b, int64_t n_b,
                 const HpArg& hp, float grad_scale, const float* coef, float* step, int step_bias, unsigned int* ticket,
                 __nv_bfloat16* shadow_hi, __nv_bfloat16* shadow_lo, int zero_grads, cudaStream_t stream);
// Gradient norm for clipping (grad_norm_kernel): the last block of a launch with `ticket` set sums parts[0, n_parts)
struct NormFinalize {
  const double* parts;
  int n_parts;
  unsigned int* ticket;   // nullptr: the launch only writes its partials
  const float* step;      // ring slot = *step mod ring_size (nullptr: slot 0)
  float* norm_out;        // nullptr: not reported
  int ring_size;
  const double* max_norm; // nullptr: no clipping factor
  float* coef_out;
};
int grad_norm_blocks(const Ctx* ctx, int64_t n);   // the fixed grid of a launch over n elements
int launch_grad_norm(Ctx* ctx, const float* g, int64_t n, int64_t off_b, int64_t n_b, double* part,
                     const NormFinalize& f, cudaStream_t stream);
int launch_hparams_eval(Ctx* ctx, const rvae_hparams* hp, const int64_t* k, int n, double* lr_out, float* beta_out,
                        cudaStream_t stream);
int launch_step_inc(Ctx* ctx, float* step, cudaStream_t stream);
// TensorBoard parameter histograms (rvae_param_histogram): record layout and size in include/rvae_b200.h
size_t param_histogram_bytes(int n_segs, int n_edges);
int launch_param_histogram(Ctx* ctx, const float* params, const int64_t* seg_offsets, const int64_t* seg_lengths,
                           int n_segs, const double* edges, int n_edges, void* record, cudaStream_t stream);
// the same over segments of seg_rows[s] rows of seg_cols[s] values at row pitch seg_pitch[s] (host arrays)
int launch_param_histogram_rows(Ctx* ctx, const float* params, const int64_t* seg_offsets, const int64_t* seg_rows,
                                const int64_t* seg_cols, const int64_t* seg_pitch, int n_segs, const double* edges,
                                int n_edges, void* record, cudaStream_t stream);

// Peer-memory all-reduce (elementwise.cu): symmetric buffers of all ranks as mapped in THIS process.
constexpr int kP2PMaxWorld = 8;
constexpr int kP2PMaxBuckets = 8;
constexpr int kP2PMaxCtas = 64;
constexpr int kP2PFlagStride = 32;            // one 128-byte line per flag: no false sharing between CTAs / ranks
constexpr size_t kP2PFlagBytes = 1024 * 1024;  // flags [bucket][cta][src rank] + epochs + tickets, at the start of the allocation
struct P2PArgs {
  float* data[kP2PMaxWorld];       // gradient buffer of rank p (peer-mapped; [rank] is local)
  float* mc_data;                  // NVLS multicast mapping of the same buffer (all ranks at once), nullptr = none:
                                   // multimem.ld_reduce sums a location over all ranks inside the switch, multimem.st
                                   // writes it to all ranks (rvae_dp_sym_adopt)
  uint32_t* flags[kP2PMaxWorld];   // flag area of rank p
  uint32_t* epoch;                 // local: [kP2PMaxBuckets]
  unsigned int* ticket;            // local: [kP2PMaxBuckets]
  uint32_t* status;                // local: 0 = healthy; else the first barrier timeout (bit 31 | peer << 8 | bucket << 4 | phase)
  long long timeout_cycles;        // SM clocks a barrier waits for a peer before it gives up (minutes, RVAE_P2P_TIMEOUT_S)
  int rank, world;
  int mode;                        // barrier flavour (experiments: RVAE_P2P_MODE)
};
struct P2PSegs {   // a bucket = concatenation of up to three segments of the flat gradient buffer (float elements)
  int64_t off[3];
  int64_t n[3];
};
int launch_allreduce_p2p(Ctx* ctx, const P2PArgs& a, const P2PSegs& sg, int bucket, int ctas, cudaStream_t stream);
// loss = acc[0]*inv_rec + kl_scale*acc[1] -> loss_out[step mod ring_size]; acc cleared; *step += 1
//   hp != nullptr: kl_scale = -0.5 * beta(k) / kl_bl instead, beta(k) from the record at k = *step
struct LossFinalize {
  double* acc;
  double inv_rec, kl_scale;
  float* loss_out;
  int ring_size;
  float* step;
  int inc_step;  // 0: the step counter is advanced elsewhere (by the last Adam launch of the step)
  const rvae_hparams* hp;
  double kl_bl;  // B * L of the loss normalisation
};
// KL gradient scale of the latent backward: c, or (float)(beta(k) / bl) with beta(k) from the record at k = *step
struct KlGrad {
  const rvae_hparams* hp;
  const float* step;
  double bl;
  float c;
  int early;  // the record and the counter are final before the kernel starts: read them before griddepcontrol.wait
};
inline KlGrad kl_grad_value(float c) { return KlGrad{nullptr, nullptr, 0.0, c, 0}; }
LossFinalize make_loss_finalize(double* acc, int64_t B, int S, int L, float beta, float* loss_out, int ring_size,
                                float* step);
int launch_loss_finalize_prepared(Ctx* ctx, const LossFinalize& f, cudaStream_t stream);
int launch_latent_bwd(Ctx* ctx, float* dz, const float* eps, const float* lv, const float* mu, const float* g_mu_ext,
                      const float* g_lv_ext, const KlGrad& kl, int64_t M, int L, __nv_bfloat16* dml_hi,
                      __nv_bfloat16* dml_lo, float* bias_grad, int clear_dz, const LossFinalize* fin,
                      cudaStream_t stream);

}  // namespace rvae
