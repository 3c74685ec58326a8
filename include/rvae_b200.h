/*
 * librvae_b200 - C ABI of the B200-native hot path for the rawaudiovae frame-level VAE.
 *
 * The reference (kelseyicotton/rawaudiovae_kelsey) is pure Python/PyTorch and has no FFI of its own; each entry
 * point below names the reference call site (file:line under the reference repo) whose work it replaces. The
 * binding a maintainer of the reference would add is a ctypes stub - see INTEGRATION.md.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in _host; the caller (PyTorch) owns every buffer,
 *     the library never allocates device memory;
 *   - `stream` is a cudaStream_t passed as void*; every call is asynchronous on it and CUDA-graph capturable;
 *   - return value 0 = ok; non-zero = error code (1 invalid argument, 2 unsupported shape, 3 driver, 4 state,
 *     1000 + cudaError_t); rvae_last_error() returns a thread-local description;
 *   - activations are row-major [frames, features]; weights are row-major [out_features, in_features] exactly
 *     as torch.nn.Linear stores them (rawvae/model.py:13-17);
 *   - bf16 planes: a tensor `t` is carried as t_hi = bf16(t) and, in fp32-emulation mode, t_lo = bf16(t - t_hi).
 *     Passing NULL for every *_lo pointer selects bf16 mode;
 *   - shapes: a plan (rvae_plan_create) accepts any positive segment_length S, n_units H and latent_dim L. It computes
 *     at Sp, Hp, Lp = the dims rounded up to multiples of 64 (rvae_param_layout_padded), with exact zeros in every
 *     padded row, column and bias, and normalises the loss by the true dims; caller tensors keep their true shapes.
 *     Dims that are multiples of 64 have no padding. The single-GEMM entry points (rvae_linear_act_fwd ..
 *     rvae_wgrad) need their GEMM dims to be multiples of 64.
 */
#ifndef RVAE_B200_H
#define RVAE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RVAE_ABI_VERSION 5

typedef struct rvae_ctx rvae_ctx;   /* per-device context (SM count, launch counter) */
typedef struct rvae_plan rvae_plan; /* a bound training / inference step for fixed shapes and buffers */

/* activation codes for rvae_linear_act_fwd */
#define RVAE_ACT_NONE 0
#define RVAE_ACT_RELU 1
#define RVAE_ACT_TANH 2        /* accurate tanhf */
#define RVAE_ACT_TANH_APPROX 3 /* tanh.approx.f32 (bf16 mode) */

/* precision modes of a plan */
#define RVAE_PRECISION_BF16 0 /* bf16 operands, fp32 accumulate */
#define RVAE_PRECISION_FP32 1 /* split-bf16 (hi+lo) operands, 3 tensor-core passes, ~2^-16 relative */

int rvae_abi_version(void);
/* 1 when the library was built with -DRVAE_EXPERIMENTS=1 (measured-and-rejected paths: chained forward launch,
 * fused latent epilogue, GEMM debug modes); 0 for the default build, which contains none of them. */
int rvae_build_experiments(void);
const char* rvae_last_error(void);

int rvae_ctx_create(int device, rvae_ctx** out);
void rvae_ctx_destroy(rvae_ctx* ctx);
int rvae_ctx_num_sms(const rvae_ctx* ctx);
/* number of kernels launched through this context so far (bench.py "gpu_launches") */
uint64_t rvae_ctx_launch_count(const rvae_ctx* ctx);

/* ---------------------------------------------------------------------------------------------------------
 * Data parallelism (no counterpart in the reference, which is single-process: SURVEY.md 2b). One process per GPU;
 * the host side (torch.distributed) only carries the 128-byte NCCL id from rank 0 to the others. Once a context
 * has a communicator, rvae_plan_train_step all-reduces every gradient bucket (SUM, fp32) on a communication stream
 * as soon as the backward stage that completes it is done, overlapped with the remaining stages, and each bucket's
 * Adam launch waits for its reduced gradient. Use rvae_plan_set_global_batch so that the sum is the gradient of the
 * concatenated batch. libnccl_path: the libnccl.so.2 to dlopen (NULL = the default search path).
 * ------------------------------------------------------------------------------------------------------- */
int rvae_dp_unique_id(rvae_ctx* ctx, const char* libnccl_path, void* out128);
int rvae_dp_init(rvae_ctx* ctx, const char* libnccl_path, const void* id128, int rank, int world);
int rvae_dp_world(const rvae_ctx* ctx);
/* Peer-memory all-reduce (our own kernel instead of NCCL): rvae_dp_sym_alloc creates this rank's symmetric
 * allocation (the library owns it - the one exception to "the caller owns every buffer", because it must be
 * IPC-exportable) and returns the device pointer of its data area plus a 64-byte CUDA IPC handle; the host side
 * gathers the handles of all ranks (torch.distributed) and passes them, indexed by rank, to rvae_dp_sym_open, which
 * maps every peer's allocation. A plan whose bufs.grads lies in the data area then all-reduces its gradient
 * buckets with a two-shot reduce-scatter / all-gather kernel that reads and writes NVLink peer memory directly
 * (csrc/elementwise.cu "Gradient all-reduce over NVLink peer memory"); other gradients fall back to NCCL. */
int rvae_dp_sym_alloc(rvae_ctx* ctx, size_t data_bytes, void** data_ptr, void* ipc_handle64);
/* In-place SUM all-reduce of `count` floats (a multiple of 4) at ptr: the peer-memory kernel when ptr lies in the
 * symmetric data area (bucket = 0..7 selects the flag set; concurrent all-reduces must use different buckets), NCCL
 * otherwise. What rvae_plan_train_step issues per gradient bucket. */
int rvae_dp_allreduce(rvae_ctx* ctx, float* ptr, int64_t count, int bucket, void* stream);
int rvae_dp_sym_open(rvae_ctx* ctx, const void* handles, int rank, int world);
/* The same set-up from a symmetric allocation the CALLER made and mapped (e.g. torch.distributed._symmetric_memory):
 * peer_bases[p] = this process' mapping of rank p's buffer ([rank] = the local one), each rvae_dp_sym_flag_bytes() of
 * zeroed flag area followed by data_bytes of gradient buffer; multicast_base = the NVLS multicast mapping of the same
 * allocation (NULL = none). With a multicast mapping the all-reduce kernel reduces each slice INSIDE THE NVSWITCH
 * (multimem.ld_reduce) and multicasts the sum to all ranks (multimem.st): 1 / W of the bucket crosses a rank's links
 * once per direction instead of (W - 1) / W peer reads + (W - 1) / W posted writes. The caller keeps the allocation
 * alive and unmaps it; RVAE_NVLS=0 ignores the multicast mapping. */
size_t rvae_dp_sym_flag_bytes(void);
int rvae_dp_sym_adopt(rvae_ctx* ctx, const void* const* peer_bases, void* multicast_base, size_t data_bytes, int rank,
                      int world);
int rvae_dp_uses_multicast(const rvae_ctx* ctx);
/* Health of the peer-memory all-reduce. Its barriers wait for a slower peer for RVAE_P2P_TIMEOUT_S seconds (default
 * 600) and never trap; the first wait that gives up records bit 31 | peer << 8 | flag set << 4 | phase here, and every
 * later wait falls through at once, so the process stays alive and the host can report the failure. 0 = healthy.
 * Synchronous 4-byte read: call it where the host synchronises anyway (loss read-back, checkpoints). */
int rvae_dp_status(rvae_ctx* ctx, unsigned int* status);

/* ---------------------------------------------------------------------------------------------------------
 * Framing and resynthesis (rawvae/dataset.py)
 * ------------------------------------------------------------------------------------------------------- */

/* Frame f of the batch = audio_pad[idx*hop : idx*hop + S] with idx = frame_idx[f] (if non-NULL) else
 * first_frame + f; samples at or beyond n_samples read as 0 (the reference zero-pads: dataset.py:102-104,
 * 141-143, 61-63). Replaces AudioDataset.__getitem__ (dataset.py:108-118), TestDataset.__getitem__ (:147-157),
 * IterableAudioDataset.process_data's slicing loop (:68-75) and default_collate's stack.
 * audio is float32 (audio_is_i16 = 0) or int16 PCM scaled by 1/32768 (audio_is_i16 = 1). Any of the three
 * outputs may be NULL (at least one of out_hi / out_f32 required). Outputs are [n_frames, S], any S > 0. */
int rvae_frame_gather(rvae_ctx* ctx, const void* audio, int audio_is_i16, int64_t n_samples,
                      const int64_t* frame_idx, int64_t first_frame, int64_t n_frames, int hop, int S,
                      void* out_hi, void* out_lo, float* out_f32, void* stream);

/* Overlap-add resynthesis: out[t - t_begin] = mean over the frames covering t of frames[i, t - i*hop], for
 * t in [t_begin, t_begin + n_out) (t_begin > 0: one window of a long signal that is resynthesised batch by batch).
 * With hop == S this is frames.view(-1) (train_iterable.py:246, tutorial.ipynb:543). frames is fp32 [n_frames, S]. */
int rvae_overlap_add(rvae_ctx* ctx, const float* frames, int64_t n_frames, int S, int hop, float* out,
                     int64_t t_begin, int64_t n_out, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Elementwise pieces of the model / loss / optimizer
 * ------------------------------------------------------------------------------------------------------- */

/* eps ~ N(0,1), Philox4x32-10 + Box-Muller keyed by (seed, offset). Replaces torch.randn_like (model.py:25).
 * out[i] is element (elem_base + i) of the logical noise tensor of that (seed, offset): a rank that owns rows
 * [r0, r1) of a global [B, L] batch passes elem_base = r0 * L (any elem_base >= 0) and draws exactly the values a
 * single process would have drawn for those rows. */
int rvae_randn(rvae_ctx* ctx, float* out, int64_t n, uint64_t seed, uint64_t offset, int64_t elem_base, void* stream);

/* Latent interpolation of the inference pattern (tutorial.ipynb:496-510, 905-932), any L > 0: per row r,
 *   mu = (1 - alpha[r]) mu_a + alpha[r] mu_b, logvar likewise, z = mu + eps * exp(logvar / 2)   (eps NULL = 0).
 * alpha: `rows` floats, or doubles when alpha_is_f64 (the notebook's interp1d output); the lerp is then carried out
 * in double. Outputs (each may be NULL, not all): z, mu_out, logvar_out, fp32 [rows, L]. */
int rvae_lerp_reparameterize(rvae_ctx* ctx, const float* mu_a, const float* logvar_a, const float* mu_b,
                             const float* logvar_b, const void* alpha, int alpha_is_f64, const float* eps,
                             int64_t rows, int L, float* z, float* mu_out, float* logvar_out, void* stream);

/* fp32 -> bf16 planes (hi, optional lo). Used for weight shadows and fp32 inputs. */
int rvae_split_bf16(rvae_ctx* ctx, const float* src, int64_t n, void* hi, void* lo, void* stream);

/* z = mu + eps * exp(0.5 * logvar) (model.py:23-26), fp32. */
int rvae_reparameterize(rvae_ctx* ctx, const float* mu, const float* logvar, const float* eps, int64_t n, float* z,
                        void* stream);

/* loss = mean((xhat-x)^2) + beta * (-0.5) * mean(1 + logvar - mu^2 - exp(logvar)) (model.py:38-46).
 * acc is a 2-double scratch accumulator; loss_out a device float. */
int rvae_loss_fwd(rvae_ctx* ctx, const float* xhat, const float* x, const float* mu, const float* logvar,
                  int64_t B, int S, int L, float beta, double* acc, float* loss_out, void* stream);

/* Per-frame loss of held-out audio: what loss_function (rawvae/model.py:38-46) measures, one value per frame instead
 * of one batch mean - the score of the reference's test_dataset (train.py:153-155, train_iterable.py:170-172), which
 * the reference only resynthesises. For f < rows, with frame f = audio[(first_frame + f) * hop + s], s < S (the
 * framing rule of rvae_frame_gather: float32, or int16 * (1/32768); zeros at and beyond n_samples):
 *   rec_out[f] = (1/S) sum_s (xhat[f,s] - x[f,s])^2
 *   kl_out[f]  = -(0.5/L) sum_l (1 + logvar[f,l] - mu[f,l]^2 - exp(logvar[f,l]))        (accurate expf)
 * so that mean_f(rec_out[f] + beta * kl_out[f]) is loss_function(xhat, x, mu, logvar, beta, S). xhat is read at row
 * pitch ld_xhat >= S, mu and logvar at ld_lat >= L: a plan's rvae_plan_xhat / rvae_plan_mu / rvae_plan_logvar can be
 * passed directly (pitches Sp, Lp). x is read from the audio itself, exact, never rounded to bf16. Each frame is
 * reduced by one fixed group of threads in a fixed order (fp64 sums, no atomics): repeated calls are bitwise equal.
 * Returns 1 for null pointers, rows, S or L <= 0, ld_xhat < S, ld_lat < L, hop <= 0, n_samples < 0 or
 * first_frame < 0 (checked before ctx is used). */
int rvae_frame_loss(rvae_ctx* ctx, const float* xhat, int ld_xhat, const float* mu, const float* logvar, int ld_lat,
                    int64_t rows, int S, int L, const void* audio, int audio_is_i16, int64_t n_samples,
                    int64_t first_frame, int hop, float* rec_out, float* kl_out, void* stream);

/* Gradients of that loss w.r.t. xhat, mu, logvar, times the upstream scalar *grad_out (NULL = 1). */
int rvae_loss_bwd(rvae_ctx* ctx, const float* xhat, const float* x, const float* mu, const float* logvar,
                  int64_t B, int S, int L, float beta, const float* grad_out, float* g_xhat, float* g_mu,
                  float* g_logvar, void* stream);

/* da4 = g_xhat * (1 - xhat^2) as bf16 planes (tanh backward, autograd's TanhBackward for model.py:30). */
int rvae_tanh_bwd(rvae_ctx* ctx, const float* g_xhat, const float* xhat, int64_t n, void* da_hi, void* da_lo,
                  void* stream);

/* out[n] (+)= sum over rows of a bf16 [M, N] matrix (hi + optional lo): bias gradients (AddmmBackward's sum). */
int rvae_colsum(rvae_ctx* ctx, const void* hi, const void* lo, int64_t M, int N, int ld, float* out, int accumulate,
                void* stream);

/* *step += 1 (device scalar), then rvae_adam_step reads it. */
int rvae_step_inc(rvae_ctx* ctx, float* step, void* stream);

/* Fused Adam over a flat fp32 buffer (torch.optim.Adam semantics; train.py:163,193; train_iterable.py:180,210):
 *   g' = g*grad_scale (+ weight_decay*p); m += (1-b1)(g'-m); v = b2 v + (1-b2) g'^2;
 *   p -= lr/(1-b1^t) * m / (sqrt(v)/sqrt(1-b2^t) + eps),  t = *step.
 * lr, beta1, beta2, eps, weight_decay are DOUBLES - what torch.optim.Adam holds - and every scalar of the update is
 * derived from them as torch derives it: 1 - beta and the bias corrections 1 - beta^t in double, then rounded to
 * fp32 (a float beta would make (1 - b2) 1.3e-5 off). The arithmetic on the tensors is fp32.
 * Optionally re-emits the bf16 shadow planes of p (what the GEMMs read). */
int rvae_adam_step(rvae_ctx* ctx, float* p, const float* g, float* m, float* v, int64_t n, double lr, double beta1,
                   double beta2, double eps, double weight_decay, float grad_scale, const float* step, void* shadow_hi,
                   void* shadow_lo, void* stream);

/* TensorBoard parameter histograms: replaces `for name, param in model.named_parameters(): writer.add_histogram(name,
 * param, step)` (train_iterable.py:216-217, train.py:203-204), which copies every parameter to the host and sorts it.
 * One launch bins n_segs segments of the fp32 buffer `params` (segment s = params[seg_offsets_host[s] ..
 * + seg_lengths_host[s]), lengths >= 1) against edges_host (n_edges strictly increasing finite doubles, e.g.
 * SummaryWriter.default_bins), with the semantics of torch.utils.tensorboard.summary.make_histogram on the values
 * converted to float64: bin i counts [edges[i], edges[i+1]), the last bin is closed, values outside
 * [edges[0], edges[n_edges-1]] and NaN are not counted; num counts every value; min / max are NaN if any value is
 * NaN. Counts, min, max and num are exact; sum and sum of squares are fp64, reduced in a fixed order (bitwise
 * reproducible, not numpy's summation order).
 * `record` (device, 16-byte aligned, rvae_param_histogram_bytes() bytes) receives, with nb = n_edges - 1 and
 * ns = n_segs, at these byte offsets:
 *   0                     int32  counts[ns][nb]
 *   A = align8(4 ns nb)   double sum[ns];  A + 8 ns: double sum_squares[ns];  A + 16 ns: int64 num[ns];
 *   A + 24 ns             float  min[ns];  A + 28 ns: float max[ns];
 * i.e. A + 32 ns bytes of results, followed by the kernel's scratch (rewritten by every call). */
#define RVAE_HIST_MAX_SEGS 16
#define RVAE_HIST_MAX_EDGES 2048
size_t rvae_param_histogram_bytes(int n_segs, int n_edges); /* 0 for unsupported sizes */
int rvae_param_histogram(rvae_ctx* ctx, const float* params, const int64_t* seg_offsets_host,
                         const int64_t* seg_lengths_host, int n_segs, const double* edges_host, int n_edges,
                         void* record, void* stream);
/* The same over strided segments: segment s = seg_rows_host[s] rows of seg_cols_host[s] values, row r starting at
 * params[seg_offsets_host[s] + r * seg_pitch_host[s]] (seg_pitch >= seg_cols): a parameter of a padded plan inside its
 * padded block, e.g. fc1.weight = H rows of S values at pitch Sp. num = rows * cols. rvae_param_histogram is the
 * one-row case. */
int rvae_param_histogram_rows(rvae_ctx* ctx, const float* params, const int64_t* seg_offsets_host,
                              const int64_t* seg_rows_host, const int64_t* seg_cols_host, const int64_t* seg_pitch_host,
                              int n_segs, const double* edges_host, int n_edges, void* record, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * tcgen05 GEMMs with fused epilogues (rawvae/model.py:19-35 forward; autograd backward of the same)
 * ------------------------------------------------------------------------------------------------------- */

/* y = act(x W^T + b): x [M,K], W [N,K], b [N] (NULL = none). Outputs: y_hi/y_lo bf16 planes and/or y_f32,
 * all [M,N]. Replaces F.relu(self.fc1(x)) (model.py:20), F.relu(self.fc3(z)) (:29), F.tanh(self.fc4(h3)) (:30). */
int rvae_linear_act_fwd(rvae_ctx* ctx, const void* x_hi, const void* x_lo, const void* w_hi, const void* w_lo,
                        const float* bias, int M, int N, int K, int act, void* y_hi, void* y_lo, float* y_f32,
                        void* stream);

/* Encoder head + reparameterisation + KL (model.py:21,23-26,45): W2 = [fc21.weight; fc22.weight] stacked [2L,K],
 * b2 = [fc21.bias; fc22.bias] [2L]; mu, logvar fp32 [M,L]; eps fp32 [M,L] (NULL = 0);
 * z = mu + eps*exp(logvar/2) as bf16 planes (optional); kl_acc[0] += sum(1+logvar-mu^2-exp(logvar)) (optional). */
int rvae_encode_head_fwd(rvae_ctx* ctx, const void* h_hi, const void* h_lo, const void* w2_hi, const void* w2_lo,
                         const float* b2, int M, int L, int K, const float* eps, float* mu, float* logvar,
                         void* z_hi, void* z_lo, double* kl_acc, void* stream);

/* Decoder output + reconstruction loss + its gradient (model.py:30,39): xhat = tanh(h3 W4^T + b4) [M,S] (fp32,
 * optional); mse_acc[0] += sum((xhat-x)^2); da4 = grad_scale*(xhat-x)*(1-xhat^2) as bf16 planes (optional),
 * grad_scale = 2/(B*S). x is given as bf16 planes. bias_grad (optional, fp32 [S]) += column sums of da4 = db4. */
int rvae_out_tanh_mse_fwd(rvae_ctx* ctx, const void* h_hi, const void* h_lo, const void* w4_hi, const void* w4_lo,
                          const float* b4, int M, int S, int K, const void* x_hi, const void* x_lo, int tanh_approx,
                          float* xhat, void* da_hi, void* da_lo, float grad_scale, double* mse_acc, float* bias_grad,
                          void* stream);

/* dX = (dY W) * [mask > 0]: dY [M,Kd], W [Kd,N] row-major (the Linear weight [out=Kd, in=N]), mask bf16 [M,N]
 * (NULL = no mask). AddmmBackward dgrad + ReluBackward (threshold_backward) for fc4->h3 and fc21/fc22->h1.
 * bias_grad (optional, fp32 [N]) += column sums of dX: the bias gradient of the layer that produced `mask`. */
int rvae_dgrad_relu(rvae_ctx* ctx, const void* dy_hi, const void* dy_lo, const void* w_hi, const void* w_lo, int M,
                    int N, int Kd, const void* mask, void* dx_hi, void* dx_lo, float* bias_grad, void* stream);

/* Latent backward: dz = da3 W3 (W3 [H,L]; split-K tcgen05 GEMM reduce-added into dz_scratch, fp32 [M,L]), then
 *   sigma = exp(logvar/2);  d_ml[:, :L] = dz + g_mu;  d_ml[:, L:] = dz*eps*sigma/2 + g_logvar   (bf16 planes [M, 2L])
 * with g_mu = kl_grad_scale*mu, g_logvar = kl_grad_scale*(sigma^2-1)/2 (the KL gradient, kl_grad_scale = beta/(B L))
 * when g_mu_ext / g_logvar_ext are NULL, else those external upstream gradients (mu may then be NULL).
 * Backward of reparameterize (model.py:24-26) merged with the KL gradient (model.py:45).
 * bias_grad (optional, fp32 [2L]) += column sums of d_ml = [db21; db22]. */
int rvae_dgrad_latent(rvae_ctx* ctx, const void* da3_hi, const void* da3_lo, const void* w3_hi, const void* w3_lo,
                      int M, int L, int H, const float* eps, const float* logvar, const float* mu,
                      const float* g_mu_ext, const float* g_logvar_ext, float kl_grad_scale, float* dz_scratch,
                      void* dml_hi, void* dml_lo, float* bias_grad, void* stream);

/* dW (+)= dY^T X: dY [B,M], X [B,N], dW fp32 [M,N]. accumulate = 0 overwrites (single split), 1 adds (red.add;
 * dW must hold the running sum, e.g. zeros). k_splits = 0 lets the library choose. AddmmBackward wgrad. */
int rvae_wgrad(rvae_ctx* ctx, const void* dy_hi, const void* dy_lo, const void* x_hi, const void* x_lo, int B, int M,
               int N, float* dW, int accumulate, int k_splits, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Plan: the whole step (forward + loss + backward + Adam) for fixed shapes and bound buffers, issued from C so
 * one call enqueues every kernel (train.py:184-193, train_iterable.py:200-210).
 * ------------------------------------------------------------------------------------------------------- */

/* Flat parameter layout (fp32 elements), used for params / grads / exp_avg / exp_avg_sq / bf16 shadows:
 *   W1 [H,S] | W2 = [fc21.weight; fc22.weight] [2L,H] | W3 [H,L] | W4 [S,H] | b1 [H] | b2 [2L] | b3 [H] | b4 [S] */
typedef struct rvae_layout {
  int64_t w1, w2, w3, w4, b1, b2, b3, b4; /* element offsets */
  int64_t total;                          /* total elements (5 772 800 for default.ini) */
} rvae_layout;

int rvae_param_layout(int S, int H, int L, rvae_layout* out);   /* S, H, L multiples of 64 */

/* Layout of the padded blocks a plan of ANY positive dims uses: *Sp, *Hp, *Lp = S, H, L rounded up to multiples of 64;
 * W1 [Hp,Sp] | W2 [2Lp,Hp] | W3 [Hp,Lp] | W4 [Sp,Hp] | b1 [Hp] | b2 [2Lp] | b3 [Hp] | b4 [Sp], i.e.
 * rvae_param_layout(Sp, Hp, Lp). A parameter is the top-left corner of its block: fc1.weight = W1[:H, :S],
 * fc21 = rows [0, L) of W2 and fc22 = rows [Lp, Lp + L), fc21.bias = b2[0:L], fc22.bias = b2[Lp:Lp+L], ... Everything
 * outside those corners is zero and stays zero through training (gradients and Adam moments included). For multiples
 * of 64 it equals rvae_param_layout. */
int rvae_param_layout_padded(int S, int H, int L, rvae_layout* out, int* Sp, int* Hp, int* Lp);

typedef struct rvae_plan_buffers {
  float* params;    /* [total] fp32 master weights */
  float* grads;     /* [total] fp32 gradients (written every step) */
  float* exp_avg;   /* [total] */
  float* exp_avg_sq;/* [total] */
  float* step;      /* device scalar, Adam step count t as fp32 (torch state format) */
  void* shadow_hi;  /* [total] bf16 */
  void* shadow_lo;  /* [total] bf16, fp32 mode only (else NULL) */
  void* workspace;  /* rvae_plan_workspace_bytes() bytes, 256-byte aligned */
} rvae_plan_buffers;

int rvae_plan_create(rvae_ctx* ctx, int S, int H, int L, int max_batch, int precision, rvae_plan** out);
void rvae_plan_destroy(rvae_plan* plan);
size_t rvae_plan_workspace_bytes(const rvae_plan* plan);
int rvae_plan_bind(rvae_plan* plan, const rvae_plan_buffers* bufs);

/* Refresh the bf16 shadow planes from the fp32 master weights (after load_state_dict / manual edits). */
int rvae_plan_sync_shadow(rvae_plan* plan, void* stream);

/* Load a batch into the plan's input buffer: `count` frames gathered from a wav buffer (see rvae_frame_gather)
 * into rows [row_offset, row_offset + count). row_offset = 0 starts a new batch; a batch that straddles several
 * files (train_iterable.py's stream) is appended run by run; the batch size becomes row_offset + count ... */
int rvae_plan_load_frames(rvae_plan* plan, const void* audio, int audio_is_i16, int64_t n_samples,
                          const int64_t* frame_idx, int64_t first_frame, int count, int hop, int row_offset,
                          void* stream);
/* ... or an fp32 [batch, S] matrix already on the device (true S; a padded plan pads it on the way in). */
int rvae_plan_load_batch(rvae_plan* plan, const float* x, int batch, void* stream);
/* ... or a RUN of `count` consecutive frames (first_frame, first_frame + 1, ...: the stream of
 * IterableAudioDataset.process_data, rawvae/dataset.py:61-69, TestDataset with hop = S, tutorial.ipynb's inference
 * loop) read IN PLACE: the run is one contiguous span of (count - 1) * hop + S samples, which is converted once
 * (fp32 / PCM16 -> bf16) into the plan's input buffer; fc1's A operand, the MSE side input and the fc1 weight
 * gradient's operand then read frame i at row pitch `hop` through overlapping-row TMA tensor maps - the [count, S]
 * frame matrix is never materialised and every sample is touched once instead of S / hop times. Results are
 * bit-identical to rvae_plan_load_frames. first_frame_dev (device int64, may be NULL) overrides first_frame and is
 * read by the kernel, so a captured CUDA graph follows the stream. Needs hop % 8 == 0, hop <= S and S % 8 == 0; with
 * S not a multiple of 64 (columns S..Sp read as zeros through the tensor maps) also bf16 mode
 * (rvae_plan_span_supported). */
int rvae_plan_span_supported(const rvae_plan* plan, int count, int hop);
int rvae_plan_load_span(rvae_plan* plan, const void* audio, int audio_is_i16, int64_t n_samples,
                        const int64_t* first_frame_dev, int64_t first_frame, int count, int hop, void* stream);

/* eps for the loaded batch: copy from a caller tensor (parity runs) or generate with Philox (seed, offset).
 * add_step != 0 adds the device-side Adam step counter (*bufs.step) to the offset inside the kernel, so a captured
 * CUDA graph draws fresh noise on every replay. */
int rvae_plan_set_eps(rvae_plan* plan, const float* eps, void* stream);
int rvae_plan_gen_eps(rvae_plan* plan, uint64_t seed, uint64_t offset, int add_step, void* stream);
/* Data parallelism: this rank's shard starts at row `first_global_row` of the global batch. The noise of
 * rvae_plan_gen_eps / rvae_plan_prefetch_frames is then drawn from Philox counters first_global_row * L onwards, so
 * with the SAME seed on every rank the shards' noise is disjoint and equal to the single-process draw. */
int rvae_plan_set_noise_rows(rvae_plan* plan, int64_t first_global_row);

/* Redirect the fp32 results of the next forward calls into caller tensors ([batch,L], [batch,L], [batch,S]);
 * NULL = keep them in the workspace. Used by the autograd wrapper so returned tensors outlive the step. */
int rvae_plan_set_outputs(rvae_plan* plan, float* mu, float* logvar, float* xhat);

/* Data parallelism: make this plan's rvae_plan_train_step all-reduce its gradient buckets over the context's
 * communicator (rvae_dp_init). Off by default, so other plans of the same device stay single-process. */
int rvae_plan_enable_dp(rvae_plan* plan, int on);
/* Data parallelism: normalise the loss (and therefore its gradients) by the GLOBAL batch size instead of the
 * local one, so that a plain SUM all-reduce over ranks yields exactly the single-process gradient of the
 * concatenated batch, also when shards are unequal. 0 (default) = use the local batch size. */
int rvae_plan_set_global_batch(rvae_plan* plan, int64_t global_batch);

/* Forward. fused_loss = 1: the epilogues also accumulate the MSE / KL sums and emit the loss gradients
 * (da4, g_mu, g_logvar) so that rvae_plan_backward can run without a separate loss kernel
 * (model.py:32-35 + :38-46 + the head of loss.backward()). fused_loss = 0: plain model(x) - xhat, mu, logvar
 * (+ what an external backward needs). want_xhat: materialise xhat fp32 (always done when fused_loss = 0). */
int rvae_plan_forward(rvae_plan* plan, float kl_beta, int fused_loss, int want_xhat, void* stream);
/* Backward from external upstream gradients (autograd path): g_xhat [batch,S], g_mu, g_logvar [batch,L] fp32,
 * xhat, logvar = the forward's outputs. Runs tanh backward then all four stages. */
int rvae_plan_backward_external(rvae_plan* plan, const float* g_xhat, const float* xhat, const float* g_mu,
                                const float* g_logvar, const float* logvar, void* stream);
/* Backward stage s = 0..3 (fc4 | fc3 | fc21+fc22 | fc1 WEIGHT gradients complete after stage s - the allreduce
 * buckets, in backward-completion order; the bias block is complete after stage 2); stage -1 runs all four.
 * Within a stage the dgrad GEMM (the critical dependency chain) is issued before the weight-gradient GEMM, both on
 * `stream`. Gradients land in bufs.grads. */
int rvae_plan_backward(rvae_plan* plan, int stage, void* stream);
/* loss -> loss_out[t mod ring_size] (device floats, may be NULL; t = *step before the call), clears the loss sums,
 * *step += 1. ring_size = 1 writes *loss_out. The value is the mean loss over this rank's frames. */
int rvae_plan_finish_loss(rvae_plan* plan, float kl_beta, float* loss_out, int ring_size, void* stream);
/* Same, but without a kernel of its own: the finalisation is carried out by the latent backward kernel of the next
 * rvae_plan_backward stage 1 (or -1) of this plan, which MUST follow on the same stream before loss_out is read, the
 * next forward is issued or Adam runs. Saves one dependent launch per training step. */
int rvae_plan_finish_loss_deferred(rvae_plan* plan, float kl_beta, float* loss_out, int ring_size);
/* Input prefetch: describe the NEXT step's batch (same arguments as rvae_plan_load_frames with row_offset 0, plus
 * the rvae_plan_gen_eps arguments for its noise). The next rvae_plan_train_step gathers it into the plan's alternate
 * input buffers on a low-priority background stream while its own GEMMs run (the reference's DataLoader prefetches
 * the next batch the same way, on the host); rvae_plan_swap_prefetched then makes it current instead of
 * rvae_plan_load_frames + rvae_plan_gen_eps. rvae_plan_prefetched_batch: frames waiting in the alternate set (0 = none). */
int rvae_plan_prefetch_frames(rvae_plan* plan, const void* audio, int audio_is_i16, int64_t n_samples,
                              const int64_t* frame_idx, int64_t first_frame, int count, int hop, uint64_t seed,
                              uint64_t offset, int add_step);
/* The same for a run of consecutive frames read in place (see rvae_plan_load_span). */
int rvae_plan_prefetch_span(rvae_plan* plan, const void* audio, int audio_is_i16, int64_t n_samples,
                            const int64_t* first_frame_dev, int64_t first_frame, int count, int hop, uint64_t seed,
                            uint64_t offset, int add_step);
int rvae_plan_swap_prefetched(rvae_plan* plan);
int rvae_plan_prefetched_batch(const rvae_plan* plan);
/* Make `stream` wait for background work of earlier calls that a later call would otherwise join (the noise of
 * rvae_plan_gen_eps). Needed before a CUDA-graph capture starts: a captured stream must not wait on uncaptured work. */
int rvae_plan_join_background(rvae_plan* plan, void* stream);
/* Host-side bookkeeping for CUDA-graph replays: a replayed rvae_plan_train_step performed the prefetch on the device
 * without running this library's host code; tell the plan that `count` frames wait in the alternate input set
 * (as gathered rows, or as a sample span at pitch span_hop: rvae_plan_prefetch_span). */
int rvae_plan_note_prefetched(rvae_plan* plan, int count, int span_hop /* 0 = gathered rows, else the run's hop */);
/* Adam over the flat buffers (+ shadow refresh). grad_scale rescales the gradients (1 for SUM all-reduced,
 * globally normalised gradients). zero_grads != 0: the kernel also clears bufs.grads after consuming it - the
 * optimizer.zero_grad() of the next iteration (train.py:184) - which lets the next backward skip its memsets. */
int rvae_plan_adam(rvae_plan* plan, double lr, double beta1, double beta2, double eps, double weight_decay,
                   float grad_scale, int zero_grads, void* stream);
/* Adam restricted to the gradient buckets in bucket_mask (bit s = bucket s of rvae_plan_bucket): lets a caller update
 * a bucket as soon as its gradient (and, under data parallelism, its all-reduce) is complete. The caller orders the
 * launch after the backward stage that completes the bucket: that stage's dgrad GEMM reads the bucket's bf16 shadow. */
int rvae_plan_adam_buckets(rvae_plan* plan, unsigned bucket_mask, double lr, double beta1, double beta2, double eps,
                           double weight_decay, float grad_scale, int zero_grads, void* stream);
/* forward + loss + backward + Adam in one call (single-GPU training step). Adam runs per bucket on an internal
 * stream underneath the later backward stages; everything is joined back into `stream` before the call returns. */
int rvae_plan_train_step(rvae_plan* plan, float kl_beta, double lr, double beta1, double beta2, double eps,
                         double weight_decay, int zero_grads, float* loss_out, int ring_size, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Scheduled hyper-parameters. The reference trains at a fixed learning rate (torch.optim.Adam, train.py:163,193)
 * and a fixed KL weight (rawvae/model.py:45); this record adds a learning-rate warm-up and decay and a KL-weight
 * ramp. It lives in device memory and the kernels of a step read it when they run, so a CUDA graph captured around
 * rvae_plan_train_step_hp holds the record's ADDRESS: every replay follows the schedule at its own step, and any
 * rewrite of the record that is stream-ordered before the replay.
 *
 * k = the device step counter (bufs.step) when the step starts; Adam's bias correction keeps t = k + 1.
 * T = total_steps, W = warmup_steps. Learning rate:
 *   k < W:       lr * (k + 1) / W
 *   otherwise    D = max(T - W, 1), u = min(k - W, D) / D, and
 *                constant lr | linear lr_min + (lr - lr_min) * (1 - u) | cosine lr_min + (lr - lr_min) * 0.5 * (1 + cos(pi u))
 * KL weight, b0 = kl_beta_start, A = kl_anneal_steps, M = kl_cycles, R = kl_cycle_ratio:
 *   constant kl_beta | linear b0 + (kl_beta - b0) * min(1, k / A)
 *   cyclical C = ceil(T / M), tau = (k mod C) / C, b0 + (kl_beta - b0) * min(1, tau / R)
 * Everything is evaluated in fp64, operation by operation in the order written, without FMA contraction. cos(pi u)
 * is a fixed polynomial: the Taylor series of cos to x^22 at x = pi * min(u, 1 - u), negated for u > 0.5, evaluated
 * by Horner's rule. So a host mirror that repeats these operations (rawaudiovae_kelsey_b200/schedule.py) gets the
 * same doubles. lr(k) reaches Adam as a double; beta(k) is rounded to float, as the kl_beta argument of
 * rvae_plan_train_step is. A record of kind constant / constant with W = 0 gives every kernel exactly the scalars
 * rvae_plan_train_step gives it. */
#define RVAE_LR_CONSTANT 0
#define RVAE_LR_LINEAR 1
#define RVAE_LR_COSINE 2
#define RVAE_KL_CONSTANT 0
#define RVAE_KL_LINEAR 1
#define RVAE_KL_CYCLICAL 2

typedef struct rvae_hparams {
  double lr;               /*   0  peak learning rate */
  double beta1;            /*   8 */
  double beta2;            /*  16 */
  double eps;              /*  24 */
  double weight_decay;     /*  32 */
  double kl_beta;          /*  40  target KL weight */
  double lr_min;           /*  48 */
  double kl_beta_start;    /*  56 */
  double kl_cycle_ratio;   /*  64  R, in (0, 1] */
  int64_t total_steps;     /*  72  T, >= 1 for a linear / cosine lr or a cyclical KL weight */
  int64_t warmup_steps;    /*  80  W, >= 0 */
  int64_t kl_anneal_steps; /*  88  A, >= 1 for a linear KL weight */
  int64_t kl_cycles;       /*  96  M, >= 1 for a cyclical KL weight */
  int32_t lr_schedule;     /* 104  RVAE_LR_* */
  int32_t kl_anneal;       /* 108  RVAE_KL_* */
} rvae_hparams;            /* 112 bytes, 8-byte aligned */

#ifdef __cplusplus
#define RVAE_STATIC_ASSERT(c, m) static_assert(c, m)
#else
#define RVAE_STATIC_ASSERT(c, m) _Static_assert(c, m)
#endif
RVAE_STATIC_ASSERT(sizeof(rvae_hparams) == 112, "rvae_hparams: 112 bytes");
RVAE_STATIC_ASSERT(offsetof(rvae_hparams, kl_beta) == 40 && offsetof(rvae_hparams, kl_cycle_ratio) == 64,
                   "rvae_hparams: double fields");
RVAE_STATIC_ASSERT(offsetof(rvae_hparams, total_steps) == 72 && offsetof(rvae_hparams, kl_cycles) == 96,
                   "rvae_hparams: integer fields");
RVAE_STATIC_ASSERT(offsetof(rvae_hparams, lr_schedule) == 104 && offsetof(rvae_hparams, kl_anneal) == 108,
                   "rvae_hparams: kinds");

/* Validate a HOST copy of a record: 0 if it is usable, 1 for an unknown kind, W < 0, T < 1 with a linear / cosine
 * learning rate or a cyclical KL weight, A < 1 with a linear KL weight, M < 1 with a cyclical one, R outside (0, 1]
 * or a non-finite value. The device entries below cannot read the record without a synchronisation: check every
 * record before it is uploaded. */
int rvae_hparams_check(const rvae_hparams* host);
/* rvae_plan_train_step with every hyper-parameter read from the device record hp_dev at run time (same data-parallel
 * path, per-kernel timing mode and results for a constant record). Returns 1 for a null hp_dev or ring_size < 1
 * (before the plan is used), 2 for the experiments-only fused latent epilogue, which takes its KL scale from the host. */
int rvae_plan_train_step_hp(rvae_plan* plan, const rvae_hparams* hp_dev, int zero_grads, float* loss_out,
                            int ring_size, void* stream);
/* Gradient-norm clipping of every later training step of the plan (rvae_plan_train_step, rvae_plan_train_step_hp),
 * as torch.nn.utils.clip_grad_norm_ with norm type 2 between backward and Adam: norm = sqrt(sum g^2) over all ten
 * parameters' gradients (after the all-reduce under data parallelism, before weight decay), and Adam consumes
 * coef * g with coef = min(1, max_norm / (norm + 1e-6)). The sum of squares is fp64 in a fixed order (bitwise
 * repeatable); coef is rounded to fp32 once. max_norm_dev: a device double, read when the kernels run, so a graph
 * captured around a step follows any rewrite ordered before its replay; +inf measures without clipping; NULL
 * switches clipping off (the step then issues exactly the launches it issues without this call). norm_out (may be
 * NULL): the pre-clip norm of the step lands in norm_out[t mod ring_size], t = the step counter when the step starts.
 * The gradients a step leaves with zero_grads = 0 are the unclipped ones. A non-finite norm propagates as in torch.
 * Returns 1 for ring_size < 1 with a non-null norm_out (before the plan is used), 2 for the experiments-only fused
 * latent epilogue. */
int rvae_plan_set_grad_clip(rvae_plan* plan, const double* max_norm_dev, float* norm_out, int ring_size);
/* The global L2 norm of the plan's bound gradient buffer with the kernels of a clipping step -> *norm_out (device
 * float); not part of any step. Returns 1 for a null norm_out (before the plan is used). */
int rvae_plan_grad_norm(rvae_plan* plan, float* norm_out, void* stream);

/* Deterministic training steps (opt-in). With a scratch bound, every output of rvae_plan_train_step(_hp) - parameters,
 * exp_avg, exp_avg_sq, bf16 shadows, the step counter, the loss ring, the norm ring and the gradients of zero_grads = 0
 * - depends only on the inputs, the state, the hyper-parameters, the dims, the batch size, the precision and the
 * world size: not on stream timing, on which CTA runs which tile, on the SM budget (RVAE_NUM_SMS,
 * RVAE_S1_WGRAD_CTAS) or on whether a GEMM runs in a fused launch. Every sum the default step does with atomics or
 * a TMA reduce-add has a fixed order instead:
 *   - split-K weight gradients and latent dgrad: split 0 stores into the gradient (dz) buffer, split k >= 1 into its
 *     own scratch slice, with plain TMA stores; the split count comes from the shapes against a fixed 74 CTA pairs.
 *     After backward stage s one grad_sum launch adds the slices of bucket s to split 0 in split order;
 *   - bias gradients: each epilogue warp writes the column sums of its 32 rows to partial row (row / 32) of the
 *     scratch, the latent backward one row per block (fixed grid of min(ceil(rows / rows per pass), 592) blocks,
 *     rows per pass = max(1, 1024 / Lp)); the grad_sum launch after stage 2 adds each bias column's rows into the
 *     bias block in a fixed order (rows r = l mod 32 by lane l in ascending order, then a fixed 32-lane tree);
 *   - dz: the latent backward adds the slices in split order;
 *   - loss: each (32-row block, 64-column group) of the MSE and of the KL term has one fp64 slot; the finalisation
 *     adds the slots in index order (fixed thread partition and tree).
 * Scratch layout (256-byte aligned sections, sized at max_batch): weight-gradient slices (the largest bucket's) |
 * latent-dgrad slices | bias partial rows [rows32][total - b1] | latent bias rows [592 max][2Lp] | MSE slots
 * [rows32][Sp/64] (fp64) | KL slots [rows32][Lp/64] (fp64), rows32 = max_batch rounded up to 256, over 32.
 * Data parallelism is covered with the peer-load all-reduce (it sums the ranks in rank order); a step whose gradients
 * go through NVLS multicast or NCCL returns 2, as do the experiments-only paths (RVAE_FUSE_LATENT, RVAE_MERGE_B3W,
 * RVAE_FUSE_FORWARD). Only the training step is covered: rvae_plan_forward / _backward / _backward_external called
 * on their own run the default kernels. rvae_plan_workspace_bytes is unchanged. */
size_t rvae_plan_deterministic_bytes(const rvae_plan* plan);   /* scratch bytes at the plan's max_batch */
/* Bind the caller-owned scratch (>= rvae_plan_deterministic_bytes, 256-byte aligned); NULL switches the mode off.
 * Returns 1 for a short or misaligned scratch. */
int rvae_plan_set_deterministic(rvae_plan* plan, void* scratch, size_t bytes);

/* Exponential moving average (EMA) of the weights, as torch.optim.swa_utils.AveragedModel with
 * multi_avg_fn = get_ema_multi_avg_fn(decay) and update_parameters(model) after every optimizer step, kept inside the
 * training step. With an EMA set, every Adam launch of every later rvae_plan_train_step(_hp) of the plan also updates
 * ema[i] for the elements it updates, from the parameter it has just computed:
 *   n_averaged == 0: ema = p;   else ema = lerp(ema, p, w), w = (float)(1 - decay), 1 - decay formed in double;
 *   lerp(e, p, w) = |w| < 0.5 ? e + w (p - e) : p - (p - e)(1 - w)   (torch's formula), in fp32;
 * and the last block of the step's final Adam launch, which advances the step counter, does *count_dev += 1. The
 * step issues the same launches as without an EMA (the EMA is 8 more bytes per parameter in each), and parameters,
 * Adam moments, shadows and the step counter are the same bit for bit. It composes with gradient clipping,
 * deterministic mode and data parallelism (each rank updates its own EMA from the all-reduced update).
 * ema: fp32, 16-byte aligned, the flat layout of the plan's parameters (rvae_param_layout_padded; padding elements
 * stay 0 when they are 0 in ema and params). decay_dev: a device double in [0, 1], read when the kernels run, so a
 * graph captured around a step follows any rewrite ordered before its replay. count_dev: the device int64 n_averaged.
 * ema == NULL switches the EMA off. rvae_plan_adam / rvae_plan_adam_buckets called on their own do not update it.
 * Returns 1 for a non-null ema with a null decay_dev or count_dev, or a misaligned ema (before the plan is used). */
int rvae_plan_set_ema(rvae_plan* plan, float* ema, const double* decay_dev, int64_t* count_dev);
/* The same EMA update as one launch over n elements: ema = lerp(ema, params, w) (a copy when *count_dev == 0), then
 * *count_dev += 1 - what follows an optimizer step of the unfused path. ema and params: 16-byte aligned fp32. Calls on
 * one ctx must be ordered (one stream, or event-ordered): they share one device ticket. Returns 1 for a null
 * pointer, n < 0, a misaligned buffer or a null ctx. */
int rvae_ema_update(rvae_ctx* ctx, float* ema, const float* params, int64_t n, const double* decay_dev,
                    int64_t* count_dev, void* stream);

/* Evaluate the record's schedule at the n step indices k_dev[0..n) with the device function the training kernels
 * use: lr_out[i] = lr(k_dev[i]), beta_out[i] = (float)beta(k_dev[i]). Returns 1 for null pointers or n < 1 (before
 * ctx is used). */
int rvae_hparams_eval(rvae_ctx* ctx, const rvae_hparams* hp_dev, const int64_t* k_dev, int n, double* lr_out,
                      float* beta_out, void* stream);

/* Device pointers into the workspace for the current batch (valid after forward): fp32 [batch, ...] at the plan's
 * padded row pitch - mu, logvar, eps [batch, Lp], xhat [batch, Sp] (rvae_param_layout_padded); only the first L (S)
 * columns of a row are the model's, the rest are zeros. */
const float* rvae_plan_mu(const rvae_plan* plan);
const float* rvae_plan_logvar(const rvae_plan* plan);
const float* rvae_plan_xhat(const rvae_plan* plan);
const float* rvae_plan_eps(const rvae_plan* plan);
/* Introspection (tests / debugging): device pointers to the bf16 planes of an intermediate of the current batch.
 * which: 0 x [B,S], 1 h1 [B,H], 2 z [B,L], 3 h3 [B,H], 4 da4 [B,S], 5 da3 [B,H], 6 d_ml [B,2L], 7 da1 [B,H], all
 * at the padded dims (*cols = the row pitch). *lo is NULL in bf16 mode. */
int rvae_plan_activation(const rvae_plan* plan, int which, void** hi, void** lo, int* cols);
/* gradient bucket s (see rvae_plan_backward): pointer into bufs.grads and element count. Buckets 0..3 are the
 * four weight matrices in backward-completion order; bucket 4 is the bias block (padded blocks of a padded plan). */
int rvae_plan_bucket(const rvae_plan* plan, int s, float** ptr, int64_t* count);

/* Per-kernel device timing (bench.py roofline): when enabled, every launch of the plan is bracketed by CUDA events
 * on the launch stream (this also disables the overlap of consecutive kernels, so use it for attribution, not for
 * the headline number). rvae_plan_read_timing synchronises those events and returns, per slot, the accumulated
 * milliseconds, launch count and - for the GEMM slots - algorithmic FLOPs per launch (2*M*N*K); it then clears the
 * accumulators. Slots 0..11 are the tcgen05 GEMMs F1, F2, F3, F4(out), F4(linear), B4w, B4d, B3w, B3d, B2w, B2d, B1w;
 * slots 12..18 the HBM-bound kernels: batch load (framing / split), eps, loss finalize, bias-gradient column sums,
 * Adam, tanh backward, latent backward. All three output arrays hold RVAE_NUM_TIMING_SLOTS entries. */
#define RVAE_NUM_GEMM_SLOTS 12
#define RVAE_NUM_TIMING_SLOTS 19
int rvae_plan_enable_timing(rvae_plan* plan, int enable);
int rvae_plan_read_timing(rvae_plan* plan, float* ms, int64_t* launches, double* flops_per_launch);

/* Debug / profiling aid: every tcgen05 GEMM prepared through `ctx` after this call writes a per-CTA, per-tile
 * timeline (clock64 stamps of the TMA-producer, MMA-issuer and epilogue roles; layout in csrc/gemm.cuh, "Timeline
 * trace") into `buf` (device memory, `launches` slabs of RVAE_TRACE_WORDS_PER_CTA * SM-count 64-bit words; successive
 * GEMM launches use successive slabs, wrapping around). NULL switches tracing off. Costs a few stores per tile;
 * never enabled on the training path. */
#define RVAE_TRACE_HEADER_WORDS 16
#define RVAE_TRACE_TILES 24
#define RVAE_TRACE_EVENTS 16
#define RVAE_TRACE_WORDS_PER_CTA (RVAE_TRACE_HEADER_WORDS + RVAE_TRACE_TILES * RVAE_TRACE_EVENTS)
int rvae_debug_set_trace(rvae_ctx* ctx, void* buf, int launches);
/* Same idea for the HBM-bound kernels (gather, randn, latent backward, Adam): launch i writes 8 words at buf + 8*i
 * (wrapping at `launches`): globaltimer of the first block's start (initialise to ~0ull) and the last block's end,
 * kind (1 gather, 2 randn, 3 latent backward, 4 Adam, 5 all-reduce), grid size, 4 kernel-specific detail words. */
int rvae_debug_set_aux_trace(rvae_ctx* ctx, void* buf, int launches);

/* Inference: decode latents z (fp32 [batch, L]) -> xhat fp32 [batch, S] (model.py:28-30). */
int rvae_plan_decode(rvae_plan* plan, const float* z, int batch, float* xhat_out, void* stream);
/* Inference, interpolation pattern (tutorial.ipynb:496-510, 905-932) as one chained enqueue: lerp of two latent
 * distributions with one alpha per frame -> reparameterize -> decode. z is written straight into fc3's bf16 operand
 * (no fp32 z round trip); arguments as rvae_lerp_reparameterize, xhat_out fp32 [batch, S]. */
int rvae_plan_decode_lerp(rvae_plan* plan, const float* mu_a, const float* logvar_a, const float* mu_b,
                          const float* logvar_b, const void* alpha, int alpha_is_f64, const float* eps, int batch,
                          float* xhat_out, void* stream);
/* Inference: encode the loaded batch -> mu, logvar (model.py:19-21); results via rvae_plan_mu/logvar. */
int rvae_plan_encode(rvae_plan* plan, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RVAE_B200_H */
