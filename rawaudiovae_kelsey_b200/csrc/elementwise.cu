// HBM-bound kernels of the hot path: framing / overlap-add, Philox normal noise, bf16 plane splitting,
// bias-gradient column sums, the fused reparameterisation + reconstruction/KL loss kernels, and fused Adam.
// All are coalesced, 128-bit vectorised, grid-strided with grids sized in multiples of the SM count.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <memory>

#include "../../include/rvae_b200.h"
#include "common.h"

namespace rvae {

static inline int grid_for(const Ctx* ctx, int64_t work_items, int threads, int max_waves = 8) {
  int64_t blocks = (work_items + threads - 1) / threads;
  const int64_t cap = static_cast<int64_t>(ctx->num_sms) * max_waves;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return static_cast<int>(blocks);
}

#define RVAE_LAUNCH_CHECK(ctx)           \
  do {                                   \
    (ctx)->launches++;                   \
  } while (0)

__device__ __forceinline__ uint32_t pack2(float a, float b) { return ptx::pack_bf16x2(a, b); }

__device__ __forceinline__ void aux_begin(const AuxTrace& t, int kind) {
  if (t.slot != nullptr && threadIdx.x == 0) {
    atomicMin(t.slot, global_timer());
    if (blockIdx.x == 0) { t.slot[2] = kind; t.slot[3] = gridDim.x; }
  }
}
__device__ __forceinline__ void aux_end(const AuxTrace& t) {
  if (t.slot != nullptr && threadIdx.x == 0) atomicMax(t.slot + 1, global_timer());
}

__device__ __forceinline__ float block_sum_to_warp0(float v, float* smem) {
  // returns the block total in every thread of warp 0
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) smem[warp] = v;
  __syncthreads();
  float t = 0.f;
  if (warp == 0) {
    const int nw = (blockDim.x + 31) >> 5;
    t = (lane < nw) ? smem[lane] : 0.f;
    t = warp_sum(t);
  }
  __syncthreads();
  return t;
}

__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;   // lane 0
}

// ------------------------------------------------------------------------------------------------
// K-D1 framing: frame f = audio_pad[idx*hop : idx*hop + S], zero beyond n_samples (the reference zero-pads the
// tail, rawvae/dataset.py:102-104,141-143). idx = frame_idx[f] (shuffled map-style batches) or first_frame + f
// (streaming / sequential). One thread converts 8 consecutive samples. Output rows are W >= S elements wide: columns
// S..W are written as zeros (the zero padding of a plan whose segment_length is not a multiple of 64).
// ------------------------------------------------------------------------------------------------
template <bool I16, int U>
__global__ void frame_gather_kernel(const void* __restrict__ audio, int64_t n_samples,
                                    const int64_t* __restrict__ frame_idx, int64_t first_frame, int64_t n_frames,
                                    int hop, int S, int W, __nv_bfloat16* __restrict__ out_hi,
                                    __nv_bfloat16* __restrict__ out_lo, float* __restrict__ out_f32, AuxTrace tr) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  aux_begin(tr, 1);
  const int vec_per_frame = (W + 7) >> 3;
  const bool vec_store = (W & 7) == 0;   // 16-byte rows: vector stores (else the row width is the caller's odd S)
  const int64_t total = n_frames * vec_per_frame;
  // U groups of 8 samples per thread and trip: the U frame indices are fetched first, then all 2 U 16-byte loads are
  // issued before the first convert / store (U = 1 by default: occupancy beats per-thread unrolling here)
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i0 < total; i0 += U * stride) {
    int64_t fr[U], s0[U];
    int col[U];
    bool fast[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t i = i0 + u * stride;
      fr[u] = i < total ? i / vec_per_frame : -1;
      col[u] = fr[u] >= 0 ? static_cast<int>(i - fr[u] * vec_per_frame) << 3 : 0;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t fi = fr[u] < 0 ? 0 : (frame_idx ? __ldg(frame_idx + fr[u]) : first_frame + fr[u]);
      s0[u] = fi * hop + col[u];
      // 16-byte aligned source address (the buffer base may itself be an unaligned view of a longer stream)
      const uintptr_t addr = reinterpret_cast<uintptr_t>(audio) + static_cast<uintptr_t>(s0[u]) * (I16 ? 2 : 4);
      fast[u] = fr[u] >= 0 && col[u] + 8 <= S && s0[u] >= 0 && s0[u] + 8 <= n_samples && (addr & 15) == 0;
    }
    float v[U][8];
    uint4 raw[U][2];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (!fast[u]) continue;
      if constexpr (I16) {
        raw[u][0] = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const int16_t*>(audio) + s0[u]));
      } else {
        const uint4* a = reinterpret_cast<const uint4*>(reinterpret_cast<const float*>(audio) + s0[u]);
        raw[u][0] = __ldg(a);
        raw[u][1] = __ldg(a + 1);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (fr[u] < 0) continue;
      if (fast[u]) {
        if constexpr (I16) {
          const int16_t* h = reinterpret_cast<const int16_t*>(&raw[u][0]);
#pragma unroll
          for (int j = 0; j < 8; ++j) v[u][j] = h[j] * (1.0f / 32768.0f);
        } else {
          const float* f = reinterpret_cast<const float*>(&raw[u][0]);
#pragma unroll
          for (int j = 0; j < 8; ++j) v[u][j] = f[j];
        }
      } else {   // unaligned start, the zero-padded tail beyond n_samples, or columns at and past S
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int64_t sidx = s0[u] + j;
          float x = 0.f;
          if (col[u] + j < S && sidx >= 0 && sidx < n_samples) {
            if constexpr (I16) x = __ldg(reinterpret_cast<const int16_t*>(audio) + sidx) * (1.0f / 32768.0f);
            else x = __ldg(reinterpret_cast<const float*>(audio) + sidx);
          }
          v[u][j] = x;
        }
      }
      const int64_t o = fr[u] * W + col[u];
      if (!vec_store) {
        for (int j = 0; j < 8 && col[u] + j < W; ++j) {
          const __nv_bfloat16 h = __float2bfloat16_rn(v[u][j]);
          if (out_hi) out_hi[o + j] = h;
          if (out_lo) out_lo[o + j] = __float2bfloat16_rn(v[u][j] - __bfloat162float(h));
          if (out_f32) out_f32[o + j] = v[u][j];
        }
        continue;
      }
      if (out_hi) {
        *reinterpret_cast<uint4*>(out_hi + o) = make_uint4(pack2(v[u][0], v[u][1]), pack2(v[u][2], v[u][3]),
                                                           pack2(v[u][4], v[u][5]), pack2(v[u][6], v[u][7]));
      }
      if (out_lo) {
        float r[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] = v[u][j] - __bfloat162float(__float2bfloat16_rn(v[u][j]));
        *reinterpret_cast<uint4*>(out_lo + o) =
            make_uint4(pack2(r[0], r[1]), pack2(r[2], r[3]), pack2(r[4], r[5]), pack2(r[6], r[7]));
      }
      if (out_f32) {
        float4* d = reinterpret_cast<float4*>(out_f32 + o);
        d[0] = make_float4(v[u][0], v[u][1], v[u][2], v[u][3]);
        d[1] = make_float4(v[u][4], v[u][5], v[u][6], v[u][7]);
      }
    }
  }
  aux_end(tr);
}

int launch_frame_gather(Ctx* ctx, const void* audio, int audio_is_i16, int64_t n_samples, const int64_t* frame_idx,
                        int64_t first_frame, int64_t n_frames, int hop, int S, int W, __nv_bfloat16* out_hi,
                        __nv_bfloat16* out_lo, float* out_f32, cudaStream_t stream) {
  RVAE_REQUIRE(audio && (out_hi || out_f32), RVAE_ERR_INVALID, "frame_gather: null buffer");
  RVAE_REQUIRE(S > 0 && hop > 0 && W >= S, RVAE_ERR_UNSUPPORTED, "frame_gather: S=%d, row width %d, hop %d", S, W, hop);
  if (n_frames <= 0) return RVAE_OK;
  const int threads = 256;
  // RVAE_GATHER_UNROLL (1 / 2 / 4 groups of 8 samples per thread and trip), RVAE_GATHER_WAVES: tuning knobs
  // measured (profiles/README.md, round 2): one group per thread and trip with 16 blocks per SM is the fastest alone
  // (16.4 us vs 24.6 us for 4 groups) and no slower inside a step, where the kernel runs on the background stream
  static const int unroll = getenv("RVAE_GATHER_UNROLL") ? atoi(getenv("RVAE_GATHER_UNROLL")) : 1;
  static const int waves = getenv("RVAE_GATHER_WAVES") ? atoi(getenv("RVAE_GATHER_WAVES")) : 16;
  const int u = unroll == 1 ? 1 : (unroll == 2 ? 2 : 4);
  const int grid = grid_for(ctx, (n_frames * ((W + 7) / 8) + u - 1) / u, threads, waves > 0 ? waves : 8);
  const AuxTrace tr = next_aux(ctx, 1);
  auto go = [&](auto kern) {
    return launch_kernel(ctx, kern, dim3(grid), dim3(threads), (size_t)0, stream, audio, n_samples, frame_idx,
                         first_frame, n_frames, hop, S, W, out_hi, out_lo, out_f32, tr);
  };
  if (audio_is_i16) {
    if (u == 1) RVAE_CUDA(go(frame_gather_kernel<true, 1>));
    else if (u == 2) RVAE_CUDA(go(frame_gather_kernel<true, 2>));
    else RVAE_CUDA(go(frame_gather_kernel<true, 4>));
  } else {
    if (u == 1) RVAE_CUDA(go(frame_gather_kernel<false, 1>));
    else if (u == 2) RVAE_CUDA(go(frame_gather_kernel<false, 2>));
    else RVAE_CUDA(go(frame_gather_kernel<false, 4>));
  }
  RVAE_LAUNCH_CHECK(ctx);
  return RVAE_OK;
}

// ------------------------------------------------------------------------------------------------
// K-D2 overlap-add resynthesis (gather form, no atomics): out[t] = sum_i frames[i, t - i*hop] / count(t)
// over the frames i that cover sample t. With hop == S this is the reference's frames.view(-1).
// ------------------------------------------------------------------------------------------------
template <bool VEC>
__global__ void overlap_add_kernel(const float* __restrict__ frames, int64_t n_frames, int S, int hop,
                                   float* __restrict__ out, int64_t t_begin, int64_t n_out) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  // VEC: S, hop and both base addresses are multiples of 4 elements, so the 4 samples of an aligned group are
  // covered by the same frames at offsets that stay 16-byte aligned; the per-sample sum order (ascending frame
  // index) is the scalar path's, hence bit-identical results. The scalar path also finishes a ragged tail.
  constexpr int W = VEC ? 4 : 1;
  const int64_t n_groups = VEC ? (n_out >> 2) : n_out;
  out -= t_begin;   // out[t - t_begin] = OLA(t) for t in [t_begin, t_begin + n_out)
  for (int64_t w = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; w < n_groups; w += (int64_t)gridDim.x * blockDim.x) {
    const int64_t t = t_begin + w * W;
    int64_t i_hi = t / hop;
    if (i_hi > n_frames - 1) i_hi = n_frames - 1;
    int64_t i_lo = (t - S + hop) / hop;  // ceil((t - S + 1) / hop) for t - S + 1 > 0
    if (t - S + 1 <= 0) i_lo = 0;
    float acc[W];
#pragma unroll
    for (int j = 0; j < W; ++j) acc[j] = 0.f;
    int cnt = 0;
    for (int64_t i = i_lo; i <= i_hi; ++i) {
      const int64_t off = t - i * hop;
      if (off >= 0 && off < S) {
        if constexpr (VEC) {
          const float4 f = __ldg(reinterpret_cast<const float4*>(frames + i * S + off));
          acc[0] += f.x; acc[1] += f.y; acc[2] += f.z; acc[3] += f.w;
        } else {
          acc[0] += __ldg(frames + i * S + off);
        }
        ++cnt;
      }
    }
    const float c = static_cast<float>(cnt);
    if constexpr (VEC) {
      float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
      if (cnt > 0) o = make_float4(acc[0] / c, acc[1] / c, acc[2] / c, acc[3] / c);
      *reinterpret_cast<float4*>(out + t) = o;
    } else {
      out[t] = cnt > 0 ? acc[0] / c : 0.f;
    }
  }
}

// samples [t0, n_out) of the scalar rule (the < 4-sample tail the vector path leaves)
__global__ void overlap_add_tail_kernel(const float* __restrict__ frames, int64_t n_frames, int S, int hop,
                                        float* __restrict__ out, int64_t t_begin, int64_t t0, int64_t t_end) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  out -= t_begin;
  for (int64_t t = t0 + threadIdx.x; t < t_end; t += blockDim.x) {
    int64_t i_hi = t / hop;
    if (i_hi > n_frames - 1) i_hi = n_frames - 1;
    int64_t i_lo = (t - S + hop) / hop;
    if (t - S + 1 <= 0) i_lo = 0;
    float acc = 0.f;
    int cnt = 0;
    for (int64_t i = i_lo; i <= i_hi; ++i) {
      const int64_t off = t - i * hop;
      if (off >= 0 && off < S) {
        acc += __ldg(frames + i * S + off);
        ++cnt;
      }
    }
    out[t] = cnt > 0 ? acc / static_cast<float>(cnt) : 0.f;
  }
}

int launch_overlap_add(Ctx* ctx, const float* frames, int64_t n_frames, int S, int hop, float* out, int64_t t_begin,
                       int64_t n_out, cudaStream_t stream) {
  RVAE_REQUIRE(frames && out, RVAE_ERR_INVALID, "overlap_add: null buffer");
  RVAE_REQUIRE(S > 0 && hop > 0 && hop <= S && t_begin >= 0, RVAE_ERR_UNSUPPORTED, "overlap_add: need 0 < hop <= S, t_begin >= 0");
  if (n_out <= 0) return RVAE_OK;
  const int threads = 256;
  const bool vec = S % 4 == 0 && hop % 4 == 0 && t_begin % 4 == 0 &&
                   ((reinterpret_cast<uintptr_t>(frames) | reinterpret_cast<uintptr_t>(out)) & 15) == 0;
  int64_t done = 0;
  if (vec && n_out >= 4) {
    done = n_out & ~(int64_t)3;
    RVAE_CUDA(launch_kernel(ctx, overlap_add_kernel<true>, dim3(grid_for(ctx, done >> 2, threads, 16)), dim3(threads), (size_t)0, stream, frames, n_frames, S, hop, out, t_begin, done));
  }
  if (done < n_out) {
    if (done == 0) {
      RVAE_CUDA(launch_kernel(ctx, overlap_add_kernel<false>, dim3(grid_for(ctx, n_out, threads, 16)), dim3(threads), (size_t)0, stream, frames, n_frames, S, hop, out, t_begin, n_out));
    } else {
      // ragged tail (< 4 samples) of the vector path
      RVAE_CUDA(launch_kernel(ctx, overlap_add_tail_kernel, dim3(1), dim3(32), (size_t)0, stream, frames, n_frames, S, hop, out, t_begin, t_begin + done, t_begin + n_out));
    }
  }
  RVAE_LAUNCH_CHECK(ctx);
  return RVAE_OK;
}

// ------------------------------------------------------------------------------------------------
// Philox4x32-10 + Box-Muller: eps ~ N(0,1) for the reparameterisation (rawvae/model.py:25, torch.randn_like).
// Counter = (element index / 4, offset); key = seed. Statistically equivalent to, not bit-identical with, torch's
// generator - parity runs inject eps explicitly.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void philox4x32_10(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
    const uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
    c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
}

// the four normal values of Philox counter ci (elements 4 ci .. 4 ci + 3 of the logical noise tensor)
__device__ __forceinline__ void randn4(int64_t ci, uint64_t seed, uint64_t offset, float (&z)[4]) {
  uint32_t c[4] = {static_cast<uint32_t>(ci), static_cast<uint32_t>(ci >> 32), static_cast<uint32_t>(offset),
                   static_cast<uint32_t>(offset >> 32)};
  philox4x32_10(c, static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32));
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const float u1 = (static_cast<float>(c[2 * h] >> 8) + 0.5f) * (1.0f / 16777216.0f);  // (0,1)
    const float u2 = (static_cast<float>(c[2 * h + 1] >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float r = sqrtf(-2.0f * __logf(u1));
    float s, co;
    __sincosf(6.283185307179586f * u2, &s, &co);
    z[2 * h] = r * co;
    z[2 * h + 1] = r * s;
  }
}

__global__ void randn_kernel(float* __restrict__ out, int64_t n, uint64_t seed, uint64_t offset,
                             const float* __restrict__ offset_src, int64_t vec_base, AuxTrace tr) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  aux_begin(tr, 2);
  // offset_src: a device-side counter (the Adam step) added to the offset, so that a CUDA graph replays fresh noise
  if (offset_src) offset += static_cast<uint64_t>(__ldg(offset_src));
  const int64_t nvec = (n + 3) >> 2;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nvec; i += (int64_t)gridDim.x * blockDim.x) {
    // vec_base: this buffer is elements [4 * vec_base, ...) of a larger logical tensor (a rank's rows of the global
    // batch under data parallelism): the ranks draw disjoint pieces of ONE stream, the single-process draw
    float z[4];
    randn4(i + vec_base, seed, offset, z);
    const int64_t o = i << 2;
    if (o + 4 <= n) {
      *reinterpret_cast<float4*>(out + o) = make_float4(z[0], z[1], z[2], z[3]);
    } else {
      for (int j = 0; j < 4 && o + j < n; ++j) out[o + j] = z[j];
    }
  }
  aux_end(tr);
}

// Row-pitched draw: out[r * ld + c] = element elem_base + r * cols + c of the logical noise tensor for c < cols, 0 for
// cols <= c < ld (the zero padding of a plan whose latent_dim is not a multiple of 64). Any elem_base. One thread per
// output element; each evaluates the Philox block of its element (the noise is a few hundred KB per step).
__global__ void randn_rows_kernel(float* __restrict__ out, int64_t rows, int64_t cols, int64_t ld, uint64_t seed,
                                  uint64_t offset, const float* __restrict__ offset_src, int64_t elem_base, AuxTrace tr) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  aux_begin(tr, 2);
  if (offset_src) offset += static_cast<uint64_t>(__ldg(offset_src));
  const int64_t n = rows * ld;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / ld;
    const int64_t c = i - r * ld;
    float v = 0.f;
    if (c < cols) {
      const int64_t e = elem_base + r * cols + c;
      float z[4];
      randn4(e >> 2, seed, offset, z);
      v = z[e & 3];
    }
    out[i] = v;
  }
  aux_end(tr);
}

int launch_randn_rows(Ctx* ctx, float* out, int64_t rows, int64_t cols, int64_t ld, uint64_t seed, uint64_t offset,
                      const float* offset_src, int64_t elem_base, cudaStream_t stream) {
  RVAE_REQUIRE(out && cols > 0 && ld >= cols && elem_base >= 0, RVAE_ERR_INVALID, "randn_rows: bad arguments");
  if (rows <= 0) return RVAE_OK;
  const int threads = 256;
  RVAE_CUDA(launch_kernel(ctx, randn_rows_kernel, dim3(grid_for(ctx, rows * ld, threads, 8)), dim3(threads), (size_t)0,
                          stream, out, rows, cols, ld, seed, offset, offset_src, elem_base, next_aux(ctx, 2)));
  RVAE_LAUNCH_CHECK(ctx);
  return RVAE_OK;
}

int launch_randn(Ctx* ctx, float* out, int64_t n, uint64_t seed, uint64_t offset, const float* offset_src,
                 int64_t elem_base, cudaStream_t stream) {
  RVAE_REQUIRE(out && (reinterpret_cast<uintptr_t>(out) & 15) == 0, RVAE_ERR_INVALID, "randn: bad output buffer");
  RVAE_REQUIRE(elem_base >= 0 && (elem_base & 3) == 0, RVAE_ERR_INVALID, "randn: elem_base must be a multiple of 4");
  if (n <= 0) return RVAE_OK;
  const int threads = 256;
  RVAE_CUDA(launch_kernel(ctx, randn_kernel, dim3(grid_for(ctx, (n + 3) / 4, threads, 8)), dim3(threads), (size_t)0, stream, out, n, seed, offset, offset_src, elem_base >> 2, next_aux(ctx, 2)));
  RVAE_LAUNCH_CHECK(ctx);
  return RVAE_OK;
}

// ------------------------------------------------------------------------------------------------
// fp32 -> bf16 hi (+ residual lo) planes
// ------------------------------------------------------------------------------------------------
__global__ void split_bf16_kernel(const float* __restrict__ src, int64_t n, __nv_bfloat16* __restrict__ hi,
                                  __nv_bfloat16* __restrict__ lo) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  const int64_t nvec = n >> 3;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nvec; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(src) + 2 * i);
    const float4 b = __ldg(reinterpret_cast<const float4*>(src) + 2 * i + 1);
    const float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    reinterpret_cast<uint4*>(hi)[i] =
        make_uint4(pack2(v[0], v[1]), pack2(v[2], v[3]), pack2(v[4], v[5]), pack2(v[6], v[7]));
    if (lo) {
      float r[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) r[j] = v[j] - __bfloat162float(__float2bfloat16_rn(v[j]));
      reinterpret_cast<uint4*>(lo)[i] =
          make_uint4(pack2(r[0], r[1]), pack2(r[2], r[3]), pack2(r[4], r[5]), pack2(r[6], r[7]));
    }
  }
  // tail (n % 8)
  if (blockIdx.x == 0) {
    for (int64_t j = (nvec << 3) + threadIdx.x; j < n; j += blockDim.x) {
      const float v = src[j];
      const __nv_bfloat16 h = __float2bfloat16_rn(v);
      hi[j] = h;
      if (lo) lo[j] = __float2bfloat16_rn(v - __bfloat162float(h));
    }
  }
}

// fp32 [rows, cols] at row pitch ld_src -> bf16 planes [rows, ld_dst], zeros in columns cols..ld_dst (caller tensors
// of a plan whose dims are not multiples of 64, on their way into the padded operands)
__global__ void split_bf16_rows_kernel(const float* __restrict__ src, int64_t rows, int cols, int ld_src, int ld_dst,
                                       __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  const int64_t n = rows * ld_dst;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / ld_dst;
    const int c = static_cast<int>(i - r * ld_dst);
    const float v = c < cols ? src[r * ld_src + c] : 0.f;
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    hi[i] = h;
    if (lo) lo[i] = __float2bfloat16_rn(v - __bfloat162float(h));
  }
}

int launch_split_bf16_rows(Ctx* ctx, const float* src, int64_t rows, int cols, int ld_src, int ld_dst,
                           __nv_bfloat16* hi, __nv_bfloat16* lo, cudaStream_t stream) {
  RVAE_REQUIRE(src && hi && cols > 0 && ld_src >= cols && ld_dst >= cols, RVAE_ERR_INVALID, "split_bf16_rows: bad arguments");
  if (rows <= 0) return RVAE_OK;
  const int threads = 256;
  RVAE_CUDA(launch_kernel(ctx, split_bf16_rows_kernel, dim3(grid_for(ctx, rows * ld_dst, threads, 8)), dim3(threads),
                          (size_t)0, stream, src, rows, cols, ld_src, ld_dst, hi, lo));
  RVAE_LAUNCH_CHECK(ctx);
  return RVAE_OK;
}

int launch_split_bf16(Ctx* ctx, const float* src, int64_t n, __nv_bfloat16* hi, __nv_bfloat16* lo,
                      cudaStream_t stream) {
  RVAE_REQUIRE(src && hi, RVAE_ERR_INVALID, "split_bf16: null buffer");
  RVAE_REQUIRE(((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(hi) |
                 reinterpret_cast<uintptr_t>(lo)) & 15) == 0,
               RVAE_ERR_INVALID, "split_bf16: buffers must be 16-byte aligned");
  if (n <= 0) return RVAE_OK;
  const int threads = 256;
  RVAE_CUDA(launch_kernel(ctx, split_bf16_kernel, dim3(grid_for(ctx, (n + 7) / 8, threads, 8)), dim3(threads), (size_t)0, stream, src, n, hi, lo));
  RVAE_LAUNCH_CHECK(ctx);
  return RVAE_OK;
}

// ------------------------------------------------------------------------------------------------
// Bias gradients: out[n] (+)= sum_m (hi[m,n] + lo[m,n]). Each block owns a 64-column strip and a slab of rows;
// a thread accumulates 2 adjacent columns (one bf16x2 load) down the slab, warps combine through smem, one
// atomicAdd per column per block.
// ------------------------------------------------------------------------------------------------
constexpr int kColsumRowsPerBlock = 256;

__global__ void colsum_kernel(const __nv_bfloat16* __restrict__ hi, const __nv_bfloat16* __restrict__ lo, int64_t M,
                              int N, int ld, float* __restrict__ out) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  __shared__ float part[8][64];
  const int strip = blockIdx.x;           // 64 columns
  const int lane = threadIdx.x & 31;      // 2 columns each
  const int warp = threadIdx.x >> 5;      // 8 warps interleave rows
  const int col = strip * 64 + lane * 2;
  const int64_t r0 = static_cast<int64_t>(blockIdx.y) * kColsumRowsPerBlock;
  int64_t r1 = r0 + kColsumRowsPerBlock;
  if (r1 > M) r1 = M;
  float s0 = 0.f, s1 = 0.f;
  if (col < N) {
    for (int64_t r = r0 + warp; r < r1; r += 8) {
      const __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(hi + r * ld + col);
      float2 f = __bfloat1622float2(h);
      if (lo) {
        const float2 g = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(lo + r * ld + col));
        f.x += g.x; f.y += g.y;
      }
      s0 += f.x; s1 += f.y;
    }
  }
  part[warp][lane * 2] = s0;
  part[warp][lane * 2 + 1] = s1;
  __syncthreads();
  if (threadIdx.x < 64) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += part[w][threadIdx.x];
    const int c = strip * 64 + threadIdx.x;
    if (c < N) atomicAdd(out + c, t);
  }
}

int launch_colsum(Ctx* ctx, const __nv_bfloat16* hi, const __nv_bfloat16* lo, int64_t M, int N, int ld, float* out,
                  int accumulate, cudaStream_t stream) {
  RVAE_REQUIRE(hi && out, RVAE_ERR_INVALID, "colsum: null buffer");
  RVAE_REQUIRE(N % 2 == 0 && ld % 2 == 0, RVAE_ERR_UNSUPPORTED, "colsum: N and ld must be even");
  if (!accumulate) RVAE_CUDA(cudaMemsetAsync(out, 0, sizeof(float) * N, stream));
  if (M <= 0) return RVAE_OK;
  dim3 grid((N + 63) / 64, static_cast<unsigned>((M + kColsumRowsPerBlock - 1) / kColsumRowsPerBlock));
  RVAE_CUDA(launch_kernel(ctx, colsum_kernel, dim3(grid), dim3(256), (size_t)0, stream, hi, lo, M, N, ld, out));
  RVAE_LAUNCH_CHECK(ctx);
  return RVAE_OK;
}

// ------------------------------------------------------------------------------------------------
// K-L1/K-L2 fused loss (rawvae/model.py:38-46): acc[0] += sum (xhat-x)^2, acc[1] += sum (1+lv-mu^2-e^lv),
// warp-shuffle + block reduction, one double atomic per block. loss_finalize turns the sums into
//   mse/(B*S) + beta * (-0.5) * kl/(B*L)   and clears the accumulators for the next step.
// ------------------------------------------------------------------------------------------------
__global__ void loss_fwd_kernel(const float* __restrict__ xhat, const float* __restrict__ x,
                                const float* __restrict__ mu, const float* __restrict__ lv, int64_t n_rec,
                                int64_t n_lat, double* __restrict__ acc) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  __shared__ float red[32];
  float mse = 0.f, kl = 0.f;
  const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t nv = n_rec >> 2;
  for (int64_t i = tid; i < nv; i += stride) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(xhat) + i);
    const float4 b = __ldg(reinterpret_cast<const float4*>(x) + i);
    const float d0 = a.x - b.x, d1 = a.y - b.y, d2 = a.z - b.z, d3 = a.w - b.w;
    mse += d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
  }
  for (int64_t i = (nv << 2) + tid; i < n_rec; i += stride) {
    const float d = xhat[i] - x[i];
    mse += d * d;
  }
  const int64_t lvn = n_lat >> 2;
  for (int64_t i = tid; i < lvn; i += stride) {
    const float4 m = __ldg(reinterpret_cast<const float4*>(mu) + i);
    const float4 l = __ldg(reinterpret_cast<const float4*>(lv) + i);
    kl += (1.f + l.x - m.x * m.x - expf(l.x)) + (1.f + l.y - m.y * m.y - expf(l.y)) +
          (1.f + l.z - m.z * m.z - expf(l.z)) + (1.f + l.w - m.w * m.w - expf(l.w));
  }
  for (int64_t i = (lvn << 2) + tid; i < n_lat; i += stride) kl += 1.f + lv[i] - mu[i] * mu[i] - expf(lv[i]);
  const float tm = block_sum_to_warp0(mse, red);
  const float tk = block_sum_to_warp0(kl, red);
  if (threadIdx.x == 0) {
    atomicAdd(acc, static_cast<double>(tm));
    atomicAdd(acc + 1, static_cast<double>(tk));
  }
}

// ------------------------------------------------------------------------------------------------
// Scheduled hyper-parameters (rvae_hparams, include/rvae_b200.h): lr(k) and beta(k) at step index k. Every operation
// is an explicitly rounded fp64 intrinsic (no FMA contraction) in the order the header writes it, so schedule.py's
// host mirror, which repeats them one by one, gets the same doubles.
// ------------------------------------------------------------------------------------------------
// cos(pi u) for u in [0, 1]: Taylor series to x^22 at x = pi * min(u, 1 - u) <= pi / 2 (truncation < 1e-19),
// negated for u > 0.5 - a fixed polynomial instead of the libm cos, whose last bit differs between device and host
__device__ __forceinline__ double cos_pi_unit(double u) {
  const double c[12] = {1.0, -0.5, 0.041666666666666664, -0.001388888888888889, 2.48015873015873e-05,
                        -2.755731922398589e-07, 2.08767569878681e-09, -1.1470745597729725e-11, 4.779477332387385e-14,
                        -1.5619206968586225e-16, 4.110317623312165e-19, -8.896791392450574e-22};
  const bool flip = u > 0.5;
  if (flip) u = __dadd_rn(1.0, -u);
  const double x = __dmul_rn(3.141592653589793, u);
  const double x2 = __dmul_rn(x, x);
  double r = c[11];
#pragma unroll
  for (int i = 10; i >= 0; --i) r = __dadd_rn(__dmul_rn(r, x2), c[i]);
  return flip ? -r : r;
}

__device__ __forceinline__ void hparams_eval(const rvae_hparams& h, double k, double* lr_out, float* beta_out) {
  const double lr = h.lr;
  const double W = static_cast<double>(h.warmup_steps);
  double a;
  if (k < W) {
    a = __ddiv_rn(__dmul_rn(lr, __dadd_rn(k, 1.0)), W);
  } else if (h.lr_schedule == RVAE_LR_CONSTANT) {
    a = lr;
  } else {
    const int64_t d = h.total_steps - h.warmup_steps;
    const double D = static_cast<double>(d > 1 ? d : 1);
    const double u = __ddiv_rn(fmin(__dadd_rn(k, -W), D), D);
    const double span = __dadd_rn(lr, -h.lr_min);
    if (h.lr_schedule == RVAE_LR_LINEAR)
      a = __dadd_rn(h.lr_min, __dmul_rn(span, __dadd_rn(1.0, -u)));
    else
      a = __dadd_rn(h.lr_min, __dmul_rn(__dmul_rn(span, 0.5), __dadd_rn(1.0, cos_pi_unit(u))));
  }
  double b = h.kl_beta;
  if (h.kl_anneal != RVAE_KL_CONSTANT) {
    double f;
    if (h.kl_anneal == RVAE_KL_LINEAR) {
      f = fmin(1.0, __ddiv_rn(k, static_cast<double>(h.kl_anneal_steps)));
    } else {
      const int64_t C = (h.total_steps + h.kl_cycles - 1) / h.kl_cycles;
      const double tau = __ddiv_rn(static_cast<double>(static_cast<int64_t>(k) % C), static_cast<double>(C));
      f = fmin(1.0, __ddiv_rn(tau, h.kl_cycle_ratio));
    }
    b = __dadd_rn(h.kl_beta_start, __dmul_rn(__dadd_rn(h.kl_beta, -h.kl_beta_start), f));
  }
  *lr_out = a;
  *beta_out = static_cast<float>(b);
}

__global__ void hparams_eval_kernel(const rvae_hparams* __restrict__ hp, const int64_t* __restrict__ k, int n,
                                    double* __restrict__ lr_out, float* __restrict__ beta_out) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) hparams_eval(*hp, static_cast<double>(k[i]), lr_out + i, beta_out + i);
}

int launch_hparams_eval(Ctx* ctx, const rvae_hparams* hp, const int64_t* k, int n, double* lr_out, float* beta_out,
                        cudaStream_t stream) {
  RVAE_REQUIRE(hp && k && lr_out && beta_out && n > 0, RVAE_ERR_INVALID, "hparams_eval: null buffer or n %d", n);
  RVAE_CUDA(launch_kernel(ctx, hparams_eval_kernel, dim3((n + 127) / 128), dim3(128), (size_t)0, stream, hp, k, n,
                          lr_out, beta_out));
  RVAE_LAUNCH_CHECK(ctx);
  return RVAE_OK;
}

HpArg hp_value(double lr, double beta1, double beta2, double eps, double weight_decay) {
  HpArg a;
  memset(&a, 0, sizeof(a));
  a.val.lr = lr; a.val.beta1 = beta1; a.val.beta2 = beta2; a.val.eps = eps; a.val.weight_decay = weight_decay;
  a.val.kl_cycle_ratio = 1.0; a.val.kl_anneal_steps = 1; a.val.kl_cycles = 1;
  a.val.lr_schedule = RVAE_LR_CONSTANT; a.val.kl_anneal = RVAE_KL_CONSTANT;
  return a;
}

__device__ __forceinline__ void loss_finalize_body(double* acc, double inv_rec, double kl_scale, float* loss_out,
                                                   int ring_size, float* step, int inc_step) {
  const double loss = acc[0] * inv_rec + kl_scale * acc[1];
  // ring_size > 1: slot = (step count before this step) mod ring_size, so a replayed CUDA graph still lands every
  // step's loss in its own slot without the host passing a new pointer
  const int slot = (ring_size > 1 && step) ? static_cast<int>(static_cast<long long>(*step) % ring_size) : 0;
  if (loss_out) loss_out[slot] = static_cast<float>(loss);
  acc[0] = 0.0;
  acc[1] = 0.0;
  if (step && inc_step) *step += 1.0f;
}

// kl_scale of a finalisation: the host's value, or -0.5 * beta(k) / (B L) from the record at k = *step
__device__ __forceinline__ double loss_kl_scale(const LossFinalize& f) {
  if (f.hp == nullptr) return f.kl_scale;
  double lr;
  float beta;
  hparams_eval(*f.hp, static_cast<double>(*f.step), &lr, &beta);
  return __ddiv_rn(__dmul_rn(-0.5, static_cast<double>(beta)), f.kl_bl);
}

__global__ void loss_finalize_kernel(LossFinalize f) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  if (threadIdx.x == 0 && blockIdx.x == 0)
    loss_finalize_body(f.acc, f.inv_rec, loss_kl_scale(f), f.loss_out, f.ring_size, f.step, f.inc_step);
}

LossFinalize make_loss_finalize(double* acc, int64_t B, int S, int L, float beta, float* loss_out, int ring_size,
                                float* step) {
  LossFinalize f;
  f.acc = acc;
  f.inv_rec = 1.0 / (static_cast<double>(B) * S);
  f.kl_scale = -0.5 * static_cast<double>(beta) / (static_cast<double>(B) * L);
  f.loss_out = loss_out;
  f.ring_size = ring_size;
  f.step = step;
  f.inc_step = 1;
  f.hp = nullptr;
  f.kl_bl = static_cast<double>(B) * L;
  return f;
}

int launch_loss_finalize(Ctx* ctx, double* acc, int64_t B, int S, int L, float beta, float* loss_out, int ring_size,
                         float* step, cudaStream_t stream) {
  RVAE_REQUIRE(acc, RVAE_ERR_INVALID, "loss_finalize: null accumulator");
  return launch_loss_finalize_prepared(ctx, make_loss_finalize(acc, B, S, L, beta, loss_out, ring_size, step), stream);
}

int launch_loss_finalize_prepared(Ctx* ctx, const LossFinalize& f, cudaStream_t stream) {
  RVAE_REQUIRE(f.acc, RVAE_ERR_INVALID, "loss_finalize: null accumulator");
  RVAE_REQUIRE(f.hp == nullptr || f.step != nullptr, RVAE_ERR_INVALID, "loss_finalize: a record needs the step counter");
  RVAE_CUDA(launch_kernel(ctx, loss_finalize_kernel, dim3(1), dim3(32), (size_t)0, stream, f));
  RVAE_LAUNCH_CHECK(ctx);
  return RVAE_OK;
}

int launch_loss_fwd(Ctx* ctx, const float* xhat, const float* x, const float* mu, const float* lv, int64_t B, int S,
                    int L, float beta, double* acc, float* loss_out, cudaStream_t stream) {
  RVAE_REQUIRE(xhat && x && mu && lv && acc && loss_out, RVAE_ERR_INVALID, "loss_fwd: null buffer");
  RVAE_REQUIRE(B > 0, RVAE_ERR_INVALID, "loss_fwd: empty batch");
  RVAE_CUDA(cudaMemsetAsync(acc, 0, 2 * sizeof(double), stream));
  const int threads = 256;
  const int grid = grid_for(ctx, B * S / 4, threads, 4);
  RVAE_CUDA(launch_kernel(ctx, loss_fwd_kernel, dim3(grid), dim3(threads), (size_t)0, stream, xhat, x, mu, lv, B * S, B * L, acc));
  RVAE_LAUNCH_CHECK(ctx);
  return launch_loss_finalize(ctx, acc, B, S, L, beta, loss_out, 1, nullptr, stream);
}

// ------------------------------------------------------------------------------------------------
// K-L3 per-frame loss of held-out audio (rawvae/model.py:38-46 per frame, no mean over the batch):
//   rec[f] = (1/S) sum_s (xhat[f,s] - x[f,s])^2,   kl[f] = -(0.5/L) sum_l (1 + lv[f,l] - mu[f,l]^2 - exp(lv[f,l]))
// x is framed straight from the audio (the rule of frame_gather_kernel: exact fp32 or int16 / 32768 samples, zeros
// at and beyond n_samples), so no bf16 rounding of x enters the score. One warp owns a frame: every lane sums a
// fixed set of columns, then a fixed shuffle tree combines the lanes - no atomics, repeated calls are bitwise equal.
// The differences and KL terms are fp32, as in the reference; their sums are fp64.
// VEC: S, ld_xhat and hop multiples of 4, xhat / audio 16-byte (int16: 8-byte) aligned: 4 columns per load.
// ------------------------------------------------------------------------------------------------
template <bool I16>
__device__ __forceinline__ float audio_sample(const void* audio, int64_t i, int64_t n_samples) {
  if (i >= n_samples) return 0.f;
  if constexpr (I16) return __ldg(reinterpret_cast<const int16_t*>(audio) + i) * (1.0f / 32768.0f);
  else return __ldg(reinterpret_cast<const float*>(audio) + i);
}

template <bool I16, bool VEC>
__global__ void frame_loss_kernel(const float* __restrict__ xhat, int ld_xhat, const float* __restrict__ mu,
                                  const float* __restrict__ lv, int ld_lat, int64_t rows, int S, int L,
                                  const void* __restrict__ audio, int64_t n_samples, int64_t first_frame, int hop,
                                  float* __restrict__ rec_out, float* __restrict__ kl_out) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t f = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5); f < rows; f += warps) {
    const float* xr = xhat + f * ld_xhat;
    const int64_t s0 = (first_frame + f) * hop;
    double rec = 0.0;
    if constexpr (VEC) {
#pragma unroll 4
      for (int c = lane * 4; c < S; c += 128) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(xr + c));
        const int64_t si = s0 + c;
        float b[4];
        if (si + 4 <= n_samples) {
          if constexpr (I16) {
            const uint2 r = __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const int16_t*>(audio) + si));
            const int16_t* h = reinterpret_cast<const int16_t*>(&r);
#pragma unroll
            for (int j = 0; j < 4; ++j) b[j] = h[j] * (1.0f / 32768.0f);
          } else {
            const float4 r = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(audio) + si));
            b[0] = r.x; b[1] = r.y; b[2] = r.z; b[3] = r.w;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j) b[j] = audio_sample<I16>(audio, si + j, n_samples);
        }
        const float d0 = a.x - b[0], d1 = a.y - b[1], d2 = a.z - b[2], d3 = a.w - b[3];
        rec = fma((double)d0, (double)d0, rec);
        rec = fma((double)d1, (double)d1, rec);
        rec = fma((double)d2, (double)d2, rec);
        rec = fma((double)d3, (double)d3, rec);
      }
    } else {
#pragma unroll 4
      for (int c = lane; c < S; c += 32) {
        const float d = __ldg(xr + c) - audio_sample<I16>(audio, s0 + c, n_samples);
        rec = fma((double)d, (double)d, rec);
      }
    }
    const float* mr = mu + f * ld_lat;
    const float* lr = lv + f * ld_lat;
    double kl = 0.0;
    for (int l = lane; l < L; l += 32) {
      const float m = __ldg(mr + l), v = __ldg(lr + l);
      kl += (double)(1.f + v - m * m - expf(v));
    }
    rec = warp_sum_f64(rec);
    kl = warp_sum_f64(kl);
    if (lane == 0) {
      rec_out[f] = static_cast<float>(rec / S);
      kl_out[f] = static_cast<float>(-0.5 * kl / L);
    }
  }
}

int launch_frame_loss(Ctx* ctx, const float* xhat, int ld_xhat, const float* mu, const float* lv, int ld_lat,
                      int64_t rows, int S, int L, const void* audio, int audio_is_i16, int64_t n_samples,
                      int64_t first_frame, int hop, float* rec_out, float* kl_out, cudaStream_t stream) {
  const int threads = 256;   // 8 frames in flight per block
  const int grid = grid_for(ctx, rows * 32, threads, 8);
  const uintptr_t align = audio_is_i16 ? 7 : 15;
  const bool vec = S % 4 == 0 && ld_xhat % 4 == 0 && hop % 4 == 0 &&
                   (reinterpret_cast<uintptr_t>(xhat) & 15) == 0 && (reinterpret_cast<uintptr_t>(audio) & align) == 0;
  auto go = [&](auto kern) {
    return launch_kernel(ctx, kern, dim3(grid), dim3(threads), (size_t)0, stream, xhat, ld_xhat, mu, lv, ld_lat, rows,
                         S, L, audio, n_samples, first_frame, hop, rec_out, kl_out);
  };
  if (audio_is_i16) {
    if (vec) RVAE_CUDA(go(frame_loss_kernel<true, true>));
    else RVAE_CUDA(go(frame_loss_kernel<true, false>));
  } else {
    if (vec) RVAE_CUDA(go(frame_loss_kernel<false, true>));
    else RVAE_CUDA(go(frame_loss_kernel<false, false>));
  }
  RVAE_LAUNCH_CHECK(ctx);
  return RVAE_OK;
}

// d loss / d xhat, mu, logvar scaled by the upstream gradient (a device scalar; nullptr = 1).
__global__ void loss_bwd_kernel(const float* __restrict__ xhat, const float* __restrict__ x,
                                const float* __restrict__ mu, const float* __restrict__ lv, int64_t n_rec,
                                int64_t n_lat, float c_rec, float c_kl, const float* __restrict__ grad_out,
                                float* __restrict__ g_xhat, float* __restrict__ g_mu, float* __restrict__ g_lv) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  const float g = grad_out ? __ldg(grad_out) : 1.f;
  const float cr = c_rec * g, ck = c_kl * g;
  const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t nv = n_rec >> 2;
  for (int64_t i = tid; i < nv; i += stride) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(xhat) + i);
    const float4 b = __ldg(reinterpret_cast<const float4*>(x) + i);
    reinterpret_cast<float4*>(g_xhat)[i] =
        make_float4(cr * (a.x - b.x), cr * (a.y - b.y), cr * (a.z - b.z), cr * (a.w - b.w));
  }
  for (int64_t i = (nv << 2) + tid; i < n_rec; i += stride) g_xhat[i] = cr * (xhat[i] - x[i]);
  for (int64_t i = tid; i < n_lat; i += stride) {
    g_mu[i] = ck * mu[i];
    g_lv[i] = 0.5f * ck * (expf(lv[i]) - 1.f);
  }
}

int launch_loss_bwd(Ctx* ctx, const float* xhat, const float* x, const float* mu, const float* lv, int64_t B, int S,
                    int L, float beta, const float* grad_out, float* g_xhat, float* g_mu, float* g_lv,
                    cudaStream_t stream) {
  RVAE_REQUIRE(xhat && x && mu && lv && g_xhat && g_mu && g_lv, RVAE_ERR_INVALID, "loss_bwd: null buffer");
  RVAE_REQUIRE(B > 0, RVAE_ERR_INVALID, "loss_bwd: empty batch");
  const float c_rec = static_cast<float>(2.0 / (static_cast<double>(B) * S));
  const float c_kl = static_cast<float>(static_cast<double>(beta) / (static_cast<double>(B) * L));
  const int threads = 256;
  RVAE_CUDA(launch_kernel(ctx, loss_bwd_kernel, dim3(grid_for(ctx, B * S / 4, threads, 8)), dim3(threads), (size_t)0, stream, xhat, x, mu, lv, B * S, B * L, c_rec,
                                                                              c_kl, grad_out, g_xhat, g_mu, g_lv));
  RVAE_LAUNCH_CHECK(ctx);
  return RVAE_OK;
}

// da4 = g_xhat * (1 - xhat^2) as bf16 planes (operand of the fc4 dgrad / wgrad GEMMs).
__global__ void tanh_bwd_kernel(const float* __restrict__ g, const float* __restrict__ xhat, int64_t n,
                                __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  const int64_t nvec = n >> 3;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nvec; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 g0 = __ldg(reinterpret_cast<const float4*>(g) + 2 * i);
    const float4 g1 = __ldg(reinterpret_cast<const float4*>(g) + 2 * i + 1);
    const float4 x0 = __ldg(reinterpret_cast<const float4*>(xhat) + 2 * i);
    const float4 x1 = __ldg(reinterpret_cast<const float4*>(xhat) + 2 * i + 1);
    const float gv[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
    const float xv[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = gv[j] * (1.f - xv[j] * xv[j]);
    reinterpret_cast<uint4*>(hi)[i] =
        make_uint4(pack2(v[0], v[1]), pack2(v[2], v[3]), pack2(v[4], v[5]), pack2(v[6], v[7]));
    if (lo) {
      float r[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) r[j] = v[j] - __bfloat162float(__float2bfloat16_rn(v[j]));
      reinterpret_cast<uint4*>(lo)[i] =
          make_uint4(pack2(r[0], r[1]), pack2(r[2], r[3]), pack2(r[4], r[5]), pack2(r[6], r[7]));
    }
  }
}

int launch_tanh_bwd(Ctx* ctx, const float* g_xhat, const float* xhat, int64_t n, __nv_bfloat16* da_hi,
                    __nv_bfloat16* da_lo, cudaStream_t stream) {
  RVAE_REQUIRE(g_xhat && xhat && da_hi, RVAE_ERR_INVALID, "tanh_bwd: null buffer");
  RVAE_REQUIRE(n % 8 == 0, RVAE_ERR_UNSUPPORTED, "tanh_bwd: element count must be a multiple of 8");
  if (n <= 0) return RVAE_OK;
  const int threads = 256;
  RVAE_CUDA(launch_kernel(ctx, tanh_bwd_kernel, dim3(grid_for(ctx, n / 8, threads, 8)), dim3(threads), (size_t)0, stream, g_xhat, xhat, n, da_hi, da_lo));
  RVAE_LAUNCH_CHECK(ctx);
  return RVAE_OK;
}

// Standalone reparameterisation z = mu + eps * exp(logvar / 2) (rawvae/model.py:23-26) for the inference API.
__global__ void reparam_kernel(const float* __restrict__ mu, const float* __restrict__ lv,
                               const float* __restrict__ eps, int64_t n, float* __restrict__ z) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  const int64_t nv = n >> 2;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nv; i += stride) {
    const float4 m = __ldcs(reinterpret_cast<const float4*>(mu) + i);
    const float4 l = __ldcs(reinterpret_cast<const float4*>(lv) + i);
    const float4 e = __ldcs(reinterpret_cast<const float4*>(eps) + i);
    reinterpret_cast<float4*>(z)[i] = make_float4(fmaf(e.x, expf(0.5f * l.x), m.x), fmaf(e.y, expf(0.5f * l.y), m.y),
                                                  fmaf(e.z, expf(0.5f * l.z), m.z), fmaf(e.w, expf(0.5f * l.w), m.w));
  }
  for (int64_t i = (nv << 2) + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += stride)
    z[i] = fmaf(eps[i], expf(0.5f * lv[i]), mu[i]);
}

int launch_reparam(Ctx* ctx, const float* mu, const float* lv, const float* eps, int64_t n, float* z,
                   cudaStream_t stream) {
  RVAE_REQUIRE(mu && lv && eps && z, RVAE_ERR_INVALID, "reparam: null buffer");
  RVAE_REQUIRE(((reinterpret_cast<uintptr_t>(mu) | reinterpret_cast<uintptr_t>(lv) | reinterpret_cast<uintptr_t>(eps) |
                 reinterpret_cast<uintptr_t>(z)) & 15) == 0, RVAE_ERR_INVALID, "reparam: buffers must be 16-byte aligned");
  if (n <= 0) return RVAE_OK;
  const int threads = 256;
  RVAE_CUDA(launch_kernel(ctx, reparam_kernel, dim3(grid_for(ctx, (n + 3) / 4, threads, 8)), dim3(threads), (size_t)0, stream, mu, lv, eps, n, z));
  RVAE_LAUNCH_CHECK(ctx);
  return RVAE_OK;
}

// Latent interpolation of the tutorial's inference pattern (tutorial.ipynb:496-510 global alpha, :905-932 per-frame
// alpha from interp1d, float64): mu = (1-a) mu_a + a mu_b, logvar likewise, z = mu + eps * exp(logvar / 2), with one
// alpha per FRAME (row). Emits z as fp32 and / or as the bf16 planes fc3's GEMM reads, so the interpolated latents
// never make an fp32 round trip through HBM before decode. The lerp itself is done in double when alpha is double
// (the notebook's dtype), then rounded to fp32 once.
template <typename AT>
__global__ void lerp_reparam_kernel(const float* __restrict__ mu_a, const float* __restrict__ lv_a,
                                    const float* __restrict__ mu_b, const float* __restrict__ lv_b,
                                    const AT* __restrict__ alpha, const float* __restrict__ eps, int64_t rows, int L,
                                    float* __restrict__ z_f32, __nv_bfloat16* __restrict__ z_hi,
                                    __nv_bfloat16* __restrict__ z_lo, float* __restrict__ mu_out,
                                    float* __restrict__ lv_out) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  const int q = L >> 2;
  const int64_t nv = rows * q;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nv; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / q;
    const AT al = alpha[r];
    const float4 ma = __ldcs(reinterpret_cast<const float4*>(mu_a) + i), mb = __ldcs(reinterpret_cast<const float4*>(mu_b) + i);
    const float4 la = __ldcs(reinterpret_cast<const float4*>(lv_a) + i), lb = __ldcs(reinterpret_cast<const float4*>(lv_b) + i);
    float4 e = make_float4(0.f, 0.f, 0.f, 0.f);
    if (eps) e = __ldcs(reinterpret_cast<const float4*>(eps) + i);
    const float* pma = reinterpret_cast<const float*>(&ma); const float* pmb = reinterpret_cast<const float*>(&mb);
    const float* pla = reinterpret_cast<const float*>(&la); const float* plb = reinterpret_cast<const float*>(&lb);
    const float* pe = reinterpret_cast<const float*>(&e);
    float m[4], l[4], z[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      m[j] = static_cast<float>((AT(1) - al) * AT(pma[j]) + al * AT(pmb[j]));
      l[j] = static_cast<float>((AT(1) - al) * AT(pla[j]) + al * AT(plb[j]));
      z[j] = fmaf(pe[j], expf(0.5f * l[j]), m[j]);
    }
    if (mu_out) reinterpret_cast<float4*>(mu_out)[i] = make_float4(m[0], m[1], m[2], m[3]);
    if (lv_out) reinterpret_cast<float4*>(lv_out)[i] = make_float4(l[0], l[1], l[2], l[3]);
    if (z_f32) reinterpret_cast<float4*>(z_f32)[i] = make_float4(z[0], z[1], z[2], z[3]);
    if (z_hi) reinterpret_cast<uint2*>(z_hi)[i] = make_uint2(pack2(z[0], z[1]), pack2(z[2], z[3]));
    if (z_lo) {
      float rr[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) rr[j] = z[j] - __bfloat162float(__float2bfloat16_rn(z[j]));
      reinterpret_cast<uint2*>(z_lo)[i] = make_uint2(pack2(rr[0], rr[1]), pack2(rr[2], rr[3]));
    }
  }
}

// Any L: one thread per element of [rows, ld_z]. The fp32 outputs are [rows, L]; the bf16 z planes have row pitch
// ld_z >= L and zeros in columns L..ld_z (fc3's operand of a plan whose latent_dim is not a multiple of 64). Same
// arithmetic as the vector kernel, so the same bits.
template <typename AT>
__global__ void lerp_reparam_rows_kernel(const float* __restrict__ mu_a, const float* __restrict__ lv_a,
                                         const float* __restrict__ mu_b, const float* __restrict__ lv_b,
                                         const AT* __restrict__ alpha, const float* __restrict__ eps, int64_t rows,
                                         int L, int ld_z, float* __restrict__ z_f32, __nv_bfloat16* __restrict__ z_hi,
                                         __nv_bfloat16* __restrict__ z_lo, float* __restrict__ mu_out,
                                         float* __restrict__ lv_out) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  const int64_t n = rows * ld_z;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / ld_z;
    const int c = static_cast<int>(i - r * ld_z);
    float z = 0.f;
    if (c < L) {
      const int64_t k = r * L + c;
      const AT al = alpha[r];
      const float e = eps ? eps[k] : 0.f;
      const float m = static_cast<float>((AT(1) - al) * AT(mu_a[k]) + al * AT(mu_b[k]));
      const float l = static_cast<float>((AT(1) - al) * AT(lv_a[k]) + al * AT(lv_b[k]));
      z = fmaf(e, expf(0.5f * l), m);
      if (mu_out) mu_out[k] = m;
      if (lv_out) lv_out[k] = l;
      if (z_f32) z_f32[k] = z;
    }
    if (z_hi) z_hi[i] = __float2bfloat16_rn(z);
    if (z_lo) z_lo[i] = __float2bfloat16_rn(z - __bfloat162float(__float2bfloat16_rn(z)));
  }
}

int launch_lerp_reparam(Ctx* ctx, const float* mu_a, const float* lv_a, const float* mu_b, const float* lv_b,
                        const void* alpha, int alpha_is_f64, const float* eps, int64_t rows, int L, int ld_z,
                        float* z_f32, __nv_bfloat16* z_hi, __nv_bfloat16* z_lo, float* mu_out, float* lv_out,
                        cudaStream_t stream) {
  RVAE_REQUIRE(mu_a && lv_a && mu_b && lv_b && alpha, RVAE_ERR_INVALID, "lerp_reparam: null buffer");
  RVAE_REQUIRE(z_f32 || z_hi || mu_out, RVAE_ERR_INVALID, "lerp_reparam: no output buffer");
  RVAE_REQUIRE(L > 0 && ld_z >= L, RVAE_ERR_UNSUPPORTED, "lerp_reparam: latent_dim=%d, z row pitch %d", L, ld_z);
  if (rows <= 0) return RVAE_OK;
  const int threads = 256;
  const bool vec = L % 4 == 0 && ld_z == L &&
                   ((reinterpret_cast<uintptr_t>(mu_a) | reinterpret_cast<uintptr_t>(lv_a) | reinterpret_cast<uintptr_t>(mu_b) |
                     reinterpret_cast<uintptr_t>(lv_b) | reinterpret_cast<uintptr_t>(eps) | reinterpret_cast<uintptr_t>(z_f32) |
                     reinterpret_cast<uintptr_t>(mu_out) | reinterpret_cast<uintptr_t>(lv_out)) & 15) == 0;
  if (!vec) {
    const dim3 grid(grid_for(ctx, rows * ld_z, threads, 8));
    if (alpha_is_f64)
      RVAE_CUDA(launch_kernel(ctx, lerp_reparam_rows_kernel<double>, grid, dim3(threads), (size_t)0, stream, mu_a, lv_a,
                              mu_b, lv_b, reinterpret_cast<const double*>(alpha), eps, rows, L, ld_z, z_f32, z_hi, z_lo,
                              mu_out, lv_out));
    else
      RVAE_CUDA(launch_kernel(ctx, lerp_reparam_rows_kernel<float>, grid, dim3(threads), (size_t)0, stream, mu_a, lv_a,
                              mu_b, lv_b, reinterpret_cast<const float*>(alpha), eps, rows, L, ld_z, z_f32, z_hi, z_lo,
                              mu_out, lv_out));
    RVAE_LAUNCH_CHECK(ctx);
    return RVAE_OK;
  }
  const dim3 grid(grid_for(ctx, rows * (L / 4), threads, 8));
  if (alpha_is_f64)
    RVAE_CUDA(launch_kernel(ctx, lerp_reparam_kernel<double>, grid, dim3(threads), (size_t)0, stream, mu_a, lv_a, mu_b, lv_b,
                            reinterpret_cast<const double*>(alpha), eps, rows, L, z_f32, z_hi, z_lo, mu_out, lv_out));
  else
    RVAE_CUDA(launch_kernel(ctx, lerp_reparam_kernel<float>, grid, dim3(threads), (size_t)0, stream, mu_a, lv_a, mu_b, lv_b,
                            reinterpret_cast<const float*>(alpha), eps, rows, L, z_f32, z_hi, z_lo, mu_out, lv_out));
  RVAE_LAUNCH_CHECK(ctx);
  return RVAE_OK;
}

// ------------------------------------------------------------------------------------------------
// K-A1 fused Adam (torch.optim.Adam defaults semantics, train.py:163,193): one pass over the flat parameter
// buffer, float4 loads/stores (28 B/param), optionally re-emitting the bf16 shadow planes the GEMMs read.
//   t = *step (already incremented); m = m + (1-b1)(g-m); v = b2 v + (1-b2) g^2;
//   p -= (lr / (1-b1^t)) * m / (sqrt(v)/sqrt(1-b2^t) + eps)
// ------------------------------------------------------------------------------------------------
// A launch covers elements [0, n) and, optionally, a second segment [off_b, off_b + n_b) of the same buffers (both
// multiples of 4 then): the per-bucket launches of a training step (W3|W4, W2, W1 + bias block).
// (4 blocks of 256 threads per SM need <= 64 registers: one register more costs a quarter of the occupancy and 30 % of
// the bandwidth - measured when the hyper-parameters became doubles)
// The hyper-parameters come from a record (HpArg: the device record of a scheduled step, read here when the kernel
// runs, or a constant record passed by value); lr is the schedule's lr(k) at k = t - 1.
// EMA = true (the training step with rvae_plan_set_ema): the launch also moves the exponential moving average e of the
// parameters toward the p it has just computed (ema_lerp), 8 more bytes per parameter; p, m and v come from the same
// adam_update as without it, so they do not change by a bit.

// One Adam update of an element, shared by both instantiations of adam_kernel
__device__ __forceinline__ void adam_update(float& p, float& m, float& v, float g, float grad_scale,
                                            float weight_decay, float omb1, float beta2, float omb2, float sqrt_bc2,
                                            float eps, float step_size) {
  float gr = g * grad_scale;
  if (weight_decay != 0.f) gr = fmaf(weight_decay, p, gr);
  m = m + omb1 * (gr - m);
  v = beta2 * v + omb2 * gr * gr;
  const float denom = sqrtf(v) / sqrt_bc2 + eps;
  p = p - step_size * (m / denom);
}

// One EMA update of an element, as torch.optim.swa_utils.AveragedModel with get_ema_multi_avg_fn: a copy of p on the
// first update, else torch.lerp(e, p, w) with w = 1 - decay (torch's two-branch formula, contracted as nvcc
// contracts torch's CUDA lerp)
__device__ __forceinline__ float ema_lerp(float e, float p, float w, bool first) {
  if (first) return p;
  const float d = p - e;
  return fabsf(w) < 0.5f ? fmaf(w, d, e) : fmaf(-d, 1.0f - w, p);
}

// The EMA's scalars, read by thread 0 of a block: w = fp32(1 - decay) (formed in double, rounded once, as a python
// float reaches torch._foreach_lerp_) and whether this is the first update (n_averaged == 0)
__device__ __forceinline__ void ema_consts(const EmaArg& ema, float* w, float* first) {
  const double decay = *reinterpret_cast<const volatile double*>(ema.decay);
  *w = static_cast<float>(1.0 - decay);
  *first = *reinterpret_cast<const volatile int64_t*>(ema.count) == 0 ? 1.f : 0.f;
}

template <int U, bool EMA>
__global__ void __launch_bounds__(256, U == 4 ? 2 : 4) adam_kernel(float* __restrict__ p, float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, int64_t n, int64_t off_b, int64_t n_b, const __grid_constant__ HpArg hp,
                            float grad_scale, const float* coef, float* step, int step_bias, unsigned int* ticket,
                            __nv_bfloat16* __restrict__ sh_hi, __nv_bfloat16* __restrict__ sh_lo, int zero_grads,
                            AuxTrace tr, const __grid_constant__ EmaArg ema) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();   // (rvae_adam_step follows the launch that advances the step counter)
  aux_begin(tr, 4);
  // The hyper-parameters are doubles - what torch.optim.Adam holds (python floats) - and every scalar the update uses
  // is derived from them exactly as torch derives it: 1 - beta in DOUBLE, then rounded to fp32 (the weight of lerp_ /
  // the value of addcmul_; (1.f - 0.999f) would be off by 1.3e-5 relative), beta2 and eps rounded to fp32. Bias
  // corrections in double, as torch computes them on the host (python floats). One thread per block reads the record,
  // does the fp64 pow()s and broadcasts the seven scalars. coef != nullptr: the gradient-clipping factor of the step
  // (grad_norm_kernel), folded into the gradient scale - g * coef in fp32, as torch.nn.utils.clip_grad_norm_ scales g.
  __shared__ float s_consts[EMA ? 10 : 8];
  if (threadIdx.x == 0) {
    if constexpr (EMA) ema_consts(ema, &s_consts[8], &s_consts[9]);
    const rvae_hparams& h = hp.dev != nullptr ? *hp.dev : hp.val;
    // t = *step + step_bias: step_bias = 1 when the step counter is advanced only at the end of the step (ticket)
    const double t = static_cast<double>(*reinterpret_cast<volatile float*>(step)) + step_bias;
    double lr;
    float beta_unused;
    hparams_eval(h, t - 1.0, &lr, &beta_unused);
    const double bc1 = 1.0 - pow(h.beta1, t);
    const double bc2 = 1.0 - pow(h.beta2, t);
    s_consts[0] = static_cast<float>(lr / bc1);
    s_consts[1] = static_cast<float>(sqrt(bc2));
    s_consts[2] = static_cast<float>(1.0 - h.beta1);
    s_consts[3] = static_cast<float>(h.beta2);
    s_consts[4] = static_cast<float>(1.0 - h.beta2);
    s_consts[5] = static_cast<float>(h.eps);
    s_consts[6] = static_cast<float>(h.weight_decay);
    s_consts[7] = coef != nullptr ? grad_scale * *coef : grad_scale;
  }
  __syncthreads();
  grad_scale = s_consts[7];
  const float step_size = s_consts[0];
  const float sqrt_bc2 = s_consts[1];
  const float omb1 = s_consts[2], beta2 = s_consts[3], omb2 = s_consts[4], eps = s_consts[5];
  const float weight_decay = s_consts[6];
  const float ema_w = EMA ? s_consts[EMA ? 8 : 0] : 0.f;
  const bool ema_first = EMA && s_consts[EMA ? 9 : 0] != 0.f;
  const int64_t nvec = n >> 2;
  const int64_t nvec_all = nvec + (n_b >> 2);
  const int64_t shift_b = (off_b >> 2) - nvec;
  // U (= 2) float4 groups per thread and trip, all 4 U loads issued before the first use: loads and the previous trip's
  // stores overlap in time, so the kernel streams instead of alternating between a read phase and a write phase.
  // p, m, v are touched once per step: streaming (evict-first) loads and stores keep them from displacing the
  // activations and bf16 shadow weights the GEMMs want in L2. The cleared gradient and the shadow use the default
  // policy: the next step's split-K reduce-adds and operand loads hit them in L2.
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t w0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; w0 < nvec_all; w0 += U * stride) {
    int64_t idx[U];
    float4 pp[U], gg[U], mm[U], vv[U];
    float4 ee[EMA ? U : 1];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t w = w0 + u * stride;
      idx[u] = w < nvec_all ? (w < nvec ? w : w + shift_b) : -1;
      if (idx[u] >= 0) {
        pp[u] = __ldcs(reinterpret_cast<const float4*>(p) + idx[u]);
        gg[u] = __ldcs(reinterpret_cast<const float4*>(g) + idx[u]);
        mm[u] = __ldcs(reinterpret_cast<const float4*>(m) + idx[u]);
        vv[u] = __ldcs(reinterpret_cast<const float4*>(v) + idx[u]);
        if constexpr (EMA) ee[u] = __ldcs(reinterpret_cast<const float4*>(ema.e) + idx[u]);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (idx[u] < 0) continue;
      const int64_t i = idx[u];
      float* pa = reinterpret_cast<float*>(&pp[u]);
      const float* ga = reinterpret_cast<const float*>(&gg[u]);
      float* ma = reinterpret_cast<float*>(&mm[u]);
      float* va = reinterpret_cast<float*>(&vv[u]);
#pragma unroll
      for (int j = 0; j < 4; ++j)
        adam_update(pa[j], ma[j], va[j], ga[j], grad_scale, weight_decay, omb1, beta2, omb2, sqrt_bc2, eps, step_size);
      __stcs(reinterpret_cast<float4*>(p) + i, pp[u]);
      __stcs(reinterpret_cast<float4*>(m) + i, mm[u]);
      __stcs(reinterpret_cast<float4*>(v) + i, vv[u]);
      if constexpr (EMA) {
        float* ea = reinterpret_cast<float*>(&ee[EMA ? u : 0]);
#pragma unroll
        for (int j = 0; j < 4; ++j) ea[j] = ema_lerp(ea[j], pa[j], ema_w, ema_first);
        __stcs(reinterpret_cast<float4*>(ema.e) + i, ee[EMA ? u : 0]);
      }
      // zero_grads: the next step's split-K weight gradients reduce-add into this buffer (saves 4 memsets / step)
      if (zero_grads) reinterpret_cast<float4*>(g)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (sh_hi) {
        reinterpret_cast<uint2*>(sh_hi)[i] = make_uint2(pack2(pa[0], pa[1]), pack2(pa[2], pa[3]));
        if (sh_lo) {
          float r[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) r[j] = pa[j] - __bfloat162float(__float2bfloat16_rn(pa[j]));
          reinterpret_cast<uint2*>(sh_lo)[i] = make_uint2(pack2(r[0], r[1]), pack2(r[2], r[3]));
        }
      }
    }
  }
  if (blockIdx.x == 0) {
    for (int64_t j = (nvec << 2) + threadIdx.x; j < n; j += blockDim.x) {
      const float gj = g[j];
      float pj = p[j], mj = m[j], vj = v[j];
      adam_update(pj, mj, vj, gj, grad_scale, weight_decay, omb1, beta2, omb2, sqrt_bc2, eps, step_size);
      m[j] = mj; v[j] = vj; p[j] = pj;
      if constexpr (EMA) ema.e[j] = ema_lerp(ema.e[j], pj, ema_w, ema_first);
      if (zero_grads) g[j] = 0.f;
      if (sh_hi) {
        const __nv_bfloat16 h = __float2bfloat16_rn(pj);
        sh_hi[j] = h;
        if (sh_lo) sh_lo[j] = __float2bfloat16_rn(pj - __bfloat162float(h));
      }
    }
  }
  aux_end(tr);
  if (ticket != nullptr) {
    // the LAST block to finish advances the step counter: every block (of this and of the earlier per-bucket
    // launches of the step, which the host joined before this launch) has read it by then
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence();
      const unsigned int done = atomicAdd(ticket, 1u);
      if (done == gridDim.x - 1) {
        *ticket = 0u;
        *step = *reinterpret_cast<volatile float*>(step) + 1.0f;
        // n_averaged advances with the step counter, once per step, after every EMA launch of the step has read it
        if constexpr (EMA) *ema.count = *reinterpret_cast<volatile int64_t*>(ema.count) + 1;
      }
    }
  }
}

int launch_adam(Ctx* ctx, float* p, float* g, float* m, float* v, int64_t n, double lr, double beta1, double beta2,
                double eps, double weight_decay, float grad_scale, const float* step, __nv_bfloat16* shadow_hi,
                __nv_bfloat16* shadow_lo, int zero_grads, cudaStream_t stream) {
  return launch_adam2(ctx, p, g, m, v, n, 0, 0, hp_value(lr, beta1, beta2, eps, weight_decay), grad_scale, nullptr,
                      const_cast<float*>(step), 0, nullptr, shadow_hi, shadow_lo, zero_grads, EmaArg{}, stream);
}

int launch_adam2(Ctx* ctx, float* p, float* g, float* m, float* v, int64_t n, int64_t off_b, int64_t n_b,
                 const HpArg& hp, float grad_scale, const float* coef, float* step, int step_bias, unsigned int* ticket,
                 __nv_bfloat16* shadow_hi, __nv_bfloat16* shadow_lo, int zero_grads, const EmaArg& ema,
                 cudaStream_t stream) {
  RVAE_REQUIRE(p && g && m && v && step, RVAE_ERR_INVALID, "adam: null buffer");
  RVAE_REQUIRE(ema.e == nullptr || (ema.decay && ema.count && (reinterpret_cast<uintptr_t>(ema.e) & 15) == 0),
               RVAE_ERR_INVALID, "adam: the EMA buffer must be 16-byte aligned, with its decay and count");
  RVAE_REQUIRE(n_b == 0 || ((n & 3) == 0 && (off_b & 3) == 0 && (n_b & 3) == 0 && off_b >= n), RVAE_ERR_INVALID,
               "adam: segments must be multiples of 4 elements");
  RVAE_REQUIRE(((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(m) |
                 reinterpret_cast<uintptr_t>(v)) & 15) == 0,
               RVAE_ERR_INVALID, "adam: p/g/m/v must be 16-byte aligned");
  RVAE_REQUIRE(((reinterpret_cast<uintptr_t>(shadow_hi) | reinterpret_cast<uintptr_t>(shadow_lo)) & 7) == 0,
               RVAE_ERR_INVALID, "adam: shadow planes must be 8-byte aligned");
  if (n + n_b <= 0) return RVAE_OK;
  const int threads = 256;
  // one wave of 4 blocks per SM (a multiple of the SM count); each thread walks ~10 float4 groups at the default
  // sizes. RVAE_ADAM_UNROLL / RVAE_ADAM_BPS: tuning knobs (tools/ncu_hbm_kernels.py sweeps them).
  static const int unroll = getenv("RVAE_ADAM_UNROLL") ? atoi(getenv("RVAE_ADAM_UNROLL")) : 2;
  static const int bps = getenv("RVAE_ADAM_BPS") ? atoi(getenv("RVAE_ADAM_BPS")) : 4;
  const int64_t groups = (n + n_b + 3) / 4;
  dim3 grid(grid_for(ctx, (groups + unroll - 1) / unroll, threads, bps > 0 ? bps : 4));
  if (ctx->aux_grid_cap > 0 && (int)grid.x > ctx->aux_grid_cap) grid.x = ctx->aux_grid_cap;
  auto kern = unroll == 1 ? adam_kernel<1, false> : (unroll == 4 ? adam_kernel<4, false> : adam_kernel<2, false>);
  if (ema.e != nullptr)
    kern = unroll == 1 ? adam_kernel<1, true> : (unroll == 4 ? adam_kernel<4, true> : adam_kernel<2, true>);
  RVAE_CUDA(launch_kernel(ctx, kern, grid, dim3(threads), (size_t)0,
                          stream, p, g, m, v, n, off_b, n_b, hp, grad_scale, coef, step, step_bias, ticket, shadow_hi,
                          shadow_lo, zero_grads, next_aux(ctx, 4), ema));
  RVAE_LAUNCH_CHECK(ctx);
  return RVAE_OK;
}

// ------------------------------------------------------------------------------------------------
// Standalone EMA update (rvae_ema_update): e = ema_lerp(e, p) over a flat buffer, with the device function of the EMA
// Adam launch - the update that follows an optimizer step of the unfused path. float4 loads and stores (12 B/param,
// streaming), a grid of 1 to 4 blocks per SM; the last block to finish advances n_averaged (ticket).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) ema_update_kernel(const float* __restrict__ p, int64_t n,
                                                         const __grid_constant__ EmaArg ema, unsigned int* ticket) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  __shared__ float s_consts[2];
  if (threadIdx.x == 0) ema_consts(ema, &s_consts[0], &s_consts[1]);
  __syncthreads();
  const float w = s_consts[0];
  const bool first = s_consts[1] != 0.f;
  constexpr int U = 4;
  const int64_t nvec = n >> 2;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  float4* e4 = reinterpret_cast<float4*>(ema.e);
  for (int64_t w0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; w0 < nvec; w0 += U * stride) {
    float4 pp[U], ee[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t i = w0 + u * stride;
      if (i < nvec) {
        pp[u] = __ldcs(reinterpret_cast<const float4*>(p) + i);
        ee[u] = __ldcs(e4 + i);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t i = w0 + u * stride;
      if (i >= nvec) continue;
      ee[u].x = ema_lerp(ee[u].x, pp[u].x, w, first);
      ee[u].y = ema_lerp(ee[u].y, pp[u].y, w, first);
      ee[u].z = ema_lerp(ee[u].z, pp[u].z, w, first);
      ee[u].w = ema_lerp(ee[u].w, pp[u].w, w, first);
      __stcs(e4 + i, ee[u]);
    }
  }
  if (blockIdx.x == 0)
    for (int64_t j = (nvec << 2) + threadIdx.x; j < n; j += blockDim.x) ema.e[j] = ema_lerp(ema.e[j], p[j], w, first);
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(ticket, 1u) == gridDim.x - 1) {
      *ticket = 0u;
      *ema.count = *reinterpret_cast<volatile int64_t*>(ema.count) + 1;
    }
  }
}

int launch_ema_update(Ctx* ctx, const float* p, int64_t n, const EmaArg& ema, unsigned int* ticket,
                      cudaStream_t stream) {
  RVAE_REQUIRE(p && ema.e && ema.decay && ema.count && ticket, RVAE_ERR_INVALID, "ema_update: null buffer");
  RVAE_REQUIRE(n >= 0, RVAE_ERR_INVALID, "ema_update: n = %lld", (long long)n);
  RVAE_REQUIRE(((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(ema.e)) & 15) == 0, RVAE_ERR_INVALID,
               "ema_update: ema and params must be 16-byte aligned");
  const int threads = 256;
  // a multiple of the SM count: one to four blocks per SM, by size (each thread covers 4 float4 groups per trip)
  const int64_t per_wave = (int64_t)ctx->num_sms_total * threads * 4 * 4;
  const int64_t waves = std::min<int64_t>(4, std::max<int64_t>(1, (n + per_wave - 1) / per_wave));
  RVAE_CUDA(launch_kernel(ctx, ema_update_kernel, dim3(ctx->num_sms_total * (int)waves), dim3(threads), (size_t)0,
                          stream, p, n, ema, ticket));
  RVAE_LAUNCH_CHECK(ctx);
  return RVAE_OK;
}

// ------------------------------------------------------------------------------------------------
// Global gradient norm for clipping (torch.nn.utils.clip_grad_norm_, norm type 2). A launch reads one or two segments
// of the flat gradient buffer (4 B/param, float4 loads), squares each fp32 element in fp64 - a gradient of 1e-30 does
// not underflow - and writes one fp64 partial per block to part[blockIdx.x]. Element-to-thread mapping, the grid
// (grad_norm_blocks) and the reduction tree are fixed, with no atomics, so a gradient buffer gives the same bits every
// time. With f.ticket set, the last block of the launch sums every partial of the reduction, f.parts[0 .. n_parts),
// in index order (earlier launches are complete: stream- or event-ordered before this one) and writes
//   norm = sqrt(sum) -> norm_out[*step mod ring_size] (fp32; slot 0 without a step counter),
//   coef = min(1, max_norm / (norm + 1e-6)) in fp64, rounded to fp32 once -> *coef_out (when max_norm != nullptr).
// A NaN norm gives a NaN coef (torch.clamp propagates it); inf gives 0, or NaN with max_norm = inf, as in torch.
// ------------------------------------------------------------------------------------------------
constexpr int kNormThreads = 256;

__device__ __forceinline__ double block_sum_f64(double v, double* smem) {
  // block total in thread 0, in a fixed order
  v = warp_sum_f64(v);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) smem[warp] = v;
  __syncthreads();
  double t = 0.0;
  if (warp == 0) t = warp_sum_f64(lane < kNormThreads / 32 ? smem[lane] : 0.0);
  return t;
}

__global__ void __launch_bounds__(kNormThreads) grad_norm_kernel(const float* __restrict__ g, int64_t n, int64_t off_b,
                                                                 int64_t n_b, double* __restrict__ part,
                                                                 NormFinalize f) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  __shared__ double red[kNormThreads / 32];
  __shared__ bool is_last;
  constexpr int U = 4;   // float4 loads in flight per thread
  const int64_t nvec = n >> 2, nvec_all = nvec + (n_b >> 2), shift_b = (off_b >> 2) - nvec;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  double acc = 0.0;
  for (int64_t w0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; w0 < nvec_all; w0 += U * stride) {
    float4 q[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t w = w0 + u * stride;
      q[u] = w < nvec_all ? __ldcg(reinterpret_cast<const float4*>(g) + (w < nvec ? w : w + shift_b))
                          : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      acc = fma((double)q[u].x, (double)q[u].x, acc);
      acc = fma((double)q[u].y, (double)q[u].y, acc);
      acc = fma((double)q[u].z, (double)q[u].z, acc);
      acc = fma((double)q[u].w, (double)q[u].w, acc);
    }
  }
  const double total = block_sum_f64(acc, red);
  if (threadIdx.x == 0) part[blockIdx.x] = total;
  if (f.ticket == nullptr) return;
  if (threadIdx.x == 0) {
    __threadfence();
    is_last = atomicAdd(f.ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  double s = 0.0;
  for (int i = threadIdx.x; i < f.n_parts; i += blockDim.x) s += __ldcg(f.parts + i);
  __syncthreads();   // red[] is reused
  s = block_sum_f64(s, red);
  if (threadIdx.x == 0) {
    *f.ticket = 0u;
    const double norm = sqrt(s);
    if (f.norm_out != nullptr) {
      const int slot = (f.ring_size > 1 && f.step) ? static_cast<int>(static_cast<long long>(*f.step) % f.ring_size) : 0;
      f.norm_out[slot] = static_cast<float>(norm);
    }
    if (f.max_norm != nullptr) {
      const double c = *f.max_norm / (norm + 1e-6);
      *f.coef_out = static_cast<float>(c > 1.0 ? 1.0 : c);   // (not fmin: a NaN must propagate)
    }
  }
}

int grad_norm_blocks(const Ctx* ctx, int64_t n) {
  // a multiple of the SM count: one to four blocks per SM, by size
  const int64_t per_wave = (int64_t)ctx->num_sms_total * kNormThreads * 4;   // elements one float4 per thread covers
  const int64_t waves = std::min<int64_t>(4, std::max<int64_t>(1, (n + per_wave - 1) / per_wave));
  return ctx->num_sms_total * (int)waves;
}

int launch_grad_norm(Ctx* ctx, const float* g, int64_t n, int64_t off_b, int64_t n_b, double* part,
                     const NormFinalize& f, cudaStream_t stream) {
  RVAE_REQUIRE(g && part, RVAE_ERR_INVALID, "grad_norm: null buffer");
  RVAE_REQUIRE((n & 3) == 0 && (off_b & 3) == 0 && (n_b & 3) == 0 && (n_b == 0 || off_b >= n) &&
                   (reinterpret_cast<uintptr_t>(g) & 15) == 0,
               RVAE_ERR_INVALID, "grad_norm: segments must be 16-byte aligned multiples of 4 elements");
  RVAE_REQUIRE(f.ticket == nullptr || (f.parts && f.n_parts > 0 && (f.max_norm == nullptr || f.coef_out)),
               RVAE_ERR_INVALID, "grad_norm: bad finalize arguments");
  RVAE_CUDA(launch_kernel(ctx, grad_norm_kernel, dim3(grad_norm_blocks(ctx, n + n_b)), dim3(kNormThreads), (size_t)0,
                          stream, g, n, off_b, n_b, part, f));
  RVAE_LAUNCH_CHECK(ctx);
  return RVAE_OK;
}

// ------------------------------------------------------------------------------------------------
// Latent backward (backward of reparameterize, rawvae/model.py:24-26, merged with the KL gradient of :45):
//   sigma = exp(lv / 2)
//   d_mu = dz + g_mu,  d_lv = dz * eps * sigma / 2 + g_lv        -> d_ml[:, :L], d_ml[:, L:]  (bf16 planes)
//   g_mu = c * mu, g_lv = c * (sigma^2 - 1) / 2 (fused loss, c = kl_beta / (B L))   or external upstream gradients
//   bias_grad[0:2L] += column sums of d_ml = [db21; db22];  dz is cleared for the next step's split-K reduce-add.
// dz is the fp32 result of the split-K latent dgrad GEMM (da3 W3). One thread handles 4 adjacent latent columns of a
// strided set of rows: float4 loads, 8-byte bf16 stores, column sums in registers -> smem -> one atomic per column
// and block.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float latent_kl_c(const KlGrad& kl) {
  double lr;
  float beta;
  hparams_eval(*kl.hp, static_cast<double>(*kl.step), &lr, &beta);
  return static_cast<float>(__ddiv_rn(static_cast<double>(beta), kl.bl));
}

// kDet (launch_latent_bwd_det): dz is the sum of its split-K slices in split order, the block's column sums go to its
// own row of det.bias_part, and the loss is finalised from the fixed loss slots - no atomics anywhere.
template <bool kDet>
__device__ __forceinline__ void latent_bwd_body(float* __restrict__ dz, const float* __restrict__ eps,
                                                const float* __restrict__ lv, const float* __restrict__ mu,
                                                const float* __restrict__ g_mu_ext, const float* __restrict__ g_lv_ext,
                                                const KlGrad& kl, int64_t M, int L, __nv_bfloat16* __restrict__ dml_hi,
                                                __nv_bfloat16* __restrict__ dml_lo, float* __restrict__ bias_grad,
                                                int clear_dz, const LossFinalize& fin, const AuxTrace& tr,
                                                const LatentDet& det) {
  ptx::pdl_launch_dependents();
  // c = (float)(beta(k) / (B L)), as the host rounds it for a kl_beta argument. kl.early: evaluated before
  // griddepcontrol.wait, overlapping the previous kernel (see rvae_plan_train_step_hp for why that is safe)
  __shared__ float s_c;
  if (kl.hp != nullptr && kl.early && threadIdx.x == 0) s_c = latent_kl_c(kl);
  ptx::pdl_wait();
  aux_begin(tr, 3);
  // the deferred loss finalisation of this step rides along (the forward that filled the sums is long complete)
  if constexpr (kDet) {
    if (fin.acc != nullptr && blockIdx.x == 0) {
      // the slots in index order: a fixed partition over the threads, then a fixed tree
      __shared__ double red[2][32];
      double a = 0.0, b = 0.0;
      for (int i = threadIdx.x; i < det.n_mse; i += blockDim.x) a += det.mse[i];
      for (int i = threadIdx.x; i < det.n_kl; i += blockDim.x) b += det.kl[i];
      a = warp_sum_f64(a);
      b = warp_sum_f64(b);
      if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = a; red[1][threadIdx.x >> 5] = b; }
      __syncthreads();
      if (threadIdx.x == 0) {
        double ta = 0.0, tb = 0.0;
        for (int w = 0; w < (int)(blockDim.x + 31) / 32; ++w) { ta += red[0][w]; tb += red[1][w]; }
        fin.acc[0] = ta;
        fin.acc[1] = tb;
        loss_finalize_body(fin.acc, fin.inv_rec, loss_kl_scale(fin), fin.loss_out, fin.ring_size, fin.step,
                           fin.inc_step);
      }
    }
  } else {
    if (fin.acc != nullptr && blockIdx.x == 0 && threadIdx.x == 0)
      loss_finalize_body(fin.acc, fin.inv_rec, loss_kl_scale(fin), fin.loss_out, fin.ring_size, fin.step, fin.inc_step);
  }
  float c = kl.c;
  if (kl.hp != nullptr) {
    if (!kl.early && threadIdx.x == 0) s_c = latent_kl_c(kl);
    __syncthreads();
    c = s_c;
  }
  extern __shared__ float s_sum[];  // [rows_per_pass][2L]
  const int q = L >> 2;                    // float4 groups per row
  const int rpp = blockDim.x / q;          // rows per pass
  const int cx = threadIdx.x % q;          // column group of this thread
  const int ry = threadIdx.x / q;
  float smu[4] = {0.f, 0.f, 0.f, 0.f}, slv[4] = {0.f, 0.f, 0.f, 0.f};
  // U rows per thread and trip, all loads (4 or 5 float4 per row) issued before the first use
  constexpr int U = 2;
  const bool ext = g_lv_ext != nullptr;
  const int64_t rstride = (int64_t)gridDim.x * rpp;
  for (int64_t r0 = (int64_t)blockIdx.x * rpp + ry; r0 < M; r0 += U * rstride) {
    float4 d4[U], e4[U], l4[U], a4[U], b4[U];
    size_t idx[U];
    bool ok[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t r = r0 + u * rstride;
      ok[u] = r < M;
      idx[u] = (size_t)(ok[u] ? r : 0) * q + cx;
      if (ok[u]) {
        d4[u] = __ldcs(reinterpret_cast<const float4*>(dz) + idx[u]);
        if constexpr (kDet) {
          for (int k = 0; k < det.n_dz_slices; ++k) {   // split order
            const float4 t = __ldcs(reinterpret_cast<const float4*>(det.dz_slices + k * det.dz_stride) + idx[u]);
            d4[u].x += t.x; d4[u].y += t.y; d4[u].z += t.z; d4[u].w += t.w;
          }
        }
        e4[u] = __ldcs(reinterpret_cast<const float4*>(eps) + idx[u]);
        l4[u] = __ldcs(reinterpret_cast<const float4*>(lv) + idx[u]);
        b4[u] = make_float4(0.f, 0.f, 0.f, 0.f);  // additive term of d_lv
        if (ext) {
          a4[u] = __ldcs(reinterpret_cast<const float4*>(g_mu_ext) + idx[u]);
          b4[u] = __ldcs(reinterpret_cast<const float4*>(g_lv_ext) + idx[u]);
        } else {
          a4[u] = __ldcs(reinterpret_cast<const float4*>(mu) + idx[u]);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (!ok[u]) continue;
      const int64_t r = r0 + u * rstride;
      const size_t i = idx[u];
      const float* d = reinterpret_cast<const float*>(&d4[u]);
      const float* e = reinterpret_cast<const float*>(&e4[u]);
      const float* l = reinterpret_cast<const float*>(&l4[u]);
      const float* a = reinterpret_cast<const float*>(&a4[u]);
      const float* b = reinterpret_cast<const float*>(&b4[u]);
      float dmu[4], dlv[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float sig = expf(0.5f * l[j]);
        const float gm = ext ? a[j] : c * a[j];
        const float gl = ext ? b[j] : 0.5f * c * (sig * sig - 1.f);
        dmu[j] = d[j] + gm;
        dlv[j] = fmaf(d[j], 0.5f * e[j] * sig, gl);
        smu[j] += dmu[j];
        slv[j] += dlv[j];
      }
      if (clear_dz) reinterpret_cast<float4*>(dz)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      const size_t o = (size_t)r * (2 * L) + 4 * cx;
      *reinterpret_cast<uint2*>(dml_hi + o) = make_uint2(pack2(dmu[0], dmu[1]), pack2(dmu[2], dmu[3]));
      *reinterpret_cast<uint2*>(dml_hi + o + L) = make_uint2(pack2(dlv[0], dlv[1]), pack2(dlv[2], dlv[3]));
      if (dml_lo) {
        float rm[4], rl[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          rm[j] = dmu[j] - __bfloat162float(__float2bfloat16_rn(dmu[j]));
          rl[j] = dlv[j] - __bfloat162float(__float2bfloat16_rn(dlv[j]));
        }
        *reinterpret_cast<uint2*>(dml_lo + o) = make_uint2(pack2(rm[0], rm[1]), pack2(rm[2], rm[3]));
        *reinterpret_cast<uint2*>(dml_lo + o + L) = make_uint2(pack2(rl[0], rl[1]), pack2(rl[2], rl[3]));
      }
    }
  }
  if (bias_grad != nullptr) {
    float* mine = s_sum + (size_t)ry * 2 * L;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      mine[4 * cx + j] = smu[j];
      mine[L + 4 * cx + j] = slv[j];
    }
    __syncthreads();
    for (int col = threadIdx.x; col < 2 * L; col += blockDim.x) {
      float t = 0.f;
      for (int y = 0; y < rpp; ++y) t += s_sum[(size_t)y * 2 * L + col];
      if constexpr (kDet) bias_grad[(size_t)blockIdx.x * 2 * L + col] = t;
      else atomicAdd(bias_grad + col, t);
    }
  }
  aux_end(tr);
}

__global__ void latent_bwd_kernel(float* __restrict__ dz, const float* __restrict__ eps, const float* __restrict__ lv,
                                  const float* __restrict__ mu, const float* __restrict__ g_mu_ext,
                                  const float* __restrict__ g_lv_ext, KlGrad kl, int64_t M, int L,
                                  __nv_bfloat16* __restrict__ dml_hi, __nv_bfloat16* __restrict__ dml_lo,
                                  float* __restrict__ bias_grad, int clear_dz, LossFinalize fin, AuxTrace tr) {
  const LatentDet none = {};
  latent_bwd_body<false>(dz, eps, lv, mu, g_mu_ext, g_lv_ext, kl, M, L, dml_hi, dml_lo, bias_grad, clear_dz, fin, tr,
                         none);
}

__global__ void latent_bwd_det_kernel(float* __restrict__ dz, const float* __restrict__ eps,
                                      const float* __restrict__ lv, const float* __restrict__ mu, KlGrad kl, int64_t M,
                                      int L, __nv_bfloat16* __restrict__ dml_hi, __nv_bfloat16* __restrict__ dml_lo,
                                      LossFinalize fin, AuxTrace tr, LatentDet det) {
  latent_bwd_body<true>(dz, eps, lv, mu, nullptr, nullptr, kl, M, L, dml_hi, dml_lo, det.bias_part, 0, fin, tr, det);
}

int launch_latent_bwd(Ctx* ctx, float* dz, const float* eps, const float* lv, const float* mu, const float* g_mu_ext,
                      const float* g_lv_ext, const KlGrad& kl, int64_t M, int L, __nv_bfloat16* dml_hi,
                      __nv_bfloat16* dml_lo, float* bias_grad, int clear_dz, const LossFinalize* fin,
                      cudaStream_t stream) {
  // every block reads k = *step: the step counter must not advance inside this launch
  RVAE_REQUIRE(kl.hp == nullptr || (kl.step != nullptr && (fin == nullptr || !fin->inc_step)), RVAE_ERR_INVALID,
               "latent_bwd: a record needs a step counter that stays put during the launch");
  RVAE_REQUIRE(dz && eps && lv && dml_hi, RVAE_ERR_INVALID, "latent_bwd: null buffer");
  RVAE_REQUIRE((g_mu_ext != nullptr) == (g_lv_ext != nullptr), RVAE_ERR_INVALID,
               "latent_bwd: external gradients come in pairs");
  RVAE_REQUIRE(g_lv_ext != nullptr || mu != nullptr, RVAE_ERR_INVALID, "latent_bwd: mu required for the fused KL gradient");
  RVAE_REQUIRE(L > 0 && L % 4 == 0 && L / 4 <= 1024, RVAE_ERR_UNSUPPORTED, "latent_bwd: latent_dim=%d", L);
  if (M <= 0) return RVAE_OK;
  const int q = L / 4;
  const int rpp = q >= 256 ? 1 : 256 / q;
  const int threads = q * rpp;
  // four blocks per SM: enough loads in flight for HBM, and only 4 x num_sms atomics per bias-gradient column
  // (measured: 2 / 4 / 8 blocks per SM -> 15.4 / 12.3 / 15.2 us)
  const int64_t want = (M + rpp - 1) / rpp;
  const int64_t cap = (int64_t)ctx->num_sms * 4;
  const int grid = (int)(want < cap ? want : cap);
  const size_t smem = bias_grad ? (size_t)rpp * 2 * L * sizeof(float) : 0;
  LossFinalize f;
  memset(&f, 0, sizeof(f));
  if (fin) f = *fin;
  RVAE_CUDA(launch_kernel(ctx, latent_bwd_kernel, dim3(grid), dim3(threads), smem, stream, dz, eps, lv, mu, g_mu_ext,
                          g_lv_ext, kl, M, L, dml_hi, dml_lo, bias_grad, clear_dz, f, next_aux(ctx, 3)));
  RVAE_LAUNCH_CHECK(ctx);
  return RVAE_OK;
}

// The deterministic launch's grid: four blocks per SM of a B200 whatever the SM budget, so the rows each block sums,
// and with them the bits of its column sums, depend on the shapes alone.
int latent_det_blocks(int64_t M, int L) {
  const int q = L / 4;
  const int rpp = q >= 256 ? 1 : 256 / q;
  const int64_t want = (M + rpp - 1) / rpp;
  return (int)(want < 148 * 4 ? want : 148 * 4);
}

int launch_latent_bwd_det(Ctx* ctx, float* dz, const float* eps, const float* lv, const float* mu, const KlGrad& kl,
                          int64_t M, int L, __nv_bfloat16* dml_hi, __nv_bfloat16* dml_lo, const LatentDet& det,
                          const LossFinalize* fin, cudaStream_t stream) {
  RVAE_REQUIRE(kl.hp == nullptr || (kl.step != nullptr && (fin == nullptr || !fin->inc_step)), RVAE_ERR_INVALID,
               "latent_bwd: a record needs a step counter that stays put during the launch");
  RVAE_REQUIRE(dz && eps && lv && mu && dml_hi && det.bias_part && (det.n_dz_slices == 0 || det.dz_slices),
               RVAE_ERR_INVALID, "latent_bwd_det: null buffer");
  RVAE_REQUIRE(fin == nullptr || (det.mse && det.kl), RVAE_ERR_INVALID, "latent_bwd_det: no loss slots");
  RVAE_REQUIRE(L > 0 && L % 4 == 0 && L / 4 <= 1024, RVAE_ERR_UNSUPPORTED, "latent_bwd: latent_dim=%d", L);
  if (M <= 0) return RVAE_OK;
  const int q = L / 4;
  const int rpp = q >= 256 ? 1 : 256 / q;
  LossFinalize f;
  memset(&f, 0, sizeof(f));
  if (fin) f = *fin;
  RVAE_CUDA(launch_kernel(ctx, latent_bwd_det_kernel, dim3(latent_det_blocks(M, L)), dim3(q * rpp),
                          (size_t)rpp * 2 * L * sizeof(float), stream, dz, eps, lv, mu, kl, M, L, dml_hi, dml_lo, f,
                          next_aux(ctx, 3), det));
  RVAE_LAUNCH_CHECK(ctx);
  return RVAE_OK;
}

// ------------------------------------------------------------------------------------------------
// Sum of one gradient bucket in deterministic mode (GradSum in common.h): the weight gradient's split-K slices added
// to split 0 in split order (one thread per float4), and the bias partial rows of each column in a fixed order (one
// warp per float4 of columns: lane-strided rows, then a butterfly tree). Neither the grid nor the SM budget enters
// the order of any sum; HBM-bound (float4 loads, grid a multiple of the SM count).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) grad_sum_kernel(const __grid_constant__ GradSum a) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  // weights: one thread per float4, the slices in split order
  const int64_t nw = a.n_slices > 0 ? a.w_count >> 2 : 0;
  for (int64_t i = tid; i < nw; i += nthreads) {
    float4 v = reinterpret_cast<const float4*>(a.w)[i];
    for (int k = 0; k < a.n_slices; ++k) {
      const float4 t = __ldcs(reinterpret_cast<const float4*>(a.w_slices + k * a.w_slice_stride) + i);
      v.x += t.x; v.y += t.y; v.z += t.z; v.w += t.w;
    }
    reinterpret_cast<float4*>(a.w)[i] = v;
  }
  // biases: one WARP per float4 of columns. Lane l adds rows l, l + 32, l + 64, ... in ascending order, then the
  // lanes' sums meet in a fixed butterfly tree: a fixed order whatever the grid, and 32 times the loads in flight of
  // a thread walking every row alone
  int64_t nb[4];
  int64_t nbt = 0;
#pragma unroll
  for (int s = 0; s < 4; ++s) { nb[s] = s < a.n_seg ? a.seg[s].cols >> 2 : 0; nbt += nb[s]; }
  const int lane = threadIdx.x & 31;
  for (int64_t wi = tid >> 5; wi < nbt; wi += nthreads >> 5) {
    int64_t j = wi;
    GradSumSeg g = a.seg[0];
    bool found = false;
#pragma unroll
    for (int s = 0; s < 4; ++s) {   // (unrolled: no dynamically indexed copy of the segment table)
      if (!found && j < nb[s]) { g = a.seg[s]; found = true; }
      else if (!found) j -= nb[s];
    }
    constexpr int kBatch = 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int r0 = lane; r0 < g.rows; r0 += 32 * kBatch) {
      float4 t[kBatch];
#pragma unroll
      for (int u = 0; u < kBatch; ++u) {
        const int r = r0 + 32 * u;
        t[u] = r < g.rows ? __ldcs(reinterpret_cast<const float4*>(g.src + r * g.pitch) + j)
                          : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int u = 0; u < kBatch; ++u) {
        if (r0 + 32 * u < g.rows) { v.x += t[u].x; v.y += t[u].y; v.z += t[u].z; v.w += t[u].w; }
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      v.x += __shfl_xor_sync(0xffffffffu, v.x, o);
      v.y += __shfl_xor_sync(0xffffffffu, v.y, o);
      v.z += __shfl_xor_sync(0xffffffffu, v.z, o);
      v.w += __shfl_xor_sync(0xffffffffu, v.w, o);
    }
    if (lane == 0) reinterpret_cast<float4*>(g.dst)[j] = v;
  }
}

int launch_grad_sum(Ctx* ctx, const GradSum& a, cudaStream_t stream) {
  RVAE_REQUIRE(a.n_seg >= 0 && a.n_seg <= 4, RVAE_ERR_INVALID, "grad_sum: %d segments", a.n_seg);
  uintptr_t align = reinterpret_cast<uintptr_t>(a.w) | reinterpret_cast<uintptr_t>(a.w_slices) |
                    (uintptr_t)(a.w_count | a.w_slice_stride);
  for (int s = 0; s < a.n_seg; ++s) {
    const GradSumSeg& g = a.seg[s];
    RVAE_REQUIRE(g.dst && g.src && g.rows >= 0, RVAE_ERR_INVALID, "grad_sum: bad bias segment %d", s);
    align |= reinterpret_cast<uintptr_t>(g.dst) | reinterpret_cast<uintptr_t>(g.src) | (uintptr_t)(g.pitch | g.cols);
  }
  RVAE_REQUIRE((align & 3) == 0 && ((reinterpret_cast<uintptr_t>(a.w) | reinterpret_cast<uintptr_t>(a.w_slices)) & 15) == 0,
               RVAE_ERR_INVALID, "grad_sum: buffers must be 16-byte aligned multiples of 4 elements");
  RVAE_REQUIRE(a.n_slices == 0 || (a.w && a.w_slices), RVAE_ERR_INVALID, "grad_sum: null weight buffer");
  for (int s = 0; s < a.n_seg; ++s)
    RVAE_REQUIRE(((reinterpret_cast<uintptr_t>(a.seg[s].dst) | reinterpret_cast<uintptr_t>(a.seg[s].src)) & 15) == 0,
                 RVAE_ERR_INVALID, "grad_sum: bias segments must be 16-byte aligned");
  const int64_t nwork = (a.n_slices > 0 ? a.w_count / 4 : 0) + [&] {
    int64_t t = 0;
    for (int s = 0; s < a.n_seg; ++s) t += a.seg[s].cols / 4 * 32;   // a warp per float4 of bias columns
    return t;
  }();
  const int threads = 256;
  // a multiple of the SM count: one to four blocks per SM, by size (every thread covers >= one float4)
  const int64_t per_sm = (int64_t)threads;
  const int64_t blocks = std::min<int64_t>(4, std::max<int64_t>(1, (nwork + per_sm * ctx->num_sms_total - 1) /
                                                                    (per_sm * ctx->num_sms_total)));
  RVAE_CUDA(launch_kernel(ctx, grad_sum_kernel, dim3((unsigned)(blocks * ctx->num_sms_total)), dim3(threads),
                          (size_t)0, stream, a));
  RVAE_LAUNCH_CHECK(ctx);
  return RVAE_OK;
}

// ------------------------------------------------------------------------------------------------
// Gradient all-reduce over NVLink peer memory (data parallelism). Every rank's flat gradient buffer lives in a
// symmetric allocation that all peers map (CUDA IPC); the kernel reads and writes peer memory directly with 128-bit
// loads - no staging copies, no NCCL. Two-shot, in place:
//   barrier 1 : every peer's bucket gradient is complete (their kernel has started)
//   reduce    : rank r sums slice r of the bucket over all ranks (W-1 peer reads + 1 local per element) and writes
//               the sum into EVERY rank's buffer (local store + W-1 posted NVLink writes)   [reduce-scatter + push]
//   barrier 2 : all slices have landed everywhere, and nobody reads this rank's buffer any more -> the caller may
//               overwrite the gradient (Adam clears it)
// A flag hop between two GPUs costs ~5 us on this fabric, so the protocol is built around the minimum of two hops.
// Work is split by CTA index: CTA c of every rank owns chunk c of each slice and synchronises only with the CTAs c
// of the other ranks (flags in the peers' symmetric memory, release / acquire at system scope), so no grid-wide
// barrier is needed and a grid of a few CTAs lives on the SMs the persistent GEMMs leave free. Flag values are
// monotonic (4 * epoch + phase); the epoch is a device counter, so CUDA-graph replays stay correct.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// NVLS (NVSwitch multicast): one load returns the SUM of the location over every rank's buffer, reduced in the switch;
// one store writes every rank's buffer
__device__ __forceinline__ float4 ld_reduce_mc(const float4* p) {
  float4 v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_mc(float4* p, const float4& v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};"
               ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ float4 ld_peer(const float4* p) {
  float4 v;
  asm volatile("ld.relaxed.sys.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
  return v;
}

// MAXW: ranks the instantiation supports; U: float4 elements per thread and trip. All (MAXW - 1) * U peer loads of a
// trip are issued before the first add, so ~16 x 16 bytes per thread are in flight (NVLink latency is ~1 us: a
// few MB in flight are needed to fill it from 16 CTAs).
template <int MAXW, int U>
__global__ void __launch_bounds__(512, 1) allreduce_p2p_kernel(P2PArgs a, P2PSegs sg, int bucket, AuxTrace tr) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  aux_begin(tr, 5);
  const int G = gridDim.x, c = blockIdx.x, W = a.world, me = a.rank;
  __shared__ uint32_t s_epoch;
  if (threadIdx.x == 0) s_epoch = *reinterpret_cast<volatile uint32_t*>(a.epoch + bucket) + 1u;
  __syncthreads();
  const uint32_t e = s_epoch;
  const int flag_row = (bucket * kP2PMaxCtas + c) * kP2PMaxWorld * kP2PFlagStride;

  auto barrier = [&](uint32_t phase) {
    __syncthreads();   // every thread's stores of the previous phase are ordered before the fence below
    const uint32_t want = 4u * e + phase;
    if (threadIdx.x < W && (int)threadIdx.x != me) {
      const int p = threadIdx.x;
      uint32_t* theirs = a.flags[p] + flag_row + me * kP2PFlagStride;
      const uint32_t* mine = a.flags[me] + flag_row + p * kP2PFlagStride;
      if (a.mode == 0) {
        __threadfence_system();
        st_release_sys(theirs, want);
      } else if (a.mode == 1) {
        st_release_sys(theirs, want);
      } else if (a.mode == 3) {   // remote atomic: performed at the destination, cannot linger in a write buffer
        __threadfence_system();
        asm volatile("red.relaxed.sys.global.max.u32 [%0], %1;" ::"l"(theirs), "r"(want) : "memory");
      } else if (a.mode == 4) {   // push the flag out with a trailing fence
        st_release_sys(theirs, want);
        __threadfence_system();
      } else {
        __threadfence_system();
        *reinterpret_cast<volatile uint32_t*>(theirs) = want;
      }
      // A peer may legitimately be seconds behind (rank 0 writing a checkpoint, a slow filesystem, a graph being
      // instantiated): wait for minutes, not seconds, and never trap - a trapped context poisons the process and
      // leaves the peers spinning. On timeout the FIRST failure is recorded in a status word the host polls
      // (rvae_dp_status), and every later wait of this context falls through at once.
      const long long t0 = clock64();
      bool dead = *reinterpret_cast<volatile uint32_t*>(a.status) != 0u;
      unsigned spins = 0;
      while (!dead && (a.mode == 0 ? ld_acquire_sys(mine) : *reinterpret_cast<const volatile uint32_t*>(mine)) < want) {
        if ((++spins & 1023u) == 0u) {
          if (clock64() - t0 > a.timeout_cycles) {
            atomicCAS(a.status, 0u, 0x80000000u | (static_cast<uint32_t>(p) << 8) | (static_cast<uint32_t>(bucket) << 4) | phase);
            dead = true;
          } else if (*reinterpret_cast<volatile uint32_t*>(a.status) != 0u) {
            dead = true;
          }
        }
        if (a.mode >= 5) __nanosleep(40);
      }
      if (a.mode != 0) __threadfence_system();
    }
    __syncthreads();
  };

  // the bucket is the concatenation of up to three segments of the flat buffer (float4 units)
  const int64_t n0 = sg.n[0] >> 2, n1 = sg.n[1] >> 2, n2 = sg.n[2] >> 2;
  const int64_t o0 = sg.off[0] >> 2, o1 = sg.off[1] >> 2, o2 = sg.off[2] >> 2;
  auto at = [&](int64_t i) -> int64_t { return i < n0 ? o0 + i : (i < n0 + n1 ? o1 + (i - n0) : o2 + (i - n0 - n1)); };
  const int64_t n4 = n0 + n1 + n2;
  const int64_t per_rank = (n4 + W - 1) / W;
  const int64_t per_cta = (per_rank + G - 1) / G;
  const int64_t T = blockDim.x;

  const unsigned long long g0 = tr.slot ? global_timer() : 0ull;
  barrier(1);
  const unsigned long long g1 = tr.slot ? global_timer() : 0ull;
  {  // my slice, my chunk: sum over all ranks, store locally AND push the result into every peer's buffer
    const int64_t s0 = (int64_t)me * per_rank;
    const int64_t s1 = min(s0 + per_rank, n4);
    const int64_t b0 = min(s0 + (int64_t)c * per_cta, s1), b1 = min(b0 + per_cta, s1);
    if (a.mc_data != nullptr) {
      // NVLS: the switch reduces my slice over all ranks (1 / W of the bucket crosses my links, once, instead of
      // (W - 1) / W peer reads) and multicasts the result back into every rank's buffer
      constexpr int UM = MAXW * U < 16 ? MAXW * U : 16;
      float4* mc = reinterpret_cast<float4*>(a.mc_data);
      for (int64_t base = b0 + threadIdx.x; base < b1; base += T * UM) {
        float4 v[UM];
#pragma unroll
        for (int u = 0; u < UM; ++u) {
          const int64_t i = base + u * T;
          if (i < b1) v[u] = ld_reduce_mc(mc + at(i));
        }
#pragma unroll
        for (int u = 0; u < UM; ++u) {
          const int64_t i = base + u * T;
          if (i < b1) st_mc(mc + at(i), v[u]);
        }
      }
    } else
    for (int64_t base = b0 + threadIdx.x; base < b1; base += T * U) {
      float4 v[MAXW][U];
#pragma unroll
      for (int p = 0; p < MAXW; ++p) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int64_t i = base + u * T;
          v[p][u] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (p < W && i < b1) {
            const float4* src = reinterpret_cast<const float4*>(a.data[p]) + at(i);
            v[p][u] = (p == me) ? *src : ld_peer(src);
          }
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int64_t i = base + u * T;
        if (i < b1) {
          float4 acc = v[0][u];
#pragma unroll
          for (int p = 1; p < MAXW; ++p) { acc.x += v[p][u].x; acc.y += v[p][u].y; acc.z += v[p][u].z; acc.w += v[p][u].w; }
#pragma unroll
          for (int p = 0; p < MAXW; ++p)
            if (p < W) reinterpret_cast<float4*>(a.data[p])[at(i)] = acc;   // p == me: local; else a posted NVLink write
        }
      }
    }
  }
  const unsigned long long g2 = tr.slot ? global_timer() : 0ull;
  // one more flag exchange ends the all-reduce: it publishes my pushes, tells me every peer's slice has landed in my
  // buffer, and - because a peer signals only after it has read my contribution - that nobody reads my buffer any
  // more, so the caller may overwrite it (Adam clears the gradient)
  barrier(2);
  if (tr.slot && threadIdx.x == 0) {  // detail words: the slowest CTA's barrier 1 / reduce+push / barrier 2
    atomicMax(tr.slot + 4, g1 - g0);
    atomicMax(tr.slot + 5, g2 - g1);
    atomicMax(tr.slot + 6, global_timer() - g2);
  }
  aux_end(tr);
  if (threadIdx.x == 0) {  // the last CTA advances the epoch of this bucket (every CTA has read it)
    const unsigned int done = atomicAdd(a.ticket + bucket, 1u);
    if (done == gridDim.x - 1) {
      a.ticket[bucket] = 0u;
      __threadfence();
      *reinterpret_cast<volatile uint32_t*>(a.epoch + bucket) = e;
    }
  }
}

int launch_allreduce_p2p(Ctx* ctx, const P2PArgs& a, const P2PSegs& sg, int bucket, int ctas, cudaStream_t stream) {
  RVAE_REQUIRE(a.world >= 2 && a.world <= kP2PMaxWorld && bucket >= 0 && bucket < kP2PMaxBuckets, RVAE_ERR_INVALID,
               "allreduce_p2p: world %d bucket %d", a.world, bucket);
  RVAE_REQUIRE(ctas >= 1 && ctas <= kP2PMaxCtas, RVAE_ERR_INVALID, "allreduce_p2p: %d CTAs", ctas);
  for (int i = 0; i < 3; ++i)
    RVAE_REQUIRE((sg.n[i] & 3) == 0 && (sg.off[i] & 3) == 0 && sg.n[i] >= 0, RVAE_ERR_INVALID,
                 "allreduce_p2p: segments must be multiples of 4 floats");
  const AuxTrace tr = next_aux(ctx, 5);
  if (a.world <= 2)
    RVAE_CUDA(launch_kernel(ctx, allreduce_p2p_kernel<2, 12>, dim3(ctas), dim3(512), (size_t)0, stream, a, sg, bucket, tr));
  else if (a.world <= 4)
    RVAE_CUDA(launch_kernel(ctx, allreduce_p2p_kernel<4, 4>, dim3(ctas), dim3(512), (size_t)0, stream, a, sg, bucket, tr));
  else
    RVAE_CUDA(launch_kernel(ctx, allreduce_p2p_kernel<8, 2>, dim3(ctas), dim3(512), (size_t)0, stream, a, sg, bucket, tr));
  RVAE_LAUNCH_CHECK(ctx);
  return RVAE_OK;
}

// ------------------------------------------------------------------------------------------------
// TensorBoard parameter histograms (writer.add_histogram, train_iterable.py:216-217, train.py:203-204): one launch
// bins every parameter segment of the flat buffer against the caller's edge table with the semantics of
// make_histogram(values.astype(float64), edges): bin i holds [e[i], e[i+1]), the last bin is closed, values outside
// [e[0], e[n]] and NaN are not counted; min / max / num / sum / sum of squares over all values, NaN and +-inf
// propagating as in numpy.
//
// Bin search. A float's order-preserving 32-bit key (sign-flipped bits) is split at its top 12 bits: a bucket spans a
// magnitude ratio of at most 1.125 (1 sign + 8 exponent + 3 mantissa bits). guide[j] = number of edges <= the
// smallest float of bucket j (computed on the host, exact in fp64), so every value of bucket j has between guide[j]
// and guide[j + 1] edges below or at it and the exact count is found by a forward scan over that window, comparing
// in fp64 against the table. TensorBoard's edges grow by 1.1 per step, so a window holds at most two edges: one or two
// fp64 compares per value instead of an 11-step binary search over 1549 edges. Nothing assumes the edges' spacing:
// a denser table only widens some windows.
//
// Contention. Initialised (and trained) weights are roughly uniform in +-1/sqrt(fan_in), and on TensorBoard's
// log-spaced bins ~90 % of them land in the top ~25 bins of each sign. Each warp therefore owns a private
// shared-memory sub-histogram (no inter-warp contention); within a warp the hottest bin sees ~2-3 lanes per
// instruction, which the shared atomic unit serialises cheaply. A warp whose 32 values all fall into one bin (a
// constant tensor, e.g. zero biases) issues a single atomic with the count. Blocks add their non-zero bins to the
// record with integer atomics - exact, so the counts do not depend on the order blocks finish in.
//
// Moments. sum and sum of squares are fp64 (each square of an fp32 value is exact in fp64) and reduced in a FIXED
// order: each thread sums its elements in index order, warps and blocks combine in fixed trees, the per-block partials
// land in the scratch tail of the record and the last block to finish (ticket) adds them in a fixed order. The grid
// depends only on the element count, so repeated calls - on any GPU - give bitwise-identical records. min / max are
// reduced through atomicMax on order-preserving keys (order-independent as well).
//
// Algorithmic traffic: read 4 B per parameter, write the record (6.2 KB per segment for TensorBoard's 1548 bins).
// ------------------------------------------------------------------------------------------------
constexpr int kHistGuideBits = 12;
constexpr int kHistGuide = 1 << kHistGuideBits;
constexpr int kHistThreads = 256;
constexpr int kHistWarps = kHistThreads / 32;
constexpr int kHistUnroll = 4;               // values per lane per iteration (independent loads in flight)
constexpr int64_t kHistMinChunk = 16384;     // elements per block (64 per thread) before the grid is capped
constexpr int kHistMaxBlocks = 1024;

struct HistArgs {
  int64_t seg_off[RVAE_HIST_MAX_SEGS];          // element offset of segment s in params
  int64_t seg_cols[RVAE_HIST_MAX_SEGS];         // segment s = rows of seg_cols values at row pitch seg_pitch
  int64_t seg_pitch[RVAE_HIST_MAX_SEGS];
  int64_t vstart[RVAE_HIST_MAX_SEGS + 1];       // prefix sums of the lengths: the segments concatenated
  int64_t chunk;                                // concatenated elements per block
  int n_segs, n_edges;
  double edges[RVAE_HIST_MAX_EDGES];
  uint16_t guide[kHistGuide + 1];
};
static_assert(sizeof(HistArgs) <= 32000, "kernel parameter space (32764 bytes on sm_70+)");

struct HistLayout {   // byte offsets into the caller's record buffer (include/rvae_b200.h)
  size_t sum, sum_sq, num, vmin, vmax, record_bytes, min_key, max_key, nan_flag, ticket, partials, total;
};
static HistLayout hist_layout(int n_segs, int n_edges) {
  HistLayout L;
  const size_t ns = static_cast<size_t>(n_segs), nb = static_cast<size_t>(n_edges - 1);
  L.sum = (4 * ns * nb + 7) / 8 * 8;
  L.sum_sq = L.sum + 8 * ns;
  L.num = L.sum_sq + 8 * ns;
  L.vmin = L.num + 8 * ns;
  L.vmax = L.vmin + 4 * ns;
  L.record_bytes = L.vmax + 4 * ns;
  L.min_key = L.record_bytes;
  L.max_key = L.min_key + 4 * ns;
  L.nan_flag = L.max_key + 4 * ns;
  L.ticket = L.nan_flag + 4 * ns;
  L.partials = (L.ticket + 4 + 7) / 8 * 8;
  L.total = L.partials + 16 * ns * kHistMaxBlocks;
  return L;
}

__host__ __device__ __forceinline__ uint32_t hist_key(float x) {   // a < b <=> key(a) < key(b) (non-NaN, -0 < +0)
  uint32_t u;
  memcpy(&u, &x, 4);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ __forceinline__ float hist_unkey(uint32_t k) {
  const uint32_t u = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
  float x;
  memcpy(&x, &u, 4);
  return x;
}

__global__ void __launch_bounds__(kHistThreads) param_histogram_kernel(const float* __restrict__ params,
                                                                       const __grid_constant__ HistArgs a,
                                                                       uint8_t* __restrict__ rec, HistLayout lay) {
  ptx::pdl_launch_dependents();
  extern __shared__ __align__(16) uint8_t hist_smem[];
  const int nb = a.n_edges - 1;
  double* edges = reinterpret_cast<double*>(hist_smem);
  uint16_t* guide = reinterpret_cast<uint16_t*>(edges + a.n_edges);
  int* sub_all = reinterpret_cast<int*>(hist_smem + ((8 * a.n_edges + 2 * (kHistGuide + 1) + 15) / 16 * 16));
  __shared__ double red_s[kHistWarps], red_ss[kHistWarps];
  __shared__ float red_mn[kHistWarps], red_mx[kHistWarps];
  __shared__ int red_nan[kHistWarps];
  __shared__ bool is_last;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int* sub = sub_all + warp * nb;
  for (int i = tid; i < a.n_edges; i += kHistThreads) edges[i] = a.edges[i];
  for (int i = tid; i <= kHistGuide; i += kHistThreads) guide[i] = a.guide[i];
  for (int i = tid; i < kHistWarps * nb; i += kHistThreads) sub_all[i] = 0;
  __syncthreads();
  ptx::pdl_wait();

  int* counts = reinterpret_cast<int*>(rec);
  uint32_t* min_key = reinterpret_cast<uint32_t*>(rec + lay.min_key);
  uint32_t* max_key = reinterpret_cast<uint32_t*>(rec + lay.max_key);
  uint32_t* nan_flag = reinterpret_cast<uint32_t*>(rec + lay.nan_flag);
  double* partials = reinterpret_cast<double*>(rec + lay.partials);   // [seg][block][2]
  const int64_t c0 = static_cast<int64_t>(blockIdx.x) * a.chunk;
  const int64_t c1 = min(c0 + a.chunk, a.vstart[a.n_segs]);
  const double e_last = edges[nb];
  for (int s = 0; s < a.n_segs; ++s) {
    const int64_t lo = max(c0, a.vstart[s]), hi = min(c1, a.vstart[s + 1]);
    if (lo >= hi) continue;   // block-uniform
    const float* p = params + a.seg_off[s];
    const int64_t v0 = a.vstart[s], cols = a.seg_cols[s], pitch = a.seg_pitch[s];
    const bool dense = cols == pitch;   // block-uniform: one contiguous run, no index arithmetic
    double sum = 0.0, sum_sq = 0.0;
    float mn = INFINITY, mx = -INFINITY;
    int nan = 0;
    for (int64_t base = lo + warp * 32 * kHistUnroll; base < hi; base += kHistThreads * kHistUnroll) {
      float x[kHistUnroll];
#pragma unroll
      for (int u = 0; u < kHistUnroll; ++u) {
        const int64_t v = base + u * 32 + lane - v0;   // index within the segment
        x[u] = v < hi - v0 ? __ldg(p + (dense ? v : v / cols * pitch + v % cols))
                           : __int_as_float(0x7fffffff);   // NaN = nothing to count
      }
#pragma unroll
      for (int u = 0; u < kHistUnroll; ++u) {
        const bool in = base + u * 32 + lane < hi;
        const double xd = static_cast<double>(x[u]);
        int bin = -1;
        if (in) {
          sum += xd;
          sum_sq += xd * xd;
          if (x[u] != x[u]) {
            nan = 1;
          } else {
            mn = fminf(mn, x[u]);
            mx = fmaxf(mx, x[u]);
            const uint32_t j = hist_key(x[u]) >> (32 - kHistGuideBits);
            int c = guide[j];
            const int c_end = guide[j + 1];
            while (c < c_end && edges[c] <= xd) ++c;
            bin = c - 1;                                  // edges <= x, minus one
            if (bin == nb && xd == e_last) bin = nb - 1;  // the last bin is closed
            if (bin >= nb) bin = -1;
          }
        }
        const int b0 = __shfl_sync(0xffffffffu, bin, 0);
        if (__all_sync(0xffffffffu, bin == b0)) {
          if (lane == 0 && b0 >= 0) atomicAdd(sub + b0, 32);
        } else if (bin >= 0) {
          atomicAdd(sub + bin, 1);
        }
      }
    }
    // block totals of this segment (fixed trees)
    sum = warp_sum_f64(sum);
    sum_sq = warp_sum_f64(sum_sq);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    nan = __any_sync(0xffffffffu, nan);
    if (lane == 0) { red_s[warp] = sum; red_ss[warp] = sum_sq; red_mn[warp] = mn; red_mx[warp] = mx; red_nan[warp] = nan; }
    __syncthreads();
    if (tid == 0) {
      double ts = 0.0, tss = 0.0;
      float tmn = INFINITY, tmx = -INFINITY;
      int tnan = 0;
      for (int w = 0; w < kHistWarps; ++w) {
        ts += red_s[w]; tss += red_ss[w];
        tmn = fminf(tmn, red_mn[w]); tmx = fmaxf(tmx, red_mx[w]);
        tnan |= red_nan[w];
      }
      partials[(static_cast<size_t>(s) * kHistMaxBlocks + blockIdx.x) * 2] = ts;
      partials[(static_cast<size_t>(s) * kHistMaxBlocks + blockIdx.x) * 2 + 1] = tss;
      // key 0 is below every real value's key, so 0 (the memset) is the identity of both maxima
      if (tmn <= tmx) {
        atomicMax(min_key + s, ~hist_key(tmn));
        atomicMax(max_key + s, hist_key(tmx));
      }
      if (tnan) atomicOr(nan_flag + s, 1u);
    }
    // fold the warps' sub-histograms into the record and clear them for the next segment
    for (int b = tid; b < nb; b += kHistThreads) {
      int t = 0;
#pragma unroll
      for (int w = 0; w < kHistWarps; ++w) { t += sub_all[w * nb + b]; sub_all[w * nb + b] = 0; }
      if (t) atomicAdd(counts + static_cast<size_t>(s) * nb + b, t);
    }
    __syncthreads();
  }

  // the last block to finish adds the per-block moments in block order and writes the scalar fields
  __threadfence();
  __syncthreads();
  if (tid == 0) is_last = atomicAdd(reinterpret_cast<unsigned int*>(rec + lay.ticket), 1u) == gridDim.x - 1;
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  // one warp per segment: lane l adds blocks b0 + l, b0 + l + 32, ... in order, then a fixed shuffle tree (32 loads
  // in flight instead of one dependent L2 round trip per block)
  for (int s = warp; s < a.n_segs; s += kHistWarps) {
    const int64_t b0 = a.vstart[s] / a.chunk, b1 = (a.vstart[s + 1] - 1) / a.chunk;
    double ts = 0.0, tss = 0.0;
    for (int64_t b = b0 + lane; b <= b1; b += 32) {
      ts += __ldcg(partials + (static_cast<size_t>(s) * kHistMaxBlocks + b) * 2);
      tss += __ldcg(partials + (static_cast<size_t>(s) * kHistMaxBlocks + b) * 2 + 1);
    }
    ts = warp_sum_f64(ts);
    tss = warp_sum_f64(tss);
    if (lane != 0) continue;
    reinterpret_cast<double*>(rec + lay.sum)[s] = ts;
    reinterpret_cast<double*>(rec + lay.sum_sq)[s] = tss;
    reinterpret_cast<int64_t*>(rec + lay.num)[s] = a.vstart[s + 1] - a.vstart[s];
    const bool has_nan = __ldcg(nan_flag + s) != 0u;
    const uint32_t kmn = ~__ldcg(min_key + s), kmx = __ldcg(max_key + s);
    reinterpret_cast<float*>(rec + lay.vmin)[s] = has_nan ? __int_as_float(0x7fffffff) : hist_unkey(kmn);
    reinterpret_cast<float*>(rec + lay.vmax)[s] = has_nan ? __int_as_float(0x7fffffff) : hist_unkey(kmx);
  }
}

size_t param_histogram_bytes(int n_segs, int n_edges) {
  if (n_segs < 1 || n_segs > RVAE_HIST_MAX_SEGS || n_edges < 2 || n_edges > RVAE_HIST_MAX_EDGES) return 0;
  return hist_layout(n_segs, n_edges).total;
}

int launch_param_histogram(Ctx* ctx, const float* params, const int64_t* seg_offsets, const int64_t* seg_lengths,
                           int n_segs, const double* edges, int n_edges, void* record, cudaStream_t stream) {
  RVAE_REQUIRE(seg_lengths, RVAE_ERR_INVALID, "param_histogram: null pointer");
  RVAE_REQUIRE(n_segs >= 1 && n_segs <= RVAE_HIST_MAX_SEGS, RVAE_ERR_INVALID,
               "param_histogram: n_segs = %d, must be 1..%d", n_segs, RVAE_HIST_MAX_SEGS);
  int64_t ones[RVAE_HIST_MAX_SEGS];
  for (int s = 0; s < n_segs; ++s) ones[s] = 1;
  return launch_param_histogram_rows(ctx, params, seg_offsets, ones, seg_lengths, seg_lengths, n_segs, edges, n_edges,
                                     record, stream);
}

int launch_param_histogram_rows(Ctx* ctx, const float* params, const int64_t* seg_offsets, const int64_t* seg_rows,
                                const int64_t* seg_cols, const int64_t* seg_pitch, int n_segs, const double* edges,
                                int n_edges, void* record, cudaStream_t stream) {
  RVAE_REQUIRE(params && seg_offsets && seg_rows && seg_cols && seg_pitch && edges && record, RVAE_ERR_INVALID,
               "param_histogram: null pointer");
  RVAE_REQUIRE(n_segs >= 1 && n_segs <= RVAE_HIST_MAX_SEGS, RVAE_ERR_INVALID,
               "param_histogram: n_segs = %d, must be 1..%d", n_segs, RVAE_HIST_MAX_SEGS);
  RVAE_REQUIRE(n_edges >= 2 && n_edges <= RVAE_HIST_MAX_EDGES, RVAE_ERR_INVALID,
               "param_histogram: n_edges = %d, must be 2..%d", n_edges, RVAE_HIST_MAX_EDGES);
  RVAE_REQUIRE(reinterpret_cast<uintptr_t>(record) % 16 == 0 && reinterpret_cast<uintptr_t>(params) % 4 == 0,
               RVAE_ERR_INVALID, "param_histogram: record must be 16-byte and params 4-byte aligned");
  for (int i = 0; i < n_edges; ++i) {
    RVAE_REQUIRE(std::isfinite(edges[i]), RVAE_ERR_INVALID, "param_histogram: edge %d is not finite", i);
    RVAE_REQUIRE(i == 0 || edges[i] > edges[i - 1], RVAE_ERR_INVALID,
                 "param_histogram: edges must increase strictly (edge %d)", i);
  }
  std::unique_ptr<HistArgs> ap(new HistArgs());   // 25 KB of kernel arguments: not on the stack
  HistArgs& a = *ap;
  a.n_segs = n_segs;
  a.n_edges = n_edges;
  a.vstart[0] = 0;
  for (int s = 0; s < n_segs; ++s) {
    RVAE_REQUIRE(seg_offsets[s] >= 0 && seg_rows[s] >= 1 && seg_cols[s] >= 1 && seg_pitch[s] >= seg_cols[s],
                 RVAE_ERR_INVALID, "param_histogram: segment %d (offset %lld, %lld rows of %lld at pitch %lld) is empty "
                 "or out of range", s, (long long)seg_offsets[s], (long long)seg_rows[s], (long long)seg_cols[s],
                 (long long)seg_pitch[s]);
    a.seg_off[s] = seg_offsets[s];
    a.seg_cols[s] = seg_cols[s];
    a.seg_pitch[s] = seg_rows[s] == 1 ? seg_cols[s] : seg_pitch[s];   // one row: contiguous, whatever the pitch
    a.vstart[s + 1] = a.vstart[s] + seg_rows[s] * seg_cols[s];
  }
  memcpy(a.edges, edges, sizeof(double) * n_edges);
  // guide[j] = #edges <= smallest float of key bucket j (NaN buckets: below / above everything); a merge walk
  int c = 0;
  for (int j = 0; j < kHistGuide; ++j) {
    const float lo = hist_unkey(static_cast<uint32_t>(j) << (32 - kHistGuideBits));
    if (lo != lo) {
      a.guide[j] = static_cast<uint16_t>(j < kHistGuide / 2 ? 0 : n_edges);
      continue;
    }
    while (c < n_edges && edges[c] <= static_cast<double>(lo)) ++c;
    a.guide[j] = static_cast<uint16_t>(c);
  }
  a.guide[kHistGuide] = static_cast<uint16_t>(n_edges);
  const int64_t total = a.vstart[n_segs];
  a.chunk = std::max<int64_t>(kHistMinChunk, (total + kHistMaxBlocks - 1) / kHistMaxBlocks);
  const int grid = static_cast<int>((total + a.chunk - 1) / a.chunk);
  const HistLayout lay = hist_layout(n_segs, n_edges);
  const size_t smem = (8 * (size_t)n_edges + 2 * (kHistGuide + 1) + 15) / 16 * 16 + 4 * (size_t)kHistWarps * (n_edges - 1);
  RVAE_CUDA(cudaFuncSetAttribute(param_histogram_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // counts, min / max keys, NaN flags and the ticket start from zero; sums and partials are overwritten
  RVAE_CUDA(cudaMemsetAsync(record, 0, lay.partials, stream));
  RVAE_CUDA(launch_kernel(ctx, param_histogram_kernel, dim3(grid), dim3(kHistThreads), smem, stream, params, *ap,
                          static_cast<uint8_t*>(record), lay));
  RVAE_LAUNCH_CHECK(ctx);
  return RVAE_OK;
}

__global__ void step_inc_kernel(float* step) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  if (threadIdx.x == 0 && blockIdx.x == 0) *step += 1.0f;
}

int launch_step_inc(Ctx* ctx, float* step, cudaStream_t stream) {
  RVAE_REQUIRE(step, RVAE_ERR_INVALID, "step_inc: null step");
  RVAE_CUDA(launch_kernel(ctx, step_inc_kernel, dim3(1), dim3(32), (size_t)0, stream, step));
  RVAE_LAUNCH_CHECK(ctx);
  return RVAE_OK;
}

}  // namespace rvae
