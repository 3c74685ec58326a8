// Persistent, warp-specialised tcgen05 GEMM for sm_100a.
//
//   D[m, n] = sum_k A[m, k] * B[n, k]        (bf16 operands, fp32 accumulation in TMEM)
//
// One CTA per SM loops over 128 x BLOCK_N output tiles (x split-K slices for the reduce-add GEMMs):
//   warp 0 (one lane)  : TMA producer   - fills a STAGES-deep ring of {A tile, B tile} in 128B-swizzled smem
//   warp 1 (one lane)  : UMMA issuer    - tcgen05.mma 128 x BLOCK_N x 16 into one of two TMEM accumulators
//   warps 2..9         : epilogue       - two teams of four warps: tcgen05.ld the finished accumulator, apply the
//                                         fused epilogue (bias/ReLU/tanh, reparameterisation+KL, tanh+MSE+dL/da,
//                                         ReLU mask, ...), stage the result in swizzled smem and TMA-store it
// so the epilogue of tile i overlaps the MMAs of tile i+1 (double-buffered TMEM, 2 x BLOCK_N columns).
//
// Every byte the epilogue exchanges with global memory moves through TMA and 128B-swizzled smem slots: the side
// inputs (ReLU mask, x for the MSE, eps for the reparameterisation) are prefetched by TMA loads while the tile's MMAs
// still run, the thread that owns a row reads them from the slot, writes its result IN PLACE, and the slot is handed
// to a TMA store (or reduce-add). Row-per-thread global loads / stores (32 cache lines per warp instruction) are
// never issued.
//
// Operands may be K-major (row = m or n, K contiguous: activations / weights in the forward pass) or
// MN-major (row = k, M or N contiguous: weights in dgrad, activations in wgrad) - no transposed copies are
// ever materialised; only the TMA box and the UMMA descriptor change.
//
// "fp32 mode" runs the same kernel with num_passes = 3 over split operands (x = hi + lo, both bf16):
// hi*hi + hi*lo + lo*hi accumulated in the same fp32 TMEM accumulator (error ~2^-16 relative).
#pragma once
#include <cstdint>
#include <cstdio>
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "ptx.cuh"

// Paths that were measured and did NOT win (profiles/README.md) are compiled only with -DRVAE_EXPERIMENTS=1
// (RVAE_EXPERIMENTS=1 python -m rawaudiovae_kelsey_b200._build): the forward pass as one launch chained by tile-level
// dependencies, the latent backward fused into the latent dgrad's epilogue (EPI_DLATENT), and the producer-only /
// MMA-only debug modes. The default build carries none of their instructions in the hot loops.
#ifndef RVAE_EXPERIMENTS
#define RVAE_EXPERIMENTS 0
#endif

namespace rvae {

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;  // 64 bf16 = 128 B = one swizzle row
constexpr int kUmmaK = 16;
constexpr int kGemmThreads = 320;  // warp 0 TMA, warp 1 MMA, warps 2..9 epilogue (two teams of four)
constexpr int kEpiTeams = 2;
constexpr int kMaxPasses = 3;
constexpr int kSlotBytes = 128 * 128;  // one epilogue slot: 128 rows x 128 bytes (64 bf16 / 32 fp32 columns)
constexpr int kSlotsPerTeam = 3;

enum : int { MAJOR_K = 0, MAJOR_MN = 1 };
enum : int { EPI_LINEAR = 0, EPI_HEAD = 1, EPI_OUT = 2, EPI_DRELU = 3, EPI_REDUCE = 5, EPI_DLATENT = 6 };
// Deterministic kinds (rvae_plan_set_deterministic): the same epilogues with every cross-CTA or cross-warp sum moved
// to fixed scratch slots, so the bits of a result never depend on which CTA ran which tile or in what order.
//   SLICE      : REDUCE with a plain store per split: split 0 -> out_f32, split k >= 1 -> out_f32_b rows
//                (k - 1) * ldp + m (ldp = the slice stride, rows)
//   HEAD_DET   : HEAD; the KL partial of each (32-row block r, 64-latent-column group c) -> loss_acc[r * L/64 + c]
//   OUT_DET    : OUT; the MSE partial of each (32-row block r, 64-column group c) -> loss_acc[r * N/64 + c], and the
//                column sums of each warp's 32 rows -> colsum[r * ldp + n] (no atomics)
//   DRELU_DET  : DRELU with the column sums as in OUT_DET
enum : int { EPI_SLICE = 7, EPI_HEAD_DET = 8, EPI_OUT_DET = 9, EPI_DRELU_DET = 10 };
__host__ __device__ constexpr int epi_base(int e) {
  return e == EPI_SLICE ? EPI_REDUCE : e == EPI_HEAD_DET ? EPI_HEAD : e == EPI_OUT_DET ? EPI_OUT
       : e == EPI_DRELU_DET ? EPI_DRELU : e;
}
__host__ __device__ constexpr bool epi_det(int e) { return e >= EPI_SLICE; }
enum : int { ACT_NONE = 0, ACT_RELU = 1, ACT_TANH = 2, ACT_TANH_APPROX = 3 };

// Epilogue arguments. Slot meaning per epilogue kind:
//   LINEAR : v = acc + bias[n]; act(v) -> out_hi (bf16) [, out_lo (bf16 residual)] [, out_f32]
//   HEAD   : tile columns [0,half) are mu, [half,BLOCK_N) are logvar of the same latent columns.
//            mu -> out_f32, logvar -> out_f32_b, eps <- in0 (f32 [M, L], NULL = 0),
//            z = mu + eps*exp(lv/2) -> out_hi/out_lo (optional), loss_acc[0] += sum(1 + lv - mu^2 - e^lv)
//   OUT    : xh = tanh(acc + bias[n]) -> out_f32 (optional); x <- in0 (bf16 hi) [+ in1 (bf16 lo)];
//            loss_acc[0] += sum((xh-x)^2); da = c0*(xh-x)*(1-xh^2) -> out_hi/out_lo
//   DRELU  : v = acc * [in0[m,n] > 0] (in0 bf16, optional) -> out_hi/out_lo
//   REDUCE : out_f32[m, n] (+)= acc   (TMA reduce-add when accumulate != 0, plain store otherwise): weight
//            gradients and the split-K latent dgrad
//   OUT / DRELU additionally accumulate the column sums of what they emit into `colsum` (the bias gradient of the
//   layer whose pre-activation gradient this is: db = sum_b da), so no separate reduction kernel is needed.
struct EpiArgs {
  const float* bias;
  __nv_bfloat16* out_hi;
  __nv_bfloat16* out_lo;
  float* out_f32;
  float* out_f32_b;
  const void* in0;
  const void* in1;
  const void* in2;  // DLATENT: mu
  double* loss_acc;
  float* colsum;  // OUT / DRELU: colsum[c] += sum over rows of the emitted values (bias gradients)
  int ldo;   // leading dimension (elements) of out_hi/out_lo/out_f32 and (when ldi == 0) of the bf16 inputs in0/in1
  int ldi;   // OUT: leading dimension of in0/in1 when it differs from ldo (frames read in place from a sample span:
             // row pitch = hop, rows overlap); 0 = ldo
  int act;   // LINEAR / OUT activation
  int L;     // HEAD latent width
  int accumulate;
  float c0;
  int ldp;   // deterministic kinds: SLICE slice stride (rows); OUT_DET / DRELU_DET row pitch of the colsum partials
};

struct alignas(64) GemmParams {
  CUtensorMap tmA[kMaxPasses];
  CUtensorMap tmB[kMaxPasses];
  CUtensorMap tmOutHi;    // bf16 output plane (box 64 cols x 128 rows, 128B swizzle)
  CUtensorMap tmOutLo;    // bf16 residual plane (fp32 emulation)
  CUtensorMap tmOutF32;   // fp32 output (box 32 cols x 128 rows, 128B swizzle)
  CUtensorMap tmOutF32b;  // HEAD: logvar
  CUtensorMap tmSide;     // side input in0: bf16 (box 64 x 128) for OUT / DRELU, fp32 (box 32 x 128) for HEAD
  int M, N, K;
  int num_passes;
  int m_blocks, n_blocks;  // m_blocks counts 128*CG-row tiles
  int k_splits, kb_per_split, kb_total;
  int b_tile_stride;  // K-major B: row advance per n-block
  int b_half_stride;  // K-major B: row offset of the second half-tile load
  int debug;          // experiments only (env RVAE_DEBUG, CG == 1): 1 = no MMA issue, 2 = no TMA loads
  unsigned long long* trace;  // experiments only (rvae_debug_set_trace): per-CTA, per-tile role timestamps
  // Tile-level dependencies between the two problems of a fused launch (a layer and the layer that consumes its
  // output): after the stores of a tile of row block m have completed, each epilogue team adds 1 to dep_signal[m];
  // a unit of row block m loads its A operand only once dep_wait[m] has reached dep_target.
  unsigned int* dep_signal;
  const unsigned int* dep_wait;
  unsigned int dep_target;
  EpiArgs epi;
};

// CG = CTAs cooperating on one tile (tcgen05 cta_group): 1 -> 128 x BLOCK_N tile per CTA; 2 -> a CTA pair computes a
// 256 x BLOCK_N tile, each CTA staging its own 128 rows of A and HALF of the B tile (the pair's tensor cores read
// both halves), which cuts L2->smem traffic per FLOP by a third and doubles the MMA's M.
template <int BLOCK_N, int CG>
struct GemmCfg {
  static constexpr int kABytes = kBlockM * kBlockK * 2;
  static constexpr int kBBytes = (BLOCK_N / CG) * kBlockK * 2;  // per CTA
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kSlotRegion = kEpiTeams * kSlotsPerTeam * kSlotBytes;  // 96 KB of epilogue slots
  static constexpr int kBiasFloats = BLOCK_N / 2 > 128 ? BLOCK_N / 2 : 128;   // a team's own columns of the tile
  static constexpr int kBiasBytes = kEpiTeams * kBiasFloats * 4;
  static constexpr int kCsumBytes = kEpiTeams * 2 * 64 * 4;
  static constexpr int kBarrierBytes = 256;                                   // <= 26 mbarriers + the TMEM slot
  static constexpr int kBudget = 232448 - kSlotRegion - kBiasBytes - kCsumBytes - kBarrierBytes;  // 227 KB per CTA
  static constexpr int kStages = kBudget / kStageBytes > 8 ? 8 : kBudget / kStageBytes;
  static constexpr int kAccStages = 2;
  static constexpr int kTmemCols = (kAccStages * BLOCK_N <= 256) ? 256 : 512;
  static constexpr int kSmemBytes = kStages * kStageBytes + kSlotRegion + kBiasBytes + kCsumBytes + kBarrierBytes;
  static_assert(kStages >= 2, "pipeline too shallow");
};

// Timeline trace (debug): per CTA a 16-word header then kTraceTiles x kTraceEvents clock64() stamps.
//   header: 0 globaltimer at entry, 1 clock at entry, 2 clock after setup, 3 clock after the PDL wait,
//           4 clock when the producer finished, 5 clock at exit, 6 globaltimer at exit
//   events: 0/1 producer tile begin / last load issued; 2/3 MMA before / after the accumulator-free wait,
//           4 first operands landed, 5 tile committed; 6/7 epilogue team 0 accumulator ready / tile released,
//           8/9 the same for team 1; 10..13 team 0's first unit: side input landed / accumulator in registers /
//           staged / store issued; 14/15 its second unit: side input landed / store issued
constexpr int kTraceHeader = 16;
constexpr int kTraceTiles = 24;
constexpr int kTraceEvents = 16;
constexpr int kTraceCtaWords = kTraceHeader + kTraceTiles * kTraceEvents;
__device__ __forceinline__ unsigned long long global_timer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void trace_hdr(const unsigned long long* trace, int word, unsigned long long v) {
  if (trace) const_cast<unsigned long long*>(trace)[static_cast<size_t>(blockIdx.x) * kTraceCtaWords + word] = v;
}
__device__ __forceinline__ void trace_ev(const unsigned long long* trace, int tile_iter, int ev) {
  if (trace && tile_iter < kTraceTiles)
    const_cast<unsigned long long*>(trace)[static_cast<size_t>(blockIdx.x) * kTraceCtaWords + kTraceHeader +
                                           tile_iter * kTraceEvents + ev] = clock64();
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <int COUNT>
__device__ __forceinline__ void load_row_bf16(const __nv_bfloat16* row, float (&v)[COUNT]) {
  const uint4* s = reinterpret_cast<const uint4*>(row);
#pragma unroll
  for (int i = 0; i < COUNT / 8; ++i) {
    uint4 t = __ldg(s + i);
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&t);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float2 f = __bfloat1622float2(h[j]);
      v[8 * i + 2 * j] = f.x;
      v[8 * i + 2 * j + 1] = f.y;
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Epilogue slots. Eight epilogue warps form two TEAMS of four (one warp per TMEM lane quarter, one output row per
// thread). The work units of a tile (64-column bf16 sub-tiles, 32-column fp32 sub-tiles) alternate between the
// teams. A team owns three 16 KB slots (128 rows x 128 bytes, 128B-swizzled: 16-byte chunk c of row r lives at chunk
// c ^ (r & 7), conflict-free for row-per-thread accesses) and uses them round-robin, one slot per unit:
//   [TMA load of the unit's side input, issued at the start of the tile] -> row owners read it, compute, write the
//   result in place -> fence.proxy.async -> team barrier -> one thread issues the TMA store (reduce-add) and then
//   waits until at most ONE store is still reading smem (cp.async.bulk.wait_group.read 1).
// Invariant: whenever the issuer passes a team barrier, every store but the most recent one has released its slot.
// A unit writes the slot used three units earlier, whose store was the most recent one two barriers ago - so by
// the time a thread has passed the previous unit's barrier that slot is free, and no store-read latency is ever on
// the critical path.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void team_bar_sync(int team) {
  asm volatile("bar.sync %0, 128;" ::"r"(team + 1) : "memory");
}
__device__ __forceinline__ uint4* slot_chunk(uint8_t* slot, int r, int c) {
  return reinterpret_cast<uint4*>(slot + r * 128 + ((c ^ (r & 7)) << 4));
}
// 64 fp32 values -> bf16 into the 8 chunks of row r
__device__ __forceinline__ void stage_bf16(uint8_t* slot, int r, const float* v) {
#pragma unroll
  for (int i = 0; i < 8; ++i)
    *slot_chunk(slot, r, i) =
        make_uint4(ptx::pack_bf16x2(v[8 * i + 0], v[8 * i + 1]), ptx::pack_bf16x2(v[8 * i + 2], v[8 * i + 3]),
                   ptx::pack_bf16x2(v[8 * i + 4], v[8 * i + 5]), ptx::pack_bf16x2(v[8 * i + 6], v[8 * i + 7]));
}
__device__ __forceinline__ float bf16_residual(float v) { return v - __bfloat162float(__float2bfloat16_rn(v)); }
__device__ __forceinline__ void stage_bf16_residual(uint8_t* slot, int r, const float* v) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    float q[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) q[j] = bf16_residual(v[8 * i + j]);
    *slot_chunk(slot, r, i) = make_uint4(ptx::pack_bf16x2(q[0], q[1]), ptx::pack_bf16x2(q[2], q[3]),
                                         ptx::pack_bf16x2(q[4], q[5]), ptx::pack_bf16x2(q[6], q[7]));
  }
}
// 32 fp32 values -> the 8 chunks of row r
__device__ __forceinline__ void stage_f32(uint8_t* slot, int r, const float* v) {
#pragma unroll
  for (int i = 0; i < 8; ++i)
    *slot_chunk(slot, r, i) = make_uint4(__float_as_uint(v[4 * i]), __float_as_uint(v[4 * i + 1]),
                                         __float_as_uint(v[4 * i + 2]), __float_as_uint(v[4 * i + 3]));
}
// row r of a bf16 slot (64 values) / an fp32 slot (32 values) -> registers
__device__ __forceinline__ void unstage_bf16(uint8_t* slot, int r, float* v) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const uint4 t = *slot_chunk(slot, r, i);
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&t);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 f = __bfloat1622float2(h[j]);
      v[8 * i + 2 * j] = f.x;
      v[8 * i + 2 * j + 1] = f.y;
    }
  }
}
__device__ __forceinline__ void unstage_f32(uint8_t* slot, int r, float* v) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const uint4 t = *slot_chunk(slot, r, i);
    v[4 * i] = __uint_as_float(t.x); v[4 * i + 1] = __uint_as_float(t.y);
    v[4 * i + 2] = __uint_as_float(t.z); v[4 * i + 3] = __uint_as_float(t.w);
  }
}

// Column sums of a [32 rows (lanes) x 64 columns] register tile: butterfly reduce-scatter over the lanes (62
// shuffles); afterwards lane l holds the sums of columns 2l and 2l+1 in v[0], v[1]. Destroys v.
__device__ __forceinline__ void warp_colsum64(float* v, int lane) {
#pragma unroll
  for (int step = 0; step < 5; ++step) {
    const int half = 32 >> step;          // values kept per lane after this step
    const int mask = 16 >> step;
    const bool upper = (lane & mask) != 0;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      if (j < half) {
        // keep columns [0, half) if the mask bit of this lane is clear, [half, 2*half) otherwise
        const float send = upper ? v[j] : v[j + half];
        const float keep = upper ? v[j + half] : v[j];
        v[j] = keep + __shfl_xor_sync(0xffffffffu, send, mask);
      }
    }
  }
}

// The same for a [32 rows x 16 columns] tile (15 + 1 shuffles): afterwards lane l holds the sum of column l >> 1
// in v[0] (both lanes of a pair hold it). Destroys v.
__device__ __forceinline__ void warp_colsum16(float* v, int lane) {
#pragma unroll
  for (int step = 0; step < 4; ++step) {
    const int half = 8 >> step;
    const int mask = 16 >> step;
    const bool upper = (lane & mask) != 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (j < half) {
        const float send = upper ? v[j] : v[j + half];
        const float keep = upper ? v[j + half] : v[j];
        v[j] = keep + __shfl_xor_sync(0xffffffffu, send, mask);
      }
    }
  }
  v[0] += __shfl_xor_sync(0xffffffffu, v[0], 1);
}

// Accurate tanh is only used by the fp32-emulation path; kept out of line so the hot epilogues stay small enough for
// the instruction cache.
static __device__ __noinline__ float tanh_accurate(float x) { return tanhf(x); }

template <int COUNT>
__device__ __forceinline__ void apply_act(float (&v)[COUNT], int act) {
  if (act == ACT_RELU) {
#pragma unroll
    for (int q = 0; q < COUNT; ++q) v[q] = fmaxf(v[q], 0.f);
  } else if (act == ACT_TANH_APPROX) {
#pragma unroll
    for (int q = 0; q < COUNT; ++q) v[q] = ptx::tanh_approx(v[q]);
  } else if (act == ACT_TANH) {
#pragma unroll
    for (int q = 0; q < COUNT; ++q) v[q] = tanh_accurate(v[q]);
  }
}

// One epilogue team's view of its slots.
struct Team {
  uint8_t* slots;     // kSlotsPerTeam x kSlotBytes
  uint64_t* in_bar;   // one mbarrier per slot: completion of the TMA load of a side input
  float* bias_s;      // bias strip of the team's own columns of the current tile
  float* csum_s;      // 2 x 64 floats: per-unit column sums, combined across the team's four warps (double-buffered)
  uint32_t use;       // running slot-use counter (identical in all threads of the team)
  uint32_t in_phase;  // bit s: parity of in_bar[s]
  uint32_t cs_par;    // which of the two column-sum strips the next unit uses
  int team;
  bool issuer;

  __device__ __forceinline__ uint8_t* slot(uint32_t u) const { return slots + (u % kSlotsPerTeam) * kSlotBytes; }
  __device__ __forceinline__ void sync() const { team_bar_sync(team); }
  // issuer only: start the TMA load of a side tile into the slot of use u
  __device__ __forceinline__ void load(uint32_t u, const CUtensorMap* tm, int c0, int c1) const {
    uint64_t* bar = &in_bar[u % kSlotsPerTeam];
    ptx::mbar_arrive_expect_tx(bar, kSlotBytes);
    ptx::tma_load_2d(slot(u), tm, bar, c0, c1);
  }
  // all threads: wait for the side tile of use u
  __device__ __forceinline__ void wait_load(uint32_t u) {
    const uint32_t s = u % kSlotsPerTeam;
    ptx::mbar_wait(&in_bar[s], (in_phase >> s) & 1u);
    in_phase ^= 1u << s;
  }
  // all threads, after writing their row of the slot of use u: publish it and hand it to the TMA unit
  __device__ __forceinline__ void store(uint32_t u, const CUtensorMap* tm, int c0, int c1, bool reduce) const {
    ptx::fence_proxy_async_smem();
    sync();
    if (issuer) {
      if (reduce) ptx::tma_reduce_add_2d(tm, slot(u), c0, c1);
      else ptx::tma_store_2d(tm, slot(u), c0, c1);
      ptx::tma_store_commit();
      ptx::tma_store_wait_read<1>();
    }
  }
  // slow paths (fp32 emulation): every slot is free and every thread knows it
  __device__ __forceinline__ void drain() const {
    if (issuer) ptx::tma_store_wait_read<0>();
    sync();
  }
};

// ---------------------------------------------------------------------------------------------------------------
// A kernel runs one GEMM ("problem") or two independent ones fused into a single persistent launch (the dgrad and the
// weight-gradient GEMM of a backward stage): the units of both share the CTAs' pipelines, so the machine is filled by
// a mixed tile list instead of two partially filled waves and one kernel boundary disappears. Per-tile code is
// templated on the problem's Kind; the role loops just dispatch.
// ---------------------------------------------------------------------------------------------------------------
template <int A_MAJOR_, int B_MAJOR_, int EPI_>
struct Kind {
  static constexpr int A = A_MAJOR_, B = B_MAJOR_, EPI = EPI_;
};

constexpr int kSchedMax = 16;  // units per CTA group in a host-built schedule (entries < 0 terminate the list)

constexpr int kMaxChain = 4;    // problems per fused launch
struct alignas(64) ChainParams {
  GemmParams p[kMaxChain];
  const int* sched;           // [groups][kSchedMax] unit indices in the combined unit space
  int base[kMaxChain + 1];    // problem i owns units [base[i], base[i + 1]); unused problems are empty ranges
};

// Units of one CTA group: strided over a single problem's unit space, or read from the schedule table.
struct UnitIter {
  const int* sched;
  int pos, u, stride, total;
  __device__ __forceinline__ UnitIter(const int* sched_, int group_id, int num_groups, int total_)
      : sched(sched_ ? sched_ + group_id * kSchedMax : nullptr), pos(0), u(group_id), stride(num_groups), total(total_) {}
  __device__ __forceinline__ bool next(int& unit) {
    if (sched) {
      if (pos >= kSchedMax) return false;
      unit = __ldg(sched + pos);
      ++pos;
      return unit >= 0;
    }
    if (u >= total) return false;
    unit = u;
    u += stride;
    return true;
  }
};

// smem carve-up and CTA identity shared by the three roles
struct Shared {
  uint8_t* smem;
  uint8_t* slot_base;
  float* bias_strips;
  float* csum_strips;
  uint64_t* full_bar;
  uint64_t* empty_bar;
  uint64_t* tmem_full_bar;
  uint64_t* tmem_empty_bar;
  uint64_t* in_bars;
  uint32_t tmem_base;
  uint32_t cta_rank;
  bool leader;
};

struct TileCoord {
  int ks, n_blk, m_blk, m0, kb_begin, kb_count;
};
template <int CG>
__device__ __forceinline__ TileCoord decode_unit(const GemmParams& p, int u, uint32_t cta_rank) {
  TileCoord t;
  const int tiles = p.m_blocks * p.n_blocks;
  t.ks = u / tiles;
  const int tile = u - t.ks * tiles;
  t.n_blk = tile / p.m_blocks;
  t.m_blk = tile - t.n_blk * p.m_blocks;
  t.m0 = (t.m_blk * CG + static_cast<int>(cta_rank)) * kBlockM;
  t.kb_begin = t.ks * p.kb_per_split;
  t.kb_count = min(p.kb_per_split, p.kb_total - t.kb_begin);
  return t;
}

struct ProdState {
  uint32_t stage, phase;
  bool slot_free;
};

template <class KD, int BLOCK_N, int CG>
__device__ __forceinline__ void produce_unit(const GemmParams& p, int u, ProdState& ps, const Shared& sh, int titer) {
  using Cfg = GemmCfg<BLOCK_N, CG>;
  constexpr int kStages = Cfg::kStages;
  constexpr int A_MAJOR = KD::A, B_MAJOR = KD::B;
  trace_ev(p.trace, titer, 0);
  const TileCoord t = decode_unit<CG>(p, u, sh.cta_rank);
  uint32_t stage = ps.stage, phase = ps.phase;
  bool slot_free = ps.slot_free;
#if RVAE_EXPERIMENTS
  if (p.dep_wait != nullptr) {
    // the rows of this unit's A operand are produced by tiles of the other problem of this launch: wait until all
    // of them have been stored (schedules list every producer unit before any consumer unit, so this cannot deadlock)
    const unsigned int* flag = p.dep_wait + t.m_blk;
    const long long t0 = clock64();
    while (ptx::ld_acquire_gpu(flag) < p.dep_target) {
      __nanosleep(64);
      if (clock64() - t0 > 2000000000ll) {
        printf("rvae: tile dependency timeout block %d row block %d (%u of %u)\n", (int)blockIdx.x, t.m_blk,
               ptx::ld_acquire_gpu(flag), p.dep_target);
        __trap();
      }
    }
    ptx::fence_proxy_async_all();  // generic-proxy acquire -> async-proxy (TMA) reads of that data
  }
#endif
  for (int pass = 0; pass < p.num_passes; ++pass) {
    const CUtensorMap* tmA = &p.tmA[pass];
    const CUtensorMap* tmB = &p.tmB[pass];
    for (int kb = t.kb_begin; kb < t.kb_begin + t.kb_count; ++kb) {
      ptx::mbar_wait_probed(slot_free, &sh.empty_bar[stage], phase ^ 1);
      {  // probe the NEXT slot now: the probe's latency overlaps the TMA issue below
        const uint32_t ns = (stage + 1 == kStages) ? 0u : stage + 1;
        const uint32_t np = (stage + 1 == kStages) ? phase ^ 1u : phase;
        slot_free = ptx::mbar_try_wait(&sh.empty_bar[ns], np ^ 1);
      }
      uint64_t* fb = &sh.full_bar[stage];
#if RVAE_EXPERIMENTS
      if (CG == 1 && (p.debug & 2)) {  // experiment: measure the MMA side alone (operands are stale smem)
        ptx::mbar_arrive(fb);
        if (++stage == kStages) { stage = 0; phase ^= 1; }
        continue;
      }
#endif
      if constexpr (CG == 1) {
        ptx::mbar_arrive_expect_tx(fb, Cfg::kStageBytes);
      } else {
        // Both CTAs' loads complete_tx on the LEADER's barrier; the leader alone arrives, announcing the pair's
        // bytes. The peer sends no arrive (a cluster-scope release per k-block would throttle its producer):
        // it cannot run a phase ahead because its smem slot is only freed by the commit that follows the MMAs
        // which consumed this phase, and a complete_tx that lands before the leader's expect_tx merely leaves
        // the tx-count transiently negative while the leader's arrival is still pending.
        if (sh.leader) ptx::mbar_arrive_expect_tx(fb, 2 * Cfg::kStageBytes);
      }
      uint8_t* sA = sh.smem + stage * Cfg::kStageBytes;
      uint8_t* sB = sA + Cfg::kABytes;
      const int k0 = kb * kBlockK;
      if constexpr (A_MAJOR == MAJOR_K) {
        ptx::tma_load_2d_cg<CG>(sA, tmA, fb, k0, t.m0);
      } else {
#pragma unroll
        for (int i = 0; i < kBlockM / 64; ++i)
          ptx::tma_load_2d_cg<CG>(sA + i * (kBlockK * 128), tmA, fb, t.m0 + i * 64, k0);
      }
      if constexpr (B_MAJOR == MAJOR_K) {
        // the B tile is staged as two boxes of BLOCK_N/2 rows: CG == 1 loads both, CG == 2 one per CTA
        const int r0 = t.n_blk * p.b_tile_stride;
        if constexpr (CG == 1) {
#pragma unroll
          for (int h = 0; h < 2; ++h)
            ptx::tma_load_2d_cg<1>(sB + h * (Cfg::kBBytes / 2), tmB, fb, k0, r0 + h * p.b_half_stride);
        } else {
          ptx::tma_load_2d_cg<2>(sB, tmB, fb, k0, r0 + static_cast<int>(sh.cta_rank) * p.b_half_stride);
        }
      } else {
        const int n0 = t.n_blk * BLOCK_N + static_cast<int>(sh.cta_rank) * (BLOCK_N / CG);
#pragma unroll
        for (int i = 0; i < BLOCK_N / CG / 64; ++i)
          ptx::tma_load_2d_cg<CG>(sB + i * (kBlockK * 128), tmB, fb, n0 + i * 64, k0);
      }
      if (++stage == kStages) { stage = 0; phase ^= 1; }
    }
  }
  ps.stage = stage; ps.phase = phase; ps.slot_free = slot_free;
  trace_ev(p.trace, titer, 1);
}

struct MmaState {
  uint32_t stage, phase, as, aphase;
  bool data_ready;
};

template <class KD, int BLOCK_N, int CG>
__device__ __forceinline__ void mma_unit(const GemmParams& p, int u, MmaState& ms, const Shared& sh, int titer) {
  using Cfg = GemmCfg<BLOCK_N, CG>;
  constexpr int kStages = Cfg::kStages;
  constexpr int A_MAJOR = KD::A, B_MAJOR = KD::B;
  constexpr uint32_t kIdesc = ptx::umma_idesc_bf16(kBlockM * CG, BLOCK_N, A_MAJOR, B_MAJOR);
  const TileCoord t = decode_unit<CG>(p, u, sh.cta_rank);
  const int iters = t.kb_count * p.num_passes;
  uint32_t stage = ms.stage, phase = ms.phase;
  bool data_ready = ms.data_ready;
  trace_ev(p.trace, titer, 2);
  ptx::mbar_wait(&sh.tmem_empty_bar[ms.as], ms.aphase ^ 1);
  ptx::tc_fence_after();
  trace_ev(p.trace, titer, 3);
  const uint32_t d_tmem = sh.tmem_base + ms.as * BLOCK_N;
  for (int it = 0; it < iters; ++it) {
    ptx::mbar_wait_probed(data_ready, &sh.full_bar[stage], phase);
    {  // probe the NEXT stage now: the MMA issue below hides the probe's latency, so the tensor pipe does not
       // drain while this thread waits on a barrier that has long completed
      const uint32_t ns = (stage + 1 == kStages) ? 0u : stage + 1;
      const uint32_t np = (stage + 1 == kStages) ? phase ^ 1u : phase;
      data_ready = ptx::mbar_try_wait(&sh.full_bar[ns], np);
    }
    ptx::tc_fence_after();
    if (it == 0) trace_ev(p.trace, titer, 4);
#if RVAE_EXPERIMENTS
    if (CG == 1 && (p.debug & 1)) {  // experiment: measure the TMA side alone
      ptx::mbar_arrive(&sh.empty_bar[stage]);
      if (++stage == kStages) { stage = 0; phase ^= 1; }
      continue;
    }
#endif
    const uint32_t a_addr = ptx::smem_u32(sh.smem + stage * Cfg::kStageBytes);
    const uint32_t b_addr = a_addr + Cfg::kABytes;
#pragma unroll
    for (int k = 0; k < kBlockK / kUmmaK; ++k) {
      const uint64_t adesc = (A_MAJOR == MAJOR_K) ? ptx::umma_desc_sw128(a_addr + k * (kUmmaK * 2), 0, 1024)
                                                  : ptx::umma_desc_sw128(a_addr + k * (kUmmaK * 128), kBlockK * 128, 1024);
      const uint64_t bdesc = (B_MAJOR == MAJOR_K) ? ptx::umma_desc_sw128(b_addr + k * (kUmmaK * 2), 0, 1024)
                                                  : ptx::umma_desc_sw128(b_addr + k * (kUmmaK * 128), kBlockK * 128, 1024);
      ptx::umma_bf16<CG>(d_tmem, adesc, bdesc, kIdesc, (it > 0 || k > 0) ? 1u : 0u);
    }
    ptx::umma_commit<CG>(&sh.empty_bar[stage]);  // frees the smem slot (in both CTAs) once these MMAs have read it
    if (++stage == kStages) { stage = 0; phase ^= 1; }
  }
#if RVAE_EXPERIMENTS
  if (CG == 1 && (p.debug & 1)) ptx::mbar_arrive(&sh.tmem_full_bar[ms.as]);
  else
#endif
  ptx::umma_commit<CG>(&sh.tmem_full_bar[ms.as]);  // accumulator complete -> epilogue (of both CTAs)
  trace_ev(p.trace, titer, 5);
  if (++ms.as == Cfg::kAccStages) { ms.as = 0; ms.aphase ^= 1; }
  ms.stage = stage; ms.phase = phase; ms.data_ready = data_ready;
}

// Per-thread state of an epilogue warp
struct EpiState {
  Team tm;
  uint32_t as, aphase;
  float loss_local;
  int team, quarter, row, team_tid, lane;
  uint32_t lane_base;
};

template <class KD, int BLOCK_N, int CG>
__device__ __forceinline__ void epilogue_unit(const GemmParams& p, int u, EpiState& es, const Shared& sh, int titer) {
  using Cfg = GemmCfg<BLOCK_N, CG>;
  constexpr int EPI = epi_base(KD::EPI);
  constexpr bool kDet = epi_det(KD::EPI);
  const EpiArgs& e = p.epi;
  Team& tm = es.tm;
  const int team = es.team, row = es.row, team_tid = es.team_tid, lane = es.lane;
  uint64_t* tmem_full_bar = sh.tmem_full_bar;
  uint32_t& as = es.as;
  uint32_t& aphase = es.aphase;
  float& loss_local = es.loss_local;
  const bool dual = e.out_lo != nullptr;
  const bool tr = team_tid == 0 && team == 0;
  const TileCoord tc = decode_unit<CG>(p, u, sh.cta_rank);
  const int n_blk = tc.n_blk, m0 = tc.m0;
  const int m = m0 + row;
  const bool row_ok = m < p.M;
  const uint32_t t_acc = sh.tmem_base + es.lane_base + as * BLOCK_N;
  const int r32 = m0 / 32 + es.quarter;   // deterministic kinds: this warp's 32-row block of the problem
  (void)lane; (void)tr; (void)dual; (void)row_ok; (void)m; (void)r32;

      if constexpr (EPI == EPI_HEAD) {
        // ---- tile columns [0, kHalf) = mu, [kHalf, BLOCK_N) = logvar of latent columns n_blk*kHalf ..; a team owns
        //      64 latent columns (BLOCK_N = 128: team 0 only). Slots A = 0, B = 1, C = 2 (drained once per tile):
        //        eps[0:32] -> A, eps[32:64] -> B (TMA loads, issued before the accumulator is ready)
        //        mu[0:32] in place in A, lv[0:32] -> C, stored; mu[32:64] in place in B, stored;
        //        then lv[32:64] -> A and z[0:64] (bf16) -> C, stored.
        constexpr int kHalf = BLOCK_N / 2;
        static_assert(kHalf / 64 <= kEpiTeams, "one HEAD unit per team per tile");
        const int L = e.L;
        const bool active = team < kHalf / 64;
        const int col0 = n_blk * kHalf + team * 64;  // latent column of this team's unit
        const bool has_eps = e.in0 != nullptr;
        if (active && team_tid < 128) {
          const int i = team_tid;  // strip: [0,64) mu bias, [64,128) logvar bias of the team's 64 latent columns
          tm.bias_s[i] = (i < 64) ? __ldg(e.bias + col0 + i) : __ldg(e.bias + L + col0 + i - 64);
        }
        if (tm.issuer && active) {
          ptx::tma_store_wait_read<0>();  // the previous tile's stores have released all three slots
          if (has_eps) {
            tm.load(0, &p.tmSide, col0, m0);
            tm.load(1, &p.tmSide, col0 + 32, m0);
          }
        }
        ptx::mbar_wait(&tmem_full_bar[as], aphase);
        ptx::tc_fence_after();
        if (team_tid == 0) trace_ev(p.trace, titer, 6 + 2 * team);
        tm.sync();  // bias strip visible; slots known to be free
        if (active) {
          float z[64];
          float lv1[32];
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int c = team * 64 + h * 32;  // accumulator column of mu; logvar sits kHalf further
            uint32_t rm[32], rl[32];
            ptx::tmem_ld_32x32(t_acc + c, rm);
            ptx::tmem_ld_32x32(t_acc + kHalf + c, rl);
            if (has_eps) tm.wait_load(h);
            ptx::tmem_ld_wait();
            uint8_t* s_mu = tm.slot(h);        // eps in, mu out (in place)
            uint8_t* s_lv = tm.slot(2);        // h == 0 only
#pragma unroll
            for (int i = 0; i < 8; ++i) {      // one 16-byte chunk (4 columns) at a time keeps the register count low
              float eps[4] = {0.f, 0.f, 0.f, 0.f};
              if (has_eps) {
                const uint4 t = *slot_chunk(s_mu, row, i);
                eps[0] = __uint_as_float(t.x); eps[1] = __uint_as_float(t.y);
                eps[2] = __uint_as_float(t.z); eps[3] = __uint_as_float(t.w);
              }
              float mu[4], lv[4];
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const int jj = 4 * i + q;
                mu[q] = __uint_as_float(rm[jj]) + tm.bias_s[h * 32 + jj];
                lv[q] = __uint_as_float(rl[jj]) + tm.bias_s[64 + h * 32 + jj];
                const float sig = expf(0.5f * lv[q]);
                z[h * 32 + jj] = fmaf(eps[q], sig, mu[q]);
                if (row_ok) loss_local += (1.f + lv[q]) - fmaf(mu[q], mu[q], sig * sig);
                if (h == 1) lv1[jj] = lv[q];
              }
              *slot_chunk(s_mu, row, i) = make_uint4(__float_as_uint(mu[0]), __float_as_uint(mu[1]),
                                                     __float_as_uint(mu[2]), __float_as_uint(mu[3]));
              if (h == 0)
                *slot_chunk(s_lv, row, i) = make_uint4(__float_as_uint(lv[0]), __float_as_uint(lv[1]),
                                                       __float_as_uint(lv[2]), __float_as_uint(lv[3]));
            }
            ptx::fence_proxy_async_smem();
            if (h == 0) {
              tm.sync();
              if (tm.issuer) {
                ptx::tma_store_2d(&p.tmOutF32, tm.slot(0), col0, m0);
                ptx::tma_store_2d(&p.tmOutF32b, tm.slot(2), col0, m0);
                ptx::tma_store_commit();
              }
            } else {
              if (tm.issuer) ptx::tma_store_wait_read<0>();  // slots A and C are free again ...
              tm.sync();                                      // ... and everyone knows
              if (tm.issuer) {
                ptx::tma_store_2d(&p.tmOutF32, tm.slot(1), col0 + 32, m0);
                ptx::tma_store_commit();
              }
              stage_f32(tm.slot(0), row, lv1);
              if (e.out_hi) stage_bf16(tm.slot(2), row, z);
              ptx::fence_proxy_async_smem();
              tm.sync();
              if (tm.issuer) {
                ptx::tma_store_2d(&p.tmOutF32b, tm.slot(0), col0 + 32, m0);
                if (e.out_hi) ptx::tma_store_2d(&p.tmOutHi, tm.slot(2), col0, m0);
                ptx::tma_store_commit();
              }
            }
          }
          if constexpr (kDet) {
            const float kl = warp_sum(loss_local);
            loss_local = 0.f;
            if (lane == 0 && e.loss_acc) e.loss_acc[static_cast<size_t>(r32) * (L / 64) + col0 / 64] = kl;
          }
          if (e.out_hi && dual) {
            tm.drain();
            stage_bf16_residual(tm.slot(0), row, z);
            ptx::fence_proxy_async_smem();
            tm.sync();
            if (tm.issuer) {
              ptx::tma_store_2d(&p.tmOutLo, tm.slot(0), col0, m0);
              ptx::tma_store_commit();
            }
          }
        }
      } else if constexpr (EPI == EPI_DLATENT) {
        // ---- latent dgrad with the backward of reparameterize + the KL gradient fused (rawvae/model.py:24-26,45):
        //        dz = acc;  sigma = exp(lv / 2)
        //        d_mu = dz + c0 * mu                          -> out_hi[:, n]      (bf16, leading dimension ldo = 2L)
        //        d_lv = dz * eps * sigma / 2 + c0 (sigma^2 - 1) / 2 -> out_hi[:, L + n]
        //        colsum[n] += sum_rows d_mu, colsum[L + n] += sum_rows d_lv      (db21, db22)
        //      Team t owns the 64-column groups t, t + 2 of the tile and walks them in 8-column pieces, one output row
        //      per thread: mu, logvar, eps (fp32) come straight from global memory (one 32-byte sector per array, row
        //      and piece; the next piece's loads are issued before this piece is computed), results go straight back
        //      as 16-byte stores. The volume is small (16 + 4 bytes per latent element) and a CTA pair runs ONE such
        //      tile per launch, so the code is kept short and rolled: a first pass through a long unrolled epilogue
        //      costs more in instruction-cache misses than the whole tile's arithmetic (measured).
        constexpr int kSubs = BLOCK_N / 64;
        constexpr int kUnitsPerTeam = (kSubs + kEpiTeams - 1) / kEpiTeams;
        constexpr int kPieces = kUnitsPerTeam * 8;
        const int L = e.L;
        const float* src[3] = {reinterpret_cast<const float*>(e.in2), reinterpret_cast<const float*>(e.in1),
                               reinterpret_cast<const float*>(e.in0)};  // mu, logvar, eps
        const size_t row_off = static_cast<size_t>(m) * L;
        auto piece_col = [&](int pc) { return n_blk * BLOCK_N + (team + (pc >> 3) * kEpiTeams) * 64 + (pc & 7) * 8; };
        float4 nx[6];  // the next piece's mu[0:8], logvar[0:8], eps[0:8]
        auto load_piece = [&](int pc) {
          const int col = pc < kPieces ? piece_col(pc) : p.N;
          if (row_ok && col < p.N) {
#pragma unroll
            for (int a = 0; a < 3; ++a) {
              const float4* g4 = reinterpret_cast<const float4*>(src[a] + row_off + col);
              nx[2 * a] = __ldg(g4);
              nx[2 * a + 1] = __ldg(g4 + 1);
            }
          } else {
#pragma unroll
            for (int a = 0; a < 6; ++a) nx[a] = make_float4(0.f, 0.f, 0.f, 0.f);
          }
        };
        if (row_ok && !(p.debug & 4)) {
          // written by the forward pass and long evicted: have the L2 fetch this row's inputs while the MMAs run
#pragma unroll
          for (int j = 0; j < kUnitsPerTeam; ++j) {
            const int n0 = n_blk * BLOCK_N + (team + j * kEpiTeams) * 64;
            if (team + j * kEpiTeams < kSubs && n0 < p.N) {
#pragma unroll
              for (int a = 0; a < 3; ++a) ptx::prefetch_l2_bulk(src[a] + row_off + n0, 256u);
            }
          }
        }
        ptx::mbar_wait(&tmem_full_bar[as], aphase);
        ptx::tc_fence_after();
        if (team_tid == 0) trace_ev(p.trace, titer, 6 + 2 * team);
        load_piece(0);
        float* cs_mu = tm.csum_s;        // both column-sum strips are zero between units
        float* cs_lv = tm.csum_s + 64;
        __nv_bfloat16* out_row = e.out_hi + static_cast<size_t>(m) * e.ldo;
#pragma unroll 1
        for (int pc = 0; pc < kPieces; ++pc) {
          const int col = piece_col(pc);
          if (col >= p.N) break;          // (uniform over the team; columns grow with pc)
          uint32_t r[8];
          ptx::tmem_ld_32x8(t_acc + (col - n_blk * BLOCK_N), r);
          float in[24];
#pragma unroll
          for (int a = 0; a < 6; ++a) {
            in[4 * a] = nx[a].x; in[4 * a + 1] = nx[a].y; in[4 * a + 2] = nx[a].z; in[4 * a + 3] = nx[a].w;
          }
          load_piece(pc + 1);
          ptx::tmem_ld_wait();
          float o[16];                    // d_mu[0:8], d_lv[0:8]
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const float d = __uint_as_float(r[q]);
            const float sig = expf(0.5f * in[8 + q]);
            const float gl = 0.5f * e.c0 * (sig * sig - 1.f);
            o[q] = row_ok ? d + e.c0 * in[q] : 0.f;
            o[8 + q] = row_ok ? fmaf(d, 0.5f * in[16 + q] * sig, gl) : 0.f;
          }
          if (row_ok) {
            *reinterpret_cast<uint4*>(out_row + col) =
                make_uint4(ptx::pack_bf16x2(o[0], o[1]), ptx::pack_bf16x2(o[2], o[3]), ptx::pack_bf16x2(o[4], o[5]),
                           ptx::pack_bf16x2(o[6], o[7]));
            *reinterpret_cast<uint4*>(out_row + L + col) =
                make_uint4(ptx::pack_bf16x2(o[8], o[9]), ptx::pack_bf16x2(o[10], o[11]),
                           ptx::pack_bf16x2(o[12], o[13]), ptx::pack_bf16x2(o[14], o[15]));
          }
          if (e.colsum) {
            warp_colsum16(o, lane);       // lane l: sum over the warp's 32 rows of value (l >> 1)
            if ((lane & 1) == 0) {
              const int idx = lane >> 1;
              atomicAdd((idx < 8 ? cs_mu : cs_lv - 8) + (pc & 7) * 8 + idx, o[0]);
            }
            if ((pc & 7) == 7) {          // the group's 64 + 64 column sums are complete: flush and clear the strips
              const int n0 = col - 56;
              tm.sync();
              if (team_tid < 64) {
                atomicAdd(e.colsum + n0 + team_tid, cs_mu[team_tid]);
                atomicAdd(e.colsum + L + n0 + team_tid, cs_lv[team_tid]);
                cs_mu[team_tid] = 0.f;
                cs_lv[team_tid] = 0.f;
              }
              tm.sync();
            }
          }
          if (tr && (pc & 7) == 7) trace_ev(p.trace, titer, 14 + (pc >> 3));   // 14 / 15: group stored
        }
      } else if constexpr (EPI == EPI_REDUCE) {
        ptx::mbar_wait(&tmem_full_bar[as], aphase);
        ptx::tc_fence_after();
        if (team_tid == 0) trace_ev(p.trace, titer, 6 + 2 * team);
        for (int piece = team; piece < BLOCK_N / 32; piece += kEpiTeams) {
          const int n = n_blk * BLOCK_N + piece * 32;
          if (n >= p.N) continue;
          uint32_t r[32];
          ptx::tmem_ld_32x32(t_acc + piece * 32, r);
          ptx::tmem_ld_wait();
          uint8_t* sl = tm.slot(tm.use);
#pragma unroll
          for (int i = 0; i < 8; ++i) *slot_chunk(sl, row, i) = make_uint4(r[4 * i], r[4 * i + 1], r[4 * i + 2], r[4 * i + 3]);
          if constexpr (kDet) {
            if (tc.ks == 0) tm.store(tm.use, &p.tmOutF32, n, m0, false);
            else tm.store(tm.use, &p.tmOutF32b, n, (tc.ks - 1) * e.ldp + m0, false);
          } else {
            tm.store(tm.use, &p.tmOutF32, n, m0, e.accumulate != 0);
          }
          ++tm.use;
        }
      } else {
        // ---- bf16 stream: LINEAR (act), DRELU (mask), OUT (da4): 64-column units, side input prefetched by TMA.
        //      Team t owns the 64-column groups t, t + 2 of the tile (bias strip: its own columns only).
        constexpr int kSubs = BLOCK_N / 64;
        constexpr int kUnitsPerTeam = (kSubs + kEpiTeams - 1) / kEpiTeams;
        static_assert(kUnitsPerTeam <= 2, "side-input prefetch covers at most two units per team and tile");
        constexpr bool kSide = (EPI == EPI_OUT || EPI == EPI_DRELU);
        constexpr bool kBias = (EPI == EPI_LINEAR || EPI == EPI_OUT);
        const bool side = kSide && e.in0 != nullptr && e.out_hi != nullptr;
        const bool do_colsum = kSide && e.colsum != nullptr;
        if constexpr (kBias) {
          if (team_tid < kUnitsPerTeam * 64) {
            const int n = n_blk * BLOCK_N + (team + (team_tid >> 6) * kEpiTeams) * 64 + (team_tid & 63);
            tm.bias_s[team_tid] = (e.bias && n < p.N) ? __ldg(e.bias + n) : 0.f;
          }
        }
        if (side && !dual && tm.issuer) {
          // the slots of the next two uses are free (see the invariant above): start this tile's side loads now,
          // while its MMAs are still running
#pragma unroll
          for (int j = 0; j < kUnitsPerTeam; ++j) {
            const int sub = team + j * kEpiTeams;
            const int n0 = n_blk * BLOCK_N + sub * 64;
            if (sub < kSubs && n0 < p.N) tm.load(tm.use + j, &p.tmSide, n0, m0);
          }
        }
        ptx::mbar_wait(&tmem_full_bar[as], aphase);
        ptx::tc_fence_after();
        if (team_tid == 0) trace_ev(p.trace, titer, 6 + 2 * team);
        if constexpr (kBias) tm.sync();  // bias strip visible
        if (e.out_hi) {
#pragma unroll 1
          for (int j = 0; j < kUnitsPerTeam; ++j) {
            const int sub = team + j * kEpiTeams;
            const int n0 = n_blk * BLOCK_N + sub * 64;
            if (sub >= kSubs || n0 >= p.N) continue;
            // 1) accumulator: both 32-column TMEM loads in flight
            uint32_t r[64];
            ptx::tmem_ld_32x32(t_acc + sub * 64, *reinterpret_cast<uint32_t(*)[32]>(&r[0]));
            ptx::tmem_ld_32x32(t_acc + sub * 64 + 32, *reinterpret_cast<uint32_t(*)[32]>(&r[32]));
            // 2) side input of this unit
            if (dual) {  // fp32 emulation: no prefetch, slots 0 (hi, in place) and 1 (residual plane)
              tm.drain();
              tm.use = 0;
              if (side && tm.issuer) tm.load(0, &p.tmSide, n0, m0);
            }
            if (side) tm.wait_load(tm.use);
            if (tr) trace_ev(p.trace, titer, j == 0 ? 10 : 14);
            ptx::tmem_ld_wait();
            if (tr && j == 0) trace_ev(p.trace, titer, 11);
            uint8_t* sl = tm.slot(tm.use);
            float v[64];
#pragma unroll
            for (int q = 0; q < 64; ++q) v[q] = __uint_as_float(r[q]);
            if constexpr (kBias) {
#pragma unroll
              for (int q = 0; q < 64; q += 4) {
                const float4 b = *reinterpret_cast<const float4*>(tm.bias_s + j * 64 + q);
                v[q] += b.x; v[q + 1] += b.y; v[q + 2] += b.z; v[q + 3] += b.w;
              }
            }
            if constexpr (EPI == EPI_LINEAR) {
              apply_act<64>(v, e.act);
            } else if constexpr (EPI == EPI_DRELU) {
              if (side) {
#pragma unroll
                for (int i = 0; i < 8; ++i) {  // ReLU mask: keep the gradient where the forward activation was > 0
                  const uint4 t = *slot_chunk(sl, row, i);
                  const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
                  for (int q = 0; q < 4; ++q) {
                    // bf16 > 0  <=>  sign clear and magnitude non-zero (per 16-bit half of the word)
                    const uint32_t lo16 = w[q] & 0xffffu, hi16 = w[q] >> 16;
                    if (!(lo16 != 0u && lo16 < 0x8000u)) v[8 * i + 2 * q] = 0.f;
                    if (!(hi16 != 0u && hi16 < 0x8000u)) v[8 * i + 2 * q + 1] = 0.f;
                  }
                }
              }
            } else {  // OUT: xh = tanh(a); d = xh - x; loss += d^2; da = c0 * d * (1 - xh^2)
              apply_act<64>(v, e.act == ACT_TANH_APPROX ? ACT_TANH_APPROX : ACT_TANH);
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                float x[8];
                if (side) {
                  const uint4 t = *slot_chunk(sl, row, i);
                  const __nv_bfloat162* hh = reinterpret_cast<const __nv_bfloat162*>(&t);
#pragma unroll
                  for (int q = 0; q < 4; ++q) {
                    const float2 f = __bfloat1622float2(hh[q]);
                    x[2 * q] = f.x; x[2 * q + 1] = f.y;
                  }
                  if (e.in1 && row_ok) {  // x = hi + lo (fp32 emulation): the residual comes straight from global
                    const uint4 t2 = __ldg(reinterpret_cast<const uint4*>(
                        reinterpret_cast<const __nv_bfloat16*>(e.in1) + static_cast<size_t>(m) * (e.ldi ? e.ldi : e.ldo) + n0 + 8 * i));
                    const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&t2);
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                      const float2 f = __bfloat1622float2(h2[q]);
                      x[2 * q] += f.x; x[2 * q + 1] += f.y;
                    }
                  }
                } else {
#pragma unroll
                  for (int q = 0; q < 8; ++q) x[q] = 0.f;
                }
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                  const float xh = v[8 * i + q];
                  const float d = xh - x[q];
                  if (row_ok) loss_local = fmaf(d, d, loss_local);
                  v[8 * i + q] = row_ok ? e.c0 * d * (1.f - xh * xh) : 0.f;
                }
              }
            }
            stage_bf16(sl, row, v);
            if (dual) stage_bf16_residual(tm.slot(tm.use + 1), row, v);
            if (tr && j == 0) trace_ev(p.trace, titer, 12);
            float* cs = tm.csum_s + (tm.cs_par << 6);
            if (do_colsum) {
              // bias gradient: column sums of this unit over the tile's 128 rows (rows >= M contribute zeros)
              warp_colsum64(v, lane);
              if constexpr (kDet) {   // this warp's 32 rows -> their own partial row, at a fixed index
                *reinterpret_cast<float2*>(e.colsum + static_cast<size_t>(r32) * e.ldp + n0 + 2 * lane) =
                    make_float2(v[0], v[1]);
              } else {
                atomicAdd(cs + 2 * lane, v[0]);
                atomicAdd(cs + 2 * lane + 1, v[1]);
              }
            }
            if constexpr (kDet && EPI == EPI_OUT) {
              const float mse = warp_sum(loss_local);
              loss_local = 0.f;
              if (lane == 0 && e.loss_acc) e.loss_acc[static_cast<size_t>(r32) * (p.N / 64) + n0 / 64] = mse;
            }
            tm.store(tm.use, &p.tmOutHi, n0, m0, false);
            if (dual && tm.issuer) {
              ptx::tma_store_2d(&p.tmOutLo, tm.slot(tm.use + 1), n0, m0);
              ptx::tma_store_commit();
            }
            if (tr) trace_ev(p.trace, titer, j == 0 ? 13 : 15);
            if (do_colsum && !kDet) {
              // the barrier inside store() ordered the four warps' smem atomics before this read; the strip is
              // cleared for its next use two units from now (the other strip serves the unit in between)
              if (team_tid < 64) {
                atomicAdd(e.colsum + n0 + team_tid, cs[team_tid]);
                cs[team_tid] = 0.f;
              }
              tm.cs_par ^= 1u;
            }
            ++tm.use;
          }
        }
        // ---- fp32 stream: LINEAR's fp32 copy / OUT's xhat: 32-column pieces of the team's own column groups
        if constexpr (kBias) {
          if (e.out_f32) {
            if (dual) { tm.drain(); tm.use = 0; }
#pragma unroll 1
            for (int jp = 0; jp < 2 * kUnitsPerTeam; ++jp) {
              const int j = jp >> 1, hf = jp & 1;
              const int sub = team + j * kEpiTeams;
              const int n = n_blk * BLOCK_N + sub * 64 + hf * 32;
              if (sub >= kSubs || n >= p.N) continue;
              uint32_t r[32];
              ptx::tmem_ld_32x32(t_acc + sub * 64 + hf * 32, r);
              ptx::tmem_ld_wait();
              float v[32];
#pragma unroll
              for (int q = 0; q < 32; ++q) v[q] = __uint_as_float(r[q]) + tm.bias_s[j * 64 + hf * 32 + q];
              apply_act<32>(v, (EPI == EPI_OUT && e.act != ACT_TANH_APPROX) ? ACT_TANH : e.act);
              if constexpr (EPI == EPI_OUT) {
                if (!e.out_hi && row_ok) {  // loss-only forward: accumulate the MSE here
                  const size_t off = static_cast<size_t>(m) * (e.ldi ? e.ldi : e.ldo) + n;
                  float x[32];
                  load_row_bf16<32>(reinterpret_cast<const __nv_bfloat16*>(e.in0) + off, x);
                  if (e.in1) {
                    float xl[32];
                    load_row_bf16<32>(reinterpret_cast<const __nv_bfloat16*>(e.in1) + off, xl);
#pragma unroll
                    for (int q = 0; q < 32; ++q) x[q] += xl[q];
                  }
#pragma unroll
                  for (int q = 0; q < 32; ++q) loss_local = fmaf(v[q] - x[q], v[q] - x[q], loss_local);
                }
              }
              stage_f32(tm.slot(tm.use), row, v);
              tm.store(tm.use, &p.tmOutF32, n, m0, false);
              ++tm.use;
            }
          }
        }
      }
      // release the accumulator back to the MMA warp
  ptx::tc_fence_before();
  __syncwarp();
  if (lane == 0) {
    if (CG == 1 || sh.leader) ptx::mbar_arrive(&sh.tmem_empty_bar[as]);
    else ptx::mbar_arrive_remote(&sh.tmem_empty_bar[as], 0);
  }
#if RVAE_EXPERIMENTS
  if (p.dep_signal != nullptr && tm.issuer) {
    // publish this team's part of the tile to the consumer problem: its bulk stores are complete (not merely read)
    ptx::tma_store_wait<0>();
    __threadfence();
    atomicAdd(p.dep_signal + tc.m_blk, 1u);
  }
#endif
  if (team_tid == 0) trace_ev(p.trace, titer, 7 + 2 * team);
  if (++as == Cfg::kAccStages) { as = 0; aphase ^= 1; }
}

struct NoKind {
  static constexpr int A = 0, B = 0, EPI = -1;
};
template <class K>
struct is_kind { static constexpr bool value = true; };
template <>
struct is_kind<NoKind> { static constexpr bool value = false; };

// The problems of a launch as the device code sees them.
struct ProblemSet {
  const GemmParams* p[kMaxChain];
  int base[kMaxChain + 1];
  const int* sched;   // nullptr: one problem, units strided over the CTA groups
};

// call FN<Ki, BLOCK_N, CG>(problem i, unit within problem i, ...) for the problem that owns unit u
#define RVAE_DISPATCH(FN, STATE)                                                                                  \
  do {                                                                                                            \
    if (u < ps.base[1]) {                                                                                         \
      FN<K0, BLOCK_N, CG>(*ps.p[0], u, STATE, sh, titer);                                                         \
    } else if (u < ps.base[2]) {                                                                                  \
      if constexpr (is_kind<K1>::value) FN<K1, BLOCK_N, CG>(*ps.p[1], u - ps.base[1], STATE, sh, titer);          \
    } else if (u < ps.base[3]) {                                                                                  \
      if constexpr (is_kind<K2>::value) FN<K2, BLOCK_N, CG>(*ps.p[2], u - ps.base[2], STATE, sh, titer);          \
    } else {                                                                                                      \
      if constexpr (is_kind<K3>::value) FN<K3, BLOCK_N, CG>(*ps.p[3], u - ps.base[3], STATE, sh, titer);          \
    }                                                                                                             \
  } while (0)

template <int BLOCK_N, int CG, class K0, class K1, class K2, class K3>
__device__ __forceinline__ void gemm_body(const ProblemSet& ps) {
  using Cfg = GemmCfg<BLOCK_N, CG>;
  constexpr int kStages = Cfg::kStages;
  const GemmParams& p = *ps.p[0];  // trace / debug switches come from the first problem

  extern __shared__ __align__(1024) uint8_t smem[];
  Shared sh;
  sh.smem = smem;
  sh.slot_base = smem + kStages * Cfg::kStageBytes;  // 1024-byte aligned (stage sizes are multiples of 1 KB)
  sh.bias_strips = reinterpret_cast<float*>(sh.slot_base + Cfg::kSlotRegion);
  sh.csum_strips = sh.bias_strips + kEpiTeams * Cfg::kBiasFloats;
  sh.full_bar = reinterpret_cast<uint64_t*>(sh.csum_strips + kEpiTeams * 128);
  sh.empty_bar = sh.full_bar + kStages;
  sh.tmem_full_bar = sh.empty_bar + kStages;
  sh.tmem_empty_bar = sh.tmem_full_bar + Cfg::kAccStages;
  sh.in_bars = sh.tmem_empty_bar + Cfg::kAccStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sh.in_bars + kEpiTeams * kSlotsPerTeam);
  static_assert((2 * 8 + 2 * 2 + kEpiTeams * kSlotsPerTeam) * 8 + 4 <= Cfg::kBarrierBytes, "barrier region");

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  sh.cta_rank = (CG == 2) ? ptx::cluster_ctarank() : 0u;
  sh.leader = sh.cta_rank == 0;
  const int group_id = (CG == 2) ? (blockIdx.x >> 1) : blockIdx.x;       // tile-owning unit: CTA or CTA pair
  const int num_groups = (CG == 2) ? (gridDim.x >> 1) : gridDim.x;

  if (threadIdx.x == 0) {
    if ((ptx::smem_u32(smem) & 1023u) != 0) {  // swizzled tiles need the declared 1 KB alignment
      printf("rvae: dynamic shared memory base is not 1024-byte aligned\n");
      __trap();
    }
    trace_hdr(p.trace, 0, global_timer());
    trace_hdr(p.trace, 1, clock64());
  }
  if (warp == 0 && lane == 0) {
#pragma unroll
    for (int q = 0; q < kMaxChain; ++q) {
      if (ps.base[q + 1] == ps.base[q]) continue;
      const GemmParams& pq = *ps.p[q];
      for (int i = 0; i < pq.num_passes; ++i) {
        ptx::prefetch_tensormap(&pq.tmA[i]);
        ptx::prefetch_tensormap(&pq.tmB[i]);
      }
      ptx::prefetch_tensormap(&pq.tmOutHi);
      ptx::prefetch_tensormap(&pq.tmOutLo);
      ptx::prefetch_tensormap(&pq.tmOutF32);
      ptx::prefetch_tensormap(&pq.tmOutF32b);
      ptx::prefetch_tensormap(&pq.tmSide);
    }
    for (int i = 0; i < kStages; ++i) {
      ptx::mbar_init(&sh.full_bar[i], 1);    // leader's barrier: its producer arrives once with the pair's byte count
      ptx::mbar_init(&sh.empty_bar[i], 1);   // per CTA: tcgen05.commit (multicast to both CTAs when CG == 2)
    }
    for (int i = 0; i < Cfg::kAccStages; ++i) {
      ptx::mbar_init(&sh.tmem_full_bar[i], 1);        // per CTA: tcgen05.commit
      ptx::mbar_init(&sh.tmem_empty_bar[i], 8 * CG);  // leader's barrier: one arrive per epilogue warp of the pair
    }
    for (int i = 0; i < kEpiTeams * kSlotsPerTeam; ++i) ptx::mbar_init(&sh.in_bars[i], 1);
    ptx::fence_barrier_init();
  }
  if (warp == 1) ptx::tmem_alloc<CG>(tmem_slot, Cfg::kTmemCols);
  if (threadIdx.x >= 64 && threadIdx.x < 64 + kEpiTeams * 128) sh.csum_strips[threadIdx.x - 64] = 0.f;
  ptx::tc_fence_before();
  if constexpr (CG == 2) ptx::cluster_sync(); else __syncthreads();
  ptx::tc_fence_after();
  sh.tmem_base = *tmem_slot;
  // PDL: everything above (barrier init, TMEM allocation, descriptor prefetch) overlaps the tail of the previous
  // kernel of the stream; from here on we read what it wrote.
  if (threadIdx.x == 0) trace_hdr(p.trace, 2, clock64());
  // (the dependents are released late, by the epilogue after its last tile: released here, their CTAs would sit on
  // the SMs this grid leaves to the step's background stream for the whole duration of this kernel)
  ptx::pdl_wait();
  if (threadIdx.x == 0) trace_hdr(p.trace, 3, clock64());

  UnitIter it(ps.sched, group_id, num_groups, ps.base[1]);

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer (one per CTA)
    if (lane == 0) {
      ProdState st{0u, 0u, ptx::mbar_try_wait(&sh.empty_bar[0], 1)};
      int titer = 0, u;
      while (it.next(u)) {
        RVAE_DISPATCH(produce_unit, st);
        ++titer;
      }
      trace_hdr(p.trace, 4, clock64());
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ UMMA issuer (leader CTA only)
    if (lane == 0 && sh.leader) {
      MmaState st{0u, 0u, 0u, 0u, false};
      int titer = 0, u;
      while (it.next(u)) {
        RVAE_DISPATCH(mma_unit, st);
        ++titer;
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue warps (2 teams x 4 warps)
    EpiState es;
    es.team = (warp - 2) >> 2;
    es.quarter = warp & 3;  // tcgen05.ld: a warp may only touch TMEM lanes 32*(warp%4) .. +31
    es.lane = lane;
    es.row = es.quarter * 32 + lane;  // row of the tile owned by this thread
    es.team_tid = (((warp - 2) & 3) << 5) | lane;  // 0..127 within the team
    es.lane_base = static_cast<uint32_t>(es.quarter * 32) << 16;
    es.tm = Team{sh.slot_base + es.team * (kSlotsPerTeam * kSlotBytes), sh.in_bars + es.team * kSlotsPerTeam,
                 sh.bias_strips + es.team * Cfg::kBiasFloats, sh.csum_strips + es.team * 128, 0u, 0u, 0u, es.team,
                 es.team_tid == 0};
    es.as = 0; es.aphase = 0; es.loss_local = 0.f;
    float loss[kMaxChain] = {0.f, 0.f, 0.f, 0.f};   // MSE / KL partial sums per problem (HEAD and OUT kinds)
    int titer = 0, u;
    while (it.next(u)) {
      RVAE_DISPATCH(epilogue_unit, es);
      const int q = (u >= ps.base[1]) + (u >= ps.base[2]) + (u >= ps.base[3]);
#pragma unroll
      for (int i = 0; i < kMaxChain; ++i)
        if (i == q) loss[i] += es.loss_local;
      es.loss_local = 0.f;
      ++titer;
    }
    ptx::pdl_launch_dependents();  // next kernel of the stream: its prologue overlaps our drain and teardown
    if (es.tm.issuer) ptx::tma_store_wait<0>();  // all bulk stores issued by this thread have completed
    auto flush_loss = [&](int i, int epi) {
      if (epi == EPI_HEAD || epi == EPI_OUT) {
        const float s = warp_sum(loss[i]);
        if (lane == 0 && ps.p[i]->epi.loss_acc) atomicAdd(ps.p[i]->epi.loss_acc, static_cast<double>(s));
      }
    };
    flush_loss(0, K0::EPI);
    if constexpr (is_kind<K1>::value) flush_loss(1, K1::EPI);
    if constexpr (is_kind<K2>::value) flush_loss(2, K2::EPI);
    if constexpr (is_kind<K3>::value) flush_loss(3, K3::EPI);
  }

  ptx::tc_fence_before();
  if constexpr (CG == 2) ptx::cluster_sync(); else __syncthreads();
  if (warp == 1) {
    __syncwarp();
    ptx::tc_fence_after();
    ptx::tmem_dealloc<CG>(sh.tmem_base, Cfg::kTmemCols);
  }
  if (threadIdx.x == 0) {
    trace_hdr(p.trace, 5, clock64());
    trace_hdr(p.trace, 6, global_timer());
  }
}

__device__ __forceinline__ ProblemSet single_problem(const GemmParams& p) {
  ProblemSet ps;
  const int total = p.m_blocks * p.n_blocks * p.k_splits;
  ps.p[0] = ps.p[1] = ps.p[2] = ps.p[3] = &p;
  ps.base[0] = 0;
  ps.base[1] = ps.base[2] = ps.base[3] = ps.base[4] = total;
  ps.sched = nullptr;
  return ps;
}

template <int BLOCK_N, int A_MAJOR, int B_MAJOR, int EPI>
__global__ void __launch_bounds__(kGemmThreads, 1) gemm_kernel(const __grid_constant__ GemmParams p) {
  gemm_body<BLOCK_N, 1, Kind<A_MAJOR, B_MAJOR, EPI>, NoKind, NoKind, NoKind>(single_problem(p));
}

template <int BLOCK_N, int A_MAJOR, int B_MAJOR, int EPI>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kGemmThreads, 1)
gemm_kernel_2cta(const __grid_constant__ GemmParams p) {
  gemm_body<BLOCK_N, 2, Kind<A_MAJOR, B_MAJOR, EPI>, NoKind, NoKind, NoKind>(single_problem(p));
}

// Up to four GEMMs in one persistent launch (CTA pairs, 256-wide tiles): independent ones (the dgrad and the weight
// gradient of a backward stage) or a chain of layers whose tiles depend on each other row block by row block (the
// forward pass). Units are assigned to the pairs by the host-built schedule cp.sched.
template <int BLOCK_N, class K0, class K1, class K2, class K3>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kGemmThreads, 1)
gemm_chain_kernel_2cta(const __grid_constant__ ChainParams cp) {
  ProblemSet ps;
#pragma unroll
  for (int i = 0; i < kMaxChain; ++i) ps.p[i] = &cp.p[i];
#pragma unroll
  for (int i = 0; i <= kMaxChain; ++i) ps.base[i] = cp.base[i];
  ps.sched = cp.sched;
  gemm_body<BLOCK_N, 2, K0, K1, K2, K3>(ps);
}

}  // namespace rvae
