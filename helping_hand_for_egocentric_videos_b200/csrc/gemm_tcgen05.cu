// Persistent, warp-specialised bf16 GEMM for sm_100a:  C[M,N] = epilogue(A[M,K] * W[N,K]^T)
//
//   * operands: TMA (cp.async.bulk.tensor, SWIZZLE_128B) into a ring of shared-memory stages
//   * math:     tcgen05.mma (cta_group::1, 128 x BLOCK_N x 16 per instruction) issued by ONE thread, fp32
//               accumulators in TMEM, double-buffered (2 x BLOCK_N columns) so the epilogue of tile i overlaps
//               the MMAs of tile i+1
//   * epilogue: 4 warps: tcgen05.ld -> registers -> bias / QuickGELU -> per-warp smem transpose -> coalesced
//               128-byte row stores (bf16) or fp32 rows with the fp32 residual added
//
// This one kernel carries every encoder contraction of the reference -- qkv / proj / fc1 / fc2 nn.Linear calls in
// model/LaviLa.py:249,281,186,189 -- plus the patch-embed conv as an im2col GEMM (:216-223), the decoder's memory
// projections (model/tfm_decoder.py:200,438-441) and class head (:208).
//
// Warp roles (256 threads): 0..3 = epilogue, 4 = TMEM allocator, 5 = residual producer (fused-LayerNorm producer GEMMs),
// 6 = TMA producer, 7 = MMA issuer (the single-thread roles on the highest warp ids: scheduler priority).
#include "hh_internal.h"
#include "hh_ptx.cuh"

#include <mutex>
#include <unordered_map>

namespace hh {

namespace {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;   // 64 bf16 = one 128-byte swizzle row
constexpr int UMMA_K = 16;
constexpr int NUM_THREADS = 256;
// Warp roles: the epilogue takes warps 0..3 and the single-thread roles the HIGHEST warp ids -- the SMSP arbiter prefers
// the highest eligible warp id (B300_MICROARCH.md), so the TMA producer and the MMA issuer are never kept waiting by the
// epilogue warp that shares their scheduler, however instruction-heavy the epilogue is.
constexpr int EPI_WARP0 = 0, W_ALLOC = 4, W_RES = 5, W_PROD = 6, W_MMA = 7;
constexpr int STAGE_LD = 33;  // per-warp transpose buffer: 32 rows x 33 words

// DEEP_EPI (the QuickGELU epilogue of the 2-SM path): a 4-slot store ring per epilogue warp and one operand stage fewer
// (same shared-memory total).  A/B on one box: fc1 43.3 -> 41.8 ms per step; the plain-bias GEMMs prefer the sixth
// operand stage (qkv 61.7 -> 62.6 ms with the deep ring), so they keep 2 slots.
// RES (the residual + LayerNorm-statistics epilogue): a per-warp ring of RES_SLOTS fp32 boxes (32 rows x 32 columns, 4 KB)
// that the residual tile streams through (TMA load -> add in place -> TMA store), paid for with two operand stages.
// It runs on 2-SM 256-wide and unclustered 128-wide tiles only (plan_tiles).
template <int BLOCK_N, bool TWOSM = false, bool DEEP_EPI = false, bool RES = false, bool LNF = false>
struct Cfg {
  static constexpr int A_BYTES = BLOCK_M * BLOCK_K * 2;
  static constexpr int B_BYTES = (TWOSM ? BLOCK_N / 2 : BLOCK_N) * BLOCK_K * 2;  // per CTA
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int RES_SLOTS = 4;
  static constexpr int RES_BYTES = RES ? 4 * RES_SLOTS * 4096 : 0;
  static constexpr int STAGES = RES ? 4 : ((BLOCK_N == 256 && !TWOSM) ? 4 : ((TWOSM && DEEP_EPI) ? 5 : 6));
  static constexpr int EPI_SLOTS = (TWOSM && DEEP_EPI) ? 4 : 2;  // per-warp ring of 32-row x 128-byte store slots
  static constexpr int EPI_BYTES = 4 * EPI_SLOTS * 4096;            // (>= the 4 x 32 x 33 words of the direct path)
  static constexpr int BIAS_BYTES = (LNF ? 2 : 1) * BLOCK_N * 4;    // bias tile (+ column-sum tile: LayerNorm-folded GEMMs)
  static constexpr int BAR_BYTES = RES ? 512 : 256;
  // The dynamic shared-memory window is declared __align__(1024) and there is no static shared memory in this kernel,
  // so the round-up below is normally a no-op; the slack is kept wherever the budget allows, and the one plan that
  // cannot afford it (folded LayerNorm on 256-wide tiles) is guarded by a device-side bounds check (traps).
  static constexpr int ALIGN_SLACK = (LNF && BLOCK_N == 256) ? 0 : 1024;
  static constexpr int SMEM_BYTES = ALIGN_SLACK + STAGES * STAGE_BYTES + EPI_BYTES + RES_BYTES + BIAS_BYTES + BAR_BYTES;
  static constexpr int TMEM_COLS = 2 * BLOCK_N;  // 256 or 512: power of two
  static_assert(SMEM_BYTES <= 232448, "shared-memory plan exceeds 227 KB");
  static_assert((2 * STAGES + 4 + (RES ? 8 * RES_SLOTS : 0)) * 8 + 4 <= BAR_BYTES, "barrier region too small");
};

struct GemmArgs {
  void* out;
  const float* bias;
  const float* residual;
  int M, N, K;
  int ldc, ldr;
  int tiles_m, tiles_n;
  // LayerNorm folded into the contraction (EPI_LN_*): per-row (sum, sum of squares) partials of the un-normalised A
  // rows [stats_parts][M][2], the column sums of the gamma-scaled weight, 1 / normalised width, eps
  const float* colsum;
  const float* stats_in;
  int stats_parts;
  float inv_d, eps;
  // EPI_RES_STATS_BF16: per-row partials of the rows this GEMM writes, [tiles_n][M][2]; write the fp32 sum back in place
  float* stats_out;
  int writeback;
  // segmented A rows (gemm_bf16_rowseg): logical row m is A row m + (m / a_seg_rows) * a_seg_skip; 0 = contiguous
  int a_seg_rows, a_seg_skip;
};

__device__ __forceinline__ float quick_gelu(float x) {
  // x * sigmoid(1.702 x) (model/openai_model.py:177-179) = 0.5 x (1 + tanh(0.851 x)): one MUFU op per element
  // (tanh.approx.f32, rel. error 2^-11, below the bf16 rounding of the output) instead of ex2 + rcp.
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(0.851f * x));
  const float hx = 0.5f * x;
  return fmaf(hx, t, hx);
}

// two elements at once: the three fp32 multiplies / FMAs are packed f32x2 instructions, tanh stays one MUFU each
__device__ __forceinline__ float2 quick_gelu2(float2 x) {
  const float2 u = __fmul2_rn(x, make_float2(0.851f, 0.851f));
  float2 t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t.x) : "f"(u.x));
  asm("tanh.approx.f32 %0, %1;" : "=f"(t.y) : "f"(u.y));
  const float2 hx = __fmul2_rn(x, make_float2(0.5f, 0.5f));
  return __ffma2_rn(hx, t, hx);
}


// HH_GEMM_TRACE (variant builds only, tools/build_variant.sh): cycles each role of every CTA spends in its waits, read
// back with hh_debug_gemm_trace.  Slots per CTA: [0] kernel cycles, producer [1] empty; MMA [2] accumulator-empty [3] full;
// epilogue warp 0 lane 0 [4] accumulator-full [5] residual-full [6] bulk-store read [7] bias / statistics prologue
// [8] tiles; epilogue warp 0 lane 1 [9] accumulator-full [10] residual-full.
#ifdef HH_GEMM_TRACE
__device__ unsigned long long g_gemm_trace[148 * 16];
#define TR_T0() const long long tr_t0_ = clock64()
#define TR_ADD(slot) tr_[slot] += static_cast<unsigned long long>(clock64() - tr_t0_)
#else
#define TR_T0() do { } while (0)
#define TR_ADD(slot) do { } while (0)
#endif

__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// TMA_STORE: the epilogue writes 32-row x 128-byte boxes through shared memory with cp.async.bulk.tensor stores
// (needs a 16-byte aligned output with a 16-byte multiple row pitch); otherwise rows are stored directly.
// CLUSTER: CTAs are launched as pairs (cluster 2x1x1) that work on two vertically adjacent output tiles with the SAME
// weight tile: each CTA fetches half of the W tile and multicasts it into both CTAs' shared memory, which cuts the
// L2 -> SM operand traffic per tile from A + W to A + W/2 (-33 %).  A stage is released to the producers only after
// BOTH CTAs' MMAs have consumed it (tcgen05.commit multicast onto both empty barriers).
// TWOSM (implies CLUSTER): the pair runs ONE tcgen05.mma.cta_group::2 of 256 x BLOCK_N x 16 per step instead of two
// independent 128 x BLOCK_N MMAs.  Each CTA stages its own 128 rows of A and only ITS half of the W tile (no multicast);
// the leader CTA's single MMA thread drives both SMs' tensor cores, which read the W halves from both shared memories.
// Shared-memory operand reads per CTA drop from 128 + BLOCK_N to 128 + BLOCK_N/2 rows per K step (-33 %), a stage is
// 32 KB instead of 48 KB (6 stages instead of 4).  Barrier protocol: both producers' TMA loads complete on the LEADER's
// full barrier (which expects both CTAs' bytes); the leader's commits are multicast to both CTAs' empty / accumulator-
// full barriers; both CTAs' epilogue warps arrive on the LEADER's accumulator-empty barrier.
template <int BLOCK_N, int EPI, bool TMA_STORE, bool CLUSTER, bool TWOSM = false>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
            const __grid_constant__ CUtensorMap tma_c, const __grid_constant__ CUtensorMap tma_r, const GemmArgs p) {
  static_assert(!TWOSM || (CLUSTER && TMA_STORE), "the 2-SM MMA path runs as a CTA pair");
  constexpr bool QGELU = (EPI == EPI_BIAS_QGELU_BF16 || EPI == EPI_LN_BIAS_QGELU_BF16);
  constexpr bool LNF = (EPI == EPI_LN_BIAS_BF16 || EPI == EPI_LN_BIAS_QGELU_BF16);   // LayerNorm folded (consumer side)
  constexpr bool RES = (EPI == EPI_RES_STATS_BF16);                                  // residual + statistics (producer)
  static_assert(!(LNF || RES) || TMA_STORE, "the fused-LayerNorm epilogues use bulk-tensor stores");
  using C = Cfg<BLOCK_N, TWOSM, QGELU, RES, LNF>;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  if constexpr (C::ALIGN_SLACK == 0) {
    if (smem != smem_raw) __trap();  // the window was not 1024-byte aligned: this plan has no room for the round-up
  }

  uint8_t* stage_base = smem;
  float* epi_stage = reinterpret_cast<float*>(smem + C::STAGES * C::STAGE_BYTES);
  uint8_t* res_stage = smem + C::STAGES * C::STAGE_BYTES + C::EPI_BYTES;
  float* bias_s = reinterpret_cast<float*>(res_stage + C::RES_BYTES);
  float* cs_s = bias_s + BLOCK_N;              // column sums (LNF only)
  uint64_t* bars = reinterpret_cast<uint64_t*>(res_stage + C::RES_BYTES + C::BIAS_BYTES);
  uint64_t* full_bar = bars;                   // [STAGES]
  uint64_t* empty_bar = bars + C::STAGES;      // [STAGES]
  uint64_t* tfull_bar = bars + 2 * C::STAGES;  // [2]
  uint64_t* tempty_bar = tfull_bar + 2;        // [2]
  uint64_t* res_full = tempty_bar + 2;         // [4 warps][RES_SLOTS] (RES only)
  uint64_t* res_empty = res_full + (RES ? 4 * C::RES_SLOTS : 0);  // [4 warps][RES_SLOTS] (RES only)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(res_empty + (RES ? 4 * C::RES_SLOTS : 0));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_kb = (p.K + BLOCK_K - 1) / BLOCK_K;
  // tile walk: a CTA (or CTA pair) takes every tile_step-th (pair of) tile(s); n_blk varies fastest
  const int cta_rank = CLUSTER ? static_cast<int>(cluster_ctarank()) : 0;
  const int tile_first = CLUSTER ? static_cast<int>(blockIdx.x >> 1) : static_cast<int>(blockIdx.x);
  const int tile_step = CLUSTER ? static_cast<int>(gridDim.x >> 1) : static_cast<int>(gridDim.x);
  const int total_tiles = CLUSTER ? ((p.tiles_m + 1) >> 1) * p.tiles_n : p.tiles_m * p.tiles_n;

  if (warp == W_PROD && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_b);
    if constexpr (TMA_STORE) tma_prefetch_desc(&tma_c);
    if constexpr (RES) tma_prefetch_desc(&tma_r);
  }
  if (warp == W_MMA && lane == 0) {
    for (int s = 0; s < C::STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], (CLUSTER && !TWOSM) ? 2 : 1);
    }
    if constexpr (RES) {
      for (int s = 0; s < 4 * C::RES_SLOTS; ++s) {
        mbar_init(&res_full[s], 1);
        mbar_init(&res_empty[s], 1);
      }
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull_bar[a], 1);
      mbar_init(&tempty_bar[a], TWOSM ? 8 : 4);   // 2-SM: the leader's barrier collects both CTAs' epilogue warps
    }
    fence_mbar_init();
  }
  if (warp == W_ALLOC) {
    if constexpr (TWOSM) {
      tmem_alloc_2sm(tmem_slot, C::TMEM_COLS);
      tmem_relinquish_2sm();
    } else {
      tmem_alloc(tmem_slot, C::TMEM_COLS);
      tmem_relinquish();
    }
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (CLUSTER) cluster_sync_all();  // the peer's barriers exist before anything is multicast to them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
#ifdef HH_GEMM_TRACE
  unsigned long long tr_[16] = {};
  const long long tr_begin_ = clock64();
#endif

  if (warp == W_PROD) {
    // ------------------------------------------------------------ TMA producer
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = tile_first; tile < total_tiles; tile += tile_step) {
        const int mp = tile / p.tiles_n;
        const int n_blk = tile - mp * p.tiles_n;
        const int m_blk = CLUSTER ? 2 * mp + cta_rank : mp;
        // A row of this tile: a 128-row box never straddles two segments (a_seg_rows % 128 == 0); a pair's padding tile
        // past M maps past the end of A as well and is zero-filled, as without segments
        int a_row = m_blk * BLOCK_M;
        if (p.a_seg_rows) a_row += (a_row / p.a_seg_rows) * p.a_seg_skip;
        for (int kb = 0; kb < num_kb; ++kb) {
          { TR_T0(); mbar_wait(&empty_bar[stage], phase ^ 1u); TR_ADD(1); }
          uint8_t* sa = stage_base + stage * C::STAGE_BYTES;
          uint8_t* sb = sa + C::A_BYTES;
          if constexpr (TWOSM) {  // my A rows + my half of the W tile, into MY smem, signalled on the leader's barrier
            if (cta_rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * C::STAGE_BYTES);
            tma_load_2d_2sm(&tma_a, &full_bar[stage], sa, kb * BLOCK_K, a_row);
            tma_load_2d_2sm(&tma_b, &full_bar[stage], sb, kb * BLOCK_K, n_blk * BLOCK_N + cta_rank * (BLOCK_N / 2));
            if (++stage == C::STAGES) {
              stage = 0;
              phase ^= 1u;
            }
            continue;
          }
          mbar_arrive_expect_tx(&full_bar[stage], C::STAGE_BYTES);
          tma_load_2d(&tma_a, &full_bar[stage], sa, kb * BLOCK_K, a_row);
          if constexpr (CLUSTER) {  // my half of the W tile, into both CTAs (box = BLOCK_N/2 rows)
            tma_load_2d_mcast(&tma_b, &full_bar[stage], sb + cta_rank * (C::B_BYTES / 2), kb * BLOCK_K,
                              n_blk * BLOCK_N + cta_rank * (BLOCK_N / 2), static_cast<uint16_t>(3));
          } else {
            tma_load_2d(&tma_b, &full_bar[stage], sb, kb * BLOCK_K, n_blk * BLOCK_N);
          }
          if (++stage == C::STAGES) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
  } else if (warp == W_MMA) {
    // ------------------------------------------------------------ MMA issuer (single thread)
    if (lane == 0 && (!TWOSM || cta_rank == 0)) {
      constexpr uint32_t idesc = umma_idesc_bf16(TWOSM ? 2 * BLOCK_M : BLOCK_M, BLOCK_N);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int tile = tile_first; tile < total_tiles; tile += tile_step) {
        { TR_T0(); mbar_wait(&tempty_bar[acc], acc_phase ^ 1u); TR_ADD(2); }  // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * BLOCK_N);
        for (int kb = 0; kb < num_kb; ++kb) {
          { TR_T0(); mbar_wait(&full_bar[stage], phase); TR_ADD(3); }
          tc_fence_after();
          const uint32_t sa = smem_u32(stage_base + stage * C::STAGE_BYTES);
          const uint32_t sb = sa + C::A_BYTES;
          const uint64_t da = umma_desc_sw128(sa);
          const uint64_t db = umma_desc_sw128(sb);
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
            // advance K inside the 128-byte swizzle row: +32 bytes => +2 in (addr >> 4) units
            if constexpr (TWOSM)
              umma_bf16_2sm(d_tmem, da + static_cast<uint64_t>(2 * k), db + static_cast<uint64_t>(2 * k), idesc,
                            (kb > 0 || k > 0) ? 1u : 0u);
            else
              umma_bf16(d_tmem, da + static_cast<uint64_t>(2 * k), db + static_cast<uint64_t>(2 * k), idesc,
                        (kb > 0 || k > 0) ? 1u : 0u);
          }
          // smem slot reusable once these MMAs retire (in a pair: tell both CTAs' producers)
          if constexpr (TWOSM) umma_commit_2sm(&empty_bar[stage], static_cast<uint16_t>(3));
          else if constexpr (CLUSTER) umma_commit_mcast(&empty_bar[stage], static_cast<uint16_t>(3));
          else umma_commit(&empty_bar[stage]);
          if (++stage == C::STAGES) {
            stage = 0;
            phase ^= 1u;
          }
        }
        if constexpr (TWOSM) umma_commit_2sm(&tfull_bar[acc], static_cast<uint16_t>(3));  // both CTAs' epilogues
        else umma_commit(&tfull_bar[acc]);  // accumulator complete -> epilogue
        if (++acc == 2) {
          acc = 0;
          acc_phase ^= 1u;
        }
      }
    }
  } else if (warp == W_RES) {
    // ------------------------------------------------------------ residual producer (RES only): lane q feeds epilogue
    // warp q's ring of fp32 boxes (32 rows x 32 columns), one box per unit, in the order the epilogue consumes them
    if constexpr (RES) {
      if (lane < 4) {
        const int q = lane;
        uint64_t* const my_full = res_full + q * C::RES_SLOTS;
        uint64_t* const my_empty = res_empty + q * C::RES_SLOTS;
        uint8_t* const my_ring = res_stage + q * C::RES_SLOTS * 4096;
        int slot = 0;
        uint32_t phase = 0;
        for (int tile = tile_first; tile < total_tiles; tile += tile_step) {
          const int mp = tile / p.tiles_n;
          const int n_blk = tile - mp * p.tiles_n;
          const int m_blk = CLUSTER ? 2 * mp + cta_rank : mp;
#pragma unroll 1
          for (int u = 0; u < BLOCK_N / 32; ++u) {
            mbar_wait(&my_empty[slot], phase ^ 1u);
            mbar_arrive_expect_tx(&my_full[slot], 4096);
            tma_load_2d(&tma_r, &my_full[slot], my_ring + slot * 4096, n_blk * BLOCK_N + u * 32, m_blk * BLOCK_M + q * 32);
            if (++slot == C::RES_SLOTS) {
              slot = 0;
              phase ^= 1u;
            }
          }
        }
      }
    }
  } else if (warp >= EPI_WARP0 && warp < EPI_WARP0 + 4) {
    // ------------------------------------------------------------ epilogue (4 warps = 128 TMEM lanes)
    const int q = warp & 3;  // TMEM lane quarter this warp may touch
    float* st = epi_stage + q * 32 * STAGE_LD;
    const int et = threadIdx.x - EPI_WARP0 * 32;  // 0..127
    int acc = 0;
    uint32_t acc_phase = 0;
    int epi_slot = 0;
    // ---- RES: the fp32 residual tile streams through this warp's ring of 32 x 32 boxes, filled by warp 3.  Units (32
    // output columns of this warp's 32 rows) are consumed in tile / column order; one bulk group is committed per unit,
    // so "every group but the newest has finished reading shared memory" frees the slot of the previous unit.
    constexpr int UNITS = BLOCK_N / 32;
    const uint32_t res_ring = smem_u32(res_stage) + static_cast<uint32_t>(q * C::RES_SLOTS * 4096);
    uint64_t* const my_res_full = res_full + q * C::RES_SLOTS;
    uint64_t* const my_res_empty = res_empty + q * C::RES_SLOTS;
    int res_slot = 0;
    uint32_t res_phase = 0;
    int res_prev = -1;                          // slot whose write-back store is still reading shared memory
    // ---- per-tile constants are fetched one tile ahead (registers), so their global-load latency hides behind the
    // previous tile's work: bias / column sums for columns et, et + 128, and this thread's row statistics
    constexpr int BPT = BLOCK_N / 128;
    float nb_bias[BPT], nb_cs[BPT];
    float n_s1 = 0.f, n_s2 = 0.f;
    auto prefetch_tile_consts = [&](int tile) {
      if (tile >= total_tiles) return;
      const int mp = tile / p.tiles_n;
      const int n_blk = tile - mp * p.tiles_n;
      const int m_blk = CLUSTER ? 2 * mp + cta_rank : mp;
#pragma unroll
      for (int i = 0; i < BPT; ++i) {
        const int col = n_blk * BLOCK_N + et + i * 128;
        nb_bias[i] = (p.bias != nullptr && col < p.N) ? __ldg(p.bias + col) : 0.0f;
        if constexpr (LNF) nb_cs[i] = (col < p.N) ? __ldg(p.colsum + col) : 0.0f;
      }
      if constexpr (LNF) {
        const int row = m_blk * BLOCK_M + q * 32 + lane;
        n_s1 = 0.f;
        n_s2 = 0.f;
        if (row < p.M) {
          float2 t[4] = {};
#pragma unroll
          for (int i = 0; i < 4; ++i)
            if (i < p.stats_parts) t[i] = __ldg(reinterpret_cast<const float2*>(p.stats_in) + static_cast<size_t>(i) * p.M + row);
          for (int i = 4; i < p.stats_parts; ++i) {
            const float2 e = __ldg(reinterpret_cast<const float2*>(p.stats_in) + static_cast<size_t>(i) * p.M + row);
            t[0].x += e.x;
            t[0].y += e.y;
          }
          n_s1 = (t[0].x + t[1].x) + (t[2].x + t[3].x);
          n_s2 = (t[0].y + t[1].y) + (t[2].y + t[3].y);
        }
      }
    };
    prefetch_tile_consts(tile_first);
    for (int tile = tile_first; tile < total_tiles; tile += tile_step) {
      const int mp = tile / p.tiles_n;
      const int n_blk = tile - mp * p.tiles_n;
      const int m_blk = CLUSTER ? 2 * mp + cta_rank : mp;
      const int row0 = m_blk * BLOCK_M + q * 32;
      const int col0 = n_blk * BLOCK_N;
#ifdef HH_GEMM_TRACE
      const long long tr_tile0_ = clock64();
#endif

      // bias tile -> smem from the registers fetched one tile ago (the previous tile's readers are done: they passed
      // the trailing named barrier)
#pragma unroll
      for (int i = 0; i < BPT; ++i) {
        bias_s[et + i * 128] = nb_bias[i];
        if constexpr (LNF) cs_s[et + i * 128] = nb_cs[i];
      }
      // folded LayerNorm: this thread's row statistics, from the producer's per-column-tile partials
      float2 ln_rs = make_float2(1.f, 1.f), ln_nm = make_float2(0.f, 0.f);
      if constexpr (LNF) {
        const float mu = n_s1 * p.inv_d;
        const float rs = rsqrtf(fmaxf(fmaf(n_s2, p.inv_d, -mu * mu), 0.f) + p.eps);
        ln_rs = make_float2(rs, rs);
        ln_nm = make_float2(-mu * rs, -mu * rs);
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");
      prefetch_tile_consts(tile + tile_step);   // in flight while this tile is processed
#ifdef HH_GEMM_TRACE
      tr_[7] += static_cast<unsigned long long>(clock64() - tr_tile0_);
      tr_[8] += 1;
#endif

      { TR_T0(); mbar_wait(&tfull_bar[acc], acc_phase); TR_ADD(4); }
      tc_fence_after();
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(acc * BLOCK_N);

      if constexpr (RES) {
        // z = acc + bias + residual: bf16 copy (next GEMM's A operand), per-row sums for the folded LayerNorm, and
        // optionally the fp32 sum written back over the residual (the stream x itself)
        const uint32_t zring = smem_u32(epi_stage) + static_cast<uint32_t>(q * C::EPI_SLOTS * 4096);
        const uint32_t sw = static_cast<uint32_t>(lane & 7);
        float s1 = 0.f, s2 = 0.f;
#pragma unroll 1
        for (int u = 0; u < UNITS; ++u) {
          const uint32_t slot = static_cast<uint32_t>(res_slot);
          uint32_t r[32];
          tmem_ld_32x32b_x32(t_row + static_cast<uint32_t>(u * 32), r);   // in flight while the residual box is awaited
          { TR_T0(); mbar_wait(&my_res_full[slot], res_phase); TR_ADD(5); }
          const uint32_t rrow = res_ring + slot * 4096u + static_cast<uint32_t>(lane * 128);
          const uint32_t zrow = zring + static_cast<uint32_t>(epi_slot * 4096 + lane * 128);
          tmem_ld_wait();
          uint32_t w[16];
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            float4 x4;
            const uint32_t ra = rrow + ((static_cast<uint32_t>(k) ^ sw) << 4);
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                         : "=f"(x4.x), "=f"(x4.y), "=f"(x4.z), "=f"(x4.w) : "r"(ra) : "memory");
            const float4 b4 = *reinterpret_cast<const float4*>(&bias_s[u * 32 + 4 * k]);
            float4 v;
            v.x = (__uint_as_float(r[4 * k + 0]) + b4.x) + x4.x;
            v.y = (__uint_as_float(r[4 * k + 1]) + b4.y) + x4.y;
            v.z = (__uint_as_float(r[4 * k + 2]) + b4.z) + x4.z;
            v.w = (__uint_as_float(r[4 * k + 3]) + b4.w) + x4.w;
            s1 += (v.x + v.y) + (v.z + v.w);
            s2 = fmaf(v.x, v.x, fmaf(v.y, v.y, fmaf(v.z, v.z, fmaf(v.w, v.w, s2))));
            if (p.writeback)
              st_shared_v4(ra, __float_as_uint(v.x), __float_as_uint(v.y), __float_as_uint(v.z), __float_as_uint(v.w));
            w[2 * k] = pack_bf16x2(v.x, v.y);
            w[2 * k + 1] = pack_bf16x2(v.z, v.w);
          }
#pragma unroll
          for (int k = 0; k < 4; ++k)  // 16-byte chunk ((u & 1) * 4 + k) of the 64-column bf16 row, 128B-swizzled
            st_shared_v4(zrow + ((static_cast<uint32_t>((u & 1) * 4 + k) ^ sw) << 4), w[4 * k], w[4 * k + 1], w[4 * k + 2],
                         w[4 * k + 3]);
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            if (p.writeback) tma_store_2d(&tma_r, res_ring + slot * 4096u, col0 + u * 32, row0);
            if (u & 1) tma_store_2d(&tma_c, zring + static_cast<uint32_t>(epi_slot * 4096), col0 + (u >> 1) * 64, row0);
            tma_store_commit();
            // every group but the newest has been read out of shared memory: with write-back that frees the previous
            // unit's box (and bounds the z ring); without it this unit's box is free as soon as the warp has read it
            { TR_T0(); tma_store_wait_read<1>(); TR_ADD(6); }
            if (p.writeback) {
              if (res_prev >= 0) mbar_arrive(&my_res_empty[res_prev]);
            } else {
              mbar_arrive(&my_res_empty[slot]);
            }
            if constexpr (C::EPI_SLOTS == 1) {   // the only z slot is rewritten by the next unit: its store must have read it
              if (u & 1) tma_store_wait_read<0>();
            }
          }
          if constexpr (C::EPI_SLOTS == 1) __syncwarp();
          res_prev = res_slot;
          if (u & 1) epi_slot = (epi_slot + 1 == C::EPI_SLOTS) ? 0 : epi_slot + 1;
          if (++res_slot == C::RES_SLOTS) {
            res_slot = 0;
            res_phase ^= 1u;
          }
        }
        const int row = row0 + lane;
        if (row < p.M)
          *reinterpret_cast<float2*>(p.stats_out + (static_cast<size_t>(n_blk) * p.M + row) * 2) = make_float2(s1, s2);
      } else
      if constexpr (TMA_STORE) {
        constexpr bool OUT16 = (EPI == EPI_BIAS_BF16 || EPI == EPI_BIAS_QGELU_BF16 || LNF);
        constexpr int CH_COLS = OUT16 ? 64 : 32;  // one chunk = 128 bytes per row
        const uint32_t ring = smem_u32(epi_stage) + static_cast<uint32_t>(q * C::EPI_SLOTS * 4096);
        const uint32_t sw = static_cast<uint32_t>(lane & 7);
#pragma unroll 1
        for (int c = 0; c < BLOCK_N / CH_COLS; ++c) {
          // the bulk store that last used this slot must have finished reading it
          if (lane == 0) { TR_T0(); tma_store_wait_read<C::EPI_SLOTS - 1>(); TR_ADD(6); }
          __syncwarp();
          const uint32_t row_addr = ring + static_cast<uint32_t>(epi_slot * 4096 + lane * 128);
          if constexpr (OUT16) {
            // both 32-column halves of the chunk are requested before the single wait: two TMEM loads in flight
            uint32_t rr[2][32];
            tmem_ld_32x32b_x32(t_row + static_cast<uint32_t>(c * 64), rr[0]);
            tmem_ld_32x32b_x32(t_row + static_cast<uint32_t>(c * 64 + 32), rr[1]);
            tmem_ld_wait();
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const uint32_t(&r)[32] = rr[h];
              uint32_t w[16];
#pragma unroll
              for (int j = 0; j < 32; j += 2) {
                // packed fp32x2 arithmetic (same IEEE results as the scalar ops, half the issue slots / energy)
                float2 v;
                if constexpr (LNF) {  // rstd * acc + (bias' - rstd * mean * colsum)
                  const float2 t = __ffma2_rn(*reinterpret_cast<const float2*>(&cs_s[c * 64 + h * 32 + j]), ln_nm,
                                              *reinterpret_cast<const float2*>(&bias_s[c * 64 + h * 32 + j]));
                  v = __ffma2_rn(make_float2(__uint_as_float(r[j]), __uint_as_float(r[j + 1])), ln_rs, t);
                } else {
                  v = __fadd2_rn(make_float2(__uint_as_float(r[j]), __uint_as_float(r[j + 1])),
                                 *reinterpret_cast<const float2*>(&bias_s[c * 64 + h * 32 + j]));
                }
                if constexpr (QGELU) v = quick_gelu2(v);
                w[j >> 1] = pack_bf16x2(v.x, v.y);
              }
#pragma unroll
              for (int k = 0; k < 4; ++k)  // 16-byte chunk (h*4 + k) of this row, 128B-swizzled
                st_shared_v4(row_addr + ((static_cast<uint32_t>(h * 4 + k) ^ sw) << 4), w[4 * k], w[4 * k + 1],
                             w[4 * k + 2], w[4 * k + 3]);
            }
          } else {
            uint32_t r[32];
            tmem_ld_32x32b_x32(t_row + static_cast<uint32_t>(c * 32), r);
            tmem_ld_wait();
#pragma unroll
            for (int k = 0; k < 8; ++k) {
              uint32_t w[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) w[e] = __float_as_uint(__uint_as_float(r[4 * k + e]) + bias_s[c * 32 + 4 * k + e]);
              st_shared_v4(row_addr + ((static_cast<uint32_t>(k) ^ sw) << 4), w[0], w[1], w[2], w[3]);
            }
          }
          fence_proxy_async_smem();  // generic-proxy smem writes -> visible to the bulk-copy engine
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&tma_c, ring + static_cast<uint32_t>(epi_slot * 4096), col0 + c * CH_COLS, row0);
            tma_store_commit();
          }
          epi_slot = (epi_slot + 1 == C::EPI_SLOTS) ? 0 : epi_slot + 1;
        }
      } else if constexpr (EPI == EPI_BIAS_BF16 || EPI == EPI_BIAS_QGELU_BF16) {
        __nv_bfloat16* out = reinterpret_cast<__nv_bfloat16*>(p.out);
#pragma unroll 1
        for (int g = 0; g < BLOCK_N / 64; ++g) {
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            uint32_t r[32];
            tmem_ld_32x32b_x32(t_row + static_cast<uint32_t>(g * 64 + h * 32), r);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; j += 2) {
              float v0 = __uint_as_float(r[j]) + bias_s[g * 64 + h * 32 + j];
              float v1 = __uint_as_float(r[j + 1]) + bias_s[g * 64 + h * 32 + j + 1];
              if constexpr (EPI == EPI_BIAS_QGELU_BF16) {
                v0 = quick_gelu(v0);
                v1 = quick_gelu(v1);
              }
              // thread = row `lane`; word index = column pair
              reinterpret_cast<uint32_t*>(st)[lane * STAGE_LD + h * 16 + (j >> 1)] = pack_bf16x2(v0, v1);
            }
          }
          __syncwarp();
          // row i of this warp's 32 rows: 32 lanes x 4 bytes = 128 contiguous bytes (64 bf16 columns)
          const int colw = col0 + g * 64 + lane * 2;
#pragma unroll 8
          for (int i = 0; i < 32; ++i) {
            const int row = row0 + i;
            const uint32_t w = reinterpret_cast<uint32_t*>(st)[i * STAGE_LD + lane];
            if (row < p.M) {
              __nv_bfloat16* dst = out + static_cast<size_t>(row) * p.ldc + colw;
              if (colw + 1 < p.N) {
                *reinterpret_cast<uint32_t*>(dst) = w;
              } else if (colw < p.N) {
                dst[0] = __ushort_as_bfloat16(static_cast<unsigned short>(w & 0xFFFFu));
              }
            }
          }
          __syncwarp();
        }
      } else {
        float* out = reinterpret_cast<float*>(p.out);
#pragma unroll 1
        for (int g = 0; g < BLOCK_N / 32; ++g) {
          uint32_t r[32];
          tmem_ld_32x32b_x32(t_row + static_cast<uint32_t>(g * 32), r);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) st[lane * STAGE_LD + j] = __uint_as_float(r[j]) + bias_s[g * 32 + j];
          __syncwarp();
          const int col = col0 + g * 32 + lane;
#pragma unroll 8
          for (int i = 0; i < 32; ++i) {
            const int row = row0 + i;
            float v = st[i * STAGE_LD + lane];
            if (row < p.M && col < p.N) {
              if constexpr (EPI == EPI_BIAS_RES_F32) v += p.residual[static_cast<size_t>(row) * p.ldr + col];
              out[static_cast<size_t>(row) * p.ldc + col] = v;
            }
          }
          __syncwarp();
        }
      }
      // all TMEM reads of this accumulator are complete (tcgen05.wait::ld above) -> hand it back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if constexpr (TWOSM) mbar_arrive_cluster(&tempty_bar[acc], 0u);
        else mbar_arrive(&tempty_bar[acc]);
      }
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1u;
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");  // bias_s free for the next tile
    }
    if constexpr (TMA_STORE) {
      if (lane == 0) tma_store_wait_read<0>();  // smem must stay valid until the last bulk store has read it
    }
    (void)epi_slot;
  }

#ifdef HH_GEMM_TRACE
  if (blockIdx.x < 148) {
    unsigned long long* g = g_gemm_trace + blockIdx.x * 16;
    if (warp == W_PROD && lane == 0) { g[0] = static_cast<unsigned long long>(clock64() - tr_begin_); g[1] = tr_[1]; }
    if (warp == W_MMA && lane == 0) { g[2] = tr_[2]; g[3] = tr_[3]; }
    if (warp == EPI_WARP0 && lane == 0) { g[4] = tr_[4]; g[5] = tr_[5]; g[6] = tr_[6]; g[7] = tr_[7]; g[8] = tr_[8]; }
    if (warp == EPI_WARP0 && lane == 1) { g[9] = tr_[4]; g[10] = tr_[5]; }
  }
#endif
  tc_fence_before();
  __syncthreads();
  if constexpr (CLUSTER) cluster_sync_all();  // no CTA leaves while its peer may still multicast into it
  if (warp == W_ALLOC) {
    tc_fence_after();
    if constexpr (TWOSM) tmem_dealloc_2sm(tmem_base, C::TMEM_COLS);
    else tmem_dealloc(tmem_base, C::TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres);
    if (e == cudaSuccess && qres == cudaDriverEntryPointSuccess) fn = reinterpret_cast<EncodeTiledFn>(ptr);
  });
  return fn;
}

// 2-D row-major [rows, cols] (cols contiguous, row stride ld elements) of bf16 (elem_bytes 2) or fp32 (4);
// box = [128 bytes of columns, box_rows rows], SWIZZLE_128B.
int make_tmap(CUtensorMap* map, const void* base, int rows, int cols, int ld, int box_rows, int elem_bytes = 2) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return fail(-3, "cuTensorMapEncodeTiled entry point not available (no CUDA driver?)");
  cuuint64_t gdim[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t gstride[1] = {static_cast<cuuint64_t>(ld) * elem_bytes};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(128 / elem_bytes), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                  const_cast<void*>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(-3, "cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r));
  return 0;
}

template <int BLOCK_N, int EPI, bool TMA_STORE, bool CLUSTER, bool TWOSM = false>
int launch(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const CUtensorMap& tr, const GemmArgs& args,
           cudaStream_t stream) {
  using C = Cfg<BLOCK_N, TWOSM, EPI == EPI_BIAS_QGELU_BF16 || EPI == EPI_LN_BIAS_QGELU_BF16, EPI == EPI_RES_STATS_BF16,
                EPI == EPI_LN_BIAS_BF16 || EPI == EPI_LN_BIAS_QGELU_BF16>;
  static bool configured = false;
  auto kern = gemm_kernel<BLOCK_N, EPI, TMA_STORE, CLUSTER, TWOSM>;
  if (!configured) {
    HH_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
    configured = true;
  }
  if constexpr (CLUSTER) {
    const int pairs = ((args.tiles_m + 1) / 2) * args.tiles_n;
    int grid = num_sms() & ~1;
    if (grid > 2 * pairs) grid = 2 * pairs;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(NUM_THREADS);
    cfg.dynamicSmemBytes = C::SMEM_BYTES;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    HH_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, ta, tb, tc, tr, args));
    return 0;
  }
  const int total = args.tiles_m * args.tiles_n;
  int grid = num_sms();
  if (grid > total) grid = total;
  kern<<<grid, NUM_THREADS, C::SMEM_BYTES, stream>>>(ta, tb, tc, tr, args);
  HH_CHECK_LAUNCH("gemm_kernel");
  return 0;
}

template <int BLOCK_N>
int dispatch_epi(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const CUtensorMap& tr, bool tma_store,
                 bool cluster, const GemmArgs& args, int epi, cudaStream_t stream) {
  // CTA pairs: one 2-SM MMA on 256-wide tiles, two 1-SM MMAs with the W tile multicast on 128-wide tiles
  constexpr bool TWOSM = BLOCK_N == 256;
  if (cluster) {
    switch (epi) {
      case EPI_BIAS_BF16: return launch<BLOCK_N, EPI_BIAS_BF16, true, true, TWOSM>(ta, tb, tc, tr, args, stream);
      case EPI_BIAS_QGELU_BF16: return launch<BLOCK_N, EPI_BIAS_QGELU_BF16, true, true, TWOSM>(ta, tb, tc, tr, args, stream);
      case EPI_BIAS_F32: return launch<BLOCK_N, EPI_BIAS_F32, true, true, TWOSM>(ta, tb, tc, tr, args, stream);
      case EPI_LN_BIAS_BF16: return launch<BLOCK_N, EPI_LN_BIAS_BF16, true, true, TWOSM>(ta, tb, tc, tr, args, stream);
      case EPI_LN_BIAS_QGELU_BF16:
        return launch<BLOCK_N, EPI_LN_BIAS_QGELU_BF16, true, true, TWOSM>(ta, tb, tc, tr, args, stream);
      case EPI_RES_STATS_BF16:
        if constexpr (TWOSM) return launch<256, EPI_RES_STATS_BF16, true, true, true>(ta, tb, tc, tr, args, stream);
        break;
    }
  }
  if (epi == EPI_RES_STATS_BF16) {  // outside the 2-SM path the residual epilogue runs unclustered on 128-wide tiles
    if constexpr (BLOCK_N == 128) {
      if (tma_store && !cluster) return launch<128, EPI_RES_STATS_BF16, true, false>(ta, tb, tc, tr, args, stream);
    }
    return fail(-2, "gemm_bf16: residual-statistics epilogue: unsupported tile configuration");
  }
  if (tma_store) {
    switch (epi) {
      case EPI_BIAS_BF16: return launch<BLOCK_N, EPI_BIAS_BF16, true, false>(ta, tb, tc, tr, args, stream);
      case EPI_BIAS_QGELU_BF16: return launch<BLOCK_N, EPI_BIAS_QGELU_BF16, true, false>(ta, tb, tc, tr, args, stream);
      case EPI_BIAS_F32: return launch<BLOCK_N, EPI_BIAS_F32, true, false>(ta, tb, tc, tr, args, stream);
      case EPI_LN_BIAS_BF16: return launch<BLOCK_N, EPI_LN_BIAS_BF16, true, false>(ta, tb, tc, tr, args, stream);
      case EPI_LN_BIAS_QGELU_BF16: return launch<BLOCK_N, EPI_LN_BIAS_QGELU_BF16, true, false>(ta, tb, tc, tr, args, stream);
    }
  }
  switch (epi) {
    case EPI_BIAS_BF16: return launch<BLOCK_N, EPI_BIAS_BF16, false, false>(ta, tb, tc, tr, args, stream);
    case EPI_BIAS_QGELU_BF16: return launch<BLOCK_N, EPI_BIAS_QGELU_BF16, false, false>(ta, tb, tc, tr, args, stream);
    case EPI_BIAS_RES_F32: return launch<BLOCK_N, EPI_BIAS_RES_F32, false, false>(ta, tb, tc, tr, args, stream);
    case EPI_BIAS_F32: return launch<BLOCK_N, EPI_BIAS_F32, false, false>(ta, tb, tc, tr, args, stream);
  }
  return fail(-2, "gemm_bf16: unknown epilogue or unsupported output alignment for a fused-LayerNorm epilogue");
}

// Tile plan shared by the launcher and by callers that size the statistics buffer.
struct TilePlan {
  int bn, tiles_m, tiles_n;
  bool cluster;
};
TilePlan plan_tiles(int M, int N, int epilogue, bool tma_store) {
  TilePlan t;
  // Tile width: 256 for the wide encoder GEMMs; 128 when N is small or the 256-wide grid would leave SMs idle.
  t.tiles_m = (M + BLOCK_M - 1) / BLOCK_M;
  t.bn = 256;
  if (N <= 128 || (N % 256 != 0 && N % 128 == 0) || t.tiles_m * ((N + 255) / 256) < num_sms()) t.bn = 128;
  // (Measured at the 5-clip EgoMCQ shape, 41 row tiles: choosing 128-wide tiles by wave count loses -- qkv 41.9 vs 31.1 us,
  // proj 22.4 vs 16.7, fc1 52.1 vs 37.3, fc2 59.2 vs 45.4 -- a 128-wide tile costs far more than half a 256-wide one.)
  // CTA pairs once there are enough row tiles to pair up: one 256-row MMA (cta_group::2) on the wide tiles, the W tile
  // multicast to two 1-SM MMAs on the 128-wide ones
  t.cluster = tma_store && t.tiles_m >= num_sms() / 2 && (num_sms() % 2 == 0);
  // the residual epilogue's shared-memory plan exists for 2-SM 256-wide and plain 128-wide tiles
  if (epilogue == EPI_RES_STATS_BF16 && !(t.cluster && t.bn == 256)) {
    t.bn = 128;
    t.cluster = false;
  }
  t.tiles_n = (N + t.bn - 1) / t.bn;
  return t;
}

}  // namespace

#ifdef HH_GEMM_TRACE
extern "C" int hh_debug_gemm_trace(unsigned long long* out, int n) {
  if (n > 148 * 16) n = 148 * 16;
  return static_cast<int>(cudaMemcpyFromSymbol(out, g_gemm_trace, sizeof(unsigned long long) * n));
}
#endif

int gemm_stats_parts(int M, int N) { return plan_tiles(M, N, EPI_RES_STATS_BF16, true).tiles_n; }

static int gemm_impl(const bf16* A, int lda, int seg_rows, int seg_pitch, const bf16* W, int ldw, void* out, int ldc,
                     const float* bias, float* residual, int ldr, int M, int N, int K, int epilogue, const GemmFuse& fuse,
                     cudaStream_t stream) {
  HH_REQUIRE(M > 0 && N > 0 && K > 0, "gemm_bf16: empty problem");
  HH_REQUIRE(lda % 8 == 0 && ldw % 8 == 0, "gemm_bf16: lda/ldw must be multiples of 8 elements (16-byte TMA strides)");
  HH_REQUIRE(K % 8 == 0, "gemm_bf16: K must be a multiple of 8");
  HH_REQUIRE((reinterpret_cast<uintptr_t>(A) & 15) == 0 && (reinterpret_cast<uintptr_t>(W) & 15) == 0,
             "gemm_bf16: A and W must be 16-byte aligned");
  const bool lnf = (epilogue == EPI_LN_BIAS_BF16 || epilogue == EPI_LN_BIAS_QGELU_BF16);
  const bool res = (epilogue == EPI_RES_STATS_BF16);
  const bool out_bf16 = (epilogue == EPI_BIAS_BF16 || epilogue == EPI_BIAS_QGELU_BF16 || lnf || res);
  if (out_bf16) {
    HH_REQUIRE(ldc % 2 == 0 && (reinterpret_cast<uintptr_t>(out) & 3) == 0, "gemm_bf16: bf16 output needs even ldc");
  }
  if (epilogue == EPI_BIAS_RES_F32) HH_REQUIRE(residual != nullptr, "gemm_bf16: residual epilogue without residual");

  // bulk-tensor stores need a 16-byte aligned base and row pitch; the residual epilogue reads while it writes
  const int esz = out_bf16 ? 2 : 4;
  const bool tma_store = epilogue != EPI_BIAS_RES_F32 && (reinterpret_cast<uintptr_t>(out) & 15) == 0 &&
                         (static_cast<size_t>(ldc) * esz) % 16 == 0;
  if (lnf) {
    HH_REQUIRE(tma_store, "gemm_bf16: folded-LayerNorm epilogue needs a 16-byte aligned output and row pitch");
    HH_REQUIRE(fuse.colsum && fuse.stats_in && fuse.stats_parts > 0 && fuse.norm_dim > 0,
               "gemm_bf16: folded-LayerNorm epilogue without colsum / statistics");
  }
  if (res) {
    HH_REQUIRE(tma_store, "gemm_bf16: residual-statistics epilogue needs a 16-byte aligned output and row pitch");
    HH_REQUIRE(residual && fuse.stats_out, "gemm_bf16: residual-statistics epilogue without residual / statistics buffer");
    HH_REQUIRE((reinterpret_cast<uintptr_t>(residual) & 15) == 0 && ldr % 4 == 0,
               "gemm_bf16: residual must be 16-byte aligned with a 16-byte multiple row pitch");
  }
  int a_rows = M;   // rows A's tensor map covers
  if (seg_rows > 0) {
    HH_REQUIRE(seg_rows % BLOCK_M == 0 && M % seg_rows == 0 && seg_pitch >= seg_rows,
               "gemm_bf16_rowseg: segments must be whole 128-row tiles, M a whole number of segments, pitch >= rows");
    const long long span = static_cast<long long>(M / seg_rows - 1) * seg_pitch + seg_rows;
    HH_REQUIRE(span <= 0x7fffffffLL, "gemm_bf16_rowseg: A spans too many rows");
    a_rows = static_cast<int>(span);
  }
  const TilePlan t = plan_tiles(M, N, epilogue, tma_store);
  const int bn = t.bn;
  CUtensorMap ta, tb, tc, tr;
  int rc = make_tmap(&ta, A, a_rows, K, lda, BLOCK_M);
  if (rc) return rc;
  rc = make_tmap(&tb, W, N, K, ldw, t.cluster ? bn / 2 : bn);
  if (rc) return rc;
  if (tma_store) {
    rc = make_tmap(&tc, out, M, N, ldc, 32, esz);
    if (rc) return rc;
  } else {
    tc = ta;
  }
  if (res) {
    rc = make_tmap(&tr, residual, M, N, ldr, 32, 4);
    if (rc) return rc;
  } else {
    tr = ta;
  }

  GemmArgs args;
  args.out = out;
  args.bias = bias;
  args.residual = residual;
  args.M = M;
  args.N = N;
  args.K = K;
  args.ldc = ldc;
  args.ldr = ldr;
  args.tiles_m = t.tiles_m;
  args.tiles_n = t.tiles_n;
  args.colsum = fuse.colsum;
  args.stats_in = fuse.stats_in;
  args.stats_parts = fuse.stats_parts;
  args.inv_d = fuse.norm_dim > 0 ? 1.0f / static_cast<float>(fuse.norm_dim) : 0.f;
  args.eps = fuse.eps;
  args.stats_out = fuse.stats_out;
  args.writeback = fuse.writeback;
  args.a_seg_rows = seg_rows > 0 ? seg_rows : 0;
  args.a_seg_skip = seg_rows > 0 ? seg_pitch - seg_rows : 0;
  if (bn == 256) return dispatch_epi<256>(ta, tb, tc, tr, tma_store, t.cluster, args, epilogue, stream);
  return dispatch_epi<128>(ta, tb, tc, tr, tma_store, t.cluster, args, epilogue, stream);
}

int gemm_bf16_fused(const bf16* A, int lda, const bf16* W, int ldw, void* out, int ldc, const float* bias,
                    float* residual, int ldr, int M, int N, int K, int epilogue, const GemmFuse& fuse,
                    cudaStream_t stream) {
  return gemm_impl(A, lda, 0, 0, W, ldw, out, ldc, bias, residual, ldr, M, N, K, epilogue, fuse, stream);
}

int gemm_bf16_rowseg(const bf16* A, int lda, int seg_rows, int seg_pitch, const bf16* W, int ldw, void* out, int ldc,
                     const float* bias, int M, int N, int K, int epilogue, cudaStream_t stream) {
  HH_REQUIRE(epilogue == EPI_BIAS_BF16 || epilogue == EPI_BIAS_F32, "gemm_bf16_rowseg: plain bias epilogues only");
  HH_REQUIRE(seg_rows > 0, "gemm_bf16_rowseg: seg_rows must be positive");
  return gemm_impl(A, lda, seg_rows, seg_pitch, W, ldw, out, ldc, bias, nullptr, 0, M, N, K, epilogue, GemmFuse{}, stream);
}

int gemm_bf16(const bf16* A, int lda, const bf16* W, int ldw, void* out, int ldc, const float* bias,
              const float* residual, int ldr, int M, int N, int K, int epilogue, cudaStream_t stream) {
  HH_REQUIRE(epilogue >= EPI_BIAS_BF16 && epilogue <= EPI_BIAS_F32, "gemm_bf16: unknown epilogue");
  return gemm_bf16_fused(A, lda, W, ldw, out, ldc, bias, const_cast<float*>(residual), ldr, M, N, K, epilogue, GemmFuse{},
                         stream);
}

}  // namespace hh
