// Spatial attention on the 5th-generation tensor cores (tcgen05 + TMEM), n <= 256 patches per frame, head dim 64.
// Same operator as attn_space.cu (VarAttention '(b f) n d', model/LaviLa.py:246-283); that file's mma.sync statement of
// it runs the frames of more than 256 patches.
//
// One task = one (clip, frame, head): Q, K, V tiles of [n x 64] bf16.  All n keys fit one accumulator tile, so the
// softmax is a single exact pass (no online rescaling):
//     S[256 x 256] = Q K^T     2 halves of 128 rows: tcgen05.mma 128x256x16, A = Q (smem), B = K (smem), D -> TMEM
//     P = exp2(S - max)        written back to TMEM as bf16 over the S columns
//     O[256 x 64]  = P V       tcgen05.mma 128x64x16, A = P (TMEM), B = V (smem, N-major), D -> TMEM
// plus the CLS key/value (one extra logit per row, folded in registers).
//
// The two 128-row halves of a task are INDEPENDENT chains (S -> max -> exp -> P V -> store) that run half a period
// apart: while one half's 8 warps are in the exp pass (MUFU), the other half's are in the phases that do not touch the
// MUFU (waiting for S, row maxima, O read-out, stores).  What keeps them apart is that nothing couples them: Q (per
// half), K and V have their own full / empty barriers, so a tile is refilled as soon as ITS last reader is done (K right
// after the second S, Q[h] after half h's output store has left its rows, V after the second P V), and the MMA thread
// polls both chains instead of waiting on either.
//
// Persistent CTA, 24 warps:
//    0      TMA producer (4-D tensor maps, 128-row boxes: rows past n are zero-filled / clipped by hardware; the next
//           task's tiles are in flight into the other smem stage while this one is processed)
//    1, 3   MMA issuers (one thread per half, each blocking on its own chain of barriers);  2  TMEM allocator
//    4-11   softmax + epilogue: ONE thread per query row (TMEM lane r = row r of a half, all 256 key columns), 4 warps per
//           half.  512 threads leave 128 registers per thread: the next 32-column chunk's tcgen05.ld is in flight under
//           the current chunk's arithmetic in both passes, and no cross-thread max / sum exchange (named barriers, shared
//           memory round trips) is left in a half's chain
//    12-15  legacy-MMA helpers (highest warp ids = highest issue priority, they gate the softmax warps): the CLS-key
//           logit of every row (q_r . k_cls) and the CLS *query*'s partial softmax over this frame's keys (merged
//           across frames by attn_cls_merge)
// TMEM (512 columns), half h owns [256h, 256h+256): S; then P (bf16 pairs) of keys 0..127 in [0,64), O in [64,128), P of
// keys 128..255 in [128,192), the CLS key's probability (one K = 16 block) in [192,200).  P V runs in two parts: keys
// 0..127 as soon as the first four chunks of the exp pass are written (under the second half of the pass), the rest
// (+ the CLS value as a 17th K step against a [16 x 64] tile whose row 0 is v_cls) when the pass is done.
#include <cstdio>
#include <cstdlib>

#include "hh_internal.h"
#include "hh_ptx.cuh"

namespace hh {

namespace {

constexpr int HD = 64;
constexpr int ROWS = 256;                 // query / key slots per task
constexpr int TILE_BYTES = ROWS * 128;    // 32 KB: [256 rows x 64 bf16], SWIZZLE_128B
constexpr int STAGE_BYTES = 3 * TILE_BYTES;
constexpr int NSTAGE = 2;
constexpr int NCLS = 4;                     // CLS-vector ring: a slot is rewritten 4 tasks later, long after its readers
constexpr int VCLS_BYTES = 16 * 128;        // [16 keys x 64] bf16 B tile of the CLS value: row 0 = v_cls, rows 1..15 zero
constexpr int HALF_BYTES = TILE_BYTES / 2; // one 128-row box
constexpr int NTHREADS = 512;                // 16 warps: 128 registers per thread
constexpr float LOG2E = 1.4426950408889634f;
constexpr int PART = HD + 2;

struct SmemExtras {
  __nv_bfloat16 cls_q[NCLS][HD];     // q, k, v of the CLS token for (clip, head): ring over the last NCLS tasks
  __nv_bfloat16 cls_k[NCLS][HD];
  float scls[NSTAGE][ROWS];          // CLS-key logit of every query row
  float merge[4][PART];              // CLS-query partials of the four helper warps
  uint64_t q_full[NSTAGE][2], k_full[NSTAGE], v_full[NSTAGE];      // per tile: Q rows of half h, K (+ CLS vectors), V
  uint64_t q_empty[NSTAGE][2], k_empty[NSTAGE], v_empty[NSTAGE];
  uint64_t scls_full[NSTAGE][2];     // CLS-key logits of half h's rows (helper warps 2h, 2h + 1)
  uint64_t s_full[2], p_full[2][2], o_full[2], t_free[2];   // p_full[h][part]: P of keys 0..127 / 128..255 (+ CLS) written
  uint64_t x_done[2][4];             // exp pass of half h, TMEM lane quarter q finished (the turn passes to the other half)
  uint32_t tmem_slot;
};
constexpr int SMEM_BYTES = 1024 + NSTAGE * STAGE_BYTES + NCLS * VCLS_BYTES + static_cast<int>(sizeof(SmemExtras)) + 64;

struct TcArgs {
  const bf16* qkv;
  float* cls_part;
  int B, T, n, H;
  unsigned long long* trace;   // debug: [role][task][event] %globaltimer stamps of CTA 0 (nullptr = off)
};

constexpr int TR_TASKS = 8, TR_EVENTS = 8, TR_ROLES = 6;
__device__ __forceinline__ void trace_ev(const TcArgs& p, int role, int it, int ev) {
  if (p.trace != nullptr && blockIdx.x == 0 && it < TR_TASKS) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    p.trace[(role * TR_TASKS + it) * TR_EVENTS + ev] = t;
  }
}

// tasks are walked from the last (clip, frame, head): those q/k/v rows were written last by the QKV GEMM and are still
// in L2, and the projection GEMM that follows reads the rows this kernel writes last (the first clips) first
__device__ __forceinline__ int task_index(int task, int ntasks) { return ntasks - 1 - task; }

__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint32_t sw128(uint32_t tile, int row, int chunk) {
  return tile + static_cast<uint32_t>(row * 128 + ((chunk ^ (row & 7)) << 4));
}

// kFull: n == 256 exactly (the L/14 geometry): no ragged-chunk code in the softmax loops (half the code bytes of the hot
// loop, compile-time trip counts).
template <bool kFull>
__global__ void __launch_bounds__(NTHREADS, 1)
attn_space_tc_kernel(const __grid_constant__ CUtensorMap tm_in, const __grid_constant__ CUtensorMap tm_out,
                     const TcArgs p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* vcls = smem + NSTAGE * STAGE_BYTES;   // NCLS tiles of VCLS_BYTES (1024-byte aligned: two SWIZZLE_128B atoms each)
  SmemExtras* ex = reinterpret_cast<SmemExtras*>(vcls + NCLS * VCLS_BYTES);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int D = p.H * HD;
  const int N = 1 + p.T * p.n;
  const int ntasks = p.B * p.T * p.H;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_in);
    tma_prefetch_desc(&tm_out);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < NSTAGE; ++s) {
      for (int h = 0; h < 2; ++h) {
        mbar_init(&ex->q_full[s][h], 1);
        mbar_init(&ex->q_empty[s][h], 5);   // the half's 4 warps (output store has left the rows) + helper warps
      }
      mbar_init(&ex->k_full[s], 1);
      mbar_init(&ex->v_full[s], 1);
      mbar_init(&ex->k_empty[s], 3);        // commit after each half's S + helper warps
      mbar_init(&ex->v_empty[s], 3);        // commit after each half's P V + helper warps
      mbar_init(&ex->scls_full[s][0], 2);
      mbar_init(&ex->scls_full[s][1], 2);
    }
    for (int h = 0; h < 2; ++h) {
      mbar_init(&ex->s_full[h], 1);
      mbar_init(&ex->p_full[h][0], 4);
      mbar_init(&ex->p_full[h][1], 4);
      mbar_init(&ex->o_full[h], 1);
      mbar_init(&ex->t_free[h], 4);
      for (int q = 0; q < 4; ++q) mbar_init(&ex->x_done[h][q], 1);
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc(&ex->tmem_slot, 512);
    tmem_relinquish();
  }
  for (int i = threadIdx.x; i < NCLS * VCLS_BYTES / 16; i += NTHREADS) reinterpret_cast<uint4*>(vcls)[i] = make_uint4(0u, 0u, 0u, 0u);
  fence_proxy_async_smem();   // rows 1..15 of the CLS-value tiles stay zero; row 0 is rewritten by the producer's bulk copies
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = ex->tmem_slot;
  if (p.trace != nullptr && blockIdx.x == 0 && threadIdx.x == 0) {   // SM clock of the run: (clock64, globaltimer) pairs
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    p.trace[TR_ROLES * TR_TASKS * TR_EVENTS + 0] = t;
    p.trace[TR_ROLES * TR_TASKS * TR_EVENTS + 1] = static_cast<unsigned long long>(clock64());
  }

  if (warp == 0) {
    // ================================================================== TMA producer
    if (lane == 0) {
      int it = 0;
      for (int task = blockIdx.x; task < ntasks; task += gridDim.x, ++it) {
        const int st = it & 1;
        const uint32_t ph = (it >> 1) & 1;
        const int tk = task_index(task, ntasks); const int h = tk % p.H, f = (tk / p.H) % p.T, b = tk / (p.H * p.T);
        const int cs = it & (NCLS - 1);
        uint8_t* base = smem + st * STAGE_BYTES;
        // tiles in the order their previous contents die: K, Q[0], V, Q[1]
        mbar_wait(&ex->k_empty[st], ph ^ 1u);
        trace_ev(p, 0, it, 0);
        mbar_arrive_expect_tx(&ex->k_full[st], TILE_BYTES + 3 * HD * 2);
        tma_load_4d(&tm_in, &ex->k_full[st], base + TILE_BYTES, D + h * HD, 0, f, b);
        tma_load_4d(&tm_in, &ex->k_full[st], base + TILE_BYTES + HALF_BYTES, D + h * HD, 128, f, b);
        const bf16* cls = p.qkv + static_cast<size_t>(b) * N * 3 * D + h * HD;
        bulk_load_1d(ex->cls_q[cs], cls, HD * 2, &ex->k_full[st]);
        bulk_load_1d(ex->cls_k[cs], cls + D, HD * 2, &ex->k_full[st]);
        bulk_load_1d(vcls + cs * VCLS_BYTES, cls + 2 * D, HD * 2, &ex->k_full[st]);   // row 0 of a swizzle atom is unswizzled
        mbar_wait(&ex->q_empty[st][0], ph ^ 1u);
        mbar_arrive_expect_tx(&ex->q_full[st][0], HALF_BYTES);
        tma_load_4d(&tm_in, &ex->q_full[st][0], base, h * HD, 0, f, b);
        mbar_wait(&ex->v_empty[st], ph ^ 1u);
        mbar_arrive_expect_tx(&ex->v_full[st], TILE_BYTES);
        tma_load_4d(&tm_in, &ex->v_full[st], base + 2 * TILE_BYTES, 2 * D + h * HD, 0, f, b);
        tma_load_4d(&tm_in, &ex->v_full[st], base + 2 * TILE_BYTES + HALF_BYTES, 2 * D + h * HD, 128, f, b);
        mbar_wait(&ex->q_empty[st][1], ph ^ 1u);
        mbar_arrive_expect_tx(&ex->q_full[st][1], HALF_BYTES);
        tma_load_4d(&tm_in, &ex->q_full[st][1], base + HALF_BYTES, h * HD, 128, f, b);
      }
    }
  } else if (warp == 1 || warp == 3) {
    // ================================================================== MMA issuers: one thread per half
    // Each half is an independent chain S -> P V (keys 0..127) -> P V (keys 128..255 + CLS) with its own issuing thread,
    // which BLOCKS on the next barrier of its chain (wake-up ~90 cycles after the arrive).  One thread polling both
    // chains with bounded mbarrier.try_wait reacted 3 000 - 7 000 cycles late: a try_wait on a barrier that does not
    // complete suspends for a hardware time far above its hint (tools/ubench_mbar.cu).
    if (lane == 0) {
      constexpr uint32_t idesc_s = umma_idesc_bf16(128, 256);
      constexpr uint32_t idesc_o = umma_idesc_bf16_bmn(128, HD);
      const int hf = warp >> 1;
      const uint32_t th = tmem_base + hf * 256;
      int u = 0;
      for (int task = blockIdx.x; task < ntasks; task += gridDim.x, ++u) {
        const int st = u & 1;
        const uint32_t ph = (u >> 1) & 1;   // parity of the stage barriers
        const uint32_t tp = u & 1;          // parity of the per-task barriers
        const uint32_t qs = smem_u32(smem + st * STAGE_BYTES);
        const uint32_t ks = qs + TILE_BYTES, vs = qs + 2 * TILE_BYTES;
        mbar_wait(&ex->t_free[hf], tp ^ 1u);   // previous task's O has left these columns
        mbar_wait(&ex->q_full[st][hf], ph);
        mbar_wait(&ex->k_full[st], ph);
        if (hf == 0) trace_ev(p, 1, u, 0);
        tc_fence_after();
        {
          const uint64_t da = umma_desc_sw128(qs + hf * HALF_BYTES);
          const uint64_t db = umma_desc_sw128(ks);
#pragma unroll
          for (int k = 0; k < HD / 16; ++k) umma_bf16(th, da + 2 * k, db + 2 * k, idesc_s, k > 0 ? 1u : 0u);
        }
        umma_commit(&ex->s_full[hf]);
        umma_commit(&ex->k_empty[st]);    // (with the other half's commit and the helpers) K may be refilled
        trace_ev(p, 1, u, 1 + hf);
        // P V, keys 0..127: P in columns [0, 64) of the half, O -> [64, 128) (S columns the exp pass has consumed)
        mbar_wait(&ex->p_full[hf][0], tp);
        mbar_wait(&ex->v_full[st], ph);
        trace_ev(p, 1, u, 3 + 2 * hf);
        tc_fence_after();
        const uint64_t dv = umma_desc_sw128_mn(vs);
#pragma unroll
        for (int k = 0; k < 8; ++k)   // 16 keys per instruction = 2 swizzle atoms of V, 8 TMEM columns of P
          umma_bf16_ts(th + 64, th + 8 * k, dv + static_cast<uint64_t>(k * 128), idesc_o, k > 0 ? 1u : 0u);
        // keys 128..255: P in [128, 192); then the CLS key: probability block in [192, 200) against the v_cls tile
        mbar_wait(&ex->p_full[hf][1], tp);
        tc_fence_after();
#pragma unroll
        for (int k = 8; k < 16; ++k)
          umma_bf16_ts(th + 64, th + 64 + 8 * k, dv + static_cast<uint64_t>(k * 128), idesc_o, 1u);
        umma_bf16_ts(th + 64, th + 192, umma_desc_sw128_mn(smem_u32(vcls + (u & (NCLS - 1)) * VCLS_BYTES)), idesc_o, 1u);
        umma_commit(&ex->o_full[hf]);
        umma_commit(&ex->v_empty[st]);
        trace_ev(p, 1, u, 4 + 2 * hf);
      }
    }
  } else if (warp >= 12) {
    // ================================================================== helpers on the legacy tensor-core path
    // 4 warps; every warp takes 4 of the 16 query-row blocks for the CLS-key logits and 64 of the 256 keys for the
    // CLS-query partial.  Fragment loads are issued in batches ahead of the MMAs that use them (one warp has no other
    // warp to hide its ldmatrix -> mma latency behind).
    const int ww = warp - 12;
    const int g = lane >> 2, t = lane & 3;
    const int mi = lane >> 3, lr = lane & 7;
    int it = 0;
    for (int task = blockIdx.x; task < ntasks; task += gridDim.x, ++it) {
      const int st = it & 1;
      const uint32_t ph = (it >> 1) & 1;
      const int tk = task_index(task, ntasks); const int h = tk % p.H, f = (tk / p.H) % p.T, b = tk / (p.H * p.T);
      const int cs = it & (NCLS - 1);
      // this warp's 64 query rows belong to half ww / 2: their CLS-key logits only need that half of Q (and k_cls)
      mbar_wait(&ex->k_full[st], ph);
      mbar_wait(&ex->q_full[st][ww >> 1], ph);
      if (ww == 0 && lane == 0) trace_ev(p, 2, it, 0);
      const uint32_t qs = smem_u32(smem + st * STAGE_BYTES);
      const uint32_t ks = qs + TILE_BYTES, vs = ks + TILE_BYTES;

      // ---- (1) CLS-key logit of every query row: S_cls = Q . k_cls, as m16n8k16 with k_cls in column 0 of B
      uint32_t kb0[4], kb1[4];
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        kb0[kk] = (g == 0) ? *reinterpret_cast<const uint32_t*>(&ex->cls_k[cs][kk * 16 + 2 * t]) : 0u;
        kb1[kk] = (g == 0) ? *reinterpret_cast<const uint32_t*>(&ex->cls_k[cs][kk * 16 + 8 + 2 * t]) : 0u;
      }
#pragma unroll
      for (int half = 0; half < 2; ++half) {   // 2 x 2 row blocks; 8 fragment loads in flight
        uint32_t qf[2][4][4];
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            ldsm_x4(qf[i][kk], sw128(qs, (ww * 4 + half * 2 + i) * 16 + (mi & 1) * 8 + lr, kk * 2 + (mi >> 1)));
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) mma_bf16_16816(acc, qf[i][kk], kb0[kk], kb1[kk]);
          if (t == 0) {  // column 0 of the 16x8 result: rows g and g+8
            const int mb = ww * 4 + half * 2 + i;
            ex->scls[st][mb * 16 + g] = acc[0];
            ex->scls[st][mb * 16 + g + 8] = acc[2];
          }
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&ex->scls_full[st][ww >> 1]);
      if (ww == 0 && lane == 0) trace_ev(p, 2, it, 1);
      mbar_wait(&ex->v_full[st], ph);   // part (2) reads K and V

      // ---- (2) CLS query vs this warp's 64 keys: online softmax over 2 blocks of 32 keys, row 0 of the A block live
      uint32_t qa0[4], qa2[4];
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        qa0[kk] = (g == 0) ? *reinterpret_cast<const uint32_t*>(&ex->cls_q[cs][kk * 16 + 2 * t]) : 0u;
        qa2[kk] = (g == 0) ? *reinterpret_cast<const uint32_t*>(&ex->cls_q[cs][kk * 16 + 8 + 2 * t]) : 0u;
      }
      float m = -INFINITY, l = 0.f;
      float o[8][4];
#pragma unroll
      for (int ni = 0; ni < 8; ++ni) o[ni][0] = o[ni][1] = o[ni][2] = o[ni][3] = 0.f;
#pragma unroll 1
      for (int blk = 0; blk < 2; ++blk) {
        const int key0 = ww * 64 + blk * 32;
        if (key0 >= p.n) break;
        uint32_t kf[8][4];
#pragma unroll
        for (int kk = 0; kk < 4; ++kk)
#pragma unroll
          for (int np = 0; np < 2; ++np)
            ldsm_x4(kf[kk * 2 + np], sw128(ks, key0 + np * 16 + (mi >> 1) * 8 + lr, kk * 2 + (mi & 1)));
        float s[4][4];
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) s[ni][0] = s[ni][1] = s[ni][2] = s[ni][3] = 0.f;
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          const uint32_t qf[4] = {qa0[kk], 0u, qa2[kk], 0u};
#pragma unroll
          for (int np = 0; np < 2; ++np) {
            mma_bf16_16816(s[2 * np], qf, kf[kk * 2 + np][0], kf[kk * 2 + np][1]);
            mma_bf16_16816(s[2 * np + 1], qf, kf[kk * 2 + np][2], kf[kk * 2 + np][3]);
          }
        }
        uint32_t vf[8][4];   // V fragments of this block: in flight during the softmax arithmetic
#pragma unroll
        for (int kk = 0; kk < 2; ++kk)
#pragma unroll
          for (int dp = 0; dp < 4; ++dp)
            ldsm_x4_trans(vf[kk * 4 + dp], sw128(vs, key0 + kk * 16 + (mi & 1) * 8 + lr, dp * 2 + (mi >> 1)));
        float mx = -INFINITY;
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) {
          const int key = key0 + ni * 8 + 2 * t;
          if (key >= p.n) s[ni][0] = -INFINITY;
          if (key + 1 >= p.n) s[ni][1] = -INFINITY;
          mx = fmaxf(mx, fmaxf(s[ni][0], s[ni][1]));
        }
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
        const float mn = fmaxf(m, mx);       // finite: key0 < n
        const float corr = fast_exp2((m - mn) * LOG2E);
        m = mn;
        l *= corr;
        uint32_t pa[2][4];
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) {
          const float p0 = fast_exp2(fmaf(s[ni][0], LOG2E, -mn * LOG2E)), p1 = fast_exp2(fmaf(s[ni][1], LOG2E, -mn * LOG2E));
          l += p0 + p1;
          pa[ni >> 1][(ni & 1) * 2 + 0] = pack_bf16x2(p0, p1);
          pa[ni >> 1][(ni & 1) * 2 + 1] = 0u;
        }
#pragma unroll
        for (int ni = 0; ni < 8; ++ni) {
          o[ni][0] *= corr;
          o[ni][1] *= corr;
        }
#pragma unroll
        for (int kk = 0; kk < 2; ++kk) {
#pragma unroll
          for (int dp = 0; dp < 4; ++dp) {
            mma_bf16_16816(o[2 * dp], pa[kk], vf[kk * 4 + dp][0], vf[kk * 4 + dp][1]);
            mma_bf16_16816(o[2 * dp + 1], pa[kk], vf[kk * 4 + dp][2], vf[kk * 4 + dp][3]);
          }
        }
      }
      l += __shfl_xor_sync(0xffffffffu, l, 1);
      l += __shfl_xor_sync(0xffffffffu, l, 2);
      // row 0 lives in lanes 0..3 (g == 0): the four warps' partials are folded by warp 4 and written to [b][h][f]
      if (g == 0) {
        float* mg = ex->merge[ww];
        if (t == 0) {
          mg[0] = m;
          mg[1] = l;
        }
#pragma unroll
        for (int ni = 0; ni < 8; ++ni) {
          mg[2 + ni * 8 + 2 * t] = o[ni][0];
          mg[2 + ni * 8 + 2 * t + 1] = o[ni][1];
        }
      }
      asm volatile("bar.sync 2, 128;" ::: "memory");
      if (ww == 0 && g == 0) {
        float mm = -INFINITY;
#pragma unroll
        for (int w = 0; w < 4; ++w) mm = fmaxf(mm, ex->merge[w][0]);
        float cw[4], ll = 0.f;
#pragma unroll
        for (int w = 0; w < 4; ++w) {
          cw[w] = (ex->merge[w][0] == -INFINITY) ? 0.f : fast_exp2((ex->merge[w][0] - mm) * LOG2E);
          ll += ex->merge[w][1] * cw[w];
        }
        float* dst = p.cls_part + ((static_cast<size_t>(b) * p.H + h) * p.T + f) * PART;
        if (t == 0) {
          dst[0] = mm;
          dst[1] = ll;
        }
#pragma unroll
        for (int ni = 0; ni < 8; ++ni) {
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int idx = 2 + ni * 8 + 2 * t + e;
            dst[idx] = ex->merge[0][idx] * cw[0] + ex->merge[1][idx] * cw[1] + ex->merge[2][idx] * cw[2] +
                       ex->merge[3][idx] * cw[3];
          }
        }
      }
      asm volatile("bar.sync 2, 128;" ::: "memory");  // merge[] reusable; all four warps are done with Q, K and V
      if (ww == 0 && lane == 0) {
        mbar_arrive(&ex->k_empty[st]);
        mbar_arrive(&ex->v_empty[st]);
        mbar_arrive(&ex->q_empty[st][0]);
        mbar_arrive(&ex->q_empty[st][1]);
        trace_ev(p, 2, it, 2);
      }
    }
  } else if (warp >= 4) {
    // ================================================================== softmax + epilogue (one thread per row)
    const int sw = warp - 4;                  // 0..7
    const int hf = sw >> 2;                   // 0: rows 0..127, 1: rows 128..255 (TMEM half hf)
    const int wq = warp & 3;                  // TMEM lane quarter of this warp
    const int rl = wq * 32 + lane;            // row within the half
    const int r = hf * 128 + rl;              // row within the task
    const int jh = hf;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(wq * 32) << 16) + static_cast<uint32_t>(hf * 256);
    const uint32_t s_col = t_lane;            // this row's 256 S columns
    const uint32_t o_col = t_lane + 64;       // its 64 O columns
    // P chunk c (32 keys = 16 packed columns) goes behind the S columns already consumed: keys 0..127 -> [0, 64), keys
    // 128..255 -> [128, 192) (chunk c <= 3: column 16c lies in S chunk c / 2; chunk c >= 4: 64 + 16c lies in S chunk c - 2 .. c)
    const int nvalid = kFull ? ROWS : min(ROWS, p.n);        // valid keys
    const int nch = kFull ? 8 : ((nvalid + 31) >> 5);        // 32-key chunks that hold valid keys (1..8)
    int u = 0;
    int release_st = -1;   // stage whose output store may still be reading its staging rows: released one task later,
                           // after the next task's first pass, instead of stalling the epilogue on the bulk-store read
    for (int task = blockIdx.x; task < ntasks; task += gridDim.x, ++u) {
      const int st = u & 1;
      const uint32_t ph = (u >> 1) & 1;
      const uint32_t tp = u & 1;
      const int tk = task_index(task, ntasks); const int h = tk % p.H, f = (tk / p.H) % p.T, b = tk / (p.H * p.T);
      const uint32_t qs = smem_u32(smem + st * STAGE_BYTES);
      mbar_wait(&ex->scls_full[st][hf], ph);
      const float s_cls = ex->scls[st][r];
      const bool tr = (wq == 0 && lane == 0);
      mbar_wait(&ex->s_full[hf], tp);
      if (tr) trace_ev(p, 3 + jh, u, 0);
      tc_fence_after();

      uint32_t va[32], vb[32];
      // ---- pass 1: row maximum; chunk c + 1 is being loaded from TMEM while chunk c is folded
      float mx = s_cls;
      float mq[4] = {s_cls, s_cls, s_cls, s_cls};   // four independent chains: one chunk's 16 three-input maxima are not serial
      {
        auto fold = [&](const uint32_t(&v)[32], int c) {
          if (kFull || c * 32 + 32 <= nvalid) {
#pragma unroll
            for (int j = 0; j < 32; j += 2)
              asm("max.f32 %0, %0, %1, %2;" : "+f"(mq[(j >> 1) & 3]) : "f"(__uint_as_float(v[j])), "f"(__uint_as_float(v[j + 1])));
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (c * 32 + j < nvalid) mx = fmaxf(mx, __uint_as_float(v[j]));
          }
        };
        tmem_ld_32x32b_x32(s_col, va);
#pragma unroll 1
        for (int c = 0; c < nch; c += 2) {
          tmem_ld_wait();
          if (c + 1 < nch) tmem_ld_32x32b_x32(s_col + (c + 1) * 32, vb);
          fold(va, c);
          if (c + 1 < nch) {
            tmem_ld_wait();
            if (c + 2 < nch) tmem_ld_32x32b_x32(s_col + (c + 2) * 32, va);
            fold(vb, c + 1);
          }
        }
        mx = fmaxf(fmaxf(mx, mq[0]), fmaxf(fmaxf(mq[1], mq[2]), mq[3]));
      }
      if (tr) trace_ev(p, 3 + jh, u, 1);
      if (release_st >= 0 && lane == 0) {
        tma_store_wait_read<0>();
        mbar_arrive(&ex->q_empty[release_st][hf]);
      }
      const float ml = mx * LOG2E;
      const float p_cls = fast_exp2(fmaf(s_cls, LOG2E, -ml));
      // The exp pass is the one phase that saturates a shared unit (MUFU: 4 lanes per clock and scheduler).  The two warps
      // of a scheduler (same TMEM lane quarter, one per half) take strict turns in it -- h0(u), h1(u), h0(u + 1), ... -- so
      // one half's exponentials always run under the other half's MUFU-free phases (P V wait, read-out, next S, row
      // maxima).  Left to themselves the two chains have the same period and nothing keeps them half a period apart:
      // they drift into phase, share the MUFU during the exp pass and leave it idle for the rest of the period.
      if (hf == 1) mbar_wait(&ex->x_done[0][wq], tp);
      else if (u > 0) mbar_wait(&ex->x_done[1][wq], tp ^ 1u);
      if (tr) trace_ev(p, 3 + jh, u, 5);

      // ---- pass 2: P = exp2(S - max) as bf16 pairs, 32 keys per iteration of ONE small loop body (next to the helper
      // warps' code the hot loop stays in the instruction cache).  Software-pipelined by hand so that ptxas sees the
      // tcgen05.ld and its consumer in the same block: the SCALED chunk t[] is carried across the back edge; an iteration
      // first issues the load of the next chunk into x[] (dead), runs this chunk's exponentials on t[], and scales x[] into
      // t[] at the bottom.  (A load whose consumer sits in the next iteration is sunk behind the last reader of its
      // registers, i.e. to the end of the body, and its whole latency is exposed in every chunk.)
      float2 l2 = make_float2(0.f, 0.f);
      {
        const float2 sc = make_float2(LOG2E, LOG2E), sh = make_float2(-ml, -ml);
        uint32_t x[32];
        float2 t[16];
        tmem_ld_32x32b_x32(s_col, x);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j)
          t[j] = __ffma2_rn(make_float2(__uint_as_float(x[2 * j]), __uint_as_float(x[2 * j + 1])), sc, sh);
#pragma unroll 1
        for (int c = 0; c < 8; ++c) {
          uint32_t w[16];
          // unconditional (the last iteration re-reads chunk 0's columns, unused): a branch here would let the
          // exponentials be hoisted above it and put the load back at the bottom of the body
          tmem_ld_32x32b_x32(s_col + ((c + 1) & 7) * 32, x);
          if (kFull || c < nch) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              float2 e = make_float2(fast_exp2(t[j].x), fast_exp2(t[j].y));
              if (!kFull) {   // ragged last chunk (n = 196)
                if (c * 32 + 2 * j >= nvalid) e.x = 0.f;
                if (c * 32 + 2 * j + 1 >= nvalid) e.y = 0.f;
              }
              l2 = __fadd2_rn(l2, e);
              w[j] = pack_bf16x2(e.x, e.y);
            }
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) w[j] = 0u;
          }
          // 16 packed columns behind the S columns already consumed: keys 0..127 -> [0, 64), keys 128..255 -> [128, 192)
          tmem_st_32x32b_x16(t_lane + (c < 4 ? 16 * c : 64 + 16 * c), w);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; ++j)
            t[j] = __ffma2_rn(make_float2(__uint_as_float(x[2 * j]), __uint_as_float(x[2 * j + 1])), sc, sh);
          if (c == 3) {   // keys 0..127 are written: their P V runs under the rest of the pass
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&ex->p_full[hf][0]);
          }
        }
      }
      const float l = (l2.x + l2.y) + p_cls;
      if (lane == 0) mbar_arrive(&ex->x_done[hf][wq]);
      if (tr) trace_ev(p, 3 + jh, u, 6);
      {   // the CLS key's probability as key 0 of a 17th K = 16 block (columns [192, 200)); its B tile holds v_cls in row 0
        uint32_t wc[8] = {pack_bf16x2(p_cls, 0.f), 0u, 0u, 0u, 0u, 0u, 0u, 0u};
        tmem_st_32x32b_x8(t_lane + 192, wc);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&ex->p_full[hf][1]);
      if (tr) trace_ev(p, 3 + jh, u, 2);

      // ---- O = P V is in TMEM columns [192, 256) of this half: all 64 output dims of this row
      mbar_wait(&ex->o_full[hf], tp);
      if (tr) trace_ev(p, 3 + jh, u, 3);
      tc_fence_after();
      tmem_ld_32x32b_x32(o_col, va);
      tmem_ld_32x32b_x32(o_col + 32, vb);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&ex->t_free[hf]);   // the next task's S may overwrite this half

      // ---- normalise, stage the 64 bf16 values (128 B) of this row, bulk-store a 32-row x 128-B box
      float inv;
      asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"(l));
      const float2 inv2 = make_float2(inv, inv);
      // staging: the 4 KB of the (consumed) Q tile that belong to these 32 rows, SWIZZLE_128B
      const uint32_t stg = qs + static_cast<uint32_t>((jh * 128 + wq * 32) * 128);
      auto stage = [&](const uint32_t(&o)[32], int half32) {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint32_t wv[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float2 r = __fmul2_rn(make_float2(__uint_as_float(o[c * 8 + 2 * q]), __uint_as_float(o[c * 8 + 2 * q + 1])), inv2);
            wv[q] = pack_bf16x2(r.x, r.y);
          }
          st_shared_v4(sw128(stg, lane, half32 * 4 + c), wv[0], wv[1], wv[2], wv[3]);
        }
      };
      stage(va, 0);
      stage(vb, 1);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        const int row0 = jh * 128 + wq * 32;
        if (row0 < p.n) {
          tma_store_4d(&tm_out, stg, h * HD, row0, f, b);
          tma_store_commit();
        }
      }
      release_st = st;
      __syncwarp();
      if (tr) trace_ev(p, 3 + jh, u, 4);
    }
    if (lane == 0) tma_store_wait_read<0>();   // shared memory stays valid until the last store has read it
  }

  tc_fence_before();
  __syncthreads();
  if (p.trace != nullptr && blockIdx.x == 0 && threadIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    p.trace[TR_ROLES * TR_TASKS * TR_EVENTS + 2] = t;
    p.trace[TR_ROLES * TR_TASKS * TR_EVENTS + 3] = static_cast<unsigned long long>(clock64());
  }
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
  }
  return fn;
}

// [cols, n, T, B] view of a token matrix whose rows are (clip, 1 + frame*n + patch): skips the CLS row of each clip.
int make_map4d(CUtensorMap* map, const bf16* base_row1, int cols, int n, int T, int B, int N, int box_cols, int box_rows,
               CUtensorMapSwizzle swz) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(-3, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t gdim[4] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(n), static_cast<cuuint64_t>(T),
                        static_cast<cuuint64_t>(B)};
  cuuint64_t gstr[3] = {static_cast<cuuint64_t>(cols) * 2, static_cast<cuuint64_t>(n) * cols * 2,
                        static_cast<cuuint64_t>(N) * cols * 2};
  cuuint32_t box[4] = {static_cast<cuuint32_t>(box_cols), static_cast<cuuint32_t>(box_rows), 1, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<bf16*>(base_row1), gdim, gstr, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(-3, "cuTensorMapEncodeTiled (4-D) failed with CUresult " + std::to_string((int)r));
  return 0;
}

}  // namespace

bool attn_space_tc_supported(int n) { return n <= ROWS; }

int attn_space_tc(const bf16* qkv, bf16* out, int B, int T, int n, int H, float* cls_ws, cudaStream_t stream) {
  HH_REQUIRE(B > 0 && T > 0 && n > 0 && n <= ROWS && H > 0, "attn_space_tc: needs 1 <= n <= 256");
  HH_REQUIRE(cls_ws != nullptr, "attn_space_tc: CLS workspace");
  HH_REQUIRE((reinterpret_cast<uintptr_t>(qkv) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0,
             "attn_space_tc: 16-byte alignment");
  const int D = H * HD, N = 1 + T * n;
  CUtensorMap tm_in, tm_out;
  int rc = make_map4d(&tm_in, qkv + static_cast<size_t>(3) * D, 3 * D, n, T, B, N, 64, ROWS / 2, CU_TENSOR_MAP_SWIZZLE_128B);  // 128-row boxes
  if (rc) return rc;
  rc = make_map4d(&tm_out, out + D, D, n, T, B, N, 64, 32, CU_TENSOR_MAP_SWIZZLE_128B);
  if (rc) return rc;
  static bool configured = false;
  if (!configured) {
    HH_CHECK_CUDA(cudaFuncSetAttribute(attn_space_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    HH_CHECK_CUDA(cudaFuncSetAttribute(attn_space_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    configured = true;
  }
  TcArgs a;
  a.qkv = qkv;
  a.cls_part = cls_ws;
  a.B = B;
  a.T = T;
  a.n = n;
  a.H = H;
  a.trace = nullptr;
  static unsigned long long* trace_buf = nullptr;
  static const bool want_trace = std::getenv("HH_ATTN_TRACE") != nullptr;
  if (want_trace) {
    if (!trace_buf) HH_CHECK_CUDA(cudaMalloc(&trace_buf, sizeof(unsigned long long) * (TR_ROLES * TR_TASKS * TR_EVENTS + 4)));
    HH_CHECK_CUDA(cudaMemsetAsync(trace_buf, 0, sizeof(unsigned long long) * (TR_ROLES * TR_TASKS * TR_EVENTS + 4), stream));
    a.trace = trace_buf;
  }
  const int ntasks = B * T * H;
  int grid = num_sms();
  if (grid > ntasks) grid = ntasks;
  if (n == ROWS) attn_space_tc_kernel<true><<<grid, NTHREADS, SMEM_BYTES, stream>>>(tm_in, tm_out, a);
  else attn_space_tc_kernel<false><<<grid, NTHREADS, SMEM_BYTES, stream>>>(tm_in, tm_out, a);
  HH_CHECK_LAUNCH("attn_space_tc_kernel");
  if (want_trace) {  // debug only: dump the timeline of CTA 0 (ns relative to the first stamp)
    static unsigned long long host[TR_ROLES * TR_TASKS * TR_EVENTS + 4];
    HH_CHECK_CUDA(cudaStreamSynchronize(stream));
    HH_CHECK_CUDA(cudaMemcpy(host, trace_buf, sizeof(host), cudaMemcpyDeviceToHost));
    {
      const unsigned long long* ck = host + TR_ROLES * TR_TASKS * TR_EVENTS;
      const double ns = static_cast<double>(ck[2] - ck[0]), cyc = static_cast<double>(ck[3] - ck[1]);
      fprintf(stderr, "[attn trace] CTA 0 ran %.0f ns = %.0f SM cycles: %.3f GHz\n", ns, cyc, ns > 0 ? cyc / ns : 0.0);
    }
    unsigned long long t0 = ~0ull;
    for (int i = 0; i < TR_ROLES * TR_TASKS * TR_EVENTS; ++i) if (host[i] && host[i] < t0) t0 = host[i];
    const char* names[TR_ROLES] = {"producer", "mma", "helper", "softmax.h0", "softmax.h1", "-"};
    for (int r = 0; r < TR_ROLES - 1; ++r)
      for (int t = 0; t < TR_TASKS; ++t) {
        std::string line = std::string(names[r]) + " task " + std::to_string(t) + ":";
        bool any = false;
        for (int e = 0; e < TR_EVENTS; ++e) {
          const unsigned long long v = host[(r * TR_TASKS + t) * TR_EVENTS + e];
          if (v) { any = true; line += " e" + std::to_string(e) + "=" + std::to_string((long long)(v - t0)); }
        }
        if (any) fprintf(stderr, "[attn trace] %s\n", line.c_str());
      }
  }
  return attn_cls_merge(qkv, cls_ws, out, B, N, H, T, stream);
}

}  // namespace hh
