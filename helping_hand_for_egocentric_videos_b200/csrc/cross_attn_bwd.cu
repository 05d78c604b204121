// Backward of the query -> patch-token cross attention (forward: cross_attn.cu; reference graph: nn.MultiheadAttention
// core at model/tfm_decoder.py:438-441 differentiated for run/train.py:196-203) on the warp tensor cores.
//
// Same decomposition as the forward: the keys of one (clip, head) are split over `splits` CTAs x 4 warps; each warp
// streams its key range in blocks of 32 through a private shared-memory tile (cp.async) and, per block and per 16-row
// query block (QB = 1 for Q <= 16, 2 for Q <= 32),
//
//   S  = q K^T,  dP = dO V^T          [16 queries x 32 keys]  q / dO as bf16 hi + lo pairs (fp32-accurate logits)
//   P  = exp(S - lse),  dS = P (m dP - D),  P' = m P          (m: the forward's dropout keep-multipliers, regenerated)
//   dq += dS K                        A operand = dS straight from the accumulator registers (hi + lo), B = K (trans)
//   dV  = P'^T dO,  dK = dS^T q       contraction over the QUERIES: the accumulator blocks are transposed in
//                                     registers with movmatrix and become the A operand; the QB query blocks are
//                                     accumulated into the same registers, so dV / dK rows of this key block are
//                                     complete after one pass and are written once (bf16)
//
// lse comes from the forward (cross_attn's lse_out) or is recomputed by cross_stats_kernel; D_i = dO_i . O_i is taken
// per CTA.  Every warp leaves a partial dq [16 QB x 64]; cross_dq_merge_kernel adds the partials in a fixed order (no
// atomics: dq is bit-reproducible).  The first-generation SIMT statement (decoder_bwd.cu: one thread per key, dS through
// HBM, 5 ms per c4 backward) serves the inputs this kernel does not take: q / dO that are not 8-byte aligned, dK / dV that
// are not 4-byte aligned, and dropout with a key count that is not a multiple of 8.
#include "hh_internal.h"
#include "hh_ptx.cuh"

namespace hh {

namespace {

constexpr int HD = 64;
constexpr int XQ = 16;        // query rows of one MMA block
static_assert(kMaxQueries % XQ == 0 && kMaxQueries / XQ == 2, "cross_attn_bwd: instantiations for QB = 1 and 2");
constexpr int XW = 4;         // warps per CTA
constexpr int XLD = 72;       // smem row stride (bf16): ldmatrix rows 16 bytes apart in banks
constexpr int KB = 32;        // keys per block
constexpr int QT = XQ * XLD;  // one [16 x 64] operand tile of one query block

int query_blocks(int Q) { return (Q + XQ - 1) / XQ; }

// dynamic shared memory: q hi / lo, dO hi / lo tiles of QB blocks, D and lse per query row, per-warp K / V tiles
constexpr size_t bwd_smem_bytes(int QB) {
  return 4 * QB * QT * sizeof(bf16) + 2 * XQ * QB * sizeof(float) + static_cast<size_t>(XW) * 2 * KB * XLD * sizeof(bf16);
}
static_assert(bwd_smem_bytes(1) <= 48 * 1024, "QB = 1 runs without the shared-memory opt-in");
static_assert(bwd_smem_bytes(kMaxQueries / XQ) <= 227 * 1024, "shared memory per block");

__device__ __forceinline__ uint32_t movmatrix_trans(uint32_t a) {
  uint32_t d;
  asm volatile("movmatrix.sync.aligned.m8n8.trans.b16 %0, %1;" : "=r"(d) : "r"(a));
  return d;
}

template <int QB>
__global__ void __launch_bounds__(XW * 32)
cross_bwd_mma_kernel(const float* __restrict__ q, const bf16* __restrict__ K, const bf16* __restrict__ V, int ldkv,
                     const float* __restrict__ O, const float* __restrict__ dO, const float* __restrict__ lse,
                     bf16* __restrict__ dK, bf16* __restrict__ dV, int lddkv, float* __restrict__ dq_part, int Q, int heads,
                     int S, int splits, int keys_per_warp, DropCfg drop, uint32_t drop_site) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  constexpr int QR = XQ * QB;                      // query rows of the tiles
  bf16* Qh = reinterpret_cast<bf16*>(smem_raw);   // q hi, q lo, dO hi, dO lo: [16 QB][XLD] each, shared by the 4 warps
  bf16* Ql = Qh + QB * QT;
  bf16* Gh = Ql + QB * QT;
  bf16* Gl = Gh + QB * QT;
  float* Dsm = reinterpret_cast<float*>(Gl + QB * QT);  // [16 QB] D_i, [16 QB] lse_i
  float* Lsm = Dsm + QR;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  bf16* Ks = reinterpret_cast<bf16*>(Lsm + QR) + static_cast<size_t>(warp) * (2 * KB * XLD);
  bf16* Vs = Ks + KB * XLD;
  const int split = blockIdx.x % splits;
  const int h = (blockIdx.x / splits) % heads;
  const int b = blockIdx.x / (splits * heads);
  const int C = heads * HD;
  const int g = lane >> 2, t = lane & 3;
  const int mi = lane >> 3, lr = lane & 7;

  // ---- CTA prologue: q / dO rows as bf16 hi + lo tiles (rows >= Q zero), D_i, lse_i (rows >= Q: +inf -> P = 0)
  for (int e = threadIdx.x; e < QR * (HD / 2); e += XW * 32) {
    const int row = e / (HD / 2), col = (e % (HD / 2)) * 2;
    float2 qv = make_float2(0.f, 0.f), gv = make_float2(0.f, 0.f);
    if (row < Q) {
      qv = *reinterpret_cast<const float2*>(q + static_cast<size_t>(b * Q + row) * C + h * HD + col);
      gv = *reinterpret_cast<const float2*>(dO + static_cast<size_t>(b * Q + row) * C + h * HD + col);
    }
    const __nv_bfloat162 qh2 = __floats2bfloat162_rn(qv.x, qv.y), gh2 = __floats2bfloat162_rn(gv.x, gv.y);
    const float2 qf = __bfloat1622float2(qh2), gf = __bfloat1622float2(gh2);
    *reinterpret_cast<__nv_bfloat162*>(Qh + row * XLD + col) = qh2;
    *reinterpret_cast<__nv_bfloat162*>(Ql + row * XLD + col) = __floats2bfloat162_rn(qv.x - qf.x, qv.y - qf.y);
    *reinterpret_cast<__nv_bfloat162*>(Gh + row * XLD + col) = gh2;
    *reinterpret_cast<__nv_bfloat162*>(Gl + row * XLD + col) = __floats2bfloat162_rn(gv.x - gf.x, gv.y - gf.y);
  }
  for (int i = warp; i < QR; i += XW) {
    float tsum = 0.f;
    if (i < Q) {
      const float* gp = dO + static_cast<size_t>(b * Q + i) * C + h * HD;
      const float* op = O + static_cast<size_t>(b * Q + i) * C + h * HD;
      tsum = gp[lane] * op[lane] + gp[lane + 32] * op[lane + 32];
    }
    tsum = warp_sum(tsum);
    if (lane == 0) {
      Dsm[i] = tsum;
      Lsm[i] = i < Q ? lse[(static_cast<size_t>(b) * heads + h) * Q + i] : INFINITY;
    }
  }
  __syncthreads();
  float D[QB][2], L[QB][2];
#pragma unroll
  for (int qb = 0; qb < QB; ++qb) {
    D[qb][0] = Dsm[XQ * qb + g];
    D[qb][1] = Dsm[XQ * qb + g + 8];
    L[qb][0] = Lsm[XQ * qb + g];
    L[qb][1] = Lsm[XQ * qb + g + 8];
  }

  const int part_id = split * XW + warp;
  const int k_begin = part_id * keys_per_warp;
  const int k_end = min(S, k_begin + keys_per_warp);
  const bf16* Kb = K + static_cast<size_t>(b) * S * ldkv + h * HD;
  const bf16* Vb = V + static_cast<size_t>(b) * S * ldkv + h * HD;
  bf16* dKb = dK + static_cast<size_t>(b) * S * lddkv + h * HD;
  bf16* dVb = dV + static_cast<size_t>(b) * S * lddkv + h * HD;

  float dqa[QB][8][4];
#pragma unroll
  for (int qb = 0; qb < QB; ++qb)
#pragma unroll
    for (int ni = 0; ni < 8; ++ni) dqa[qb][ni][0] = dqa[qb][ni][1] = dqa[qb][ni][2] = dqa[qb][ni][3] = 0.f;

  for (int kb = k_begin; kb < k_end; kb += KB) {
    // ---- stage 32 keys x 64 dims of K and V (zero-filled past k_end)
    for (int c = lane; c < KB * 8; c += 32) {
      const int r = c >> 3, ch = c & 7;
      const bool valid = kb + r < k_end;
      const size_t off = static_cast<size_t>(valid ? kb + r : kb) * ldkv + ch * 8;
      cp_async_16(Ks + r * XLD + ch * 8, Kb + off, valid);
      cp_async_16(Vs + r * XLD + ch * 8, Vb + off, valid);
    }
    cp_async_commit();
    cp_async_wait<0>();
    __syncwarp();

    // ---- per query block: S, dP, P, dS, P', dq; the transposed dS / P' blocks wait for dK / dV below
    uint32_t ds_hi[QB][4][2], pm_hi[QB][4][2];
#pragma unroll
    for (int qb = 0; qb < QB; ++qb) {
      // ---- S = q K^T and dP = dO V^T: [16 x 32], n-tile ni = keys 8 ni .. 8 ni + 7
      float s[4][4], dp[4][4];
#pragma unroll
      for (int ni = 0; ni < 4; ++ni) {
        s[ni][0] = s[ni][1] = s[ni][2] = s[ni][3] = 0.f;
        dp[ni][0] = dp[ni][1] = dp[ni][2] = dp[ni][3] = 0.f;
      }
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        uint32_t ah[4], al[4], bh[4], bl[4];
        const int aoff = ((mi & 1) * 8 + lr) * XLD + ks * 16 + (mi >> 1) * 8;
        ldmatrix_x4(ah, smem_u32(Qh + qb * QT + aoff));
        ldmatrix_x4(al, smem_u32(Ql + qb * QT + aoff));
        ldmatrix_x4(bh, smem_u32(Gh + qb * QT + aoff));
        ldmatrix_x4(bl, smem_u32(Gl + qb * QT + aoff));
#pragma unroll
        for (int np = 0; np < 2; ++np) {
          uint32_t kf[4], vf[4];
          const int boff = (np * 16 + (mi >> 1) * 8 + lr) * XLD + ks * 16 + (mi & 1) * 8;
          ldmatrix_x4(kf, smem_u32(Ks + boff));
          ldmatrix_x4(vf, smem_u32(Vs + boff));
          mma_bf16_16816(s[2 * np], ah, kf[0], kf[1]);
          mma_bf16_16816(s[2 * np], al, kf[0], kf[1]);
          mma_bf16_16816(s[2 * np + 1], ah, kf[2], kf[3]);
          mma_bf16_16816(s[2 * np + 1], al, kf[2], kf[3]);
          mma_bf16_16816(dp[2 * np], bh, vf[0], vf[1]);
          mma_bf16_16816(dp[2 * np], bl, vf[0], vf[1]);
          mma_bf16_16816(dp[2 * np + 1], bh, vf[2], vf[3]);
          mma_bf16_16816(dp[2 * np + 1], bl, vf[2], vf[3]);
        }
      }

      // ---- P, dS, P' (this thread: rows 16 qb + g / + 8, keys 8 ni + 2t, + 1); packed bf16 blocks for the MMAs below
      uint32_t ds_lo[4][2];
      const int row0 = XQ * qb + g, row1 = row0 + 8;
#pragma unroll
      for (int ni = 0; ni < 4; ++ni) {
        const int key = kb + ni * 8 + 2 * t;
        const bool v0 = key < k_end, v1 = key + 1 < k_end;
        float p[4];
        p[0] = v0 ? __expf(s[ni][0] - L[qb][0]) : 0.f;
        p[1] = v1 ? __expf(s[ni][1] - L[qb][0]) : 0.f;
        p[2] = v0 ? __expf(s[ni][2] - L[qb][1]) : 0.f;
        p[3] = v1 ? __expf(s[ni][3] - L[qb][1]) : 0.f;
        float m[4] = {1.f, 1.f, 1.f, 1.f};
        if (drop.thr) {  // keys 8 ni .. 8 ni + 7 of a row are one Philox block (S % 8 == 0), as in the forward
          uint32_t rb[4];
          if (row0 < Q) {
            drop_block8(drop, drop_site, ((static_cast<uint64_t>(b) * heads + h) * Q + row0) * (S >> 3) + ((kb + ni * 8) >> 3), rb);
            const uint32_t w = t == 0 ? rb[0] : t == 1 ? rb[1] : t == 2 ? rb[2] : rb[3];
            m[0] = (w & 0xFFFFu) < drop.thr ? 0.f : drop.scale;
            m[1] = (w >> 16) < drop.thr ? 0.f : drop.scale;
          }
          if (row1 < Q) {
            drop_block8(drop, drop_site, ((static_cast<uint64_t>(b) * heads + h) * Q + row1) * (S >> 3) + ((kb + ni * 8) >> 3), rb);
            const uint32_t w = t == 0 ? rb[0] : t == 1 ? rb[1] : t == 2 ? rb[2] : rb[3];
            m[2] = (w & 0xFFFFu) < drop.thr ? 0.f : drop.scale;
            m[3] = (w >> 16) < drop.thr ? 0.f : drop.scale;
          }
        }
        float dsv[4];
        dsv[0] = p[0] * (m[0] * dp[ni][0] - D[qb][0]);
        dsv[1] = p[1] * (m[1] * dp[ni][1] - D[qb][0]);
        dsv[2] = p[2] * (m[2] * dp[ni][2] - D[qb][1]);
        dsv[3] = p[3] * (m[3] * dp[ni][3] - D[qb][1]);
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const __nv_bfloat162 hi = __floats2bfloat162_rn(dsv[2 * e], dsv[2 * e + 1]);
          const float2 hf = __bfloat1622float2(hi);
          ds_hi[qb][ni][e] = *reinterpret_cast<const uint32_t*>(&hi);
          ds_lo[ni][e] = pack_bf16x2(dsv[2 * e] - hf.x, dsv[2 * e + 1] - hf.y);
          pm_hi[qb][ni][e] = pack_bf16x2(p[2 * e] * m[2 * e], p[2 * e + 1] * m[2 * e + 1]);
        }
      }

      // ---- dq += dS K: A = dS from the registers (rows = queries, k = 16 keys), B = K[key][d] read transposed
#pragma unroll
      for (int kk = 0; kk < 2; ++kk) {
        const uint32_t ahi[4] = {ds_hi[qb][2 * kk][0], ds_hi[qb][2 * kk][1], ds_hi[qb][2 * kk + 1][0], ds_hi[qb][2 * kk + 1][1]};
        const uint32_t alo[4] = {ds_lo[2 * kk][0], ds_lo[2 * kk][1], ds_lo[2 * kk + 1][0], ds_lo[2 * kk + 1][1]};
#pragma unroll
        for (int dpi = 0; dpi < 4; ++dpi) {
          uint32_t kf[4];
          ldmatrix_x4_trans(kf, smem_u32(Ks + (kk * 16 + (mi & 1) * 8 + lr) * XLD + dpi * 16 + (mi >> 1) * 8));
          mma_bf16_16816(dqa[qb][2 * dpi], ahi, kf[0], kf[1]);
          mma_bf16_16816(dqa[qb][2 * dpi], alo, kf[0], kf[1]);
          mma_bf16_16816(dqa[qb][2 * dpi + 1], ahi, kf[2], kf[3]);
          mma_bf16_16816(dqa[qb][2 * dpi + 1], alo, kf[2], kf[3]);
        }
      }
    }

    // ---- dV = P'^T dO, dK = dS^T q for the two 16-key groups: the [queries x keys] blocks transposed in registers,
    // the QB query blocks accumulated in the same registers (one k16 MMA each) before the single bf16 write
#pragma unroll
    for (int kg = 0; kg < 2; ++kg) {
      uint32_t ap[QB][4], ad[QB][4];
#pragma unroll
      for (int qb = 0; qb < QB; ++qb) {
        ap[qb][0] = movmatrix_trans(pm_hi[qb][2 * kg][0]);     // keys 0-7 of the group x queries 0-7 of the block
        ap[qb][1] = movmatrix_trans(pm_hi[qb][2 * kg + 1][0]); // keys 8-15 x queries 0-7
        ap[qb][2] = movmatrix_trans(pm_hi[qb][2 * kg][1]);     // keys 0-7 x queries 8-15
        ap[qb][3] = movmatrix_trans(pm_hi[qb][2 * kg + 1][1]);
        ad[qb][0] = movmatrix_trans(ds_hi[qb][2 * kg][0]);
        ad[qb][1] = movmatrix_trans(ds_hi[qb][2 * kg + 1][0]);
        ad[qb][2] = movmatrix_trans(ds_hi[qb][2 * kg][1]);
        ad[qb][3] = movmatrix_trans(ds_hi[qb][2 * kg + 1][1]);
      }
      const int key0 = kb + kg * 16 + g, key1 = key0 + 8;
#pragma unroll
      for (int dpi = 0; dpi < 4; ++dpi) {
        float dv0[4] = {0.f, 0.f, 0.f, 0.f}, dv1[4] = {0.f, 0.f, 0.f, 0.f};
        float dk0[4] = {0.f, 0.f, 0.f, 0.f}, dk1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int qb = 0; qb < QB; ++qb) {
          uint32_t gf[4], qf[4];
          const int boff = qb * QT + ((mi & 1) * 8 + lr) * XLD + dpi * 16 + (mi >> 1) * 8;
          ldmatrix_x4_trans(gf, smem_u32(Gh + boff));
          ldmatrix_x4_trans(qf, smem_u32(Qh + boff));
          mma_bf16_16816(dv0, ap[qb], gf[0], gf[1]);
          mma_bf16_16816(dv1, ap[qb], gf[2], gf[3]);
          mma_bf16_16816(dk0, ad[qb], qf[0], qf[1]);
          mma_bf16_16816(dk1, ad[qb], qf[2], qf[3]);
        }
        const int d0 = dpi * 16 + 2 * t;
        if (key0 < k_end) {
          *reinterpret_cast<uint32_t*>(dVb + static_cast<size_t>(key0) * lddkv + d0) = pack_bf16x2(dv0[0], dv0[1]);
          *reinterpret_cast<uint32_t*>(dVb + static_cast<size_t>(key0) * lddkv + d0 + 8) = pack_bf16x2(dv1[0], dv1[1]);
          *reinterpret_cast<uint32_t*>(dKb + static_cast<size_t>(key0) * lddkv + d0) = pack_bf16x2(dk0[0], dk0[1]);
          *reinterpret_cast<uint32_t*>(dKb + static_cast<size_t>(key0) * lddkv + d0 + 8) = pack_bf16x2(dk1[0], dk1[1]);
        }
        if (key1 < k_end) {
          *reinterpret_cast<uint32_t*>(dVb + static_cast<size_t>(key1) * lddkv + d0) = pack_bf16x2(dv0[2], dv0[3]);
          *reinterpret_cast<uint32_t*>(dVb + static_cast<size_t>(key1) * lddkv + d0 + 8) = pack_bf16x2(dv1[2], dv1[3]);
          *reinterpret_cast<uint32_t*>(dKb + static_cast<size_t>(key1) * lddkv + d0) = pack_bf16x2(dk0[2], dk0[3]);
          *reinterpret_cast<uint32_t*>(dKb + static_cast<size_t>(key1) * lddkv + d0 + 8) = pack_bf16x2(dk1[2], dk1[3]);
        }
      }
    }
    __syncwarp();  // the tile is overwritten by the next block's copies
  }

  // ---- partial dq of this warp: [(b*heads + h)][part_id][query (pitch 16 QB)][64]
  float* dst = dq_part + ((static_cast<size_t>(b) * heads + h) * (splits * XW) + part_id) * QR * HD;
#pragma unroll
  for (int qb = 0; qb < QB; ++qb) {
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int row = XQ * qb + g + e * 8;
      if (row < Q) {
#pragma unroll
        for (int ni = 0; ni < 8; ++ni)
          *reinterpret_cast<float2*>(dst + row * HD + ni * 8 + 2 * t) =
              make_float2(dqa[qb][ni][2 * e], dqa[qb][ni][2 * e + 1]);
      }
    }
  }
}

__global__ void __launch_bounds__(4 * HD)
cross_dq_merge_kernel(const float* __restrict__ part, float* __restrict__ dq, int Q, int heads, int nparts, int rows) {
  const int h = blockIdx.x % heads, b = blockIdx.x / heads;
  const int d = threadIdx.x & (HD - 1);
  const int C = heads * HD;
  const float* base = part + static_cast<size_t>(blockIdx.x) * nparts * rows * HD;   // rows = 16 QB
  for (int i = threadIdx.x / HD; i < Q; i += 4) {   // four query rows per pass
    float t = 0.f;
    for (int s = 0; s < nparts; ++s) t += base[(s * rows + i) * HD + d];
    dq[static_cast<size_t>(b * Q + i) * C + h * HD + d] = t;
  }
}

int bwd_splits(int B, int heads, int S) {
  int splits = (4 * num_sms() + B * heads - 1) / (B * heads);
  const int max_splits = (S + XW * KB - 1) / (XW * KB);
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  return splits;
}

template <int QB>
int cross_bwd_launch(const float* q, const bf16* K, const bf16* V, int ldkv, const float* O, const float* dO, const float* lse,
                     float* dq, bf16* dK, bf16* dV, int lddkv, float* part, int B, int Q, int heads, int S, cudaStream_t s,
                     DropCfg drop, uint32_t drop_site) {
  const int splits = bwd_splits(B, heads, S);
  const int nparts = splits * XW;
  const int keys_per_warp = ((S + nparts - 1) / nparts + KB - 1) / KB * KB;
  constexpr size_t smem = bwd_smem_bytes(QB);
  if (smem > 48 * 1024) {
    static bool configured = false;   // one flag per instantiation
    if (!configured) {
      HH_CHECK_CUDA(cudaFuncSetAttribute(cross_bwd_mma_kernel<QB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         static_cast<int>(smem)));
      configured = true;
    }
  }
  cross_bwd_mma_kernel<QB><<<B * heads * splits, XW * 32, smem, s>>>(q, K, V, ldkv, O, dO, lse, dK, dV, lddkv, part, Q, heads,
                                                                     S, splits, keys_per_warp, drop, drop_site);
  HH_CHECK_LAUNCH("cross_bwd_mma_kernel");
  cross_dq_merge_kernel<<<B * heads, 4 * HD, 0, s>>>(part, dq, Q, heads, nparts, XQ * QB);
  HH_CHECK_LAUNCH("cross_dq_merge_kernel");
  return 0;
}

}  // namespace

size_t cross_attn_bwd_workspace_bytes(int B, int Q, int heads, int S) {
  const size_t simt = cross_attn_bwd_simt_workspace_bytes(B, Q, heads, S);
  const size_t mma = static_cast<size_t>(B) * heads * Q * sizeof(float) +
                     static_cast<size_t>(B) * heads * bwd_splits(B, heads, S) * XW * XQ * query_blocks(Q) * HD * sizeof(float);
  return simt > mma ? simt : mma;
}

int cross_attn_bwd(const float* q, const bf16* K, const bf16* V, int ldkv, const float* O, const float* dO, float* dq,
                   bf16* dK, bf16* dV, int lddkv, int B, int Q, int heads, int S, void* workspace, cudaStream_t s,
                   DropCfg drop, uint32_t drop_site, const float* lse_saved) {
  HH_REQUIRE(B > 0 && Q >= 1 && Q <= kMaxQueries && heads > 0 && S > 0, "cross_attn_bwd: 1..32 queries");
  HH_REQUIRE(q && K && V && O && dO && dq && dK && dV && workspace, "cross_attn_bwd: null buffer");
  HH_REQUIRE(ldkv % 8 == 0 && lddkv % 2 == 0, "cross_attn_bwd: row pitch");
  const bool aligned = (reinterpret_cast<uintptr_t>(K) & 15) == 0 && (reinterpret_cast<uintptr_t>(V) & 15) == 0 &&
                       (reinterpret_cast<uintptr_t>(q) & 7) == 0 && (reinterpret_cast<uintptr_t>(dO) & 7) == 0 &&
                       (reinterpret_cast<uintptr_t>(dK) & 3) == 0 && (reinterpret_cast<uintptr_t>(dV) & 3) == 0;
  if (!aligned || (drop.thr != 0 && S % 8 != 0))
    return cross_attn_bwd_simt(q, K, V, ldkv, O, dO, dq, dK, dV, lddkv, B, Q, heads, S, workspace, s, drop, drop_site, lse_saved);
  float* lse_ws = static_cast<float*>(workspace);
  float* part = lse_ws + static_cast<size_t>(B) * heads * Q;
  const float* lse = lse_saved;
  if (lse == nullptr) {
    if (int rc = cross_lse(q, K, ldkv, lse_ws, B, Q, heads, S, s)) return rc;
    lse = lse_ws;
  }
  if (Q <= XQ)
    return cross_bwd_launch<1>(q, K, V, ldkv, O, dO, lse, dq, dK, dV, lddkv, part, B, Q, heads, S, s, drop, drop_site);
  return cross_bwd_launch<2>(q, K, V, ldkv, O, dO, lse, dq, dK, dV, lddkv, part, B, Q, heads, S, s, drop, drop_site);
}

}  // namespace hh
