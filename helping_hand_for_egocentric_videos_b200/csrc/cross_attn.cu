// Query -> patch-token cross attention of the object-aware decoder (nn.MultiheadAttention core at
// model/tfm_decoder.py:438-441): Q <= kMaxQueries (32) learned queries per clip against S = T*n keys, 8 heads of 64.
//
// HBM-bound (K and V of a layer are read once: 2 * B*S*C bf16).  Flash-decode layout: the keys of one (clip, head)
// are split over `splits` CTAs x 4 warps; each warp streams its key range in blocks of 64 through a private
// shared-memory tile (cp.async, 16 B per lane) and runs S = Q K^T and O = P V on mma.sync m16n8k16 with an fp32 online
// softmax.  The queries form QB blocks of 16 rows (QB = 1 for Q <= 16, 2 for Q <= 32): each staged K/V block serves
// every query block, so the K/V bytes do not grow with Q; fragments, accumulators and softmax state are per block.
// The fp32 queries enter the tensor cores as a bf16 hi + lo pair (two MMAs), so the logits keep fp32-level accuracy in
// q.  Every warp writes an unnormalised partial (max, sum, o[64]) per query; cross_merge_kernel folds them exactly.
// The head-averaged attention map that the reference computes and discards (:271-295) is not produced.
#include "hh_internal.h"
#include "hh_ptx.cuh"

namespace hh {

namespace {

constexpr float LOG2E = 1.4426950408889634f;
constexpr int HD = 64;
constexpr int XQ = 16;          // query rows of one MMA block
constexpr int XQB = kMaxQueries / XQ;  // query blocks of the largest instantiation
static_assert(kMaxQueries % XQ == 0 && XQB == 2, "cross_attn: instantiations for QB = 1 and 2");
constexpr int XW = 4;           // warps per CTA
constexpr int XLD = 72;         // smem row stride (bf16)
constexpr int XPART = HD + 2;   // per query: m, l, o[64]
constexpr int XBLK = 64;        // keys per block

int query_blocks(int Q) { return (Q + XQ - 1) / XQ; }

// QB = 2 holds twice the query fragments and accumulators: 2 CTAs per SM instead of 3 keep it free of spills
template <int QB>
__global__ void __launch_bounds__(XW * 32, QB == 1 ? 3 : 2)
cross_attn_mma_kernel(const float* __restrict__ q, const bf16* __restrict__ K, const bf16* __restrict__ V, int ldkv,
                      float* __restrict__ part, int Q, int heads, int S, int splits, int keys_per_warp, DropCfg drop,
                      uint32_t drop_site) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  bf16* Ks = reinterpret_cast<bf16*>(smem_raw) + static_cast<size_t>(warp) * (2 * XBLK * XLD);
  bf16* Vs = Ks + XBLK * XLD;
  const int split = blockIdx.x % splits;
  const int h = (blockIdx.x / splits) % heads;
  const int b = blockIdx.x / (splits * heads);
  const int C = heads * HD;
  const int g = lane >> 2, t = lane & 3;
  const int mi = lane >> 3, lr = lane & 7;

  // ---- query fragments of block qb (rows 16 qb + g, + 8; columns 16ks + 2t + {0,1,8,9}) as bf16 hi / lo pairs
  uint32_t qh[QB][4][4], ql[QB][4][4];
#pragma unroll
  for (int qb = 0; qb < QB; ++qb) {
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int row = XQ * qb + g + (e & 1) * 8;
        const int col = ks * 16 + 2 * t + (e >> 1) * 8;
        float2 v = make_float2(0.f, 0.f);
        if (row < Q) v = *reinterpret_cast<const float2*>(q + static_cast<size_t>(b * Q + row) * C + h * HD + col);
        const __nv_bfloat162 hi = __floats2bfloat162_rn(v.x, v.y);
        const float2 hf = __bfloat1622float2(hi);
        qh[qb][ks][e] = *reinterpret_cast<const uint32_t*>(&hi);
        ql[qb][ks][e] = pack_bf16x2(v.x - hf.x, v.y - hf.y);
      }
    }
  }

  const int part_id = split * XW + warp;
  const int k_begin = part_id * keys_per_warp;
  const int k_end = min(S, k_begin + keys_per_warp);
  const bf16* Kb = K + static_cast<size_t>(b) * S * ldkv + h * HD;
  const bf16* Vb = V + static_cast<size_t>(b) * S * ldkv + h * HD;

  float m[QB][2], l[QB][2];
  float o[QB][8][4];
#pragma unroll
  for (int qb = 0; qb < QB; ++qb) {
    m[qb][0] = m[qb][1] = -INFINITY;
    l[qb][0] = l[qb][1] = 0.f;
#pragma unroll
    for (int ni = 0; ni < 8; ++ni) o[qb][ni][0] = o[qb][ni][1] = o[qb][ni][2] = o[qb][ni][3] = 0.f;
  }

  for (int kb = k_begin; kb < k_end; kb += XBLK) {
    // ---- stage 64 keys x 64 dims of K and V (zero-filled past k_end), once for all query blocks
    for (int c = lane; c < XBLK * 8; c += 32) {
      const int r = c >> 3, ch = c & 7;
      const bool valid = kb + r < k_end;
      const size_t off = static_cast<size_t>(valid ? kb + r : kb) * ldkv + ch * 8;
      cp_async_16(Ks + r * XLD + ch * 8, Kb + off, valid);
      cp_async_16(Vs + r * XLD + ch * 8, Vb + off, valid);
    }
    cp_async_commit();
    cp_async_wait<0>();
    __syncwarp();

#pragma unroll
    for (int qb = 0; qb < QB; ++qb) {
      float s[8][4];
#pragma unroll
      for (int ni = 0; ni < 8; ++ni) s[ni][0] = s[ni][1] = s[ni][2] = s[ni][3] = 0.f;
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
        for (int np = 0; np < 4; ++np) {
          uint32_t kf[4];
          ldmatrix_x4(kf, smem_u32(Ks + (np * 16 + (mi >> 1) * 8 + lr) * XLD + ks * 16 + (mi & 1) * 8));
          mma_bf16_16816(s[2 * np], qh[qb][ks], kf[0], kf[1]);
          mma_bf16_16816(s[2 * np], ql[qb][ks], kf[0], kf[1]);
          mma_bf16_16816(s[2 * np + 1], qh[qb][ks], kf[2], kf[3]);
          mma_bf16_16816(s[2 * np + 1], ql[qb][ks], kf[2], kf[3]);
        }
      }
      float mx0 = -INFINITY, mx1 = -INFINITY;
      if (kb + XBLK > k_end) {
#pragma unroll
        for (int ni = 0; ni < 8; ++ni) {
          const int key = kb + ni * 8 + 2 * t;
          if (key >= k_end) s[ni][0] = s[ni][2] = -INFINITY;
          if (key + 1 >= k_end) s[ni][1] = s[ni][3] = -INFINITY;
        }
      }
#pragma unroll
      for (int ni = 0; ni < 8; ++ni) {
        mx0 = fmaxf(mx0, fmaxf(s[ni][0], s[ni][1]));
        mx1 = fmaxf(mx1, fmaxf(s[ni][2], s[ni][3]));
      }
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
      const float mn0 = fmaxf(m[qb][0], mx0), mn1 = fmaxf(m[qb][1], mx1);  // finite: key kb is always valid
      const float ml0 = mn0 * LOG2E, ml1 = mn1 * LOG2E;
      const float c0 = fast_exp2(m[qb][0] * LOG2E - ml0), c1 = fast_exp2(m[qb][1] * LOG2E - ml1);
      m[qb][0] = mn0;
      m[qb][1] = mn1;
      l[qb][0] *= c0;
      l[qb][1] *= c1;
      const int row0 = XQ * qb + g, row1 = row0 + 8;
      uint32_t pa[4][4];
#pragma unroll
      for (int ni = 0; ni < 8; ++ni) {
        const float p0 = fast_exp2(fmaf(s[ni][0], LOG2E, -ml0)), p1 = fast_exp2(fmaf(s[ni][1], LOG2E, -ml0));
        const float p2 = fast_exp2(fmaf(s[ni][2], LOG2E, -ml1)), p3 = fast_exp2(fmaf(s[ni][3], LOG2E, -ml1));
        l[qb][0] += p0 + p1;
        l[qb][1] += p2 + p3;
        float d0 = p0, d1 = p1, d2 = p2, d3 = p3;
        if (drop.thr) {  // training: probabilities are dropped AFTER normalisation -> l keeps every key, P V only the kept
          // keys 8*ni .. 8*ni+7 of a row are one Philox block (S % 8 == 0); this thread owns lanes 2t, 2t+1 of two rows
          const int key = kb + ni * 8;
          uint32_t rb[4];
          if (row0 < Q) {
            drop_block8(drop, drop_site, ((static_cast<uint64_t>(b) * heads + h) * Q + row0) * (S >> 3) + (key >> 3), rb);
            const uint32_t w = t == 0 ? rb[0] : t == 1 ? rb[1] : t == 2 ? rb[2] : rb[3];
            if ((w & 0xFFFFu) < drop.thr) d0 = 0.f;
            if ((w >> 16) < drop.thr) d1 = 0.f;
          }
          if (row1 < Q) {
            drop_block8(drop, drop_site, ((static_cast<uint64_t>(b) * heads + h) * Q + row1) * (S >> 3) + (key >> 3), rb);
            const uint32_t w = t == 0 ? rb[0] : t == 1 ? rb[1] : t == 2 ? rb[2] : rb[3];
            if ((w & 0xFFFFu) < drop.thr) d2 = 0.f;
            if ((w >> 16) < drop.thr) d3 = 0.f;
          }
        }
        pa[ni >> 1][(ni & 1) * 2 + 0] = pack_bf16x2(d0, d1);
        pa[ni >> 1][(ni & 1) * 2 + 1] = pack_bf16x2(d2, d3);
        o[qb][ni][0] *= c0; o[qb][ni][1] *= c0; o[qb][ni][2] *= c1; o[qb][ni][3] *= c1;
      }
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
#pragma unroll
        for (int dp = 0; dp < 4; ++dp) {
          uint32_t vf[4];
          ldmatrix_x4_trans(vf, smem_u32(Vs + (kk * 16 + (mi & 1) * 8 + lr) * XLD + dp * 16 + (mi >> 1) * 8));
          mma_bf16_16816(o[qb][2 * dp], pa[kk], vf[0], vf[1]);
          mma_bf16_16816(o[qb][2 * dp + 1], pa[kk], vf[2], vf[3]);
        }
      }
    }
    __syncwarp();  // the tile is overwritten by the next block's copies
  }

  // ---- partial of this warp: [(b*heads + h)][part_id][query (pitch 16 QB)][m, l, o[64]]
  float* dst = part + ((static_cast<size_t>(b) * heads + h) * (splits * XW) + part_id) * (XQ * QB) * XPART;
#pragma unroll
  for (int qb = 0; qb < QB; ++qb) {
    float l0 = l[qb][0], l1 = l[qb][1];
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
    l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int row = XQ * qb + g + e * 8;
      if (row < Q) {
        float* pr = dst + row * XPART;
        if (t == 0) {
          pr[0] = m[qb][e];
          pr[1] = e ? l1 : l0;
        }
#pragma unroll
        for (int ni = 0; ni < 8; ++ni) {
          pr[2 + ni * 8 + 2 * t] = o[qb][ni][2 * e];
          pr[2 + ni * 8 + 2 * t + 1] = o[qb][ni][2 * e + 1];
        }
      }
    }
  }
}

// part: [(b*heads + h)][nparts][rows][XPART], rows = 16 QB of the producing instantiation
__global__ void __launch_bounds__(4 * HD)
cross_merge_kernel(const float* __restrict__ part, float* __restrict__ out, float* __restrict__ lse, int Q, int heads,
                   int nparts, int rows, float oscale) {
  const int h = blockIdx.x % heads, b = blockIdx.x / heads;
  const int d = threadIdx.x & (HD - 1);
  const int C = heads * HD;
  const float* base = part + static_cast<size_t>(blockIdx.x) * nparts * rows * XPART;
  for (int i = threadIdx.x / HD; i < Q; i += 4) {   // four query rows per pass
    float mm = -INFINITY;
    for (int s = 0; s < nparts; ++s) mm = fmaxf(mm, base[(s * rows + i) * XPART]);
    float ll = 0.f, oo = 0.f;
    for (int s = 0; s < nparts; ++s) {
      const float* pr = base + (s * rows + i) * XPART;
      const float c = (pr[0] == -INFINITY) ? 0.f : exp2f((pr[0] - mm) * LOG2E);
      ll += pr[1] * c;
      oo += pr[2 + d] * c;
    }
    out[static_cast<size_t>(b * Q + i) * C + h * HD + d] = oo * oscale / ll;
    // log-sum-exp of the row's logits, kept for cross_attn_bwd (dropout does not enter: it acts after normalisation)
    if (lse != nullptr && d == 0) lse[static_cast<size_t>(blockIdx.x) * Q + i] = mm + logf(ll);
  }
}

int cross_splits(int B, int heads, int S) {
  int splits = (6 * num_sms() + B * heads - 1) / (B * heads);  // ~2 waves of 3 CTAs per SM
  const int max_splits = (S + XW * XBLK - 1) / (XW * XBLK);
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  return splits;
}

template <int QB>
int cross_attn_launch(const float* q, const bf16* K, const bf16* V, int ldkv, float* out, int B, int Q, int heads, int S,
                      float* part, cudaStream_t stream, DropCfg drop, uint32_t drop_site, float* lse_out) {
  const int splits = cross_splits(B, heads, S);
  const int nparts = splits * XW;
  const int keys_per_warp = ((S + nparts - 1) / nparts + XBLK - 1) / XBLK * XBLK;
  const size_t smem = static_cast<size_t>(XW) * 2 * XBLK * XLD * sizeof(bf16);
  static bool configured = false;   // one flag per instantiation
  if (!configured) {
    HH_CHECK_CUDA(cudaFuncSetAttribute(cross_attn_mma_kernel<QB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>(smem)));
    configured = true;
  }
  cross_attn_mma_kernel<QB><<<B * heads * splits, XW * 32, smem, stream>>>(q, K, V, ldkv, part, Q, heads, S, splits,
                                                                          keys_per_warp, drop, drop_site);
  HH_CHECK_LAUNCH("cross_attn_mma_kernel");
  cross_merge_kernel<<<B * heads, 4 * HD, 0, stream>>>(part, out, lse_out, Q, heads, nparts, XQ * QB,
                                                   drop.thr ? drop.scale : 1.f);
  HH_CHECK_LAUNCH("cross_merge_kernel");
  return 0;
}

}  // namespace

size_t cross_attn_workspace_bytes(int B, int Q, int heads, int S) {
  return static_cast<size_t>(B) * heads * cross_splits(B, heads, S) * XW * XQ * query_blocks(Q) * XPART * sizeof(float);
}

int cross_attn(const float* q, const bf16* K, const bf16* V, int ldkv, float* out, int B, int Q, int heads, int S,
               void* workspace, cudaStream_t stream, DropCfg drop, uint32_t drop_site, float* lse_out) {
  HH_REQUIRE(drop.thr == 0 || S % 8 == 0, "cross_attn: dropout needs a multiple of 8 keys");
  HH_REQUIRE(Q >= 1 && Q <= kMaxQueries, "cross_attn: 1..32 queries supported");
  HH_REQUIRE(ldkv % 8 == 0, "cross_attn: K/V row stride must be a multiple of 8 elements");
  HH_REQUIRE((reinterpret_cast<uintptr_t>(K) & 15) == 0 && (reinterpret_cast<uintptr_t>(V) & 15) == 0 &&
                 (reinterpret_cast<uintptr_t>(q) & 7) == 0,
             "cross_attn: K/V must be 16-byte aligned, q 8-byte aligned");
  HH_REQUIRE(workspace != nullptr, "cross_attn: workspace");
  float* part = static_cast<float*>(workspace);   // sized by cross_attn_workspace_bytes(B, Q, heads, S)
  if (Q <= XQ) return cross_attn_launch<1>(q, K, V, ldkv, out, B, Q, heads, S, part, stream, drop, drop_site, lse_out);
  return cross_attn_launch<2>(q, K, V, ldkv, out, B, Q, heads, S, part, stream, drop, drop_site, lse_out);
}

}  // namespace hh
