// Temporal attention for T <= 16 (attn_time in attn_time.cu): patch query (f,p) attends {CLS key} U {(f',p) : f'} --
// T+1 <= 17 keys of 64 dims, 16 queries.  HBM-bound (q,k,v read once, o written once).  One warp owns one head of one clip
// and walks a chunk of patch positions; per position it runs the 16x24x64 and 16x64x32 products on the legacy
// tensor-core path (mma.sync m16n8k16, fp32 accumulate) with an fp32 softmax in registers.  The 8 warps of a CTA cover 8
// adjacent heads, so every global row access of the CTA is a 1 KB contiguous span.  The CLS *query* rides along as a
// second 16-row MMA block whose only live row is q_cls: each warp keeps a running (max, sum, o[64]) over the keys it sees
// and writes ONE partial per (clip, head, patch-chunk) for attn_cls_merge.
//   * per-warp shared-memory tiles are 128-byte rows with an XOR swizzle instead of padded rows, and the key / value /
//     query slots that are constant (CLS row) or always zero are single shared rows addressed per lane by ldmatrix,
//     so a warp needs 12.5 KB and its loads can be DOUBLE-BUFFERED: the 3*T row segments of patch position p+1 are in
//     flight (cp.async) while position p is computed -> twice the bytes in flight per SM for this HBM-bound kernel.
//   * the frame count is a template parameter for T = 4 / 8 / 16 (every configuration the reference runs): the copy
//     loops are fully unrolled over per-lane base pointers + warp-uniform offsets, so a 16-byte cp.async costs ~2
//     instructions instead of the ~60 of the runtime-T index arithmetic (integer division by T, swizzle, 64-bit
//     address) that made the first version issue-bound at 46 % of HBM bandwidth. TT = 0 runs the runtime-T loops for
//     every other T.
#include "hh_internal.h"
#include "hh_ptx.cuh"

namespace hh {

namespace {

constexpr int HD = 64;
constexpr float LOG2E = 1.4426950408889634f;
constexpr int TW = 8;                 // warps (= adjacent heads) per CTA
constexpr int BUF_ROWS = 48;          // 16 q + 16 k + 16 v frame rows
constexpr int ROW_QCLS = 96, ROW_KCLS = 97, ROW_VCLS = 98, ROW_ZERO = 99;
constexpr int WARP_ROWS = 100;
constexpr int WARP_BYTES = WARP_ROWS * 128;

__device__ __forceinline__ uint32_t sw_addr(uint32_t base, int row, int chunk) {
  return base + static_cast<uint32_t>(row * 128 + ((chunk ^ (row & 7)) << 4));
}
__device__ __forceinline__ void cp16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}

template <int TT>
__global__ void __launch_bounds__(TW * 32, 2)
attn_time_v2_kernel(const bf16* __restrict__ qkv, bf16* __restrict__ out, float* __restrict__ cls_part, int Trt, int n,
                    int H, int pchunk, int nchunks) {
  const int T = TT ? TT : Trt;
  extern __shared__ __align__(128) uint8_t smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t base = smem_u32(smem_raw) + static_cast<uint32_t>(warp * WARP_BYTES);

  const int D = H * HD;
  const int N = 1 + T * n;
  const int hgroups = (H + TW - 1) / TW;
  const int chunk = blockIdx.x % nchunks;
  const int hg = (blockIdx.x / nchunks) % hgroups;
  // last clips first: their q/k/v rows were written last by the QKV GEMM and are still in L2 (see rows.cu)
  const int b = static_cast<int>(gridDim.x) / (nchunks * hgroups) - 1 - static_cast<int>(blockIdx.x) / (nchunks * hgroups);
  const int h = hg * TW + warp;
  if (h >= H) return;  // whole warp; no block-level barriers below
  const size_t ld = static_cast<size_t>(3) * D;
  const bf16* clip = qkv + static_cast<size_t>(b) * N * ld + h * HD;

  // ---- zero the private tile once, then the per-warp constants: q, k, v of the CLS token
  for (int i = lane; i < WARP_BYTES / 16; i += 32)
    asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(base + i * 16), "r"(0u) : "memory");
  __syncwarp();
  if (lane < 24) {
    const int which = lane >> 3, ch = lane & 7;  // 0: q_cls, 1: k_cls, 2: v_cls
    cp16(sw_addr(base, ROW_QCLS + which, ch), clip + which * D + ch * 8);
  }
  cp_async_commit();

  const int g = lane >> 2, t = lane & 3;
  const int mi = lane >> 3, lr = lane & 7;
  const int nkeys = T + 1;

  // ---- per-lane ldmatrix row selectors (row index relative to the buffer, or an absolute constant row if >= 96)
  // Q block 0: frames (mi&1)*8 + lr ; block 1: row 16 = q_cls, rest zero
  const int q0_row = (mi & 1) * 8 + lr;
  const int q1_row = ((mi & 1) == 0 && lr == 0) ? ROW_QCLS : ROW_ZERO;
  // K n-tiles 0,1: key = (mi>>1)*8 + lr ; key 0 = CLS, key j = frame j-1
  const int k01_key = (mi >> 1) * 8 + lr;
  const int k01_row = (k01_key == 0) ? ROW_KCLS : 16 + k01_key - 1;
  // K n-tile 2: key = 16 + lr ; key 16 = frame 15, rest zero
  const int k2_row = (lr == 0) ? 16 + 15 : ROW_ZERO;
  // V k-step 0: key = (mi&1)*8 + lr ; k-step 1: key = 16 + (mi&1)*8 + lr
  const int v0_key = (mi & 1) * 8 + lr;
  const int v0_row = (v0_key == 0) ? ROW_VCLS : 32 + v0_key - 1;
  const int v1_row = ((mi & 1) == 0 && lr == 0) ? 32 + 15 : ROW_ZERO;
  auto row_abs = [](int r, int buf) { return r >= 96 ? r : buf * BUF_ROWS + r; };

  float cm = -INFINITY, cl = 0.f;
  float co[8][4];
#pragma unroll
  for (int ni = 0; ni < 8; ++ni) co[ni][0] = co[ni][1] = co[ni][2] = co[ni][3] = 0.f;

  const int p_begin = chunk * pchunk;
  const int p_end = min(n, p_begin + pchunk);

  // fast path (TT % 4 == 0): lane -> (frame row lrow + 4i, 16-byte chunk lch); row & 7 = lrow + 4 * (i & 1)
  const int lrow = lane >> 3, lch = lane & 7;
  const bf16* ld_lane = clip + (1 + static_cast<size_t>(lrow) * n) * ld + lch * 8;
  const size_t ld_step4 = static_cast<size_t>(4) * n * ld;          // four frames further
  const uint32_t sm_lane0 = base + lrow * 128 + ((lch ^ lrow) << 4);        // rows lrow + 8j
  const uint32_t sm_lane1 = base + (lrow + 4) * 128 + ((lch ^ (lrow + 4)) << 4);  // rows lrow + 4 + 8j
  bf16* st_lane = out + (static_cast<size_t>(b) * N + 1 + static_cast<size_t>(lrow) * n) * D + h * HD + lch * 8;
  const size_t st_step4 = static_cast<size_t>(4) * n * D;

  auto issue_loads = [&](int buf, int p) {
    if constexpr (TT != 0) {
      const bf16* src = ld_lane + static_cast<size_t>(p) * ld;
      const uint32_t boff = buf * (BUF_ROWS * 128);
#pragma unroll
      for (int i = 0; i < 3 * TT / 4; ++i) {
        const int which = (4 * i) / TT, f4 = ((4 * i) % TT) / 4;   // compile-time after unrolling
        const int row = which * 16 + 4 * f4;                       // + lrow, folded into sm_lane*
        const uint32_t dst = ((f4 & 1) ? sm_lane1 + (row - 4) * 128 : sm_lane0 + row * 128) + boff;
        cp16(dst, src + f4 * ld_step4 + which * D);
      }
    } else {
      for (int c = lane; c < 3 * T * 8; c += 32) {
        const int ch = c & 7;
        const int r = c >> 3;
        const int which = r / T, f = r - which * T;
        const bf16* src = clip + (1 + static_cast<size_t>(f) * n + p) * ld + which * D + ch * 8;
        cp16(sw_addr(base, buf * BUF_ROWS + which * 16 + f, ch), src);
      }
    }
    cp_async_commit();
  };

  issue_loads(0, p_begin);
  int it = 0;
  for (int p = p_begin; p < p_end; ++p, ++it) {
    const int buf = it & 1;
    if (p + 1 < p_end) {
      issue_loads(buf ^ 1, p + 1);   // prefetch the next position while this one is computed
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncwarp();

    // ---- S = Q K^T for both 16-row blocks (block 1: only row 16 = q_cls is live)
    float s[2][3][4];
#pragma unroll
    for (int mb = 0; mb < 2; ++mb)
#pragma unroll
      for (int ni = 0; ni < 3; ++ni) s[mb][ni][0] = s[mb][ni][1] = s[mb][ni][2] = s[mb][ni][3] = 0.f;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      uint32_t k01[4], k2[4], qf[4];
      ldmatrix_x4(k01, sw_addr(base, row_abs(k01_row, buf), ks * 2 + (mi & 1)));
      ldmatrix_x4(k2, sw_addr(base, row_abs(k2_row, buf), ks * 2 + (mi & 1)));
      ldmatrix_x4(qf, sw_addr(base, row_abs(q0_row, buf), ks * 2 + (mi >> 1)));
      mma_bf16_16816(s[0][0], qf, k01[0], k01[1]);
      mma_bf16_16816(s[0][1], qf, k01[2], k01[3]);
      mma_bf16_16816(s[0][2], qf, k2[0], k2[1]);
      ldmatrix_x4(qf, sw_addr(base, q1_row, ks * 2 + (mi >> 1)));
      mma_bf16_16816(s[1][0], qf, k01[0], k01[1]);
      mma_bf16_16816(s[1][1], qf, k01[2], k01[3]);
      mma_bf16_16816(s[1][2], qf, k2[0], k2[1]);
    }

    // ---- patch queries: softmax over the nkeys valid slots
    float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
    for (int ni = 0; ni < 3; ++ni) {
      const int key = ni * 8 + 2 * t;
      if (key >= nkeys) s[0][ni][0] = s[0][ni][2] = -INFINITY;
      if (key + 1 >= nkeys) s[0][ni][1] = s[0][ni][3] = -INFINITY;
      mx0 = fmaxf(mx0, fmaxf(s[0][ni][0], s[0][ni][1]));
      mx1 = fmaxf(mx1, fmaxf(s[0][ni][2], s[0][ni][3]));
    }
    mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
    mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
    mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
    mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
    float l0 = 0.f, l1 = 0.f;
    uint32_t pa[2][4];
    const float ml0 = mx0 * LOG2E, ml1 = mx1 * LOG2E;
#pragma unroll
    for (int ni = 0; ni < 3; ++ni) {
      const float p0 = fast_exp2(fmaf(s[0][ni][0], LOG2E, -ml0)), p1 = fast_exp2(fmaf(s[0][ni][1], LOG2E, -ml0));
      const float p2 = fast_exp2(fmaf(s[0][ni][2], LOG2E, -ml1)), p3 = fast_exp2(fmaf(s[0][ni][3], LOG2E, -ml1));
      l0 += p0 + p1;
      l1 += p2 + p3;
      pa[ni >> 1][(ni & 1) * 2 + 0] = pack_bf16x2(p0, p1);
      pa[ni >> 1][(ni & 1) * 2 + 1] = pack_bf16x2(p2, p3);
    }
    pa[1][2] = pa[1][3] = 0u;
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
    l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 2);

    // ---- CLS query (row g of block 1): keys 1..T of this position join its running softmax
    float cmx = -INFINITY;
#pragma unroll
    for (int ni = 0; ni < 3; ++ni) {
      const int key = ni * 8 + 2 * t;
      if (key >= nkeys || key == 0) s[1][ni][0] = -INFINITY;
      if (key + 1 >= nkeys) s[1][ni][1] = -INFINITY;
      cmx = fmaxf(cmx, fmaxf(s[1][ni][0], s[1][ni][1]));
    }
    cmx = fmaxf(cmx, __shfl_xor_sync(0xffffffffu, cmx, 1));
    cmx = fmaxf(cmx, __shfl_xor_sync(0xffffffffu, cmx, 2));
    const float cmn = fmaxf(cm, cmx);  // finite: T >= 1 gives at least one valid key
    const float ccorr = fast_exp2((cm - cmn) * LOG2E);
    cm = cmn;
    cl *= ccorr;
    uint32_t pc[2][4];
#pragma unroll
    for (int ni = 0; ni < 3; ++ni) {
      const float p0 = fast_exp2(fmaf(s[1][ni][0], LOG2E, -cmn * LOG2E)), p1 = fast_exp2(fmaf(s[1][ni][1], LOG2E, -cmn * LOG2E));
      cl += p0 + p1;
      pc[ni >> 1][(ni & 1) * 2 + 0] = pack_bf16x2(p0, p1);
      pc[ni >> 1][(ni & 1) * 2 + 1] = 0u;
    }
    pc[1][2] = pc[1][3] = 0u;
#pragma unroll
    for (int ni = 0; ni < 8; ++ni) {
      co[ni][0] *= ccorr;
      co[ni][1] *= ccorr;
    }

    float o[8][4];
#pragma unroll
    for (int ni = 0; ni < 8; ++ni) o[ni][0] = o[ni][1] = o[ni][2] = o[ni][3] = 0.f;
#pragma unroll
    for (int dp = 0; dp < 4; ++dp) {
      uint32_t vf[4];
      ldmatrix_x4_trans(vf, sw_addr(base, row_abs(v0_row, buf), dp * 2 + (mi >> 1)));
      mma_bf16_16816(o[2 * dp], pa[0], vf[0], vf[1]);
      mma_bf16_16816(o[2 * dp + 1], pa[0], vf[2], vf[3]);
      mma_bf16_16816(co[2 * dp], pc[0], vf[0], vf[1]);
      mma_bf16_16816(co[2 * dp + 1], pc[0], vf[2], vf[3]);
      ldmatrix_x4_trans(vf, sw_addr(base, row_abs(v1_row, buf), dp * 2 + (mi >> 1)));
      mma_bf16_16816(o[2 * dp], pa[1], vf[0], vf[1]);
      mma_bf16_16816(o[2 * dp + 1], pa[1], vf[2], vf[3]);
      mma_bf16_16816(co[2 * dp], pc[1], vf[0], vf[1]);
      mma_bf16_16816(co[2 * dp + 1], pc[1], vf[2], vf[3]);
    }

    // ---- stage the 16x64 result over this buffer's (consumed) query rows, then 16-byte coalesced row stores
    const float i0 = 1.f / l0, i1 = 1.f / l1;
    __syncwarp();
    const int qb = buf * BUF_ROWS;
#pragma unroll
    for (int ni = 0; ni < 8; ++ni) {
      const uint32_t a0 = sw_addr(base, qb + g, ni) + 4 * t;
      const uint32_t a1 = sw_addr(base, qb + g + 8, ni) + 4 * t;
      asm volatile("st.shared.b32 [%0], %1;" ::"r"(a0), "r"(pack_bf16x2(o[ni][0] * i0, o[ni][1] * i0)) : "memory");
      asm volatile("st.shared.b32 [%0], %1;" ::"r"(a1), "r"(pack_bf16x2(o[ni][2] * i1, o[ni][3] * i1)) : "memory");
    }
    __syncwarp();
    if constexpr (TT != 0) {
      bf16* dstp = st_lane + static_cast<size_t>(p) * D;
      const uint32_t boff = buf * (BUF_ROWS * 128);
#pragma unroll
      for (int j = 0; j < TT / 4; ++j) {
        uint4 v;
        const uint32_t src = ((j & 1) ? sm_lane1 + (4 * j - 4) * 128 : sm_lane0 + 4 * j * 128) + boff;
        asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                     : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                     : "r"(src));
        *reinterpret_cast<uint4*>(dstp + j * st_step4) = v;
      }
    } else {
      for (int c = lane; c < T * 8; c += 32) {
        const int f = c >> 3, ch = c & 7;
        uint4 v;
        asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                     : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                     : "r"(sw_addr(base, qb + f, ch)));
        bf16* dst = out + (static_cast<size_t>(b) * N + 1 + static_cast<size_t>(f) * n + p) * D + h * HD + ch * 8;
        *reinterpret_cast<uint4*>(dst) = v;
      }
    }
    __syncwarp();  // this buffer is refilled by the prefetch issued at the top of the next iteration
  }

  cl += __shfl_xor_sync(0xffffffffu, cl, 1);
  cl += __shfl_xor_sync(0xffffffffu, cl, 2);
  if (g == 0) {
    float* dst = cls_part + ((static_cast<size_t>(b) * H + h) * nchunks + chunk) * (HD + 2);
    if (t == 0) {
      dst[0] = cm;
      dst[1] = cl;
    }
#pragma unroll
    for (int ni = 0; ni < 8; ++ni) {
      dst[2 + ni * 8 + 2 * t] = co[ni][0];
      dst[2 + ni * 8 + 2 * t + 1] = co[ni][1];
    }
  }
}

}  // namespace

template <int TT>
static int launch_v2(const bf16* qkv, bf16* out, int B, int T, int n, int H, float* cls_ws, int pchunk, int nchunks,
                     cudaStream_t stream) {
  const size_t smem = static_cast<size_t>(TW) * WARP_BYTES;
  static bool configured = false;
  if (!configured) {
    HH_CHECK_CUDA(cudaFuncSetAttribute(attn_time_v2_kernel<TT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>(smem)));
    configured = true;
  }
  const long long blocks = static_cast<long long>(B) * ((H + TW - 1) / TW) * nchunks;
  HH_REQUIRE(blocks < (1ll << 31), "attn_time: grid too large");
  attn_time_v2_kernel<TT><<<static_cast<unsigned>(blocks), TW * 32, smem, stream>>>(qkv, out, cls_ws, T, n, H, pchunk,
                                                                                     nchunks);
  HH_CHECK_LAUNCH("attn_time_v2_kernel");
  return 0;
}

int attn_time_v2(const bf16* qkv, bf16* out, int B, int T, int n, int H, float* cls_ws, int pchunk, int nchunks,
                 cudaStream_t stream) {
  if (T == 16) return launch_v2<16>(qkv, out, B, T, n, H, cls_ws, pchunk, nchunks, stream);
  if (T == 8) return launch_v2<8>(qkv, out, B, T, n, H, cls_ws, pchunk, nchunks, stream);
  if (T == 4) return launch_v2<4>(qkv, out, B, T, n, H, cls_ws, pchunk, nchunks, stream);
  return launch_v2<0>(qkv, out, B, T, n, H, cls_ws, pchunk, nchunks, stream);
}

}  // namespace hh
