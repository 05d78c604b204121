// Temporal half of the divided space-time attention (VarAttention with einops '(b n) f d', model/LaviLa.py:246-283)
// and the CLS query row shared by both halves.
//
// attn_time (T <= 16) runs the tensor-core kernel of attn_time_v2.cu, which writes one partial of the CLS *query*
// (which attends all 1+T*n keys, LaviLa.py:258) per (clip, head, patch-chunk); attn_cls_merge folds the partials and the
// CLS key itself into output row 0.
// attn_time (16 < T <= 32) keeps the simple SIMT kernel + the stand-alone CLS kernel.
#include "hh_internal.h"
#include "hh_ptx.cuh"

namespace hh {

namespace {

constexpr int HD = 64;
constexpr float LOG2E = 1.4426950408889634f;

__device__ __forceinline__ void unpack8(const uint4& u, float* f) {
  float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y), c = unpack_bf16x2(u.z), d = unpack_bf16x2(u.w);
  f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
}

// Folds the per-chunk partials of the CLS query and the CLS key/value itself into output row 0 of every (clip, head).
__global__ void __launch_bounds__(HD)
attn_cls_merge_kernel(const bf16* __restrict__ qkv, const float* __restrict__ part, bf16* __restrict__ out, int N, int H,
                      int nparts) {
  __shared__ float red[2];
  const int h = blockIdx.x % H, b = blockIdx.x / H;
  const int d = threadIdx.x;
  const int D = H * HD;
  const bf16* cls = qkv + static_cast<size_t>(b) * N * 3 * D + h * HD;
  // s_cls = q_cls . k_cls (q pre-scaled)
  float prod = __bfloat162float(cls[d]) * __bfloat162float(cls[D + d]);
  prod = warp_sum(prod);
  if ((d & 31) == 0) red[d >> 5] = prod;
  __syncthreads();
  const float s_cls = red[0] + red[1];
  const float* base = part + static_cast<size_t>(blockIdx.x) * nparts * (HD + 2);
  float mm = s_cls;
  for (int i = 0; i < nparts; ++i) mm = fmaxf(mm, base[i * (HD + 2)]);
  float ll = exp2f((s_cls - mm) * LOG2E);
  float oo = ll * __bfloat162float(cls[2 * D + d]);
  for (int i = 0; i < nparts; ++i) {
    const float* pr = base + i * (HD + 2);
    const float c = (pr[0] == -INFINITY) ? 0.f : exp2f((pr[0] - mm) * LOG2E);
    ll += pr[1] * c;
    oo += pr[2 + d] * c;
  }
  out[static_cast<size_t>(b) * N * D + h * HD + d] = __float2bfloat16(oo / ll);
}

// ============================================================================================ SIMT kernel (T > 16)
constexpr int TIME_WARPS = 4;

// TP: padded frame count (lanes per sub-problem). Keys per problem: T + 1 <= TP + 1.
template <int TP>
__global__ void __launch_bounds__(TIME_WARPS * 32)
attn_time_kernel(const bf16* __restrict__ qkv, bf16* __restrict__ out, int B, int T, int n, int H) {
  constexpr int PPW = 32 / TP;       // problems (heads) per warp
  constexpr int NK = TP + 1;         // key slots per problem
  extern __shared__ __align__(16) uint8_t smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* Ks = reinterpret_cast<float*>(smem_raw) + static_cast<size_t>(warp) * (2 * PPW * NK * HD);
  float* Vs = Ks + PPW * NK * HD;

  const int D = H * HD;
  const int N = 1 + T * n;
  const int hgroups = (H + PPW - 1) / PPW;
  const long long task = static_cast<long long>(blockIdx.x) * TIME_WARPS + warp;
  const long long ntasks = static_cast<long long>(B) * n * hgroups;
  if (task >= ntasks) return;
  const int hg = static_cast<int>(task % hgroups);
  const int p = static_cast<int>((task / hgroups) % n);
  const int b = static_cast<int>(task / (static_cast<long long>(hgroups) * n));
  const int h0 = hg * PPW;
  const size_t ld = static_cast<size_t>(3) * D;
  const bf16* clip = qkv + static_cast<size_t>(b) * N * ld;

  const int nkeys = T + 1;
  for (int c = lane; c < PPW * nkeys * 8; c += 32) {
    const int ch = c & 7;
    const int slot = (c >> 3) % nkeys;
    const int sp = (c >> 3) / nkeys;
    if (h0 + sp < H) {
      const size_t tokrow = (slot == 0) ? 0 : (1 + static_cast<size_t>(slot - 1) * n + p);
      const bf16* src = clip + tokrow * ld + (h0 + sp) * HD + ch * 8;
      const uint4 ku = *reinterpret_cast<const uint4*>(src + D);
      const uint4 vu = *reinterpret_cast<const uint4*>(src + 2 * D);
      float kf[8], vf[8];
      unpack8(ku, kf);
      unpack8(vu, vf);
      float* kd = Ks + (sp * NK + slot) * HD + ch * 8;
      float* vd = Vs + (sp * NK + slot) * HD + ch * 8;
      *reinterpret_cast<float4*>(kd) = make_float4(kf[0], kf[1], kf[2], kf[3]);
      *reinterpret_cast<float4*>(kd + 4) = make_float4(kf[4], kf[5], kf[6], kf[7]);
      *reinterpret_cast<float4*>(vd) = make_float4(vf[0], vf[1], vf[2], vf[3]);
      *reinterpret_cast<float4*>(vd + 4) = make_float4(vf[4], vf[5], vf[6], vf[7]);
    }
  }
  __syncwarp();

  const int sp = lane / TP, f = lane % TP;
  const bool active = (f < T) && (h0 + sp < H);
  if (!active) return;
  const size_t qrow = 1 + static_cast<size_t>(f) * n + p;
  const bf16* qsrc = clip + qrow * ld + (h0 + sp) * HD;
  float q[HD];
#pragma unroll
  for (int c = 0; c < 8; ++c) unpack8(*reinterpret_cast<const uint4*>(qsrc + c * 8), q + c * 8);

  const float* Kp = Ks + sp * NK * HD;
  const float* Vp = Vs + sp * NK * HD;
  float s[NK];
  float mx = -INFINITY;
#pragma unroll
  for (int j = 0; j < NK; ++j) {
    if (j < nkeys) {
      float acc = 0.f;
#pragma unroll
      for (int d = 0; d < HD; d += 4) {
        const float4 k4 = *reinterpret_cast<const float4*>(Kp + j * HD + d);
        acc += q[d] * k4.x + q[d + 1] * k4.y + q[d + 2] * k4.z + q[d + 3] * k4.w;
      }
      s[j] = acc;
      mx = fmaxf(mx, acc);
    } else {
      s[j] = -INFINITY;
    }
  }
  float l = 0.f;
#pragma unroll
  for (int j = 0; j < NK; ++j) {
    s[j] = exp2f((s[j] - mx) * LOG2E);
    l += s[j];
  }
  const float inv = 1.f / l;
#pragma unroll
  for (int d = 0; d < HD; ++d) q[d] = 0.f;
#pragma unroll
  for (int j = 0; j < NK; ++j) {
    if (j < nkeys) {
      const float pj = s[j] * inv;
#pragma unroll
      for (int d = 0; d < HD; d += 4) {
        const float4 v4 = *reinterpret_cast<const float4*>(Vp + j * HD + d);
        q[d] += pj * v4.x; q[d + 1] += pj * v4.y; q[d + 2] += pj * v4.z; q[d + 3] += pj * v4.w;
      }
    }
  }
  bf16* dst = out + (static_cast<size_t>(b) * N + qrow) * D + (h0 + sp) * HD;
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    uint4 u;
    u.x = pack_bf16x2(q[c * 8 + 0], q[c * 8 + 1]);
    u.y = pack_bf16x2(q[c * 8 + 2], q[c * 8 + 3]);
    u.z = pack_bf16x2(q[c * 8 + 4], q[c * 8 + 5]);
    u.w = pack_bf16x2(q[c * 8 + 6], q[c * 8 + 7]);
    *reinterpret_cast<uint4*>(dst + c * 8) = u;
  }
}

template <int TP>
int launch_time(const bf16* qkv, bf16* out, int B, int T, int n, int H, cudaStream_t stream) {
  constexpr int PPW = 32 / TP;
  const size_t smem = static_cast<size_t>(TIME_WARPS) * 2 * PPW * (TP + 1) * HD * sizeof(float);
  static bool configured = false;
  if (!configured) {
    HH_CHECK_CUDA(cudaFuncSetAttribute(attn_time_kernel<TP>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>(smem)));
    configured = true;
  }
  const long long ntasks = static_cast<long long>(B) * n * ((H + PPW - 1) / PPW);
  const long long blocks = (ntasks + TIME_WARPS - 1) / TIME_WARPS;
  HH_REQUIRE(blocks < (1ll << 31), "attn_time: grid too large");
  attn_time_kernel<TP><<<static_cast<unsigned>(blocks), TIME_WARPS * 32, smem, stream>>>(qkv, out, B, T, n, H);
  HH_CHECK_LAUNCH("attn_time_kernel");
  return 0;
}

// ------------------------------------------------------------------------------------------ stand-alone CLS query row
constexpr int CLS_WARPS = 8;

__global__ void __launch_bounds__(CLS_WARPS * 32)
attn_cls_kernel(const bf16* __restrict__ qkv, bf16* __restrict__ out, int N, int H) {
  __shared__ float sm_m[CLS_WARPS * 4];
  __shared__ float sm_l[CLS_WARPS * 4];
  __shared__ float sm_o[CLS_WARPS * 4][HD];
  const int D = H * HD;
  const int h = blockIdx.x % H, b = blockIdx.x / H;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int grp = lane >> 3, sub = lane & 7;  // 4 key groups per warp, 8 lanes x 8 dims per key
  const size_t ld = static_cast<size_t>(3) * D;
  const bf16* clip = qkv + static_cast<size_t>(b) * N * ld + h * HD + sub * 8;

  float q[8];
  unpack8(*reinterpret_cast<const uint4*>(clip), q);  // CLS token is row 0; q section is columns [0, D)
  float m = -INFINITY, l = 0.f, o[8];
#pragma unroll
  for (int d = 0; d < 8; ++d) o[d] = 0.f;

  const int step = CLS_WARPS * 4;
  for (int j0 = 0; j0 < N; j0 += step) {  // uniform trip count: the shuffles below need the whole warp
    const int j = j0 + warp * 4 + grp;
    const bool valid = j < N;
    float s = 0.f, v[8];
    if (valid) {
      const bf16* row = clip + static_cast<size_t>(j) * ld;
      float k[8];
      unpack8(*reinterpret_cast<const uint4*>(row + D), k);
      unpack8(*reinterpret_cast<const uint4*>(row + 2 * D), v);
#pragma unroll
      for (int d = 0; d < 8; ++d) s += q[d] * k[d];
    } else {
#pragma unroll
      for (int d = 0; d < 8; ++d) v[d] = 0.f;
    }
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    s += __shfl_xor_sync(0xffffffffu, s, 4);
    if (valid) {
      const float mn = fmaxf(m, s);
      const float c = exp2f((m - mn) * LOG2E);  // m = -inf on first key -> 0
      const float pj = exp2f((s - mn) * LOG2E);
      l = l * c + pj;
#pragma unroll
      for (int d = 0; d < 8; ++d) o[d] = o[d] * c + pj * v[d];
      m = mn;
    }
  }
  const int slot = warp * 4 + grp;
  if (sub == 0) {
    sm_m[slot] = m;
    sm_l[slot] = l;
  }
#pragma unroll
  for (int d = 0; d < 8; ++d) sm_o[slot][sub * 8 + d] = o[d];
  __syncthreads();
  if (threadIdx.x < HD) {
    float mm = -INFINITY;
    for (int s2 = 0; s2 < CLS_WARPS * 4; ++s2) mm = fmaxf(mm, sm_m[s2]);
    float ll = 0.f, acc = 0.f;
    for (int s2 = 0; s2 < CLS_WARPS * 4; ++s2) {
      const float c = (sm_m[s2] == -INFINITY) ? 0.f : exp2f((sm_m[s2] - mm) * LOG2E);
      ll += sm_l[s2] * c;
      acc += sm_o[s2][threadIdx.x] * c;
    }
    out[static_cast<size_t>(b) * N * D + h * HD + threadIdx.x] = __float2bfloat16(acc / ll);
  }
}

}  // namespace

size_t attn_cls_workspace_bytes(int B, int T, int n, int H) {
  const int parts = (T > (n + 15) / 16) ? T : (n + 15) / 16;
  return static_cast<size_t>(B) * H * parts * (HD + 2) * sizeof(float);
}

int attn_cls_merge(const bf16* qkv, const float* parts, bf16* out, int B, int N, int H, int nparts, cudaStream_t stream) {
  attn_cls_merge_kernel<<<B * H, HD, 0, stream>>>(qkv, parts, out, N, H, nparts);
  HH_CHECK_LAUNCH("attn_cls_merge_kernel");
  return 0;
}

int attn_time(const bf16* qkv, bf16* out, int B, int T, int n, int H, float* cls_ws, cudaStream_t stream) {
  HH_REQUIRE(B > 0 && T > 0 && n > 0 && H > 0, "attn_time: empty problem");
  HH_REQUIRE(T <= 32, "attn_time: at most 32 frames");
  if (T <= 16) {
    HH_REQUIRE(cls_ws != nullptr, "attn_time: CLS workspace");
    const int pchunk = 16;
    const int nchunks = (n + pchunk - 1) / pchunk;
    int rc = attn_time_v2(qkv, out, B, T, n, H, cls_ws, pchunk, nchunks, stream);
    if (rc) return rc;
    return attn_cls_merge(qkv, cls_ws, out, B, 1 + T * n, H, nchunks, stream);
  }
  int rc = launch_time<32>(qkv, out, B, T, n, H, stream);
  if (rc) return rc;
  return attn_cls(qkv, out, B, 1 + T * n, H, stream);
}

int attn_cls(const bf16* qkv, bf16* out, int B, int N, int H, cudaStream_t stream) {
  HH_REQUIRE(B > 0 && N > 0 && H > 0, "attn_cls: empty problem");
  attn_cls_kernel<<<B * H, CLS_WARPS * 32, 0, stream>>>(qkv, out, N, H);
  HH_CHECK_LAUNCH("attn_cls_kernel");
  return 0;
}

}  // namespace hh
