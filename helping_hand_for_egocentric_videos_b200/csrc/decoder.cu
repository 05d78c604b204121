// Query-side kernels of the object-aware decoder (model/tfm_decoder.py).  The decoder's heavy contractions (memory
// projection, the 6 layers' K/V projections, the class head) run on the tcgen05 GEMM; what is left operates on the
// Q <= kMaxQueries (32) learned queries per clip and is latency-, not FLOP-bound.  Everything here is fp32.
//
//   linear_f32          small-M nn.Linear (+ query_pos add on the input, bias, ReLU/sigmoid, residual); fp32 operands on
//                       the tensor cores as error-compensated TF32 (3 MMAs per product, fp32-level accuracy)
//   self_attn_queries   nn.MultiheadAttention core over the Q queries (tfm_decoder.py:433)
//   cross_attn          query -> patch-token attention core (tfm_decoder.py:438-441), split over keys (flash-decode
//                       style) with an exact merge; the head-averaged attention map the reference computes and
//                       discards (:271-295) is not produced
#include "hh_internal.h"
#include "hh_ptx.cuh"

namespace hh {

namespace {

constexpr float LOG2E = 1.4426950408889634f;
constexpr int HD = 64;

// ------------------------------------------------------------------------------------------ linear_f32
constexpr int LBM = 32, LBN = 64, LBK = 32;

// Tensor-core inner product (3xTF32, fp32-level accuracy): 8 warps = 2 row blocks of 16 x 4 column blocks of 16.
constexpr int LSA = LBK + 4;   // smem row stride: fragment loads (rows g, columns t) hit 32 distinct banks

__global__ void __launch_bounds__(256) linear_f32_kernel(const LinArgs a) {
  __shared__ __align__(16) float As[LBM][LSA];
  __shared__ __align__(16) float Ws[LBN][LSA];
  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  const int wm = warp & 1, wn = warp >> 1;
  const int r0 = blockIdx.y * LBM, n0 = blockIdx.x * LBN;
  float acc[2][4];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  // software pipeline: the next K tile's global loads are issued before this tile's MMAs and land in registers while
  // they run (few CTAs per SM here: the load latency is otherwise fully exposed every iteration)
  float4 ra, rw[2];
  auto load_tiles = [&](int k0) {
    {  // A tile: 32 rows x 32 k, one float4 per thread
      const int r = tid >> 3, kk = (tid & 7) * 4;
      const int row = r0 + r;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (row < a.R) {
        v = *reinterpret_cast<const float4*>(a.in + static_cast<size_t>(row) * a.ldi + k0 + kk);
        if (a.in_add) {
          const float4 q = *reinterpret_cast<const float4*>(a.in_add + static_cast<size_t>(row % a.add_mod) * a.K + k0 + kk);
          v.x += q.x; v.y += q.y; v.z += q.z; v.w += q.w;
        }
        if (a.in_relu) {
          v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f);
        }
      }
      ra = v;
    }
#pragma unroll
    for (int it = 0; it < 2; ++it) {  // W tile: 64 n x 32 k
      const int idx = tid + it * 256;
      const int nn = idx >> 3, kk = (idx & 7) * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (n0 + nn < a.N) v = *reinterpret_cast<const float4*>(a.W + static_cast<size_t>(n0 + nn) * a.K + k0 + kk);
      rw[it] = v;
    }
  };
  load_tiles(0);
  for (int k0 = 0; k0 < a.K; k0 += LBK) {
    *reinterpret_cast<float4*>(&As[tid >> 3][(tid & 7) * 4]) = ra;
#pragma unroll
    for (int it = 0; it < 2; ++it) {
      const int idx = tid + it * 256;
      *reinterpret_cast<float4*>(&Ws[idx >> 3][(idx & 7) * 4]) = rw[it];
    }
    __syncthreads();
    if (k0 + LBK < a.K) load_tiles(k0 + LBK);
    // the tensor core truncates when it accumulates: chain only this tile's 4 k-steps there and add the tile's
    // partial to the running sum with a rounded fp32 add (keeps the result within ~5e-7 of an fp32 FMA chain)
    float part[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
#pragma unroll
    for (int ks = 0; ks < LBK / 8; ++ks) {
      const float af[4] = {As[wm * 16 + g][ks * 8 + t], As[wm * 16 + g + 8][ks * 8 + t], As[wm * 16 + g][ks * 8 + t + 4],
                           As[wm * 16 + g + 8][ks * 8 + t + 4]};
#pragma unroll
      for (int j = 0; j < 2; ++j)
        mma_3xtf32(part[j], af, Ws[wn * 16 + j * 8 + g][ks * 8 + t], Ws[wn * 16 + j * 8 + g][ks * 8 + t + 4]);
    }
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[j][e] += part[j][e];
    __syncthreads();
  }
#pragma unroll
  for (int j = 0; j < 2; ++j) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int row = r0 + wm * 16 + g + (e >> 1) * 8;
      const int col = n0 + wn * 16 + j * 8 + 2 * t + (e & 1);
      if (row >= a.R || col >= a.N) continue;
      float v = acc[j][e] + (a.bias ? a.bias[col] : 0.f);
      if (a.act == 1) v = fmaxf(v, 0.f);
      else if (a.act == 2) v = 1.f / (1.f + __expf(-v));
      if (a.drop.thr) v *= drop_mult(a.drop, a.drop_site, static_cast<uint64_t>(row) * a.N + col);
      if (a.residual) v += a.residual[static_cast<size_t>(row) * a.ldres + col];
      a.out[static_cast<size_t>(row) * a.ldo + col] = v;
    }
  }
}

// ------------------------------------------------------------------------------------------ self attention
// one warp per (clip, head), lane = query: a warp holds every query the decoder takes; terms for j >= Q are exact zeros
static_assert(kMaxQueries <= 32, "self_attn_kernel: one lane per query");
__global__ void __launch_bounds__(32)
self_attn_kernel(const float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v, int ld,
                 float* __restrict__ out, int Q, int heads, DropCfg drop, uint32_t drop_site) {
  __shared__ float Ks[kMaxQueries][HD + 1];
  __shared__ float Vs[kMaxQueries][HD + 1];
  const int h = blockIdx.x % heads, b = blockIdx.x / heads;
  const int lane = threadIdx.x;
  const int C = heads * HD;
  for (int i = lane; i < Q * HD; i += 32) {
    const int r = i / HD, d = i - r * HD;
    Ks[r][d] = k[static_cast<size_t>(b * Q + r) * ld + h * HD + d];
    Vs[r][d] = v[static_cast<size_t>(b * Q + r) * ld + h * HD + d];
  }
  __syncwarp();
  if (lane >= Q) return;
  const float* qr = q + static_cast<size_t>(b * Q + lane) * ld + h * HD;
  float s[kMaxQueries];
  float mx = -INFINITY;
#pragma unroll
  for (int j = 0; j < kMaxQueries; ++j) {
    if (j < Q) {
      float acc = 0.f;
      for (int d = 0; d < HD; ++d) acc += qr[d] * Ks[j][d];
      s[j] = acc;
      mx = fmaxf(mx, acc);
    } else {
      s[j] = -INFINITY;
    }
  }
  float l = 0.f;
#pragma unroll
  for (int j = 0; j < kMaxQueries; ++j) {
    s[j] = exp2f((s[j] - mx) * LOG2E);
    l += s[j];
  }
  const float inv = 1.f / l;
  if (drop.thr) {  // dropout on the normalised probabilities (nn.MultiheadAttention, training mode)
    const uint64_t base = (static_cast<uint64_t>(blockIdx.x) * Q + lane) * Q;
#pragma unroll
    for (int j = 0; j < kMaxQueries; ++j)
      if (j < Q) s[j] *= drop_mult(drop, drop_site, base + j);
  }
  float* o = out + static_cast<size_t>(b * Q + lane) * C + h * HD;
  for (int d = 0; d < HD; ++d) {
    float acc = 0.f;
#pragma unroll
    for (int j = 0; j < kMaxQueries; ++j)
      if (j < Q) acc += s[j] * Vs[j][d];
    o[d] = acc * inv;
  }
}

// ------------------------------------------------------------------------------------------ cross attention
constexpr int XQ = 16;       // max queries of this differential-test statement (static smem: 48 KB at 16)
constexpr int XWARPS = 4;
constexpr int XPART = HD + 2;  // per (query): m, l, o[64]

__global__ void __launch_bounds__(XWARPS * 32)
cross_attn_kernel(const float* __restrict__ q, const bf16* __restrict__ K, const bf16* __restrict__ V, int ldkv,
                  float* __restrict__ part, int Q, int heads, int S, int splits) {
  __shared__ __align__(16) float qs[XQ][HD];
  __shared__ float ps[XWARPS][XQ][32];
  __shared__ float wm[XWARPS][XQ], wl[XWARPS][XQ];
  __shared__ float wo[XWARPS][XQ][HD];
  const int split = blockIdx.x % splits;
  const int h = (blockIdx.x / splits) % heads;
  const int b = blockIdx.x / (splits * heads);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int C = heads * HD;

  for (int i = threadIdx.x; i < XQ * HD; i += blockDim.x) {
    const int r = i / HD, d = i - r * HD;
    qs[r][d] = (r < Q) ? q[static_cast<size_t>(b * Q + r) * C + h * HD + d] : 0.f;
  }
  __syncthreads();

  const int per = ((S + splits - 1) / splits + 31) & ~31;  // keys per split, multiple of 32
  const int k_begin = split * per;
  const int k_end = min(S, k_begin + per);
  const bf16* Kb = K + static_cast<size_t>(b) * S * ldkv + h * HD;
  const bf16* Vb = V + static_cast<size_t>(b) * S * ldkv + h * HD;

  float m[XQ], l[XQ], acc[XQ][2];
#pragma unroll
  for (int i = 0; i < XQ; ++i) {
    m[i] = -INFINITY;
    l[i] = 0.f;
    acc[i][0] = acc[i][1] = 0.f;
  }

  for (int kb = k_begin + warp * 32; kb < k_end; kb += XWARPS * 32) {
    // ---- phase 1: lane = key
    const int key = kb + lane;
    const bool valid = key < k_end;
    float kf[HD];
    if (valid) {
      const uint4* src = reinterpret_cast<const uint4*>(Kb + static_cast<size_t>(key) * ldkv);
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const uint4 u = src[c];
        float2 t0 = unpack_bf16x2(u.x), t1 = unpack_bf16x2(u.y), t2 = unpack_bf16x2(u.z), t3 = unpack_bf16x2(u.w);
        kf[c * 8 + 0] = t0.x; kf[c * 8 + 1] = t0.y; kf[c * 8 + 2] = t1.x; kf[c * 8 + 3] = t1.y;
        kf[c * 8 + 4] = t2.x; kf[c * 8 + 5] = t2.y; kf[c * 8 + 6] = t3.x; kf[c * 8 + 7] = t3.y;
      }
    } else {
#pragma unroll
      for (int d = 0; d < HD; ++d) kf[d] = 0.f;
    }
    float cfac[XQ];
#pragma unroll
    for (int i = 0; i < XQ; ++i) {
      if (i < Q) {  // Q is block-uniform
        float s = 0.f;
#pragma unroll
        for (int d = 0; d < HD; d += 4) {
          const float4 q4 = *reinterpret_cast<const float4*>(&qs[i][d]);
          s += kf[d] * q4.x + kf[d + 1] * q4.y + kf[d + 2] * q4.z + kf[d + 3] * q4.w;
        }
        if (!valid) s = -INFINITY;
        const float bm = warp_max(s);            // finite: lane 0 of every visited block is a valid key
        const float mn = fmaxf(m[i], bm);
        const float p = exp2f((s - mn) * LOG2E);
        cfac[i] = exp2f((m[i] - mn) * LOG2E);
        m[i] = mn;
        l[i] = l[i] * cfac[i] + warp_sum(p);
        ps[warp][i][lane] = p;
      } else {
        cfac[i] = 1.f;
      }
    }
    __syncwarp();
    // ---- phase 2: lane = output dim pair (2*lane, 2*lane+1)
#pragma unroll
    for (int i = 0; i < XQ; ++i) {
      acc[i][0] *= cfac[i];
      acc[i][1] *= cfac[i];
    }
    const int nvalid = min(32, k_end - kb);
    for (int j = 0; j < nvalid; ++j) {
      const float2 v2 = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(Vb + static_cast<size_t>(kb + j) * ldkv + 2 * lane));
#pragma unroll
      for (int i = 0; i < XQ; ++i) {
        if (i < Q) {
          const float p = ps[warp][i][j];
          acc[i][0] += p * v2.x;
          acc[i][1] += p * v2.y;
        }
      }
    }
    __syncwarp();
  }

  // ---- merge the 4 warps, write the split's partial (m, l, unnormalised o)
#pragma unroll
  for (int i = 0; i < XQ; ++i) {
    if (i < Q) {
      if (lane == 0) {
        wm[warp][i] = m[i];
        wl[warp][i] = l[i];
      }
      wo[warp][i][2 * lane] = acc[i][0];
      wo[warp][i][2 * lane + 1] = acc[i][1];
    }
  }
  __syncthreads();
  float* dst = part + static_cast<size_t>(blockIdx.x) * XQ * XPART;
  for (int idx = threadIdx.x; idx < Q * HD; idx += blockDim.x) {
    const int i = idx / HD, d = idx - i * HD;
    float mm = -INFINITY;
#pragma unroll
    for (int w = 0; w < XWARPS; ++w) mm = fmaxf(mm, wm[w][i]);
    float ll = 0.f, oo = 0.f;
#pragma unroll
    for (int w = 0; w < XWARPS; ++w) {
      const float c = (wm[w][i] == -INFINITY) ? 0.f : exp2f((wm[w][i] - mm) * LOG2E);
      ll += wl[w][i] * c;
      oo += wo[w][i][d] * c;
    }
    dst[i * XPART + 2 + d] = oo;
    if (d == 0) {
      dst[i * XPART] = mm;
      dst[i * XPART + 1] = ll;
    }
  }
}

__global__ void __launch_bounds__(HD)
cross_merge_kernel(const float* __restrict__ part, float* __restrict__ out, int Q, int heads, int splits) {
  const int h = blockIdx.x % heads, b = blockIdx.x / heads;
  const int d = threadIdx.x;
  const int C = heads * HD;
  const float* base = part + static_cast<size_t>(blockIdx.x) * splits * XQ * XPART;
  for (int i = 0; i < Q; ++i) {
    float mm = -INFINITY;
    for (int s = 0; s < splits; ++s) mm = fmaxf(mm, base[(s * XQ + i) * XPART]);
    float ll = 0.f, oo = 0.f;
    for (int s = 0; s < splits; ++s) {
      const float* pr = base + (s * XQ + i) * XPART;
      const float c = (pr[0] == -INFINITY) ? 0.f : exp2f((pr[0] - mm) * LOG2E);
      ll += pr[1] * c;
      oo += pr[2 + d] * c;
    }
    out[static_cast<size_t>(b * Q + i) * C + h * HD + d] = oo / ll;
  }
}

int cross_splits(int B, int heads, int S) {
  int splits = (4 * num_sms() + B * heads - 1) / (B * heads);
  const int max_splits = (S + 127) / 128;
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  return splits;
}

// ------------------------------------------------------------------------------------------ head helpers
__global__ void __launch_bounds__(256)
add_frame_term_kernel(const float* __restrict__ hsproj, const float* __restrict__ frameterm, float* __restrict__ out,
                      int LB, int T, int Q, int C) {
  const int c4 = C >> 2;
  const long long total = static_cast<long long>(LB) * T * Q * c4;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % c4) * 4;
    const long long r = i / c4;  // (lb, t, q)
    const int qi = static_cast<int>(r % Q);
    const int t = static_cast<int>((r / Q) % T);
    const long long lb = r / (static_cast<long long>(Q) * T);
    const float4 a = *reinterpret_cast<const float4*>(hsproj + (lb * Q + qi) * C + c);
    const float4 f = *reinterpret_cast<const float4*>(frameterm + static_cast<size_t>(t) * C + c);
    *reinterpret_cast<float4*>(out + r * C + c) = make_float4(a.x + f.x, a.y + f.y, a.z + f.z, a.w + f.w);
  }
}

__global__ void __launch_bounds__(256)
expand_rows_kernel(const float* __restrict__ src, float* __restrict__ dst, int LB, int rep, size_t per4) {
  const size_t total = static_cast<size_t>(LB) * rep * per4;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const size_t e = i % per4;
    const size_t lb = i / (per4 * rep);
    reinterpret_cast<float4*>(dst)[i] = reinterpret_cast<const float4*>(src)[lb * per4 + e];
  }
}

__global__ void __launch_bounds__(256)
expand_rows_scalar_kernel(const float* __restrict__ src, float* __restrict__ dst, int LB, int rep, size_t per) {
  const size_t total = static_cast<size_t>(LB) * rep * per;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x)
    dst[i] = src[(i / (per * rep)) * per + i % per];
}

}  // namespace

int linear_f32_legacy(const LinArgs& a, cudaStream_t stream) {
  HH_REQUIRE(a.R > 0 && a.N > 0 && a.K > 0, "linear_f32: empty problem");
  HH_REQUIRE(a.K % LBK == 0 && a.ldi % 4 == 0, "linear_f32: K must be a multiple of 32 and ldi of 4");
  HH_REQUIRE(a.in_add == nullptr || a.add_mod > 0, "linear_f32: add_mod");
  dim3 grid((a.N + LBN - 1) / LBN, (a.R + LBM - 1) / LBM);
  linear_f32_kernel<<<grid, 256, 0, stream>>>(a);
  HH_CHECK_LAUNCH("linear_f32_kernel");
  return 0;
}

int self_attn_queries(const float* q, const float* k, const float* v, int ld, float* out, int B, int Q, int heads,
                      cudaStream_t stream, DropCfg drop, uint32_t drop_site) {
  HH_REQUIRE(Q >= 1 && Q <= kMaxQueries, "self_attn_queries: 1..32 queries supported");
  self_attn_kernel<<<B * heads, 32, 0, stream>>>(q, k, v, ld, out, Q, heads, drop, drop_site);
  HH_CHECK_LAUNCH("self_attn_kernel");
  return 0;
}

size_t cross_attn_simt_workspace_bytes(int B, int Q, int heads, int S) {
  (void)Q;
  return static_cast<size_t>(B) * heads * cross_splits(B, heads, S) * XQ * XPART * sizeof(float);
}

// fp32 SIMT statement of the cross attention (kept as a second implementation for differential tests; Q <= 16 only,
// tests compare larger Q with float64 torch)
int cross_attn_simt(const float* q, const bf16* K, const bf16* V, int ldkv, float* out, int B, int Q, int heads, int S,
                    void* workspace, cudaStream_t stream) {
  HH_REQUIRE(Q >= 1 && Q <= XQ, "cross_attn: 1..16 queries supported");
  HH_REQUIRE(ldkv % 8 == 0, "cross_attn: K/V row stride must be a multiple of 8 elements");
  HH_REQUIRE(workspace != nullptr, "cross_attn: workspace");
  const int splits = cross_splits(B, heads, S);
  cross_attn_kernel<<<B * heads * splits, XWARPS * 32, 0, stream>>>(q, K, V, ldkv, static_cast<float*>(workspace), Q,
                                                                   heads, S, splits);
  HH_CHECK_LAUNCH("cross_attn_kernel");
  cross_merge_kernel<<<B * heads, HD, 0, stream>>>(static_cast<const float*>(workspace), out, Q, heads, splits);
  HH_CHECK_LAUNCH("cross_merge_kernel");
  return 0;
}

int add_frame_term(const float* hsproj, const float* frameterm, float* out, int LB, int T, int Q, int C,
                   cudaStream_t stream) {
  HH_REQUIRE(C % 4 == 0, "add_frame_term: C must be a multiple of 4");
  const long long total = static_cast<long long>(LB) * T * Q * (C / 4);
  long long blocks = (total + 255) / 256;
  const long long cap = static_cast<long long>(num_sms()) * 16;
  if (blocks > cap) blocks = cap;
  add_frame_term_kernel<<<static_cast<int>(blocks), 256, 0, stream>>>(hsproj, frameterm, out, LB, T, Q, C);
  HH_CHECK_LAUNCH("add_frame_term_kernel");
  return 0;
}

int expand_logits(const float* src, float* dst, int LB, int rep, size_t per, cudaStream_t stream) {
  const bool vec = per % 4 == 0 && (reinterpret_cast<uintptr_t>(src) & 15) == 0 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0;
  const size_t total = static_cast<size_t>(LB) * rep * (vec ? per / 4 : per);
  size_t blocks = (total + 255) / 256;
  const size_t cap = static_cast<size_t>(num_sms()) * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  if (vec) expand_rows_kernel<<<static_cast<int>(blocks), 256, 0, stream>>>(src, dst, LB, rep, per / 4);
  else expand_rows_scalar_kernel<<<static_cast<int>(blocks), 256, 0, stream>>>(src, dst, LB, rep, per);
  HH_CHECK_LAUNCH("expand_rows_kernel");
  return 0;
}

}  // namespace hh
