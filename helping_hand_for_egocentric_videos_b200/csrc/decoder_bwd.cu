// Backward primitives of the object-aware decoder (SURVEY.md section 8f row 2: "decoder / heads backward").
// The query side (Q <= kMaxQueries = 32 rows per clip) keeps fp32 operands like its forward (linears as
// error-compensated TF32 on the tensor cores, the rest SIMT); the memory side (B*S patch tokens) reuses
// the tcgen05 GEMM for its data- and weight-gradient contractions (engine_bwd.cu) and needs from here only the
// cross-attention backward, LayerNorm backward, column sums and transposes.
//
//   linear_dgrad_f32 / linear_wgrad_f32   nn.Linear backward (activation derivative and query_pos add folded in)
//   ln_backward_rows                       LayerNorm backward: dx per row + two-stage deterministic dgamma / dbeta
//   self_attn_bwd                          nn.MultiheadAttention core over the queries
//   cross_attn_bwd                         query -> patch attention core: softmax statistics, per-key dK / dV / dS,
//                                          then dQ = dS K
//   colsum_rows, transpose_to_bf16         reductions / layout changes feeding the weight-gradient GEMMs
#include "hh_internal.h"
#include "hh_ptx.cuh"

namespace hh {

namespace {

constexpr int HD = 64;

__device__ __forceinline__ float act_grad(float dy, float y, int act) {
  if (act == 1) return y > 0.f ? dy : 0.f;        // ReLU (y is the saved output)
  if (act == 2) return dy * y * (1.f - y);        // sigmoid
  return dy;
}

// ------------------------------------------------------------------------------------------ linear backward
// dX[r, k] = beta * dX[r, k] + sum_n g[r, n] * W[n, k],  g = act'(dY, Y)
// Inner products on the tensor cores as error-compensated TF32 (mma_3xtf32: fp32-level accuracy); 8 warps = 2 row
// blocks of 16 x 4 column blocks of 16; smem strides chosen so that fragment loads are bank-conflict free.
__global__ void __launch_bounds__(256) linear_dgrad_kernel(const LinBwdArgs a) {
  __shared__ float Gs[32][36];   // [r][n]
  __shared__ float Ws[32][72];   // [n][k]
  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  const int wm = warp & 1, wn = warp >> 1;
  const int r0 = blockIdx.y * 32, k0 = blockIdx.x * 64;
  float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
  // split-N: CTA z reduces output features [z * n_per_split, ...) and adds its partial tile atomically (host wrapper)
  const int n_begin = blockIdx.z * a.rows_per_split;
  const int n_end = (n_begin + a.rows_per_split < a.N) ? n_begin + a.rows_per_split : a.N;
  // software pipeline: the next tile's global loads are in flight (registers) while this tile's MMAs run
  float gr[4], wr[8];
  auto load_tiles = [&](int n0) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int idx = tid + i * 256;
      const int r = idx >> 5, n = idx & 31;
      float v = 0.f;
      if (r0 + r < a.R && n0 + n < n_end) {
        v = a.dY[static_cast<size_t>(r0 + r) * a.ldy + n0 + n];
        if (a.drop.thr) v *= drop_mult(a.drop, a.drop_site, static_cast<uint64_t>(r0 + r) * a.N + n0 + n);
        if (a.act) v = act_grad(v, a.Y[static_cast<size_t>(r0 + r) * a.ldyo + n0 + n], a.act) * (a.act_scale != 0.f ? a.act_scale : 1.f);
      }
      gr[i] = v;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int idx = tid + i * 256;
      const int n = idx >> 6, k = idx & 63;
      wr[i] = (n0 + n < n_end && k0 + k < a.K) ? a.W[static_cast<size_t>(n0 + n) * a.K + k0 + k] : 0.f;
    }
  };
  load_tiles(n_begin);
  for (int n0 = n_begin; n0 < n_end; n0 += 32) {
#pragma unroll
    for (int i = 0; i < 4; ++i) Gs[(tid + i * 256) >> 5][(tid + i * 256) & 31] = gr[i];
#pragma unroll
    for (int i = 0; i < 8; ++i) Ws[(tid + i * 256) >> 6][(tid + i * 256) & 63] = wr[i];
    __syncthreads();
    if (n0 + 32 < n_end) load_tiles(n0 + 32);
    float part[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};   // per-tile partial, see linear_f32_kernel
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {   // A = G (rows r, reduction n), B[n][k] = W
      const float af[4] = {Gs[wm * 16 + g][ks * 8 + t], Gs[wm * 16 + g + 8][ks * 8 + t], Gs[wm * 16 + g][ks * 8 + t + 4],
                           Gs[wm * 16 + g + 8][ks * 8 + t + 4]};
#pragma unroll
      for (int j = 0; j < 2; ++j)
        mma_3xtf32(part[j], af, Ws[ks * 8 + t][wn * 16 + j * 8 + g], Ws[ks * 8 + t + 4][wn * 16 + j * 8 + g]);
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
      const int col = k0 + wn * 16 + j * 8 + 2 * t + (e & 1);
      if (row >= a.R || col >= a.K) continue;
      float* d = a.dX + static_cast<size_t>(row) * a.lddx + col;
      if (gridDim.z > 1) atomicAdd(d, acc[j][e]);
      else *d = (a.beta != 0.f ? a.beta * *d : 0.f) + acc[j][e];
    }
  }
}

// dW[n, k] = beta * dW[n, k] + scale * sum_r g[r, n] * x[r, k],  x = relu?(X + x_add[r % mod]);  db[n] likewise
__global__ void __launch_bounds__(256) linear_wgrad_kernel(const LinBwdArgs a) {
  __shared__ float Gs[32][40];   // [r][n]
  __shared__ float Xs[32][72];   // [r][k]
  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  const int wm = warp & 1, wn = warp >> 1;
  const int n0 = blockIdx.y * 32, k0 = blockIdx.x * 64;
  float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
  float bsum = 0.f;  // threads 0..31 of the k-tile-0 CTAs own one bias entry
  // split-R: CTA z reduces rows [z * rows_per_split, ...) and adds its partial tile atomically (outputs pre-zeroed or
  // accumulating, see the host wrapper)
  const int r_begin = blockIdx.z * a.rows_per_split;
  const int r_end = (r_begin + a.rows_per_split < a.R) ? r_begin + a.rows_per_split : a.R;
  // (no register prefetch here: the row split already keeps ~4 CTAs per SM in flight, and the extra registers of a
  // software pipeline cost more occupancy than the overlap returns -- measured 4.4 vs 5.9 ms per c4 backward)
  for (int r0 = r_begin; r0 < r_end; r0 += 32) {
    for (int idx = tid; idx < 32 * 32; idx += 256) {
      const int r = idx >> 5, n = idx & 31;
      float v = 0.f;
      if (r0 + r < r_end && n0 + n < a.N) {
        v = a.dY[static_cast<size_t>(r0 + r) * a.ldy + n0 + n];
        if (a.drop.thr) v *= drop_mult(a.drop, a.drop_site, static_cast<uint64_t>(r0 + r) * a.N + n0 + n);
        if (a.act) v = act_grad(v, a.Y[static_cast<size_t>(r0 + r) * a.ldyo + n0 + n], a.act) * (a.act_scale != 0.f ? a.act_scale : 1.f);
      }
      Gs[r][n] = v;
    }
    for (int idx = tid; idx < 32 * 64; idx += 256) {
      const int r = idx >> 6, k = idx & 63;
      float v = 0.f;
      if (r0 + r < r_end && k0 + k < a.K) {
        v = a.X[static_cast<size_t>(r0 + r) * a.ldx + k0 + k];
        if (a.x_add) v += a.x_add[static_cast<size_t>((r0 + r) % a.add_mod) * a.K + k0 + k];
        if (a.in_relu) v = fmaxf(v, 0.f);
      }
      Xs[r][k] = v;
    }
    __syncthreads();
    float part[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};   // per-tile partial, see linear_f32_kernel
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {   // A[n][r] = G^T (rows n, reduction r), B[r][k] = X
      const float af[4] = {Gs[ks * 8 + t][wm * 16 + g], Gs[ks * 8 + t][wm * 16 + g + 8], Gs[ks * 8 + t + 4][wm * 16 + g],
                           Gs[ks * 8 + t + 4][wm * 16 + g + 8]};
#pragma unroll
      for (int j = 0; j < 2; ++j)
        mma_3xtf32(part[j], af, Xs[ks * 8 + t][wn * 16 + j * 8 + g], Xs[ks * 8 + t + 4][wn * 16 + j * 8 + g]);
    }
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[j][e] += part[j][e];
    if (a.db && blockIdx.x == 0 && tid < 32)
      for (int r = 0; r < 32; ++r) bsum += Gs[r][tid];
    __syncthreads();
  }
#pragma unroll
  for (int j = 0; j < 2; ++j) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int n = n0 + wm * 16 + g + (e >> 1) * 8;
      const int k = k0 + wn * 16 + j * 8 + 2 * t + (e & 1);
      if (n >= a.N || k >= a.K) continue;
      float* d = a.dW + static_cast<size_t>(n) * a.ldw + k;
      if (gridDim.z > 1) atomicAdd(d, a.scale * acc[j][e]);
      else *d = (a.beta != 0.f ? a.beta * *d : 0.f) + a.scale * acc[j][e];
    }
  }
  if (a.db && blockIdx.x == 0 && tid < 32 && n0 + tid < a.N) {
    float* d = a.db + n0 + tid;
    if (gridDim.z > 1) atomicAdd(d, a.scale * bsum);
    else *d = (a.beta != 0.f ? a.beta * *d : 0.f) + a.scale * bsum;
  }
}

// ------------------------------------------------------------------------------------------ LayerNorm backward
// one warp per row (D <= 1024, multiple of 128); per-CTA partial dgamma / dbeta -> part[blockIdx.x][2][D]
constexpr int LNB_MAXV = 8;
__global__ void __launch_bounds__(256)
ln_bwd_kernel(const float* __restrict__ x, int ldx, const bf16* __restrict__ delta, const float* __restrict__ w,
              const float* __restrict__ dy, const float* __restrict__ dy2, const bf16* __restrict__ dy16, int lddy,
              float eps, float beta,
              float* __restrict__ dx, bf16* __restrict__ dx16, float* __restrict__ part, int M, int D) {
  extern __shared__ float sred[];  // [8 warps][2][D]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nv = D >> 7;
  float4 gsum[LNB_MAXV], bsum[LNB_MAXV];
#pragma unroll
  for (int j = 0; j < LNB_MAXV; ++j) gsum[j] = bsum[j] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int row = blockIdx.x * 8 + warp; row < M; row += gridDim.x * 8) {
    float4 v[LNB_MAXV], g[LNB_MAXV];
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < LNB_MAXV; ++j)
      if (j < nv) {
        const int c = (j * 32 + lane) * 4;
        v[j] = *reinterpret_cast<const float4*>(x + static_cast<size_t>(row) * ldx + c);
        if (delta) {
          const uint2 d2 = *reinterpret_cast<const uint2*>(delta + static_cast<size_t>(row) * D + c);
          const float2 a0 = unpack_bf16x2(d2.x), a1 = unpack_bf16x2(d2.y);
          v[j].x += a0.x; v[j].y += a0.y; v[j].z += a1.x; v[j].w += a1.y;
        }
        if (dy) {
          g[j] = *reinterpret_cast<const float4*>(dy + static_cast<size_t>(row) * lddy + c);
          if (dy2) {   // second fp32 addend of the upstream gradient (same pitch)
            const float4 g2 = *reinterpret_cast<const float4*>(dy2 + static_cast<size_t>(row) * lddy + c);
            g[j].x += g2.x; g[j].y += g2.y; g[j].z += g2.z; g[j].w += g2.w;
          }
        } else {
          const uint2 d2 = *reinterpret_cast<const uint2*>(dy16 + static_cast<size_t>(row) * lddy + c);
          const float2 a0 = unpack_bf16x2(d2.x), a1 = unpack_bf16x2(d2.y);
          g[j] = make_float4(a0.x, a0.y, a1.x, a1.y);
        }
        s += v[j].x + v[j].y + v[j].z + v[j].w;
      }
    const float mean = warp_sum(s) / D;
    float q = 0.f;
#pragma unroll
    for (int j = 0; j < LNB_MAXV; ++j)
      if (j < nv) {
        v[j].x -= mean; v[j].y -= mean; v[j].z -= mean; v[j].w -= mean;
        q += v[j].x * v[j].x + v[j].y * v[j].y + v[j].z * v[j].z + v[j].w * v[j].w;
      }
    const float rstd = rsqrtf(warp_sum(q) / D + eps);
    float m1 = 0.f, m2 = 0.f;  // mean(g*w), mean(g*w*xhat)
#pragma unroll
    for (int j = 0; j < LNB_MAXV; ++j)
      if (j < nv) {
        const int c = (j * 32 + lane) * 4;
        const float4 ww = *reinterpret_cast<const float4*>(w + c);
        v[j].x *= rstd; v[j].y *= rstd; v[j].z *= rstd; v[j].w *= rstd;  // xhat
        gsum[j].x += g[j].x * v[j].x; gsum[j].y += g[j].y * v[j].y; gsum[j].z += g[j].z * v[j].z; gsum[j].w += g[j].w * v[j].w;
        bsum[j].x += g[j].x; bsum[j].y += g[j].y; bsum[j].z += g[j].z; bsum[j].w += g[j].w;
        g[j].x *= ww.x; g[j].y *= ww.y; g[j].z *= ww.z; g[j].w *= ww.w;
        m1 += g[j].x + g[j].y + g[j].z + g[j].w;
        m2 += g[j].x * v[j].x + g[j].y * v[j].y + g[j].z * v[j].z + g[j].w * v[j].w;
      }
    m1 = warp_sum(m1) / D;
    m2 = warp_sum(m2) / D;
#pragma unroll
    for (int j = 0; j < LNB_MAXV; ++j)
      if (j < nv) {
        const int c = (j * 32 + lane) * 4;
        float4 o;
        o.x = rstd * (g[j].x - m1 - v[j].x * m2);
        o.y = rstd * (g[j].y - m1 - v[j].y * m2);
        o.z = rstd * (g[j].z - m1 - v[j].z * m2);
        o.w = rstd * (g[j].w - m1 - v[j].w * m2);
        if (dx) {
          float4* d = reinterpret_cast<float4*>(dx + static_cast<size_t>(row) * D + c);
          if (beta != 0.f) {
            const float4 p = *d;
            o.x += beta * p.x; o.y += beta * p.y; o.z += beta * p.z; o.w += beta * p.w;
          }
          *d = o;
        }
        if (dx16) {
          uint2 pk;
          pk.x = pack_bf16x2(o.x, o.y);
          pk.y = pack_bf16x2(o.z, o.w);
          *reinterpret_cast<uint2*>(dx16 + static_cast<size_t>(row) * D + c) = pk;
        }
      }
  }
  if (!part) return;
  float* mine = sred + static_cast<size_t>(warp) * 2 * D;
#pragma unroll
  for (int j = 0; j < LNB_MAXV; ++j)
    if (j < nv) {
      const int c = (j * 32 + lane) * 4;
      *reinterpret_cast<float4*>(mine + c) = gsum[j];
      *reinterpret_cast<float4*>(mine + D + c) = bsum[j];
    }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * D; i += blockDim.x) {
    float t = 0.f;
    for (int ww = 0; ww < 8; ++ww) t += sred[static_cast<size_t>(ww) * 2 * D + i];
    part[static_cast<size_t>(blockIdx.x) * 2 * D + i] = t;
  }
}

// out[c] = beta * out[c] + sum_p part[p][c]   (fixed order)
__global__ void reduce_parts_kernel(const float* __restrict__ part, int P, int n, int stride, float beta,
                                    float* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n) return;
  float t = 0.f;
  for (int p = 0; p < P; ++p) t += part[static_cast<size_t>(p) * stride + c];
  out[c] = (beta != 0.f ? beta * out[c] : 0.f) + t;
}

// ------------------------------------------------------------------------------------------ self-attention backward
// one warp per (clip, head); lane i = query row i
static_assert(kMaxQueries <= 32, "self_attn_bwd_kernel: one lane per query");
__global__ void __launch_bounds__(32)
self_attn_bwd_kernel(const float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v, int ld,
                     const float* __restrict__ dO, float* __restrict__ dq, float* __restrict__ dk, float* __restrict__ dv,
                     int ldg, int Q, int heads, DropCfg drop, uint32_t drop_site) {
  __shared__ float Qs[kMaxQueries][HD + 1], Ks[kMaxQueries][HD + 1], Vs[kMaxQueries][HD + 1], Gs[kMaxQueries][HD + 1];
  __shared__ float Ps[kMaxQueries][kMaxQueries + 1], Ss[kMaxQueries][kMaxQueries + 1];
  const int h = blockIdx.x % heads, b = blockIdx.x / heads;
  const int lane = threadIdx.x;
  for (int i = lane; i < Q * HD; i += 32) {
    const int r = i / HD, d = i - r * HD;
    const size_t src = static_cast<size_t>(b * Q + r) * ld + h * HD + d;
    Qs[r][d] = q[src];
    Ks[r][d] = k[src];
    Vs[r][d] = v[src];
    Gs[r][d] = dO[static_cast<size_t>(b * Q + r) * (heads * HD) + h * HD + d];
  }
  __syncwarp();
  if (lane < Q) {
    float s[kMaxQueries], mx = -INFINITY;
    for (int j = 0; j < Q; ++j) {
      float acc = 0.f;
      for (int d = 0; d < HD; ++d) acc += Qs[lane][d] * Ks[j][d];
      s[j] = acc;
      mx = fmaxf(mx, acc);
    }
    float l = 0.f;
    for (int j = 0; j < Q; ++j) {
      s[j] = __expf(s[j] - mx);
      l += s[j];
    }
    const float inv = 1.f / l;
    // with dropout (training): O = sum_j (m_j p_j) v_j, m_j in {0, 1/(1-p)}: dP_j = m_j (dO . v_j), dV_j gets m_j p_j dO
    float dp[kMaxQueries], mult[kMaxQueries], Dsum = 0.f;
    for (int j = 0; j < Q; ++j) {
      s[j] *= inv;
      mult[j] = drop.thr ? drop_mult(drop, drop_site, (static_cast<uint64_t>(blockIdx.x) * Q + lane) * Q + j) : 1.f;
      float acc = 0.f;
      for (int d = 0; d < HD; ++d) acc += Gs[lane][d] * Vs[j][d];
      dp[j] = acc * mult[j];
      Dsum += s[j] * dp[j];
    }
    for (int j = 0; j < Q; ++j) {
      Ps[lane][j] = s[j] * mult[j];
      Ss[lane][j] = s[j] * (dp[j] - Dsum);
    }
    float* o = dq + static_cast<size_t>(b * Q + lane) * ldg + h * HD;
    for (int d = 0; d < HD; ++d) {
      float acc = 0.f;
      for (int j = 0; j < Q; ++j) acc += Ss[lane][j] * Ks[j][d];
      o[d] = acc;
    }
  }
  __syncwarp();
  if (lane < Q) {
    float* ok = dk + static_cast<size_t>(b * Q + lane) * ldg + h * HD;
    float* ov = dv + static_cast<size_t>(b * Q + lane) * ldg + h * HD;
    for (int d = 0; d < HD; ++d) {
      float ak = 0.f, av = 0.f;
      for (int i = 0; i < Q; ++i) {
        ak += Ss[i][lane] * Qs[i][d];
        av += Ps[i][lane] * Gs[i][d];
      }
      ok[d] = ak;
      ov[d] = av;
    }
  }
}

// ------------------------------------------------------------------------------------------ cross-attention backward
// (i) per (clip, head): lse_i over the S keys -- only when the forward did not keep it (cross_attn's lse_out).  Up to 16
// warps; warp w owns query rows w, w + warps, ...; lanes stride over keys.
constexpr int kStatsWarps = 16;
__global__ void __launch_bounds__(kStatsWarps * 32)
cross_stats_kernel(const float* __restrict__ q, const bf16* __restrict__ K, int ldkv, float* __restrict__ lse, int Q,
                   int heads, int S) {
  __shared__ float qs[kMaxQueries][HD];
  const int h = blockIdx.x % heads, b = blockIdx.x / heads;
  const int C = heads * HD;
  const int tid = threadIdx.x, lane = tid & 31;
  for (int e = tid; e < Q * HD; e += blockDim.x) qs[e / HD][e % HD] = q[static_cast<size_t>(b * Q + e / HD) * C + h * HD + e % HD];
  __syncthreads();
  for (int i = tid >> 5; i < Q; i += blockDim.x >> 5) {
    float m = -INFINITY, sacc = 0.f;
    for (int j = lane; j < S; j += 32) {
      const uint4* kr = reinterpret_cast<const uint4*>(K + (static_cast<size_t>(b) * S + j) * ldkv + h * HD);
      float sc = 0.f;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const uint4 u = kr[c];
        const float2 a0 = unpack_bf16x2(u.x), a1 = unpack_bf16x2(u.y), a2 = unpack_bf16x2(u.z), a3 = unpack_bf16x2(u.w);
        const float* qq = &qs[i][c * 8];
        sc += qq[0] * a0.x + qq[1] * a0.y + qq[2] * a1.x + qq[3] * a1.y + qq[4] * a2.x + qq[5] * a2.y + qq[6] * a3.x + qq[7] * a3.y;
      }
      const float nm = fmaxf(m, sc);
      sacc = sacc * __expf(m - nm) + __expf(sc - nm);
      m = nm;
    }
    for (int o = 16; o; o >>= 1) {
      const float om = __shfl_xor_sync(0xffffffffu, m, o), os = __shfl_xor_sync(0xffffffffu, sacc, o);
      const float nm = fmaxf(m, om);
      sacc = (m == -INFINITY ? 0.f : sacc * __expf(m - nm)) + (om == -INFINITY ? 0.f : os * __expf(om - nm));
      m = nm;
    }
    if (lane == 0) lse[(static_cast<size_t>(b) * heads + h) * Q + i] = m + logf(sacc);
  }
}

// (ii) one thread per key: p_ij, dS_ij, dV_j = sum_i p_ij dO_i, dK_j = sum_i dS_ij q_i;  D_i = dO_i . O_i is recomputed by
// every CTA of the (clip, head) (13 x 64 products) instead of a pass of its own
__global__ void __launch_bounds__(128)
cross_keys_kernel(const float* __restrict__ q, const bf16* __restrict__ K, const bf16* __restrict__ V, int ldkv,
                  const float* __restrict__ dO, const float* __restrict__ O, const float* __restrict__ lse,
                  bf16* __restrict__ dK, bf16* __restrict__ dV, int lddkv, float* __restrict__ dS, int Q, int heads, int S,
                  DropCfg drop, uint32_t drop_site) {
  __shared__ float qs[kMaxQueries][HD], gs[kMaxQueries][HD];
  __shared__ float ls[kMaxQueries], ds_[kMaxQueries];
  const int h = blockIdx.y % heads, b = blockIdx.y / heads;
  const int C = heads * HD;
  for (int i = threadIdx.x; i < Q * HD; i += blockDim.x) {
    qs[i / HD][i % HD] = q[static_cast<size_t>(b * Q + i / HD) * C + h * HD + i % HD];
    gs[i / HD][i % HD] = dO[static_cast<size_t>(b * Q + i / HD) * C + h * HD + i % HD];
  }
  if (threadIdx.x < Q) ls[threadIdx.x] = lse[(static_cast<size_t>(b) * heads + h) * Q + threadIdx.x];
  for (int i = threadIdx.x >> 5; i < Q; i += 4) {
    const int lane = threadIdx.x & 31;
    const float* g = dO + static_cast<size_t>(b * Q + i) * C + h * HD;
    const float* o = O + static_cast<size_t>(b * Q + i) * C + h * HD;
    const float t = warp_sum(g[lane] * o[lane] + g[lane + 32] * o[lane + 32]);
    if (lane == 0) ds_[i] = t;
  }
  __syncthreads();
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= S) return;
  const size_t rowoff = (static_cast<size_t>(b) * S + j);
  float p[kMaxQueries], dsv[kMaxQueries];
  {
    float kf[HD], vf[HD];
    const uint4* kr = reinterpret_cast<const uint4*>(K + rowoff * ldkv + h * HD);
    const uint4* vr = reinterpret_cast<const uint4*>(V + rowoff * ldkv + h * HD);
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      uint4 u = kr[c];
      float2 a0 = unpack_bf16x2(u.x), a1 = unpack_bf16x2(u.y), a2 = unpack_bf16x2(u.z), a3 = unpack_bf16x2(u.w);
      kf[c * 8 + 0] = a0.x; kf[c * 8 + 1] = a0.y; kf[c * 8 + 2] = a1.x; kf[c * 8 + 3] = a1.y;
      kf[c * 8 + 4] = a2.x; kf[c * 8 + 5] = a2.y; kf[c * 8 + 6] = a3.x; kf[c * 8 + 7] = a3.y;
      u = vr[c];
      a0 = unpack_bf16x2(u.x); a1 = unpack_bf16x2(u.y); a2 = unpack_bf16x2(u.z); a3 = unpack_bf16x2(u.w);
      vf[c * 8 + 0] = a0.x; vf[c * 8 + 1] = a0.y; vf[c * 8 + 2] = a1.x; vf[c * 8 + 3] = a1.y;
      vf[c * 8 + 4] = a2.x; vf[c * 8 + 5] = a2.y; vf[c * 8 + 6] = a3.x; vf[c * 8 + 7] = a3.y;
    }
#pragma unroll
    for (int i = 0; i < kMaxQueries; ++i) {
      p[i] = dsv[i] = 0.f;
      if (i < Q) {
        float s = 0.f, dp = 0.f;
#pragma unroll
        for (int d = 0; d < HD; ++d) {
          s += qs[i][d] * kf[d];
          dp += gs[i][d] * vf[d];
        }
        p[i] = __expf(s - ls[i]);
        // dropout on the probabilities (training): dP = m (dO . v), dV weight = m p;  D_i = dO_i . O_i is unchanged
        const float mult = drop.thr ? drop_mult(drop, drop_site, ((static_cast<uint64_t>(b) * heads + h) * Q + i) * S + j) : 1.f;
        dsv[i] = p[i] * (mult * dp - ds_[i]);
        dS[((static_cast<size_t>(b) * heads + h) * Q + i) * S + j] = dsv[i];
        p[i] *= mult;
      }
    }
  }
  uint32_t* okv = reinterpret_cast<uint32_t*>(dV + rowoff * lddkv + h * HD);
  uint32_t* okk = reinterpret_cast<uint32_t*>(dK + rowoff * lddkv + h * HD);
#pragma unroll 4
  for (int d = 0; d < HD; d += 2) {
    float v0 = 0.f, v1 = 0.f, k0 = 0.f, k1 = 0.f;
#pragma unroll
    for (int i = 0; i < kMaxQueries; ++i)
      if (i < Q) {
        v0 += p[i] * gs[i][d];
        v1 += p[i] * gs[i][d + 1];
        k0 += dsv[i] * qs[i][d];
        k1 += dsv[i] * qs[i][d + 1];
      }
    okv[d >> 1] = pack_bf16x2(v0, v1);
    okk[d >> 1] = pack_bf16x2(k0, k1);
  }
}

// (iii) dQ[b, i, h*64 + d] = sum_j dS[b,h,i,j] * K[b, j, h*64 + d]
__global__ void __launch_bounds__(256)
cross_dq_kernel(const float* __restrict__ dS, const bf16* __restrict__ K, int ldkv, float* __restrict__ dq, int Q, int heads,
                int S) {
  __shared__ float part[4][kMaxQueries][HD];
  const int h = blockIdx.x % heads, b = blockIdx.x / heads;
  const int C = heads * HD;
  const int d = threadIdx.x & 63, grp = threadIdx.x >> 6;  // 4 key groups x 64 dims
  float acc[kMaxQueries];
#pragma unroll
  for (int i = 0; i < kMaxQueries; ++i) acc[i] = 0.f;
  const float* ds = dS + (static_cast<size_t>(b) * heads + h) * Q * S;
  for (int j = grp; j < S; j += 4) {
    const float kv = __bfloat162float(K[(static_cast<size_t>(b) * S + j) * ldkv + h * HD + d]);
#pragma unroll
    for (int i = 0; i < kMaxQueries; ++i)
      if (i < Q) acc[i] += ds[static_cast<size_t>(i) * S + j] * kv;
  }
#pragma unroll
  for (int i = 0; i < kMaxQueries; ++i) part[grp][i][d] = acc[i];
  __syncthreads();
  for (int idx = threadIdx.x; idx < Q * HD; idx += 256) {
    const int i = idx / HD, dd = idx - i * HD;
    dq[static_cast<size_t>(b * Q + i) * C + h * HD + dd] = part[0][i][dd] + part[1][i][dd] + part[2][i][dd] + part[3][i][dd];
  }
}

// ------------------------------------------------------------------------------------------ reductions / layouts
// part[gy][c] = sum over the gy-th slice of rows of X[r, c]
template <typename T>
__global__ void __launch_bounds__(256)
colsum_part_kernel(const T* __restrict__ X, long long ld, long long rows, long long cols, float* __restrict__ part) {
  const long long c = blockIdx.x * 256LL + threadIdx.x;
  if (c >= cols) return;
  const long long per = (rows + gridDim.y - 1) / gridDim.y;
  const long long r0 = blockIdx.y * per, r1 = (r0 + per < rows) ? r0 + per : rows;
  float t = 0.f;
  for (long long r = r0; r < r1; ++r) {
    if constexpr (sizeof(T) == 2) t += __bfloat162float(X[r * ld + c]);
    else t += X[r * ld + c];
  }
  part[blockIdx.y * cols + c] = t;
}

// out bf16 [cols, rows] = transpose(in [rows, cols])   (in fp32 or bf16)
template <typename T>
__global__ void __launch_bounds__(256)
transpose_bf16_kernel(const T* __restrict__ in, long long ld, bf16* __restrict__ out, long long rows, long long cols) {
  __shared__ float tile[32][33];
  const long long c0 = blockIdx.x * 32LL, r0 = blockIdx.y * 32LL;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int i = ty; i < 32; i += 8) {
    const long long r = r0 + i, c = c0 + tx;
    float v = 0.f;
    if (r < rows && c < cols) {
      if constexpr (sizeof(T) == 2) v = __bfloat162float(in[r * ld + c]);
      else v = in[r * ld + c];
    }
    tile[i][tx] = v;
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const long long c = c0 + i, r = r0 + tx;
    if (r < rows && c < cols) out[c * rows + r] = __float2bfloat16(tile[tx][i]);
  }
}

// bf16 -> bf16, every dimension a multiple of 8: 64 x 64 tiles, 16-byte global loads and stores (the element-wise kernel
// above moved the 403 MB all-layer dK / dV matrices at 1.7 TB/s)
__global__ void __launch_bounds__(256)
transpose_bf16x8_kernel(const bf16* __restrict__ in, long long ld, bf16* __restrict__ out, long long rows, long long cols) {
  __shared__ __align__(16) bf16 tile[64][72];
  const long long c0 = blockIdx.x * 64LL, r0 = blockIdx.y * 64LL;
  for (int i = threadIdx.x; i < 512; i += 256) {
    const int r = i >> 3, ch = i & 7;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (r0 + r < rows && c0 + ch * 8 < cols) v = *reinterpret_cast<const uint4*>(in + (r0 + r) * ld + c0 + ch * 8);
    *reinterpret_cast<uint4*>(&tile[r][ch * 8]) = v;
  }
  __syncthreads();
  const uint16_t* t16 = reinterpret_cast<const uint16_t*>(&tile[0][0]);
  for (int i = threadIdx.x; i < 512; i += 256) {
    const int c = (i >> 1) & 63, rh = ((i >> 7) << 1) | (i & 1);   // two lanes fill one 32-byte sector of an output row
    if (c0 + c < cols && r0 + rh * 8 < rows) {
      uint32_t w[4];
#pragma unroll
      for (int k = 0; k < 4; ++k)
        w[k] = static_cast<uint32_t>(t16[(rh * 8 + 2 * k) * 72 + c]) | (static_cast<uint32_t>(t16[(rh * 8 + 2 * k + 1) * 72 + c]) << 16);
      *reinterpret_cast<uint4*>(out + (c0 + c) * rows + r0 + rh * 8) = make_uint4(w[0], w[1], w[2], w[3]);
    }
  }
}

}  // namespace

// ================================================================================================ host wrappers
int linear_dgrad_f32_legacy(const LinBwdArgs& a_in, cudaStream_t s) {
  LinBwdArgs a = a_in;
  HH_REQUIRE(a.R > 0 && a.N > 0 && a.K > 0 && a.dY && a.W && a.dX, "linear_dgrad: bad argument");
  HH_REQUIRE(a.act == 0 || a.Y != nullptr, "linear_dgrad: activation derivative needs the saved output");
  dim3 grid((a.K + 63) / 64, (a.R + 31) / 32);
  // Few output tiles but a long reduction (FFN: N = 2048 against 208 tiles): split the reduction over gridDim.z so that
  // ~4 CTAs per SM are in flight; partial tiles are combined with fp32 atomics (last bits vary from run to run, as for
  // the weight gradients).
  int split = (4 * num_sms() + static_cast<int>(grid.x * grid.y) - 1) / static_cast<int>(grid.x * grid.y);
  const int max_split = a.N / 256;  // at least 256 reduction steps per CTA
  if (split > max_split) split = max_split;
  if (split < 1 || (a.beta != 0.f && a.beta != 1.f)) split = 1;
  a.rows_per_split = ((a.N + split - 1) / split + 31) / 32 * 32;   // (field shared with wgrad's row split)
  split = (a.N + a.rows_per_split - 1) / a.rows_per_split;
  grid.z = split;
  if (split > 1 && a.beta == 0.f)
    HH_CHECK_CUDA(cudaMemset2DAsync(a.dX, static_cast<size_t>(a.lddx) * 4, 0, static_cast<size_t>(a.K) * 4, a.R, s));
  linear_dgrad_kernel<<<grid, 256, 0, s>>>(a);
  HH_CHECK_LAUNCH("linear_dgrad_kernel");
  return 0;
}

int linear_wgrad_f32_legacy(const LinBwdArgs& a_in, cudaStream_t s) {
  LinBwdArgs a = a_in;
  HH_REQUIRE(a.R > 0 && a.N > 0 && a.K > 0 && a.dY && a.X && a.dW, "linear_wgrad: bad argument");
  HH_REQUIRE(a.act == 0 || a.Y != nullptr, "linear_wgrad: activation derivative needs the saved output");
  dim3 grid((a.K + 63) / 64, (a.N + 31) / 32);
  // Few output tiles but many rows: split the row reduction over gridDim.z so that ~4 CTAs per SM are in flight; the
  // partial tiles are combined with fp32 atomics (summation order, hence the last bits, vary from run to run).
  int split = (4 * num_sms() + static_cast<int>(grid.x * grid.y) - 1) / static_cast<int>(grid.x * grid.y);
  const int max_split = (a.R + 127) / 128;  // at least 128 rows per CTA
  if (split > max_split) split = max_split;
  if (split > 64) split = 64;
  if (split < 1 || (a.beta != 0.f && a.beta != 1.f)) split = 1;
  a.rows_per_split = ((a.R + split - 1) / split + 31) / 32 * 32;
  split = (a.R + a.rows_per_split - 1) / a.rows_per_split;
  grid.z = split;
  if (split > 1 && a.beta == 0.f) {
    HH_CHECK_CUDA(cudaMemset2DAsync(a.dW, static_cast<size_t>(a.ldw) * 4, 0, static_cast<size_t>(a.K) * 4, a.N, s));
    if (a.db) HH_CHECK_CUDA(cudaMemsetAsync(a.db, 0, static_cast<size_t>(a.N) * 4, s));
  }
  linear_wgrad_kernel<<<grid, 256, 0, s>>>(a);
  HH_CHECK_LAUNCH("linear_wgrad_kernel");
  return 0;
}

size_t ln_backward_workspace_bytes(int M, int D) {
  int blocks = (M + 7) / 8;
  const int cap = num_sms() * 4;
  if (blocks > cap) blocks = cap;
  return static_cast<size_t>(blocks) * 2 * D * sizeof(float);
}

int ln_backward_rows(const LnBwdArgs& a, cudaStream_t s) {
  HH_REQUIRE(a.M > 0 && a.D % 128 == 0 && a.D <= 128 * LNB_MAXV, "ln_backward: D must be a multiple of 128, <= 1024");
  HH_REQUIRE(a.x && a.w && (a.dy || a.dy16) && (a.dx || a.dx16), "ln_backward: null buffer");
  HH_REQUIRE((a.dgamma == nullptr) == (a.dbeta == nullptr), "ln_backward: dgamma and dbeta go together");
  HH_REQUIRE(a.dgamma == nullptr || a.workspace != nullptr, "ln_backward: workspace");
  int blocks = (a.M + 7) / 8;
  const int cap = num_sms() * 4;
  if (blocks > cap) blocks = cap;
  const size_t smem = static_cast<size_t>(8) * 2 * a.D * sizeof(float);
  static bool configured = false;
  if (!configured) {
    HH_CHECK_CUDA(cudaFuncSetAttribute(ln_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * 2 * 1024 * 4));
    configured = true;
  }
  float* part = a.dgamma ? static_cast<float*>(a.workspace) : nullptr;
  ln_bwd_kernel<<<blocks, 256, smem, s>>>(a.x, a.ldx, a.delta, a.w, a.dy, a.dy2, a.dy16, a.lddy, a.eps, a.beta_dx, a.dx, a.dx16, part,
                                          a.M, a.D);
  HH_CHECK_LAUNCH("ln_bwd_kernel");
  if (a.dgamma) {
    reduce_parts_kernel<<<(a.D + 255) / 256, 256, 0, s>>>(part, blocks, a.D, 2 * a.D, a.beta_w, a.dgamma);
    reduce_parts_kernel<<<(a.D + 255) / 256, 256, 0, s>>>(part + a.D, blocks, a.D, 2 * a.D, a.beta_w, a.dbeta);
    HH_CHECK_LAUNCH("reduce_parts_kernel");
  }
  return 0;
}

int self_attn_bwd(const float* q, const float* k, const float* v, int ld, const float* dO, float* dq, float* dk, float* dv,
                  int ldg, int B, int Q, int heads, cudaStream_t s, DropCfg drop, uint32_t drop_site) {
  HH_REQUIRE(B > 0 && Q >= 1 && Q <= kMaxQueries && heads > 0, "self_attn_bwd: 1..32 queries");
  self_attn_bwd_kernel<<<B * heads, 32, 0, s>>>(q, k, v, ld, dO, dq, dk, dv, ldg, Q, heads, drop, drop_site);
  HH_CHECK_LAUNCH("self_attn_bwd_kernel");
  return 0;
}

size_t cross_attn_bwd_simt_workspace_bytes(int B, int Q, int heads, int S) {
  return static_cast<size_t>(B) * heads * Q * (static_cast<size_t>(S) + 1) * sizeof(float);
}

int cross_lse(const float* q, const bf16* K, int ldkv, float* lse, int B, int Q, int heads, int S, cudaStream_t s) {
  HH_REQUIRE(Q >= 1 && Q <= kMaxQueries, "cross_lse: 1..32 queries");
  cross_stats_kernel<<<B * heads, 32 * (Q < kStatsWarps ? Q : kStatsWarps), 0, s>>>(q, K, ldkv, lse, Q, heads, S);
  HH_CHECK_LAUNCH("cross_stats_kernel");
  return 0;
}

int cross_attn_bwd_simt(const float* q, const bf16* K, const bf16* V, int ldkv, const float* O, const float* dO, float* dq,
                        bf16* dK, bf16* dV, int lddkv, int B, int Q, int heads, int S, void* workspace, cudaStream_t s,
                        DropCfg drop, uint32_t drop_site, const float* lse_saved) {
  HH_REQUIRE(B > 0 && Q >= 1 && Q <= kMaxQueries && heads > 0 && S > 0, "cross_attn_bwd: 1..32 queries");
  float* lse_ws = static_cast<float*>(workspace);
  float* dS = lse_ws + static_cast<size_t>(B) * heads * Q;
  const float* lse = lse_saved;
  if (lse == nullptr) {
    if (int rc = cross_lse(q, K, ldkv, lse_ws, B, Q, heads, S, s)) return rc;
    lse = lse_ws;
  }
  dim3 grid((S + 127) / 128, B * heads);
  cross_keys_kernel<<<grid, 128, 0, s>>>(q, K, V, ldkv, dO, O, lse, dK, dV, lddkv, dS, Q, heads, S, drop, drop_site);
  cross_dq_kernel<<<B * heads, 256, 0, s>>>(dS, K, ldkv, dq, Q, heads, S);
  HH_CHECK_LAUNCH("cross_attn_bwd kernels");
  return 0;
}

size_t colsum_workspace_bytes(long long cols) { return static_cast<size_t>(64) * cols * sizeof(float); }

int colsum_rows(const void* X, int is_bf16, long long ld, long long rows, long long cols, float beta, float* out,
                void* workspace, cudaStream_t s) {
  HH_REQUIRE(rows > 0 && cols > 0 && X && out && workspace, "colsum_rows: bad argument");
  const int gy = rows < 64 ? static_cast<int>(rows) : 64;
  dim3 grid(static_cast<unsigned>((cols + 255) / 256), gy);
  float* part = static_cast<float*>(workspace);
  if (is_bf16) colsum_part_kernel<bf16><<<grid, 256, 0, s>>>(static_cast<const bf16*>(X), ld, rows, cols, part);
  else colsum_part_kernel<float><<<grid, 256, 0, s>>>(static_cast<const float*>(X), ld, rows, cols, part);
  reduce_parts_kernel<<<static_cast<unsigned>((cols + 255) / 256), 256, 0, s>>>(part, gy, static_cast<int>(cols),
                                                                               static_cast<int>(cols), beta, out);
  HH_CHECK_LAUNCH("colsum kernels");
  return 0;
}

int transpose_to_bf16(const void* in, int is_bf16, long long ld, bf16* out, long long rows, long long cols, cudaStream_t s) {
  HH_REQUIRE(rows > 0 && cols > 0 && in && out, "transpose_to_bf16: bad argument");
  if (is_bf16 && rows % 8 == 0 && cols % 8 == 0 && ld % 8 == 0 && (reinterpret_cast<uintptr_t>(in) & 15) == 0 &&
      (reinterpret_cast<uintptr_t>(out) & 15) == 0 && (rows + 63) / 64 < 65536) {
    dim3 g8(static_cast<unsigned>((cols + 63) / 64), static_cast<unsigned>((rows + 63) / 64));
    transpose_bf16x8_kernel<<<g8, 256, 0, s>>>(static_cast<const bf16*>(in), ld, out, rows, cols);
    HH_CHECK_LAUNCH("transpose_bf16x8_kernel");
    return 0;
  }
  dim3 grid(static_cast<unsigned>((cols + 31) / 32), static_cast<unsigned>((rows + 31) / 32));
  HH_REQUIRE(grid.y < 65536, "transpose_to_bf16: too many rows");
  if (is_bf16) transpose_bf16_kernel<bf16><<<grid, 256, 0, s>>>(static_cast<const bf16*>(in), ld, out, rows, cols);
  else transpose_bf16_kernel<float><<<grid, 256, 0, s>>>(static_cast<const float*>(in), ld, out, rows, cols);
  HH_CHECK_LAUNCH("transpose_bf16_kernel");
  return 0;
}

}  // namespace hh
