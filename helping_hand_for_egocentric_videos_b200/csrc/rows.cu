// Row-wise HBM-bound kernels: LayerNorm (fp32 in, fp32 statistics, bf16 and/or fp32 out) and fp32->bf16 row gathers.
// One warp per row, 128-bit loads, two-pass statistics held in registers (mean, then centred variance), matching
// torch.nn.LayerNorm's biased variance (model/LaviLa.py:439,456,570; model/tfm_decoder.py:57,61,375-377).
#include "hh_internal.h"
#include "hh_ptx.cuh"

namespace hh {

namespace {

constexpr int LN_MAX_VEC = 8;  // D <= 8 * 128 = 1024

__global__ void __launch_bounds__(256) ln_rows_kernel(const LnArgs a) {
  const int warp_lin = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp_lin >= a.M) return;
  // Rows are walked from the END of the matrix: the GEMM that produced `delta` wrote its last row tiles last, so they
  // are still in the 126 MB L2, and the GEMM that follows reads the rows written last here (the first ones) first.
  // Measured +0.5 ... 0.7 % clips/s with the same walk in the attention kernels (A/B on one box against a forward walk).
  const int warp = a.M - 1 - warp_lin;
  const int nv = a.D >> 7;  // float4 per lane
  const float* xr = a.x + static_cast<size_t>(warp) * a.ldx;
  float4 v[LN_MAX_VEC];
  uint2 dv[LN_MAX_VEC];
  float s = 0.f;
  // All loads of the row are issued before anything is stored: xsum_out may alias x, and a store in between would
  // serialise the loads behind it.  Streaming (evict-first) accesses: every byte here is touched exactly once.
#pragma unroll
  for (int j = 0; j < LN_MAX_VEC; ++j)
    if (j < nv) v[j] = __ldcs(reinterpret_cast<const float4*>(xr + (j * 32 + lane) * 4));
  if (a.delta) {  // residual branch output (bf16) folded in here: x <- x + delta
    const bf16* dr = a.delta + static_cast<size_t>(warp) * a.D;
#pragma unroll
    for (int j = 0; j < LN_MAX_VEC; ++j)
      if (j < nv) dv[j] = __ldcs(reinterpret_cast<const uint2*>(dr + (j * 32 + lane) * 4));
#pragma unroll
    for (int j = 0; j < LN_MAX_VEC; ++j) {
      if (j < nv) {
        const float2 d0 = unpack_bf16x2(dv[j].x), d1 = unpack_bf16x2(dv[j].y);
        v[j].x += d0.x; v[j].y += d0.y; v[j].z += d1.x; v[j].w += d1.y;
      }
    }
    if (a.delta2) {  // second pending branch output, added after the first: (x + delta) + delta2
      const bf16* dr2 = a.delta2 + static_cast<size_t>(warp) * a.D;
#pragma unroll
      for (int j = 0; j < LN_MAX_VEC; ++j)
        if (j < nv) dv[j] = __ldcs(reinterpret_cast<const uint2*>(dr2 + (j * 32 + lane) * 4));
#pragma unroll
      for (int j = 0; j < LN_MAX_VEC; ++j) {
        if (j < nv) {
          const float2 d0 = unpack_bf16x2(dv[j].x), d1 = unpack_bf16x2(dv[j].y);
          v[j].x += d0.x; v[j].y += d0.y; v[j].z += d1.x; v[j].w += d1.y;
        }
      }
    }
    if (a.xsum_out) {
      float* xo = a.xsum_out + static_cast<size_t>(warp) * a.D;
#pragma unroll
      for (int j = 0; j < LN_MAX_VEC; ++j)
        if (j < nv) __stcs(reinterpret_cast<float4*>(xo + (j * 32 + lane) * 4), v[j]);
    }
  }
#pragma unroll
  for (int j = 0; j < LN_MAX_VEC; ++j)
    if (j < nv) s += (v[j].x + v[j].y) + (v[j].z + v[j].w);
  const float mean = warp_sum(s) / static_cast<float>(a.D);
  float ss = 0.f;
#pragma unroll
  for (int j = 0; j < LN_MAX_VEC; ++j) {
    if (j < nv) {
      v[j].x -= mean; v[j].y -= mean; v[j].z -= mean; v[j].w -= mean;
      ss += (v[j].x * v[j].x + v[j].y * v[j].y) + (v[j].z * v[j].z + v[j].w * v[j].w);
    }
  }
  const float rstd = rsqrtf(warp_sum(ss) / static_cast<float>(a.D) + a.eps);
  const size_t orow = static_cast<size_t>(warp) * a.D;
  const float* padd = a.post_add ? a.post_add + static_cast<size_t>(warp % a.post_mod) * a.D : nullptr;
  float* const crow = (a.cls_f32 && warp % a.cls_mod == 0) ? a.cls_f32 + static_cast<size_t>(warp / a.cls_mod) * a.D : nullptr;
#pragma unroll
  for (int j = 0; j < LN_MAX_VEC; ++j) {
    if (j < nv) {
      const int c = (j * 32 + lane) * 4;
      const float4 w = __ldg(reinterpret_cast<const float4*>(a.w + c));  // read-only path: not ordered behind the stores
      const float4 b = __ldg(reinterpret_cast<const float4*>(a.b + c));
      float4 y;
      y.x = v[j].x * rstd * w.x + b.x;
      y.y = v[j].y * rstd * w.y + b.y;
      y.z = v[j].z * rstd * w.z + b.z;
      y.w = v[j].w * rstd * w.w + b.w;
      if (a.out_f32) *reinterpret_cast<float4*>(a.out_f32 + orow + c) = y;
      if (crow) *reinterpret_cast<float4*>(crow + c) = y;
      if (a.out_bf16) {
        uint2 pk = make_uint2(pack_bf16x2(y.x, y.y), pack_bf16x2(y.z, y.w));
        *reinterpret_cast<uint2*>(a.out_bf16 + orow + c) = pk;
      }
      if (padd) {
        const float4 q = *reinterpret_cast<const float4*>(padd + c);
        y.x += q.x; y.y += q.y; y.z += q.z; y.w += q.w;
        if (a.out2_f32) *reinterpret_cast<float4*>(a.out2_f32 + orow + c) = y;
        if (a.out2_bf16) {
          uint2 pk = make_uint2(pack_bf16x2(y.x, y.y), pack_bf16x2(y.z, y.w));
          *reinterpret_cast<uint2*>(a.out2_bf16 + orow + c) = pk;
        }
      }
    }
  }
}

// 4 columns per step: float4 -> packed bf16 (fp32 rows) or a plain 8-byte copy (bf16 rows, the gather alone)
__device__ __forceinline__ uint2 load4_bf16(const float* s) {
  const float4 v = *reinterpret_cast<const float4*>(s);
  return make_uint2(pack_bf16x2(v.x, v.y), pack_bf16x2(v.z, v.w));
}
__device__ __forceinline__ uint2 load4_bf16(const bf16* s) { return *reinterpret_cast<const uint2*>(s); }

template <typename Src>
__global__ void __launch_bounds__(256) cast_rows_kernel(const Src* __restrict__ src, long long outer_stride,
                                                        long long row_stride, int inner, bf16* __restrict__ dst,
                                                        int rows, int cols) {
  const int vec_per_row = cols >> 2;
  const long long total = static_cast<long long>(rows) * vec_per_row;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int r = static_cast<int>(i / vec_per_row);
    const int c = static_cast<int>(i - static_cast<long long>(r) * vec_per_row) * 4;
    const Src* s = src + (r / inner) * outer_stride + (r % inner) * row_stride + c;
    *reinterpret_cast<uint2*>(dst + static_cast<size_t>(r) * cols + c) = load4_bf16(s);
  }
}

__global__ void __launch_bounds__(256) f32_to_bf16_kernel(const float* __restrict__ src, bf16* __restrict__ dst,
                                                          size_t n4) {
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const float4 v = reinterpret_cast<const float4*>(src)[i];
    reinterpret_cast<uint2*>(dst)[i] = make_uint2(pack_bf16x2(v.x, v.y), pack_bf16x2(v.z, v.w));
  }
}

__global__ void __launch_bounds__(256)
pack_weight_kernel(const float* __restrict__ src, bf16* __restrict__ dst, int rows, int cols_in, int cols_out,
                   int scaled_rows, float scale) {
  const long long total = static_cast<long long>(rows) * cols_out;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int r = static_cast<int>(i / cols_out), c = static_cast<int>(i % cols_out);
    float v = (c < cols_in) ? src[static_cast<size_t>(r) * cols_in + c] : 0.f;
    if (r < scaled_rows) v *= scale;
    dst[i] = __float2bfloat16(v);
  }
}

// LayerNorm folded into the following nn.Linear (model/LaviLa.py:353,372,388): with z the un-normalised row,
//   Linear(LN(z)) = rstd * (z W'^T - mean * colsum) + bias',  W'[r,k] = W[r,k] gamma[k],  bias'[r] = bias[r] + sum_k W[r,k] beta[k],
// colsum[r] = sum_k W'[r,k] taken over the bf16-ROUNDED W' (the values the tensor cores multiply), so that a constant row
// z = c maps to exactly bias'.  One warp per weight row; rows below `scaled_rows` (the q third) also carry `scale`.
__global__ void __launch_bounds__(256)
fold_ln_weight_kernel(const float* __restrict__ W, const float* __restrict__ gamma, const float* __restrict__ beta,
                      const float* __restrict__ bias, bf16* __restrict__ Wf, float* __restrict__ colsum,
                      float* __restrict__ bias_f, int rows, int K, int scaled_rows, float scale) {
  const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= rows) return;
  const float sc = r < scaled_rows ? scale : 1.f;
  const float* wr = W + static_cast<size_t>(r) * K;
  float cs = 0.f, bb = 0.f;
  for (int k = lane; k < K; k += 32) {
    const float w = wr[k];
    const bf16 wf = __float2bfloat16(w * gamma[k] * sc);
    Wf[static_cast<size_t>(r) * K + k] = wf;
    cs += __bfloat162float(wf);
    bb = fmaf(w, beta[k], bb);
  }
  cs = warp_sum(cs);
  bb = warp_sum(bb);
  if (lane == 0) {
    colsum[r] = cs;
    bias_f[r] = ((bias ? bias[r] : 0.f) + bb) * sc;
  }
}

__global__ void __launch_bounds__(256)
scale_copy_kernel(const float* __restrict__ src, float* __restrict__ dst, size_t n, size_t scaled, float scale) {
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x)
    dst[i] = (i < scaled) ? src[i] * scale : src[i];
}

__global__ void __launch_bounds__(256)
slice_cols_kernel(const float* __restrict__ src, int lds, int col0, float* __restrict__ dst, int rows, int cols) {
  const long long total = static_cast<long long>(rows) * cols;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int r = static_cast<int>(i / cols), c = static_cast<int>(i % cols);
    dst[i] = src[static_cast<size_t>(r) * lds + col0 + c];
  }
}

__global__ void __launch_bounds__(256)
build_pos3d_kernel(const float* __restrict__ pos_embed, const float* __restrict__ temporal, float* __restrict__ out,
                   int T, int n, int C) {
  const long long total = static_cast<long long>(T) * n * C;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % C);
    const int s = static_cast<int>(i / C);
    const int t = s / n, p = s - t * n;
    out[i] = pos_embed[static_cast<size_t>(1 + p) * C + c] + temporal[static_cast<size_t>(t) * C + c];
  }
}

__global__ void __launch_bounds__(256)
l2norm_rows_kernel(const float* __restrict__ x, float* __restrict__ out, int rows, int cols, float eps) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* xr = x + static_cast<size_t>(row) * cols;
  float ss = 0.f;
  for (int c = lane; c < cols; c += 32) ss += xr[c] * xr[c];
  const float nrm = fmaxf(sqrtf(warp_sum(ss)), eps);
  for (int c = lane; c < cols; c += 32) out[static_cast<size_t>(row) * cols + c] = xr[c] / nrm;
}

int grid_for(long long n) {
  long long blocks = (n + 255) / 256;
  const long long cap = static_cast<long long>(num_sms()) * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return static_cast<int>(blocks);
}

}  // namespace

int pack_weight_bf16(const float* src, bf16* dst, int rows, int cols_in, int cols_out, int scaled_rows, float scale,
                     cudaStream_t stream) {
  HH_REQUIRE(rows > 0 && cols_in > 0 && cols_out >= cols_in, "pack_weight_bf16: shape");
  pack_weight_kernel<<<grid_for(static_cast<long long>(rows) * cols_out), 256, 0, stream>>>(src, dst, rows, cols_in,
                                                                                          cols_out, scaled_rows, scale);
  HH_CHECK_LAUNCH("pack_weight_kernel");
  return 0;
}

int fold_ln_weight(const float* W, const float* gamma, const float* beta, const float* bias, bf16* Wf, float* colsum,
                   float* bias_f, int rows, int K, int scaled_rows, float scale, cudaStream_t stream) {
  HH_REQUIRE(rows > 0 && K > 0 && W && gamma && beta && Wf && colsum && bias_f, "fold_ln_weight: bad arguments");
  fold_ln_weight_kernel<<<(rows + 7) / 8, 256, 0, stream>>>(W, gamma, beta, bias, Wf, colsum, bias_f, rows, K, scaled_rows,
                                                           scale);
  HH_CHECK_LAUNCH("fold_ln_weight_kernel");
  return 0;
}

int scale_copy_f32(const float* src, float* dst, size_t n, size_t scaled, float scale, cudaStream_t stream) {
  if (n == 0) return 0;
  scale_copy_kernel<<<grid_for(static_cast<long long>(n)), 256, 0, stream>>>(src, dst, n, scaled, scale);
  HH_CHECK_LAUNCH("scale_copy_kernel");
  return 0;
}

int slice_cols_f32(const float* src, int lds, int col0, float* dst, int rows, int cols, cudaStream_t stream) {
  slice_cols_kernel<<<grid_for(static_cast<long long>(rows) * cols), 256, 0, stream>>>(src, lds, col0, dst, rows, cols);
  HH_CHECK_LAUNCH("slice_cols_kernel");
  return 0;
}

int build_pos3d(const float* pos_embed, const float* temporal, float* out, int T, int n, int C, cudaStream_t stream) {
  build_pos3d_kernel<<<grid_for(static_cast<long long>(T) * n * C), 256, 0, stream>>>(pos_embed, temporal, out, T, n, C);
  HH_CHECK_LAUNCH("build_pos3d_kernel");
  return 0;
}

int l2_normalize_rows(const float* x, float* out, int rows, int cols, float eps, cudaStream_t stream) {
  HH_REQUIRE(rows > 0 && cols > 0, "l2_normalize_rows: empty");
  l2norm_rows_kernel<<<(rows + 7) / 8, 256, 0, stream>>>(x, out, rows, cols, eps);
  HH_CHECK_LAUNCH("l2norm_rows_kernel");
  return 0;
}

int layernorm_rows(const LnArgs& a, cudaStream_t stream) {
  HH_REQUIRE(a.M > 0, "layernorm_rows: no rows");
  HH_REQUIRE(a.D % 128 == 0 && a.D <= 128 * LN_MAX_VEC, "layernorm_rows: D must be a multiple of 128, at most 1024");
  HH_REQUIRE(a.ldx % 4 == 0, "layernorm_rows: ldx must be a multiple of 4");
  HH_REQUIRE(a.post_add == nullptr || a.post_mod > 0, "layernorm_rows: post_mod");
  const int rows_per_block = 8;
  const int grid = (a.M + rows_per_block - 1) / rows_per_block;
  ln_rows_kernel<<<grid, rows_per_block * 32, 0, stream>>>(a);
  HH_CHECK_LAUNCH("ln_rows_kernel");
  return 0;
}

template <typename Src>
static int cast_rows_impl(const Src* src, long long outer_stride, long long row_stride, int inner, bf16* dst, int rows,
                          int cols, cudaStream_t stream) {
  HH_REQUIRE(rows > 0 && cols > 0 && cols % 4 == 0, "cast_rows_bf16: cols must be a multiple of 4");
  HH_REQUIRE(outer_stride % 4 == 0 && row_stride % 4 == 0, "cast_rows_bf16: strides must keep 4-element alignment");
  HH_REQUIRE((reinterpret_cast<uintptr_t>(src) & (4 * sizeof(Src) - 1)) == 0, "cast_rows_bf16: misaligned source");
  const long long total = static_cast<long long>(rows) * (cols / 4);
  long long blocks = (total + 255) / 256;
  const long long cap = static_cast<long long>(num_sms()) * 16;
  if (blocks > cap) blocks = cap;
  cast_rows_kernel<Src><<<static_cast<int>(blocks), 256, 0, stream>>>(src, outer_stride, row_stride, inner, dst, rows, cols);
  HH_CHECK_LAUNCH("cast_rows_kernel");
  return 0;
}

int cast_rows_bf16(const float* src, long long outer_stride, long long row_stride, int inner, bf16* dst, int rows,
                   int cols, cudaStream_t stream) {
  return cast_rows_impl(src, outer_stride, row_stride, inner, dst, rows, cols, stream);
}

int cast_rows_bf16(const bf16* src, long long outer_stride, long long row_stride, int inner, bf16* dst, int rows,
                   int cols, cudaStream_t stream) {
  return cast_rows_impl(src, outer_stride, row_stride, inner, dst, rows, cols, stream);
}

int f32_to_bf16(const float* src, bf16* dst, size_t n, cudaStream_t stream) {
  HH_REQUIRE(n % 4 == 0, "f32_to_bf16: element count must be a multiple of 4");
  size_t n4 = n / 4;
  if (n4 == 0) return 0;
  size_t blocks = (n4 + 255) / 256;
  const size_t cap = static_cast<size_t>(num_sms()) * 16;
  if (blocks > cap) blocks = cap;
  f32_to_bf16_kernel<<<static_cast<int>(blocks), 256, 0, stream>>>(src, dst, n4);
  HH_CHECK_LAUNCH("f32_to_bf16_kernel");
  return 0;
}

}  // namespace hh
