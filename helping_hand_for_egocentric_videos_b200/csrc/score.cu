// Video-text scoring (model/metric.py:363-375 sim_matrix, :218 argmax; model/loss.py:61-69 softmax at 1/temperature).
//
// sim_matrix: fused L2-normalise + similarity.  A 32x64 output tile streams the embedding dimension once and
// accumulates the dot products together with the squared row norms of both operands, so the embeddings are read
// once and never written back normalised:  out = a.b / (max(|a|, eps) * max(|b|, eps)).
// Large problems (EPIC-MIR: 9728 x 9728 x 256, the c4 EgoNCE matrix) run on the tcgen05 GEMM instead: rows are normalised
// in fp32 and split into a bf16 (hi, lo) pair by split_normalize_kernel, and out = [hi hi lo lo] . [hi lo hi lo]^T is one
// bf16 GEMM with K = 4 d and fp32 accumulation -- every product of two bf16 values is exact in fp32, the pair carries
// 16 mantissa bits, so the result stays within ~2e-6 of the fp32 statement (test: 1e-5 against fp64) while the kernel
// becomes output-write bound.
// row_reduce: one warp per row -- argmax (first maximum, like torch.argmax), softmax or log_softmax of scale * x.
#include "hh_internal.h"
#include "hh_ptx.cuh"
#include "engine.h"

namespace hh {

namespace {

constexpr int SBM = 32, SBN = 64, SBK = 32;

__global__ void __launch_bounds__(256)
sim_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ out, int Na, int Nb, int d,
           float eps) {
  __shared__ float As[SBM][SBK + 1];
  __shared__ float Bs[SBN][SBK + 1];
  __shared__ float na[SBM], nb[SBN];
  const int tid = threadIdx.x;
  const int ty = tid >> 4, tx = tid & 15;
  const int r0 = blockIdx.y * SBM, n0 = blockIdx.x * SBN;
  float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
  float sq_a = 0.f, sq_b = 0.f;  // threads 0..31 own an A row, 0..63 a B row
  for (int k0 = 0; k0 < d; k0 += SBK) {
    for (int idx = tid; idx < SBM * SBK; idx += 256) {
      const int r = idx / SBK, k = idx - r * SBK;
      As[r][k] = (r0 + r < Na && k0 + k < d) ? a[static_cast<size_t>(r0 + r) * d + k0 + k] : 0.f;
    }
    for (int idx = tid; idx < SBN * SBK; idx += 256) {
      const int r = idx / SBK, k = idx - r * SBK;
      Bs[r][k] = (n0 + r < Nb && k0 + k < d) ? b[static_cast<size_t>(n0 + r) * d + k0 + k] : 0.f;
    }
    __syncthreads();
    if (tid < SBM)
      for (int k = 0; k < SBK; ++k) sq_a += As[tid][k] * As[tid][k];
    if (tid < SBN)
      for (int k = 0; k < SBK; ++k) sq_b += Bs[tid][k] * Bs[tid][k];
#pragma unroll
    for (int k = 0; k < SBK; ++k) {
      const float a0 = As[ty * 2][k], a1 = As[ty * 2 + 1][k];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float w = Bs[tx + 16 * j][k];
        acc[0][j] += a0 * w;
        acc[1][j] += a1 * w;
      }
    }
    __syncthreads();
  }
  if (tid < SBM) na[tid] = fmaxf(sqrtf(sq_a), eps);
  if (tid < SBN) nb[tid] = fmaxf(sqrtf(sq_b), eps);
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int row = r0 + ty * 2 + i;
    if (row >= Na) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int col = n0 + tx + 16 * j;
      if (col < Nb) out[static_cast<size_t>(row) * Nb + col] = acc[i][j] / (na[ty * 2 + i] * nb[tx + 16 * j]);
    }
  }
}

// warp per row: y = x / max(|x|, eps); out row = [hi hi lo lo] (order 0) or [hi lo hi lo] (order 1), hi = bf16(y),
// lo = bf16(y - hi)
__global__ void __launch_bounds__(256)
split_normalize_kernel(const float* __restrict__ x, bf16* __restrict__ out, int rows, int d, float eps, int order) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* xr = x + static_cast<size_t>(row) * d;
  float sq = 0.f;
  for (int c = lane; c < d; c += 32) sq = fmaf(xr[c], xr[c], sq);
  sq = warp_sum(sq);
  const float inv = 1.0f / fmaxf(sqrtf(sq), eps);
  bf16* o = out + static_cast<size_t>(row) * 4 * d;
  for (int c = lane; c < d; c += 32) {
    const float y = xr[c] * inv;
    const bf16 hi = __float2bfloat16_rn(y);
    const bf16 lo = __float2bfloat16_rn(y - __bfloat162float(hi));
    o[c] = hi;
    o[d + c] = order ? lo : hi;
    o[2 * d + c] = order ? hi : lo;
    o[3 * d + c] = lo;
  }
}

__global__ void __launch_bounds__(256)
row_reduce_kernel(const float* __restrict__ x, int rows, int cols, float scale, int mode, void* __restrict__ out) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* xr = x + static_cast<size_t>(row) * cols;
  float mx = -INFINITY;
  int arg = 0x7fffffff;
  for (int c = lane; c < cols; c += 32) {
    const float v = xr[c] * scale;
    if (v > mx || (v == mx && c < arg)) {
      mx = v;
      arg = c;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float om = __shfl_xor_sync(0xffffffffu, mx, o);
    const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
    if (om > mx || (om == mx && oa < arg)) {
      mx = om;
      arg = oa;
    }
  }
  if (mode == 0) {
    if (lane == 0) reinterpret_cast<long long*>(out)[row] = arg;
    return;
  }
  float l = 0.f;
  for (int c = lane; c < cols; c += 32) l += __expf(xr[c] * scale - mx);
  l = warp_sum(l);
  float* o = reinterpret_cast<float*>(out) + static_cast<size_t>(row) * cols;
  if (mode == 1) {
    const float inv = 1.f / l;
    for (int c = lane; c < cols; c += 32) o[c] = __expf(xr[c] * scale - mx) * inv;
  } else {
    const float lse = mx + logf(l);
    for (int c = lane; c < cols; c += 32) o[c] = xr[c] * scale - lse;
  }
}

}  // namespace

// operand workspace of the tensor-core path: grow-only, one per process (the C ABI is not re-entrant per device)
static DevBuf g_sim_ws;

int sim_matrix(const float* a, const float* b, float* out, int Na, int Nb, int d, float eps, cudaStream_t stream) {
  HH_REQUIRE(Na > 0 && Nb > 0 && d > 0, "sim_matrix: empty problem");
  if (Na >= 128 && Nb >= 128 && d % 8 == 0 && (reinterpret_cast<uintptr_t>(out) & 3) == 0) {
    const size_t abytes = (static_cast<size_t>(Na) * 4 * d * 2 + 255) & ~size_t(255);
    const size_t bbytes = static_cast<size_t>(Nb) * 4 * d * 2;
    int rc = g_sim_ws.reserve(abytes + bbytes);
    if (rc) return rc;
    bf16* a4 = static_cast<bf16*>(g_sim_ws.ptr);
    bf16* b4 = reinterpret_cast<bf16*>(static_cast<uint8_t*>(g_sim_ws.ptr) + abytes);
    split_normalize_kernel<<<(Na + 7) / 8, 256, 0, stream>>>(a, a4, Na, d, eps, 0);
    HH_CHECK_LAUNCH("split_normalize_kernel");
    split_normalize_kernel<<<(Nb + 7) / 8, 256, 0, stream>>>(b, b4, Nb, d, eps, 1);
    HH_CHECK_LAUNCH("split_normalize_kernel");
    return gemm_bf16(a4, 4 * d, b4, 4 * d, out, Nb, nullptr, nullptr, 0, Na, Nb, 4 * d, EPI_BIAS_F32, stream);
  }
  dim3 grid((Nb + SBN - 1) / SBN, (Na + SBM - 1) / SBM);
  HH_REQUIRE(grid.y < 65536, "sim_matrix: too many rows for one launch");
  sim_kernel<<<grid, 256, 0, stream>>>(a, b, out, Na, Nb, d, eps);
  HH_CHECK_LAUNCH("sim_kernel");
  return 0;
}

int row_reduce(const float* x, int rows, int cols, float scale, int mode, void* out, cudaStream_t stream) {
  HH_REQUIRE(rows > 0 && cols > 0, "row_reduce: empty problem");
  HH_REQUIRE(mode >= 0 && mode <= 2, "row_reduce: mode");
  const int grid = (rows + 7) / 8;
  row_reduce_kernel<<<grid, 256, 0, stream>>>(x, rows, cols, scale, mode, out);
  HH_CHECK_LAUNCH("row_reduce_kernel");
  return 0;
}

}  // namespace hh
