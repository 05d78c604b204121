// Small fp32 nn.Linear family of the decoder's query side and heads (model/tfm_decoder.py:420-461 forward_pre, :208-228
// heads; their backward for run/train.py:196-203): forward, data gradient and weight gradient as ONE pipelined kernel
//
//     C[M, N] (+)= sum_red A(m, red) * B(red, n)
//
//   forward   M = rows,  N = out features, red = in features;  A = x [m][red],  B = W [n][red]
//   dgrad     M = rows,  N = in features,  red = out features; A = g [m][red],  B = W [red][n]
//   wgrad     M = out features, N = in features, red = rows;   A = g [red][m],  B = x [red][n]
//
// fp32 operands on the tensor cores as error-compensated TF32 (3 mma.sync per product: fp32-level accuracy, see
// hh_ptx.cuh).  These problems are tiny (832 rows x 256 x 256 at the c2 / c4 shapes): what bounds them is latency, not
// FLOPs.  The first-generation kernels (decoder.cu / decoder_bwd.cu, kept as *_legacy for shapes this file refuses)
// staged one 32-wide reduction chunk through registers per iteration, which exposed a full global-load round trip per
// chunk (30 us for a 256-deep reduction).  Here a 4-stage cp.async ring keeps three chunks in flight (the whole
// reduction of the K = 256 layers is requested before the first MMA), one __syncthreads per chunk, and the element-wise
// prologues (query_pos add, ReLU, dropout mask and activation derivative of the incoming gradient) run in shared memory
// on the 16-byte pieces each thread copied itself -- once per element instead of once per consuming warp, with one
// Philox block per four dropout decisions.
#include "hh_internal.h"
#include "hh_ptx.cuh"

namespace hh {

namespace {

constexpr int BM = 32, BN = 64, BK = 32, NST = 4;
constexpr int LDK = BK + 4;     // reduction-contiguous tiles [rows][36]: fragment loads (row g, column t) hit 32 banks
constexpr int LDA_R = BM + 8;   // reduction-major A tile [32][40]: (row t, column g) -> bank 8 t + g
constexpr int LDB_R = BN + 8;   // reduction-major B tile [32][72]
constexpr int A_FLOATS = BK * LDA_R;   // 1280 >= BM * LDK
constexpr int B_FLOATS = BN * LDK;     // 2304 == BK * LDB_R
static_assert(BM * LDK <= A_FLOATS && BK * LDB_R <= B_FLOATS, "tile regions");

enum { MODE_FWD = 0, MODE_DGRAD = 1, MODE_WGRAD = 2 };
enum { TA_NONE = 0, TA_ADD = 1, TA_GRAD = 2 };

struct Lin3Args {
  const float* A; long long lda;
  const float* Ax; long long ldax; int ax_mod;   // TA_ADD: row-periodic addend (query_pos); TA_GRAD: saved output Y
  const float* B; long long ldb;
  const float* Bx; long long ldbx; int bx_mod;   // wgrad: row-periodic addend of x
  int ta, a_relu, b_relu;
  int act; float act_scale;                      // TA_GRAD: g = act'(dY * mask, Y) * act_scale
  DropCfg drop; uint32_t drop_site; int drop_ld; // mask index = row * drop_ld + col (forward epilogue and TA_GRAD)
  int M, N, RED, red_per_split;
  float* C; long long ldc;
  const float* bias; const float* residual; long long ldres;   // forward epilogue
  int out_act;
  float beta, scale;                              // dgrad / wgrad: C = beta C + scale acc
  float* db;                                      // wgrad: column sums of g
};

__device__ __forceinline__ float act_grad3(float dy, float y, int act) {
  if (act == 1) return y > 0.f ? dy : 0.f;
  if (act == 2) return dy * y * (1.f - y);
  return dy;
}

// x = hi + lo for the 3xTF32 product.  `cvt.rna.tf32.f32` is not a native conversion on sm_100a (ptxas expands it to
// an Inf test, an integer add, a select and a mask: with the subtraction 9 instructions per operand element, which made
// the first version of this kernel issue-bound at 17 instructions per MMA).  Here: hi = x rounded to the 10-bit TF32
// mantissa by an integer add of half an ulp and a mask (round-half-away; operands are finite), lo = x - hi exactly; the
// tensor core itself ignores the low 13 bits of lo, so lo enters truncated: |x - hi - lo_used| <= 2^-21 |x|.
__device__ __forceinline__ void split_fast(float x, uint32_t& hi, uint32_t& lo) {
  hi = (__float_as_uint(x) + 0x1000u) & 0xffffe000u;
  lo = __float_as_uint(x - __uint_as_float(hi));
}

// keep-multipliers of the four consecutive elements idx .. idx + 3 (idx a multiple of 4): half a Philox block
__device__ __forceinline__ void drop_mult4(const DropCfg& d, uint32_t site, uint64_t idx, float (&m)[4]) {
  uint32_t o[4];
  drop_block8(d, site, idx >> 3, o);
  const bool up = (idx & 4u) != 0;
  const uint32_t w0 = up ? o[2] : o[0], w1 = up ? o[3] : o[1];
  m[0] = (w0 & 0xFFFFu) >= d.thr ? d.scale : 0.f;
  m[1] = (w0 >> 16) >= d.thr ? d.scale : 0.f;
  m[2] = (w1 & 0xFFFFu) >= d.thr ? d.scale : 0.f;
  m[3] = (w1 >> 16) >= d.thr ? d.scale : 0.f;
}

template <int MODE>
__global__ void __launch_bounds__(256) lin3_kernel(const Lin3Args a) {
  constexpr bool A_KM = MODE != MODE_WGRAD;   // A tile stored [m][red] (else [red][m])
  constexpr bool B_KM = MODE == MODE_FWD;     // B tile stored [n][red] (else [red][n])
  extern __shared__ __align__(16) float smem[];
  const bool has_ax = a.Ax != nullptr, has_bx = a.Bx != nullptr;
  const int off_b = A_FLOATS, off_ax = A_FLOATS + B_FLOATS, off_bx = off_ax + (has_ax ? A_FLOATS : 0);
  const int stage_floats = off_bx + (has_bx ? B_FLOATS : 0);

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  const int wm = warp & 1, wn = warp >> 1;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  const int red_begin = blockIdx.z * a.red_per_split;
  const int red_end = min(red_begin + a.red_per_split, a.RED);
  const int nch = (red_end - red_begin + BK - 1) / BK;

  // ---- the 16-byte pieces this thread copies (and later transforms): one of A, two of B
  // A piece: source element (arow, acol) of the row-major matrix A (+ red0 along the reduction), smem offset a_dst
  int arow, acol, a_dst;
  if (A_KM) { arow = m0 + (tid >> 3); acol = (tid & 7) * 4; a_dst = (tid >> 3) * LDK + (tid & 7) * 4; }
  else { arow = tid >> 3; acol = m0 + (tid & 7) * 4; a_dst = (tid >> 3) * LDA_R + (tid & 7) * 4; }
  int brow[2], bcol[2], b_dst[2];
#pragma unroll
  for (int it = 0; it < 2; ++it) {
    const int idx = tid + it * 256;
    if (B_KM) { brow[it] = n0 + (idx >> 3); bcol[it] = (idx & 7) * 4; b_dst[it] = (idx >> 3) * LDK + (idx & 7) * 4; }
    else { brow[it] = idx >> 4; bcol[it] = n0 + (idx & 15) * 4; b_dst[it] = (idx >> 4) * LDB_R + (idx & 15) * 4; }
  }
  auto a_valid = [&](int red0) {
    return A_KM ? (arow < a.M && red0 + acol < red_end) : (red0 + arow < red_end && acol < a.M);
  };
  // Running source pointers of this thread's pieces: chunks are requested strictly in order, so every request is one
  // compare, one select and one pointer increment (recomputing row * ld + col, and the row modulo of the periodic
  // addends, per request cost as many instructions as the MMAs of the chunk).
  const bool a_ok = A_KM ? arow < a.M : acol < a.M;
  const float* pa = a.A + (A_KM ? static_cast<long long>(arow) * a.lda + red_begin + acol
                                : static_cast<long long>(red_begin + arow) * a.lda + acol);
  const long long step_a = A_KM ? BK : static_cast<long long>(BK) * a.lda;
  const float* pax = a.Ax;
  long long step_ax = 0;
  if (has_ax) {
    if (a.ta == TA_ADD) pax += static_cast<long long>(arow % a.ax_mod) * a.ldax + red_begin + acol;   // forward only (A_KM)
    else pax += A_KM ? static_cast<long long>(arow) * a.ldax + red_begin + acol
                     : static_cast<long long>(red_begin + arow) * a.ldax + acol;
    step_ax = (A_KM || a.ta == TA_ADD) ? BK : static_cast<long long>(BK) * a.ldax;
  }
  bool b_ok[2];
  const float* pb[2];
  int bxmod[2];
#pragma unroll
  for (int it = 0; it < 2; ++it) {
    b_ok[it] = B_KM ? brow[it] < a.N : bcol[it] < a.N;
    pb[it] = a.B + (B_KM ? static_cast<long long>(brow[it]) * a.ldb + red_begin + bcol[it]
                         : static_cast<long long>(red_begin + brow[it]) * a.ldb + bcol[it]);
    bxmod[it] = has_bx ? (red_begin + brow[it]) % a.bx_mod : 0;   // wgrad only (rows of x run along the reduction)
  }
  const long long step_b = B_KM ? BK : static_cast<long long>(BK) * a.ldb;
  const int bx_step = has_bx ? BK % a.bx_mod : 0;
  int ld_red0 = red_begin;
  auto load_stage = [&](int c) {
    float* st = smem + (c % NST) * stage_floats;
    {
      const bool v = a_ok && ld_red0 + (A_KM ? acol : arow) < red_end;
      cp_async_16(st + a_dst, v ? pa : a.A, v);
      pa += step_a;
      if (has_ax) {
        cp_async_16(st + off_ax + a_dst, v ? pax : a.Ax, v);
        pax += step_ax;
      }
    }
#pragma unroll
    for (int it = 0; it < 2; ++it) {
      const bool v = b_ok[it] && ld_red0 + (B_KM ? bcol[it] : brow[it]) < red_end;
      cp_async_16(st + off_b + b_dst[it], v ? pb[it] : a.B, v);
      pb[it] += step_b;
      if (has_bx) {
        cp_async_16(st + off_bx + b_dst[it], v ? a.Bx + static_cast<long long>(bxmod[it]) * a.ldbx + bcol[it] : a.Bx, v);
        bxmod[it] += bx_step;
        if (bxmod[it] >= a.bx_mod) bxmod[it] -= a.bx_mod;
      }
    }
    ld_red0 += BK;
  };
  // element-wise prologue on this thread's own pieces (its cp.async data is visible to it after wait_group)
  auto transform_stage = [&](int c) {
    float* st = smem + (c % NST) * stage_floats;
    const int red0 = red_begin + c * BK;
    if (a.ta != TA_NONE || a.a_relu) {
      float4 v = *reinterpret_cast<float4*>(st + a_dst);
      if (a.ta == TA_ADD) {
        const float4 x = *reinterpret_cast<const float4*>(st + off_ax + a_dst);
        v.x += x.x; v.y += x.y; v.z += x.z; v.w += x.w;
      } else if (a.ta == TA_GRAD && a_valid(red0)) {
        if (a.drop.thr) {
          const int r = A_KM ? arow : red0 + arow, cc = A_KM ? red0 + acol : acol;
          float mk[4];
          drop_mult4(a.drop, a.drop_site, static_cast<uint64_t>(r) * a.drop_ld + cc, mk);
          v.x *= mk[0]; v.y *= mk[1]; v.z *= mk[2]; v.w *= mk[3];
        }
        if (a.act) {
          const float4 y = *reinterpret_cast<const float4*>(st + off_ax + a_dst);
          v.x = act_grad3(v.x, y.x, a.act) * a.act_scale; v.y = act_grad3(v.y, y.y, a.act) * a.act_scale;
          v.z = act_grad3(v.z, y.z, a.act) * a.act_scale; v.w = act_grad3(v.w, y.w, a.act) * a.act_scale;
        }
      }
      if (a.a_relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
      *reinterpret_cast<float4*>(st + a_dst) = v;
    }
    if (has_bx || a.b_relu) {
#pragma unroll
      for (int it = 0; it < 2; ++it) {
        float4 v = *reinterpret_cast<float4*>(st + off_b + b_dst[it]);
        if (has_bx) {
          const float4 x = *reinterpret_cast<const float4*>(st + off_bx + b_dst[it]);
          v.x += x.x; v.y += x.y; v.z += x.z; v.w += x.w;
        }
        if (a.b_relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
        *reinterpret_cast<float4*>(st + off_b + b_dst[it]) = v;
      }
    }
  };

  float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
  float bsum = 0.f;   // wgrad: threads 0..31 of the column-tile-0 CTAs own one bias-gradient entry
#pragma unroll
  for (int s = 0; s < NST - 1; ++s) {
    if (s < nch) load_stage(s);
    cp_async_commit();
  }
  for (int c = 0; c < nch; ++c) {
    cp_async_wait<NST - 2>();
    transform_stage(c);
    __syncthreads();   // chunk c complete for everyone; everyone is done with chunk c - 1 (whose stage is refilled next)
    if (c + NST - 1 < nch) load_stage(c + NST - 1);
    cp_async_commit();
    const float* As = smem + (c % NST) * stage_floats;
    const float* Bs = As + off_b;
    // The tensor core truncates when it accumulates: chain only this chunk's 4 k-steps there (the two small correction
    // products in their own accumulator) and add the chunk's partial to the running sum with a rounded fp32 add.
    // (One accumulator set: splitting the k-steps over 2 or 4 sets measured slower -- registers (occupancy) matter more
    // than MMA chain length.)
    float ph[2][4], pc[2][4];
#pragma unroll
    for (int i = 0; i < 8; ++i) (&ph[0][0])[i] = (&pc[0][0])[i] = 0.f;
    // Forward (both tiles reduction-contiguous): the MMA's reduction index is a free permutation as long as A and B use
    // the same one -- thread t takes the chunk's elements 8t .. 8t+7 (k-step ks: 8t + 2ks as k = t, 8t + 2ks + 1 as
    // k = t + 4), so a fragment row is two 16-byte loads per chunk instead of eight 4-byte ones (rows of 36 floats:
    // the eight lanes of a quarter-warp phase cover all 32 banks).
    float av[2][8], bv[2][8];
    if (MODE == MODE_FWD) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const float4* ap = reinterpret_cast<const float4*>(As + (wm * 16 + g + h * 8) * LDK + 8 * t);
        const float4* bp = reinterpret_cast<const float4*>(Bs + (wn * 16 + h * 8 + g) * LDK + 8 * t);
        *reinterpret_cast<float4*>(&av[h][0]) = ap[0];
        *reinterpret_cast<float4*>(&av[h][4]) = ap[1];
        *reinterpret_cast<float4*>(&bv[h][0]) = bp[0];
        *reinterpret_cast<float4*>(&bv[h][4]) = bp[1];
      }
    }
#pragma unroll
    for (int ks = 0; ks < BK / 8; ++ks) {
      float af[4];
      if (MODE == MODE_FWD) {
        af[0] = av[0][2 * ks]; af[1] = av[1][2 * ks]; af[2] = av[0][2 * ks + 1]; af[3] = av[1][2 * ks + 1];
      } else if (A_KM) {
        af[0] = As[(wm * 16 + g) * LDK + ks * 8 + t];     af[1] = As[(wm * 16 + g + 8) * LDK + ks * 8 + t];
        af[2] = As[(wm * 16 + g) * LDK + ks * 8 + t + 4]; af[3] = As[(wm * 16 + g + 8) * LDK + ks * 8 + t + 4];
      } else {
        af[0] = As[(ks * 8 + t) * LDA_R + wm * 16 + g];     af[1] = As[(ks * 8 + t) * LDA_R + wm * 16 + g + 8];
        af[2] = As[(ks * 8 + t + 4) * LDA_R + wm * 16 + g]; af[3] = As[(ks * 8 + t + 4) * LDA_R + wm * 16 + g + 8];
      }
      uint32_t ah[4], al[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) split_fast(af[i], ah[i], al[i]);
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int n = wn * 16 + j * 8 + g;
        float b0, b1;
        if (MODE == MODE_FWD) { b0 = bv[j][2 * ks]; b1 = bv[j][2 * ks + 1]; }
        else { b0 = Bs[(ks * 8 + t) * LDB_R + n]; b1 = Bs[(ks * 8 + t + 4) * LDB_R + n]; }
        uint32_t bh0, bl0, bh1, bl1;
        split_fast(b0, bh0, bl0);
        split_fast(b1, bh1, bl1);
        mma_tf32_1688(pc[j], al, bh0, bh1);
        mma_tf32_1688(ph[j], ah, bh0, bh1);
        mma_tf32_1688(pc[j], ah, bl0, bl1);
      }
    }
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[j][e] += ph[j][e] + pc[j][e];
    if (MODE == MODE_WGRAD && a.db && blockIdx.x == 0 && tid < BM) {
#pragma unroll 8
      for (int r = 0; r < BK; ++r) bsum += As[r * LDA_R + tid];
    }
  }

  // ---- epilogue
#pragma unroll
  for (int j = 0; j < 2; ++j) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int row = m0 + wm * 16 + g + h * 8;
      const int col = n0 + wn * 16 + j * 8 + 2 * t;
      if (row >= a.M || col >= a.N) continue;   // N is a multiple of 4 and col is even: col + 1 < N as well
      float v0 = acc[j][h * 2], v1 = acc[j][h * 2 + 1];
      float* d = a.C + static_cast<long long>(row) * a.ldc + col;
      if (MODE == MODE_FWD) {
        if (a.bias) { v0 += a.bias[col]; v1 += a.bias[col + 1]; }
        if (a.out_act == 1) { v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f); }
        else if (a.out_act == 2) { v0 = 1.f / (1.f + __expf(-v0)); v1 = 1.f / (1.f + __expf(-v1)); }
        if (a.drop.thr) {
          const uint64_t idx = static_cast<uint64_t>(row) * a.drop_ld + col;
          uint32_t o[4];
          drop_block8(a.drop, a.drop_site, idx >> 3, o);
          const uint32_t wi = (static_cast<uint32_t>(idx) & 7u) >> 1;
          const uint32_t w = wi == 0 ? o[0] : wi == 1 ? o[1] : wi == 2 ? o[2] : o[3];
          v0 *= (w & 0xFFFFu) >= a.drop.thr ? a.drop.scale : 0.f;
          v1 *= (w >> 16) >= a.drop.thr ? a.drop.scale : 0.f;
        }
        if (a.residual) {
          const float* r = a.residual + static_cast<long long>(row) * a.ldres + col;
          v0 += r[0]; v1 += r[1];
        }
        d[0] = v0; d[1] = v1;
      } else {
        v0 *= a.scale; v1 *= a.scale;
        if (gridDim.z > 1) { atomicAdd(d, v0); atomicAdd(d + 1, v1); }
        else if (a.beta != 0.f) { d[0] = a.beta * d[0] + v0; d[1] = a.beta * d[1] + v1; }
        else { d[0] = v0; d[1] = v1; }
      }
    }
  }
  if (MODE == MODE_WGRAD && a.db && blockIdx.x == 0 && tid < BM && m0 + tid < a.M) {
    float* d = a.db + m0 + tid;
    if (gridDim.z > 1) atomicAdd(d, a.scale * bsum);
    else *d = (a.beta != 0.f ? a.beta * *d : 0.f) + a.scale * bsum;
  }
}

inline bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

template <int MODE>
int launch_lin3(const Lin3Args& a, int split, cudaStream_t s) {
  const size_t stage = A_FLOATS + B_FLOATS + (a.Ax ? A_FLOATS : 0) + (a.Bx ? B_FLOATS : 0);
  const size_t bytes = stage * NST * sizeof(float);
  static bool configured = false;   // (one device per process)
  if (!configured) {
    HH_CHECK_CUDA(cudaFuncSetAttribute(lin3_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>(2 * (A_FLOATS + B_FLOATS) * NST * sizeof(float))));
    configured = true;
  }
  dim3 grid((a.N + BN - 1) / BN, (a.M + BM - 1) / BM, split);
  lin3_kernel<MODE><<<grid, 256, bytes, s>>>(a);
  HH_CHECK_LAUNCH("lin3_kernel");
  return 0;
}

}  // namespace

int linear_f32(const LinArgs& a, cudaStream_t stream) {
  HH_REQUIRE(a.R > 0 && a.N > 0 && a.K > 0, "linear_f32: empty problem");
  // both generations read the operands in 16-byte pieces
  HH_REQUIRE(a.K % 4 == 0 && a.ldi % 4 == 0 && al16(a.in) && al16(a.W) && (a.in_add == nullptr || al16(a.in_add)),
             "linear_f32: input, weight and addend rows must be 16-byte aligned (K and ldi multiples of 4)");
  HH_REQUIRE(a.in_add == nullptr || a.add_mod > 0, "linear_f32: add_mod");
  if (a.N % 2 != 0) return linear_f32_legacy(a, stream);
  Lin3Args l{};
  l.A = a.in; l.lda = a.ldi; l.Ax = a.in_add; l.ldax = a.K; l.ax_mod = a.in_add ? a.add_mod : 1;
  l.B = a.W; l.ldb = a.K;
  l.ta = a.in_add ? TA_ADD : TA_NONE; l.a_relu = a.in_relu;
  l.drop = a.drop; l.drop_site = a.drop_site; l.drop_ld = a.N;
  l.M = a.R; l.N = a.N; l.RED = a.K; l.red_per_split = a.K;
  l.C = a.out; l.ldc = a.ldo; l.bias = a.bias; l.residual = a.residual; l.ldres = a.ldres; l.out_act = a.act;
  l.scale = 1.f;
  return launch_lin3<MODE_FWD>(l, 1, stream);
}

namespace {
// g = act'(dY * mask, Y) * act_scale as the A operand of dgrad / wgrad
void grad_operand(const LinBwdArgs& a, Lin3Args& l) {
  l.A = a.dY; l.lda = a.ldy;
  if (a.act || a.drop.thr) {
    l.ta = TA_GRAD;
    l.Ax = a.act ? a.Y : nullptr; l.ldax = a.ldyo; l.ax_mod = 1;
    l.act = a.act; l.act_scale = a.act_scale != 0.f ? a.act_scale : 1.f;
    l.drop = a.drop; l.drop_site = a.drop_site; l.drop_ld = a.N;
  }
}
bool grad_operand_ok(const LinBwdArgs& a) {
  return a.N % 4 == 0 && a.ldy % 4 == 0 && al16(a.dY) && (!a.act || (a.Y && a.ldyo % 4 == 0 && al16(a.Y)));
}
}  // namespace

int linear_dgrad_f32(const LinBwdArgs& a, cudaStream_t s) {
  HH_REQUIRE(a.R > 0 && a.N > 0 && a.K > 0 && a.dY && a.W && a.dX, "linear_dgrad: bad argument");
  HH_REQUIRE(a.act == 0 || a.Y != nullptr, "linear_dgrad: activation derivative needs the saved output");
  const bool ok = grad_operand_ok(a) && a.K % 4 == 0 && al16(a.W);
  if (!ok) return linear_dgrad_f32_legacy(a, s);
  Lin3Args l{};
  grad_operand(a, l);
  l.B = a.W; l.ldb = a.K;
  l.M = a.R; l.N = a.K; l.RED = a.N; l.red_per_split = (a.N + BK - 1) / BK * BK;
  l.C = a.dX; l.ldc = a.lddx; l.beta = a.beta; l.scale = 1.f;
  return launch_lin3<MODE_DGRAD>(l, 1, s);
}

int linear_wgrad_f32(const LinBwdArgs& a, cudaStream_t s) {
  HH_REQUIRE(a.R > 0 && a.N > 0 && a.K > 0 && a.dY && a.X && a.dW, "linear_wgrad: bad argument");
  HH_REQUIRE(a.act == 0 || a.Y != nullptr, "linear_wgrad: activation derivative needs the saved output");
  const bool ok = grad_operand_ok(a) && a.K % 4 == 0 && a.ldx % 4 == 0 && al16(a.X) &&
                  (a.x_add == nullptr || (al16(a.x_add) && a.add_mod > 0));
  if (!ok) return linear_wgrad_f32_legacy(a, s);
  Lin3Args l{};
  grad_operand(a, l);
  l.B = a.X; l.ldb = a.ldx; l.Bx = a.x_add; l.ldbx = a.K; l.bx_mod = a.x_add ? a.add_mod : 1; l.b_relu = a.in_relu;
  l.M = a.N; l.N = a.K; l.RED = a.R;
  l.C = a.dW; l.ldc = a.ldw; l.db = a.db; l.beta = a.beta; l.scale = a.scale;
  // Few output tiles but many rows: split the row reduction over gridDim.z so that ~4 CTAs per SM are in flight; the
  // partial tiles are combined with fp32 atomics (summation order, hence the last bits, vary from run to run).
  const int tiles = ((a.K + BN - 1) / BN) * ((a.N + BM - 1) / BM);
  int split = (4 * num_sms() + tiles - 1) / tiles;
  // at least 128 rows (4 chunks: one full ring) per CTA; 64 and 256 measured within noise of it
  const int max_split = (a.R + 127) / 128;
  if (split > max_split) split = max_split;
  if (split > 64) split = 64;
  if (split < 1 || (a.beta != 0.f && a.beta != 1.f)) split = 1;
  l.red_per_split = ((a.R + split - 1) / split + BK - 1) / BK * BK;
  split = (a.R + l.red_per_split - 1) / l.red_per_split;
  if (split > 1 && a.beta == 0.f) {
    HH_CHECK_CUDA(cudaMemset2DAsync(a.dW, static_cast<size_t>(a.ldw) * 4, 0, static_cast<size_t>(a.K) * 4, a.N, s));
    if (a.db) HH_CHECK_CUDA(cudaMemsetAsync(a.db, 0, static_cast<size_t>(a.N) * 4, s));
  }
  return launch_lin3<MODE_WGRAD>(l, split, s);
}

}  // namespace hh
