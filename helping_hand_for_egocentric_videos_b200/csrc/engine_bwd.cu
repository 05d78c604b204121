// Decoder::backward -- gradients of every ObjDecoder parameter the engine owns, for the activations kept by the last
// forward(save = true).  Reference graph: ObjDecoder.forward (model/tfm_decoder.py:183-233) -> Cross_Attention.forward
// (:76-93) -> TransformerDecoderLayer.forward_pre (:420-461) x L, differentiated by hand in reverse order:
//
//   heads      bbox MLP (sigmoid / ReLU derivatives folded into the dgrad / wgrad loads), frame_proj split, final norm
//   layers     FFN, cross attention (dQ fp32; dK / dV bf16 into the all-layer [B*S, L*C] matrices), self attention;
//              every LayerNorm backward accumulates straight into the residual-stream gradient
//   memory     d(mem + pos) = dK_all Wk, d mem += dV_all Wv on the tcgen05 GEMM; weight gradients dK_all^T (mem + pos),
//              dV_all^T mem and d memf^T feat as GEMMs over the B*S reduction dimension (operands transposed to
//              K-major bf16 first); pre_norm backward; position-embedding reductions
//
// The class head has no loss in the reference's criterion (losses = ['boxes', 'cardinality'], run/train.py:471;
// exclude_class=True), so class_embed receives zero gradients.  Host-side C++ only (kernels: decoder_bwd.cu).
#include <cmath>

#include "engine.h"

namespace hh {

#define RC(expr)         \
  do {                   \
    int _rc = (expr);    \
    if (_rc) return _rc; \
  } while (0)

namespace {

// dhsproj[lb, q, :] = sum_t dcond[lb, t, q, :] ;  dft[t, :] = sum_{lb, q} dcond[lb, t, q, :]
// (blockIdx.y + y_off selects the row: [0, LB*Q) the dhsproj rows, then the T rows of dft)
__global__ void frame_term_bwd_kernel(const float* __restrict__ dcond, float* __restrict__ dhsproj, float* __restrict__ dft,
                                      int LB, int T, int Q, int C, int y_off) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const int by = static_cast<int>(blockIdx.y) + y_off;
  if (by < LB * Q) {
    const int lb = by / Q, q = by % Q;
    float t = 0.f;
    for (int f = 0; f < T; ++f) t += dcond[((static_cast<size_t>(lb) * T + f) * Q + q) * C + c];
    dhsproj[(static_cast<size_t>(lb) * Q + q) * C + c] = t;
  } else {
    const int f = by - LB * Q;
    float t = 0.f;
    for (int lb = 0; lb < LB; ++lb)
      for (int q = 0; q < Q; ++q) t += dcond[((static_cast<size_t>(lb) * T + f) * Q + q) * C + c];
    dft[static_cast<size_t>(f) * C + c] = t;
  }
}

// d pos_embed[0] = 0, d pos_embed[1 + p] = sum_t dpos3d[t*n + p] ; d temporal[t] = sum_p dpos3d[t*n + p]
__global__ void pos3d_bwd_kernel(const float* __restrict__ dpos, float* __restrict__ dpe, float* __restrict__ dte, int T,
                                 int n, int C) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const int r = blockIdx.y;
  if (r == 0) {
    dpe[c] = 0.f;
  } else if (r <= n) {
    float t = 0.f;
    for (int f = 0; f < T; ++f) t += dpos[(static_cast<size_t>(f) * n + r - 1) * C + c];
    dpe[static_cast<size_t>(r) * C + c] = t;
  } else {
    const int f = r - n - 1;
    float t = 0.f;
    for (int p = 0; p < n; ++p) t += dpos[(static_cast<size_t>(f) * n + p) * C + c];
    dte[static_cast<size_t>(f) * C + c] = t;
  }
}

int dgrad(const float* dY, int ldy, const float* Y, int ldyo, int act, const float* W, float* dX, int lddx, int R, int N,
          int K, float beta, cudaStream_t s, DropCfg drop = drop_off(), uint32_t drop_site = 0, float act_scale = 1.f) {
  LinBwdArgs a{};
  a.dY = dY; a.ldy = ldy; a.Y = Y; a.ldyo = ldyo; a.act = act; a.W = W; a.dX = dX; a.lddx = lddx; a.R = R; a.N = N; a.K = K;
  a.beta = beta; a.scale = 1.f;
  a.drop = drop; a.drop_site = drop_site; a.act_scale = act_scale;
  return linear_dgrad_f32(a, s);
}

int wgrad(const float* dY, int ldy, const float* Y, int ldyo, int act, const float* X, int ldx, const float* x_add,
          int add_mod, float* dW, int ldw, float* db, int R, int N, int K, float beta, float scale, cudaStream_t s,
          DropCfg drop = drop_off(), uint32_t drop_site = 0, float act_scale = 1.f) {
  LinBwdArgs a{};
  a.dY = dY; a.ldy = ldy; a.Y = Y; a.ldyo = ldyo; a.act = act; a.X = X; a.ldx = ldx; a.x_add = x_add; a.add_mod = add_mod;
  a.dW = dW; a.ldw = ldw; a.db = db; a.R = R; a.N = N; a.K = K; a.beta = beta; a.scale = scale;
  a.drop = drop; a.drop_site = drop_site; a.act_scale = act_scale;
  return linear_wgrad_f32(a, s);
}

}  // namespace

Decoder::~Decoder() {
  if (bw_side) cudaStreamDestroy(bw_side);
  if (bw_fork) cudaEventDestroy(bw_fork);
  for (cudaEvent_t e : bw_done)
    if (e) cudaEventDestroy(e);
}

const float* Decoder::grad(const std::string& key) const {
  auto it = grads.find(key);
  return it == grads.end() ? nullptr : static_cast<const float*>(it->second.ptr);
}

int Decoder::backward(const float* hs, const float* boxes, const float* d_hs, const float* d_boxes, cudaStream_t s) {
  HH_REQUIRE(saved_B > 0 && !saved.empty(), "decoder backward: no saved forward (call the training forward first)");
  HH_REQUIRE(hs && boxes, "decoder backward: the forward outputs hs / boxes are required");
  HH_REQUIRE(!weights.dirty, "decoder backward: parameters changed since the forward");
  const int C = cfg.d_model, Lr = cfg.num_layers, F = cfg.feature_dim, Q = cfg.num_queries, Fd = cfg.dim_feedforward;
  const int B = saved_B, T = saved_T, n = cfg.patches_per_frame, S = T * n, heads = cfg.nhead;
  const int R = B * Q;
  const size_t BS = static_cast<size_t>(B) * S;
  HH_REQUIRE(BS % 8 == 0, "decoder backward: clips x patch tokens must be a multiple of 8");
  const bool traj = cfg.pred_traj && T == cfg.num_frames;
  const size_t LR = static_cast<size_t>(Lr) * R;
  const size_t rows_box = LR * (traj ? T : 1);
  const float qscale = 1.0f / std::sqrt(64.0f);
  const size_t RC_ = static_cast<size_t>(R) * C;

  // ---- gradient buffers (one per parameter key), zeroed: parameters outside the loss graph keep a zero gradient
  for (const auto& kv : weights.expected) {
    DevBuf& g = grads[kv.first];
    RC(g.reserve(static_cast<size_t>(kv.second) * 4));
    HH_CHECK_CUDA(cudaMemsetAsync(g.ptr, 0, static_cast<size_t>(kv.second) * 4, s));
  }
  auto G = [&](const std::string& k) { return static_cast<float*>(grads[k].ptr); };

  // ---- scratch (all reserved up front: growing a buffer later would free storage that queued kernels still use)
  const int M = static_cast<int>(BS);
  const int LC = Lr * C;
  size_t big = (rows_box + T) * C;
  if (static_cast<size_t>(R) * Fd > big) big = static_cast<size_t>(R) * Fd;
  if (BS * C > big) big = BS * C;
  if (static_cast<size_t>(S) * C > big) big = static_cast<size_t>(S) * C;
  RC(bw_a.reserve(big * 4));
  RC(bw_b.reserve(big * 4));
  RC(bw_c.reserve(LR * C * 4));       // d hs of all layers
  RC(bw_d.reserve(RC_ * 3 * 4));      // dx, tmp, tmp2
  RC(bw_t3.reserve(RC_ * 3 * 4));     // d qkv of the self attention
  RC(bw_dk.reserve(BS * LC * 2));
  RC(bw_dv.reserve(BS * LC * 2));
  RC(bw_t1.reserve(static_cast<size_t>(LC) * 4 * 2 + static_cast<size_t>(LC) * C * 4 * 2));
  RC(bw_t2.reserve((static_cast<size_t>(LC) + C + (C > F ? C : F)) * BS * 2));
  size_t wsb = ln_backward_workspace_bytes(M, C);
  const size_t w2 = cross_attn_bwd_workspace_bytes(B, Q, heads, S);
  if (w2 > wsb) wsb = w2;
  const size_t w3 = colsum_workspace_bytes(static_cast<long long>(S) * C);
  if (w3 > wsb) wsb = w3;
  const size_t w4 = colsum_workspace_bytes(static_cast<long long>(LC));
  if (w4 > wsb) wsb = w4;
  const size_t w5 = colsum_workspace_bytes(static_cast<long long>(T) * Q * C);   // frame-term reduction
  if (w5 > wsb) wsb = w5;
  RC(bw_ws.reserve(wsb));
  float* ga = static_cast<float*>(bw_a.ptr);
  float* gb = static_cast<float*>(bw_b.ptr);
  float* dhs = static_cast<float*>(bw_c.ptr);
  float* dx = static_cast<float*>(bw_d.ptr);
  float* tmp = dx + RC_;
  float* tmp2 = tmp + RC_;
  float* dqkv = static_cast<float*>(bw_t3.ptr);
  bf16* dKall = static_cast<bf16*>(bw_dk.ptr);
  bf16* dVall = static_cast<bf16*>(bw_dv.ptr);
  const float* qpos = weights.get("query_embed.weight");
  const bf16* Kall = static_cast<const bf16*>(ws_k.ptr);
  const bf16* Vall = static_cast<const bf16*>(ws_v.ptr);

  // ---- The weight gradients run on a second stream beside the data-gradient chain: at the query side's sizes neither
  // fills the GPU (208-CTA launches, latency-bound).  fork() orders a weight gradient after everything issued so far;
  // side_reads(slot) marks the scratch buffer it still reads, before_write(slot) makes the main stream wait for that
  // reader before a later kernel overwrites the buffer.
  enum { SL_DX = 0, SL_GA, SL_GB, SL_TMP2, SL_DQKV, SL_N };
  if (bw_side == nullptr) {
    HH_CHECK_CUDA(cudaStreamCreateWithFlags(&bw_side, cudaStreamNonBlocking));
    HH_CHECK_CUDA(cudaEventCreateWithFlags(&bw_fork, cudaEventDisableTiming));
    for (int i = 0; i < SL_N; ++i) HH_CHECK_CUDA(cudaEventCreateWithFlags(&bw_done[i], cudaEventDisableTiming));
  }
  cudaStream_t sw = bw_side;
  bool pending[SL_N] = {false, false, false, false, false};
  auto fork = [&]() -> int {
    HH_CHECK_CUDA(cudaEventRecord(bw_fork, s));
    HH_CHECK_CUDA(cudaStreamWaitEvent(sw, bw_fork, 0));
    return 0;
  };
  auto side_reads = [&](int slot) -> int {
    HH_CHECK_CUDA(cudaEventRecord(bw_done[slot], sw));
    pending[slot] = true;
    return 0;
  };
  auto before_write = [&](int slot) -> int {
    if (!pending[slot]) return 0;
    HH_CHECK_CUDA(cudaStreamWaitEvent(s, bw_done[slot], 0));
    pending[slot] = false;
    return 0;
  };

  if (d_hs) HH_CHECK_CUDA(cudaMemcpyAsync(dhs, d_hs, LR * C * 4, cudaMemcpyDeviceToDevice, s));
  else HH_CHECK_CUDA(cudaMemsetAsync(dhs, 0, LR * C * 4, s));

  // =========================================================================================== heads
  if (d_boxes) {
    const float* box_in = traj ? sv_cond : hs;
    const int RB = static_cast<int>(rows_box);
    // layer 2: boxes = sigmoid(x2 W3^T + b3)
    RC(fork());
    RC(wgrad(d_boxes, 4, boxes, 4, 2, sv_x2, C, nullptr, 0, G("bbox_embed.layers.2.weight"), C, G("bbox_embed.layers.2.bias"), RB,
             4, C, 0.f, 1.f, sw));
    RC(dgrad(d_boxes, 4, boxes, 4, 2, weights.get("bbox_embed.layers.2.weight"), ga, C, RB, 4, C, 0.f, s));
    // layer 1: x2 = relu(x1 W2^T + b2)
    RC(fork());
    RC(wgrad(ga, C, sv_x2, C, 1, sv_x1, C, nullptr, 0, G("bbox_embed.layers.1.weight"), C, G("bbox_embed.layers.1.bias"), RB, C, C,
             0.f, 1.f, sw));
    RC(side_reads(SL_GA));
    RC(dgrad(ga, C, sv_x2, C, 1, weights.get("bbox_embed.layers.1.weight"), gb, C, RB, C, C, 0.f, s));
    // layer 0: x1 = relu(box_in W1^T + b1)
    RC(fork());
    RC(wgrad(gb, C, sv_x1, C, 1, box_in, C, nullptr, 0, G("bbox_embed.layers.0.weight"), C, G("bbox_embed.layers.0.bias"), RB, C, C,
             0.f, 1.f, sw));
    RC(side_reads(SL_GB));
    if (!traj) {
      RC(dgrad(gb, C, sv_x1, C, 1, weights.get("bbox_embed.layers.0.weight"), dhs, C, RB, C, C, 1.f, s));  // box_in = hs
    } else {
      RC(before_write(SL_GA));
      RC(dgrad(gb, C, sv_x1, C, 1, weights.get("bbox_embed.layers.0.weight"), ga, C, RB, C, C, 0.f, s));   // ga = d cond
      RC(before_write(SL_GB));   // dhsproj / dft / dsum live in gb
      // cond[lb,t,q] = hs[lb,q] Wf1^T + (frame_index[t] Wf2^T + bf)      (tfm_decoder.py:212-215)
      float* dhsproj = gb;
      float* dft = gb + LR * C;
      float* dsum = dft + static_cast<size_t>(T) * C;   // [T, Q, C]: d cond summed over (layer, clip)
      if (static_cast<size_t>(T) * Q * C + LR * C + static_cast<size_t>(T) * C <= big) {
        // dft sums 4992 rows per output at the c4 shape: the (layer, clip) reduction goes through the 64-way column-sum
        // kernels first (one thread per output walking all rows took 0.83 ms), the T rows of dft only sum Q rows then
        dim3 grid((C + 127) / 128, static_cast<unsigned>(LR));
        frame_term_bwd_kernel<<<grid, 128, 0, s>>>(ga, dhsproj, dft, Lr * B, T, Q, C, 0);
        const long long tqc = static_cast<long long>(T) * Q * C;
        RC(colsum_rows(ga, 0, tqc, static_cast<long long>(Lr) * B, tqc, 0.f, dsum, bw_ws.ptr, s));
        dim3 grid2((C + 127) / 128, static_cast<unsigned>(T));
        frame_term_bwd_kernel<<<grid2, 128, 0, s>>>(dsum, dhsproj, dft, 1, T, Q, C, Q);
      } else {
        dim3 grid((C + 127) / 128, static_cast<unsigned>(LR + T));
        frame_term_bwd_kernel<<<grid, 128, 0, s>>>(ga, dhsproj, dft, Lr * B, T, Q, C, 0);
      }
      HH_CHECK_LAUNCH("frame_term_bwd_kernel");
      float* dWf = G("frame_proj.weight");  // [C, 2C] = [Wf1 | Wf2]
      RC(fork());
      RC(wgrad(dhsproj, C, nullptr, 0, 0, hs, C, nullptr, 0, dWf, 2 * C, nullptr, static_cast<int>(LR), C, C, 0.f, 1.f, sw));
      RC(dgrad(dhsproj, C, nullptr, 0, 0, static_cast<const float*>(w_f1.ptr), dhs, C, static_cast<int>(LR), C, C, 1.f, s));
      RC(fork());
      RC(wgrad(dft, C, nullptr, 0, 0, weights.get("frame_index.weight"), C, nullptr, 0, dWf + C, 2 * C, G("frame_proj.bias"), T, C,
               C, 0.f, 1.f, sw));
      RC(side_reads(SL_GB));
      RC(dgrad(dft, C, nullptr, 0, 0, static_cast<const float*>(w_f2.ptr), G("frame_index.weight"), C, T, C, C, 0.f, s));
    }
  }

  // =========================================================================================== decoder layers
  HH_CHECK_CUDA(cudaMemsetAsync(dx, 0, RC_ * 4, s));  // gradient w.r.t. the residual stream after the current layer
  const DropCfg dr = saved_drop;   // the masks of the matching forward, regenerated
  auto ln_bwd = [&](const float* x, const std::string& nm, const float* dy, float beta_w) {
    LnBwdArgs a{};
    a.x = x; a.ldx = C; a.w = weights.get(nm + ".weight"); a.eps = 1e-5f; a.dy = dy; a.lddy = C;
    a.dx = dx; a.beta_dx = 1.f;  // accumulates into the residual-stream gradient
    a.dgamma = G(nm + ".weight"); a.dbeta = G(nm + ".bias"); a.beta_w = beta_w;
    a.workspace = bw_ws.ptr; a.M = R; a.D = C;
    return ln_backward_rows(a, s);
  };
  for (int i = Lr - 1; i >= 0; --i) {
    const std::string p = "transformer.decoder.layers." + std::to_string(i) + ".";
    const LayerBufs& A = saved[i];
    const float* wsa = static_cast<const float*>(w_sa.ptr) + static_cast<size_t>(i) * 3 * C * C;
    // hs_i = norm(x3): its gradient joins the stream (the norm's weights are shared by all layers: accumulate)
    RC(before_write(SL_DX));
    RC(ln_bwd(A.x3, "transformer.decoder.norm", dhs + static_cast<size_t>(i) * RC_, i == Lr - 1 ? 0.f : 1.f));
    // ---- FFN: x3 = x2 + drop3(drop(relu(n3 W1^T + b1)) W2^T + b2).  A.f is the hidden AFTER its dropout, so
    // f > 0 <=> (ReLU active and kept) and the inner dropout is only the factor 1/(1-p) on the ReLU derivative
    const uint32_t st0 = static_cast<uint32_t>(i) * 8;
    const float fscale = dr.thr ? dr.scale : 1.f;
    RC(fork());
    RC(wgrad(dx, C, nullptr, 0, 0, A.f, Fd, nullptr, 0, G(p + "linear2.weight"), Fd, G(p + "linear2.bias"), R, C, Fd, 0.f, 1.f, sw,
             dr, st0 + 5));
    RC(side_reads(SL_DX));
    RC(before_write(SL_GA));
    RC(dgrad(dx, C, nullptr, 0, 0, weights.get(p + "linear2.weight"), ga, Fd, R, C, Fd, 0.f, s, dr, st0 + 5));  // ga = d f
    RC(fork());
    RC(wgrad(ga, Fd, A.f, Fd, 1, A.n3, C, nullptr, 0, G(p + "linear1.weight"), C, G(p + "linear1.bias"), R, Fd, C, 0.f, 1.f, sw,
             drop_off(), 0, fscale));
    RC(side_reads(SL_GA));
    RC(dgrad(ga, Fd, A.f, Fd, 1, weights.get(p + "linear1.weight"), tmp, C, R, Fd, C, 0.f, s, drop_off(), 0, fscale));  // tmp = d n3
    RC(before_write(SL_DX));
    RC(ln_bwd(A.x2, p + "norm3", tmp, 0.f));
    // ---- cross attention: x2 = x1 + CA(qc, K_i, V_i) Wo^T + bo,  qc = s ((n2 + qpos) Wq^T + bq)
    RC(fork());
    RC(wgrad(dx, C, nullptr, 0, 0, A.o2, C, nullptr, 0, G(p + "multihead_attn.out_proj.weight"), C,
             G(p + "multihead_attn.out_proj.bias"), R, C, C, 0.f, 1.f, sw, dr, st0 + 3));
    RC(side_reads(SL_DX));
    RC(dgrad(dx, C, nullptr, 0, 0, weights.get(p + "multihead_attn.out_proj.weight"), tmp, C, R, C, C, 0.f, s, dr, st0 + 3));  // tmp = d o2
    RC(before_write(SL_TMP2));
    RC(cross_attn_bwd(A.qc, Kall + static_cast<size_t>(i) * C, Vall + static_cast<size_t>(i) * C, Lr * C, A.o2, tmp, tmp2,
                      dKall + static_cast<size_t>(i) * C, dVall + static_cast<size_t>(i) * C, Lr * C, B, Q, heads, S, bw_ws.ptr, s,
                      dr, st0 + 2, A.lse));
    float* dWca = G(p + "multihead_attn.in_proj_weight");
    float* dbca = G(p + "multihead_attn.in_proj_bias");
    RC(fork());
    RC(wgrad(tmp2, C, nullptr, 0, 0, A.n2, C, qpos, Q, dWca, C, dbca, R, C, C, 0.f, qscale, sw));                // rows [0, C): Wq
    RC(side_reads(SL_TMP2));
    RC(dgrad(tmp2, C, nullptr, 0, 0, static_cast<const float*>(w_caq.ptr) + static_cast<size_t>(i) * C * C, tmp, C, R, C, C, 0.f, s));
    RC(colsum_rows(tmp, 0, static_cast<long long>(Q) * C, B, static_cast<long long>(Q) * C, 1.f, G("query_embed.weight"),
                   bw_ws.ptr, s));                                                                               // d qpos
    RC(before_write(SL_DX));
    RC(ln_bwd(A.x1, p + "norm2", tmp, 0.f));
    // ---- self attention: x1 = x0 + SA(q, k, v) Wo^T + bo;  q, k from n1 + qpos, v from n1
    RC(fork());
    RC(wgrad(dx, C, nullptr, 0, 0, A.o1, C, nullptr, 0, G(p + "self_attn.out_proj.weight"), C, G(p + "self_attn.out_proj.bias"),
             R, C, C, 0.f, 1.f, sw, dr, st0 + 1));
    RC(side_reads(SL_DX));
    RC(dgrad(dx, C, nullptr, 0, 0, weights.get(p + "self_attn.out_proj.weight"), tmp, C, R, C, C, 0.f, s, dr, st0 + 1));  // tmp = d o1
    RC(before_write(SL_DQKV));
    RC(self_attn_bwd(A.qkv, A.qkv + C, A.qkv + 2 * C, 3 * C, tmp, dqkv, dqkv + C, dqkv + 2 * C, 3 * C, B, Q, heads, s, dr, st0 + 0));
    float* dWsa = G(p + "self_attn.in_proj_weight");
    float* dbsa = G(p + "self_attn.in_proj_bias");
    RC(fork());
    RC(wgrad(dqkv, 3 * C, nullptr, 0, 0, A.n1, C, qpos, Q, dWsa, C, dbsa, R, C, C, 0.f, qscale, sw));            // Wq (pre-scaled q)
    RC(fork());
    RC(wgrad(dqkv + C, 3 * C, nullptr, 0, 0, A.n1, C, qpos, Q, dWsa + static_cast<size_t>(C) * C, C, dbsa + C, R, C, C, 0.f, 1.f, sw));
    RC(fork());
    RC(wgrad(dqkv + 2 * C, 3 * C, nullptr, 0, 0, A.n1, C, nullptr, 0, dWsa + static_cast<size_t>(2) * C * C, C, dbsa + 2 * C, R, C,
             C, 0.f, 1.f, sw));
    RC(side_reads(SL_DQKV));
    RC(dgrad(dqkv, 3 * C, nullptr, 0, 0, wsa, tmp, C, R, 2 * C, C, 0.f, s));                                     // d(n1 + qpos) via q, k
    RC(colsum_rows(tmp, 0, static_cast<long long>(Q) * C, B, static_cast<long long>(Q) * C, 1.f, G("query_embed.weight"),
                   bw_ws.ptr, s));
    RC(dgrad(dqkv + 2 * C, 3 * C, nullptr, 0, 0, wsa + static_cast<size_t>(2) * C * C, tmp, C, R, C, C, 1.f, s));  // + via v
    RC(before_write(SL_DX));
    RC(ln_bwd(A.x0, p + "norm1", tmp, 0.f));
  }
  // join: the memory side reuses ga / gb, and the caller reads the gradients in stream order
  HH_CHECK_CUDA(cudaEventRecord(bw_fork, sw));
  HH_CHECK_CUDA(cudaStreamWaitEvent(s, bw_fork, 0));
  // dx now holds the gradient w.r.t. the zero-initialised tgt: no parameter behind it

  // =========================================================================================== memory side
  // bias gradients of the K / V projections: column sums over all tokens
  float* dbk = static_cast<float*>(bw_t1.ptr);
  float* dbv = dbk + LC;
  float* dWk = dbv + LC;
  float* dWv = dWk + static_cast<size_t>(LC) * C;
  RC(colsum_rows(dKall, 1, LC, M, LC, 0.f, dbk, bw_ws.ptr, s));
  RC(colsum_rows(dVall, 1, LC, M, LC, 0.f, dbv, bw_ws.ptr, s));
  // weight gradients: dWk_all [L*C, C] = dK_all^T (mem + pos), dWv_all = dV_all^T mem   (reduction over B*S)
  bf16* gT = static_cast<bf16*>(bw_t2.ptr);             // [L*C, BS]
  bf16* xT = gT + static_cast<size_t>(LC) * BS;         // [C, BS]
  bf16* fT = xT + static_cast<size_t>(C) * BS;          // [F, BS] (later)
  RC(transpose_to_bf16(dKall, 1, LC, gT, M, LC, s));
  RC(transpose_to_bf16(ws_mempos.ptr, 1, C, xT, M, C, s));
  RC(gemm_bf16(gT, M, xT, M, dWk, C, nullptr, nullptr, 0, LC, C, M, EPI_BIAS_F32, s));
  RC(transpose_to_bf16(dVall, 1, LC, gT, M, LC, s));
  RC(transpose_to_bf16(ws_mem.ptr, 1, C, xT, M, C, s));
  RC(gemm_bf16(gT, M, xT, M, dWv, C, nullptr, nullptr, 0, LC, C, M, EPI_BIAS_F32, s));
  for (int i = 0; i < Lr; ++i) {
    const std::string p = "transformer.decoder.layers." + std::to_string(i) + ".";
    float* dWca = G(p + "multihead_attn.in_proj_weight");
    float* dbca = G(p + "multihead_attn.in_proj_bias");
    const size_t cc = static_cast<size_t>(C) * C;
    HH_CHECK_CUDA(cudaMemcpyAsync(dWca + cc, dWk + i * cc, cc * 4, cudaMemcpyDeviceToDevice, s));
    HH_CHECK_CUDA(cudaMemcpyAsync(dWca + 2 * cc, dWv + i * cc, cc * 4, cudaMemcpyDeviceToDevice, s));
    HH_CHECK_CUDA(cudaMemcpyAsync(dbca + C, dbk + static_cast<size_t>(i) * C, C * 4, cudaMemcpyDeviceToDevice, s));
    HH_CHECK_CUDA(cudaMemcpyAsync(dbca + 2 * C, dbv + static_cast<size_t>(i) * C, C * 4, cudaMemcpyDeviceToDevice, s));
  }
  // data gradients: d(mem + pos) = dK_all Wk_all ; d mem = d(mem + pos) + dV_all Wv_all
  float* dmem = ga;
  RC(gemm_bf16(dKall, LC, static_cast<const bf16*>(w_kallT.ptr), LC, dmem, C, nullptr, nullptr, 0, M, C, LC, EPI_BIAS_F32, s));
  float* dpos = gb;
  RC(colsum_rows(dmem, 0, static_cast<long long>(S) * C, B, static_cast<long long>(S) * C, 0.f, dpos, bw_ws.ptr, s));
  {
    dim3 grid((C + 127) / 128, static_cast<unsigned>(1 + n + T));
    pos3d_bwd_kernel<<<grid, 128, 0, s>>>(dpos, G("pos_embed"), G("temporal_embed"), T, n, C);
    HH_CHECK_LAUNCH("pos3d_bwd_kernel");
  }
  // d mem = d(mem + pos) + dV_all Wv_all.  The second product goes to its own buffer (gb: the position sums above are consumed)
  // and pre_norm's backward adds the two: the in-place residual epilogue only exists on the unclustered 1-SM GEMM path
  // (0.87 ms for this launch against 0.13 ms for its twin above).
  float* dmem2 = gb;
  RC(gemm_bf16(dVall, LC, static_cast<const bf16*>(w_vallT.ptr), LC, dmem2, C, nullptr, nullptr, 0, M, C, LC, EPI_BIAS_F32, s));
  // pre_norm backward: memf (fp32, pre-norm) saved by the forward; the bf16 gradient feeds the proj weight GEMM
  bf16* dmemf16 = dKall;  // dK_all is dead: reuse its storage ([BS, C] bf16 fits)
  {
    LnBwdArgs a{};
    a.x = static_cast<const float*>(ws_memf.ptr); a.ldx = C; a.w = weights.get("transformer.pre_norm.weight"); a.eps = 1e-5f;
    a.dy = dmem; a.dy2 = dmem2; a.lddy = C; a.dx16 = dmemf16;
    a.dgamma = G("transformer.pre_norm.weight"); a.dbeta = G("transformer.pre_norm.bias"); a.beta_w = 0.f;
    a.workspace = bw_ws.ptr; a.M = M; a.D = C;
    RC(ln_backward_rows(a, s));
  }
  // proj.weight [C, F] = d memf^T feat
  RC(transpose_to_bf16(dmemf16, 1, C, xT, M, C, s));
  RC(transpose_to_bf16(ws_feat.ptr, 1, F, fT, M, F, s));
  RC(gemm_bf16(xT, M, fT, M, G("proj.weight"), F, nullptr, nullptr, 0, C, F, M, EPI_BIAS_F32, s));
  return 0;
}

}  // namespace hh
