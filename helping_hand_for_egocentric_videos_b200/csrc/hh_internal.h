// Internal (C++) interface between the kernel translation units and the C-ABI layer.
#pragma once
#include <cstddef>
#include <cstdint>
#include <string>

#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "hh_rng.cuh"

namespace hh {

typedef __nv_bfloat16 bf16;

// Thread-local last error (reported through hh_last_error()).
void set_error(const std::string& msg);
const char* last_error_cstr();
int fail(int code, const std::string& msg);  // records msg, returns code

#define HH_CHECK_CUDA(expr)                                                                         \
  do {                                                                                              \
    cudaError_t _e = (expr);                                                                        \
    if (_e != cudaSuccess)                                                                          \
      return ::hh::fail(-3, std::string(#expr) + ": " + cudaGetErrorString(_e));                    \
  } while (0)

#define HH_CHECK_LAUNCH(name)                                                                       \
  do {                                                                                              \
    cudaError_t _e = cudaGetLastError();                                                            \
    if (_e != cudaSuccess) return ::hh::fail(-3, std::string(name) + ": " + cudaGetErrorString(_e)); \
  } while (0)

#define HH_REQUIRE(cond, msg)                                         \
  do {                                                                \
    if (!(cond)) return ::hh::fail(-2, std::string(msg) + " [" #cond "]"); \
  } while (0)

int num_sms();

// ---------------------------------------------------------------- GEMM (gemm_tcgen05.cu)
enum GemmEpilogue {
  EPI_BIAS_BF16 = 0,        // out bf16 = acc + bias
  EPI_BIAS_QGELU_BF16 = 1,  // out bf16 = quickgelu(acc + bias)
  EPI_BIAS_RES_F32 = 2,     // out f32  = acc + bias + residual (residual may alias out)
  EPI_BIAS_F32 = 3,         // out f32  = acc + bias
  // LayerNorm folded into the contraction (GemmFuse): A holds the UN-normalised rows z (bf16), W the gamma-scaled
  // weight; out = act(rstd * (acc - mean * colsum) + bias') with mean / rstd from the producer's row statistics
  EPI_LN_BIAS_BF16 = 4,
  EPI_LN_BIAS_QGELU_BF16 = 5,
  // out bf16 = z = acc + bias + residual (fp32), per-row (sum z, sum z^2) partials per column tile, optionally
  // residual <- z in place (fp32): the producer side of the folded LayerNorm
  EPI_RES_STATS_BF16 = 6,
};
// Extra operands of the fused-LayerNorm epilogues (model/LaviLa.py:353-388: norm1/2/3 + residual adds).
struct GemmFuse {
  const float* colsum = nullptr;    // EPI_LN_*: fp32 [N], sum_k W'[n, k] of the bf16 weight actually multiplied
  const float* stats_in = nullptr;  // EPI_LN_*: fp32 [parts][M][2]
  int stats_parts = 0;
  int norm_dim = 0;                 // width the statistics were taken over (= K)
  float eps = 0.f;
  float* stats_out = nullptr;       // EPI_RES_STATS_BF16: fp32 [gemm_stats_parts(M, N)][M][2]
  int writeback = 0;                // EPI_RES_STATS_BF16: residual <- acc + bias + residual (fp32, in place)
};
// Number of column tiles (= statistics partials per row) EPI_RES_STATS_BF16 uses for an [M, N] output.
int gemm_stats_parts(int M, int N);
int gemm_bf16_fused(const bf16* A, int lda, const bf16* W, int ldw, void* out, int ldc, const float* bias,
                    float* residual, int ldr, int M, int N, int K, int epilogue, const GemmFuse& fuse,
                    cudaStream_t stream);
// C[M,N] = epilogue(A[M,K] * W[N,K]^T); A, W bf16 with K contiguous. bias fp32 [N] or nullptr.
int gemm_bf16(const bf16* A, int lda, const bf16* W, int ldw, void* out, int ldc, const float* bias,
              const float* residual, int ldr, int M, int N, int K, int epilogue, cudaStream_t stream);
// gemm_bf16 (EPI_BIAS_BF16 / EPI_BIAS_F32) over A rows in segments: logical row m is row m + (m / seg_rows) *
// (seg_pitch - seg_rows) of A (row stride lda), i.e. M / seg_rows segments of seg_rows rows that start seg_pitch rows
// apart (per-clip patch rows of a feature map whose CLS rows are skipped).  seg_rows % 128 == 0 (every 128-row tile
// lies in one segment), M % seg_rows == 0, seg_pitch >= seg_rows.
int gemm_bf16_rowseg(const bf16* A, int lda, int seg_rows, int seg_pitch, const bf16* W, int ldw, void* out, int ldc,
                     const float* bias, int M, int N, int K, int epilogue, cudaStream_t stream);

// ---------------------------------------------------------------- row-wise kernels (rows.cu)
// y = LayerNorm(x (+ add_rows_mod)) * w + b.  x fp32 [M, D] (row stride ldx). Outputs (any may be null):
//   out_f32 [M,D], out_bf16 [M,D], and out2 = y + post_add[row % post_mod] (bf16 and/or f32).
struct LnArgs {
  const float* x; int ldx;
  const bf16* delta;    // optional bf16 [M, D]: the norm is taken of x + delta (fused residual add)
  const bf16* delta2;   // optional second bf16 [M, D] (only with delta): (x + delta) + delta2
  float* xsum_out;      // optional fp32 [M, D]: receives x + delta (may alias x)
  const float* w; const float* b; float eps;
  float* out_f32; bf16* out_bf16;
  const float* post_add; int post_mod;   // optional positional term added after the norm
  float* out2_f32; bf16* out2_bf16;
  int M, D;
  float* cls_f32; int cls_mod;   // optional fp32 [M / cls_mod, D]: rows with row % cls_mod == 0 also go here (CLS rows)
};
int layernorm_rows(const LnArgs& a, cudaStream_t stream);

// fp32 or bf16 (strided rows) -> bf16 contiguous [rows, cols]: row r = (r / inner) * outer_stride + (r % inner) * row_stride.
int cast_rows_bf16(const float* src, long long outer_stride, long long row_stride, int inner, bf16* dst, int rows,
                   int cols, cudaStream_t stream);
int cast_rows_bf16(const bf16* src, long long outer_stride, long long row_stride, int inner, bf16* dst, int rows,
                   int cols, cudaStream_t stream);

// ---------------------------------------------------------------- encoder satellites (embed.cu)
// video fp32 [B*T,3,H,W] -> patches bf16 [B*T*n, Kp] (k = c*p*p + i*p + j, zero padded to Kp).
int im2col_patches(const float* video, bf16* out, int BT, int H, int W, int p, int Kp, cudaStream_t stream);
// frames uint8 [B*T,H,W,3] -> the same patch matrix with ((u/255) - mean[c]) / std[c] applied on the fly (host arrays).
int im2col_patches_u8(const uint8_t* frames, const float* mean, const float* stdv, bf16* out, int BT, int H, int W, int p,
                      int Kp, cudaStream_t stream);
// x[b, 0] = LN(cls + pos[0]); x[b, 1 + f*n + q] = LN(tok[(b*T+f)*n + q] + pos[1+q] + temporal[f]);  eps 1e-5
// Optional (both or neither): z16 bf16 [B*N, D] = bf16(x) and stats fp32 [B*N][2] = per-row (sum x, sum x^2) -- the
// operands of the first folded-LayerNorm GEMM (one statistics partial per row).
int assemble_tokens_ln(const float* tok, const float* cls, const float* pos, const float* temporal, const float* w,
                       const float* b, float eps, float* x, int B, int T, int n, int D, cudaStream_t stream,
                       bf16* z16 = nullptr, float* stats = nullptr);

// ---------------------------------------------------------------- divided space-time attention (attn_*.cu)
// qkv bf16 [B*N, 3*D] (q pre-scaled), N = 1 + T*n, heads of 64. out bf16 [B*N, D]; patch rows only.
// Both write every row of out, including the CLS query row (out[b*N + 0]), which attends all N keys; its partial
// softmax states go through `cls_ws` (attn_cls_workspace_bytes) and are folded by attn_cls_merge.
size_t attn_cls_workspace_bytes(int B, int T, int n, int H);
int attn_space(const bf16* qkv, bf16* out, int B, int T, int n, int H, float* cls_ws, cudaStream_t stream);
int attn_time(const bf16* qkv, bf16* out, int B, int T, int n, int H, float* cls_ws, cudaStream_t stream);
// attn_time for T <= 16 (attn_time_v2.cu)
int attn_time_v2(const bf16* qkv, bf16* out, int B, int T, int n, int H, float* cls_ws, int pchunk, int nchunks,
                 cudaStream_t stream);
// tcgen05/TMEM implementation of attn_space for n <= 256 (attn_space dispatches to it)
bool attn_space_tc_supported(int n);
int attn_space_tc(const bf16* qkv, bf16* out, int B, int T, int n, int H, float* cls_ws, cudaStream_t stream);
int attn_cls_merge(const bf16* qkv, const float* parts, bf16* out, int B, int N, int H, int nparts, cudaStream_t stream);
// Stand-alone CLS query row (reference statement of the fused path; used when T > 16).
int attn_cls(const bf16* qkv, bf16* out, int B, int N, int H, cudaStream_t stream);

// Causal self-attention of the CLIP text tower (text.cu): qkv bf16 [G*L, 3*H*64] (q pre-scaled) -> out bf16 [G*L, H*64]
int attn_causal(const bf16* qkv, bf16* out, int G, int L, int H, cudaStream_t stream);

// ---------------------------------------------------------------- decoder satellites (decoder.cu)
// Most learned queries per clip the decoder takes (ObjDecoder num_queries = nq + 1).  Every query-side array, tile and
// workspace size is derived from it: one warp lane per query in the self attention, two 16-row query blocks in the
// tensor-core cross-attention kernels.
constexpr int kMaxQueries = 32;
// Small-M fp32 linear: out[R,N] = act((in[R,K] (+ in_add[r % add_mod, K])) * W[N,K]^T + bias) (+ residual[R,N]).
struct LinArgs {
  const float* in; int ldi;
  const float* in_add; int add_mod;       // optional, row-periodic (query_pos)
  const float* W; const float* bias;      // W fp32 [N,K] row-major
  const float* residual; int ldres;       // optional
  float* out; int ldo;
  int R, N, K;
  int act;                                // 0 none, 1 relu, 2 sigmoid
  int in_relu;                            // 1: apply ReLU to the input first (txt_proj = ReLU -> Linear)
  DropCfg drop; uint32_t drop_site;       // training: dropout on act(x W^T + b) before the residual add, idx = row*N + col
};
int linear_f32(const LinArgs& a, cudaStream_t stream);          // lin3.cu (pipelined); shapes it refuses go to:
int linear_f32_legacy(const LinArgs& a, cudaStream_t stream);   // decoder.cu
// Query self-attention: q,k,v fp32 [B*Q, C] (q pre-scaled), heads of 64 -> out fp32 [B*Q, C].
// drop: dropout on the attention probabilities (training), idx = ((b*heads + h)*Q + i)*Q + j
int self_attn_queries(const float* q, const float* k, const float* v, int ld, float* out, int B, int Q, int heads,
                      cudaStream_t stream, DropCfg drop = drop_off(), uint32_t drop_site = 0);
// Query -> patch cross attention. q fp32 [B*Q, C] (pre-scaled); K,V bf16 rows [B*S] with row stride ldkv, head h at
// column h*64.  Output fp32 [B*Q, C].  workspace: see cross_attn_workspace_bytes.
size_t cross_attn_workspace_bytes(int B, int Q, int heads, int S);
// drop: dropout on the attention probabilities (training), idx = ((b*heads + h)*Q + i)*S + j
int cross_attn(const float* q, const bf16* K, const bf16* V, int ldkv, float* out, int B, int Q, int heads, int S,
               void* workspace, cudaStream_t stream, DropCfg drop = drop_off(), uint32_t drop_site = 0,
               float* lse_out = nullptr);   // lse_out: optional fp32 [B*heads, Q] row log-sum-exp for cross_attn_bwd
// fp32 SIMT statement of cross_attn for differential tests: Q <= 16 only
size_t cross_attn_simt_workspace_bytes(int B, int Q, int heads, int S);
int cross_attn_simt(const float* q, const bf16* K, const bf16* V, int ldkv, float* out, int B, int Q, int heads, int S,
                    void* workspace, cudaStream_t stream);
// boxes[l, b*T+t, q, :] head input: cond = hsproj[l,b,q,:] + frameterm[t,:]  (ObjDecoder frame_proj split)
int add_frame_term(const float* hsproj, const float* frameterm, float* out, int LB, int T, int Q, int C,
                   cudaStream_t stream);
int f32_to_bf16(const float* src, bf16* dst, size_t n, cudaStream_t stream);
// weight packing: dst bf16 [rows, cols_out] = src fp32 [rows, cols_in] (zero padded), first `scaled_rows` rows * scale
int pack_weight_bf16(const float* src, bf16* dst, int rows, int cols_in, int cols_out, int scaled_rows, float scale,
                     cudaStream_t stream);
// LayerNorm(gamma, beta) folded into the Linear (W fp32 [rows, K], bias may be null) that follows it: Wf bf16 [rows, K],
// colsum fp32 [rows], bias_f fp32 [rows]; the first `scaled_rows` rows (and their bias) are multiplied by `scale`.
int fold_ln_weight(const float* W, const float* gamma, const float* beta, const float* bias, bf16* Wf, float* colsum,
                   float* bias_f, int rows, int K, int scaled_rows, float scale, cudaStream_t stream);
// dst[i] = src[i] * (i < scaled ? scale : 1)
int scale_copy_f32(const float* src, float* dst, size_t n, size_t scaled, float scale, cudaStream_t stream);
// dst[r, :cols] = src[r, col0 : col0+cols]  (src row stride lds)
int slice_cols_f32(const float* src, int lds, int col0, float* dst, int rows, int cols, cudaStream_t stream);
// pos[t*n + p, :] = pos_embed[1 + p, :] + temporal[t, :]   (both encoders' tiled position embedding)
int build_pos3d(const float* pos_embed, const float* temporal, float* out, int T, int n, int C, cudaStream_t stream);
// x / max(||x||, eps) per row
int l2_normalize_rows(const float* x, float* out, int rows, int cols, float eps, cudaStream_t stream);
int expand_logits(const float* src, float* dst, int LB, int rep, size_t per, cudaStream_t stream);

// ---------------------------------------------------------------- decoder backward primitives (decoder_bwd.cu)
// nn.Linear backward.  g = act'(dY, Y) (act 0 none, 1 relu, 2 sigmoid; Y = saved output).
//   dgrad: dX[R,K] = beta*dX + g W           (W fp32 [N,K])
//   wgrad: dW[N,K] = beta*dW + scale * g^T x,  x = relu?(X + x_add[r % add_mod]);  db[N] = beta*db + scale * sum_r g
struct LinBwdArgs {
  const float* dY; int ldy;
  const float* Y; int ldyo; int act;
  const float* W;
  const float* X; int ldx;
  const float* x_add; int add_mod; int in_relu;
  float* dX; int lddx;  // dgrad output
  float* dW; int ldw;   // wgrad outputs
  float* db;
  int R, N, K;
  float beta, scale;
  int rows_per_split;   // set by linear_wgrad_f32
  DropCfg drop; uint32_t drop_site;   // the forward dropped act(.) [R, N] (idx = row*N + col): g = act'(dY * mult, Y)
  float act_scale;                    // 0 = 1; extra factor on act'(.) (ReLU followed by dropout: kept <=> Y > 0)
};
int linear_dgrad_f32(const LinBwdArgs& a, cudaStream_t s);
int linear_wgrad_f32(const LinBwdArgs& a, cudaStream_t s);
int linear_dgrad_f32_legacy(const LinBwdArgs& a, cudaStream_t s);
int linear_wgrad_f32_legacy(const LinBwdArgs& a, cudaStream_t s);
// LayerNorm backward over rows of x (+ optional bf16 delta, as in the forward).  dy fp32 or bf16 (row stride lddy).
// dx = beta_dx * dx + grad (fp32, contiguous rows) and/or dx16 (bf16);  dgamma/dbeta = beta_w * old + sum over rows.
struct LnBwdArgs {
  const float* x; int ldx; const bf16* delta;
  const float* w; float eps;
  const float* dy; const bf16* dy16; int lddy;
  const float* dy2;                 // optional second fp32 addend of dy (same pitch)
  float* dx; bf16* dx16; float beta_dx;
  float* dgamma; float* dbeta; float beta_w;
  void* workspace;  // ln_backward_workspace_bytes(M, D) when dgamma is requested
  int M, D;
};
size_t ln_backward_workspace_bytes(int M, int D);
int ln_backward_rows(const LnBwdArgs& a, cudaStream_t s);
// backward of self_attn_queries: dq/dk/dv rows have stride ldg (same packing as the forward's q/k/v with stride ld)
int self_attn_bwd(const float* q, const float* k, const float* v, int ld, const float* dO, float* dq, float* dk, float* dv,
                  int ldg, int B, int Q, int heads, cudaStream_t s, DropCfg drop = drop_off(), uint32_t drop_site = 0);
// backward of cross_attn: dq fp32 [B*Q, C]; dK, dV bf16 rows [B*S] with stride lddkv (head h at column h*64)
size_t cross_attn_bwd_workspace_bytes(int B, int Q, int heads, int S);
int cross_attn_bwd(const float* q, const bf16* K, const bf16* V, int ldkv, const float* O, const float* dO, float* dq,
                   bf16* dK, bf16* dV, int lddkv, int B, int Q, int heads, int S, void* workspace, cudaStream_t s,
                   DropCfg drop = drop_off(), uint32_t drop_site = 0,
                   const float* lse_saved = nullptr);   // the forward's lse_out; recomputed from q, K when absent
// cross_attn_bwd.cu runs the tensor-core kernel; the first-generation SIMT statement (decoder_bwd.cu) serves unaligned
// q / dO / dK / dV and dropout with S % 8 != 0
size_t cross_attn_bwd_simt_workspace_bytes(int B, int Q, int heads, int S);
int cross_attn_bwd_simt(const float* q, const bf16* K, const bf16* V, int ldkv, const float* O, const float* dO, float* dq,
                        bf16* dK, bf16* dV, int lddkv, int B, int Q, int heads, int S, void* workspace, cudaStream_t s,
                        DropCfg drop, uint32_t drop_site, const float* lse_saved);
int cross_lse(const float* q, const bf16* K, int ldkv, float* lse, int B, int Q, int heads, int S, cudaStream_t s);
// out[c] = beta*out[c] + sum_r X[r, c]  (X fp32 or bf16, row stride ld); workspace colsum_workspace_bytes(cols)
size_t colsum_workspace_bytes(long long cols);
int colsum_rows(const void* X, int is_bf16, long long ld, long long rows, long long cols, float beta, float* out,
                void* workspace, cudaStream_t s);
// out bf16 [cols, rows] = transpose(in [rows, cols]) (in fp32 or bf16, row stride ld)
int transpose_to_bf16(const void* in, int is_bf16, long long ld, bf16* out, long long rows, long long cols, cudaStream_t s);

// ---------------------------------------------------------------- scoring / boxes (score.cu, box.cu)
int sim_matrix(const float* a, const float* b, float* out, int Na, int Nb, int d, float eps, cudaStream_t stream);
// mode 0: argmax over columns -> int64 ; 1: row softmax(x*scale) ; 2: row log_softmax(x*scale)
int row_reduce(const float* x, int rows, int cols, float scale, int mode, void* out, cudaStream_t stream);
int box_cxcywh_to_xyxy(const float* in, float* out, long long nboxes, cudaStream_t stream);
int box_xyxy_to_cxcywh(const float* in, float* out, long long nboxes, cudaStream_t stream);
// pairwise on xyxy boxes: iou, union, giou (each [N,M], any may be null)
int box_pairwise(const float* b1, const float* b2, int N, int M, float* iou, float* uni, float* giou,
                 cudaStream_t stream);
// matcher cost on cxcywh boxes: w_bbox * L1 + w_giou * (-GIoU)  -> [N,M]
int box_match_cost(const float* pred, const float* tgt, int N, int M, float w_bbox, float w_giou, float* cost,
                   cudaStream_t stream);

// matched-pair box loss (SetCriterion.loss_boxes, model/box_utils.py:157-173): losses[0] = L1 / num_boxes,
// losses[1] = sum(1 - giou) / num_boxes over pairs (pred[src_row[k]], tgt[k]), both cxcywh; and its gradient w.r.t. pred.
int box_loss_forward(const float* pred, const long long* src_row, const float* tgt, int K, float num_boxes, float* losses,
                     cudaStream_t stream);
int box_loss_backward(const float* pred, const long long* src_row, const float* tgt, int K, float num_boxes,
                      const float* g_losses, float* grad_pred, long long pred_rows, cudaStream_t stream);

// ---------------------------------------------------------------- assignment (assign.cu)
// P independent rectangular linear-sum-assignment problems (scipy.optimize.linear_sum_assignment semantics and index
// order).  Problem p: rows nr[p] (optionally filtered by row_valid[p, :]), columns nc[p], entry (i,j) at
// cost[offset[p] + i*ld[p] + j].  Outputs padded with -1; count[p] = pairs found, -1 if infeasible / oversized.
int assign_lsa(const float* cost, const long long* offset, const int* ld, const int* nr, const int* nc,
               const unsigned char* row_valid, int row_valid_ld, int P, int max_dim, long long* row_ind,
               long long* col_ind, int* count, int out_ld, cudaStream_t stream);
// cost[r, t] += w * -softmax(logits[r, :ncls])[ids[t]]   (matcher class term, model/box_utils.py:66,83-85)
int match_cost_class(const float* logits, int N, int ncls, const long long* ids, int M, float w, float* cost,
                     cudaStream_t stream);

// ---------------------------------------------------------------- losses (loss.cu)
// Gradient of sim_matrix(a, b) (eps-clamped cosine): G [Na, Nb] (scaled by *gscale when given) -> da [Na,d], db [Nb,d]
// (either may be null).
size_t sim_matrix_backward_workspace_bytes(int Na, int Nb);
int sim_matrix_backward(const float* a, const float* b, const float* G, const float* gscale, float* da, float* db, int Na,
                        int Nb, int d, float eps, void* workspace, cudaStream_t s);
// EgoNCE (model/loss.py:15-70).  saved: fp32 [3N + 3M + 2]; saved[3N + 3M] = loss, [3N + 3M + 1] = kept rows.
int egonce_forward(const float* x, int N, int M, const float* mask_v, const float* mask_n, int R, const float* pad,
                   float temperature, float vn_threshold, unsigned char* mask_bool, unsigned char* keep, float* saved,
                   cudaStream_t s);
int egonce_backward(const float* x, int N, int M, float temperature, const unsigned char* mask_bool,
                    const unsigned char* keep, const float* saved, const float* grad_loss, float* grad_x, cudaStream_t s);
// WordContrastiveLoss (model/loss.py:78-106).  stats fp32 [4]: loss, matched nouns, 1/matched, scratch.
size_t word_loss_workspace_bytes(int V, int d, int B2, int Q, int Wm);
int word_loss_forward(const float* nouns, int V, int d, const float* pred, int B2, int Q, const long long* gt_inds, int Wm,
                      float temperature, float noun_threshold, long long* col_ind, float* sel, long long* sel_row,
                      float* dlogits, float* stats, void* workspace, cudaStream_t s);
int word_loss_backward(const float* nouns, int V, int d, int B2, int Q, int Wm, const float* sel, const long long* sel_row,
                       const float* dlogits, const float* stats, const float* grad_loss, float* d_pred, float* d_nouns,
                       void* workspace, cudaStream_t s);

// ---------------------------------------------------------------- retrieval metrics (retrieval.cu)
// Per query row of sim [N, M] (float64): mode 0 -> average precision (utils/mAP.py), mode 1 -> DCG (utils/nDCG.py) with
// logs[k] = log2(k + 2) and the optional k_counts mask (null: first #(rel > 0) ranks).  out float64 [N].
int retrieval_rows(const double* sim, const double* rel, const double* logs, const int* kcounts, int N, int M, int mode,
                   double* out, cudaStream_t stream);

}  // namespace hh
