/* libhh_b200.so -- C ABI of the B200-native Helping-Hands video-side forward path.
 *
 * The reference (Chuhanxx/helping_hand_for_egocentric_videos) has no FFI: its operator API for this path is the
 * Python nn.Module boundary of model/LaviLa.py, model/tfm_decoder.py, model/metric.py and utils/box_ops.py.  The
 * Python mirror of those modules (helping_hand_for_egocentric_videos_b200/model/*.py) binds exactly the entry points
 * below through ctypes; each one names the reference interface it replaces (paths relative to the reference root).
 *
 * Conventions
 *   - every pointer argument is a DEVICE pointer to a contiguous buffer owned by the caller, unless stated otherwise;
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); nothing synchronises the device;
 *   - return value 0 = OK, negative = error (-1 bad handle, -2 bad argument, -3 CUDA failure);
 *     hh_last_error() returns the message for the calling thread;
 *   - there is no CPU fallback anywhere: without a CUDA device every compute entry point fails with -3.
 */
#ifndef HH_B200_H_
#define HH_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct hh_encoder hh_encoder;
typedef struct hh_decoder hh_decoder;
typedef struct hh_text hh_text;

const char* hh_last_error(void);
int hh_version(void);

/* ------------------------------------------------------------------------------------------------------------------
 * Video encoder: SpaceTimeTransformer.forward_features  (model/LaviLa.py:537-573; blocks :345-390; attention :246-283)
 * ---------------------------------------------------------------------------------------------------------------- */
typedef struct {
  int img_size;    /* 224 */
  int patch_size;  /* 14 (L/14) or 16 (B/16) */
  int num_frames;  /* T; forward requires exactly T frames (LaviLa.py:549-553) */
  int embed_dim;   /* D: multiple of 128, <= 1024 */
  int depth;       /* number of SpaceTimeBlocks */
  int num_heads;   /* D / num_heads must be 64 */
  int mlp_hidden;  /* 4 * D */
} hh_encoder_cfg;

int hh_encoder_create(hh_encoder** out, const hh_encoder_cfg* cfg);
void hh_encoder_destroy(hh_encoder* enc);
/* Copies one parameter (fp32, contiguous, `numel` elements) out of the caller's tensor.  `key` is the reference
 * state_dict key relative to `visual.` (e.g. "blocks.3.timeattn.qkv.weight", "pos_embed", "ln_pre.bias";
 * SURVEY.md section 8b).  Call again after the tensor changes (load_state_dict / .to() / inflate_positional_embeds). */
int hh_encoder_set_weight(hh_encoder* enc, const char* key, const float* data, int64_t numel, void* stream);
/* video fp32 [B,T,3,H,W] -> fmap fp32 [B, 1+T*n, D] (final norm applied to every token, LaviLa.py:573).
 * x_cls of the reference is fmap[:,0,:] (LaviLa.py:570). */
int hh_encoder_forward(hh_encoder* enc, const float* video, int B, float* fmap, void* stream);
/* Test hook: fp32 residual stream after block `block` (0-based) of the last forward is not retained; instead run a
 * truncated forward: blocks [0, nblocks) then the final norm. nblocks < 0 means all. */
int hh_encoder_forward_n(hh_encoder* enc, const float* video, int B, int nblocks, float* fmap, void* stream);
/* Same forward from raw decoder output: frames uint8 [B,T,H,W,3] (decord / cv2 layout, base/base_dataset.py:322-323).
 * The loader tail `frames.float()/255 -> permute -> NormalizeVideo(mean, std)` (data_loader/transforms.py:48-51; constants
 * run/test_EgoMCQ.py:230-233) is applied inside the patch loader in the reference's fp32 operation order, so the result
 * is bit-identical to hh_encoder_forward on the host-normalised clip, at a quarter of the input bytes.
 * mean / std: 3 host floats each (per channel, in [0,1] units). */
int hh_encoder_forward_u8(hh_encoder* enc, const uint8_t* frames, int B, const float* mean, const float* std,
                          float* fmap, void* stream);
/* The same two forwards with the feature map handed over in bf16: fmap bf16 [B, 1+T*n, D] holds every row of the fp32
 * map rounded to nearest-even, and cls fp32 [B, D] (may be NULL) receives the CLS rows fmap32[:, 0] unrounded, so x_cls
 * and the image embedding stay bit-identical to the fp32 entry points.  Half the bytes written and held; the decoder
 * rounds its input to bf16 anyway, so hh_decoder_forward_bf16 on this map gives what hh_decoder_forward gives on the
 * fp32 one, bit for bit. */
int hh_encoder_forward_bf16(hh_encoder* enc, const float* video, int B, void* fmap, float* cls, void* stream);
int hh_encoder_forward_u8_bf16(hh_encoder* enc, const uint8_t* frames, int B, const float* mean, const float* std,
                               void* fmap, float* cls, void* stream);
/* Algorithmic FLOPs of one clip through the encoder (SURVEY.md section 8d formula). */
double hh_encoder_flops_per_clip(const hh_encoder* enc);
/* Number of kernel launches issued by the last hh_encoder_forward call. */
int hh_encoder_last_launches(const hh_encoder* enc);

/* ------------------------------------------------------------------------------------------------------------------
 * Object-aware decoder: ObjDecoder.forward  (model/tfm_decoder.py:183-233) with Cross_Attention.forward (:76-93),
 * TransformerDecoder.forward (:255-295) and TransformerDecoderLayer.forward_pre (:420-461), eval mode (no dropout).
 * ---------------------------------------------------------------------------------------------------------------- */
typedef struct {
  int d_model;           /* C: 512 (multiple of 128, <= 1024; heads of 64) */
  int nhead;             /* C / nhead must be 64 */
  int num_layers;        /* 6 */
  int dim_feedforward;   /* 2048 */
  int num_queries;       /* Q = nq + 1 <= 16 */
  int num_classes1;      /* num_classes + 1 = 22048 */
  int feature_dim;       /* F: 1024 (L/14) or 768 (B/16) */
  int num_frames;        /* T the position embedding was built for */
  int patches_per_frame; /* n */
  int pred_traj;         /* ObjDecoder(pred_traj=...) */
} hh_decoder_cfg;

int hh_decoder_create(hh_decoder** out, const hh_decoder_cfg* cfg);
void hh_decoder_destroy(hh_decoder* dec);
/* `key`: ObjDecoder state_dict key (e.g. "transformer.decoder.layers.0.multihead_attn.in_proj_weight"). */
int hh_decoder_set_weight(hh_decoder* dec, const char* key, const float* data, int64_t numel, void* stream);
/* features fp32 [B,T,n,F] given as a strided view: element (b,t,p,c) at features[b*stride_b + (t*n+p)*stride_row + c]
 * (this is how run/test_EgoMCQ.py:69-70 slices image_feature_map[:,1:]).  Outputs (caller-allocated, fp32):
 *   hs     [L, B, Q, C]
 *   logits [L, B*rep, Q, num_classes1]   rep = 4 if pred_traj and T == num_frames (the reference's literal 4,
 *                                        tfm_decoder.py:216) else 1
 *   boxes  [L, B*Tb, Q, 4]               Tb = T if pred_traj and T == num_frames else 1
 */
int hh_decoder_forward(hh_decoder* dec, const float* features, int64_t stride_b, int64_t stride_row, int B, int T,
                       float* hs, float* logits, float* boxes, void* stream);
/* The same forward on bf16 features [B,T,n,F] (same strided layout, strides in elements; rows 8-byte aligned).  When
 * T*n is a multiple of 128, the rows are 16-byte aligned and stride_b is a multiple of stride_row (image_feature_map[:, 1:]
 * of a bf16 map qualifies), the first GEMM reads the caller's rows in place: no copy, no feature workspace, one launch
 * fewer.  Otherwise the rows are first gathered into the engine's workspace. */
int hh_decoder_forward_bf16(hh_decoder* dec, const void* features, int64_t stride_b, int64_t stride_row, int B, int T,
                            float* hs, float* logits, float* boxes, void* stream);
/* Training: the same forward that also keeps every layer's activations inside the engine, then hh_decoder_backward
 * differentiates it.  Dropout of the reference's training mode (nn.Dropout x4 per layer, tfm_decoder.py:372-386, and
 * nn.MultiheadAttention(dropout=p) on the self- and cross-attention probabilities, :365-366) is applied by the training
 * forward when hh_decoder_set_dropout was called with p > 0: masks come from a counter-based generator (Philox4x32-10,
 * keyed by `seed`, stream position `offset`; csrc/hh_rng.cuh), so hh_decoder_backward regenerates them instead of storing
 * them.  The setting persists until changed; callers advance `offset` every step.  p = 0 (the default) = eval arithmetic.
 * hh_decoder_backward: hs / boxes are the outputs of that forward; d_hs [L,B,Q,C] and d_boxes [L,B*Tb,Q,4] are the
 * upstream gradients (either may be NULL = zero).  Class logits carry no gradient (the reference criterion has no class
 * loss, run/train.py:471, exclude_class=True): class_embed.* get zeros.  Gradients of every parameter key are then read
 * with hh_decoder_get_grad (fp32, `numel` elements, device memory). */
int hh_decoder_forward_train(hh_decoder* dec, const float* features, int64_t stride_b, int64_t stride_row, int B, int T,
                             float* hs, float* logits, float* boxes, void* stream);
/* Training forward on bf16 features.  It always copies the rows into the engine (backward reads that copy), so the
 * caller may overwrite `features` between this call and hh_decoder_backward. */
int hh_decoder_forward_train_bf16(hh_decoder* dec, const void* features, int64_t stride_b, int64_t stride_row, int B,
                                  int T, float* hs, float* logits, float* boxes, void* stream);
int hh_decoder_set_dropout(hh_decoder* dec, float p, uint64_t seed, uint32_t offset);
int hh_decoder_backward(hh_decoder* dec, const float* hs, const float* boxes, const float* d_hs, const float* d_boxes,
                        void* stream);
/* The engine keeps ONE set of saved activations.  hh_decoder_generation returns the ordinal of the last forward (every
 * forward, training or not, bumps it); hh_decoder_backward_checked refuses (-2) when `generation` is not that ordinal,
 * i.e. when another forward ran between the training forward being differentiated and this call. */
uint64_t hh_decoder_generation(const hh_decoder* dec);
int hh_decoder_backward_checked(hh_decoder* dec, uint64_t generation, const float* hs, const float* boxes,
                                const float* d_hs, const float* d_boxes, void* stream);
int hh_decoder_get_grad(hh_decoder* dec, const char* key, float* out, int64_t numel, void* stream);
/* Batched forms (one call per training step instead of one per parameter: the step's 135 keys made the Python side of
 * the backward host-bound).  get_grads packs the gradients of keys[0..n) back to back into `out` (`total` = sum of
 * numels); set_weights is hh_decoder_set_weight over n (key, data, numel) triples. */
int hh_decoder_get_grads(hh_decoder* dec, const char* const* keys, const int64_t* numels, int n, float* out, int64_t total,
                         void* stream);
int hh_decoder_set_weights(hh_decoder* dec, const char* const* keys, const float* const* data, const int64_t* numels, int n,
                           void* stream);
double hh_decoder_flops_per_clip(const hh_decoder* dec, int T);
int hh_decoder_last_launches(const hh_decoder* dec);

/* ------------------------------------------------------------------------------------------------------------------
 * CLIP text tower: CLIP.encode_text  (model/LaviLa.py:660-670) over ResidualAttentionBlock (model/openai_model.py:
 * 182-216): token + positional embedding, `layers` pre-norm blocks with causal attention and QuickGELU MLP, ln_final,
 * end-of-text row (argmax of the token ids) @ text_projection.
 * ---------------------------------------------------------------------------------------------------------------- */
typedef struct {
  int vocab_size;      /* 49408 */
  int context_length;  /* 77 */
  int width;           /* 512 (BASE) / 768 (LARGE); heads of 64 */
  int heads;
  int layers;          /* 12 */
  int embed_dim;       /* projection width, 256 */
} hh_text_cfg;

int hh_text_create(hh_text** out, const hh_text_cfg* cfg);
void hh_text_destroy(hh_text* txt);
/* `key`: CLIP state_dict key of the text side ("token_embedding.weight", "positional_embedding",
 * "transformer.resblocks.3.attn.in_proj_weight", "ln_final.bias", "text_projection", ...). */
int hh_text_set_weight(hh_text* txt, const char* key, const float* data, int64_t numel, void* stream);
/* tokens int64 [G, context_length] (device) -> embed fp32 [G, embed_dim] (un-normalised x_cls, LaviLa.py:669) and
 * fmap fp32 [G, context_length, width] (ln_final of every token, :667).  Either output may be NULL.  Synchronises the
 * stream once to report token ids outside [0, vocab_size) (the reference's nn.Embedding device-asserts on those). */
int hh_text_forward(hh_text* txt, const int64_t* tokens, int G, float* embed, float* fmap, void* stream);
double hh_text_flops_per_sequence(const hh_text* txt);
int hh_text_last_launches(const hh_text* txt);

/* Per-kernel-class device timing (CUDA events recorded on the launching stream around every launch while enabled).
 * hh_*_profile waits for the recorded events, writes the summed milliseconds and launch counts of every class
 * (arrays of hh_profile_num_classes() entries) since the previous call, and resets the recorder. */
int hh_profile_num_classes(void);
const char* hh_profile_class_name(int cls);
int hh_encoder_set_profile(hh_encoder* enc, int on);
int hh_encoder_profile(hh_encoder* enc, double* ms, int* counts);
int hh_decoder_set_profile(hh_decoder* dec, int on);
int hh_decoder_profile(hh_decoder* dec, double* ms, int* counts);

/* ------------------------------------------------------------------------------------------------------------------
 * Stateless operators
 * ---------------------------------------------------------------------------------------------------------------- */
/* sim_matrix(a, b) (model/metric.py:363-375): out[Na,Nb] = (a/max(|a|,eps)) . (b/max(|b|,eps))^T, fp32. */
int hh_sim_matrix(const float* a, const float* b, float* out, int Na, int Nb, int d, float eps, void* stream);
/* Row-wise reductions of scale*x [rows, cols]: mode 0 = argmax -> int64 out[rows] (EgoMCQ choice, metric.py:218);
 * 1 = softmax, 2 = log_softmax -> fp32 out[rows, cols] (EgoNCE at scale 1/0.07, model/loss.py:61-69). */
int hh_row_reduce(const float* x, int rows, int cols, float scale, int mode, void* out, void* stream);
/* F.normalize(x, dim=-1) with eps (CLIP.forward, model/LaviLa.py:676-677). */
int hh_l2_normalize(const float* x, float* out, int rows, int cols, float eps, void* stream);
/* nn.Linear on fp32 rows: out = act(relu_in?(in (+ in_add[row % add_mod])) W^T + bias) (+ residual).
 * W [N,K] row-major, K % 32 == 0.  act: 0 none, 1 ReLU, 2 sigmoid.  (ObjDecoder.obj_proj / txt_proj,
 * tfm_decoder.py:168-180; CLIP image_projection, LaviLa.py:657.) */
int hh_linear_f32(const float* in, int ldi, const float* in_add, int add_mod, const float* W, const float* bias,
                  const float* residual, int ldres, float* out, int ldo, int R, int N, int K, int act, int in_relu,
                  void* stream);
/* utils/box_ops.py:9-13, :16-20 */
int hh_box_cxcywh_to_xyxy(const float* in, float* out, int64_t nboxes, void* stream);
int hh_box_xyxy_to_cxcywh(const float* in, float* out, int64_t nboxes, void* stream);
/* box_iou + generalized_box_iou (utils/box_ops.py:24-61) on xyxy boxes; each output [N,M] may be NULL. */
int hh_box_pairwise(const float* boxes1, const float* boxes2, int N, int M, float* iou, float* uni, float* giou,
                    void* stream);
/* HungarianMatcher cost with exclude_class (model/box_utils.py:75-88): w_bbox*L1 + w_giou*(-GIoU), cxcywh in. */
int hh_box_match_cost(const float* pred, const float* tgt, int N, int M, float w_bbox, float w_giou, float* cost,
                      void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Kernel-level entry points (used by the parity tests and the roofline bench; same kernels the engines launch)
 * ---------------------------------------------------------------------------------------------------------------- */
/* C[M,N] = epilogue(A[M,K] W[N,K]^T): A, W bf16 (uint16 storage), K contiguous.  epilogue: 0 bias->bf16,
 * 1 bias+QuickGELU->bf16, 2 bias+fp32 residual->fp32, 3 bias->fp32.  (nn.Linear calls of LaviLa.py:249,281,186,189) */
int hh_gemm_bf16(const void* A, int lda, const void* W, int ldw, void* out, int ldc, const float* bias,
                 const float* residual, int ldr, int M, int N, int K, int epilogue, void* stream);
/* LayerNorm folded into the contractions around it (norm1 / norm2 / norm3 + residual adds of SpaceTimeBlock.forward,
 * model/LaviLa.py:353-388; north_star "fused LayerNorm+bias+GELU epilogues").  With z the UN-normalised row,
 *   Linear(LayerNorm(z)) = rstd * (z W'^T - mean * colsum) + bias',   W' = W diag(gamma),  bias' = bias + W beta.
 * hh_fold_layernorm_weight: W fp32 [N,K], gamma / beta fp32 [K], bias fp32 [N] or NULL -> Wf bf16 [N,K], colsum fp32 [N]
 *   (column sums of the bf16-rounded W'), bias_f fp32 [N]; the first `scaled_rows` rows and their bias also carry `scale`.
 * hh_gemm_bf16_res_stats (producer): z16 bf16 [M,N] = A W^T + bias + residual (fp32 [M,N], row pitch ldr); per-row
 *   (sum z, sum z^2) partials, one per column tile: stats fp32 [hh_gemm_stats_parts(M,N)][M][2]; writeback != 0 also stores
 *   the fp32 sum over `residual` in place (the residual stream itself).
 * hh_gemm_bf16_ln (consumer): out bf16 [M,N] = act(rstd * (A Wf^T - mean * colsum) + bias_f), mean / rstd per row from
 *   `parts` statistics partials taken over norm_dim (= K) columns; act = QuickGELU when qgelu != 0. */
int hh_gemm_stats_parts(int M, int N);
int hh_fold_layernorm_weight(const float* W, const float* gamma, const float* beta, const float* bias, int N, int K,
                             int scaled_rows, float scale, void* Wf, float* colsum, float* bias_f, void* stream);
int hh_gemm_bf16_res_stats(const void* A, int lda, const void* W, int ldw, void* z16, int ldz, const float* bias,
                           float* residual, int ldr, int writeback, float* stats, int M, int N, int K, void* stream);
int hh_gemm_bf16_ln(const void* A, int lda, const void* Wf, int ldw, void* out, int ldc, const float* bias_f,
                    const float* colsum, const float* stats, int parts, int norm_dim, float eps, int M, int N, int K,
                    int qgelu, void* stream);
/* LayerNorm rows (fp32 in): optional fp32 and bf16 outputs. */
int hh_layernorm(const float* x, int ldx, const float* w, const float* b, float eps, float* out_f32, void* out_bf16,
                 int M, int D, void* stream);
int hh_f32_to_bf16(const float* src, void* dst, int64_t n, void* stream);
/* Divided attention on packed qkv bf16 [B*(1+T*n), 3*H*64] with q pre-scaled -> out bf16 [B*(1+T*n), H*64].
 * kind 0 = space, 1 = time (patch rows), 2 = CLS row. */
int hh_attention(const void* qkv, void* out, int B, int T, int n, int H, int kind, void* stream);
/* Query->patch cross attention (tfm_decoder.py:438-441 core): q fp32 [B*Q, heads*64] pre-scaled, K/V bf16 [B*S, ldkv]. */
int hh_cross_attention(const float* q, const void* K, const void* V, int ldkv, float* out, int B, int Q, int heads,
                       int S, void* stream);
/* Causal self-attention core of the text tower: qkv bf16 [G*L, 3*H*64] (q pre-scaled) -> out bf16 [G*L, H*64]. */
int hh_attention_causal(const void* qkv, void* out, int G, int L, int H, void* stream);
/* Same operator on the fp32 SIMT kernel (second implementation kept for differential testing). */
int hh_cross_attention_simt(const float* q, const void* K, const void* V, int ldkv, float* out, int B, int Q, int heads,
                            int S, void* stream);

/* SetCriterion.loss_boxes (model/box_utils.py:157-173) on matched pairs: pair k = (pred[src_row[k]], tgt[k]), boxes in
 * cxcywh.  losses[0] = sum |p - t| / num_boxes, losses[1] = sum (1 - GIoU(p, t)) / num_boxes (GIoU as in
 * utils/box_ops.py:24-61).  backward: grad_pred [pred_rows, 4] (zero-filled, then one row per pair) for upstream
 * gradients g_losses[0..1]; follows the eager reference's autograd conventions (ties of max/min split 0.5/0.5). */
int hh_box_loss_forward(const float* pred, const int64_t* src_row, const float* tgt, int K, float num_boxes,
                        float* losses, void* stream);
int hh_box_loss_backward(const float* pred, const int64_t* src_row, const float* tgt, int K, float num_boxes,
                         const float* g_losses, float* grad_pred, int64_t pred_rows, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Assignment: the per-image / per-clip scipy.optimize.linear_sum_assignment calls of HungarianMatcher.forward
 * (model/box_utils.py:89-92) and WordContrastiveLoss.forward (model/loss.py:88-93), batched on the device.
 * Problem p has nr[p] rows (only those with row_valid[p*row_valid_ld + r] != 0 when row_valid is given; the kept rows
 * are renumbered 0..) and nc[p] columns (each <= max_dim <= 32); entry (i, j) = cost[offset[p] + i*ld[p] + j].
 * row_ind / col_ind [P, out_ld] int64 receive the pairs in scipy's order (ascending row), -1 padded;
 * count[p] = number of pairs (min(rows, cols)), or -1 when the problem is infeasible (inf / nan) or oversized.
 * All arrays are device memory.
 * ---------------------------------------------------------------------------------------------------------------- */
int hh_assign(const float* cost, const int64_t* offset, const int32_t* ld, const int32_t* nr, const int32_t* nc,
              const uint8_t* row_valid, int row_valid_ld, int P, int max_dim, int64_t* row_ind, int64_t* col_ind,
              int32_t* count, int out_ld, void* stream);
/* cost[r, t] += w * -softmax(logits[r, :])[ids[t]]  for r < N, t < M: the classification term of the matcher cost
 * (model/box_utils.py:66,83-85; only evaluated when exclude_class=False). */
int hh_match_cost_class(const float* logits, int N, int ncls, const int64_t* ids, int M, float w, float* cost,
                        void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Training-side scoring losses (forward + backward).  All buffers are device memory owned by the caller.
 * ---------------------------------------------------------------------------------------------------------------- */
/* Gradient of hh_sim_matrix: G fp32 [Na, Nb] (multiplied by *gscale when gscale != NULL) -> da [Na, d], db [Nb, d]
 * (either may be NULL).  workspace: hh_sim_matrix_backward_workspace_bytes(Na, Nb) bytes. */
size_t hh_sim_matrix_backward_workspace_bytes(int Na, int Nb);
int hh_sim_matrix_backward(const float* a, const float* b, const float* G, const float* gscale, float* da, float* db,
                           int Na, int Nb, int d, float eps, void* workspace, void* stream);
/* EgoNCE.forward (model/loss.py:15-70).  x fp32 [N, M] similarities, N = R * M (R captions per video, video-major);
 * mask_v / mask_n fp32 [M, M] (either may be NULL); pad fp32 [N, M] or NULL (single-positive branch, R = 1).
 * Outputs: mask_bool uint8 [N, M] (before the padded rows are dropped), keep uint8 [N] (row survives
 * `masked_x.sum(-1) != -inf`), saved fp32 [3N + 3M + 2] (row/column log-sum-exp, positive counts, per-row/column terms;
 * saved[3N + 3M] = loss, saved[3N + 3M + 1] = number of kept rows). */
int hh_egonce_forward(const float* x, int N, int M, const float* mask_v, const float* mask_n, int R, const float* pad,
                      float temperature, float vn_threshold, uint8_t* mask_bool, uint8_t* keep, float* saved,
                      void* stream);
/* grad_x [N, M] = d loss / d x * (*grad_loss); rows dropped by `keep` get 0. */
int hh_egonce_backward(const float* x, int N, int M, float temperature, const uint8_t* mask_bool, const uint8_t* keep,
                       const float* saved, const float* grad_loss, float* grad_x, void* stream);
/* WordContrastiveLoss.forward (model/loss.py:78-106).  noun_embeds fp32 [V, d]; pred fp32 [B2, Q, d] (object-query
 * embeddings); gt_inds int64 [B2, Wm] (0 = no noun).  Outputs: col_ind int64 [B2, Wm] = query matched to each noun slot
 * (-1 for empty slots; the k-th non-empty slot of a clip carries scipy's col_ind[k]), sel fp32 [B2*Wm, d] (matched query
 * rows), sel_row int64 [B2*Wm] (row of pred, -1 if empty), dlogits fp32 [B2*Wm, V] (d loss_slot / d similarity),
 * stats fp32 [4] (stats[0] = loss, stats[1] = matched nouns).  A noun id outside [0, V) makes the loss NaN. */
size_t hh_word_loss_workspace_bytes(int V, int d, int B2, int Q, int Wm);
int hh_word_loss_forward(const float* noun_embeds, int V, int d, const float* pred, int B2, int Q,
                         const int64_t* gt_inds, int Wm, float temperature, float noun_threshold, int64_t* col_ind,
                         float* sel, int64_t* sel_row, float* dlogits, float* stats, void* workspace, void* stream);
/* d_pred fp32 [B2*Q, d] and d_nouns fp32 [V, d] (either may be NULL), scaled by *grad_loss. */
int hh_word_loss_backward(const float* noun_embeds, int V, int d, int B2, int Q, int Wm, const float* sel,
                          const int64_t* sel_row, const float* dlogits, float* stats, const float* grad_loss,
                          float* d_pred, float* d_nouns, void* workspace, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Retrieval metrics (run/test_epic.py:262-283): per-query average precision (utils/mAP.py:4-44, mode 0) or discounted
 * cumulative gain (utils/nDCG.py:3-44, mode 1) of sim [N, M] against rel [N, M], all float64 device arrays, M <= 16384.
 * logs [M] = log2(k + 2) (mode 1; pass numpy's table so the divisors are the reference's own); kcounts int32 [N, M] or
 * NULL (= calculate_k_counts(rel), utils/nDCG.py:46-75).  out float64 [N].  Summation follows numpy's order (sequential
 * cumsum, pairwise np.sum), so results equal the reference's bit for bit when no two similarities of a row tie. */
int hh_retrieval_rows(const double* sim, const double* rel, const double* logs, const int32_t* kcounts, int N, int M,
                      int mode, double* out, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Decoder backward primitives (kernel-level entry points; the decoder engine sequences them in hh_decoder_backward).
 * ---------------------------------------------------------------------------------------------------------------- */
/* nn.Linear backward for y = act(x W^T + b), x = relu?(X + x_add[r % add_mod]).  g = act'(dY, Y) with Y the saved output
 * (act 0 none / 1 relu / 2 sigmoid).  dX [R,K] = beta*dX + g W (skipped when NULL); dW [N,K] = beta*dW + scale * g^T x and
 * db [N] = beta*db + scale * colsum(g) (skipped when dW is NULL; db may be NULL). */
int hh_linear_f32_backward(const float* dY, int ldy, const float* Y, int ldyo, int act, const float* W, const float* X,
                           int ldx, const float* x_add, int add_mod, int in_relu, float* dX, int lddx, float* dW,
                           float* db, int R, int N, int K, float beta, float scale, void* stream);
/* LayerNorm backward over M rows of width D (multiple of 128, <= 1024): dx (overwritten), dgamma / dbeta (overwritten;
 * both or neither). */
int hh_layernorm_backward(const float* x, int ldx, const float* w, float eps, const float* dy, int lddy, float* dx,
                          float* dgamma, float* dbeta, int M, int D, void* stream);
/* Backward of the query self-attention core (hh_decoder's self_attn): q,k,v fp32 rows with stride ld (q pre-scaled),
 * dO fp32 [B*Q, heads*64] -> dq, dk, dv rows with stride ldg. */
int hh_self_attention_backward(const float* q, const float* k, const float* v, int ld, const float* dO, float* dq,
                               float* dk, float* dv, int ldg, int B, int Q, int heads, void* stream);
/* Backward of hh_cross_attention: O = forward output, dO its gradient (fp32 [B*Q, heads*64]) -> dq fp32 [B*Q, heads*64],
 * dK / dV bf16 rows [B*S] with stride lddkv. */
int hh_cross_attention_backward(const float* q, const void* K, const void* V, int ldkv, const float* O, const float* dO,
                                float* dq, void* dK, void* dV, int lddkv, int B, int Q, int heads, int S, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Data-parallel exchange: the one collective of the path (all-gather of embeddings for the cross-rank similarity
 * matrix, run/train.py:36-37,126-128; _valid_all_gather, utils/train_utils.py:51-59).  NCCL is resolved at run time
 * (dlopen of the libnccl.so.2 already loaded by the host framework); one communicator per process / GPU.
 * ---------------------------------------------------------------------------------------------------------------- */
#define HH_NCCL_ID_BYTES 128
int hh_comm_unique_id(void* id_host);                                     /* rank 0: fills 128 host bytes */
int hh_comm_create(void** comm, int nranks, int rank, const void* id_host); /* collective over all ranks */
int hh_comm_destroy(void* comm);
/* recv[r*bytes_per_rank ...] = rank r's send buffer, for every rank (ncclAllGather on `stream`). */
int hh_allgather(void* comm, const void* send, void* recv, size_t bytes_per_rank, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HH_B200_H_ */
