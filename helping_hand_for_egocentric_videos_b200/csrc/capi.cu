// extern "C" surface declared in include/hh_b200.h.  No C++ types or exceptions cross this boundary.
#include <dlfcn.h>

#include <cstring>

#include <new>

#include "engine.h"

using namespace hh;

struct hh_encoder {
  Encoder impl;
  explicit hh_encoder(const hh_encoder_cfg& c) : impl(c) {}
};
struct hh_decoder {
  Decoder impl;
  explicit hh_decoder(const hh_decoder_cfg& c) : impl(c) {}
};

struct hh_text {
  TextEncoder impl;
  explicit hh_text(const hh_text_cfg& c) : impl(c) {}
};

#define HH_GUARD_BEGIN try {
#define HH_GUARD_END                                              \
  }                                                               \
  catch (const std::bad_alloc&) { return fail(-3, "host out of memory"); } \
  catch (const std::exception& e) { return fail(-3, std::string("internal error: ") + e.what()); } \
  catch (...) { return fail(-3, "internal error"); }

static inline cudaStream_t S(void* s) { return static_cast<cudaStream_t>(s); }

extern "C" {

const char* hh_last_error(void) { return last_error_cstr(); }
int hh_version(void) { return 100; }

// ------------------------------------------------------------------------------------------ encoder
int hh_encoder_create(hh_encoder** out, const hh_encoder_cfg* cfg) {
  HH_GUARD_BEGIN
  if (!out || !cfg) return fail(-2, "hh_encoder_create: null argument");
  int rc = Encoder::validate(*cfg);
  if (rc) return rc;
  *out = new hh_encoder(*cfg);
  return 0;
  HH_GUARD_END
}
void hh_encoder_destroy(hh_encoder* enc) { delete enc; }
int hh_encoder_set_weight(hh_encoder* enc, const char* key, const float* data, int64_t numel, void* stream) {
  HH_GUARD_BEGIN
  if (!enc) return fail(-1, "hh_encoder_set_weight: null handle");
  if (!key || !data) return fail(-2, "hh_encoder_set_weight: null argument");
  return enc->impl.weights.set(key, data, numel, S(stream));
  HH_GUARD_END
}
int hh_encoder_forward_n(hh_encoder* enc, const float* video, int B, int nblocks, float* fmap, void* stream) {
  HH_GUARD_BEGIN
  if (!enc) return fail(-1, "hh_encoder_forward: null handle");
  Encoder::Fmap o;
  o.f32 = fmap;
  return enc->impl.forward(video, B, nblocks, o, S(stream));
  HH_GUARD_END
}
int hh_encoder_forward(hh_encoder* enc, const float* video, int B, float* fmap, void* stream) {
  return hh_encoder_forward_n(enc, video, B, -1, fmap, stream);
}
int hh_encoder_forward_u8(hh_encoder* enc, const uint8_t* frames, int B, const float* mean, const float* stdv, float* fmap,
                          void* stream) {
  HH_GUARD_BEGIN
  if (!enc) return fail(-1, "hh_encoder_forward_u8: null handle");
  Encoder::Fmap o;
  o.f32 = fmap;
  return enc->impl.forward_u8(frames, mean, stdv, B, o, S(stream));
  HH_GUARD_END
}
int hh_encoder_forward_bf16(hh_encoder* enc, const float* video, int B, void* fmap, float* cls, void* stream) {
  HH_GUARD_BEGIN
  if (!enc) return fail(-1, "hh_encoder_forward_bf16: null handle");
  Encoder::Fmap o;
  o.b16 = static_cast<bf16*>(fmap);
  o.cls = cls;
  return enc->impl.forward(video, B, -1, o, S(stream));
  HH_GUARD_END
}
int hh_encoder_forward_u8_bf16(hh_encoder* enc, const uint8_t* frames, int B, const float* mean, const float* stdv,
                               void* fmap, float* cls, void* stream) {
  HH_GUARD_BEGIN
  if (!enc) return fail(-1, "hh_encoder_forward_u8_bf16: null handle");
  Encoder::Fmap o;
  o.b16 = static_cast<bf16*>(fmap);
  o.cls = cls;
  return enc->impl.forward_u8(frames, mean, stdv, B, o, S(stream));
  HH_GUARD_END
}
double hh_encoder_flops_per_clip(const hh_encoder* enc) { return enc ? enc->impl.flops_per_clip() : 0.0; }
int hh_encoder_last_launches(const hh_encoder* enc) { return enc ? enc->impl.launches : 0; }

// ------------------------------------------------------------------------------------------ decoder
int hh_decoder_create(hh_decoder** out, const hh_decoder_cfg* cfg) {
  HH_GUARD_BEGIN
  if (!out || !cfg) return fail(-2, "hh_decoder_create: null argument");
  int rc = Decoder::validate(*cfg);
  if (rc) return rc;
  *out = new hh_decoder(*cfg);
  return 0;
  HH_GUARD_END
}
void hh_decoder_destroy(hh_decoder* dec) { delete dec; }
int hh_decoder_set_weight(hh_decoder* dec, const char* key, const float* data, int64_t numel, void* stream) {
  HH_GUARD_BEGIN
  if (!dec) return fail(-1, "hh_decoder_set_weight: null handle");
  if (!key || !data) return fail(-2, "hh_decoder_set_weight: null argument");
  return dec->impl.weights.set(key, data, numel, S(stream));
  HH_GUARD_END
}
int hh_decoder_forward(hh_decoder* dec, const float* features, int64_t stride_b, int64_t stride_row, int B, int T,
                       float* hs, float* logits, float* boxes, void* stream) {
  HH_GUARD_BEGIN
  if (!dec) return fail(-1, "hh_decoder_forward: null handle");
  return dec->impl.forward(features, false, stride_b, stride_row, B, T, hs, logits, boxes, S(stream));
  HH_GUARD_END
}
int hh_decoder_forward_bf16(hh_decoder* dec, const void* features, int64_t stride_b, int64_t stride_row, int B, int T,
                            float* hs, float* logits, float* boxes, void* stream) {
  HH_GUARD_BEGIN
  if (!dec) return fail(-1, "hh_decoder_forward_bf16: null handle");
  return dec->impl.forward(features, true, stride_b, stride_row, B, T, hs, logits, boxes, S(stream));
  HH_GUARD_END
}
int hh_decoder_forward_train(hh_decoder* dec, const float* features, int64_t stride_b, int64_t stride_row, int B, int T,
                             float* hs, float* logits, float* boxes, void* stream) {
  HH_GUARD_BEGIN
  if (!dec) return fail(-1, "hh_decoder_forward_train: null handle");
  return dec->impl.forward(features, false, stride_b, stride_row, B, T, hs, logits, boxes, S(stream), true);
  HH_GUARD_END
}
int hh_decoder_forward_train_bf16(hh_decoder* dec, const void* features, int64_t stride_b, int64_t stride_row, int B,
                                  int T, float* hs, float* logits, float* boxes, void* stream) {
  HH_GUARD_BEGIN
  if (!dec) return fail(-1, "hh_decoder_forward_train_bf16: null handle");
  return dec->impl.forward(features, true, stride_b, stride_row, B, T, hs, logits, boxes, S(stream), true);
  HH_GUARD_END
}
int hh_decoder_set_dropout(hh_decoder* dec, float p, uint64_t seed, uint32_t offset) {
  HH_GUARD_BEGIN
  if (!dec) return fail(-1, "hh_decoder_set_dropout: null handle");
  if (!(p >= 0.f && p < 1.f)) return fail(-2, "hh_decoder_set_dropout: p must be in [0, 1)");
  DropCfg d = drop_off();
  if (p > 0.f) {
    d.thr = static_cast<uint32_t>(p * 65536.0f + 0.5f);   // keep <=> 16-bit lane >= thr
    if (d.thr == 0) d.thr = 1;
    d.scale = 1.0f / (1.0f - p);
    d.seed_lo = static_cast<uint32_t>(seed);
    d.seed_hi = static_cast<uint32_t>(seed >> 32);
    d.offset = offset;
  }
  dec->impl.next_drop = d;
  return 0;
  HH_GUARD_END
}
int hh_decoder_backward(hh_decoder* dec, const float* hs, const float* boxes, const float* d_hs, const float* d_boxes,
                        void* stream) {
  HH_GUARD_BEGIN
  if (!dec) return fail(-1, "hh_decoder_backward: null handle");
  return dec->impl.backward(hs, boxes, d_hs, d_boxes, S(stream));
  HH_GUARD_END
}
uint64_t hh_decoder_generation(const hh_decoder* dec) { return dec ? dec->impl.generation : 0; }
int hh_decoder_backward_checked(hh_decoder* dec, uint64_t generation, const float* hs, const float* boxes, const float* d_hs,
                                const float* d_boxes, void* stream) {
  HH_GUARD_BEGIN
  if (!dec) return fail(-1, "hh_decoder_backward_checked: null handle");
  if (dec->impl.generation != generation)
    return fail(-2, "hh_decoder_backward: the engine's saved activations belong to forward #" +
                        std::to_string(dec->impl.generation) + ", not to forward #" + std::to_string(generation) +
                        " (another forward ran in between; call backward before the next forward)");
  return dec->impl.backward(hs, boxes, d_hs, d_boxes, S(stream));
  HH_GUARD_END
}
int hh_decoder_get_grad(hh_decoder* dec, const char* key, float* out, int64_t numel, void* stream) {
  HH_GUARD_BEGIN
  if (!dec || !key || !out) return fail(-2, "hh_decoder_get_grad: null argument");
  auto it = dec->impl.weights.expected.find(key);
  if (it == dec->impl.weights.expected.end()) return fail(-2, std::string("unknown parameter key '") + key + "'");
  if (it->second != numel) return fail(-2, std::string("parameter '") + key + "': wrong element count");
  const float* g = dec->impl.grad(key);
  if (!g) return fail(-2, "hh_decoder_get_grad: no gradient yet (run hh_decoder_backward)");
  HH_CHECK_CUDA(cudaMemcpyAsync(out, g, static_cast<size_t>(numel) * 4, cudaMemcpyDeviceToDevice, S(stream)));
  return 0;
  HH_GUARD_END
}
int hh_decoder_get_grads(hh_decoder* dec, const char* const* keys, const int64_t* numels, int n, float* out, int64_t total,
                         void* stream) {
  HH_GUARD_BEGIN
  if (!dec || !keys || !numels || !out || n < 0) return fail(-2, "hh_decoder_get_grads: null argument");
  int64_t off = 0;
  for (int i = 0; i < n; ++i) {
    auto it = dec->impl.weights.expected.find(keys[i]);
    if (it == dec->impl.weights.expected.end()) return fail(-2, std::string("unknown parameter key '") + keys[i] + "'");
    if (it->second != numels[i]) return fail(-2, std::string("parameter '") + keys[i] + "': wrong element count");
    if (off + numels[i] > total) return fail(-2, "hh_decoder_get_grads: output too small");
    const float* g = dec->impl.grad(keys[i]);
    if (!g) return fail(-2, "hh_decoder_get_grads: no gradient yet (run hh_decoder_backward)");
    HH_CHECK_CUDA(cudaMemcpyAsync(out + off, g, static_cast<size_t>(numels[i]) * 4, cudaMemcpyDeviceToDevice, S(stream)));
    off += numels[i];
  }
  if (off != total) return fail(-2, "hh_decoder_get_grads: total does not match the keys");
  return 0;
  HH_GUARD_END
}
int hh_decoder_set_weights(hh_decoder* dec, const char* const* keys, const float* const* data, const int64_t* numels, int n,
                           void* stream) {
  HH_GUARD_BEGIN
  if (!dec || !keys || !data || !numels || n < 0) return fail(-2, "hh_decoder_set_weights: null argument");
  for (int i = 0; i < n; ++i) {
    if (!keys[i] || !data[i]) return fail(-2, "hh_decoder_set_weights: null entry");
    int rc = dec->impl.weights.set(keys[i], data[i], numels[i], S(stream));
    if (rc) return rc;
  }
  return 0;
  HH_GUARD_END
}
double hh_decoder_flops_per_clip(const hh_decoder* dec, int T) { return dec ? dec->impl.flops_per_clip(T) : 0.0; }
int hh_decoder_last_launches(const hh_decoder* dec) { return dec ? dec->impl.launches : 0; }

// ------------------------------------------------------------------------------------------ text tower
int hh_text_create(hh_text** out, const hh_text_cfg* cfg) {
  HH_GUARD_BEGIN
  if (!out || !cfg) return fail(-2, "hh_text_create: null argument");
  int rc = TextEncoder::validate(*cfg);
  if (rc) return rc;
  *out = new hh_text(*cfg);
  return 0;
  HH_GUARD_END
}
void hh_text_destroy(hh_text* txt) { delete txt; }
int hh_text_set_weight(hh_text* txt, const char* key, const float* data, int64_t numel, void* stream) {
  HH_GUARD_BEGIN
  if (!txt) return fail(-1, "hh_text_set_weight: null handle");
  if (!key || !data) return fail(-2, "hh_text_set_weight: null argument");
  return txt->impl.weights.set(key, data, numel, S(stream));
  HH_GUARD_END
}
int hh_text_forward(hh_text* txt, const int64_t* tokens, int G, float* embed, float* fmap, void* stream) {
  HH_GUARD_BEGIN
  if (!txt) return fail(-1, "hh_text_forward: null handle");
  return txt->impl.forward(tokens, G, embed, fmap, S(stream));
  HH_GUARD_END
}
double hh_text_flops_per_sequence(const hh_text* txt) { return txt ? txt->impl.flops_per_sequence() : 0.0; }
int hh_text_last_launches(const hh_text* txt) { return txt ? txt->impl.launches : 0; }

// ------------------------------------------------------------------------------------------ event profiler
static const char* kClassNames[K_NUM] = {"gemm_qkv", "gemm_proj", "gemm_fc1", "gemm_fc2", "gemm_patch", "layernorm",
                                         "attn_time", "attn_space", "attn_cls", "embed", "dec_memory_gemm",
                                         "dec_cross_attn", "dec_query_side", "dec_heads"};
int hh_profile_num_classes(void) { return K_NUM; }
const char* hh_profile_class_name(int i) { return (i >= 0 && i < K_NUM) ? kClassNames[i] : ""; }
int hh_encoder_set_profile(hh_encoder* enc, int on) {
  if (!enc) return fail(-1, "hh_encoder_set_profile: null handle");
  enc->impl.prof.enabled = on != 0;
  return 0;
}
int hh_encoder_profile(hh_encoder* enc, double* ms, int* counts) {
  HH_GUARD_BEGIN
  if (!enc || !ms || !counts) return fail(-2, "hh_encoder_profile: null argument");
  return enc->impl.prof.collect(ms, counts);
  HH_GUARD_END
}
int hh_decoder_set_profile(hh_decoder* dec, int on) {
  if (!dec) return fail(-1, "hh_decoder_set_profile: null handle");
  dec->impl.prof.enabled = on != 0;
  return 0;
}
int hh_decoder_profile(hh_decoder* dec, double* ms, int* counts) {
  HH_GUARD_BEGIN
  if (!dec || !ms || !counts) return fail(-2, "hh_decoder_profile: null argument");
  return dec->impl.prof.collect(ms, counts);
  HH_GUARD_END
}

// ------------------------------------------------------------------------------------------ stateless operators
int hh_sim_matrix(const float* a, const float* b, float* out, int Na, int Nb, int d, float eps, void* stream) {
  return sim_matrix(a, b, out, Na, Nb, d, eps, S(stream));
}
int hh_row_reduce(const float* x, int rows, int cols, float scale, int mode, void* out, void* stream) {
  return row_reduce(x, rows, cols, scale, mode, out, S(stream));
}
int hh_l2_normalize(const float* x, float* out, int rows, int cols, float eps, void* stream) {
  return l2_normalize_rows(x, out, rows, cols, eps, S(stream));
}
int hh_linear_f32(const float* in, int ldi, const float* in_add, int add_mod, const float* W, const float* bias,
                  const float* residual, int ldres, float* out, int ldo, int R, int N, int K, int act, int in_relu,
                  void* stream) {
  LinArgs la{};
  la.in = in; la.ldi = ldi; la.in_add = in_add; la.add_mod = add_mod; la.W = W; la.bias = bias;
  la.residual = residual; la.ldres = ldres; la.out = out; la.ldo = ldo; la.R = R; la.N = N; la.K = K;
  la.act = act; la.in_relu = in_relu;
  return linear_f32(la, S(stream));
}
int hh_box_cxcywh_to_xyxy(const float* in, float* out, int64_t nboxes, void* stream) {
  return box_cxcywh_to_xyxy(in, out, nboxes, S(stream));
}
int hh_box_xyxy_to_cxcywh(const float* in, float* out, int64_t nboxes, void* stream) {
  return box_xyxy_to_cxcywh(in, out, nboxes, S(stream));
}
int hh_box_pairwise(const float* boxes1, const float* boxes2, int N, int M, float* iou, float* uni, float* giou,
                    void* stream) {
  return box_pairwise(boxes1, boxes2, N, M, iou, uni, giou, S(stream));
}
int hh_box_match_cost(const float* pred, const float* tgt, int N, int M, float w_bbox, float w_giou, float* cost,
                      void* stream) {
  return box_match_cost(pred, tgt, N, M, w_bbox, w_giou, cost, S(stream));
}

int hh_box_loss_forward(const float* pred, const int64_t* src_row, const float* tgt, int K, float num_boxes,
                        float* losses, void* stream) {
  return box_loss_forward(pred, reinterpret_cast<const long long*>(src_row), tgt, K, num_boxes, losses, S(stream));
}
int hh_box_loss_backward(const float* pred, const int64_t* src_row, const float* tgt, int K, float num_boxes,
                         const float* g_losses, float* grad_pred, int64_t pred_rows, void* stream) {
  return box_loss_backward(pred, reinterpret_cast<const long long*>(src_row), tgt, K, num_boxes, g_losses, grad_pred,
                           pred_rows, S(stream));
}
int hh_assign(const float* cost, const int64_t* offset, const int32_t* ld, const int32_t* nr, const int32_t* nc,
              const uint8_t* row_valid, int row_valid_ld, int P, int max_dim, int64_t* row_ind, int64_t* col_ind,
              int32_t* count, int out_ld, void* stream) {
  return assign_lsa(cost, reinterpret_cast<const long long*>(offset), ld, nr, nc, row_valid, row_valid_ld, P,
                    max_dim, reinterpret_cast<long long*>(row_ind), reinterpret_cast<long long*>(col_ind), count, out_ld,
                    S(stream));
}
int hh_match_cost_class(const float* logits, int N, int ncls, const int64_t* ids, int M, float w, float* cost,
                        void* stream) {
  return match_cost_class(logits, N, ncls, reinterpret_cast<const long long*>(ids), M, w, cost, S(stream));
}

// ------------------------------------------------------------------------------------------ losses
size_t hh_sim_matrix_backward_workspace_bytes(int Na, int Nb) { return sim_matrix_backward_workspace_bytes(Na, Nb); }
int hh_sim_matrix_backward(const float* a, const float* b, const float* G, const float* gscale, float* da, float* db,
                           int Na, int Nb, int d, float eps, void* workspace, void* stream) {
  return sim_matrix_backward(a, b, G, gscale, da, db, Na, Nb, d, eps, workspace, S(stream));
}
int hh_egonce_forward(const float* x, int N, int M, const float* mask_v, const float* mask_n, int R, const float* pad,
                      float temperature, float vn_threshold, uint8_t* mask_bool, uint8_t* keep, float* saved,
                      void* stream) {
  return egonce_forward(x, N, M, mask_v, mask_n, R, pad, temperature, vn_threshold, mask_bool, keep, saved, S(stream));
}
int hh_egonce_backward(const float* x, int N, int M, float temperature, const uint8_t* mask_bool, const uint8_t* keep,
                       const float* saved, const float* grad_loss, float* grad_x, void* stream) {
  return egonce_backward(x, N, M, temperature, mask_bool, keep, saved, grad_loss, grad_x, S(stream));
}
size_t hh_word_loss_workspace_bytes(int V, int d, int B2, int Q, int Wm) {
  return word_loss_workspace_bytes(V, d, B2, Q, Wm);
}
int hh_word_loss_forward(const float* noun_embeds, int V, int d, const float* pred, int B2, int Q,
                         const int64_t* gt_inds, int Wm, float temperature, float noun_threshold, int64_t* col_ind,
                         float* sel, int64_t* sel_row, float* dlogits, float* stats, void* workspace, void* stream) {
  return word_loss_forward(noun_embeds, V, d, pred, B2, Q, reinterpret_cast<const long long*>(gt_inds), Wm, temperature,
                           noun_threshold, reinterpret_cast<long long*>(col_ind), sel,
                           reinterpret_cast<long long*>(sel_row), dlogits, stats, workspace, S(stream));
}
int hh_word_loss_backward(const float* noun_embeds, int V, int d, int B2, int Q, int Wm, const float* sel,
                          const int64_t* sel_row, const float* dlogits, float* stats, const float* grad_loss,
                          float* d_pred, float* d_nouns, void* workspace, void* stream) {
  return word_loss_backward(noun_embeds, V, d, B2, Q, Wm, sel, reinterpret_cast<const long long*>(sel_row), dlogits,
                            stats, grad_loss, d_pred, d_nouns, workspace, S(stream));
}

int hh_retrieval_rows(const double* sim, const double* rel, const double* logs, const int32_t* kcounts, int N, int M,
                      int mode, double* out, void* stream) {
  return retrieval_rows(sim, rel, logs, kcounts, N, M, mode, out, S(stream));
}

// ------------------------------------------------------------------------------------------ decoder backward primitives
int hh_linear_f32_backward(const float* dY, int ldy, const float* Y, int ldyo, int act, const float* W, const float* X,
                           int ldx, const float* x_add, int add_mod, int in_relu, float* dX, int lddx, float* dW,
                           float* db, int R, int N, int K, float beta, float scale, void* stream) {
  LinBwdArgs a{};
  a.dY = dY; a.ldy = ldy; a.Y = Y; a.ldyo = ldyo; a.act = act; a.W = W; a.X = X; a.ldx = ldx; a.x_add = x_add;
  a.add_mod = add_mod; a.in_relu = in_relu; a.dX = dX; a.lddx = lddx; a.dW = dW; a.ldw = K; a.db = db; a.R = R; a.N = N;
  a.K = K; a.beta = beta; a.scale = scale;
  if (dX) {
    int rc = linear_dgrad_f32(a, S(stream));
    if (rc) return rc;
  }
  if (dW) return linear_wgrad_f32(a, S(stream));
  return 0;
}
int hh_layernorm_backward(const float* x, int ldx, const float* w, float eps, const float* dy, int lddy, float* dx,
                          float* dgamma, float* dbeta, int M, int D, void* stream) {
  HH_GUARD_BEGIN
  static thread_local DevBuf ws;
  int rc = ws.reserve(ln_backward_workspace_bytes(M, D));
  if (rc) return rc;
  LnBwdArgs a{};
  a.x = x; a.ldx = ldx; a.w = w; a.eps = eps; a.dy = dy; a.lddy = lddy; a.dx = dx; a.dgamma = dgamma; a.dbeta = dbeta;
  a.workspace = ws.ptr; a.M = M; a.D = D;
  return ln_backward_rows(a, S(stream));
  HH_GUARD_END
}
int hh_self_attention_backward(const float* q, const float* k, const float* v, int ld, const float* dO, float* dq,
                               float* dk, float* dv, int ldg, int B, int Q, int heads, void* stream) {
  return self_attn_bwd(q, k, v, ld, dO, dq, dk, dv, ldg, B, Q, heads, S(stream));
}
int hh_cross_attention_backward(const float* q, const void* K, const void* V, int ldkv, const float* O, const float* dO,
                                float* dq, void* dK, void* dV, int lddkv, int B, int Q, int heads, int S_, void* stream) {
  HH_GUARD_BEGIN
  static thread_local DevBuf ws;
  int rc = ws.reserve(cross_attn_bwd_workspace_bytes(B, Q, heads, S_));
  if (rc) return rc;
  return cross_attn_bwd(q, static_cast<const bf16*>(K), static_cast<const bf16*>(V), ldkv, O, dO, dq,
                        static_cast<bf16*>(dK), static_cast<bf16*>(dV), lddkv, B, Q, heads, S_, ws.ptr, S(stream));
  HH_GUARD_END
}

// ------------------------------------------------------------------------------------------ kernel-level entry points
int hh_gemm_bf16(const void* A, int lda, const void* W, int ldw, void* out, int ldc, const float* bias,
                 const float* residual, int ldr, int M, int N, int K, int epilogue, void* stream) {
  return gemm_bf16(static_cast<const bf16*>(A), lda, static_cast<const bf16*>(W), ldw, out, ldc, bias, residual, ldr, M,
                   N, K, epilogue, S(stream));
}
int hh_gemm_stats_parts(int M, int N) { return gemm_stats_parts(M, N); }
int hh_fold_layernorm_weight(const float* W, const float* gamma, const float* beta, const float* bias, int N, int K,
                             int scaled_rows, float scale, void* Wf, float* colsum, float* bias_f, void* stream) {
  return fold_ln_weight(W, gamma, beta, bias, static_cast<bf16*>(Wf), colsum, bias_f, N, K, scaled_rows, scale, S(stream));
}
int hh_gemm_bf16_res_stats(const void* A, int lda, const void* W, int ldw, void* z16, int ldz, const float* bias,
                           float* residual, int ldr, int writeback, float* stats, int M, int N, int K, void* stream) {
  GemmFuse f;
  f.stats_out = stats;
  f.writeback = writeback;
  return gemm_bf16_fused(static_cast<const bf16*>(A), lda, static_cast<const bf16*>(W), ldw, z16, ldz, bias, residual, ldr, M,
                         N, K, EPI_RES_STATS_BF16, f, S(stream));
}
int hh_gemm_bf16_ln(const void* A, int lda, const void* Wf, int ldw, void* out, int ldc, const float* bias_f,
                    const float* colsum, const float* stats, int parts, int norm_dim, float eps, int M, int N, int K,
                    int qgelu, void* stream) {
  GemmFuse f;
  f.colsum = colsum;
  f.stats_in = stats;
  f.stats_parts = parts;
  f.norm_dim = norm_dim;
  f.eps = eps;
  return gemm_bf16_fused(static_cast<const bf16*>(A), lda, static_cast<const bf16*>(Wf), ldw, out, ldc, bias_f, nullptr, 0, M,
                         N, K, qgelu ? EPI_LN_BIAS_QGELU_BF16 : EPI_LN_BIAS_BF16, f, S(stream));
}
int hh_layernorm(const float* x, int ldx, const float* w, const float* b, float eps, float* out_f32, void* out_bf16,
                 int M, int D, void* stream) {
  LnArgs a{};
  a.x = x; a.ldx = ldx; a.w = w; a.b = b; a.eps = eps; a.out_f32 = out_f32; a.out_bf16 = static_cast<bf16*>(out_bf16);
  a.M = M; a.D = D;
  return layernorm_rows(a, S(stream));
}
int hh_f32_to_bf16(const float* src, void* dst, int64_t n, void* stream) {
  return f32_to_bf16(src, static_cast<bf16*>(dst), static_cast<size_t>(n), S(stream));
}
int hh_attention(const void* qkv, void* out, int B, int T, int n, int H, int kind, void* stream) {
  HH_GUARD_BEGIN
  const bf16* q = static_cast<const bf16*>(qkv);
  bf16* o = static_cast<bf16*>(out);
  static thread_local DevBuf ws;
  int rc = ws.reserve(attn_cls_workspace_bytes(B, T, n, H));
  if (rc) return rc;
  switch (kind) {
    case 0: return attn_space(q, o, B, T, n, H, static_cast<float*>(ws.ptr), S(stream));
    case 1: return attn_time(q, o, B, T, n, H, static_cast<float*>(ws.ptr), S(stream));
    case 2: return attn_cls(q, o, B, 1 + T * n, H, S(stream));
  }
  return fail(-2, "hh_attention: kind must be 0 (space), 1 (time) or 2 (stand-alone CLS row)");
  HH_GUARD_END
}
int hh_cross_attention(const float* q, const void* K, const void* V, int ldkv, float* out, int B, int Q, int heads,
                       int S_, void* stream) {
  HH_GUARD_BEGIN
  static thread_local DevBuf ws;
  int rc = ws.reserve(cross_attn_workspace_bytes(B, Q, heads, S_));
  if (rc) return rc;
  return cross_attn(q, static_cast<const bf16*>(K), static_cast<const bf16*>(V), ldkv, out, B, Q, heads, S_, ws.ptr,
                    S(stream));
  HH_GUARD_END
}

int hh_attention_causal(const void* qkv, void* out, int G, int L, int H, void* stream) {
  return attn_causal(static_cast<const bf16*>(qkv), static_cast<bf16*>(out), G, L, H, S(stream));
}

int hh_cross_attention_simt(const float* q, const void* K, const void* V, int ldkv, float* out, int B, int Q, int heads,
                            int S_, void* stream) {
  HH_GUARD_BEGIN
  static thread_local DevBuf ws;
  int rc = ws.reserve(cross_attn_simt_workspace_bytes(B, Q, heads, S_));
  if (rc) return rc;
  return cross_attn_simt(q, static_cast<const bf16*>(K), static_cast<const bf16*>(V), ldkv, out, B, Q, heads, S_, ws.ptr,
                         S(stream));
  HH_GUARD_END
}

// ------------------------------------------------------------------------------------------ NCCL all-gather
namespace {
typedef int (*nccl_get_uid_t)(void*);
struct HhNcclId {  // ncclUniqueId is passed BY VALUE to ncclCommInitRank: 128 opaque bytes
  char internal[HH_NCCL_ID_BYTES];
};
typedef int (*nccl_allgather_t)(const void*, void*, size_t, int, void*, cudaStream_t);
typedef int (*nccl_destroy_t)(void*);
typedef const char* (*nccl_errstr_t)(int);

struct NcclApi {
  void* handle = nullptr;
  nccl_get_uid_t get_uid = nullptr;
  int (*init_rank)(void**, int, HhNcclId, int) = nullptr;
  nccl_allgather_t allgather = nullptr;
  nccl_destroy_t destroy = nullptr;
  nccl_errstr_t errstr = nullptr;
};

NcclApi* nccl_api() {
  static NcclApi api;
  static bool tried = false;
  if (!tried) {
    tried = true;
    // RTLD_NOLOAD first: reuse the copy the host framework (torch) already mapped, so both share one NCCL.
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) {
      api.handle = dlopen(nm, RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);
      if (api.handle) break;
    }
    if (!api.handle)
      for (const char* nm : names) {
        api.handle = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
        if (api.handle) break;
      }
    if (api.handle) {
      api.get_uid = reinterpret_cast<nccl_get_uid_t>(dlsym(api.handle, "ncclGetUniqueId"));
      api.init_rank = reinterpret_cast<int (*)(void**, int, HhNcclId, int)>(dlsym(api.handle, "ncclCommInitRank"));
      api.allgather = reinterpret_cast<nccl_allgather_t>(dlsym(api.handle, "ncclAllGather"));
      api.destroy = reinterpret_cast<nccl_destroy_t>(dlsym(api.handle, "ncclCommDestroy"));
      api.errstr = reinterpret_cast<nccl_errstr_t>(dlsym(api.handle, "ncclGetErrorString"));
    }
  }
  if (!api.handle || !api.get_uid || !api.init_rank || !api.allgather || !api.destroy) return nullptr;
  return &api;
}

int nccl_fail(NcclApi* api, const char* what, int code) {
  return fail(-3, std::string(what) + ": NCCL error " + std::to_string(code) +
                      (api->errstr ? std::string(" (") + api->errstr(code) + ")" : std::string()));
}
}  // namespace

int hh_comm_unique_id(void* id_host) {
  NcclApi* api = nccl_api();
  if (!api) return fail(-3, "hh_comm: libnccl.so.2 not found (load torch, or put NCCL on the library path)");
  if (!id_host) return fail(-2, "hh_comm_unique_id: null buffer");
  int rc = api->get_uid(id_host);
  return rc ? nccl_fail(api, "ncclGetUniqueId", rc) : 0;
}
int hh_comm_create(void** comm, int nranks, int rank, const void* id_host) {
  NcclApi* api = nccl_api();
  if (!api) return fail(-3, "hh_comm: libnccl.so.2 not found (load torch, or put NCCL on the library path)");
  if (!comm || !id_host || nranks < 1 || rank < 0 || rank >= nranks) return fail(-2, "hh_comm_create: bad argument");
  HhNcclId id;
  memcpy(id.internal, id_host, HH_NCCL_ID_BYTES);
  int rc = api->init_rank(comm, nranks, id, rank);
  return rc ? nccl_fail(api, "ncclCommInitRank", rc) : 0;
}
int hh_comm_destroy(void* comm) {
  NcclApi* api = nccl_api();
  if (!api || !comm) return 0;
  int rc = api->destroy(comm);
  return rc ? nccl_fail(api, "ncclCommDestroy", rc) : 0;
}
int hh_allgather(void* comm, const void* send, void* recv, size_t bytes_per_rank, void* stream) {
  NcclApi* api = nccl_api();
  if (!api) return fail(-3, "hh_allgather: NCCL not available");
  if (!comm || !send || !recv) return fail(-2, "hh_allgather: null argument");
  // ncclInt8 == 0 : gather raw bytes so one packed buffer can carry mixed dtypes
  int rc = api->allgather(send, recv, bytes_per_rank, /*ncclInt8*/ 0, comm, S(stream));
  return rc ? nccl_fail(api, "ncclAllGather", rc) : 0;
}

}  // extern "C"
