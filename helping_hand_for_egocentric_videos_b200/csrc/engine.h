// Engine objects behind the opaque hh_encoder / hh_decoder handles of include/hh_b200.h.
#pragma once
#include <map>
#include <string>
#include <vector>

#include "../../include/hh_b200.h"
#include "hh_internal.h"

namespace hh {

struct DevBuf {
  void* ptr = nullptr;
  size_t bytes = 0;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  DevBuf(DevBuf&& o) noexcept : ptr(o.ptr), bytes(o.bytes) { o.ptr = nullptr; o.bytes = 0; }
  ~DevBuf();
  int reserve(size_t nbytes);  // grow-only
  void release();
};

// fp32 master copies of the module's parameters, keyed by reference state_dict name.
struct WeightStore {
  std::map<std::string, int64_t> expected;  // key -> numel
  std::map<std::string, DevBuf> bufs;
  bool dirty = true;
  int set(const std::string& key, const float* data, int64_t numel, cudaStream_t stream);
  const float* get(const std::string& key) const;
  int check_complete() const;
};

// Kernel classes reported by the event profiler (hh_encoder_profile / hh_decoder_profile).
enum KernelClass {
  K_GEMM_QKV = 0, K_GEMM_PROJ, K_GEMM_FC1, K_GEMM_FC2, K_GEMM_PATCH, K_LN, K_ATTN_TIME, K_ATTN_SPACE, K_ATTN_CLS,
  K_EMBED, K_DEC_GEMM, K_DEC_CROSS, K_DEC_QUERY, K_DEC_HEADS, K_NUM
};

struct Profiler {
  bool enabled = false;
  bool open = false;
  struct Rec { int cls; size_t e0, e1; };
  std::vector<cudaEvent_t> pool;
  size_t used = 0;
  std::vector<Rec> recs;
  ~Profiler();
  void begin(int cls, cudaStream_t s);
  void end(cudaStream_t s);
  int collect(double* ms, int* counts);  // waits for the recorded events; sums per class; resets
};

struct Encoder {
  Profiler prof;
  hh_encoder_cfg cfg;
  int grid, n, N, Kpatch, Kp;
  int max_chunk = 64;  // clips per pass through the workspace
  int launches = 0;
  WeightStore weights;
  struct Layer {
    DevBuf w_qkv[2], b_qkv[2], w_proj[2];  // [0] = timeattn, [1] = attn (space)
    DevBuf w_fc1, w_fc2;
    // LayerNorm folded into the contraction (fused_ln): norm3 -> timeattn.qkv, norm1 -> attn.qkv, norm2 -> mlp.fc1
    DevBuf cs_qkv[2], cs_fc1, b_fc1;       // column sums of the gamma-scaled bf16 weights; folded fc1 bias
  };
  std::vector<Layer> layers;
  DevBuf w_patch;
  DevBuf ws_patches, ws_tok, ws_x, ws_dl, ws_dl2, ws_a, ws_qkv, ws_h, ws_cls, ws_stats;
  // true (default): norm1/2/3 and the residual adds live in the GEMM epilogues (model/LaviLa.py:353-388), the stand-alone
  // LayerNorm kernel only runs for the final norm.  HH_LN_UNFUSED=1 keeps the round-1 sequence (A/B and differential tests).
  bool fused_ln = true;

  explicit Encoder(const hh_encoder_cfg& c);
  static int validate(const hh_encoder_cfg& c);
  int pack(cudaStream_t s);
  // The feature map leaves the final norm as fp32 (Fmap::f32) or as bf16 (Fmap::b16, with the CLS rows also written in
  // fp32 to Fmap::cls [B, D] when it is set: the same values as the fp32 map's rows b * N).
  struct Fmap {
    float* f32 = nullptr;
    bf16* b16 = nullptr;
    float* cls = nullptr;
  };
  int forward(const float* video, int B, int nblocks, const Fmap& out, cudaStream_t s);
  // raw frames uint8 [B,T,H,W,3] with the loader's /255 + mean/std normalisation fused into the patch loader
  int forward_u8(const uint8_t* frames, const float* mean, const float* stdv, int B, const Fmap& out, cudaStream_t s);
  double flops_per_clip() const;

 private:
  int run(const float* video, const uint8_t* frames, const float* mean, const float* stdv, int B, int nblocks,
          const Fmap& out, cudaStream_t s);
  int run_blocks_fused(const float* tok, int Bc, int nblocks, LnArgs& final_norm, cudaStream_t s);

 public:
};

struct Decoder {
  Profiler prof;
  hh_decoder_cfg cfg;
  int launches = 0;
  WeightStore weights;
  DevBuf w_proj, w_cls, w_kall, w_vall, b_kall, b_vall, w_sa, b_sa, w_caq, b_caq, pos3d, w_f1, w_f2, frameterm;
  DevBuf ws_feat, ws_memf, ws_mem, ws_mempos, ws_k, ws_v, ws_q, ws_cross, ws_head;

  // ---- training state (engine_bwd.cu): activations of the last forward(save = true) and the parameter gradients
  struct LayerBufs {  // fp32 [B*Q, .] each; in inference mode every layer aliases one set
    float *x0, *x1, *x2, *x3;   // residual stream before norm1 / norm2 / norm3 / after the FFN
    float *n1, *n2, *n3;        // LayerNorm outputs
    float *qkv, *o1;            // self-attention packed projections (q pre-scaled) and core output
    float *qc, *o2;             // cross-attention query projection (pre-scaled) and core output
    float* f;                   // FFN hidden after ReLU
    float* lse;                 // training only: cross-attention row log-sum-exp [B*heads, Q] (nullptr in inference)
  };
  std::vector<LayerBufs> saved;
  int saved_B = 0, saved_T = 0;
  // bumped by EVERY forward (the engine holds one activation set): backward() of an older forward must be refused
  uint64_t generation = 0;
  // dropout of the training forward (hh_decoder_set_dropout): `next_drop` applies to the next forward(save = true),
  // `saved_drop` is what that forward used -- backward() regenerates the same masks from it
  DropCfg next_drop = drop_off(), saved_drop = drop_off();
  float *sv_cond = nullptr, *sv_x1 = nullptr, *sv_x2 = nullptr, *sv_hsproj = nullptr;
  DevBuf ws_train, w_kallT, w_vallT;
  DevBuf bw_a, bw_b, bw_c, bw_d, bw_dk, bw_dv, bw_t1, bw_t2, bw_t3, bw_ws;
  std::map<std::string, DevBuf> grads;
  // second stream of backward() (weight gradients beside the data-gradient chain) and its ordering events
  cudaStream_t bw_side = nullptr;
  cudaEvent_t bw_fork = nullptr, bw_done[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};

  explicit Decoder(const hh_decoder_cfg& c);
  ~Decoder();
  static int validate(const hh_decoder_cfg& c);
  int pack(cudaStream_t s);
  // save = true keeps every layer's activations for backward() (training forward; dropout per next_drop).
  // features: fp32, or bf16 when feat_bf16; inference reads a suitably laid out bf16 map in place (no ws_feat copy)
  int forward(const void* features, bool feat_bf16, int64_t stride_b, int64_t stride_row, int B, int T, float* hs,
              float* logits, float* boxes, cudaStream_t s, bool save = false);
  // Gradients of all decoder parameters for upstream d_hs [L,B,Q,C] and d_boxes [L,B*Tb,Q,4] (either may be null = 0);
  // hs / boxes are the outputs of the matching forward(save = true).  Results are read with grad().
  int backward(const float* hs, const float* boxes, const float* d_hs, const float* d_boxes, cudaStream_t s);
  const float* grad(const std::string& key) const;
  double flops_per_clip(int T) const;
};

// CLIP text tower (text.cu): CLIP.encode_text, model/LaviLa.py:660-670.
struct TextEncoder {
  hh_text_cfg cfg;
  int max_chunk = 1024;  // sequences per pass through the workspace
  int launches = 0;
  WeightStore weights;
  struct Layer {
    DevBuf w_qkv, b_qkv, w_proj, w_fc1, w_fc2;
  };
  std::vector<Layer> layers;
  DevBuf w_projT, flag;
  DevBuf ws_x, ws_dl, ws_a, ws_qkv, ws_h, ws_out, ws_cls;

  explicit TextEncoder(const hh_text_cfg& c);
  static int validate(const hh_text_cfg& c);
  int pack(cudaStream_t s);
  // tokens int64 [G, L] -> embed fp32 [G, E] (x[eot] @ text_projection, may be null), fmap fp32 [G, L, W] (may be null)
  int forward(const int64_t* tokens, int G, float* embed, float* fmap, cudaStream_t s);
  double flops_per_sequence() const;
};

}  // namespace hh
