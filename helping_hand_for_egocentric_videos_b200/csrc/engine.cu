// Encoder / decoder engines: own the packed weights and the workspace arena, sequence the kernels of one forward.
// Host-side C++ only (no kernels here).  Reference call order: model/LaviLa.py:537-573 (encoder) and
// model/tfm_decoder.py:183-233 (decoder); see DESIGN.md for the kernel-by-kernel mapping.
#include "engine.h"

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>

namespace hh {

// ------------------------------------------------------------------------------------------ small utilities
static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }
const char* last_error_cstr() { return g_err.c_str(); }
int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}

int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
        n <= 0)
      n = 148;
  }
  return n;
}

DevBuf::~DevBuf() { release(); }
void DevBuf::release() {
  if (ptr) cudaFree(ptr);
  ptr = nullptr;
  bytes = 0;
}
int DevBuf::reserve(size_t nbytes) {
  if (nbytes <= bytes) return 0;
  release();
  cudaError_t e = cudaMalloc(&ptr, nbytes);
  if (e != cudaSuccess) {
    ptr = nullptr;
    return fail(-3, std::string("cudaMalloc(") + std::to_string(nbytes) + "): " + cudaGetErrorString(e));
  }
  bytes = nbytes;
  return 0;
}

int WeightStore::set(const std::string& key, const float* data, int64_t numel, cudaStream_t stream) {
  auto it = expected.find(key);
  if (it == expected.end()) return fail(-2, "unknown parameter key '" + key + "'");
  if (it->second != numel)
    return fail(-2, "parameter '" + key + "': expected " + std::to_string(it->second) + " elements, got " +
                        std::to_string(numel));
  DevBuf& b = bufs[key];
  int rc = b.reserve(static_cast<size_t>(numel) * sizeof(float));
  if (rc) return rc;
  HH_CHECK_CUDA(cudaMemcpyAsync(b.ptr, data, static_cast<size_t>(numel) * sizeof(float), cudaMemcpyDeviceToDevice, stream));
  dirty = true;
  return 0;
}
const float* WeightStore::get(const std::string& key) const {
  auto it = bufs.find(key);
  return it == bufs.end() ? nullptr : static_cast<const float*>(it->second.ptr);
}
int WeightStore::check_complete() const {
  for (const auto& kv : expected)
    if (bufs.find(kv.first) == bufs.end()) return fail(-2, "parameter '" + kv.first + "' was never set");
  return 0;
}

#define RC(expr)          \
  do {                    \
    int _rc = (expr);     \
    if (_rc) return _rc;  \
  } while (0)

// Launch `expr` bracketed by CUDA events of kernel class `cls` when profiling is on (hh_*_set_profile).
#define PROF(cls, expr)       \
  do {                        \
    prof.begin(cls, s);       \
    int _rc = (expr);         \
    if (_rc) return _rc;      \
    prof.end(s);              \
  } while (0)

// ------------------------------------------------------------------------------------------ event profiler
Profiler::~Profiler() {
  for (cudaEvent_t e : pool) cudaEventDestroy(e);
}
void Profiler::begin(int cls, cudaStream_t s) {
  if (!enabled) return;
  if (used + 2 > pool.size()) {
    for (int i = 0; i < 256; ++i) {
      cudaEvent_t e;
      if (cudaEventCreate(&e) != cudaSuccess) return;
      pool.push_back(e);
    }
  }
  recs.push_back({cls, used, used + 1});
  cudaEventRecord(pool[used], s);
  used += 2;
  open = true;
}
void Profiler::end(cudaStream_t s) {
  if (!enabled || !open) return;
  cudaEventRecord(pool[recs.back().e1], s);
  open = false;
}
int Profiler::collect(double* ms, int* counts) {
  for (int i = 0; i < K_NUM; ++i) {
    ms[i] = 0.0;
    counts[i] = 0;
  }
  for (const Rec& r : recs) {
    HH_CHECK_CUDA(cudaEventSynchronize(pool[r.e1]));
    float t = 0.f;
    HH_CHECK_CUDA(cudaEventElapsedTime(&t, pool[r.e0], pool[r.e1]));
    ms[r.cls] += t;
    counts[r.cls] += 1;
  }
  recs.clear();
  used = 0;
  return 0;
}

// ========================================================================================== encoder
Encoder::Encoder(const hh_encoder_cfg& c) : cfg(c) {
  if (const char* e = std::getenv("HH_ENCODER_CHUNK")) {  // clips per pass through the workspace (tuning knob)
    const int v = std::atoi(e);
    if (v > 0) max_chunk = v;
  }
  if (const char* e = std::getenv("HH_LN_UNFUSED")) fused_ln = !(e[0] && e[0] != '0');
  grid = cfg.img_size / cfg.patch_size;
  n = grid * grid;
  N = 1 + cfg.num_frames * n;
  Kpatch = 3 * cfg.patch_size * cfg.patch_size;
  Kp = (Kpatch + 63) / 64 * 64;
  const int64_t D = cfg.embed_dim, Hd = cfg.mlp_hidden;
  auto& e = weights.expected;
  e["cls_token"] = D;
  e["pos_embed"] = (n + 1) * D;
  e["temporal_embed"] = cfg.num_frames * D;
  e["patch_embed.proj.weight"] = D * Kpatch;
  for (const char* nm : {"ln_pre", "norm"}) {
    e[std::string(nm) + ".weight"] = D;
    e[std::string(nm) + ".bias"] = D;
  }
  for (int i = 0; i < cfg.depth; ++i) {
    const std::string p = "blocks." + std::to_string(i) + ".";
    for (const char* nm : {"norm1", "norm2", "norm3"}) {
      e[p + nm + ".weight"] = D;
      e[p + nm + ".bias"] = D;
    }
    for (const char* at : {"attn", "timeattn"}) {
      e[p + at + ".qkv.weight"] = 3 * D * D;
      e[p + at + ".qkv.bias"] = 3 * D;
      e[p + at + ".proj.weight"] = D * D;
      e[p + at + ".proj.bias"] = D;
    }
    e[p + "mlp.fc1.weight"] = Hd * D;
    e[p + "mlp.fc1.bias"] = Hd;
    e[p + "mlp.fc2.weight"] = D * Hd;
    e[p + "mlp.fc2.bias"] = D;
  }
}

int Encoder::validate(const hh_encoder_cfg& c) {
  HH_REQUIRE(c.embed_dim % 128 == 0 && c.embed_dim <= 1024, "encoder: embed_dim must be a multiple of 128, <= 1024");
  HH_REQUIRE(c.num_heads > 0 && c.embed_dim == c.num_heads * 64, "encoder: head dim must be 64");
  HH_REQUIRE(c.patch_size > 0 && c.patch_size % 2 == 0 && c.img_size % c.patch_size == 0, "encoder: patch/img size");
  HH_REQUIRE(c.num_frames >= 1 && c.num_frames <= 32, "encoder: 1..32 frames");
  HH_REQUIRE(c.depth >= 1 && c.mlp_hidden % 64 == 0, "encoder: depth / mlp_hidden");
  return 0;
}

int Encoder::pack(cudaStream_t s) {
  RC(weights.check_complete());
  const int D = cfg.embed_dim, Hd = cfg.mlp_hidden;
  const float qscale = 1.0f / std::sqrt(64.0f);  // VarAttention.scale (LaviLa.py:233,252), folded into Wq / bq
  RC(w_patch.reserve(static_cast<size_t>(D) * Kp * 2));
  RC(pack_weight_bf16(weights.get("patch_embed.proj.weight"), static_cast<bf16*>(w_patch.ptr), D, Kpatch, Kp, 0, 1.f, s));
  layers.resize(cfg.depth);
  for (int i = 0; i < cfg.depth; ++i) {
    const std::string p = "blocks." + std::to_string(i) + ".";
    Layer& L = layers[i];
    const char* ats[2] = {"timeattn", "attn"};
    const char* nms[2] = {"norm3", "norm1"};  // the LayerNorm in front of each attention's qkv (LaviLa.py:353,372)
    for (int a = 0; a < 2; ++a) {
      const std::string q = p + ats[a];
      RC(L.w_qkv[a].reserve(static_cast<size_t>(3) * D * D * 2));
      RC(L.b_qkv[a].reserve(static_cast<size_t>(3) * D * 4));
      if (fused_ln) {
        RC(L.cs_qkv[a].reserve(static_cast<size_t>(3) * D * 4));
        RC(fold_ln_weight(weights.get(q + ".qkv.weight"), weights.get(p + nms[a] + ".weight"), weights.get(p + nms[a] + ".bias"),
                          weights.get(q + ".qkv.bias"), static_cast<bf16*>(L.w_qkv[a].ptr), static_cast<float*>(L.cs_qkv[a].ptr),
                          static_cast<float*>(L.b_qkv[a].ptr), 3 * D, D, D, qscale, s));
      } else {
        RC(pack_weight_bf16(weights.get(q + ".qkv.weight"), static_cast<bf16*>(L.w_qkv[a].ptr), 3 * D, D, D, D, qscale, s));
        RC(scale_copy_f32(weights.get(q + ".qkv.bias"), static_cast<float*>(L.b_qkv[a].ptr), 3 * D, D, qscale, s));
      }
      RC(L.w_proj[a].reserve(static_cast<size_t>(D) * D * 2));
      RC(pack_weight_bf16(weights.get(q + ".proj.weight"), static_cast<bf16*>(L.w_proj[a].ptr), D, D, D, 0, 1.f, s));
    }
    RC(L.w_fc1.reserve(static_cast<size_t>(Hd) * D * 2));
    if (fused_ln) {  // norm2 -> fc1 (LaviLa.py:388)
      RC(L.cs_fc1.reserve(static_cast<size_t>(Hd) * 4));
      RC(L.b_fc1.reserve(static_cast<size_t>(Hd) * 4));
      RC(fold_ln_weight(weights.get(p + "mlp.fc1.weight"), weights.get(p + "norm2.weight"), weights.get(p + "norm2.bias"),
                        weights.get(p + "mlp.fc1.bias"), static_cast<bf16*>(L.w_fc1.ptr), static_cast<float*>(L.cs_fc1.ptr),
                        static_cast<float*>(L.b_fc1.ptr), Hd, D, 0, 1.f, s));
    } else {
      RC(pack_weight_bf16(weights.get(p + "mlp.fc1.weight"), static_cast<bf16*>(L.w_fc1.ptr), Hd, D, D, 0, 1.f, s));
    }
    RC(L.w_fc2.reserve(static_cast<size_t>(D) * Hd * 2));
    RC(pack_weight_bf16(weights.get(p + "mlp.fc2.weight"), static_cast<bf16*>(L.w_fc2.ptr), D, Hd, Hd, 0, 1.f, s));
  }
  weights.dirty = false;
  return 0;
}

int Encoder::forward(const float* video, int B, int nblocks, const Fmap& out, cudaStream_t s) {
  HH_REQUIRE(video != nullptr, "encoder forward: null buffer");
  return run(video, nullptr, nullptr, nullptr, B, nblocks, out, s);
}

int Encoder::forward_u8(const uint8_t* frames, const float* mean, const float* stdv, int B, const Fmap& out, cudaStream_t s) {
  HH_REQUIRE(frames != nullptr && mean != nullptr && stdv != nullptr, "encoder forward_u8: null buffer");
  return run(nullptr, frames, mean, stdv, B, -1, out, s);
}

int Encoder::run(const float* video, const uint8_t* frames, const float* mean, const float* stdv, int B, int nblocks,
                 const Fmap& out, cudaStream_t s) {
  HH_REQUIRE(B > 0, "encoder forward: empty batch");
  HH_REQUIRE((out.f32 != nullptr) != (out.b16 != nullptr), "encoder forward: exactly one feature-map buffer");
  HH_REQUIRE(out.cls == nullptr || out.b16 != nullptr, "encoder forward: the CLS buffer goes with the bf16 map");
  if (weights.dirty) RC(pack(s));
  if (nblocks < 0 || nblocks > cfg.depth) nblocks = cfg.depth;
  launches = 0;
  const int T = cfg.num_frames, D = cfg.embed_dim, H = cfg.num_heads, Hd = cfg.mlp_hidden;
  const int chunk = B < max_chunk ? B : max_chunk;
  // workspace for one chunk
  const size_t Mc = static_cast<size_t>(chunk) * N;
  const size_t Pc = static_cast<size_t>(chunk) * T * n;
  RC(ws_patches.reserve(Pc * Kp * 2));
  RC(ws_tok.reserve(Pc * D * 4));
  RC(ws_x.reserve(Mc * D * 4));
  RC(ws_dl.reserve(Mc * D * 2));
  RC(ws_dl2.reserve(Mc * D * 2));
  RC(ws_a.reserve(Mc * D * 2));
  RC(ws_qkv.reserve(Mc * 3 * D * 2));
  RC(ws_h.reserve(Mc * Hd * 2));
  RC(ws_cls.reserve(attn_cls_workspace_bytes(chunk, T, n, H)));
  if (fused_ln) RC(ws_stats.reserve(Mc * 2 * 4 * static_cast<size_t>(D / 128 > 1 ? D / 128 : 1)));
  bf16* patches = static_cast<bf16*>(ws_patches.ptr);
  float* tok = static_cast<float*>(ws_tok.ptr);
  float* x = static_cast<float*>(ws_x.ptr);
  bf16* dl = static_cast<bf16*>(ws_dl.ptr);
  bf16* dls = static_cast<bf16*>(ws_dl2.ptr);   // spatial branch output, pending until the next layer's norm3
  bf16* a = static_cast<bf16*>(ws_a.ptr);
  bf16* qkv = static_cast<bf16*>(ws_qkv.ptr);
  bf16* h = static_cast<bf16*>(ws_h.ptr);
  float* cls_ws = static_cast<float*>(ws_cls.ptr);
  const size_t frame_elems = static_cast<size_t>(3) * cfg.img_size * cfg.img_size;

  for (int b0 = 0; b0 < B; b0 += chunk) {
    const int Bc = (B - b0) < chunk ? (B - b0) : chunk;
    const int M = Bc * N;
    const int P = Bc * T * n;
    // this chunk's rows of the final norm's outputs (fp32 map, or bf16 map + fp32 CLS rows)
    LnArgs fin{};
    fin.out_f32 = out.f32 ? out.f32 + static_cast<size_t>(b0) * N * D : nullptr;
    fin.out_bf16 = out.b16 ? out.b16 + static_cast<size_t>(b0) * N * D : nullptr;
    fin.cls_f32 = out.cls ? out.cls + static_cast<size_t>(b0) * D : nullptr;
    fin.cls_mod = N;
    // patch embed (LaviLa.py:218-223,540-542) + CLS/pos/temporal + ln_pre (:545-559)
    if (frames) {
      PROF(K_EMBED, im2col_patches_u8(frames + static_cast<size_t>(b0) * T * frame_elems, mean, stdv, patches, Bc * T,
                                      cfg.img_size, cfg.img_size, cfg.patch_size, Kp, s));
    } else {
      PROF(K_EMBED, im2col_patches(video + static_cast<size_t>(b0) * T * frame_elems, patches, Bc * T, cfg.img_size,
                                   cfg.img_size, cfg.patch_size, Kp, s));
    }
    PROF(K_GEMM_PATCH, gemm_bf16(patches, Kp, static_cast<const bf16*>(w_patch.ptr), Kp, tok, D, nullptr, nullptr, 0, P, D,
                                 Kp, EPI_BIAS_F32, s));
    if (fused_ln) {
      RC(run_blocks_fused(tok, Bc, nblocks, fin, s));
      continue;
    }
    PROF(K_EMBED, assemble_tokens_ln(tok, weights.get("cls_token"), weights.get("pos_embed"), weights.get("temporal_embed"),
                                     weights.get("ln_pre.weight"), weights.get("ln_pre.bias"), 1e-5f, x, Bc, T, n, D, s));
    launches += 3;
    // bf16 branch outputs not yet folded into the fp32 residual stream x: the spatial-attention output and the MLP
    // output of a layer are BOTH added by the next layer's norm3 pass, x <- (x + space_out) + mlp_out -- the same two
    // fp32 additions in the same order as adding them one at a time, but x is written once per layer instead of twice
    const bf16* pending = nullptr;
    const bf16* pending2 = nullptr;
    auto ln_fused = [&](const bf16* delta, const bf16* delta2, bool write_x, const std::string& nm, float eps,
                        bf16* out16, float* out32, float* cls32 = nullptr) {
      LnArgs ln{};
      ln.x = x;
      ln.ldx = D;
      ln.delta = delta;
      ln.delta2 = delta2;
      ln.xsum_out = (delta && write_x) ? x : nullptr;
      ln.w = weights.get(nm + ".weight");
      ln.b = weights.get(nm + ".bias");
      ln.eps = eps;
      ln.out_bf16 = out16;
      ln.out_f32 = out32;
      ln.cls_f32 = cls32;
      ln.cls_mod = N;
      ln.M = M;
      ln.D = D;
      prof.begin(K_LN, s);
      int rc = layernorm_rows(ln, s);
      prof.end(s);
      return rc;
    };
    for (int i = 0; i < nblocks; ++i) {
      const std::string p = "blocks." + std::to_string(i) + ".";
      const Layer& L = layers[i];
      // Residual adds are folded into the LayerNorms (fp32 passes instead of GEMM-epilogue read-modify-writes):
      //   norm3 reads x + space_out(prev) + mlp_out(prev) and stores it as the new x;
      //   norm1 reads x + time_out (never stored: 'frozen-in-time' discards it, LaviLa.py:364,384);
      //   norm2 reads x + space_out (not stored either: the sum is formed again, bit-identically, by the next norm3).
      for (int at = 0; at < 2; ++at) {  // 0 = time (norm3), 1 = space (norm1)
        const std::string q = p + (at == 0 ? "timeattn" : "attn");
        if (at == 0) RC(ln_fused(pending, pending2, true, p + "norm3", 1e-6f, a, nullptr));
        else RC(ln_fused(dl, nullptr, false, p + "norm1", 1e-6f, a, nullptr));
        PROF(K_GEMM_QKV, gemm_bf16(a, D, static_cast<const bf16*>(L.w_qkv[at].ptr), D, qkv, 3 * D,
                                   static_cast<const float*>(L.b_qkv[at].ptr), nullptr, 0, M, 3 * D, D, EPI_BIAS_BF16, s));
        if (at == 0) PROF(K_ATTN_TIME, attn_time(qkv, a, Bc, T, n, H, cls_ws, s));
        else PROF(K_ATTN_SPACE, attn_space(qkv, a, Bc, T, n, H, cls_ws, s));
        PROF(K_GEMM_PROJ, gemm_bf16(a, D, static_cast<const bf16*>(L.w_proj[at].ptr), D, at == 0 ? dl : dls, D,
                                    weights.get(q + ".proj.bias"), nullptr, 0, M, D, D, EPI_BIAS_BF16, s));
        launches += 5;
      }
      RC(ln_fused(dls, nullptr, false, p + "norm2", 1e-6f, a, nullptr));  // a = norm2(x + space_out)
      PROF(K_GEMM_FC1, gemm_bf16(a, D, static_cast<const bf16*>(L.w_fc1.ptr), D, h, Hd, weights.get(p + "mlp.fc1.bias"), nullptr,
                                 0, M, Hd, D, EPI_BIAS_QGELU_BF16, s));
      PROF(K_GEMM_FC2, gemm_bf16(h, Hd, static_cast<const bf16*>(L.w_fc2.ptr), Hd, dl, D, weights.get(p + "mlp.fc2.bias"), nullptr,
                                 0, M, D, Hd, EPI_BIAS_BF16, s));
      pending = dls;   // x + space_out + mlp_out is formed by the next norm3 (or the final norm)
      pending2 = dl;
      launches += 3;
    }
    RC(ln_fused(pending, pending2, false, "norm", 1e-6f, fin.out_bf16, fin.out_f32, fin.cls_f32));
    launches += 1;
  }
  return 0;
}

// Blocks with norm1 / norm2 / norm3 and the residual adds folded into the contractions (model/LaviLa.py:345-390).
// Per layer, with x the fp32 stream, z a bf16 copy of the un-normalised GEMM input and (sum, sum^2) row statistics:
//   qkv_t = Linear'(z, stats)                          norm3 folded into timeattn.qkv         (:353)
//   z     = x + proj_t(attn_time(qkv_t)), stats        x itself untouched: 'frozen-in-time'   (:364)
//   qkv_s = Linear'(z, stats)                          norm1 folded into attn.qkv             (:372)
//   x, z  = x + proj_s(attn_space(qkv_s)), stats       fp32 sum written back in place         (:384)
//   h     = QuickGELU(Linear'(z, stats))               norm2 folded into mlp.fc1              (:388)
//   x, z  = x + fc2(h), stats                                                                 (:388)
// x moves 26 bytes per element per layer (3 reads, 2 writes, 3 bf16 copies) instead of 36, in 8 launches instead of 11.
int Encoder::run_blocks_fused(const float* tok, int Bc, int nblocks, LnArgs& ln, cudaStream_t s) {
  const int T = cfg.num_frames, D = cfg.embed_dim, H = cfg.num_heads, Hd = cfg.mlp_hidden;
  const int M = Bc * N;
  float* x = static_cast<float*>(ws_x.ptr);
  bf16* z = static_cast<bf16*>(ws_dl.ptr);
  bf16* a = static_cast<bf16*>(ws_a.ptr);
  bf16* qkv = static_cast<bf16*>(ws_qkv.ptr);
  bf16* h = static_cast<bf16*>(ws_h.ptr);
  float* stats = static_cast<float*>(ws_stats.ptr);
  float* cls_ws = static_cast<float*>(ws_cls.ptr);
  PROF(K_EMBED, assemble_tokens_ln(tok, weights.get("cls_token"), weights.get("pos_embed"), weights.get("temporal_embed"),
                                   weights.get("ln_pre.weight"), weights.get("ln_pre.bias"), 1e-5f, x, Bc, T, n, D, s, z, stats));
  launches += 3;
  int parts = 1;  // statistics partials per row currently in `stats`
  const int parts_d = gemm_stats_parts(M, D);
  auto consume = [&](const DevBuf& W, const DevBuf& bias, const DevBuf& cs, bf16* out, int Nout, int epi) {
    GemmFuse f;
    f.colsum = static_cast<const float*>(cs.ptr);
    f.stats_in = stats;
    f.stats_parts = parts;
    f.norm_dim = D;
    f.eps = 1e-6f;
    return gemm_bf16_fused(z, D, static_cast<const bf16*>(W.ptr), D, out, Nout, static_cast<const float*>(bias.ptr), nullptr, 0,
                           M, Nout, D, epi, f, s);
  };
  auto produce = [&](const bf16* A, int K, const DevBuf& W, const float* bias, bool writeback) {
    GemmFuse f;
    f.stats_out = stats;
    f.writeback = writeback ? 1 : 0;
    const int rc = gemm_bf16_fused(A, K, static_cast<const bf16*>(W.ptr), K, z, D, bias, x, D, M, D, K, EPI_RES_STATS_BF16, f, s);
    parts = parts_d;
    return rc;
  };
  for (int i = 0; i < nblocks; ++i) {
    const std::string p = "blocks." + std::to_string(i) + ".";
    const Layer& L = layers[i];
    PROF(K_GEMM_QKV, consume(L.w_qkv[0], L.b_qkv[0], L.cs_qkv[0], qkv, 3 * D, EPI_LN_BIAS_BF16));
    PROF(K_ATTN_TIME, attn_time(qkv, a, Bc, T, n, H, cls_ws, s));
    PROF(K_GEMM_PROJ, produce(a, D, L.w_proj[0], weights.get(p + "timeattn.proj.bias"), false));
    PROF(K_GEMM_QKV, consume(L.w_qkv[1], L.b_qkv[1], L.cs_qkv[1], qkv, 3 * D, EPI_LN_BIAS_BF16));
    PROF(K_ATTN_SPACE, attn_space(qkv, a, Bc, T, n, H, cls_ws, s));
    PROF(K_GEMM_PROJ, produce(a, D, L.w_proj[1], weights.get(p + "attn.proj.bias"), true));
    PROF(K_GEMM_FC1, consume(L.w_fc1, L.b_fc1, L.cs_fc1, h, Hd, EPI_LN_BIAS_QGELU_BF16));
    PROF(K_GEMM_FC2, produce(h, Hd, L.w_fc2, weights.get(p + "mlp.fc2.bias"), true));
    launches += 8;
  }
  // final norm into the outputs the caller set in `ln`
  ln.x = x;
  ln.ldx = D;
  ln.w = weights.get("norm.weight");
  ln.b = weights.get("norm.bias");
  ln.eps = 1e-6f;
  ln.M = M;
  ln.D = D;
  PROF(K_LN, layernorm_rows(ln, s));
  launches += 1;
  return 0;
}

double Encoder::flops_per_clip() const {
  // SURVEY.md section 8(d): F_enc = 2 nT 3p^2 D + L [32 N D^2 + 4 D (n T (T+1) + N) + 4 D (T n (n+1) + N)] + 2 D 256
  const double D = cfg.embed_dim, T = cfg.num_frames, nn = n, NN = N, L = cfg.depth;
  const double ratio = static_cast<double>(cfg.mlp_hidden) / cfg.embed_dim;
  const double lin = (16.0 + 4.0 * ratio) * NN * D * D;  // qkv x2 (12) + proj x2 (4) + mlp (4*ratio) -> 32 at ratio 4
  return 2.0 * nn * T * Kpatch * D + L * (lin + 4.0 * D * (nn * T * (T + 1) + NN) + 4.0 * D * (T * nn * (nn + 1) + NN)) +
         2.0 * D * 256.0;
}

// ========================================================================================== decoder
Decoder::Decoder(const hh_decoder_cfg& c) : cfg(c) {
  const int64_t C = cfg.d_model, Fd = cfg.dim_feedforward;
  auto& e = weights.expected;
  e["pos_embed"] = (cfg.patches_per_frame + 1) * C;
  e["temporal_embed"] = cfg.num_frames * C;
  e["transformer.pre_norm.weight"] = C;
  e["transformer.pre_norm.bias"] = C;
  e["transformer.decoder.norm.weight"] = C;
  e["transformer.decoder.norm.bias"] = C;
  e["class_embed.weight"] = static_cast<int64_t>(cfg.num_classes1) * C;
  e["class_embed.bias"] = cfg.num_classes1;
  e["query_embed.weight"] = cfg.num_queries * C;
  e["proj.weight"] = C * cfg.feature_dim;
  const int64_t dims[4] = {C, C, C, 4};
  for (int j = 0; j < 3; ++j) {
    e["bbox_embed.layers." + std::to_string(j) + ".weight"] = dims[j + 1] * dims[j];
    e["bbox_embed.layers." + std::to_string(j) + ".bias"] = dims[j + 1];
  }
  if (cfg.pred_traj) {
    e["frame_index.weight"] = cfg.num_frames * C;
    e["frame_proj.weight"] = C * 2 * C;
    e["frame_proj.bias"] = C;
  }
  for (int i = 0; i < cfg.num_layers; ++i) {
    const std::string p = "transformer.decoder.layers." + std::to_string(i) + ".";
    for (const char* at : {"multihead_attn", "self_attn"}) {
      e[p + at + ".in_proj_weight"] = 3 * C * C;
      e[p + at + ".in_proj_bias"] = 3 * C;
      e[p + at + ".out_proj.weight"] = C * C;
      e[p + at + ".out_proj.bias"] = C;
    }
    e[p + "linear1.weight"] = Fd * C;
    e[p + "linear1.bias"] = Fd;
    e[p + "linear2.weight"] = C * Fd;
    e[p + "linear2.bias"] = C;
    for (const char* nm : {"norm1", "norm2", "norm3"}) {
      e[p + nm + ".weight"] = C;
      e[p + nm + ".bias"] = C;
    }
  }
}

int Decoder::validate(const hh_decoder_cfg& c) {
  HH_REQUIRE(c.d_model % 128 == 0 && c.d_model <= 1024, "decoder: d_model must be a multiple of 128, <= 1024");
  HH_REQUIRE(c.nhead > 0 && c.d_model == c.nhead * 64, "decoder: head dim must be 64");
  HH_REQUIRE(c.num_queries >= 1 && c.num_queries <= kMaxQueries,
             "decoder: 1..32 queries (num_queries==1 n_decode path unsupported)");
  HH_REQUIRE(c.num_layers >= 1 && c.dim_feedforward % 32 == 0, "decoder: layers / ffn");
  HH_REQUIRE(c.feature_dim % 8 == 0 && c.num_classes1 >= 1, "decoder: feature_dim must be a multiple of 8");
  HH_REQUIRE(c.num_frames >= 1 && c.patches_per_frame >= 1, "decoder: frames / patches");
  return 0;
}

int Decoder::pack(cudaStream_t s) {
  RC(weights.check_complete());
  const int C = cfg.d_model, Lr = cfg.num_layers, F = cfg.feature_dim;
  const float qscale = 1.0f / std::sqrt(64.0f);  // nn.MultiheadAttention scales q by head_dim^-0.5
  RC(w_proj.reserve(static_cast<size_t>(C) * F * 2));
  RC(pack_weight_bf16(weights.get("proj.weight"), static_cast<bf16*>(w_proj.ptr), C, F, F, 0, 1.f, s));
  RC(w_cls.reserve(static_cast<size_t>(cfg.num_classes1) * C * 2));
  RC(pack_weight_bf16(weights.get("class_embed.weight"), static_cast<bf16*>(w_cls.ptr), cfg.num_classes1, C, C, 0, 1.f, s));
  // memory is layer-invariant: the 6 layers' cross-attention K (resp. V) projections become ONE GEMM each
  RC(w_kall.reserve(static_cast<size_t>(Lr) * C * C * 2));
  RC(w_vall.reserve(static_cast<size_t>(Lr) * C * C * 2));
  RC(b_kall.reserve(static_cast<size_t>(Lr) * C * 4));
  RC(b_vall.reserve(static_cast<size_t>(Lr) * C * 4));
  RC(w_sa.reserve(static_cast<size_t>(Lr) * 3 * C * C * 4));
  RC(b_sa.reserve(static_cast<size_t>(Lr) * 3 * C * 4));
  RC(w_caq.reserve(static_cast<size_t>(Lr) * C * C * 4));
  RC(b_caq.reserve(static_cast<size_t>(Lr) * C * 4));
  for (int i = 0; i < Lr; ++i) {
    const std::string p = "transformer.decoder.layers." + std::to_string(i) + ".";
    const float* wca = weights.get(p + "multihead_attn.in_proj_weight");
    const float* bca = weights.get(p + "multihead_attn.in_proj_bias");
    RC(pack_weight_bf16(wca + static_cast<size_t>(C) * C, static_cast<bf16*>(w_kall.ptr) + static_cast<size_t>(i) * C * C, C, C,
                        C, 0, 1.f, s));
    RC(pack_weight_bf16(wca + static_cast<size_t>(2) * C * C, static_cast<bf16*>(w_vall.ptr) + static_cast<size_t>(i) * C * C,
                        C, C, C, 0, 1.f, s));
    RC(scale_copy_f32(bca + C, static_cast<float*>(b_kall.ptr) + static_cast<size_t>(i) * C, C, 0, 1.f, s));
    RC(scale_copy_f32(bca + 2 * C, static_cast<float*>(b_vall.ptr) + static_cast<size_t>(i) * C, C, 0, 1.f, s));
    RC(scale_copy_f32(wca, static_cast<float*>(w_caq.ptr) + static_cast<size_t>(i) * C * C, static_cast<size_t>(C) * C,
                      static_cast<size_t>(C) * C, qscale, s));
    RC(scale_copy_f32(bca, static_cast<float*>(b_caq.ptr) + static_cast<size_t>(i) * C, C, C, qscale, s));
    RC(scale_copy_f32(weights.get(p + "self_attn.in_proj_weight"), static_cast<float*>(w_sa.ptr) + static_cast<size_t>(i) * 3 * C * C,
                      static_cast<size_t>(3) * C * C, static_cast<size_t>(C) * C, qscale, s));
    RC(scale_copy_f32(weights.get(p + "self_attn.in_proj_bias"), static_cast<float*>(b_sa.ptr) + static_cast<size_t>(i) * 3 * C,
                      3 * C, C, qscale, s));
  }
  // K-major copies of the K / V projection weights for the data-gradient GEMMs of backward(): [C, L*C]
  RC(w_kallT.reserve(static_cast<size_t>(Lr) * C * C * 2));
  RC(w_vallT.reserve(static_cast<size_t>(Lr) * C * C * 2));
  RC(transpose_to_bf16(w_kall.ptr, 1, C, static_cast<bf16*>(w_kallT.ptr), static_cast<long long>(Lr) * C, C, s));
  RC(transpose_to_bf16(w_vall.ptr, 1, C, static_cast<bf16*>(w_vallT.ptr), static_cast<long long>(Lr) * C, C, s));
  // constant 3-D position embedding (tfm_decoder.py:161-166)
  const int S = cfg.num_frames * cfg.patches_per_frame;
  RC(pos3d.reserve(static_cast<size_t>(S) * C * 4));
  RC(build_pos3d(weights.get("pos_embed"), weights.get("temporal_embed"), static_cast<float*>(pos3d.ptr), cfg.num_frames,
                 cfg.patches_per_frame, C, s));
  if (cfg.pred_traj) {
    // frame_proj([hs ; frame_index[t]]) = hs W1^T + (frame_index[t] W2^T + b)   (tfm_decoder.py:212-215)
    RC(w_f1.reserve(static_cast<size_t>(C) * C * 4));
    RC(w_f2.reserve(static_cast<size_t>(C) * C * 4));
    RC(frameterm.reserve(static_cast<size_t>(cfg.num_frames) * C * 4));
    RC(slice_cols_f32(weights.get("frame_proj.weight"), 2 * C, 0, static_cast<float*>(w_f1.ptr), C, C, s));
    RC(slice_cols_f32(weights.get("frame_proj.weight"), 2 * C, C, static_cast<float*>(w_f2.ptr), C, C, s));
    LinArgs la{};
    la.in = weights.get("frame_index.weight");
    la.ldi = C;
    la.W = static_cast<const float*>(w_f2.ptr);
    la.bias = weights.get("frame_proj.bias");
    la.out = static_cast<float*>(frameterm.ptr);
    la.ldo = C;
    la.R = cfg.num_frames;
    la.N = C;
    la.K = C;
    RC(linear_f32(la, s));
  }
  weights.dirty = false;
  return 0;
}

static int lin(const float* in, int ldi, const float* in_add, int add_mod, const float* W, const float* bias,
               const float* residual, int ldres, float* out, int ldo, int R, int N, int K, int act, cudaStream_t s,
               DropCfg drop = drop_off(), uint32_t drop_site = 0) {
  LinArgs la{};
  la.in = in; la.ldi = ldi; la.in_add = in_add; la.add_mod = add_mod; la.W = W; la.bias = bias;
  la.residual = residual; la.ldres = ldres; la.out = out; la.ldo = ldo; la.R = R; la.N = N; la.K = K; la.act = act;
  la.drop = drop; la.drop_site = drop_site;
  return linear_f32(la, s);
}

int Decoder::forward(const void* features, bool feat_bf16, int64_t stride_b, int64_t stride_row, int B, int T, float* hs,
                     float* logits, float* boxes, cudaStream_t s, bool save) {
  HH_REQUIRE(B > 0 && features && hs && logits && boxes, "decoder forward: bad arguments");
  HH_REQUIRE(T == cfg.num_frames, "decoder forward: T must equal num_frames (construct_3d_pos_embed, tfm_decoder.py:161-166)");
  if (weights.dirty) RC(pack(s));
  launches = 0;
  ++generation;
  const int C = cfg.d_model, Lr = cfg.num_layers, F = cfg.feature_dim, Q = cfg.num_queries, Fd = cfg.dim_feedforward;
  const int n = cfg.patches_per_frame, S = T * n, heads = cfg.nhead, ncls = cfg.num_classes1;
  const int R = B * Q;
  const size_t BS = static_cast<size_t>(B) * S;
  // Direct path (inference, bf16 map): the proj GEMM reads A from the caller's rows, clip b's S patch rows starting at
  // row b * pitch (pitch = stride_b / stride_row: image_feature_map[:, 1:] skips each clip's CLS row).  TMA needs 16-byte
  // rows and segments of whole 128-row tiles.  Every other case gathers the rows into ws_feat first; the training
  // forward always does, because backward() reads that copy (the caller may reuse its tensor before backward()).
  const int64_t pitch = (B == 1) ? S : (stride_row > 0 ? stride_b / stride_row : 0);
  const bool direct = feat_bf16 && !save && S % 128 == 0 && (reinterpret_cast<uintptr_t>(features) & 15) == 0 &&
                      stride_row > 0 && stride_row % 8 == 0 && (B == 1 || (stride_b % stride_row == 0 && pitch >= S)) &&
                      stride_row <= 0x7fffffff && pitch <= 0x7fffffff;
  if (!direct) RC(ws_feat.reserve(BS * F * 2));
  RC(ws_memf.reserve(BS * C * 4));
  RC(ws_mem.reserve(BS * C * 2));
  RC(ws_mempos.reserve(BS * C * 2));
  RC(ws_k.reserve(BS * Lr * C * 2));
  RC(ws_v.reserve(BS * Lr * C * 2));
  RC(ws_q.reserve(static_cast<size_t>(R) * (3 * C /*tgt,t2,o*/ + 3 * C /*qkv*/ + Fd) * 4));
  RC(ws_cross.reserve(cross_attn_workspace_bytes(B, Q, heads, S)));
  const bool traj = cfg.pred_traj && T == cfg.num_frames;
  const size_t LR = static_cast<size_t>(Lr) * R;
  RC(ws_head.reserve((LR * C * 2 /*bf16 hs*/) + LR * C * 4 /*hsproj*/ + LR * (traj ? T : 1) * C * 4 * 3 /*cond,x1,x2*/ +
                     (traj ? LR * static_cast<size_t>(ncls) * 4 : 0)));

  bf16* feat = static_cast<bf16*>(ws_feat.ptr);
  float* memf = static_cast<float*>(ws_memf.ptr);
  bf16* mem = static_cast<bf16*>(ws_mem.ptr);
  bf16* mempos = static_cast<bf16*>(ws_mempos.ptr);
  bf16* Kall = static_cast<bf16*>(ws_k.ptr);
  bf16* Vall = static_cast<bf16*>(ws_v.ptr);
  float* tgt = static_cast<float*>(ws_q.ptr);
  const float* qpos = weights.get("query_embed.weight");
  // per-layer activation buffers: one shared set in inference, one set per layer when saving for backward()
  saved.assign(Lr, LayerBufs{});
  {
    const size_t RC_ = static_cast<size_t>(R) * C;
    if (!save) {
      float* t2 = tgt + RC_;
      float* o = t2 + RC_;
      float* qkv = o + RC_;
      float* ffn = qkv + 3 * RC_;
      for (auto& b : saved) b = LayerBufs{tgt, tgt, tgt, tgt, t2, t2, t2, qkv, o, qkv, o, ffn, nullptr};
      saved_B = 0;
    } else {
      const size_t per = 12 * RC_ + static_cast<size_t>(R) * Fd;  // x0,x1,x2,n1,n2,n3 (6) qkv (3) o1,qc,o2 (3) + f
      const size_t nlse = static_cast<size_t>(B) * heads * Q;     // cross-attention lse per layer (after the last x3)
      RC(ws_train.reserve((per * Lr + RC_ + nlse * Lr) * 4));
      float* p0 = static_cast<float*>(ws_train.ptr);
      for (int i = 0; i < Lr; ++i) {
        float* b = p0 + per * i;
        LayerBufs& L = saved[i];
        L.x0 = b; L.x1 = b + RC_; L.x2 = b + 2 * RC_; L.n1 = b + 3 * RC_; L.n2 = b + 4 * RC_; L.n3 = b + 5 * RC_;
        L.qkv = b + 6 * RC_; L.o1 = b + 9 * RC_; L.qc = b + 10 * RC_; L.o2 = b + 11 * RC_; L.f = b + 12 * RC_;
        L.x3 = (i + 1 < Lr) ? p0 + per * (i + 1) : p0 + per * Lr;  // = x0 of the next layer
        L.lse = p0 + per * Lr + RC_ + nlse * i;
      }
      tgt = saved[0].x0;
      saved_B = B;
      saved_T = T;
    }
  }
  // dropout sites of TransformerDecoderLayer.forward_pre in training mode (tfm_decoder.py:372-386,431-459): site =
  // layer * 8 + {0 self-attention probabilities, 1 dropout1, 2 cross-attention probabilities, 3 dropout2, 4 FFN inner
  // dropout, 5 dropout3}.  Only the training forward drops; backward() regenerates the masks from saved_drop.
  const DropCfg dr = save ? next_drop : drop_off();
  if (save) saved_drop = dr;

  // proj (no bias, :200) -> pre_norm (:86) ; memory and memory+pos in bf16 for the K/V GEMMs
  if (direct) {
    PROF(K_DEC_GEMM, gemm_bf16_rowseg(static_cast<const bf16*>(features), static_cast<int>(stride_row), S, static_cast<int>(pitch),
                                      static_cast<const bf16*>(w_proj.ptr), F, memf, C, nullptr, static_cast<int>(BS), C, F,
                                      EPI_BIAS_F32, s));
  } else {
    if (feat_bf16)
      PROF(K_DEC_GEMM, cast_rows_bf16(static_cast<const bf16*>(features), stride_b, stride_row, S, feat, static_cast<int>(BS), F, s));
    else
      PROF(K_DEC_GEMM, cast_rows_bf16(static_cast<const float*>(features), stride_b, stride_row, S, feat, static_cast<int>(BS), F, s));
    PROF(K_DEC_GEMM, gemm_bf16(feat, F, static_cast<const bf16*>(w_proj.ptr), F, memf, C, nullptr, nullptr, 0, static_cast<int>(BS), C,
                               F, EPI_BIAS_F32, s));
  }
  LnArgs ln{};
  ln.x = memf; ln.ldx = C;
  ln.w = weights.get("transformer.pre_norm.weight"); ln.b = weights.get("transformer.pre_norm.bias"); ln.eps = 1e-5f;
  ln.out_bf16 = mem;
  ln.post_add = static_cast<const float*>(pos3d.ptr); ln.post_mod = S; ln.out2_bf16 = mempos;
  ln.M = static_cast<int>(BS); ln.D = C;
  PROF(K_DEC_GEMM, layernorm_rows(ln, s));
  PROF(K_DEC_GEMM, gemm_bf16(mempos, C, static_cast<const bf16*>(w_kall.ptr), C, Kall, Lr * C, static_cast<const float*>(b_kall.ptr),
               nullptr, 0, static_cast<int>(BS), Lr * C, C, EPI_BIAS_BF16, s));
  PROF(K_DEC_GEMM, gemm_bf16(mem, C, static_cast<const bf16*>(w_vall.ptr), C, Vall, Lr * C, static_cast<const float*>(b_vall.ptr), nullptr,
               0, static_cast<int>(BS), Lr * C, C, EPI_BIAS_BF16, s));
  HH_CHECK_CUDA(cudaMemsetAsync(tgt, 0, static_cast<size_t>(R) * C * 4, s));  // tgt = zeros (:84)
  launches += direct ? 5 : 6;

  auto lnq = [&](const float* x, const std::string& nm, float* out) {
    LnArgs a{};
    a.x = x; a.ldx = C; a.w = weights.get(nm + ".weight"); a.b = weights.get(nm + ".bias"); a.eps = 1e-5f;
    a.out_f32 = out; a.M = R; a.D = C;
    return layernorm_rows(a, s);
  };
  for (int i = 0; i < Lr; ++i) {
    const std::string p = "transformer.decoder.layers." + std::to_string(i) + ".";
    const float* wsa = static_cast<const float*>(w_sa.ptr) + static_cast<size_t>(i) * 3 * C * C;
    const float* bsa = static_cast<const float*>(b_sa.ptr) + static_cast<size_t>(i) * 3 * C;
    const LayerBufs& A = saved[i];
    // self attention over the queries (:431-435)
    PROF(K_DEC_QUERY, lnq(A.x0, p + "norm1", A.n1));
    PROF(K_DEC_QUERY, lin(A.n1, C, qpos, Q, wsa, bsa, nullptr, 0, A.qkv, 3 * C, R, 2 * C, C, 0, s));                   // q,k <- n1+qpos
    PROF(K_DEC_QUERY, lin(A.n1, C, nullptr, 0, wsa + static_cast<size_t>(2) * C * C, bsa + 2 * C, nullptr, 0, A.qkv + 2 * C, 3 * C, R, C, C, 0, s));
    PROF(K_DEC_QUERY, self_attn_queries(A.qkv, A.qkv + C, A.qkv + 2 * C, 3 * C, A.o1, B, Q, heads, s, dr, i * 8 + 0));
    PROF(K_DEC_QUERY, lin(A.o1, C, nullptr, 0, weights.get(p + "self_attn.out_proj.weight"), weights.get(p + "self_attn.out_proj.bias"), A.x0, C,
           A.x1, C, R, C, C, 0, s, dr, i * 8 + 1));
    // cross attention to the patch tokens (:436-441,456)
    PROF(K_DEC_QUERY, lnq(A.x1, p + "norm2", A.n2));
    PROF(K_DEC_QUERY, lin(A.n2, C, qpos, Q, static_cast<const float*>(w_caq.ptr) + static_cast<size_t>(i) * C * C,
           static_cast<const float*>(b_caq.ptr) + static_cast<size_t>(i) * C, nullptr, 0, A.qc, C, R, C, C, 0, s));
    PROF(K_DEC_CROSS, cross_attn(A.qc, Kall + static_cast<size_t>(i) * C, Vall + static_cast<size_t>(i) * C, Lr * C, A.o2, B, Q, heads, S,
                  ws_cross.ptr, s, dr, i * 8 + 2, A.lse));
    PROF(K_DEC_QUERY, lin(A.o2, C, nullptr, 0, weights.get(p + "multihead_attn.out_proj.weight"), weights.get(p + "multihead_attn.out_proj.bias"),
           A.x1, C, A.x2, C, R, C, C, 0, s, dr, i * 8 + 3));
    // FFN (:457-459)
    PROF(K_DEC_QUERY, lnq(A.x2, p + "norm3", A.n3));
    PROF(K_DEC_QUERY, lin(A.n3, C, nullptr, 0, weights.get(p + "linear1.weight"), weights.get(p + "linear1.bias"), nullptr, 0, A.f, Fd, R, Fd, C,
           1, s, dr, i * 8 + 4));
    PROF(K_DEC_QUERY, lin(A.f, Fd, nullptr, 0, weights.get(p + "linear2.weight"), weights.get(p + "linear2.bias"), A.x2, C, A.x3, C, R, C, Fd, 0,
           s, dr, i * 8 + 5));
    // intermediate output through the shared final norm (:282,287-291)
    PROF(K_DEC_QUERY, lnq(A.x3, "transformer.decoder.norm", hs + static_cast<size_t>(i) * R * C));
    launches += 15;
  }

  // ---- heads
  uint8_t* hp = static_cast<uint8_t*>(ws_head.ptr);
  bf16* hs16 = reinterpret_cast<bf16*>(hp);
  hp += LR * C * 2;
  float* hsproj = reinterpret_cast<float*>(hp);
  hp += LR * C * 4;
  const size_t rows_box = LR * (traj ? T : 1);
  float* cond = reinterpret_cast<float*>(hp);
  hp += rows_box * C * 4;
  float* x1 = reinterpret_cast<float*>(hp);
  hp += rows_box * C * 4;
  float* x2 = reinterpret_cast<float*>(hp);
  hp += rows_box * C * 4;
  float* logits_raw = traj ? reinterpret_cast<float*>(hp) : logits;
  sv_cond = cond; sv_x1 = x1; sv_x2 = x2; sv_hsproj = hsproj;

  PROF(K_DEC_HEADS, f32_to_bf16(hs, hs16, LR * C, s));
  PROF(K_DEC_HEADS, gemm_bf16(hs16, C, static_cast<const bf16*>(w_cls.ptr), C, logits_raw, ncls, weights.get("class_embed.bias"), nullptr, 0,
               static_cast<int>(LR), ncls, C, EPI_BIAS_F32, s));  // class_embed (:208)
  launches += 2;
  const float* box_in = hs;
  if (traj) {
    PROF(K_DEC_HEADS, expand_logits(logits_raw, logits, Lr * B, 4, static_cast<size_t>(Q) * ncls, s));  // literal 4 (:216)
    PROF(K_DEC_HEADS, lin(hs, C, nullptr, 0, static_cast<const float*>(w_f1.ptr), nullptr, nullptr, 0, hsproj, C, static_cast<int>(LR), C, C, 0, s));
    PROF(K_DEC_HEADS, add_frame_term(hsproj, static_cast<const float*>(frameterm.ptr), cond, Lr * B, T, Q, C, s));
    box_in = cond;
    launches += 3;
  }
  // bbox_embed: 3-layer MLP + sigmoid (:228)
  PROF(K_DEC_HEADS, lin(box_in, C, nullptr, 0, weights.get("bbox_embed.layers.0.weight"), weights.get("bbox_embed.layers.0.bias"), nullptr, 0, x1,
         C, static_cast<int>(rows_box), C, C, 1, s));
  PROF(K_DEC_HEADS, lin(x1, C, nullptr, 0, weights.get("bbox_embed.layers.1.weight"), weights.get("bbox_embed.layers.1.bias"), nullptr, 0, x2, C,
         static_cast<int>(rows_box), C, C, 1, s));
  PROF(K_DEC_HEADS, lin(x2, C, nullptr, 0, weights.get("bbox_embed.layers.2.weight"), weights.get("bbox_embed.layers.2.bias"), nullptr, 0, boxes,
         4, static_cast<int>(rows_box), 4, C, 2, s));
  launches += 3;
  return 0;
}

double Decoder::flops_per_clip(int T) const {
  // SURVEY.md section 8(d): F_dec
  const double C = cfg.d_model, S = static_cast<double>(T) * cfg.patches_per_frame, Q = cfg.num_queries, F = cfg.feature_dim;
  const double Lr = cfg.num_layers, ffn = cfg.dim_feedforward, ncls = cfg.num_classes1;
  const bool traj = cfg.pred_traj && T == cfg.num_frames;
  const double Rr = Lr * Q * (traj ? T : 1);
  double fl = 2 * S * F * C + Lr * (4 * S * C * C + 4 * Q * S * C + (12 * Q * C * C + 4 * Q * Q * C) + 4 * Q * C * ffn) +
              Lr * 2 * Q * C * ncls + Rr * 2 * (2 * C * C + 4 * C) + 2 * Q * (C * C + 256 * C);
  if (traj) fl += Rr * 2 * 2 * C * C;
  return fl;
}

}  // namespace hh
