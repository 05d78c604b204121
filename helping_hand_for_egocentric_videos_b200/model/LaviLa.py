"""Drop-in mirror of the reference's ``model/LaviLa.py`` whose video tower runs on libhh_b200.so.

Same class names, constructor keywords, ``forward`` signatures, attribute names and ``state_dict`` keys as the
reference (SURVEY.md section 8b), so ``run/test_EgoMCQ.py`` / ``run/train.py`` / ``run/test_epic.py`` can import this
module in place of the reference's:

    from model.LaviLa import CLIP_OPENAI_TIMESFORMER_LARGE        # reference
    from helping_hand_for_egocentric_videos_b200.model.LaviLa import CLIP_OPENAI_TIMESFORMER_LARGE   # this repo

The nn.Module tree below only *holds parameters* (so load_state_dict / .to() / named_parameters() behave); the video
forward (SpaceTimeTransformer.forward_features, reference model/LaviLa.py:537-573) is one call into the C ABI
(hh_encoder_forward).  There is no PyTorch fallback for it.  The CLIP text tower (reference :660-670; SURVEY.md
section 8f, row 1) is likewise one call (hh_text_forward) over parameter containers with reference-identical keys.
"""
from __future__ import annotations

import ctypes as C
import os
from collections import OrderedDict
from functools import partial

import numpy as np
import torch
import torch.nn as nn

from .. import _lib as L
from .. import ops
from ..utils.checkpoint import remap_keys  # noqa: F401  (reference model/LaviLa.py:19-53 lives in this module)


class QuickGELU(nn.Module):
    """x * sigmoid(1.702 x) (reference model/openai_model.py:177-179).  Marker class: the encoder kernels fuse it."""

    def forward(self, x):
        return x * torch.sigmoid(1.702 * x)


# ---------------------------------------------------------------------------------------------- parameter containers
class Mlp(nn.Module):
    def __init__(self, in_features, hidden_features=None, out_features=None, act_layer=QuickGELU, drop=0.):
        super().__init__()
        self.fc1 = nn.Linear(in_features, hidden_features or in_features)
        self.act = act_layer()
        self.fc2 = nn.Linear(hidden_features or in_features, out_features or in_features)


class VideoPatchEmbed(nn.Module):
    def __init__(self, img_size=224, patch_size=16, in_chans=3, embed_dim=768, num_frames=8, ln_pre=False):
        super().__init__()
        self.img_size = (img_size, img_size)
        self.patch_size = (patch_size, patch_size)
        self.num_patches = (img_size // patch_size) ** 2 * num_frames
        self.num_frames = num_frames
        self.embed_dim = embed_dim
        self.proj = nn.Conv2d(in_chans, embed_dim, kernel_size=patch_size, stride=patch_size, bias=not ln_pre)


class VarAttention(nn.Module):
    def __init__(self, dim, num_heads=8, qkv_bias=False, qk_scale=None, attn_drop=0., proj_drop=0., initialize='random'):
        super().__init__()
        self.num_heads = num_heads
        self.scale = qk_scale or (dim // num_heads) ** -0.5
        self.qkv = nn.Linear(dim, dim * 3, bias=qkv_bias)
        self.proj = nn.Linear(dim, dim)
        if initialize == 'zeros':     # reference :236-242
            self.qkv.weight.data.fill_(0)
            self.qkv.bias.data.fill_(0)
            self.proj.weight.data.fill_(1)
            self.proj.bias.data.fill_(0)


class SpaceTimeBlock(nn.Module):
    def __init__(self, dim, num_heads, mlp_ratio=4., qkv_bias=False, qk_scale=None, n_layer=0, drop=0., attn_drop=0.,
                 drop_path=0., act_layer=QuickGELU, norm_layer=nn.LayerNorm, time_init='zeros',
                 attention_style='frozen-in-time', is_tanh_gating=False, use_adapter=False):
        super().__init__()
        self.norm1 = norm_layer(dim)
        self.attn = VarAttention(dim, num_heads=num_heads, qkv_bias=qkv_bias, qk_scale=qk_scale)
        self.timeattn = VarAttention(dim, num_heads=num_heads, qkv_bias=qkv_bias, qk_scale=qk_scale, initialize=time_init)
        self.norm2 = norm_layer(dim)
        self.mlp = Mlp(in_features=dim, hidden_features=int(dim * mlp_ratio), act_layer=act_layer, drop=drop)
        self.norm3 = norm_layer(dim)
        self.attention_style = attention_style
        self.use_adapter = False


class _ParamSync:
    """Pushes nn.Parameters into the C engine when (and only when) they changed: a tensor is re-sent if its storage
    pointer or its in-place version counter differs from what was last uploaded (load_state_dict, .to(),
    inflate_positional_embeds, optimizer steps all trip one of the two).

    Writes through ``param.data`` (``p.data.copy_(...)``, the pattern of reference model/LaviLa.py:164-170, EMA updates,
    ``clamp_`` via .data) do NOT bump the version counter: call ``module.mark_dirty()`` after them.  load_state_dict and
    every ``_apply`` (.to / .cuda / .float) mark the module dirty by themselves.  HH_PARAM_CHECKSUM=1 additionally
    compares a per-tensor checksum on every sync (debug aid: one small reduction per parameter per forward)."""

    def __init__(self):
        self.seen = {}
        self.checks = {}
        self.debug = bool(int(os.environ.get("HH_PARAM_CHECKSUM", "0") or 0))

    def clear(self):
        self.seen.clear()
        self.checks.clear()

    def sync(self, named, setter, batch_setter=None):
        """`setter(key, tensor)` per changed parameter, or `batch_setter([(key, tensor), ...])` once for all of them."""
        batch = []
        for key, t in named:
            tag = (t.data_ptr(), t._version, t.dtype)
            if self.seen.get(key) == tag:
                if not self.debug:
                    continue
                chk = float(t.detach().double().sum().item())
                if self.checks.get(key) == chk:
                    continue
            src = t.detach()
            if src.dtype != torch.float32 or not src.is_contiguous():
                src = src.float().contiguous()
            if batch_setter is not None:
                batch.append((key, src))
            else:
                setter(key, src)
            self.seen[key] = tag
            if self.debug:
                self.checks[key] = float(t.detach().double().sum().item())
        if batch:
            batch_setter(batch)


class _DirtyHooks:
    """Mixin for the engine-backed modules: everything that can rewrite parameters behind the version counters'
    back marks the uploaded copies stale."""

    def _sync_states(self):
        return [v for k, v in vars(self).items() if isinstance(v, _ParamSync)]

    def mark_dirty(self):
        """Force a re-upload of every parameter on the next forward (needed after writes through ``.data``)."""
        for st in self._sync_states():
            st.clear()
        for m in self.children():
            if isinstance(m, _DirtyHooks):
                m.mark_dirty()
        return self

    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)
        self.mark_dirty()
        return out

    def load_state_dict(self, *args, **kwargs):
        out = super().load_state_dict(*args, **kwargs)
        self.mark_dirty()
        return out


class SpaceTimeTransformer(_DirtyHooks, nn.Module):
    """Divided space-time ViT, reference model/LaviLa.py:393-581 (only the LaViLa configuration is implemented:
    ``ln_pre=True``, QuickGELU MLP, 'frozen-in-time' residual wiring, qkv_bias=True, no dropout / drop-path)."""

    def __init__(self, img_size=224, patch_size=16, in_chans=3, num_classes=1000, embed_dim=768, depth=12,
                 num_heads=12, mlp_ratio=4., qkv_bias=True, qk_scale=None, representation_size=None,
                 drop_rate=0., attn_drop_rate=0., drop_path_rate=0., hybrid_backbone=None, norm_layer=None,
                 num_frames=8, time_init='rand', attention_style='frozen-in-time', ln_pre=False,
                 act_layer=nn.GELU, is_tanh_gating=False, use_adapter=False):
        super().__init__()
        if not ln_pre or act_layer is not QuickGELU or attention_style != 'frozen-in-time' or not qkv_bias \
                or is_tanh_gating or use_adapter or hybrid_backbone is not None or in_chans != 3 \
                or drop_rate or attn_drop_rate or drop_path_rate or qk_scale is not None or representation_size:
            raise NotImplementedError(
                "helping_hand_for_egocentric_videos_b200 implements the LaViLa TimeSformer configuration only "
                "(ln_pre=True, act_layer=QuickGELU, 'frozen-in-time', qkv_bias=True, no gating/adapter/dropout)")
        self.num_classes = num_classes
        self.num_features = self.embed_dim = embed_dim
        self.num_frames = num_frames
        norm_layer = norm_layer or partial(nn.LayerNorm, eps=1e-6)
        self.patch_embed = VideoPatchEmbed(img_size=img_size, patch_size=patch_size, in_chans=in_chans,
                                           embed_dim=embed_dim, num_frames=num_frames, ln_pre=ln_pre)
        self.patches_per_frame = self.patch_embed.num_patches // num_frames
        self.cls_token = nn.Parameter(torch.zeros(1, 1, embed_dim))
        self.pos_embed = nn.Parameter(torch.zeros(1, self.patches_per_frame + 1, embed_dim))
        self.temporal_embed = nn.Parameter(torch.zeros(1, num_frames, embed_dim))
        self.ln_pre = nn.LayerNorm(embed_dim)
        self.blocks = nn.ModuleList([
            SpaceTimeBlock(dim=embed_dim, num_heads=num_heads, mlp_ratio=mlp_ratio, qkv_bias=qkv_bias, n_layer=i,
                           norm_layer=norm_layer, time_init=time_init, attention_style=attention_style,
                           act_layer=act_layer) for i in range(depth)])
        self.norm = norm_layer(embed_dim)
        self.pre_logits = nn.Identity()
        self.head = nn.Linear(self.num_features, num_classes) if num_classes > 0 else nn.Identity()
        nn.init.trunc_normal_(self.pos_embed, std=.02)
        nn.init.trunc_normal_(self.cls_token, std=.02)
        self._cfg = L.EncoderCfg(img_size, patch_size, num_frames, embed_dim, depth, num_heads, int(embed_dim * mlp_ratio))
        self._handle = None
        self._sync = _ParamSync()
        self.feature_map_dtype = torch.float32

    @property
    def feature_map_dtype(self):
        """dtype of the feature map forward_features returns: torch.float32 (default) or torch.bfloat16.  The bf16 map
        is the fp32 one rounded to nearest-even at half the bytes; x_cls stays fp32 and bit-identical, and ObjDecoder
        gives the same outputs on either map (it rounds its input to bf16 itself)."""
        return self._feature_map_dtype

    @feature_map_dtype.setter
    def feature_map_dtype(self, dtype):
        if dtype not in (torch.float32, torch.bfloat16):
            raise ValueError("feature_map_dtype must be torch.float32 or torch.bfloat16, got %r" % (dtype,))
        self._feature_map_dtype = dtype

    # -- engine plumbing ---------------------------------------------------------------------------------------
    def _engine(self):
        if self._handle is None:
            h = C.c_void_p()
            L.check(L.load().hh_encoder_create(C.byref(h), C.byref(self._cfg)), "hh_encoder_create")
            self._handle = h
        return self._handle

    def __del__(self):
        h = getattr(self, "_handle", None)
        if h is not None and L._lib is not None:
            L._lib.hh_encoder_destroy(h)
            self._handle = None

    def _engine_params(self):
        skip = ("head.", "pre_logits.", "fc.")
        for k, p in self.named_parameters():
            if not k.startswith(skip):
                yield k, p

    def sync_weights(self):
        h, lib = self._engine(), L.load()
        # the temporal embedding may have been inflated (run/test_egtea.py:46-96): the engine is rebuilt for the new T
        T = self.temporal_embed.shape[1]
        if T != self._cfg.num_frames:
            lib.hh_encoder_destroy(h)
            self._handle = None
            self._cfg.num_frames = T
            self.num_frames = T
            self._sync = _ParamSync()
            h = self._engine()

        def setter(key, src):
            L.check(lib.hh_encoder_set_weight(h, key.encode(), L.ptr(src), src.numel(), L.stream_ptr()),
                    "hh_encoder_set_weight(%s)" % key)
        self._sync.sync(self._engine_params(), setter)

    def flops_per_clip(self) -> float:
        return L.load().hh_encoder_flops_per_clip(self._engine())

    def last_launches(self) -> int:
        return L.load().hh_encoder_last_launches(self._engine())

    def set_profile(self, on: bool):
        """Record CUDA events around every kernel launch of the engine (see profile())."""
        L.check(L.load().hh_encoder_set_profile(self._engine(), 1 if on else 0), "hh_encoder_set_profile")

    def profile(self):
        """{kernel class: (milliseconds, launches)} since the last call; waits for the recorded events."""
        lib = L.load()
        k = lib.hh_profile_num_classes()
        ms, cnt = (C.c_double * k)(), (C.c_int * k)()
        L.check(lib.hh_encoder_profile(self._engine(), ms, cnt), "hh_encoder_profile")
        return {lib.hh_profile_class_name(i).decode(): (ms[i], cnt[i]) for i in range(k) if cnt[i]}

    # -- reference API -----------------------------------------------------------------------------------------
    @torch.jit.ignore
    def no_weight_decay(self):
        return {'pos_embed', 'cls_token'}

    def freeze_spatial_weights(self):
        for n, p in self.named_parameters():
            if not ('temporal_embed' in n or 'timeattn' in n or 'norm3' in n):
                p.requires_grad = False

    def freeze_temporal_weights(self):
        for n, p in self.named_parameters():
            if 'temporal_embed' in n or 'timeattn' in n or 'norm3' in n:
                p.requires_grad = False

    @torch.no_grad()
    def forward_features(self, x, use_checkpoint=False, cls_at_last=True, _nblocks=-1):
        """x [B,T,3,H,W] -> (x_cls [B,D], fmap [B,1+T*n,D]); the tower is frozen in every reference script
        (run/train.py:109 runs it under no_grad), so no autograd graph is recorded.  fmap has feature_map_dtype
        (x_cls is fp32 either way); the `_nblocks` test hook always returns fp32."""
        if not x.is_cuda:
            raise RuntimeError("SpaceTimeTransformer (B200): input is on %s; there is no CPU fallback" % x.device)
        b, t, c, hh, ww = x.shape
        if t != self.temporal_embed.shape[1]:
            raise RuntimeError("got %d frames, model built for %d (reference LaviLa.py:549-553 needs them equal)"
                               % (t, self.temporal_embed.shape[1]))
        if c != 3 or hh != self._cfg.img_size or ww != self._cfg.img_size:
            raise RuntimeError("expected [B,T,3,%d,%d] clips, got %s" % (self._cfg.img_size, self._cfg.img_size,
                                                                         tuple(x.shape)))
        self.sync_weights()
        x = x.float().contiguous()
        n_tok = 1 + t * self.patches_per_frame
        if self.feature_map_dtype == torch.bfloat16 and _nblocks == -1:     # the truncated-forward hook stays fp32
            fmap = torch.empty(b, n_tok, self.embed_dim, dtype=torch.bfloat16, device=x.device)
            cls = torch.empty(b, self.embed_dim, dtype=torch.float32, device=x.device)
            L.check(L.load().hh_encoder_forward_bf16(self._engine(), L.ptr(x), b, L.ptr(fmap), L.ptr(cls), L.stream_ptr()),
                    "hh_encoder_forward_bf16")
            return self.pre_logits(cls), fmap
        fmap = torch.empty(b, n_tok, self.embed_dim, dtype=torch.float32, device=x.device)
        L.check(L.load().hh_encoder_forward_n(self._engine(), L.ptr(x), b, _nblocks, L.ptr(fmap), L.stream_ptr()),
                "hh_encoder_forward")
        x_cls = self.pre_logits(fmap[:, 0])
        return x_cls, fmap

    @torch.no_grad()
    def forward_features_u8(self, frames, norm_mean, norm_std):
        """Raw decoder output uint8 [B,T,H,W,3] -> (x_cls, fmap), with the loader tail of the reference
        (frames.float()/255, permute, NormalizeVideo(mean, std): base/base_dataset.py:322-323,
        data_loader/transforms.py:48-51) fused into the patch loader.  Bit-identical to
        forward_features(((frames.float() / 255).permute(0, 1, 4, 2, 3) - mean) / std)."""
        if not frames.is_cuda:
            raise RuntimeError("SpaceTimeTransformer (B200): input is on %s; there is no CPU fallback" % frames.device)
        if frames.dtype != torch.uint8:
            raise TypeError("forward_features_u8 expects uint8 frames, got %s" % frames.dtype)
        b, t, hh, ww, c = frames.shape
        if t != self.temporal_embed.shape[1]:
            raise RuntimeError("got %d frames, model built for %d" % (t, self.temporal_embed.shape[1]))
        if c != 3 or hh != self._cfg.img_size or ww != self._cfg.img_size:
            raise RuntimeError("expected [B,T,%d,%d,3] frames, got %s" % (self._cfg.img_size, self._cfg.img_size,
                                                                         tuple(frames.shape)))
        self.sync_weights()
        frames = frames.contiguous()
        mean = (C.c_float * 3)(*[float(v) for v in norm_mean])
        std = (C.c_float * 3)(*[float(v) for v in norm_std])
        n_tok = 1 + t * self.patches_per_frame
        if self.feature_map_dtype == torch.bfloat16:
            fmap = torch.empty(b, n_tok, self.embed_dim, dtype=torch.bfloat16, device=frames.device)
            cls = torch.empty(b, self.embed_dim, dtype=torch.float32, device=frames.device)
            L.check(L.load().hh_encoder_forward_u8_bf16(self._engine(), L.ptr(frames), b, mean, std, L.ptr(fmap), L.ptr(cls),
                                                        L.stream_ptr()), "hh_encoder_forward_u8_bf16")
            return self.pre_logits(cls), fmap
        fmap = torch.empty(b, n_tok, self.embed_dim, dtype=torch.float32, device=frames.device)
        L.check(L.load().hh_encoder_forward_u8(self._engine(), L.ptr(frames), b, mean, std, L.ptr(fmap), L.stream_ptr()),
                "hh_encoder_forward_u8")
        return self.pre_logits(fmap[:, 0]), fmap

    def forward(self, x, use_checkpoint=False):
        x_cls, x = self.forward_features(x, use_checkpoint=use_checkpoint)
        return self.head(x_cls), x


# ---------------------------------------------------------------------------------------------- text tower
class ResidualAttentionBlock(nn.Module):
    """Parameter container with the keys of reference model/openai_model.py:182-216 (attn.in_proj_weight, ln_1, mlp.c_fc,
    ...).  The arithmetic runs in the C engine (CLIP.encode_text)."""

    def __init__(self, d_model: int, n_head: int, attn_mask: torch.Tensor = None):
        super().__init__()
        self.attn = nn.MultiheadAttention(d_model, n_head)
        self.ln_1 = nn.LayerNorm(d_model)
        self.mlp = nn.Sequential(OrderedDict([("c_fc", nn.Linear(d_model, d_model * 4)), ("gelu", QuickGELU()),
                                              ("c_proj", nn.Linear(d_model * 4, d_model))]))
        self.ln_2 = nn.LayerNorm(d_model)
        self.attn_mask = attn_mask

    def forward(self, x: torch.Tensor, use_checkpoint=False):
        raise NotImplementedError("the text blocks run inside hh_text_forward; call CLIP.encode_text")


class Transformer(nn.Module):
    def __init__(self, width: int, layers: int, heads: int, attn_mask: torch.Tensor = None):
        super().__init__()
        self.width = width
        self.layers = layers
        self.heads = heads
        self.resblocks = nn.Sequential(*[ResidualAttentionBlock(width, heads, attn_mask) for _ in range(layers)])

    def forward(self, x: torch.Tensor, use_checkpoint=False):
        raise NotImplementedError("the text blocks run inside hh_text_forward; call CLIP.encode_text")


class CLIP(_DirtyHooks, nn.Module):
    """Reference model/LaviLa.py:586-687 (dual encoder wrapper)."""

    def __init__(self, embed_dim: int, vision_width: int, vision_model: nn.Module, context_length: int,
                 vocab_size: int, transformer_width: int, transformer_heads: int, transformer_layers: int,
                 tempearture_init=0.07, **kwargs):
        super().__init__()
        self.context_length = context_length
        self.vision_width = vision_width
        self.visual = vision_model
        self.transformer = Transformer(width=transformer_width, layers=transformer_layers, heads=transformer_heads,
                                       attn_mask=self.build_attention_mask())
        self.vocab_size = vocab_size
        self.token_embedding = nn.Embedding(vocab_size, transformer_width)
        self.positional_embedding = nn.Parameter(torch.empty(self.context_length, transformer_width))
        self.ln_final = nn.LayerNorm(transformer_width)
        self.image_projection = nn.Parameter(torch.empty(vision_width, embed_dim))
        self.text_projection = nn.Parameter(torch.empty(transformer_width, embed_dim))
        self.logit_scale = nn.Parameter(torch.ones([]) * np.log(1 / tempearture_init))
        self.initialize_parameters()
        self._proj_t = None
        self._text_cfg = L.TextCfg(vocab_size=vocab_size, context_length=context_length, width=transformer_width,
                                   heads=transformer_heads, layers=transformer_layers, embed_dim=embed_dim)
        self._text_handle = None
        self._text_sync = _ParamSync()

    def initialize_parameters(self):
        nn.init.normal_(self.token_embedding.weight, std=0.02)
        nn.init.normal_(self.positional_embedding, std=0.01)
        proj_std = (self.transformer.width ** -0.5) * ((2 * self.transformer.layers) ** -0.5)
        attn_std = self.transformer.width ** -0.5
        fc_std = (2 * self.transformer.width) ** -0.5
        for block in self.transformer.resblocks:
            nn.init.normal_(block.attn.in_proj_weight, std=attn_std)
            nn.init.normal_(block.attn.out_proj.weight, std=proj_std)
            nn.init.normal_(block.mlp.c_fc.weight, std=fc_std)
            nn.init.normal_(block.mlp.c_proj.weight, std=proj_std)
        nn.init.normal_(self.image_projection, std=self.vision_width ** -0.5)
        nn.init.normal_(self.text_projection, std=self.transformer.width ** -0.5)

    def build_attention_mask(self):
        mask = torch.empty(self.context_length, self.context_length)
        mask.fill_(float("-inf"))
        mask.triu_(1)
        return mask

    def mark_dirty(self):
        self._proj_t = None
        return super().mark_dirty()

    def _image_projection_t(self):
        p = self.image_projection
        tag = (p.data_ptr(), p._version)
        if self._proj_t is None or self._proj_t[0] != tag:
            self._proj_t = (tag, p.detach().float().t().contiguous())
        return self._proj_t[1]

    def encode_image(self, image, use_checkpoint=False, apply_project=True):
        x_cls, x = self.visual(image, use_checkpoint=use_checkpoint)
        if not apply_project:
            return x_cls, x
        x_cls = ops.linear_f32(x_cls.contiguous(), self._image_projection_t())      # x_cls @ image_projection (:657)
        return x_cls, x

    # -- text engine plumbing ----------------------------------------------------------------------------------
    def _text_engine(self):
        if self._text_handle is None:
            h = C.c_void_p()
            L.check(L.load().hh_text_create(C.byref(h), C.byref(self._text_cfg)), "hh_text_create")
            self._text_handle = h
        return self._text_handle

    def __del__(self):
        h = getattr(self, "_text_handle", None)
        if h is not None and L._lib is not None:
            L._lib.hh_text_destroy(h)
            self._text_handle = None

    def _text_params(self):
        keep = ("transformer.", "token_embedding.", "positional_embedding", "ln_final.", "text_projection")
        for k, p in self.named_parameters():
            if k.startswith(keep):
                yield k, p

    def sync_text_weights(self):
        h, lib = self._text_engine(), L.load()

        def setter(key, src):
            L.check(lib.hh_text_set_weight(h, key.encode(), L.ptr(src), src.numel(), L.stream_ptr()),
                    "hh_text_set_weight(%s)" % key)
        self._text_sync.sync(self._text_params(), setter)

    def text_flops_per_sequence(self) -> float:
        return L.load().hh_text_flops_per_sequence(self._text_engine())

    @torch.no_grad()
    def encode_text(self, text, use_checkpoint=False):
        """text int64 [G, context_length] -> (x_cls [G, embed_dim], x [G, context_length, width]); reference
        model/LaviLa.py:660-670.  The tower is frozen in every reference script (run/train.py:88,109)."""
        if not text.is_cuda:
            raise RuntimeError("helping_hand_for_egocentric_videos_b200: the text tower runs on CUDA only "
                               "(got a %s tensor); there is no CPU fallback" % text.device)
        if text.dim() != 2 or text.shape[1] != self.context_length:
            raise ValueError("text must be [G, %d] token ids, got %s" % (self.context_length, tuple(text.shape)))
        if text.dtype not in (torch.int64, torch.int32):
            raise TypeError("text must hold integer token ids, got %s" % text.dtype)
        with torch.cuda.device(text.device):
            self.sync_text_weights()
            tok = text.to(torch.int64).contiguous()
            G = tok.shape[0]
            x_cls = torch.empty(G, self._text_cfg.embed_dim, device=text.device, dtype=torch.float32)
            x = torch.empty(G, self.context_length, self._text_cfg.width, device=text.device, dtype=torch.float32)
            L.check(L.load().hh_text_forward(self._text_engine(), L.ptr(tok), G, L.ptr(x_cls), L.ptr(x), L.stream_ptr()),
                    "hh_text_forward")
        return x_cls, x

    def forward(self, image, text, use_checkpoint=False, norm_embed=True, return_feature_map=False):
        image_embed, image_fmap = self.encode_image(image, use_checkpoint=use_checkpoint)
        text_embed, text_fmap = self.encode_text(text, use_checkpoint=use_checkpoint)
        if norm_embed:
            image_embed = ops.l2_normalize(image_embed, 1e-12)
            text_embed = ops.l2_normalize(text_embed, 1e-12)
        out = {'image_embed': image_embed, 'text_embed': text_embed, 'logit_scale': self.logit_scale.exp()}
        if return_feature_map:
            out['image_feature_map'] = image_fmap
            out['text_feature_map'] = text_fmap
        return out


def _timesformer_clip(patch_size, embed_dim, depth, num_heads, text_width, text_heads, num_frames, temperature_init,
                      project_embed_dim, timesformer_gated_xattn, drop_path_rate, use_adapter, kwargs):
    if timesformer_gated_xattn or use_adapter or drop_path_rate:
        raise NotImplementedError("gated x-attn / adapters / drop-path are not part of the accelerated path")
    vision_model = SpaceTimeTransformer(
        img_size=224, patch_size=patch_size, embed_dim=embed_dim, depth=depth, num_heads=num_heads,
        num_frames=num_frames, time_init='zeros', attention_style='frozen-in-time', ln_pre=True, act_layer=QuickGELU)
    vision_model.head = nn.Identity()
    vision_model.pre_logits = nn.Identity()
    vision_model.fc = nn.Identity()
    if kwargs.get("timesformer_freeze_space"):
        # reference :74-85 / :135-146: everything the OpenAI-CLIP image tower provides is frozen; the temporal parts
        # (absent from that checkpoint: timeattn.*, norm3.*, temporal_embed) and cls_token stay trainable
        for n, p in vision_model.named_parameters():
            p.requires_grad = ('temporal_embed' in n or 'timeattn' in n or 'norm3' in n or n == 'cls_token')
    kwargs = {k: v for k, v in kwargs.items() if k not in ("pretrained", "text_use_cls_token", "timesformer_freeze_space")}
    return CLIP(embed_dim=project_embed_dim, vision_width=embed_dim, vision_model=vision_model, context_length=77,
                vocab_size=49408, transformer_width=text_width, transformer_heads=text_heads, transformer_layers=12,
                tempearture_init=temperature_init, **kwargs)


def CLIP_OPENAI_TIMESFORMER_BASE(num_frames=4, timesformer_gated_xattn=False, drop_path_rate=0,
                                 timesformer_freeze_space=False, temperature_init=0.07, project_embed_dim=256,
                                 use_adapter=False, **kwargs):
    """Reference model/LaviLa.py:55-111 without the OpenAI-CLIP download (:69): weights start random and are expected
    to be overwritten by a LaViLa checkpoint, exactly as run/test_EgoMCQ.py:221-227 does."""
    kwargs["timesformer_freeze_space"] = timesformer_freeze_space
    return _timesformer_clip(16, 768, 12, 12, 512, 8, num_frames, temperature_init, project_embed_dim,
                             timesformer_gated_xattn, drop_path_rate, use_adapter, kwargs)


def CLIP_OPENAI_TIMESFORMER_LARGE(num_frames=4, timesformer_gated_xattn=False, drop_path_rate=0,
                                  timesformer_freeze_space=False, temperature_init=0.07, project_embed_dim=256,
                                  use_adapter=False, **kwargs):
    """Reference model/LaviLa.py:114-172 without the network access (:130)."""
    kwargs["timesformer_freeze_space"] = timesformer_freeze_space
    return _timesformer_clip(14, 1024, 24, 16, 768, 12, num_frames, temperature_init, project_embed_dim,
                             timesformer_gated_xattn, drop_path_rate, use_adapter, kwargs)
