"""Drop-in mirror of the reference's ``model/tfm_decoder.py`` (object-aware decoder) running on libhh_b200.so.

``Cross_Attention`` / ``ObjDecoder`` keep the reference's constructor keywords, attributes (``.txt_proj``,
``.obj_proj``, ``.transformer`` ...), ``state_dict`` keys and return values:

    out, hs, attn, self_attn = model(video_grid)        # run/test_EgoMCQ.py:73 ; attn == self_attn == []

The module tree holds parameters; ``ObjDecoder.forward`` (reference :183-233) is one C-ABI call (hh_decoder_forward)
and the small projection heads are hh_linear_f32 calls.  In ``train()`` mode the reference's dropout (nn.Dropout x4
per layer and the attention-probability dropout of both nn.MultiheadAttention modules, p = ``dropout``) is applied by
the engine's training forward with counter-based masks (hh_decoder_set_dropout); ``eval()`` is the inference arithmetic.
"""
from __future__ import annotations

import copy
import ctypes as C
import math
import warnings

import torch
import torch.nn as nn

from .. import _lib as L
from .. import ops
from .LaviLa import _DirtyHooks, _ParamSync


class _LinearFn(torch.autograd.Function):
    """y = act(relu?(x) W^T + b) on hh_linear_f32 with the backward kernels of hh_linear_f32_backward."""

    @staticmethod
    def forward(ctx, x, weight, bias, act, in_relu):
        shp = x.shape
        x2 = x.reshape(-1, shp[-1])
        x2 = x2 if (x2.dtype == torch.float32 and x2.is_contiguous()) else x2.float().contiguous()
        y = ops.linear_f32(x2, weight.detach(), bias.detach() if bias is not None else None, act=act, in_relu=in_relu)
        ctx.save_for_backward(x2, weight, y)
        ctx.act, ctx.in_relu, ctx.shape, ctx.has_bias = act, in_relu, shp, bias is not None
        return y.reshape(*shp[:-1], weight.shape[0])

    @staticmethod
    def backward(ctx, dy):
        x2, weight, y = ctx.saved_tensors
        need_dx = ctx.needs_input_grad[0]
        if need_dx and ctx.in_relu:
            raise NotImplementedError("gradient through a leading ReLU of a native head is not implemented "
                                      "(txt_proj's input comes from the frozen text tower)")
        dy2 = dy.reshape(-1, weight.shape[0]).float().contiguous()
        dx, dw, db = ops.linear_f32_backward(dy2, y, ctx.act, weight.detach().float().contiguous(), x2, None, ctx.in_relu,
                                             need_dx=need_dx, need_dw=ctx.needs_input_grad[1])
        return (dx.reshape(ctx.shape) if need_dx else None, dw, db if ctx.has_bias else None, None, None)


class _NativeHead(nn.Sequential):
    """nn.Sequential of Linear / ReLU layers (same child indices => same state_dict keys as the reference's
    nn.Sequential heads, tfm_decoder.py:168-180) evaluated with hh_linear_f32, ReLUs fused into the linears.  With
    autograd enabled and trainable parameters, every linear records its hand-written backward."""

    def forward(self, x):
        track = torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.parameters()))
        mods = list(self)
        pending_relu = False
        i = 0
        while i < len(mods):
            m = mods[i]
            if isinstance(m, nn.ReLU):
                pending_relu = True
                i += 1
                continue
            assert isinstance(m, nn.Linear)
            fuse_out = i + 1 < len(mods) and isinstance(mods[i + 1], nn.ReLU)
            if track:
                x = _LinearFn.apply(x, m.weight, m.bias, 1 if fuse_out else 0, pending_relu)
            else:
                with torch.no_grad():
                    x = ops.linear_f32(x, m.weight.detach(), m.bias.detach() if m.bias is not None else None,
                                       act=1 if fuse_out else 0, in_relu=pending_relu)
            pending_relu = False
            i += 2 if fuse_out else 1
        if pending_relu:
            x = torch.relu(x)
        return x


class _DecoderFn(torch.autograd.Function):
    """ObjDecoder forward + hand-written backward (hh_decoder_forward_train / hh_decoder_backward).  The parameters are
    passed as inputs only so that autograd routes their gradients; the arithmetic reads the engine's packed copies."""

    @staticmethod
    def forward(ctx, module, features, *params):
        hs, logits, boxes = module._run_engine(features, train=True)
        # the engine holds one activation set: stamp this graph with the forward's ordinal so that a backward issued
        # after ANOTHER forward of the same module (two clips then a summed backward, ...) fails instead of silently
        # differentiating the wrong activations / dropout masks
        ctx.generation = L.load().hh_decoder_generation(module._engine())
        ctx.module = module
        ctx.keys = [k for k, _ in module._engine_params()]
        ctx.shapes = [tuple(p.shape) for p in params]
        ctx.save_for_backward(hs, boxes)
        ctx.mark_non_differentiable(logits)
        return hs, logits, boxes

    @staticmethod
    def backward(ctx, d_hs, d_logits, d_boxes):
        hs, boxes = ctx.saved_tensors
        m = ctx.module
        lib = L.load()

        def prep(g):
            return None if g is None else (g if (g.dtype == torch.float32 and g.is_contiguous()) else g.float().contiguous())
        d_hs, d_boxes = prep(d_hs), prep(d_boxes)
        L.check(lib.hh_decoder_backward_checked(m._engine(), ctx.generation, L.ptr(hs), L.ptr(boxes), L.ptr(d_hs),
                                                L.ptr(d_boxes), L.stream_ptr()), "hh_decoder_backward")
        # one packed read of every requested gradient (135 keys at the c4 step: per-key calls and allocations made this
        # function host-bound); the returned gradients are views of the one flat tensor
        needs = tuple(bool(n) for n in ctx.needs_input_grad[2:])
        want = [(k, shp) for k, shp, need in zip(ctx.keys, ctx.shapes, needs) if need]
        grads = [None] * len(ctx.keys)
        if want:
            cache = getattr(m, "_grad_pack", None)
            if cache is None or cache[0] != (needs, tuple(ctx.keys), tuple(ctx.shapes)):
                numels = [int(math.prod(shp)) for _, shp in want]
                keys_c = (C.c_char_p * len(want))(*[k.encode() for k, _ in want])
                numels_c = (C.c_int64 * len(want))(*numels)
                cache = ((needs, tuple(ctx.keys), tuple(ctx.shapes)), keys_c, numels_c, numels, sum(numels))
                m._grad_pack = cache
            _, keys_c, numels_c, numels, total = cache
            flat = torch.empty(total, dtype=torch.float32, device=hs.device)
            L.check(lib.hh_decoder_get_grads(m._engine(), keys_c, numels_c, len(want), L.ptr(flat), total, L.stream_ptr()),
                    "hh_decoder_get_grads")
            pieces = iter(flat.split(numels))
            for i, (need, shp) in enumerate(zip(needs, ctx.shapes)):
                if need:
                    grads[i] = next(pieces).view(shp)
        return (None, None, *grads)


class MLP(nn.Module):
    """Parameter container for bbox_embed (reference :96-108)."""

    def __init__(self, input_dim, hidden_dim, output_dim, num_layers):
        super().__init__()
        self.num_layers = num_layers
        h = [hidden_dim] * (num_layers - 1)
        self.layers = nn.ModuleList(nn.Linear(n, k) for n, k in zip([input_dim] + h, h + [output_dim]))


class TransformerDecoderLayer(nn.Module):
    def __init__(self, d_model, nhead, dim_feedforward=2048, dropout=0.1, activation="relu", normalize_before=False,
                 sa_first=True):
        super().__init__()
        self.sa_first = sa_first
        self.multihead_attn = nn.MultiheadAttention(d_model, nhead, dropout=dropout)
        self.self_attn = nn.MultiheadAttention(d_model, nhead, dropout=dropout)
        self.linear1 = nn.Linear(d_model, dim_feedforward)
        self.dropout = nn.Dropout(dropout)
        self.linear2 = nn.Linear(dim_feedforward, d_model)
        self.norm1 = nn.LayerNorm(d_model)
        self.norm2 = nn.LayerNorm(d_model)
        self.norm3 = nn.LayerNorm(d_model)
        self.dropout1 = nn.Dropout(dropout)
        self.dropout2 = nn.Dropout(dropout)
        self.dropout3 = nn.Dropout(dropout)
        self.normalize_before = normalize_before


class TransformerDecoder(nn.Module):
    def __init__(self, decoder_layer, num_layers, norm=None, return_intermediate=False):
        super().__init__()
        self.layers = nn.ModuleList([copy.deepcopy(decoder_layer) for _ in range(num_layers)])
        self.num_layers = num_layers
        self.norm = norm
        self.return_intermediate = return_intermediate


class Cross_Attention(nn.Module):
    """Reference :50-93.  Only the configuration every reference script uses is implemented: pre-norm
    (``normalize_before=True`` -- the post-norm branch of the reference cannot run, SURVEY.md appendix A),
    ``return_intermediate_dec=True``, ReLU FFN, self-attention first."""

    def __init__(self, d_model=512, nhead=8, num_encoder_layers=6, num_decoder_layers=6, dim_feedforward=2048,
                 dropout=0.1, activation="relu", normalize_before=False, hidden_dim=768,
                 return_intermediate_dec=False, sa_first=True):
        super().__init__()
        if not normalize_before or not return_intermediate_dec or activation != "relu" or not sa_first:
            raise NotImplementedError("Cross_Attention (B200): normalize_before=True, return_intermediate_dec=True, "
                                      "activation='relu', sa_first=True is the supported configuration")
        self.pre_norm = nn.LayerNorm(d_model)
        layer = TransformerDecoderLayer(d_model, nhead, dim_feedforward, dropout, activation, normalize_before,
                                        sa_first=sa_first)
        self.decoder = TransformerDecoder(layer, num_decoder_layers, nn.LayerNorm(d_model),
                                          return_intermediate=return_intermediate_dec)
        for p in self.parameters():
            if p.dim() > 1:
                nn.init.xavier_uniform_(p)
        self.d_model = d_model
        self.nhead = nhead
        self.dec_layers = num_decoder_layers
        self.enc_layers = num_encoder_layers
        self.dim_feedforward = dim_feedforward
        self.dropout_p = dropout


class ObjDecoder(_DirtyHooks, nn.Module):
    """Reference :111-241.  num_queries (the scripts pass `--num_queries` + 1) may be 2 .. 32, in inference and in
    training; 1 (the reference's n_decode = 10 branch) raises NotImplementedError, above 32 hh_decoder_create refuses."""

    def __init__(self, transformer, num_classes, num_queries, feature_dim=768, aux_loss=False, pred_traj=True,
                 num_frames=4, patches_per_frame=256, backbone='LaviLa', self_attn=False):
        super().__init__()
        if self_attn:
            raise NotImplementedError("ObjDecoder(self_attn=True) is not used by any reference script")
        if num_queries == 1:
            raise NotImplementedError("the num_queries == 1 / n_decode = 10 branch (reference :135-137) is not implemented")
        self.backbone = backbone
        self.txt_proj = _NativeHead(nn.ReLU(), nn.Linear(768, 256))
        self.vid_proj = _NativeHead(nn.Linear(768, 256))
        self.num_queries = num_queries
        self.transformer = transformer
        hidden_dim = transformer.d_model
        self.hidden_dim = hidden_dim
        self.class_embed = nn.Linear(hidden_dim, num_classes + 1)
        self.bbox_embed = MLP(hidden_dim, hidden_dim, 4, 3)
        self.query_embed = nn.Embedding(num_queries, hidden_dim)
        self.pred_traj = pred_traj
        self.n_decode = 1
        if self.pred_traj:
            self.frame_index = nn.Embedding(num_frames, hidden_dim)
            self.frame_proj = nn.Linear(hidden_dim * 2, hidden_dim)
        self.aux_loss = aux_loss
        self.pos_embed = nn.Parameter(torch.zeros(1, patches_per_frame + 1, hidden_dim))
        self.temporal_embed = nn.Parameter(torch.zeros(1, num_frames, hidden_dim))
        nn.init.trunc_normal_(self.pos_embed, std=.02)
        nn.init.trunc_normal_(self.temporal_embed, std=.02)
        self.patches_per_frame = patches_per_frame
        self.proj = nn.Linear(feature_dim, hidden_dim, bias=False)
        self.num_frames = num_frames
        self.obj_proj = _NativeHead(nn.Linear(hidden_dim, hidden_dim), nn.ReLU(), nn.Linear(hidden_dim, 256))
        self._cfg = L.DecoderCfg(hidden_dim, transformer.nhead, transformer.dec_layers, transformer.dim_feedforward,
                                 num_queries, num_classes + 1, feature_dim, num_frames, patches_per_frame,
                                 1 if pred_traj else 0)
        self._handle = None
        self._sync = _ParamSync()
        # dropout stream of the training forward: seed (None -> torch.initial_seed(), i.e. torch.manual_seed governs it)
        # and a per-module step counter; `last_dropout` records what the most recent forward used (None = no dropout)
        self.dropout_seed = None
        self._drop_step = 0
        self.last_dropout = None

    # -- engine plumbing ---------------------------------------------------------------------------------------
    def _engine(self):
        if self._handle is None:
            h = C.c_void_p()
            L.check(L.load().hh_decoder_create(C.byref(h), C.byref(self._cfg)), "hh_decoder_create")
            self._handle = h
        return self._handle

    def __del__(self):
        h = getattr(self, "_handle", None)
        if h is not None and L._lib is not None:
            L._lib.hh_decoder_destroy(h)
            self._handle = None

    def _engine_params(self):
        skip = ("txt_proj.", "vid_proj.", "obj_proj.")
        for k, p in self.named_parameters():
            if not k.startswith(skip):
                yield k, p

    def sync_weights(self):
        lib = L.load()
        T = self.temporal_embed.shape[1]       # inflate_positional_embeds may have stretched it (run/test_epic.py:168-173)
        if T != self._cfg.num_frames and not self.pred_traj:
            if self._handle is not None:
                lib.hh_decoder_destroy(self._handle)
                self._handle = None
            self._cfg.num_frames = T
            self.num_frames = T
            self._sync = _ParamSync()
        h = self._engine()

        def setter(items):   # every changed parameter in one call (an optimizer step changes all 135)
            n = len(items)
            keys_c = (C.c_char_p * n)(*[k.encode() for k, _ in items])
            ptrs_c = (C.c_void_p * n)(*[L.ptr(t) for _, t in items])
            numels_c = (C.c_int64 * n)(*[t.numel() for _, t in items])
            L.check(lib.hh_decoder_set_weights(h, keys_c, ptrs_c, numels_c, n, L.stream_ptr()), "hh_decoder_set_weights")
        self._sync.sync(self._engine_params(), None, batch_setter=setter)

    def flops_per_clip(self, T=None) -> float:
        return L.load().hh_decoder_flops_per_clip(self._engine(), int(T or self.num_frames))

    def last_launches(self) -> int:
        return L.load().hh_decoder_last_launches(self._engine())

    def set_profile(self, on: bool):
        """Record CUDA events around every kernel launch of the engine (see profile())."""
        L.check(L.load().hh_decoder_set_profile(self._engine(), 1 if on else 0), "hh_decoder_set_profile")

    def profile(self):
        """{kernel class: (milliseconds, launches)} since the last call; waits for the recorded events."""
        lib = L.load()
        k = lib.hh_profile_num_classes()
        ms, cnt = (C.c_double * k)(), (C.c_int * k)()
        L.check(lib.hh_decoder_profile(self._engine(), ms, cnt), "hh_decoder_profile")
        return {lib.hh_profile_class_name(i).decode(): (ms[i], cnt[i]) for i in range(k) if cnt[i]}

    # -- reference API -----------------------------------------------------------------------------------------
    def construct_3d_pos_embed(self, T):
        tile_pos_embed = self.pos_embed[:, 1:, :].repeat(1, T, 1)
        tile_temporal_embed = self.temporal_embed.repeat_interleave(self.patches_per_frame, 1)
        return (tile_pos_embed + tile_temporal_embed).view(1, T, self.patches_per_frame, self.pos_embed.shape[-1])

    def _run_engine(self, features, train: bool):
        B, T, n, F = features.shape
        L_, Q, Cd, ncls = self._cfg.num_layers, self.num_queries, self.hidden_dim, self._cfg.num_classes1
        traj = self.pred_traj and T == self.num_frames
        dev = features.device
        hs = torch.empty(L_, B, Q, Cd, dtype=torch.float32, device=dev)
        logits = torch.empty(L_, B * (4 if traj else 1), Q, ncls, dtype=torch.float32, device=dev)
        boxes = torch.empty(L_, B * (T if traj else 1), Q, 4, dtype=torch.float32, device=dev)
        lib = L.load()
        if features.dtype == torch.bfloat16:
            fn = lib.hh_decoder_forward_train_bf16 if train else lib.hh_decoder_forward_bf16
        else:
            fn = lib.hh_decoder_forward_train if train else lib.hh_decoder_forward
        self.last_dropout = None
        if train:
            p = float(self.transformer.dropout_p) if self.training else 0.0
            seed = int(self.dropout_seed if self.dropout_seed is not None else torch.initial_seed()) & ((1 << 64) - 1)
            offset = self._drop_step & 0xFFFFFFFF
            L.check(L.load().hh_decoder_set_dropout(self._engine(), p, seed, offset), "hh_decoder_set_dropout")
            if p > 0:
                self.last_dropout = {"p": p, "seed": seed, "offset": offset}
                self._drop_step += 1
        L.check(fn(self._engine(), features.data_ptr(), features.stride(0), features.stride(2), B, T, L.ptr(hs),
                   L.ptr(logits), L.ptr(boxes), L.stream_ptr()), "hh_decoder_forward")
        return hs, logits, boxes

    def forward(self, features, use_checkpoint=False):
        """features [B,T,n,F] (fp32 or bf16, any strides with a unit innermost stride) -> (out, hs, [], []).  bf16
        features give the same outputs as their fp32 source (the engine rounds fp32 features to bf16 itself); in eval a
        bf16 image_feature_map[:, 1:] view is read in place.  With autograd enabled and trainable parameters the engine
        keeps its activations (and its own copy of the features) and the outputs carry the hand-written backward
        (gradients for every decoder parameter; `features` come from the frozen backbone and get none)."""
        if not features.is_cuda:
            raise RuntimeError("ObjDecoder (B200): input is on %s; there is no CPU fallback" % features.device)
        B, T, n, F = features.shape
        if n != self.patches_per_frame or F != self._cfg.feature_dim:
            raise RuntimeError("expected features [B,T,%d,%d], got %s" % (self.patches_per_frame, self._cfg.feature_dim,
                                                                          tuple(features.shape)))
        features = features.detach()
        if features.dtype not in (torch.float32, torch.bfloat16):
            features = features.float()
        vec = 16 // features.element_size()          # elements per 16 bytes
        if features.stride(3) != 1 or features.stride(1) != n * features.stride(2) or features.stride(2) % vec \
                or features.stride(0) % vec or features.data_ptr() % 16:
            features = features.contiguous()
        self.sync_weights()
        params = [p for _, p in self._engine_params()]
        if torch.is_grad_enabled() and any(p.requires_grad for p in params):
            if self.class_embed.weight.requires_grad and not getattr(self, "_warned_logits", False):
                # the reference criterion has no class loss (run/train.py:471, exclude_class=True): the hand-written
                # backward leaves class_embed.* at zero and pred_logits is a constant of the graph -- say so once
                # instead of letting a 'labels' loss train nothing in silence
                warnings.warn("ObjDecoder (B200): pred_logits carries no gradient (the reference training loop has no "
                              "class loss); a loss built on pred_logits will not train the decoder", stacklevel=2)
                self._warned_logits = True
            hs, logits, boxes = _DecoderFn.apply(self, features, *params)
        else:
            with torch.no_grad():  # train() mode drops activations even when no gradient is recorded, as nn.Dropout does
                hs, logits, boxes = self._run_engine(features, train=self.training and self.transformer.dropout_p > 0)
        out = {'pred_logits': logits[-1], 'pred_boxes': boxes[-1]}
        if self.aux_loss:
            out['aux_outputs'] = [{'pred_logits': a, 'pred_boxes': b} for a, b in zip(logits[:-1], boxes[:-1])]
        return out, hs, [], []
