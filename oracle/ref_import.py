"""Import the *unmodified* reference modules from a checkout of the original project named by $HH_REFERENCE_ROOT.

TEST INFRASTRUCTURE ONLY.  The original project is not part of this repository, so nothing
reachable from `pytest -m gpu`, smoke() or bench.py may call into this file; it is used
by `oracle/make_golden.py` and by the CPU tests that are skipped when no checkout is named.

The reference imports two packages the image lacks (SURVEY.md §8c):
  * ``timm.models.layers`` -- only DropPath / to_2tuple / trunc_normal_ are used
    (model/LaviLa.py:12, model/tfm_decoder.py:11); drop_path_rate is always 0.
  * ``ftfy`` -- tokenizer only (model/tokenizer.py:16).
Both get tiny stand-ins.  The factory functions CLIP_OPENAI_TIMESFORMER_* download CLIP
weights (model/LaviLa.py:69,130), so the builders below construct SpaceTimeTransformer /
CLIP directly with the factory's kwargs (model/LaviLa.py:118-162).
"""
import os
import sys
import types
import contextlib
import io

REFERENCE_ROOT = os.environ.get("HH_REFERENCE_ROOT", "")


def reference_available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isfile(os.path.join(REFERENCE_ROOT, "model", "LaviLa.py"))


def _install_shims():
    import torch
    import torch.nn as nn
    try:  # transformers probes timm.__spec__; import it before the stub exists
        import transformers  # noqa: F401
    except Exception:
        pass
    if "timm" not in sys.modules:
        timm = types.ModuleType("timm")
        timm.__path__ = []
        models = types.ModuleType("timm.models")
        models.__path__ = []
        layers = types.ModuleType("timm.models.layers")

        class DropPath(nn.Module):
            def __init__(self, p=0.0):
                super().__init__()
                assert p == 0.0, "reference always uses drop_path_rate=0"

            def forward(self, x):
                return x

        def to_2tuple(v):
            return tuple(v) if isinstance(v, (tuple, list)) else (v, v)

        layers.DropPath = DropPath
        layers.to_2tuple = to_2tuple
        layers.trunc_normal_ = torch.nn.init.trunc_normal_
        timm.models = models
        models.layers = layers
        sys.modules["timm"] = timm
        sys.modules["timm.models"] = models
        sys.modules["timm.models.layers"] = layers
    if "ftfy" not in sys.modules:
        ftfy = types.ModuleType("ftfy")
        ftfy.fix_text = lambda s: s
        sys.modules["ftfy"] = ftfy


def import_reference():
    """Returns a namespace with the reference modules (LaviLa, tfm_decoder, metric, box_ops, ...)."""
    if not reference_available():
        raise RuntimeError("HH_REFERENCE_ROOT (%r) does not name a checkout of the original project" % REFERENCE_ROOT)
    _install_shims()
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import importlib
    ns = types.SimpleNamespace()
    ns.LaviLa = importlib.import_module("model.LaviLa")
    ns.tfm_decoder = importlib.import_module("model.tfm_decoder")
    ns.openai_model = importlib.import_module("model.openai_model")
    ns.metric = importlib.import_module("model.metric")
    ns.box_ops = importlib.import_module("utils.box_ops")
    return ns


def build_reference_backbone(ns, *, img_size=224, patch_size=14, embed_dim=1024, depth=24, num_heads=16,
                             num_frames=4, text_width=768, text_heads=12, text_layers=12,
                             project_embed_dim=256, vocab_size=49408, context_length=77):
    """CLIP(SpaceTimeTransformer) with the kwargs of CLIP_OPENAI_TIMESFORMER_LARGE (model/LaviLa.py:118-162)."""
    import torch.nn as nn
    with contextlib.redirect_stdout(io.StringIO()):
        vis = ns.LaviLa.SpaceTimeTransformer(
            img_size=img_size, patch_size=patch_size, embed_dim=embed_dim, depth=depth, num_heads=num_heads,
            num_frames=num_frames, time_init='zeros', attention_style='frozen-in-time', ln_pre=True,
            act_layer=ns.openai_model.QuickGELU, is_tanh_gating=False, drop_path_rate=0, use_adapter=False)
        vis.head = nn.Identity()
        vis.pre_logits = nn.Identity()
        vis.fc = nn.Identity()
        clip = ns.LaviLa.CLIP(embed_dim=project_embed_dim, vision_width=embed_dim, vision_model=vis,
                              context_length=context_length, vocab_size=vocab_size, transformer_width=text_width,
                              transformer_heads=text_heads, transformer_layers=text_layers, tempearture_init=0.07)
    return clip.eval()


def build_reference_decoder(ns, *, num_queries=5, feature_dim=1024, num_frames=4, patches_per_frame=256,
                            pred_traj=True, num_classes=22047, d_model=512, nhead=8, dec_layers=6, ffn=2048):
    """Cross_Attention + ObjDecoder as constructed in run/test_EgoMCQ.py:237-243."""
    tr = ns.tfm_decoder.Cross_Attention(d_model=d_model, nhead=nhead, num_decoder_layers=dec_layers,
                                        dim_feedforward=ffn, normalize_before=True, return_intermediate_dec=True)
    dec = ns.tfm_decoder.ObjDecoder(transformer=tr, num_classes=num_classes, num_queries=num_queries, aux_loss=True,
                                    pred_traj=pred_traj, feature_dim=feature_dim, num_frames=num_frames,
                                    patches_per_frame=patches_per_frame, self_attn=False)
    return dec.eval()
