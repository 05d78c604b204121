"""CPU: the drop-in modules keep the reference's state_dict key/shape contract (SURVEY.md section 8b) and the
reference's module-level API (constructor keywords, attributes the run scripts touch).

tests/golden/state_dict_layout.json holds the state_dict keys and shapes the interchange with the reference depends on
(_layout of a small backbone and decoder): it was recorded from this repository's modules, is compared with them
everywhere, and is itself compared with the original project's modules by the live test whenever $HH_REFERENCE_ROOT
names a checkout of it."""
import json
import os

import pytest
import torch

from oracle import hh_oracle as O
from oracle import ref_import
from helping_hand_for_egocentric_videos_b200.model import LaviLa, tfm_decoder


def test_backbone_keys_match_survey_counts():
    m = LaviLa.CLIP_OPENAI_TIMESFORMER_LARGE(num_frames=4, pretrained=None, text_use_cls_token=False)
    sd = m.state_dict()
    assert len(sd) == 591
    assert sum(p.numel() for p in m.parameters()) == 527513857          # 527.5 M (SURVEY.md section 8b)
    want = O.clip_param_shapes(1024, 24, 14, 256, 4)
    assert set(sd) == set(want)
    for k, shp in want.items():
        assert tuple(sd[k].shape) == tuple(shp), k
    # the scripts strip 'module.' and load strict (run/test_EgoMCQ.py:223-227)
    m.load_state_dict({k: torch.zeros_like(v) for k, v in sd.items()}, strict=True)
    # freshly built temporal attention is the reference's zero init (model/LaviLa.py:236-242)
    m2 = LaviLa.CLIP_OPENAI_TIMESFORMER_LARGE(num_frames=4)
    assert float(m2.visual.blocks[0].timeattn.qkv.weight.abs().sum()) == 0.0
    assert float(m2.visual.blocks[0].timeattn.proj.weight.min()) == 1.0


def test_decoder_keys_match_survey_counts():
    for traj, nkeys in ((True, 135), (False, 132)):
        tr = tfm_decoder.Cross_Attention(normalize_before=True, return_intermediate_dec=True)
        d = tfm_decoder.ObjDecoder(tr, num_classes=22047, num_queries=13, aux_loss=True, pred_traj=traj,
                                   feature_dim=1024, num_frames=4)
        sd = d.state_dict()
        assert len(sd) == nkeys
        want = O.decoder_param_shapes(512, 13, 256, 4, 1024, 22048, pred_traj=traj)
        assert set(sd) == set(want)
        for k, shp in want.items():
            assert tuple(sd[k].shape) == tuple(shp), k
    assert hasattr(d, "txt_proj") and hasattr(d, "obj_proj") and hasattr(d, "vid_proj")
    names = [n for n, _ in d.named_parameters()]
    assert any(".bias" in n for n in names) and any("norm" in n for n in names)   # optim_policy groups by these


def test_unsupported_configurations_are_refused():
    with pytest.raises(NotImplementedError):
        LaviLa.SpaceTimeTransformer()                      # default: GELU, no ln_pre -> not the LaViLa tower
    with pytest.raises(NotImplementedError):
        tfm_decoder.Cross_Attention(normalize_before=False)


GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "state_dict_layout.json")


def _layout(backbone, decoder):
    return {name: {k: list(v.shape) for k, v in m.state_dict().items()}
            for name, m in (("backbone", backbone), ("decoder", decoder))}


def _small_modules():
    vis = LaviLa.SpaceTimeTransformer(img_size=56, patch_size=14, embed_dim=128, depth=2, num_heads=2, num_frames=3,
                                      time_init='zeros', ln_pre=True, act_layer=LaviLa.QuickGELU)
    vis.head = torch.nn.Identity()
    mine = LaviLa.CLIP(embed_dim=256, vision_width=128, vision_model=vis, context_length=77, vocab_size=128,
                       transformer_width=768, transformer_heads=12, transformer_layers=1)
    tr = tfm_decoder.Cross_Attention(d_model=128, nhead=2, num_decoder_layers=2, dim_feedforward=256,
                                     normalize_before=True, return_intermediate_dec=True)
    mdec = tfm_decoder.ObjDecoder(tr, num_classes=30, num_queries=5, aux_loss=True, feature_dim=128, num_frames=3,
                                  patches_per_frame=16)
    return mine, mdec


def test_state_dicts_match_the_stored_reference_layout():
    with open(GOLDEN) as f:
        assert _layout(*_small_modules()) == json.load(f)


@pytest.mark.skipif(not ref_import.reference_available(), reason="needs a checkout of the original project (HH_REFERENCE_ROOT)")
def test_state_dicts_interchange_with_the_live_reference():
    ns = ref_import.import_reference()
    ref = ref_import.build_reference_backbone(ns, img_size=56, patch_size=14, embed_dim=128, depth=2, num_heads=2,
                                              num_frames=3, text_layers=1, vocab_size=128)
    rdec = ref_import.build_reference_decoder(ns, num_queries=5, feature_dim=128, num_frames=3, patches_per_frame=16,
                                              num_classes=30, d_model=128, nhead=2, dec_layers=2, ffn=256)
    mine, mdec = _small_modules()
    mine.load_state_dict(ref.state_dict(), strict=True)
    ref.load_state_dict(mine.state_dict(), strict=True)
    mdec.load_state_dict(rdec.state_dict(), strict=True)
    rdec.load_state_dict(mdec.state_dict(), strict=True)
    with open(GOLDEN) as f:
        assert _layout(ref, rdec) == json.load(f)
