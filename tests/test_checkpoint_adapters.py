"""Host-side checkpoint adapters (SURVEY.md section 8f row 4) against the reference's own functions.

tests/golden/checkpoint_adapters.pt holds what the comparison with the reference looks at (_adapter_outputs): it was
recorded from this repository's adapters, is compared with them everywhere, and is itself compared with the original
project's functions by the live test whenever $HH_REFERENCE_ROOT names a checkout of it."""
import ast
import os

import pytest
import torch

from helping_hand_for_egocentric_videos_b200.utils import checkpoint as ck
from oracle import ref_import


def _clip_visual_sd(layers=2, width=8):
    g = torch.Generator().manual_seed(0)
    sd = {"class_embedding": torch.randn(width, generator=g), "positional_embedding": torch.randn(5, width, generator=g),
          "conv1.weight": torch.randn(width, 3, 2, 2, generator=g), "proj": torch.randn(width, 4, generator=g)}
    for k in ("ln_pre", "ln_post"):
        sd[k + ".weight"], sd[k + ".bias"] = torch.randn(width, generator=g), torch.randn(width, generator=g)
    for i in range(layers):
        p = "transformer.resblocks.%d." % i
        for k, shp in (("attn.in_proj_weight", (3 * width, width)), ("attn.in_proj_bias", (3 * width,)),
                       ("attn.out_proj.weight", (width, width)), ("attn.out_proj.bias", (width,)),
                       ("ln_1.weight", (width,)), ("ln_1.bias", (width,)), ("ln_2.weight", (width,)),
                       ("ln_2.bias", (width,)), ("mlp.c_fc.weight", (4 * width, width)), ("mlp.c_fc.bias", (4 * width,)),
                       ("mlp.c_proj.weight", (width, 4 * width)), ("mlp.c_proj.bias", (width,))):
            sd[p + k] = torch.randn(*shp, generator=g)
    return sd


GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "checkpoint_adapters.pt")
INFLATE_CASES = [(4, 16, "bilinear"), (4, 16, "interp"), (4, 16, "zeros"), (16, 4, "bilinear"), (4, 4, "zeros")]


def _adapter_outputs(remap_keys, inflate_positional_embeds):
    out = {"remap_keys": remap_keys(_clip_visual_sd(), transformer_layers=2)}
    for have, want_t, fix in INFLATE_CASES:
        cur = {"visual.temporal_embed": torch.zeros(1, want_t, 8)}
        new = {"visual.temporal_embed": torch.arange(have * 8.).view(1, have, 8)}
        out["inflate_%d_%d_%s" % (have, want_t, fix)] = inflate_positional_embeds(
            cur, new, num_frames=want_t, load_temporal_fix=fix)["visual.temporal_embed"]
    return out


def _assert_same(got, want):
    assert list(got) == list(want)
    assert list(got["remap_keys"]) == list(want["remap_keys"])
    assert all(torch.equal(got["remap_keys"][k], v) for k, v in want["remap_keys"].items())
    for k, v in want.items():
        if k != "remap_keys":
            assert torch.equal(got[k], v), k


def test_adapters_equal_the_stored_reference_outputs():
    _assert_same(_adapter_outputs(ck.remap_keys, ck.inflate_positional_embeds), torch.load(GOLDEN))


def test_strip_module_prefix():
    sd = {"module.visual.cls_token": 1, "logit_scale": 2}
    assert list(ck.strip_module_prefix(sd)) == ["visual.cls_token", "logit_scale"]


def test_remap_keys_contract():
    out = ck.remap_keys(_clip_visual_sd(), transformer_layers=2)
    assert "proj" not in out and out["cls_token"].shape == (1, 1, 8) and out["pos_embed"].shape == (1, 5, 8)
    assert "blocks.1.attn.qkv.weight" in out and "blocks.0.mlp.fc2.bias" in out and "norm.weight" in out
    with pytest.raises(KeyError):
        ck.remap_keys(_clip_visual_sd(layers=3), transformer_layers=2)


def test_inflate_contract():
    cur = {"visual.temporal_embed": torch.zeros(1, 16, 8)}
    for fix in ("zeros", "interp", "bilinear"):
        new = {"visual.temporal_embed": torch.arange(32.).view(1, 4, 8)}
        out = ck.inflate_positional_embeds(cur, new, num_frames=16, load_temporal_fix=fix)
        assert out["visual.temporal_embed"].shape == (1, 16, 8)
    new = {"visual.temporal_embed": torch.arange(32.).view(1, 4, 8)}
    assert ck.inflate_positional_embeds({"visual.temporal_embed": torch.zeros(1, 2, 8)}, new, num_frames=2)[
        "visual.temporal_embed"].shape == (1, 2, 8)
    with pytest.raises(NotImplementedError):
        ck.inflate_positional_embeds(cur, {"visual.temporal_embed": torch.zeros(1, 4, 8)}, num_frames=8)


@pytest.mark.skipif(not ref_import.reference_available(), reason="needs a checkout of the original project (HH_REFERENCE_ROOT)")
def test_adapters_equal_the_reference(capsys):
    ns = ref_import.import_reference()
    # run/test_egtea.py imports sacred at module level; execute only its inflate_positional_embeds definition
    src = open(ref_import.REFERENCE_ROOT + "/run/test_egtea.py").read()
    fn = next(n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == "inflate_positional_embeds")
    scope = {"torch": torch, "F": torch.nn.functional}
    exec(compile(ast.Module(body=[fn], type_ignores=[]), "ref_inflate", "exec"), scope)
    want = _adapter_outputs(ns.LaviLa.remap_keys, scope["inflate_positional_embeds"])
    _assert_same(_adapter_outputs(ck.remap_keys, ck.inflate_positional_embeds), want)
    _assert_same(torch.load(GOLDEN), want)
