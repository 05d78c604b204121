"""bf16 hand-over of the video tower's feature map (SpaceTimeTransformer.feature_map_dtype = torch.bfloat16).

The encoder's bf16 map must be its fp32 map rounded to nearest-even, with x_cls / image_embed unchanged; the decoder
rounds its input to bf16 itself, so on a bf16 map it must give the fp32 run's outputs bit for bit, whether it reads the
caller's rows in place (inference, T*n a multiple of 128) or gathers them first (every other case, and training)."""
import os

import pytest
import torch

from oracle import golden_cases as gc


def _mods():
    from helping_hand_for_egocentric_videos_b200.model import LaviLa, tfm_decoder
    return LaviLa, tfm_decoder


def _backbone(case, unfused=False):
    LaviLa, _ = _mods()
    c = case["cfg"]
    old = os.environ.get("HH_LN_UNFUSED")
    os.environ["HH_LN_UNFUSED"] = "1" if unfused else "0"
    try:
        vis = LaviLa.SpaceTimeTransformer(img_size=c["img"], patch_size=c["patch"], embed_dim=c["D"], depth=c["L"],
                                          num_heads=c["H"], num_frames=c["T"], time_init='zeros', ln_pre=True,
                                          act_layer=LaviLa.QuickGELU)
        vis.head = torch.nn.Identity()
        clip = LaviLa.CLIP(embed_dim=256, vision_width=c["D"], vision_model=vis, context_length=77, vocab_size=c["vocab"],
                           transformer_width=c["text_width"], transformer_heads=c["text_heads"],
                           transformer_layers=c["text_layers"])
        clip.load_state_dict(gc.backbone_state_dict(case), strict=True)
        clip = clip.cuda().eval()
        clip.visual._engine()          # the engine reads HH_LN_UNFUSED when it is created
    finally:
        if old is None:
            del os.environ["HH_LN_UNFUSED"]
        else:
            os.environ["HH_LN_UNFUSED"] = old
    return clip


def _decoder(cfg, dropout=0.1):
    _, D = _mods()
    tr = D.Cross_Attention(d_model=cfg["C"], nhead=cfg["heads"], num_decoder_layers=cfg["layers"],
                           dim_feedforward=cfg["ffn"], dropout=dropout, normalize_before=True,
                           return_intermediate_dec=True)
    return D.ObjDecoder(transformer=tr, num_classes=cfg["ncls"], num_queries=cfg["Q"], aux_loss=True,
                        pred_traj=cfg["pred_traj"], feature_dim=cfg["F"], num_frames=cfg["T"],
                        patches_per_frame=cfg["n"])


def _equal_outputs(a, b):
    (oa, hsa, _, _), (ob, hsb, _, _) = a, b
    assert torch.equal(hsa, hsb)
    assert torch.equal(oa["pred_logits"], ob["pred_logits"]) and torch.equal(oa["pred_boxes"], ob["pred_boxes"])
    assert len(oa["aux_outputs"]) == len(ob["aux_outputs"])
    for x, y in zip(oa["aux_outputs"], ob["aux_outputs"]):
        assert torch.equal(x["pred_logits"], y["pred_logits"]) and torch.equal(x["pred_boxes"], y["pred_boxes"])


# ------------------------------------------------------------------------------------------ CPU
def test_feature_map_dtype_accepts_fp32_and_bf16_only():
    LaviLa, _ = _mods()
    vis = LaviLa.SpaceTimeTransformer(img_size=56, patch_size=14, embed_dim=128, depth=1, num_heads=2, num_frames=2,
                                      ln_pre=True, act_layer=LaviLa.QuickGELU, time_init='zeros', num_classes=0)
    assert vis.feature_map_dtype == torch.float32
    vis.feature_map_dtype = torch.bfloat16
    assert vis.feature_map_dtype == torch.bfloat16
    for bad in (torch.float16, torch.float64, "bfloat16", None):
        with pytest.raises(ValueError):
            vis.feature_map_dtype = bad
    assert vis.feature_map_dtype == torch.bfloat16


# ------------------------------------------------------------------------------------------ encoder
@pytest.mark.gpu
@pytest.mark.parametrize("name,u8,unfused", [("enc_tiny", False, False), ("enc_tiny", True, False),
                                             ("enc_tiny", False, True), ("enc_c0", False, False),
                                             ("enc_c0", True, False), ("enc_l14", False, False),
                                             ("enc_l14_t16", False, False)])
def test_encoder_bf16_map_is_the_rounded_fp32_map(name, u8, unfused):
    case = gc.CASES[name]
    c = case["cfg"]
    clip = _backbone(case, unfused=unfused)
    vis = clip.visual
    if u8:
        g = torch.Generator().manual_seed(78)
        frames = torch.randint(0, 256, (2, c["T"], c["img"], c["img"], 3), generator=g, dtype=torch.uint8).cuda()
        mean, std = [0.42, 0.46, 0.41], [0.27, 0.26, 0.28]

        def run():
            return vis.forward_features_u8(frames, mean, std)
    else:
        video, tokens = gc.make_inputs(case)
        video, tokens = video.cuda(), tokens.cuda()

        def run():
            out = clip(video, tokens)
            x_cls, fmap = vis.forward_features(video)
            return x_cls, fmap, out["image_embed"]
    a = run()
    n32 = vis.last_launches()
    vis.feature_map_dtype = torch.bfloat16
    b = run()
    n16 = vis.last_launches()
    assert a[1].dtype == torch.float32 and b[1].dtype == torch.bfloat16 and b[0].dtype == torch.float32
    assert torch.equal(b[1], a[1].to(torch.bfloat16))
    assert torch.equal(b[0], a[0])                 # x_cls
    if not u8:
        assert torch.equal(b[2], a[2])             # image_embed (projected, normalised)
    assert n16 == n32
    # the truncated-forward test hook keeps returning fp32
    if not u8 and name == "enc_tiny":
        _, f1 = vis.forward_features(gc.make_inputs(case)[0].cuda(), _nblocks=1)
        assert f1.dtype == torch.float32


# ------------------------------------------------------------------------------------------ decoder, eval
def _check_decoder_eval(cfg, feats, sd=None):
    """feats fp32 [B,T,n,F] on the device: contiguous input and the [:, 1:] view of a full map, fp32 vs bf16."""
    dec = _decoder(cfg)
    if sd is not None:
        dec.load_state_dict(sd, strict=True)
    dec = dec.cuda().eval()
    B, T, n, F = feats.shape
    S = T * n
    fmap = torch.randn(B, 1 + S, F, device=feats.device)
    fmap[:, 1:] = feats.reshape(B, S, F)
    fmap16 = fmap.to(torch.bfloat16)
    cases = [(feats, feats.to(torch.bfloat16)),
             (fmap[:, 1:].unflatten(1, (T, n)), fmap16[:, 1:].unflatten(1, (T, n)))]
    direct = S % 128 == 0
    for f32, f16 in cases:
        assert torch.equal(f16.float(), f32.to(torch.bfloat16).float())
        # inference forward (under autograd with trainable parameters the module runs the training forward, which
        # always copies the features: covered by the training test below)
        with torch.no_grad():
            r32 = dec(f32)
            n32 = dec.last_launches()
            r16 = dec(f16)
            n16 = dec.last_launches()
        _equal_outputs(r32, r16)
        assert n16 == n32 - (1 if direct else 0), (n32, n16, S)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["dec_tiny_traj", "dec_tiny_notraj", "dec_c0", "dec_c1", "dec_c2", "dec_c4"])
def test_decoder_eval_bf16_features_bit_identical(name):
    case = gc.CASES[name]
    feats, _ = gc.make_inputs(case)
    _check_decoder_eval(case["cfg"], feats.cuda(), gc.decoder_state_dict(case))


@pytest.mark.gpu
@pytest.mark.parametrize("name,B", [("dec_c2", 4), ("dec_c4", 16)])
def test_decoder_eval_bf16_on_the_cta_pair_plan(name, B):
    """B * T * n = 16384 rows: 128 row tiles, enough for the proj GEMM to run as CTA pairs (>= 74 row tiles)."""
    case = gc.CASES[name]
    c = case["cfg"]
    g = torch.Generator().manual_seed(900 + B)
    feats = torch.randn(B, c["T"], c["n"], c["F"], generator=g)
    _check_decoder_eval(c, feats.cuda(), gc.decoder_state_dict(case))


# ------------------------------------------------------------------------------------------ decoder, training
def _train_grads(cfg, sd, feats, overwrite=False):
    dec = _decoder(cfg, dropout=0.1)
    dec.load_state_dict(sd, strict=True)
    dec = dec.cuda().train()
    dec.dropout_seed = 0x5EED0123456789
    g = torch.Generator().manual_seed(5)
    w_hs = torch.randn(cfg["layers"], *feats.shape[:1], cfg["Q"], cfg["C"], generator=g).cuda()
    out, hs, _, _ = dec(feats)
    boxes = torch.stack([a["pred_boxes"] for a in out["aux_outputs"]] + [out["pred_boxes"]])
    loss = (hs * w_hs).sum() + boxes.square().sum()
    if overwrite:
        feats.normal_()        # the engine keeps its own copy of the features for backward()
    loss.backward()
    grads = {k: p.grad.detach().clone() for k, p in dec.named_parameters() if p.grad is not None}
    return (out, hs), grads


def _grads_equal(ga, gb):
    """The weight-gradient kernels combine partial tiles with fp32 atomics where a reduction is split (last bits vary
    from run to run), so tensors are compared to fp32 summation noise; any other difference would be of the order of
    the features' bf16 rounding or the gradients themselves."""
    assert ga.keys() == gb.keys()
    for k in ga:
        a, b = ga[k], gb[k]
        if torch.equal(a, b):
            continue
        scale = a.abs().max().item()
        err = (a - b).abs().max().item()
        assert err <= 1e-5 * max(scale, 1e-3), (k, err, scale)


@pytest.mark.gpu
@pytest.mark.parametrize("name,B", [("dec_train_dropout", 2), ("dec_c4", 3)])
def test_decoder_training_bf16_features(name, B):
    case = gc.CASES[name]
    c = case["cfg"]
    sd = gc.decoder_state_dict(case)
    g = torch.Generator().manual_seed(31 + B)
    S = c["T"] * c["n"]
    fmap = torch.randn(B, 1 + S, c["F"], generator=g).cuda()
    feats32 = fmap[:, 1:].unflatten(1, (c["T"], c["n"]))
    fmap16 = fmap.to(torch.bfloat16)
    (o32, hs32), g32 = _train_grads(c, sd, feats32)
    (o16, hs16), g16 = _train_grads(c, sd, fmap16[:, 1:].unflatten(1, (c["T"], c["n"])))
    assert torch.equal(hs32, hs16)
    assert torch.equal(o32["pred_boxes"], o16["pred_boxes"]) and torch.equal(o32["pred_logits"], o16["pred_logits"])
    assert "proj.weight" in g16
    _grads_equal(g32, g16)
    # overwriting the caller's bf16 map between forward and backward changes nothing
    scratch = fmap16.clone()
    (_, hs16b), g16b = _train_grads(c, sd, scratch[:, 1:].unflatten(1, (c["T"], c["n"])), overwrite=True)
    assert torch.equal(hs16b, hs16)
    _grads_equal(g16, g16b)
