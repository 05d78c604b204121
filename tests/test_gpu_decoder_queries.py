"""17 .. 32 queries per clip (`--num_queries` 16 .. 31): the second 16-row query block of the tensor-core cross-attention
kernels (QB = 2), the 32-lane self attention and the 32-row SIMT cross-attention backward, from the kernels up to the
public modules.

- kernels against float64 / fp32 torch with the tolerances of test_gpu_kernels.py and test_gpu_backward.py;
- the second query block against the first, bit for bit: the QB = 2 instantiation does the QB = 1 arithmetic per block;
- the training step, one kernel step at a time, against float64 (test_gpu_decoder_steps._run_case);
- the module against the oracle: gradients, L/14 inference (fp32 and bf16 feature maps) and a training step at nq = 31;
- refusals: Q = 33 everywhere, Q = 17 on the SIMT forward (a differential reference kept at 16 queries)."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from oracle import golden_cases as gc
from oracle import hh_oracle as O
from test_gpu_backward import _check_grads, _decoder_grads_case
from test_gpu_decoder_steps import C4, _cfg, _run_case


def _ops():
    from helping_hand_for_egocentric_videos_b200 import ops
    return ops


def _off8(t):
    """A contiguous copy 4 bytes off an 8-byte boundary: the tensor-core backward does not take it, the SIMT one does."""
    flat = torch.empty(t.numel() + 1, device="cuda")
    flat[1:] = t.flatten().cuda()
    out = flat[1:].view(t.shape)
    assert out.data_ptr() % 8 != 0
    return out


# ------------------------------------------------------------------------------------------ kernels
@pytest.mark.gpu
@pytest.mark.parametrize("B,Q,heads,S", [(2, 17, 8, 1024), (1, 32, 8, 4096), (3, 24, 2, 77), (1, 32, 1, 31),
                                         (2, 32, 2, 100)])
def test_cross_attention(B, Q, heads, S):
    """Tolerance of test_gpu_kernels.test_cross_attention: P is rounded to bf16 for P.V (2^-7 rel + 4e-3)."""
    g = torch.Generator().manual_seed(B * 1000 + Q * 10 + heads)
    Cc = heads * 64
    q = (torch.randn(B * Q, Cc, generator=g) * 0.3).double()
    K = torch.randn(B * S, Cc, generator=g).bfloat16()
    V = torch.randn(B * S, Cc, generator=g).bfloat16()
    got = _ops().cross_attention(q.float().cuda(), K.cuda(), V.cuda(), B, Q, heads, S).cpu().double()
    qh = q.view(B, Q, heads, 64).transpose(1, 2)
    kh = K.double().view(B, S, heads, 64).transpose(1, 2)
    vh = V.double().view(B, S, heads, 64).transpose(1, 2)
    ref = (torch.softmax(qh @ kh.transpose(-1, -2), -1) @ vh).transpose(1, 2).reshape(B * Q, Cc)
    err = (got - ref).abs()
    assert bool((err <= 4e-3 + 2 ** -7 * ref.abs()).all()), err.max().item()


@pytest.mark.gpu
@pytest.mark.parametrize("B,Q,heads", [(3, 17, 8), (2, 32, 2), (1, 32, 8)])
def test_self_attention_backward(B, Q, heads):
    """Tolerance of test_gpu_backward.test_self_attention_backward (5e-5 of max(1, max|ref|))."""
    g = torch.Generator().manual_seed(B * 10 + Q)
    Cc = heads * 64
    qkv = torch.randn(B * Q, 3 * Cc, generator=g) * 0.5
    dO = torch.randn(B * Q, Cc, generator=g)
    t = qkv.double().requires_grad_(True)
    x = t.view(B, Q, 3, heads, 64).permute(2, 0, 3, 1, 4)
    o = (torch.softmax(x[0] @ x[1].transpose(-1, -2), -1) @ x[2]).permute(0, 2, 1, 3).reshape(B * Q, Cc)
    o.backward(dO.double())
    got = _ops().self_attention_backward(qkv.cuda(), dO.cuda(), B, Q, heads).cpu().double()
    err = (got - t.grad).abs().max().item()
    assert err <= 5e-5 * max(1.0, t.grad.abs().max().item()), err


@pytest.mark.gpu
@pytest.mark.parametrize("B,Q,heads,S", [(2, 17, 8, 1024), (1, 32, 2, 196), (3, 32, 2, 77), (1, 24, 1, 300)])
def test_cross_attention_backward(B, Q, heads, S):
    """Tolerances of test_gpu_backward.test_cross_attention_backward (dq 1e-4, dK / dV 2^-7 + 1e-4), aligned operands
    (tensor-core kernel) and q / dO 4 bytes off an 8-byte boundary (SIMT kernels)."""
    g = torch.Generator().manual_seed(S + Q)
    Cc = heads * 64
    q = torch.randn(B * Q, Cc, generator=g) * 0.3
    K = torch.randn(B * S, Cc, generator=g).to(torch.bfloat16)
    V = torch.randn(B * S, Cc, generator=g).to(torch.bfloat16)
    dO = torch.randn(B * Q, Cc, generator=g)
    q0, K0, V0 = q.double().requires_grad_(True), K.double().requires_grad_(True), V.double().requires_grad_(True)
    qh = q0.view(B, Q, heads, 64).transpose(1, 2)
    kh, vh = K0.view(B, S, heads, 64).transpose(1, 2), V0.view(B, S, heads, 64).transpose(1, 2)
    O_ = (torch.softmax(qh @ kh.transpose(-1, -2), -1) @ vh).transpose(1, 2).reshape(B * Q, Cc)
    O_.backward(dO.double())
    Of = O_.detach().float().cuda()

    def close(got, want, name, rtol, atol=0.0):
        err = (got.detach().cpu().double() - want).abs().max().item()
        assert err <= atol + rtol * max(1.0, want.abs().max().item()), (name, err)
    for tag, qq, gg in (("tensor core", q.cuda(), dO.cuda()), ("SIMT", _off8(q), _off8(dO))):
        dq, dK, dV = _ops().cross_attention_backward(qq, K.cuda(), V.cuda(), Of, gg, B, Q, heads, S)
        close(dq, q0.grad, "dq " + tag, 1e-4)
        close(dK, K0.grad, "dK " + tag, 2 ** -7, 1e-4)
        close(dV, V0.grad, "dV " + tag, 2 ** -7, 1e-4)


@pytest.mark.gpu
@pytest.mark.parametrize("B,heads,S", [(2, 8, 1024), (1, 2, 77), (3, 8, 4096)])
def test_second_query_block_matches_the_first_bit_for_bit(B, heads, S):
    """q rows 16 .. 31 equal to rows 0 .. 15 (no dropout): the forward output and the tensor-core backward's dq of the
    second block equal those of the first, and both equal the rows of the Q = 16 call."""
    ops = _ops()
    g = torch.Generator().manual_seed(S + heads)
    Cc = heads * 64
    q16 = torch.randn(B, 16, Cc, generator=g) * 0.3
    dO16 = torch.randn(B, 16, Cc, generator=g)
    K = torch.randn(B * S, Cc, generator=g).to(torch.bfloat16).cuda()
    V = torch.randn(B * S, Cc, generator=g).to(torch.bfloat16).cuda()
    q32, dO32 = torch.cat([q16, q16], 1).cuda(), torch.cat([dO16, dO16], 1).cuda()
    q16, dO16 = q16.cuda(), dO16.cuda()
    o32 = ops.cross_attention(q32.reshape(B * 32, Cc), K, V, B, 32, heads, S).view(B, 32, Cc)
    o16 = ops.cross_attention(q16.reshape(B * 16, Cc), K, V, B, 16, heads, S).view(B, 16, Cc)
    assert torch.equal(o32[:, 16:], o32[:, :16])
    assert torch.equal(o32[:, :16], o16)
    dq32, _, _ = ops.cross_attention_backward(q32.reshape(B * 32, Cc), K, V, o32.reshape(B * 32, Cc),
                                              dO32.reshape(B * 32, Cc), B, 32, heads, S)
    dq16, _, _ = ops.cross_attention_backward(q16.reshape(B * 16, Cc), K, V, o16.reshape(B * 16, Cc),
                                              dO16.reshape(B * 16, Cc), B, 16, heads, S)
    dq32 = dq32.view(B, 32, Cc)
    assert torch.equal(dq32[:, 16:], dq32[:, :16])
    assert torch.equal(dq32[:, :16], dq16.view(B, 16, Cc))


# ------------------------------------------------------------------------------------------ step by step against float64
CASES = {
    # both query blocks of the tensor-core kernels, the second one partly (17) and fully (32) occupied
    "tiny_traj_q17_p0.1": ("dec_tiny_traj", dict(Q=17), 2, 0.1),
    "tiny_traj_q32_p0.1": ("dec_tiny_traj", dict(Q=32), 2, 0.1),
    "tiny_notraj_q32_p0": ("dec_tiny_notraj", dict(Q=32), 4, 0.0),
    # T * n = 60 keys, not a multiple of 8: a partial last key block in both query blocks (the forward takes dropout
    # only for multiples of 8 keys; test_cross_attention_backward runs the SIMT backward at 24 and 32 queries)
    "tiny_traj_n20_q32_p0": ("dec_tiny_traj", dict(Q=32, n=20), 2, 0.0),
    "c4_q32_b3_p0.1": (C4, dict(Q=32), 3, 0.1),
    # R = 2048 query rows: split-K weight gradients; B*S = 65536: the CTA-pair memory-side GEMMs
    "c4_q32_b64_p0.1": (C4, dict(Q=32), 64, 0.1),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_decoder_training_step_against_float64(case):
    base, patch, B, p = CASES[case]
    _run_case(_cfg(base, patch), B, 60 + list(CASES).index(case), p).finish(case)


# ------------------------------------------------------------------------------------------ module against the oracle
@pytest.mark.gpu
def test_decoder_backward_tiny_q32():
    ref, params = _decoder_grads_case(_cfg("dec_tiny_traj", dict(Q=32)), 2, 31, dropout_p=0.1)
    _check_grads(ref, params, tol_cos=0.99, tol_rel=0.15)


@pytest.mark.gpu
def test_decoder_dropout_c4_geometry_q32():
    ref, params = _decoder_grads_case(dict(C4, Q=32), 3, 79, dropout_p=0.1)
    _check_grads(ref, params)


@pytest.mark.gpu
@pytest.mark.parametrize("name,B", [("dec_c4", 2), ("dec_c2", 1)])
def test_decoder_eval_l14_q32_against_oracle(name, B):
    """ObjDecoder(num_queries=32) inference on L/14-sized features (F = 1024, 256 patches): T = 4 with the trajectory
    head (c4) and T = 16 without (c2).  Box L1 <= 1e-2 against the oracle, as for the golden geometries; a bf16
    image_feature_map[:, 1:] view gives the fp32 hand-over's outputs bit for bit."""
    from test_gpu_feature_map_bf16 import _check_decoder_eval, _decoder
    cfg = dict(gc.CASES[name]["cfg"], Q=32)
    sd = gc.decoder_state_dict(dict(cfg=cfg, seed=300 + B))
    g = torch.Generator().manual_seed(301 + B)
    feats = torch.randn(B, cfg["T"], cfg["n"], cfg["F"], generator=g)
    dec = _decoder(cfg)
    dec.load_state_dict(sd, strict=True)
    dec = dec.cuda().eval()
    with torch.no_grad():
        out, hs, _, _ = dec(feats.cuda())
        rout, rhs, _, _ = O.decoder_forward(feats, sd, heads=cfg["heads"], pred_traj=cfg["pred_traj"])
    assert out["pred_boxes"].shape == rout["pred_boxes"].shape and hs.shape == rhs.shape
    assert (out["pred_boxes"].cpu() - rout["pred_boxes"]).abs().max().item() <= 1e-2
    for a, b in zip(out["aux_outputs"], rout["aux_outputs"]):
        assert (a["pred_boxes"].cpu() - b["pred_boxes"]).abs().max().item() <= 1e-2
    _check_decoder_eval(cfg, feats.cuda(), sd)


@pytest.mark.gpu
def test_train_step_nq31_matches_oracle_autograd():
    """test_gpu_train_step at --num_queries 31 (Q = 32), decoder in train() with dropout 0.1: hands on queries 0:2,
    objects on 2:31, WordContrastiveLoss on the 31 query embeddings.  Box and noun assignments equal the oracle's; losses
    and gradients within that test's tolerances."""
    from test_gpu_train_step import _inputs
    from helping_hand_for_egocentric_videos_b200.model import LaviLa, box_utils, loss, metric, tfm_decoder as D
    drop = {"p": 0.1, "seed": 0xBEEF4321, "offset": 0}
    B, T, img, R, V, nq = 4, 4, 56, 5, 40, 31
    Q = nq + 1
    enc = dict(img=img, patch=14, D=128, L=2, H=2, T=T, text_width=768, text_heads=12, text_layers=1, vocab=128)
    dec_cfg = dict(C=128, heads=2, layers=2, ffn=256, Q=Q, n=16, T=T, F=128, ncls=30, pred_traj=True)
    bsd = gc.backbone_state_dict(dict(cfg=enc, seed=111))
    dsd = gc.decoder_state_dict(dict(cfg=dec_cfg, seed=112))
    inp = _inputs(B, T, img, R, V, torch.Generator().manual_seed(113))
    eot = inp["tokens"].argmax(-1)
    wd = {"loss_bbox_hand_boxes": 5, "loss_bbox_obj_boxes": 5, "loss_giou_hand_boxes": 2, "loss_giou_obj_boxes": 2}

    # ---------------- oracle / autograd
    ref = {k: v.clone().requires_grad_(True) for k, v in dsd.items()}
    with torch.no_grad():
        bo = O.clip_forward(inp["video"], inp["tokens"], bsd, heads=2, text_heads=12)
    grid = bo["image_feature_map"][:, 1:].unflatten(1, (T, 16))
    out, hs, _, _ = O.decoder_forward(grid, ref, heads=2, pred_traj=True, dropout=drop)
    txt = O.txt_proj(bo["text_feature_map"][torch.arange(B * R), eot], ref)
    vid = O.obj_proj(hs[-1], ref)[:, -1]
    nce, _ = O.egonce_loss(O.sim_matrix(txt, vid), O.sim_matrix(inp["verb"], inp["verb"]),
                           O.sim_matrix(inp["noun"], inp["noun"]), inp["pad"])
    lh, idx_h = O.box_loss(out["pred_boxes"], inp["px"][:, :2], 0, 2)
    lo_, idx_o = O.box_loss(out["pred_boxes"], inp["px"][:, 2:], 2, nq)
    word, cols = O.word_contrastive_loss(O.txt_proj(inp["noun_feats"], ref), O.obj_proj(hs[-1], ref)[:, :-1], inp["inds"])
    total = nce + lh + lo_ + 0.5 * word
    total.backward()

    # ---------------- CUDA mirrors
    vis = LaviLa.SpaceTimeTransformer(img_size=img, patch_size=14, embed_dim=128, depth=2, num_heads=2, num_frames=T,
                                      time_init='zeros', ln_pre=True, act_layer=LaviLa.QuickGELU)
    vis.head = torch.nn.Identity()
    clip = LaviLa.CLIP(embed_dim=256, vision_width=128, vision_model=vis, context_length=77, vocab_size=128,
                       transformer_width=768, transformer_heads=12, transformer_layers=1)
    clip.load_state_dict(bsd, strict=True)
    clip = clip.cuda().eval()
    for p in clip.parameters():
        p.requires_grad = False
    tr = D.Cross_Attention(d_model=128, nhead=2, num_decoder_layers=2, dim_feedforward=256, normalize_before=True,
                           return_intermediate_dec=True)
    model = D.ObjDecoder(transformer=tr, num_classes=30, num_queries=Q, aux_loss=True, pred_traj=True, feature_dim=128,
                         num_frames=T, patches_per_frame=16)
    model.load_state_dict(dsd, strict=True)
    model = model.cuda().train()
    model.dropout_seed, model._drop_step = drop["seed"], drop["offset"]
    crit = box_utils.SetCriterion(22047, matcher=box_utils.build_matcher(None), weight_dict=wd, eos_coef=0.1,
                                  losses=["boxes", "cardinality"]).cuda()
    dev = {k: v.cuda() for k, v in inp.items()}
    with torch.no_grad():
        o2 = clip(dev["video"], dev["tokens"], return_feature_map=True)
    grid2 = o2["image_feature_map"][:, 1:].unflatten(1, (T, 16))
    mo, hs2, _, _ = model(grid2)
    txt2 = model.txt_proj(o2["text_feature_map"][torch.arange(B * R), dev["tokens"].argmax(-1)])
    emb2 = model.obj_proj(hs2[-1])
    sim2 = metric.sim_matrix(txt2, emb2[:, -1].contiguous())
    nce2, _ = loss.EgoNCE()(sim2, metric.sim_matrix(dev["verb"], dev["verb"]), metric.sim_matrix(dev["noun"], dev["noun"]),
                            multi_pad_mask=dev["pad"], strict_mask=True)
    sizes = torch.full((B * T, 2), 224.0, device="cuda")
    lh2, idx_h2 = box_utils.compute_box_loss('hand_boxes', crit, mo, dev["px"][:, :2].clone(), None, sizes, n_queries=nq)
    lo2, idx_o2 = box_utils.compute_box_loss('obj_boxes', crit, mo, dev["px"][:, 2:].clone(), None, sizes, n_queries=nq)
    wl = loss.WordContrastiveLoss()
    word2 = wl(model.txt_proj(dev["noun_feats"]), emb2[:, :-1].contiguous(), dev["inds"])
    total2 = nce2 + lh2 + lo2 + 0.5 * word2
    total2.backward()
    assert model.last_dropout == drop
    assert emb2.shape == (B, Q, 256) and mo["pred_boxes"].shape == (B * T, Q, 4)

    for got, want in ((idx_h2, idx_h), (idx_o2, idx_o)):
        assert len(got) == len(want)
        for (gs, gt), (ws, wt) in zip(got, want):
            assert torch.equal(torch.as_tensor(gs).long(), torch.as_tensor(ws).long())
            assert torch.equal(torch.as_tensor(gt).long(), torch.as_tensor(wt).long())
    col = wl.last_col_ind.cpu()
    with_nouns = [b for b in range(B) if bool((inp["inds"][b] != 0).any())]
    assert len(with_nouns) == len(cols)
    for b, want in zip(with_nouns, cols):
        assert torch.equal(col[b][inp["inds"][b] != 0], want)
    for a, b, nm in ((nce2, nce, "nce"), (lh2, lh, "hand"), (lo2, lo_, "obj"), (word2, word, "word")):
        assert abs(a.item() - b.item()) <= 2e-2 * max(1.0, abs(b.item())), (nm, a.item(), b.item())
    bad = []
    for k, p in model.named_parameters():
        want = ref[k].grad
        if want is None or want.abs().max() == 0:
            assert p.grad is None or p.grad.abs().max().item() <= 1e-6, k
            continue
        assert p.grad is not None, k
        cos = F.cosine_similarity(p.grad.float().cpu().reshape(want.shape).flatten(), want.flatten(), dim=0).item()
        if cos < 0.99:
            bad.append((k, round(cos, 4)))
    assert not bad, bad


# ------------------------------------------------------------------------------------------ refusals
def _decoder_cfg(L, Q):
    return L.DecoderCfg(512, 8, 6, 2048, Q, 22048, 1024, 4, 256, 1)


def test_decoder_create_accepts_32_queries_without_a_gpu():
    """The configuration check is host logic: Q = 32 is accepted, Q = 33 refused, with or without a device."""
    import __graft_entry__ as g
    g.build()
    from helping_hand_for_egocentric_videos_b200 import _lib as L
    lib = L.load()
    h = C.c_void_p()
    assert lib.hh_decoder_create(C.byref(h), C.byref(_decoder_cfg(L, 32))) == 0, L.last_error()
    lib.hh_decoder_destroy(h)
    h2 = C.c_void_p()
    assert lib.hh_decoder_create(C.byref(h2), C.byref(_decoder_cfg(L, 33))) == -2
    assert "1..32 queries" in L.last_error()


@pytest.mark.gpu
def test_refusals_before_any_launch():
    """Q = 33 at every kernel entry point and Q = 17 at the 16-query SIMT forward return -2 from the host check: the
    outputs keep their sentinel and the stream holds no error."""
    from helping_hand_for_egocentric_videos_b200 import _lib as L
    lib = L.load()
    h = C.c_void_p()
    assert lib.hh_decoder_create(C.byref(h), C.byref(_decoder_cfg(L, 33))) == -2
    B, heads, S = 2, 2, 64
    Cc = heads * 64
    st = L.stream_ptr()

    def bufs(Q):
        q = torch.randn(B * Q, 3 * Cc, device="cuda") * 0.3
        K = torch.randn(B * S, Cc, device="cuda").bfloat16()
        V = torch.randn(B * S, Cc, device="cuda").bfloat16()
        return q, K, V, torch.full((B * Q, 3 * Cc), float("nan"), device="cuda")

    def untouched(out):
        torch.cuda.synchronize()
        assert bool(out.isnan().all())
    q, K, V, out = bufs(33)
    assert lib.hh_cross_attention(L.ptr(q), L.ptr(K), L.ptr(V), Cc, L.ptr(out), B, 33, heads, S, st) == -2
    assert "1..32 queries" in L.last_error()
    untouched(out)
    dK, dV = torch.full_like(K, float("nan")), torch.full_like(V, float("nan"))
    assert lib.hh_cross_attention_backward(L.ptr(q), L.ptr(K), L.ptr(V), Cc, L.ptr(q), L.ptr(q), L.ptr(out), L.ptr(dK),
                                           L.ptr(dV), Cc, B, 33, heads, S, st) == -2
    assert "1..32 queries" in L.last_error()
    untouched(out)
    assert bool(dK.isnan().all()) and bool(dV.isnan().all())
    p, po = L.ptr(q), L.ptr(out)
    assert lib.hh_self_attention_backward(p, p + 4 * Cc, p + 8 * Cc, 3 * Cc, p, po, po + 4 * Cc, po + 8 * Cc, 3 * Cc,
                                          B, 33, heads, st) == -2
    assert "1..32 queries" in L.last_error()
    untouched(out)
    q, K, V, out = bufs(17)
    assert lib.hh_cross_attention_simt(L.ptr(q), L.ptr(K), L.ptr(V), Cc, L.ptr(out), B, 17, heads, S, st) == -2
    assert "1..16 queries" in L.last_error()
    untouched(out)
