"""Backward kernels of the decoder (SURVEY.md section 8f row 2) against torch autograd on the same fp32 statement of
each operator, through the C ABI.  fp32 kernels: rel 2e-5 (different summation order); the cross-attention backward
reads bf16 K/V and writes bf16 dK/dV: compared on the same bf16-rounded inputs, output rounding 2^-8."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _ops():
    from helping_hand_for_egocentric_videos_b200 import ops
    return ops


def _close(got, want, name, rtol=2e-5, atol=None):
    got, want = got.detach().float().cpu(), want.detach().float().cpu()
    assert got.shape == want.shape, (name, got.shape, want.shape)
    err = (got - want).abs().max().item()
    lim = (atol if atol is not None else 0.0) + rtol * max(1.0, want.abs().max().item())
    assert err <= lim, (name, err, lim)


@pytest.mark.parametrize("R,N,K,act,add,in_relu", [(65, 512, 512, 0, True, False), (832, 2048, 512, 1, False, False),
                                                   (100, 4, 512, 2, False, False), (37, 256, 768, 0, False, True),
                                                   (5, 40, 24, 1, True, False), (70, 30, 64, 1, True, False)])
def test_linear_backward(R, N, K, act, add, in_relu):
    """N = 30 (not a multiple of 4) runs both gradients on the first-generation kernels instead of lin3_kernel."""
    g = torch.Generator().manual_seed(R + N)
    x = torch.randn(R, K, generator=g)
    w = torch.randn(N, K, generator=g) / K ** 0.5
    b = torch.randn(N, generator=g) * 0.1
    xa = torch.randn(13 if R >= 13 else R, K, generator=g) if add else None
    dy = torch.randn(R, N, generator=g)
    x0, w0, b0 = x.clone().requires_grad_(True), w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    xin = x0 + (xa.repeat((R + xa.shape[0] - 1) // xa.shape[0], 1)[:R] if add else 0)
    if in_relu:
        xin = F.relu(xin)
    y = F.linear(xin, w0, b0)
    y = F.relu(y) if act == 1 else (torch.sigmoid(y) if act == 2 else y)
    y.backward(dy)
    dx, dw, db = _ops().linear_f32_backward(dy.cuda(), y.detach().cuda(), act, w.cuda(), x.cuda(),
                                            xa.cuda() if add else None, in_relu)
    _close(dw, w0.grad, "dw", 5e-5)
    _close(db, b0.grad, "db", 5e-5)
    if not in_relu:          # the kernel returns d(relu(x)) there; the caller applies the mask
        _close(dx, x0.grad, "dx", 5e-5)


@pytest.mark.parametrize("M,D", [(832, 512), (3000, 1024), (7, 128)])
def test_layernorm_backward(M, D):
    g = torch.Generator().manual_seed(M)
    x = torch.randn(M, D, generator=g) * 2 + 0.3
    w = 1 + 0.1 * torch.randn(D, generator=g)
    b = 0.1 * torch.randn(D, generator=g)
    dy = torch.randn(M, D, generator=g)
    x0, w0, b0 = x.clone().requires_grad_(True), w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    F.layer_norm(x0, (D,), w0, b0, 1e-5).backward(dy)
    dx, dg, db = _ops().layernorm_backward(x.cuda(), w.cuda(), dy.cuda(), 1e-5)
    _close(dx, x0.grad, "dx", 5e-5)
    _close(dg, w0.grad, "dgamma", 1e-4)
    _close(db, b0.grad, "dbeta", 1e-4)


@pytest.mark.parametrize("B,Q,heads", [(3, 13, 8), (2, 5, 2), (1, 16, 1), (4, 1, 2)])
def test_self_attention_backward(B, Q, heads):
    g = torch.Generator().manual_seed(B * 10 + Q)
    Cc = heads * 64
    qkv = torch.randn(B * Q, 3 * Cc, generator=g) * 0.5
    dO = torch.randn(B * Q, Cc, generator=g)
    t = qkv.clone().requires_grad_(True)
    x = t.view(B, Q, 3, heads, 64).permute(2, 0, 3, 1, 4)
    o = (torch.softmax(x[0] @ x[1].transpose(-1, -2), -1) @ x[2]).permute(0, 2, 1, 3).reshape(B * Q, Cc)
    o.backward(dO)
    got = _ops().self_attention_backward(qkv.cuda(), dO.cuda(), B, Q, heads)
    _close(got, t.grad, "dqkv", 5e-5)


@pytest.mark.parametrize("B,Q,heads,S", [(2, 13, 8, 1024), (1, 5, 2, 196), (3, 13, 2, 77), (1, 16, 1, 300)])
def test_cross_attention_backward(B, Q, heads, S):
    g = torch.Generator().manual_seed(S + Q)
    Cc = heads * 64
    q = torch.randn(B * Q, Cc, generator=g) * 0.3
    K = torch.randn(B * S, Cc, generator=g).to(torch.bfloat16)
    V = torch.randn(B * S, Cc, generator=g).to(torch.bfloat16)
    dO = torch.randn(B * Q, Cc, generator=g)
    q0, K0, V0 = q.clone().requires_grad_(True), K.float().requires_grad_(True), V.float().requires_grad_(True)
    qh = q0.view(B, Q, heads, 64).transpose(1, 2)
    kh, vh = K0.view(B, S, heads, 64).transpose(1, 2), V0.view(B, S, heads, 64).transpose(1, 2)
    O = (torch.softmax(qh @ kh.transpose(-1, -2), -1) @ vh).transpose(1, 2).reshape(B * Q, Cc)
    O.backward(dO)
    dq, dK, dV = _ops().cross_attention_backward(q.cuda(), K.cuda(), V.cuda(), O.detach().cuda(), dO.cuda(), B, Q, heads, S)
    _close(dq, q0.grad, "dq", 1e-4)
    _close(dK, K0.grad, "dK", 2 ** -7, atol=1e-4)
    _close(dV, V0.grad, "dV", 2 ** -7, atol=1e-4)
    # q and dO 4 bytes off an 8-byte boundary: the tensor-core kernel does not take them, the SIMT kernels do
    def off8(t):
        flat = torch.empty(t.numel() + 1, device="cuda")
        flat[1:] = t.flatten().cuda()
        return flat[1:].view(t.shape)
    qu, dOu = off8(q), off8(dO)
    assert qu.data_ptr() % 8 != 0 and dOu.data_ptr() % 8 != 0
    dq, dK, dV = _ops().cross_attention_backward(qu, K.cuda(), V.cuda(), O.detach().cuda(), dOu, B, Q, heads, S)
    _close(dq, q0.grad, "dq (SIMT)", 1e-4)
    _close(dK, K0.grad, "dK (SIMT)", 2 ** -7, atol=1e-4)
    _close(dV, V0.grad, "dV (SIMT)", 2 ** -7, atol=1e-4)


# ------------------------------------------------------------------------------------------ whole-decoder backward
def _decoder_grads_case(cfg, B, seed, dropout_p=0.0):
    """Gradients of a random linear functional of (hs, all layers' boxes, obj_proj embeddings) w.r.t. every decoder
    parameter: hand-written backward (hh_decoder_backward via autograd.Function) against autograd through the oracle.
    dropout_p > 0: the module runs in train() mode (the reference's training mode, dropout at six sites per layer) and
    the oracle graph is run with the very masks the engine drew (oracle philox_keep restates csrc/hh_rng.cuh)."""
    from oracle import hh_oracle as O
    from helping_hand_for_egocentric_videos_b200.model import tfm_decoder as D
    c = cfg
    shapes = O.decoder_param_shapes(c["C"], c["Q"], c["n"], c["T"], c["F"], c["ncls"] + 1, layers=c["layers"], ffn=c["ffn"],
                                    pred_traj=c["pred_traj"])
    sd = O.synth_state_dict(shapes, seed)
    g = torch.Generator().manual_seed(seed + 1)
    feats = torch.randn(B, c["T"], c["n"], c["F"], generator=g)
    Tb = c["T"] if c["pred_traj"] else 1
    w_hs = torch.randn(c["layers"], B, c["Q"], c["C"], generator=g)
    w_box = torch.randn(c["layers"], B * Tb, c["Q"], 4, generator=g)
    w_emb = torch.randn(B, c["Q"], 256, generator=g)

    # CUDA side
    tr = D.Cross_Attention(d_model=c["C"], nhead=c["heads"], num_decoder_layers=c["layers"], dim_feedforward=c["ffn"],
                           dropout=dropout_p if dropout_p > 0 else 0.1, normalize_before=True, return_intermediate_dec=True)
    dec = D.ObjDecoder(transformer=tr, num_classes=c["ncls"], num_queries=c["Q"], aux_loss=True, pred_traj=c["pred_traj"],
                       feature_dim=c["F"], num_frames=c["T"], patches_per_frame=c["n"])
    dec.load_state_dict(sd, strict=True)
    dec = dec.cuda()
    if dropout_p > 0:
        dec.train()
        dec.dropout_seed = 0x1234ABCD5678 + seed
        dec._drop_step = 3
    else:
        dec.eval()                          # eval: the inference arithmetic, no dropout
    o2, hs2, _, _ = dec(feats.cuda())
    boxes2 = torch.stack([a["pred_boxes"] for a in o2["aux_outputs"]] + [o2["pred_boxes"]])
    loss2 = (hs2 * w_hs.cuda()).sum() + (boxes2 * w_box.cuda()).sum() + (dec.obj_proj(hs2[-1]) * w_emb.cuda()).sum()
    loss2.backward()
    drop = dec.last_dropout
    assert (drop is not None) == (dropout_p > 0)

    # oracle side (same dropout masks)
    ref = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    out, hs, _, _ = O.decoder_forward(feats, ref, heads=c["heads"], pred_traj=c["pred_traj"], dropout=drop)
    boxes = torch.stack([a["pred_boxes"] for a in out["aux_outputs"]] + [out["pred_boxes"]])
    loss = (hs * w_hs).sum() + (boxes * w_box).sum() + (O.obj_proj(hs[-1], ref) * w_emb).sum()
    loss.backward()
    assert abs(loss2.item() - loss.item()) <= 2e-2 * max(1.0, abs(loss.item()))
    hs_err = (hs2.detach().cpu() - hs.detach()).abs().max().item()
    assert hs_err <= 3e-2, hs_err             # a single mismatched mask element would show up at the 0.1 .. 1 level
    return ref, dict(dec.named_parameters())


def _check_grads(ref, params, tol_cos=0.995, tol_rel=0.1):
    """Per-tensor cosine >= 0.995 and relative L2 error <= 10 % against fp32 autograd.  The forward runs its memory side
    in bf16 (the reference trains under fp16 autocast), so a few ReLU units near zero take the other branch than in the
    fp32 oracle: whole gradient rows of the weights in front of a ReLU then differ, which bounds the achievable
    max-norm agreement; direction and norm of every gradient tensor are what is asserted."""
    worst = (1.0, None)
    bad = []
    for k, p in params.items():
        want = ref[k].grad
        if k.startswith(("txt_proj.", "vid_proj.")):
            assert p.grad is None or float(p.grad.abs().max()) == 0.0
            continue
        if k.startswith("class_embed."):
            assert p.grad is not None and float(p.grad.abs().max()) == 0.0      # no class loss in the graph
            continue
        assert p.grad is not None, k
        got = p.grad.detach().float().cpu().reshape(want.shape)
        scale = want.abs().max().item()
        if scale == 0.0:
            assert got.abs().max().item() <= 1e-6, k
            continue
        cos = F.cosine_similarity(got.flatten(), want.flatten(), dim=0).item()
        rel = ((got - want).norm() / want.norm()).item()
        if cos < worst[0]:
            worst = (cos, k)
        if not (cos >= tol_cos and rel <= tol_rel):
            bad.append((k, round(cos, 5), round(rel, 4)))
    assert not bad, bad
    return worst


@pytest.mark.parametrize("name", ["dec_tiny_traj", "dec_tiny_notraj"])
def test_decoder_backward_tiny(name):
    from oracle import golden_cases as gc
    case = gc.CASES[name]
    B = 2 if name == "dec_tiny_traj" else 4            # clips x patch tokens must be a multiple of 8
    ref, params = _decoder_grads_case(case["cfg"], B, case["seed"])
    _check_grads(ref, params, tol_cos=0.99, tol_rel=0.15)     # 60-150 rows only: one flipped ReLU unit is visible


def test_decoder_backward_c4_geometry():
    """BASELINE c4 decoder geometry (C=512, 8 heads, 6 layers, nq=12 -> Q=13, 4 frames x 256 patches of 1024-d
    features, trajectory head) on 3 clips."""
    cfg = dict(C=512, heads=8, layers=6, ffn=2048, Q=13, n=256, T=4, F=1024, ncls=63, pred_traj=True)
    ref, params = _decoder_grads_case(cfg, 3, 77)
    _check_grads(ref, params)


# ------------------------------------------------------------------------------------------ training-mode dropout
@pytest.mark.parametrize("name", ["dec_tiny_traj", "dec_tiny_notraj"])
def test_decoder_dropout_forward_backward_tiny(name):
    """train() mode, p = 0.1 (the reference's Cross_Attention default): outputs and every parameter gradient against the
    oracle graph run with the same masks."""
    from oracle import golden_cases as gc
    case = gc.CASES[name]
    B = 2 if name == "dec_tiny_traj" else 4
    ref, params = _decoder_grads_case(case["cfg"], B, case["seed"], dropout_p=0.1)
    _check_grads(ref, params, tol_cos=0.99, tol_rel=0.15)


def test_decoder_dropout_c4_geometry():
    """BASELINE c4 decoder geometry in training mode with dropout 0.1 (run/train.py trains the decoder in train())."""
    cfg = dict(C=512, heads=8, layers=6, ffn=2048, Q=13, n=256, T=4, F=1024, ncls=63, pred_traj=True)
    ref, params = _decoder_grads_case(cfg, 3, 78, dropout_p=0.1)
    _check_grads(ref, params)


def test_decoder_dropout_stream_semantics():
    """eval() never drops; train() draws a new mask every step (offset advances), the same (seed, step) reproduces the
    same output bit for bit, and a large p visibly changes the result."""
    from oracle import hh_oracle as O
    from oracle import golden_cases as gc
    from helping_hand_for_egocentric_videos_b200.model import tfm_decoder as D
    c = gc.CASES["dec_tiny_traj"]["cfg"]
    sd = O.synth_state_dict(O.decoder_param_shapes(c["C"], c["Q"], c["n"], c["T"], c["F"], c["ncls"] + 1, layers=c["layers"],
                                                   ffn=c["ffn"], pred_traj=c["pred_traj"]), 5)
    tr = D.Cross_Attention(d_model=c["C"], nhead=c["heads"], num_decoder_layers=c["layers"], dim_feedforward=c["ffn"],
                           dropout=0.3, normalize_before=True, return_intermediate_dec=True)
    dec = D.ObjDecoder(transformer=tr, num_classes=c["ncls"], num_queries=c["Q"], aux_loss=True, pred_traj=c["pred_traj"],
                       feature_dim=c["F"], num_frames=c["T"], patches_per_frame=c["n"])
    dec.load_state_dict(sd, strict=True)
    dec = dec.cuda()
    x = torch.randn(2, c["T"], c["n"], c["F"], generator=torch.Generator().manual_seed(6)).cuda()
    with torch.no_grad():
        dec.eval()
        e1 = dec(x)[1].clone()
        e2 = dec(x)[1].clone()
        assert torch.equal(e1, e2) and dec.last_dropout is None
        dec.train()
        dec.dropout_seed, dec._drop_step = 99, 0
        t1 = dec(x)[1].clone()
        assert dec.last_dropout == {"p": 0.3, "seed": 99, "offset": 0}
        t2 = dec(x)[1].clone()
        assert dec.last_dropout["offset"] == 1
        dec._drop_step = 0
        t3 = dec(x)[1].clone()
    assert torch.equal(t1, t3)
    assert not torch.equal(t1, t2)
    assert (t1 - e1).abs().max().item() > 1e-2


def test_decoder_dropout_against_reference_fixture():
    """The CUDA decoder in train() mode against tests/golden/dec_train_dropout.pt: outputs and parameter gradients of the
    UNMODIFIED reference run with the same dropout masks (oracle/make_golden.py injects hh_oracle.philox_keep through
    torch.nn.functional.dropout)."""
    import os
    from oracle import golden_cases as gc
    from helping_hand_for_egocentric_videos_b200.model import tfm_decoder as D
    case = gc.CASES["dec_train_dropout"]
    c, dr = case["cfg"], case["dropout"]
    ref = torch.load(os.path.join(gc.GOLDEN_DIR, "dec_train_dropout.pt"))
    tr = D.Cross_Attention(d_model=c["C"], nhead=c["heads"], num_decoder_layers=c["layers"], dim_feedforward=c["ffn"],
                           dropout=dr["p"], normalize_before=True, return_intermediate_dec=True)
    dec = D.ObjDecoder(transformer=tr, num_classes=c["ncls"], num_queries=c["Q"], aux_loss=True, pred_traj=c["pred_traj"],
                       feature_dim=c["F"], num_frames=c["T"], patches_per_frame=c["n"])
    dec.load_state_dict(gc.decoder_state_dict(case), strict=True)
    dec = dec.cuda().train()
    dec.dropout_seed, dec._drop_step = dr["seed"], dr["offset"]


    def fwd(feats):
        out, hs, _, _ = dec(feats.cuda())
        out = {"pred_boxes": out["pred_boxes"].cpu(), "aux_outputs": [{"pred_boxes": a["pred_boxes"].cpu()} for a in out["aux_outputs"]]}
        return out, hs.cpu()
    got = gc.train_functional(case, fwd, lambda h: dec.obj_proj(h.cuda()).cpu(), dict(dec.named_parameters()))
    assert dec.last_dropout == {"p": dr["p"], "seed": dr["seed"], "offset": dr["offset"]}
    assert (got["hs"] - ref["hs"]).abs().max().item() <= 3e-2
    assert (got["boxes"] - ref["boxes"]).abs().max().item() <= 1e-2                      # box L1 gate
    assert F.cosine_similarity(got["embed"].flatten(1), ref["embed"].flatten(1), dim=-1).min().item() >= 0.999
    assert abs(got["loss"].item() - ref["loss"].item()) <= 2e-2 * max(1.0, abs(ref["loss"].item()))
    bad = []
    for k, v in ref.items():
        if not k.startswith("gnorm/"):
            continue
        name = k[len("gnorm/"):]
        if name.startswith("class_embed.") or v.item() == 0.0:       # no class loss in the graph / unused parameters
            assert got[k].item() <= 1e-6, name
            continue
        rel = abs(got[k].item() - v.item()) / v.item()
        sub_ref, sub_got = ref["grad/" + name], got["grad/" + name].cpu()
        cos = F.cosine_similarity(sub_got.flatten(), sub_ref.flatten(), dim=0).item() if sub_ref.norm() > 0 else 1.0
        # 64-element subsamples of 10-row problems: one ReLU unit that takes the other branch under the bf16 memory side
        # moves a subsample's cosine by a few per cent (see _check_grads); the norm is held to 15 %
        if rel > 0.15 or cos < 0.95:
            bad.append((name, round(rel, 4), round(cos, 4)))
    assert not bad, bad
