"""The decoder's training step, one kernel step at a time, against float64.

`ObjDecoder` runs its normal training path (`_DecoderFn` -> hh_decoder_forward_train / hh_decoder_backward_checked) on
a random linear functional of hs, all layers' boxes and obj_proj(hs[-1]).  Between the forward and `backward()` the
test reads what the engine saved (hh_decoder_get_saved) and recomputes every saved tensor in float64 from the engine's
PREVIOUS saved tensor.  The float64 backward is then evaluated at the engine's own activations: each recomputed
tensor is pinned to the engine's value (`_pin`: the engine's value forward, the reference's derivative backward).

Wherever the engine made a discrete choice, the reference takes it from the saved tensors: the dropout masks
(hh_oracle.philox_keep, restated on the GPU by `_keep` and checked against it), the FFN and bbox ReLU decisions
(`f > 0`, `box_x1 > 0`, `box_x2 > 0`) and the bf16 roundings the engine documents (proj and the K / V projection
weights and activations in the forward; dK, dV and the pre_norm input gradient in the backward).  What is left is
summation order, so the tolerances are those of the per-kernel tests:

  forward     fp32 steps 1e-5; self attention 5e-5; cross attention 2^-7 rel + 4e-3 (P is rounded to bf16 for P.V);
              bf16 steps (mem, mempos, k, v) within one bf16 ulp of the float64 value, at most 1 % of them not the
              nearest bf16
  backward    query side (fp32 end to end: 3xTF32 linears, fp32 attention backward): max error <= 3e-5 max|ref|,
              measured worst 6.4e-6 (test_cross_attention_backward holds dq to 1e-4);
              memory side: relative L2 <= 2^-7 and max error <= 2^-7 max|ref| per tensor, measured worst 3.9e-3
              (~2^-8.0, proj.weight, tiny geometry) and 4.4e-3 max|ref|.  The cross-attention backward forms dK / dV
              from bf16 operands before it writes them in bf16 (test_cross_attention_backward holds them to 2^-7), so
              2^-8 would sit at the measured error.  Sums of dK that cancel (the K biases, exactly zero in exact
              arithmetic, and the position embeddings) are held elementwise to 2^-8 of the sum of the terms'
              magnitudes, measured worst 0.41 of that bound

Every case prints the worst error / bound ratio of each tolerance class (pytest -s shows it).
"""
import math

import pytest
import torch
import torch.nn.functional as F

C4 = dict(C=512, heads=8, layers=6, ffn=2048, Q=13, n=256, T=4, F=1024, ncls=63, pred_traj=True)


# ------------------------------------------------------------------------------------------ dropout masks
def _keep(drop, site, shape, device="cuda"):
    """oracle.hh_oracle.philox_keep (Philox4x32-10, csrc/hh_rng.cuh) in int64 torch ops: multipliers 0 or fp32(1/(1-p))
    in float64, row-major over `shape`; None without dropout.  64-bit products wrap, so only their low 32 bits of each
    half are used, as in the 32-bit reference."""
    if drop is None:
        return None
    numel = math.prod(shape)
    M = 0xFFFFFFFF
    idx = torch.arange(numel, dtype=torch.int64, device=device)
    c0, c1 = (idx >> 3) & M, (idx >> 35) & M
    c2 = torch.full_like(idx, site)
    c3 = torch.full_like(idx, drop["offset"])
    k0, k1 = drop["seed"] & M, (drop["seed"] >> 32) & M
    for _ in range(10):
        p0, p1 = c0 * 0xD2511F53, c2 * 0xCD9E8D57
        c0, c1, c2, c3 = ((p1 >> 32) & M) ^ c1 ^ k0, p1 & M, ((p0 >> 32) & M) ^ c3 ^ k1, p0 & M
        k0, k1 = (k0 + 0x9E3779B9) & M, (k1 + 0xBB67AE85) & M
    words = torch.stack([c0, c1, c2, c3], 1)
    lane = idx & 7
    w = words.gather(1, (lane >> 1)[:, None])[:, 0]
    r = (w >> (16 * (lane & 1))) & 0xFFFF
    thr = max(1, int(drop["p"] * 65536.0 + 0.5))
    scale = torch.tensor(1.0 / (1.0 - drop["p"]), dtype=torch.float32).item()      # the engine's fp32 1/(1-p)
    return ((r >= thr).double() * scale).view(shape)


def test_keep_matches_oracle():
    """The GPU restatement of the masks draws exactly oracle.hh_oracle.philox_keep's (runs on the CPU)."""
    from oracle import hh_oracle as O
    for seed, offset, site, numel, p in [(0x1234ABCD5678, 3, 2, 5000, 0.1), (99, 0, 45, 777, 0.3), ((1 << 63) + 5, 7, 8, 64, 0.5)]:
        drop = {"p": p, "seed": seed, "offset": offset}
        want = O.philox_keep(seed, offset, site, numel, p).double()
        assert torch.equal(_keep(drop, site, (numel,), device="cpu"), want)


# ------------------------------------------------------------------------------------------ float64 reference pieces
def _pin(comp, saved):
    """The engine's value, with the reference's derivative."""
    return comp + (saved.double() - comp).detach()


def _bf16(t):
    return t.float().bfloat16().double()


def _w16(w):
    """A weight the engine reads as bf16: rounded forward, straight through backward."""
    return w + (_bf16(w) - w).detach()


class _GradBf16(torch.autograd.Function):
    """Identity whose backward rounds the gradient to bf16, where the engine writes that gradient in bf16."""

    @staticmethod
    def forward(ctx, x):
        return x.view_as(x)

    @staticmethod
    def backward(ctx, g):
        return _bf16(g)


class _CrossCore(torch.autograd.Function):
    """softmax(q k^T) (dropout) v per head, float64.  Backward as cross_attn_bwd states it: D = rowsum(dO * O) with the
    engine's saved O."""

    @staticmethod
    def forward(ctx, q, k, v, keep, o_saved):
        p = torch.softmax(q @ k.transpose(-1, -2), -1)
        ctx.save_for_backward(q, k, v, p, keep, o_saved)
        return (p if keep is None else p * keep) @ v

    @staticmethod
    def backward(ctx, do):
        q, k, v, p, keep, o = ctx.saved_tensors
        dv = (p if keep is None else p * keep).transpose(-1, -2) @ do
        dp = do @ v.transpose(-1, -2)
        if keep is not None:
            dp = dp * keep
        ds = p * (dp - (do * o).sum(-1, keepdim=True))
        return ds @ k, ds.transpose(-1, -2) @ q, dv, None, None


class _Tally:
    """Checks one case: keeps the worst error / bound ratio of each tolerance class and every failure, so that one run
    shows all of them (the first failing forward step is where a bug lives)."""

    def __init__(self):
        self.worst = {}
        self.bad = []

    def _note(self, cls, name, err, lim):
        r = err / lim if lim > 0 else (0.0 if err == 0 else math.inf)
        if r >= self.worst.get(cls, (-1.0,))[0]:
            self.worst[cls] = (r, name, err, lim)
        if not r <= 1.0:
            self.bad.append((cls, name, err, lim))

    def close(self, cls, name, got, want, rtol, atol=0.0, floor=1.0):
        """max |got - want| <= atol + rtol * max(floor, max|want|)"""
        got, want = got.double(), want.detach().double()
        assert got.shape == want.shape, (name, got.shape, want.shape)
        err = (got - want).abs().max().item()
        self._note(cls, name, err, atol + rtol * max(floor, want.abs().max().item()))

    def bf16(self, name, got, want):
        """bf16 `got` against the float64 `want`: every element within one bf16 ulp of `want` (plus 1e-5 max|want| for
        values that cancel to near zero in the engine's fp32 accumulation), at most 1 % of them not bf16(want)."""
        want = want.detach().double()
        nearest = want.float().bfloat16()
        ulp = torch.exp2((torch.frexp(want.float())[1] - 8).double())                     # bf16 spacing at |want|
        err = (got.double() - want).abs() / (ulp + 1e-5 * want.abs().max().item())
        self._note("bf16 steps (ulp)", name, err.max().item(), 1.0)
        self._note("bf16 steps (share not nearest)", name, (got != nearest).double().mean().item(), 0.01)

    def grad_query(self, name, got, want):
        got, want = got.double(), want.double()
        self._note("backward query side (max)", name, (got - want).abs().max().item(), 3e-5 * want.abs().max().item())

    def grad_memory(self, name, got, want):
        got, want = got.double(), want.double()
        self._note("backward memory side (rel L2)", name, ((got - want).norm() / want.norm()).item(), 2 ** -7)
        self._note("backward memory side (max)", name, (got - want).abs().max().item(), 2 ** -7 * want.abs().max().item())

    def grad_sum(self, name, got, want, mag):
        """A gradient that is a sum of bf16-rounded dK terms that cancel (exactly, for the K bias: softmax ignores a
        shift shared by all keys): |got - want| <= 2^-8 times the same sum over the terms' magnitudes, elementwise."""
        diff, lim = (got.double() - want.double()).abs(), 2 ** -8 * mag
        ratio = torch.where(lim > 0, diff / lim.clamp_min(1e-300), torch.where(diff == 0, 0.0, math.inf))
        self._note("backward memory side (sums of dK)", name, ratio.max().item(), 1.0)

    def finish(self, tag):
        for cls, (r, name, err, lim) in sorted(self.worst.items()):
            print("[%s] %-36s worst %.3g of the bound (%s: %.3g vs %.3g)" % (tag, cls, r, name, err, lim))
        assert not self.bad, self.bad


def _ln(x, ref, nm):
    return F.layer_norm(x, (x.shape[-1],), ref[nm + ".weight"], ref[nm + ".bias"], 1e-5)


def _heads(t, B, L, h):
    return t.reshape(B, L, h, 64).transpose(1, 2)


def _merge(t):
    B, h, L, d = t.shape
    return t.transpose(1, 2).reshape(B * L, h * d)


# ------------------------------------------------------------------------------------------ one training step
def _module(cfg, seed, p):
    from oracle import hh_oracle as O
    from helping_hand_for_egocentric_videos_b200.model import tfm_decoder as D
    c = cfg
    sd = O.synth_state_dict(O.decoder_param_shapes(c["C"], c["Q"], c["n"], c["T"], c["F"], c["ncls"] + 1, layers=c["layers"],
                                                   ffn=c["ffn"], pred_traj=c["pred_traj"]), seed)
    tr = D.Cross_Attention(d_model=c["C"], nhead=c["heads"], num_decoder_layers=c["layers"], dim_feedforward=c["ffn"],
                           dropout=p if p > 0 else 0.1, normalize_before=True, return_intermediate_dec=True)
    dec = D.ObjDecoder(transformer=tr, num_classes=c["ncls"], num_queries=c["Q"], aux_loss=True, pred_traj=c["pred_traj"],
                       feature_dim=c["F"], num_frames=c["T"], patches_per_frame=c["n"])
    dec.load_state_dict(sd, strict=True)
    dec = dec.cuda()
    if p > 0:
        dec.train()
        dec.dropout_seed, dec._drop_step = 0x5EED0000 + seed, 11
    else:
        dec.eval()
    return dec


def _saved(dec, name, layer, shape, dtype=torch.float32):
    from helping_hand_for_egocentric_videos_b200 import _lib as L
    t = torch.empty(shape, dtype=dtype, device="cuda")
    L.check(L.load().hh_decoder_get_saved(dec._engine(), name.encode(), layer, L.ptr(t), t.numel() * t.element_size(),
                                          L.stream_ptr()), "hh_decoder_get_saved(%s, %d)" % (name, layer))
    return t


def _engine_step(cfg, B, seed, p, stream):
    """Training step of the module on `stream`: (module, features, saved state, functional weights, hs, boxes)."""
    from helping_hand_for_egocentric_videos_b200 import ops
    c = cfg
    Lr, Q, Cd, T, S = c["layers"], c["Q"], c["C"], c["T"], c["T"] * c["n"]
    Tb = T if c["pred_traj"] else 1
    R = B * Q
    g = torch.Generator(device="cuda").manual_seed(seed + 1)
    feats = torch.randn(B, T, c["n"], c["F"], generator=g, device="cuda")
    w_hs = torch.randn(Lr, B, Q, Cd, generator=g, device="cuda")
    w_box = torch.randn(Lr, B * Tb, Q, 4, generator=g, device="cuda")
    w_emb = torch.randn(B, Q, 256, generator=g, device="cuda")
    dec = _module(cfg, seed, p)
    torch.cuda.synchronize()
    with torch.cuda.stream(stream):
        out, hs, _, _ = dec(feats)
        boxes = torch.stack([a["pred_boxes"] for a in out["aux_outputs"]] + [out["pred_boxes"]])
        loss = (hs * w_hs).sum() + (boxes * w_box).sum() + (dec.obj_proj(hs[-1]) * w_emb).sum()
        sv = {"memf": _saved(dec, "memf", -1, (B * S, Cd)),
              "mem": _saved(dec, "mem", -1, (B * S, Cd), torch.bfloat16),
              "mempos": _saved(dec, "mempos", -1, (B * S, Cd), torch.bfloat16),
              "k": _saved(dec, "k", -1, (B * S, Lr * Cd), torch.bfloat16),
              "v": _saved(dec, "v", -1, (B * S, Lr * Cd), torch.bfloat16)}
        rows_box = Lr * R * Tb
        for nm in ("box_x1", "box_x2") + (("cond",) if c["pred_traj"] else ()):
            sv[nm] = _saved(dec, nm, -1, (rows_box, Cd))
        widths = dict(x0=Cd, x1=Cd, x2=Cd, x3=Cd, n1=Cd, n2=Cd, n3=Cd, qkv=3 * Cd, o1=Cd, qc=Cd, o2=Cd, f=c["ffn"])
        for i in range(Lr):
            for nm, w in widths.items():
                sv[nm, i] = _saved(dec, nm, i, (R, w))
            sv["lse", i] = _saved(dec, "lse", i, (B * c["heads"], Q))
        # obj_proj's hidden ReLU decisions, as its native forward takes them
        sv["obj_h"] = ops.linear_f32(hs[-1].detach().reshape(R, Cd), dec.obj_proj[0].weight.detach(),
                                     dec.obj_proj[0].bias.detach(), act=1)
        loss.backward()
    torch.cuda.current_stream().wait_stream(stream)
    torch.cuda.synchronize()
    return dec, feats, sv, (w_hs, w_box, w_emb), hs.detach(), boxes.detach()


def _relu_decisions(name, kept_out, pre, keep=None):
    """The engine's ReLU (and dropout) decisions against the float64 pre-activation: exactly zero where dropped or
    where pre < -1e-4, positive where kept and pre > 1e-4."""
    if keep is not None:
        assert bool((kept_out[keep == 0] == 0).all()), name + ": a dropped unit is not zero"
    far = pre.abs() > 1e-4
    assert bool((kept_out[far & (pre < 0)] == 0).all()), name + ": a negative pre-activation passed the ReLU"
    live = far & (pre > 0)
    if keep is not None:
        live &= keep != 0
    assert bool((kept_out[live] > 0).all()), name + ": a positive kept pre-activation was zeroed"


def _run_case(cfg, B, seed, p, stream=None):
    c = cfg
    Lr, Q, Cd, T, n, h, Fd = c["layers"], c["Q"], c["C"], c["T"], c["n"], c["heads"], c["ffn"]
    S, R = T * n, B * Q
    traj = c["pred_traj"]
    dec, feats, sv, (w_hs, w_box, w_emb), hs_e, boxes_e = _engine_step(cfg, B, seed, p, stream or torch.cuda.current_stream())
    drop = dec.last_dropout
    assert (drop is not None) == (p > 0)
    t = _Tally()
    ref = {k: v.detach().double().clone().requires_grad_(True) for k, v in dec.named_parameters()}
    qs = 0.125                                                           # 64 ** -0.5, folded into the engine's Wq / bq

    # ---- memory side: proj -> pre_norm -> (mem, mem + pos) -> all layers' K / V
    feat = _bf16(feats.reshape(B * S, c["F"]))
    memf_c = feat @ _w16(ref["proj.weight"]).t()
    t.close("fp32 steps", "memf", sv["memf"], memf_c, 1e-5, floor=0.0)
    memf = _GradBf16.apply(_pin(memf_c, sv["memf"]))                    # the pre_norm input gradient is written in bf16
    mem_c = _ln(memf, ref, "transformer.pre_norm")
    pos = (ref["pos_embed"][0, 1:][None] + ref["temporal_embed"][0][:, None]).reshape(S, Cd)
    mempos_c = mem_c + pos.repeat(B, 1)
    t.bf16("mem", sv["mem"], mem_c)
    t.bf16("mempos", sv["mempos"], mempos_c)
    mem, mempos = _pin(mem_c, sv["mem"]), _pin(mempos_c, sv["mempos"])
    K, V, Kpin = [], [], []
    for i in range(Lr):
        p_ = "transformer.decoder.layers.%d.multihead_attn." % i
        w, b = ref[p_ + "in_proj_weight"], ref[p_ + "in_proj_bias"]
        k_c = mempos @ _w16(w[Cd:2 * Cd]).t() + b[Cd:2 * Cd]
        v_c = mem @ _w16(w[2 * Cd:]).t() + b[2 * Cd:]
        t.bf16("k[%d]" % i, sv["k"][:, i * Cd:(i + 1) * Cd], k_c)
        t.bf16("v[%d]" % i, sv["v"][:, i * Cd:(i + 1) * Cd], v_c)
        Kpin.append(_pin(k_c, sv["k"][:, i * Cd:(i + 1) * Cd]))
        Kpin[-1].retain_grad()                                            # bf16(dK), for the bounds of its sums
        K.append(_GradBf16.apply(Kpin[-1]))                               # dK / dV are written in bf16
        V.append(_GradBf16.apply(_pin(v_c, sv["v"][:, i * Cd:(i + 1) * Cd])))

    # ---- query side, layer by layer, each step from the engine's previous saved tensor
    qpos = ref["query_embed.weight"].repeat(B, 1)
    assert bool((sv["x0", 0] == 0).all()), "x0 of layer 0 is not zero"
    x = sv["x0", 0].double()
    hs = []
    for i in range(Lr):
        p_ = "transformer.decoder.layers.%d." % i
        st = 8 * i
        n1 = _ln(x, ref, p_ + "norm1")
        t.close("fp32 steps", "n1[%d]" % i, sv["n1", i], n1, 1e-5)
        n1 = _pin(n1, sv["n1", i])
        w, b = ref[p_ + "self_attn.in_proj_weight"], ref[p_ + "self_attn.in_proj_bias"]
        qkv = torch.cat([((n1 + qpos) @ w[:Cd].t() + b[:Cd]) * qs, (n1 + qpos) @ w[Cd:2 * Cd].t() + b[Cd:2 * Cd],
                         n1 @ w[2 * Cd:].t() + b[2 * Cd:]], 1)
        t.close("fp32 steps", "qkv[%d]" % i, sv["qkv", i], qkv, 1e-5)
        qkv = _pin(qkv, sv["qkv", i])
        q_, k_, v_ = (_heads(qkv[:, j * Cd:(j + 1) * Cd], B, Q, h) for j in range(3))
        pr = torch.softmax(q_ @ k_.transpose(-1, -2), -1)
        keep = _keep(drop, st + 0, (B, h, Q, Q))
        o1 = _merge((pr if keep is None else pr * keep) @ v_)
        t.close("self attention", "o1[%d]" % i, sv["o1", i], o1, 5e-5)
        o1 = _pin(o1, sv["o1", i])
        y = o1 @ ref[p_ + "self_attn.out_proj.weight"].t() + ref[p_ + "self_attn.out_proj.bias"]
        keep = _keep(drop, st + 1, (R, Cd))
        x1 = x + (y if keep is None else y * keep)
        t.close("fp32 steps", "x1[%d]" % i, sv["x1", i], x1, 1e-5)
        x1 = _pin(x1, sv["x1", i])
        n2 = _ln(x1, ref, p_ + "norm2")
        t.close("fp32 steps", "n2[%d]" % i, sv["n2", i], n2, 1e-5)
        n2 = _pin(n2, sv["n2", i])
        w, b = ref[p_ + "multihead_attn.in_proj_weight"], ref[p_ + "multihead_attn.in_proj_bias"]
        qc = ((n2 + qpos) @ w[:Cd].t() + b[:Cd]) * qs
        t.close("fp32 steps", "qc[%d]" % i, sv["qc", i], qc, 1e-5)
        qc = _pin(qc, sv["qc", i])
        qh, kh, vh = _heads(qc, B, Q, h), _heads(K[i], B, S, h), _heads(V[i], B, S, h)
        lse = torch.logsumexp(qh.detach() @ kh.detach().transpose(-1, -2), -1).reshape(B * h, Q)
        t.close("fp32 steps", "lse[%d]" % i, sv["lse", i], lse, 1e-5, floor=0.0)
        keep = _keep(drop, st + 2, (B, h, Q, S))
        o2 = _merge(_CrossCore.apply(qh, kh, vh, keep, _heads(sv["o2", i].double(), B, Q, h)))
        t.close("cross attention", "o2[%d]" % i, sv["o2", i], o2, 2 ** -7, atol=4e-3)
        o2 = _pin(o2, sv["o2", i])
        y = o2 @ ref[p_ + "multihead_attn.out_proj.weight"].t() + ref[p_ + "multihead_attn.out_proj.bias"]
        keep = _keep(drop, st + 3, (R, Cd))
        x2 = x1 + (y if keep is None else y * keep)
        t.close("fp32 steps", "x2[%d]" % i, sv["x2", i], x2, 1e-5)
        x2 = _pin(x2, sv["x2", i])
        n3 = _ln(x2, ref, p_ + "norm3")
        t.close("fp32 steps", "n3[%d]" % i, sv["n3", i], n3, 1e-5)
        n3 = _pin(n3, sv["n3", i])
        pre = n3 @ ref[p_ + "linear1.weight"].t() + ref[p_ + "linear1.bias"]
        keep = _keep(drop, st + 4, (R, Fd))
        _relu_decisions("f[%d]" % i, sv["f", i], pre.detach(), keep)
        f = pre * (sv["f", i] > 0).double() * (keep.max().item() if drop else 1.0)     # ReLU' times 1/(1-p)
        t.close("fp32 steps", "f[%d]" % i, sv["f", i], f, 1e-5)
        f = _pin(f, sv["f", i])
        y = f @ ref[p_ + "linear2.weight"].t() + ref[p_ + "linear2.bias"]
        keep = _keep(drop, st + 5, (R, Cd))
        x3 = x2 + (y if keep is None else y * keep)
        x3_saved = sv["x0", i + 1] if i + 1 < Lr else sv["x3", i]
        assert torch.equal(sv["x3", i], x3_saved)
        t.close("fp32 steps", "x3[%d]" % i, sv["x3", i], x3, 1e-5)
        x = _pin(x3, sv["x3", i])
        hs_i = _ln(x, ref, "transformer.decoder.norm")
        t.close("fp32 steps", "hs[%d]" % i, hs_e[i].reshape(R, Cd), hs_i, 1e-5)
        hs.append(_pin(hs_i, hs_e[i].reshape(R, Cd)))
    hs = torch.stack(hs)                                                  # [L, R, C]

    # ---- heads: frame_proj split (trajectory head), bbox MLP, obj_proj
    if traj:
        wf = ref["frame_proj.weight"]
        ft = ref["frame_index.weight"] @ wf[:, Cd:].t() + ref["frame_proj.bias"]          # [T, C]
        cond = (hs.reshape(Lr * B, 1, Q, Cd) @ wf[:, :Cd].t()) + ft[None, :, None, :]   # [(l, b), t, q, C]
        cond = cond.reshape(Lr * B * T * Q, Cd)
        t.close("fp32 steps", "cond", sv["cond"], cond, 1e-5)
        box_in = _pin(cond, sv["cond"])
    else:
        box_in = hs.reshape(Lr * R, Cd)
    xb = box_in
    for j, nm in ((0, "box_x1"), (1, "box_x2")):
        pre = xb @ ref["bbox_embed.layers.%d.weight" % j].t() + ref["bbox_embed.layers.%d.bias" % j]
        _relu_decisions(nm, sv[nm], pre.detach())
        xb = pre * (sv[nm] > 0).double()
        t.close("fp32 steps", nm, sv[nm], xb, 1e-5)
        xb = _pin(xb, sv[nm])
    boxes = torch.sigmoid(xb @ ref["bbox_embed.layers.2.weight"].t() + ref["bbox_embed.layers.2.bias"])
    t.close("fp32 steps", "boxes", boxes_e.reshape(-1, 4), boxes, 1e-5)
    hid = (hs[-1] @ ref["obj_proj.0.weight"].t() + ref["obj_proj.0.bias"]) * (sv["obj_h"] > 0).double()
    emb = hid @ ref["obj_proj.2.weight"].t() + ref["obj_proj.2.bias"]
    loss = (hs * w_hs.double().reshape(Lr, R, Cd)).sum() + (boxes * w_box.double().reshape(-1, 4)).sum() + \
        (emb * w_emb.double().reshape(R, 256)).sum()
    loss.backward()

    # ---- every parameter gradient.  Magnitudes of the cancelling dK sums: |dK| per K-bias column, and for the position
    # embeddings the clip-summed |dK| |Wk| rows (d(mem + pos) = sum over layers of dK Wk), reduced as pos3d_bwd reduces
    dK = [kp.grad for kp in Kpin]
    with torch.no_grad():
        mag_mp = sum(d.abs() @ _bf16(ref["transformer.decoder.layers.%d.multihead_attn.in_proj_weight" % i][Cd:2 * Cd]).abs()
                     for i, d in enumerate(dK)).reshape(B, T, n, Cd).sum(0)
    mag = {"pos_embed": torch.cat([torch.zeros(1, Cd, dtype=torch.float64, device="cuda"), mag_mp.sum(0)])[None],
           "temporal_embed": mag_mp.sum(1)[None]}
    mem_keys = ("transformer.pre_norm.weight", "transformer.pre_norm.bias", "proj.weight", "pos_embed", "temporal_embed")
    for k, prm in dec.named_parameters():
        if k.startswith(("txt_proj.", "vid_proj.")):
            assert prm.grad is None or float(prm.grad.abs().max()) == 0.0, k
            continue
        assert prm.grad is not None, k
        got, want = prm.grad.detach(), ref[k].grad
        if k.startswith("class_embed."):
            assert float(got.abs().max()) == 0.0, k                    # no class loss in the graph
            continue
        if k in mag:
            t.grad_sum(k, got, want, mag[k])
        elif k in mem_keys:
            t.grad_memory(k, got, want)
        elif k.endswith("multihead_attn.in_proj_weight") or k.endswith("multihead_attn.in_proj_bias"):
            t.grad_query(k + "[q]", got[:Cd], want[:Cd])
            if k.endswith("bias"):
                i = int(k.split(".")[3])
                t.grad_sum(k + "[k]", got[Cd:2 * Cd], want[Cd:2 * Cd], dK[i].abs().sum(0))
            else:
                t.grad_memory(k + "[k]", got[Cd:2 * Cd], want[Cd:2 * Cd])
            t.grad_memory(k + "[v]", got[2 * Cd:], want[2 * Cd:])
        else:
            t.grad_query(k, got, want)
    return t


CASES = {
    # trajectory head, frame_term_bwd with its column-sum pre-reduction; p = 0 and p = 0.1
    "tiny_traj_p0": ("dec_tiny_traj", None, 2, 0.0),
    "tiny_traj_p0.1": ("dec_tiny_traj", None, 2, 0.1),
    # no trajectory head (box_in = hs), T = 2, 3 layers
    "tiny_notraj_p0.1": ("dec_tiny_notraj", None, 4, 0.1),
    # 16 queries: the full query block of both cross-attention kernels
    "tiny_traj_q16_p0.1": ("dec_tiny_traj", dict(Q=16), 2, 0.1),
    # c4 geometry, R = 39: every query-side weight gradient on the single-split plan
    "c4_b3_p0.1": (C4, None, 3, 0.1),
}


def _cfg(base, patch):
    from oracle import golden_cases as gc
    cfg = dict(gc.CASES[base]["cfg"]) if isinstance(base, str) else dict(base)
    cfg.update(patch or {})
    return cfg


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_decoder_training_step_against_float64(case):
    base, patch, B, p = CASES[case]
    _run_case(_cfg(base, patch), B, 40 + list(CASES).index(case), p).finish(case)


@pytest.mark.gpu
@pytest.mark.parametrize("side_stream", [False, True], ids=["default_stream", "side_stream"])
def test_decoder_training_step_c4_batch64_against_float64(side_stream):
    """The benchmarked c4 share (bench.py c4, 64 clips): R = 832 takes the split-K fp32-atomic weight gradients and
    B*S = 65536 the CTA-pair memory-side GEMMs.  On a non-default torch stream the backward's side stream must order
    against the caller's stream, not only against the default stream."""
    st = torch.cuda.Stream() if side_stream else None
    _run_case(C4, 64, 50, 0.1, stream=st).finish("c4_b64" + ("_side_stream" if side_stream else ""))


@pytest.mark.gpu
def test_get_saved_refusals():
    """hh_decoder_get_saved refuses (-2) a wrong byte count, an unknown name, a layer out of range and any read after an
    inference forward (which aliases every layer onto one buffer set)."""
    from helping_hand_for_egocentric_videos_b200 import _lib as L
    cfg = _cfg("dec_tiny_traj", None)
    dec = _module(cfg, 7, 0.1)
    lib = L.load()
    feats = torch.randn(2, cfg["T"], cfg["n"], cfg["F"], device="cuda")
    R, Cd = 2 * cfg["Q"], cfg["C"]
    buf = torch.empty(max(R * cfg["ffn"], 2 * cfg["T"] * cfg["n"] * Cd), device="cuda")

    def get(name, layer, nbytes):
        return lib.hh_decoder_get_saved(dec._engine(), name.encode(), layer, L.ptr(buf), nbytes, L.stream_ptr())
    assert get("x1", 0, R * Cd * 4) == -2                           # no forward yet
    dec(feats)[1].sum().backward()                                  # training forward + backward
    assert get("x1", 0, R * Cd * 4) == 0
    assert torch.equal(buf[:R * Cd].view(R, Cd), _saved(dec, "x1", 0, (R, Cd)))
    assert get("f", cfg["layers"] - 1, R * cfg["ffn"] * 4) == 0
    assert get("x1", 0, R * Cd * 4 - 4) == -2 and "bytes" in L.last_error()
    assert get("x4", 0, R * Cd * 4) == -2
    assert get("memf", 0, R * Cd * 4) == -2                         # memory-side names are layer -1
    assert get("x1", cfg["layers"], R * Cd * 4) == -2
    assert get("x1", -2, R * Cd * 4) == -2
    with torch.no_grad():
        dec.eval()
        dec(feats)                                                  # inference forward
    assert get("x1", 0, R * Cd * 4) == -2 and "no training forward" in L.last_error()
    assert get("memf", -1, 2 * cfg["T"] * cfg["n"] * Cd * 4) == -2
