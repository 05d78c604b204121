"""Generate tests/golden/*.pt by running the UNMODIFIED reference (a checkout of the original project).

TEST INFRASTRUCTURE ONLY.  Usage:  HH_REFERENCE_ROOT=<checkout> python -m oracle.make_golden  [--check]

Each fixture holds the *reference's* outputs for a seeded synthetic state_dict + input (both
regenerated from the seed by `hh_oracle.synth_state_dict` / `golden_cases.make_inputs`, so only the
outputs are stored).  Loading uses `load_state_dict(strict=True)`, which also pins the key/shape
lists of `hh_oracle.*_param_shapes` against the reference modules.
"""
import argparse
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import golden_cases as gc  # noqa: E402
from oracle import ref_import  # noqa: E402


def run_reference(case):
    ns = ref_import.import_reference()
    kind = case["kind"]
    torch.manual_seed(0)
    if kind == "losses":
        import importlib
        loss_mod = importlib.import_module("model.loss")
        box_utils = importlib.import_module("model.box_utils")
        nce, wl = loss_mod.EgoNCE(), loss_mod.WordContrastiveLoss()
        m = box_utils.build_matcher(None)

        def word(nouns, pred, inds):
            # the reference does not return col_ind; recompute it exactly as model/loss.py:85-93 does
            from scipy.optimize import linear_sum_assignment
            cols = []
            for b in range(inds.shape[0]):
                ids = inds[b][inds[b] != 0]
                if len(ids):
                    cost = -ns.metric.sim_matrix(nouns[ids], pred[b]).detach()
                    cols.append(torch.as_tensor(linear_sum_assignment(cost)[1], dtype=torch.int64))
            return wl(nouns, pred, inds), torch.cat(cols)
        crit = box_utils.SetCriterion(22047, matcher=m, eos_coef=0.1, losses=["boxes", "cardinality"],
                                      weight_dict={"loss_bbox_hand_boxes": 5, "loss_bbox_obj_boxes": 5,
                                                   "loss_giou_hand_boxes": 2, "loss_giou_obj_boxes": 2})   # run/train.py:460-472

        def box(detr_out, px, box_type):
            sizes = torch.full((px.shape[0], 2), 224.0)
            keep = torch.Tensor.cuda
            torch.Tensor.cuda = lambda self, *a, **k: self      # prepare_targets hard-codes .cuda() (model/box_utils.py:255)
            try:
                return box_utils.compute_box_loss(box_type, crit, detr_out, px, None, sizes, n_queries=12)
            finally:
                torch.Tensor.cuda = keep
        return gc.run_losses(gc.make_inputs(case), ns.metric.sim_matrix,
                             lambda x, mv, mn, pad: nce(x, mv, mn, multi_pad_mask=pad, strict_mask=True), word,
                             lambda o, t, e: m(o, t, exclude_class=e), box)
    if kind == "decoder_train":
        # The UNMODIFIED reference decoder in train() mode.  Only torch's dropout primitive is swapped: every call of
        # torch.nn.functional.dropout (nn.Dropout.forward and the attention-weight dropout inside
        # F.multi_head_attention_forward both resolve to it) draws its mask from hh_oracle.philox_keep, site = call
        # order within the forward: per layer [self-attn probs, dropout1, cross-attn probs, dropout2, FFN inner, dropout3]
        # (model/tfm_decoder.py:431-459).  The reference's tensors are sequence-first [Q, B, C]; the mask index is
        # defined batch-first (b, q, c), hence the transpose for those sites.
        import torch.nn.functional as F
        from oracle import hh_oracle as O
        c, dr = case["cfg"], case["dropout"]
        dec = ref_import.build_reference_decoder(
            ns, num_queries=c["Q"], feature_dim=c["F"], num_frames=c["T"], patches_per_frame=c["n"],
            pred_traj=c["pred_traj"], num_classes=c["ncls"], d_model=c["C"], nhead=c["heads"],
            dec_layers=c["layers"], ffn=c["ffn"])
        dec.load_state_dict(gc.decoder_state_dict(case), strict=True)
        dec.train()
        assert dec.transformer.decoder.layers[0].dropout1.p == dr["p"]        # Cross_Attention default dropout=0.1
        calls = {"k": 0}
        real_dropout = F.dropout

        def philox_dropout(input, p=0.5, training=True, inplace=False):
            if not training or p == 0.0:
                return input
            k = calls["k"]
            calls["k"] += 1
            layer, kind_ = divmod(k, 6)
            site = layer * 8 + kind_
            assert abs(p - dr["p"]) < 1e-12
            m = O.philox_keep(dr["seed"], dr["offset"], site, input.numel(), p)
            if kind_ in (0, 2):                                   # attention probabilities [B*heads, Lq, Lk]
                m = m.view(input.shape)
            else:                                                 # [Q, B, C] sequence-first
                qn, bn, cn = input.shape
                m = m.view(bn, qn, cn).transpose(0, 1)
            return input * m
        F.dropout = philox_dropout
        try:
            params = dict(dec.named_parameters())

            def fwd(feats):
                out, hs, _, _ = dec(feats)
                return out, hs
            res = gc.train_functional(case, fwd, dec.obj_proj, params)
        finally:
            F.dropout = real_dropout
        assert calls["k"] == 6 * c["layers"], calls
        return res
    with torch.no_grad():
        if kind == "encoder":
            c = case["cfg"]
            clip = ref_import.build_reference_backbone(
                ns, img_size=c["img"], patch_size=c["patch"], embed_dim=c["D"], depth=c["L"], num_heads=c["H"],
                num_frames=c["T"], text_width=c["text_width"], text_heads=c["text_heads"],
                text_layers=c["text_layers"], vocab_size=c["vocab"])
            sd = gc.backbone_state_dict(case)
            clip.load_state_dict(sd, strict=True)
            video, tokens = gc.make_inputs(case)
            out = clip(video, tokens, return_feature_map=True)
            res = {k: out[k] for k in ("image_embed", "text_embed", "image_feature_map", "text_feature_map")}
            # per-block activations through forward hooks would touch reference internals; block parity is
            # covered by running depth-truncated state_dicts instead (see golden_cases).
            return gc.subsample(case, res)
        if kind == "decoder":
            c = case["cfg"]
            dec = ref_import.build_reference_decoder(
                ns, num_queries=c["Q"], feature_dim=c["F"], num_frames=c["T"], patches_per_frame=c["n"],
                pred_traj=c["pred_traj"], num_classes=c["ncls"], d_model=c["C"], nhead=c["heads"],
                dec_layers=c["layers"], ffn=c["ffn"])
            sd = gc.decoder_state_dict(case)
            dec.load_state_dict(sd, strict=True)
            feats, text_feat = gc.make_inputs(case)
            out, hs, a, b = dec(feats)
            assert a == [] and b == []
            vid = dec.obj_proj(hs[-1])[:, -1]
            txt = dec.txt_proj(text_feat)
            sim = ns.metric.sim_matrix(txt, vid)
            res = {"pred_logits": out["pred_logits"], "pred_boxes": out["pred_boxes"], "hs": hs,
                   "aux_boxes": torch.stack([a_["pred_boxes"] for a_ in out["aux_outputs"]]),
                   "aux_logits0": out["aux_outputs"][0]["pred_logits"],
                   "video_embed": vid, "text_embed": txt, "sim": sim}
            return gc.subsample(case, res)
        if kind == "boxes":
            p, t = gc.make_inputs(case)
            pxy, txy = ns.box_ops.box_cxcywh_to_xyxy(p), ns.box_ops.box_cxcywh_to_xyxy(t)
            iou, union = ns.box_ops.box_iou(pxy, txy)
            giou = ns.box_ops.generalized_box_iou(pxy, txy)
            cost = 5.0 * torch.cdist(p, t, p=1) + 2.0 * (-giou)      # model/box_utils.py:75-88, weights :96
            return {"xyxy": pxy, "back": ns.box_ops.box_xyxy_to_cxcywh(pxy), "iou": iou, "union": union,
                    "giou": giou, "cost": cost}
        if kind == "score":
            a, b, preds, labels, types = gc.make_inputs(case)
            return {"sim": ns.metric.sim_matrix(a, b), "sim3": ns.metric.sim_matrix(a[None], b[None]),
                    "acc": ns.metric.egomcq_accuracy_metrics(preds, labels, types)}
    raise ValueError(kind)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--check", action="store_true", help="compare live reference with committed fixtures")
    ap.add_argument("--only", default=None, help="comma-separated case names (default: all)")
    args = ap.parse_args()
    os.makedirs(gc.GOLDEN_DIR, exist_ok=True)
    for name, case in gc.CASES.items():
        if args.only and name not in args.only.split(","):
            continue
        res = run_reference(case)
        path = os.path.join(gc.GOLDEN_DIR, name + ".pt")
        if args.check:
            old = torch.load(path)
            for k in res:
                if isinstance(res[k], torch.Tensor):
                    assert torch.equal(old[k], res[k]), (name, k)
            print("ok", name)
        else:
            torch.save(res, path)
            sz = os.path.getsize(path)
            print("wrote %s (%.1f KB)" % (path, sz / 1024))


if __name__ == "__main__":
    main()
