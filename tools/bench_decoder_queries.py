"""Decoder step time against the number of queries per clip (Q = nq + 1 in {13, 17, 32}), in one process.

  c2 share:  ObjDecoder inference (eval), 64 clips x 16 frames x 256 patches of 1024-d features, no trajectory head
  c4 share:  ObjDecoder training forward + backward, 64 clips x 4 frames x 256 patches, trajectory head, dropout 0.1,
             on a fixed linear functional of hs and all layers' boxes

Q <= 16 runs the one-query-block instantiations of the cross-attention kernels, Q = 17 .. 32 the two-block ones.  The
three decoders alternate after a warm-up and are timed with CUDA events (median over `rounds` samples of `iters` steps
each); per-class times come from the engine's event profiler in a separate pass.  Writes one JSON object with the GPU
name and power limit read in the same run.

    python tools/bench_decoder_queries.py --out profiles/decoder_queries.json [--rounds 10]
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_feature_map_bf16 import alternate, gpu_info, summary  # noqa: E402

QS = (13, 17, 32)


def decoder(Q, frames, pred_traj, seed):
    from helping_hand_for_egocentric_videos_b200.model import tfm_decoder
    from helping_hand_for_egocentric_videos_b200 import synthetic
    tr = tfm_decoder.Cross_Attention(dropout=0.1, normalize_before=True, return_intermediate_dec=True)
    dec = tfm_decoder.ObjDecoder(tr, num_classes=22047, num_queries=Q, aux_loss=True, pred_traj=pred_traj,
                                 feature_dim=1024, num_frames=frames, patches_per_frame=256)
    synthetic.randomize_(dec, seed)
    return dec.cuda()


def profiled(steps, decs, reps=3):
    """Q -> {class: ms per step} from the decoder's event profiler (a pass of its own: events slow the host)."""
    res = {}
    for q, fn in steps.items():
        decs[q].set_profile(True)
        decs[q].profile()
        acc = {}
        for _ in range(reps):
            fn()
            torch.cuda.synchronize()
            for k, (t, _) in decs[q].profile().items():
                acc[k] = acc.get(k, 0.0) + t / reps
        decs[q].set_profile(False)
        res[q] = acc
    return res


def c2(rounds, iters):
    B, T, n = 64, 16, 256
    g = torch.Generator().manual_seed(5)
    feats = torch.randn(B, T, n, 1024, generator=g).cuda()
    decs = {q: decoder(q, T, False, seed=20 + q).eval() for q in QS}

    def make(q):
        def step():
            with torch.no_grad():
                decs[q](feats)
        return step
    steps = {q: make(q) for q in QS}
    ms = alternate(steps, rounds, iters)
    prof = profiled(steps, decs)
    return {"what": "c2 share: decoder eval, 64 clips x 16 frames x 256 patches x 1024, no trajectory head",
            "step": {q: summary(v) for q, v in ms.items()}, "profiled_ms_per_step": prof}


def c4(rounds, iters):
    B, T, n, L = 64, 4, 256, 6
    g = torch.Generator().manual_seed(6)
    feats = torch.randn(B, T, n, 1024, generator=g).cuda()
    decs, w = {}, {}
    for q in QS:
        decs[q] = decoder(q, T, True, seed=40 + q).train()
        decs[q].dropout_seed = 0x5EED
        w[q] = (torch.randn(L, B, q, 512, generator=g).cuda(), torch.randn(L, B * T, q, 4, generator=g).cuda())

    def make(q):
        def step():
            dec = decs[q]
            dec.zero_grad(set_to_none=True)
            out, hs, _, _ = dec(feats)
            boxes = torch.stack([a["pred_boxes"] for a in out["aux_outputs"]] + [out["pred_boxes"]])
            ((hs * w[q][0]).sum() + (boxes * w[q][1]).sum()).backward()
        return step
    steps = {q: make(q) for q in QS}
    ms = alternate(steps, rounds, iters)
    prof = profiled(steps, decs)
    return {"what": "c4 share: decoder training forward + backward, 64 clips x 4 frames x 256 patches x 1024, "
                    "trajectory head, dropout 0.1, fixed linear functional of hs and all layers' boxes",
            "step": {q: summary(v) for q, v in ms.items()}, "profiled_ms_per_step": prof}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--iters", type=int, default=3, help="steps per timed sample")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    torch.cuda.set_device(0)
    res = {"gpu": gpu_info(), "torch": torch.__version__, "rounds": args.rounds, "iters_per_sample": args.iters,
           "queries": list(QS), "c2": c2(args.rounds, args.iters), "c4": c4(args.rounds, args.iters)}
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    for k in ("c2", "c4"):
        print(k, {q: round(v["median_ms"], 3) for q, v in res[k]["step"].items()})
        for q, p in res[k]["profiled_ms_per_step"].items():
            print("  Q=%d" % q, {c: round(t, 3) for c, t in sorted(p.items())})


if __name__ == "__main__":
    main()
