"""fp32 vs bf16 hand-over of the video tower's feature map (SpaceTimeTransformer.feature_map_dtype), in one process.

  c2 step:  64 clips x 16 frames through TimeSformer-L/14, then ObjDecoder (nq = 12) in eval on image_feature_map[:, 1:]
  c4 step:  ObjDecoder training forward + backward (64 clips x 4 frames x 256 patches, nq = 12, trajectory head,
            dropout 0.1) on a [:, 1:] view of a feature map

The two modes alternate after a warm-up and are timed with CUDA events; per-class times (encoder `layernorm`, decoder
`dec_memory_gemm`) come from the engines' event profiler in a separate pass.  The outputs of the two modes are compared
(forward outputs bit for bit; gradients to fp32 summation noise, the weight-gradient reductions use atomics).  Writes one
JSON object with the GPU name and power limit read in the same run.

    python tools/bench_feature_map_bf16.py --out profiles/feature_map_bf16.json [--rounds 10]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

MODES = {"fp32": torch.float32, "bf16": torch.bfloat16}


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"] = float(out[0])
        info["sm_max_mhz"] = float(out[1])
    except Exception as e:          # the numbers are reported without it, marked as such
        info["power_limit_error"] = str(e)
    return info


def build(frames, nq, pred_traj, seed, dropout=0.1):
    from helping_hand_for_egocentric_videos_b200.model import LaviLa, tfm_decoder
    from helping_hand_for_egocentric_videos_b200 import synthetic
    vis = LaviLa.SpaceTimeTransformer(img_size=224, patch_size=14, embed_dim=1024, depth=24, num_heads=16,
                                      num_frames=frames, time_init='zeros', ln_pre=True, act_layer=LaviLa.QuickGELU,
                                      num_classes=0)
    tr = tfm_decoder.Cross_Attention(dropout=dropout, normalize_before=True, return_intermediate_dec=True)
    dec = tfm_decoder.ObjDecoder(tr, num_classes=22047, num_queries=nq + 1, aux_loss=True, pred_traj=pred_traj,
                                 feature_dim=1024, num_frames=frames, patches_per_frame=256)
    synthetic.randomize_(vis, seed)
    synthetic.randomize_(dec, seed + 1)
    return vis.cuda().eval(), dec.cuda()


def timed(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / iters


def alternate(steps, rounds, iters):
    """steps: mode -> callable.  Warm both, then `rounds` x (each mode `iters` times); per-mode list of ms per step."""
    for fn in steps.values():
        for _ in range(2):
            fn()
    torch.cuda.synchronize()
    ms = {m: [] for m in steps}
    for r in range(rounds):
        order = list(steps) if r % 2 == 0 else list(steps)[::-1]
        for m in order:
            ms[m].append(timed(steps[m], iters))
    return ms


def summary(v):
    s = sorted(v)
    return {"median_ms": s[len(s) // 2], "min_ms": s[0], "max_ms": s[-1], "samples_ms": v}


def profiled(mods_steps, classes, reps=3):
    """mode -> {class: ms per step} from the engines' event profilers (a separate pass: events slow the host)."""
    res = {}
    for m, (mods, fn) in mods_steps.items():
        for mod in mods:
            mod.set_profile(True)
            mod.profile()
        acc = {}
        for _ in range(reps):
            fn()
            torch.cuda.synchronize()
            for mod in mods:
                for k, (t, _) in mod.profile().items():
                    if k in classes:
                        acc[k] = acc.get(k, 0.0) + t / reps
        for mod in mods:
            mod.set_profile(False)
        res[m] = acc
    return res


def c2(rounds, iters):
    from helping_hand_for_egocentric_videos_b200 import synthetic
    B, T, n = 64, 16, 256
    vis, dec = build(T, 12, False, seed=0)
    dec.eval()
    video = synthetic.synthetic_clips(B, T, 224, seed=1234, device="cuda")
    outs = {}

    def make(m):
        def step():
            vis.feature_map_dtype = MODES[m]
            with torch.no_grad():
                x_cls, fmap = vis.forward_features(video)
                out, hs, _, _ = dec(fmap[:, 1:].unflatten(1, (T, n)))
            outs[m] = (x_cls, out, hs, fmap.dtype, dec.last_launches())
        return step
    steps = {m: make(m) for m in MODES}
    ms = alternate(steps, rounds, iters)
    prof = profiled({m: ((vis, dec), steps[m]) for m in MODES}, ("layernorm", "dec_memory_gemm"))
    a, b = outs["fp32"], outs["bf16"]
    equal = {"x_cls": torch.equal(a[0], b[0]), "hs": torch.equal(a[2], b[2]),
             "pred_logits": torch.equal(a[1]["pred_logits"], b[1]["pred_logits"]),
             "pred_boxes": torch.equal(a[1]["pred_boxes"], b[1]["pred_boxes"]),
             "aux_outputs": all(torch.equal(x["pred_boxes"], y["pred_boxes"]) and torch.equal(x["pred_logits"], y["pred_logits"])
                                for x, y in zip(a[1]["aux_outputs"], b[1]["aux_outputs"]))}
    return {"what": "c2 step: encoder 64 x 16 frames L/14 + decoder eval (nq = 12) on image_feature_map[:, 1:]",
            "feature_map_bytes": {m: B * (1 + T * n) * 1024 * (4 if m == "fp32" else 2) for m in MODES},
            "decoder_launches": {"fp32": a[4], "bf16": b[4]},
            "step": {m: summary(v) for m, v in ms.items()}, "profiled_ms_per_step": prof, "outputs_equal": equal}


def c4(rounds, iters):
    B, T, n = 64, 4, 256
    _, dec = build(T, 12, True, seed=10)
    dec.train()
    dec.dropout_seed = 0x5EED
    g = torch.Generator().manual_seed(3)
    fmap32 = torch.randn(B, 1 + T * n, 1024, generator=g).cuda()
    maps = {"fp32": fmap32, "bf16": fmap32.to(torch.bfloat16)}
    res = {}

    def make(m):
        def step():
            dec.zero_grad(set_to_none=True)
            out, hs, _, _ = dec(maps[m][:, 1:].unflatten(1, (T, n)))
            loss = hs.square().mean() + out["pred_boxes"].square().mean()
            loss.backward()
            res[m] = (hs.detach(), out["pred_boxes"].detach())
        return step
    steps = {m: make(m) for m in MODES}
    ms = alternate(steps, rounds, iters)
    prof = profiled({m: ((dec,), steps[m]) for m in MODES}, ("dec_memory_gemm",))
    # equality at one fixed dropout step
    grads = {}
    for m in MODES:
        dec._drop_step = 1000
        steps[m]()
        grads[m] = {k: p.grad.detach().clone() for k, p in dec.named_parameters() if p.grad is not None}
    torch.cuda.synchronize()
    worst = 0.0
    for k in grads["fp32"]:
        a, b = grads["fp32"][k], grads["bf16"][k]
        worst = max(worst, (a - b).abs().max().item() / max(a.abs().max().item(), 1e-12))
    dec._drop_step = 2000
    steps["fp32"]()
    h32 = res["fp32"]
    dec._drop_step = 2000
    steps["bf16"]()
    h16 = res["bf16"]
    return {"what": "c4 decoder training forward + backward, 64 clips x 4 frames x 256 patches, nq = 12, dropout 0.1, "
                    "on a [:, 1:] view of the feature map",
            "step": {m: summary(v) for m, v in ms.items()}, "profiled_ms_per_step": prof,
            "outputs_equal": {"hs": torch.equal(h32[0], h16[0]), "pred_boxes": torch.equal(h32[1], h16[1])},
            "grad_max_rel_diff": worst}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--iters", type=int, default=3, help="steps per timed sample")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    import __graft_entry__  # noqa: F401  (puts the repository root on sys.path)
    torch.cuda.set_device(0)
    res = {"gpu": gpu_info(), "torch": torch.__version__, "rounds": args.rounds, "iters_per_sample": args.iters,
           "c2": c2(args.rounds, args.iters), "c4": c4(args.rounds, args.iters)}
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    for k in ("c2", "c4"):
        print(k, {m: round(v["median_ms"], 2) for m, v in res[k]["step"].items()}, res[k]["profiled_ms_per_step"],
              res[k]["outputs_equal"])


if __name__ == "__main__":
    main()
