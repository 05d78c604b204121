#!/usr/bin/env python
"""Headline benchmark: clips/sec of the video-side forward path (TimeSformer-L/14 encoder -> object-aware decoder ->
obj_proj -> similarity scoring).  Default workload = BASELINE.json configs[2] (16 frames x 224^2, nq = 12, 64 clips per GPU).

  python bench.py --gpus 1 --steps K --warmup W                      # this repo (hand-written sm_100a path), config c2
  python bench.py --config c1|c2|c3|c4 ...                           # the other BASELINE.json configurations
  torchrun ... bench.py --gpus N ...                                 # one rank per GPU, weak scaling, 1 all-gather / step
  python bench.py --impl reference ...                               # reference algorithm on the host CPU cores
  python bench.py ... --dump-outputs DIR                             # also write the last timed step's outputs, DIR/*.npy

One JSON line is printed by rank 0 (contract: task description / DESIGN.md section "Measurement").

  c1  L/14 + decoder nq=4 (pred_traj), 4 frames, 32 clips per GPU                        forward, clips/s
  c2  L/14 + decoder nq=12, 16 frames, 64 clips per GPU, EgoMCQ-style scoring            forward, clips/s   (default)
  c3  EPIC-MIR: c2's forward feeding a bank of 9728 / N video embeddings per rank; every step the banks are all-gathered
      and the rank's 9728 / N text rows are scored against all 9728 videos                forward + sharded sim, clips/s
  c4  one GPU's share of the pre-training step: 64 clips x 4 frames + 320 captions through the frozen backbone, decoder
      in train() mode, EgoNCE + box + word losses, decoder / heads backward, AdamW        training step, clips/s

The default (c2, N = 1) line also carries `gpu_eager_baseline` (the reference algorithm as plain torch ops on the same
GPU) and `extra` (c4 step, 9728^2 scoring, EgoMCQ question latency), each measured in this very run.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

UNIT = "clips/s"

CONFIGS = {
    "c1": dict(frames=4, nq=4, batch=32, pred_traj=True, idx=1,
               what="TimeSformer-L/14 + tfm_decoder nq=%(nq)d, %(frames)d frames 224^2, batch %(batch)d clips/GPU, "
                    "EgoMCQ-style scoring (BASELINE.json configs[1])"),
    "c2": dict(frames=16, nq=12, batch=64, pred_traj=False, idx=2,
               what="TimeSformer-L/14 + tfm_decoder nq=%(nq)d, %(frames)d frames 224^2, batch %(batch)d clips/GPU, "
                    "EgoMCQ-style scoring (BASELINE.json configs[2])"),
    "c3": dict(frames=16, nq=12, batch=64, pred_traj=False, idx=3, mir_rows=9728,
               what="EPIC-MIR zero-shot: TimeSformer-L/14 + tfm_decoder nq=%(nq)d, %(frames)d frames, batch %(batch)d "
                    "clips/GPU into a 9728-row embedding bank, all-gathered, full video x text similarity every step "
                    "(BASELINE.json configs[3])"),
    "c4": dict(frames=4, nq=12, batch=64, pred_traj=True, idx=4, train=True,
               what="pre-training step, one GPU's share: %(batch)d clips x %(frames)d frames + 5 captions per clip, frozen "
                    "L/14 backbone, tfm_decoder nq=%(nq)d in train() mode, EgoNCE + GIoU/L1 box + noun losses, decoder/heads "
                    "backward, AdamW (BASELINE.json configs[4])"),
}


def metric_name(frames, nq):
    return "clips/sec (%df x 224^2, nq=%d)" % (frames, nq)


def env_int(k, d):
    try:
        return int(os.environ.get(k, d))
    except ValueError:
        return d


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        with open(p) as f:
            d = json.load(f)
        return dict(burst=d.get("bf16_tflops", 1590.0), sustained=d.get("bf16_tflops_sustained", 1400.0),
                    hbm=d.get("hbm_gbs", 6650.0), source="MEASURED_PEAKS.json")
    return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the timed region runs (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return

        def pump():
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 8:
                continue
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                pw.append(float(r[3]))
            except ValueError:
                continue
            for nm, v in zip(names, r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def gpu_ms(fn, iters=5, warm=2):
    """Mean CUDA-event milliseconds of fn() on the current stream, after `warm` untimed calls."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def write_outputs(out_dir, arrays, sample=1 << 20, limit=64 << 20):
    """--dump-outputs: each tensor of `arrays` (name -> tensor) as <out_dir>/<name>.npy, floating point as float32 and
    integers as float64 (exact).  A tensor of more than `sample` elements is written as its flattened values at `sample`
    positions drawn from a fixed seed: the same positions in every run, so that two builds compare element for element."""
    import numpy as np
    host = {}
    for name, t in arrays.items():
        t = t.detach()
        t = t.double() if t.dtype == torch.float64 or not t.is_floating_point() else t.float()
        if t.numel() > sample:
            idx = torch.randint(t.numel(), (sample,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t.flatten()[idx.to(t.device)]
        host[name] = t.cpu().numpy()
    total = sum(a.nbytes for a in host.values())
    assert total <= limit, "--dump-outputs: %d bytes of outputs, more than %d" % (total, limit)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------- model construction
def build_modules(frames, nq, seed=0, pred_traj=False, device=None):
    """Random-init L/14 video tower + object decoder.  device=None: parameters drawn on the host from a seeded generator
    (identical on every rank); a CUDA device: constructed and re-drawn on the GPU (the extras' second set of modules)."""
    from helping_hand_for_egocentric_videos_b200.model import LaviLa, tfm_decoder
    from helping_hand_for_egocentric_videos_b200 import synthetic
    import contextlib
    ctx = torch.device(device) if device is not None else contextlib.nullcontext()
    with ctx:
        vis = LaviLa.SpaceTimeTransformer(img_size=224, patch_size=14, embed_dim=1024, depth=24, num_heads=16,
                                          num_frames=frames, time_init='zeros', attention_style='frozen-in-time',
                                          ln_pre=True, act_layer=LaviLa.QuickGELU, num_classes=0)
        tr = tfm_decoder.Cross_Attention(normalize_before=True, return_intermediate_dec=True)
        # run/test_epic.py:150-153 construction (the 16-frame path): pred_traj=False, num_queries = nq + 1;
        # run/test_EgoMCQ.py:236 / run/train.py (4 frames): pred_traj=True
        dec = tfm_decoder.ObjDecoder(tr, num_classes=22047, num_queries=nq + 1, aux_loss=True, pred_traj=pred_traj,
                                     feature_dim=1024, num_frames=frames, patches_per_frame=256)
    if device is not None:
        synthetic.randomize_on_device_(vis, seed)
        synthetic.randomize_on_device_(dec, seed + 1)
    else:
        synthetic.randomize_(vis, seed)
        synthetic.randomize_(dec, seed + 1)
    return vis.eval(), dec.eval()


def cpu_forward_clips(vsd, dsd, frames, nclips, threads, nq=12, pred_traj=False):
    """Reference algorithm (oracle port) on the host: encoder + decoder + obj_proj + sim, fp32."""
    from oracle import hh_oracle as O
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(99)
    video = torch.randn(nclips, frames, 3, 224, 224, generator=g)
    text = torch.randn(nq + 1, 256, generator=g)
    t0 = time.perf_counter()
    with torch.no_grad():
        _, fmap = O.encoder_forward(video, vsd, 16)
        _, hs, _, _ = O.decoder_forward(fmap[:, 1:].unflatten(1, (frames, 256)), dsd, heads=8, pred_traj=pred_traj)
        vid = O.obj_proj(hs[-1], dsd)[:, -1]
        O.sim_matrix(text, vid).argmax(-1)
    return time.perf_counter() - t0


def workload_string(cfg):
    return cfg["what"] % cfg


def run_reference(args, cfg, rank, emit):
    """--impl reference: the reference's algorithm on all host cores.  This is the oracle PORT (kind "port"): the
    reference is Python that imports from /root/reference, which does not exist on the GPU box; the port leaves out the
    reference's rearrange / cat copies, so it is, if anything, faster than the reference modules on the same cores.
    Bounded sample of 4 clips per step of the configuration's forward path (c4: its forward share only)."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    T, nq = cfg["frames"], cfg["nq"]
    vis, dec = build_modules(T, nq, pred_traj=cfg["pred_traj"])
    vsd = {k: v.detach() for k, v in vis.state_dict().items()}
    dsd = {k: v.detach() for k, v in dec.state_dict().items()}
    sample = 4                                    # ~10 s of host work per step on a 16-core box at 16 frames
    for _ in range(min(args.warmup, 1)):
        cpu_forward_clips(vsd, dsd, T, sample, cores, nq, cfg["pred_traj"])
    steps = args.steps
    dts = [cpu_forward_clips(vsd, dsd, T, sample, cores, nq, cfg["pred_traj"]) for _ in range(steps)]
    dt = sum(dts) / len(dts)
    val = sample / dt
    line = {"impl": "reference", "metric": metric_name(T, nq), "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": min(args.warmup, 1), "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_string(cfg), "name": args.config,
                       "frames": T, "nq": nq, "clips_per_step": sample,
                       "sample": "bounded sample of the workload: %d clips per step on the host cores%s" % (
                           sample, " (forward share of the training step only)" if cfg.get("train") else "")},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": "%d clip(s) per step, %d steps, oracle/hh_oracle.py fp32 torch CPU (a port of the "
                                       "reference's algorithm, not the reference modules)" % (sample, steps)},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ---------------------------------------------------------------------------------------------- c4: the training step
class TrainShare:
    """One GPU's share of BASELINE config c4 (run/train.py:104-203): `B` clips x 4 frames with 5 captions each through the
    frozen backbone (video + text towers), ObjDecoder in train() mode (dropout 0.1), txt_proj / obj_proj, EgoNCE +
    hand / object box losses + word loss, backward through heads and decoder, AdamW.  At world > 1 the text / video
    embeddings and the EgoNCE masks' operands are all-gathered with ONE packed differentiable collective."""

    def __init__(self, B, dev, world=1, rank=0, on_device_init=True):
        from helping_hand_for_egocentric_videos_b200 import synthetic
        from helping_hand_for_egocentric_videos_b200.model import LaviLa, box_utils, tfm_decoder as D
        import contextlib
        self.B, self.T, self.R, self.V = B, 4, 5, 2000
        T, R, V = self.T, self.R, self.V
        self.world = world
        ctx = torch.device(dev) if on_device_init else contextlib.nullcontext()
        with ctx:
            clip = LaviLa.CLIP_OPENAI_TIMESFORMER_LARGE(num_frames=T)
            tr = D.Cross_Attention(normalize_before=True, return_intermediate_dec=True)
            model = D.ObjDecoder(transformer=tr, num_classes=22047, num_queries=13, aux_loss=True, pred_traj=True,
                                 feature_dim=1024, num_frames=T, patches_per_frame=256)
        rnd = synthetic.randomize_on_device_ if on_device_init else synthetic.randomize_
        rnd(clip, 0)
        rnd(model, 1)
        self.clip = clip.to(dev).eval()
        for p in self.clip.parameters():
            p.requires_grad = False                                # run/train.py:88 freezes the backbone
        self.model = model.to(dev).train()                         # run/train.py trains the decoder in train() mode
        self.opt = torch.optim.AdamW(self.model.parameters(), lr=1e-5)
        self.crit = box_utils.SetCriterion(22047, matcher=box_utils.build_matcher(None), eos_coef=0.1,
                                           losses=["boxes", "cardinality"],
                                           weight_dict={"loss_bbox_hand_boxes": 5, "loss_bbox_obj_boxes": 5,
                                                        "loss_giou_hand_boxes": 2, "loss_giou_obj_boxes": 2}).to(dev)
        g = torch.Generator().manual_seed(5 + rank)
        self.host_video = torch.randn(B, T, 3, 224, 224, generator=g).pin_memory()
        self.video = self.host_video.to(dev)
        tokens = torch.zeros(B * R, 77, dtype=torch.long)
        for i in range(B * R):
            ln = int(torch.randint(3, 30, (1,), generator=g))
            tokens[i, :ln] = torch.randint(1, 49405, (ln,), generator=g)
            tokens[i, ln] = 49407
        self.tokens = tokens.to(dev)
        pad = (torch.rand(B * R, generator=g) > 0.4).float()
        pad[::R] = 1
        self.pad_rows = pad.to(dev)                                   # [B*R]; the mask is pad[:, None].repeat(1, B_glob)
        self.verb = (torch.rand(B, 118, generator=g) < 0.012).float().to(dev)
        self.noun = (torch.rand(B, 582, generator=g) < 0.004).float().to(dev)
        lo = 224 * torch.rand(B * T, 4, 2, generator=g) * 0.7
        px = torch.cat([lo, lo + 10 + 60 * torch.rand(B * T, 4, 2, generator=g)], -1)
        px[torch.rand(B * T, 4, generator=g) < 0.3] = 0.0
        self.px = px.to(dev)
        self.noun_feats = torch.randn(V, 768, generator=torch.Generator().manual_seed(6)).to(dev)
        inds = torch.randint(1, V, (B, 4), generator=g)
        inds[torch.rand(B, 4, generator=g) < 0.4] = 0
        self.inds = inds.to(dev)
        self.sizes = torch.full((B * T, 2), 224.0, device=dev)
        self.marks = {}
        self.ar = torch.arange(B * R, device=dev)

    def flops_per_clip(self):
        """Forward algorithmic FLOPs per clip (video tower + decoder + 5 captions through the text tower); the decoder /
        heads backward adds ~2x the decoder's forward share (SURVEY section 8d)."""
        return (self.clip.visual.flops_per_clip() + self.model.flops_per_clip(self.T)
                + self.R * self.clip.text_flops_per_sequence())

    def step(self, video=None, timed_parts=False, wrap=None):
        """`wrap`: optional {"decoder" | "losses" | "backward": context-manager factory} put around that part (tools/prof_c4.py)."""
        import contextlib
        from helping_hand_for_egocentric_videos_b200 import parallel
        wrap = wrap or {}
        around = lambda k: wrap[k]() if k in wrap else contextlib.nullcontext()  # noqa: E731
        from helping_hand_for_egocentric_videos_b200.model import box_utils, loss, metric
        B, T, R = self.B, self.T, self.R
        video = self.video if video is None else video
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)] if timed_parts else None
        if ev:
            ev[0].record()
        with torch.no_grad():
            out = self.clip(video, self.tokens, return_feature_map=True)
        if ev:
            ev[1].record()
        grid = out["image_feature_map"][:, 1:].unflatten(1, (T, 256))
        with around("decoder"):
            mo, hs, _, _ = self.model(grid)
        if ev:
            ev[2].record()
        with around("losses"):
            txt = self.model.txt_proj(out["text_feature_map"][self.ar, self.tokens.argmax(-1)])
            emb = self.model.obj_proj(hs[-1])
            vid = emb[:, -1].contiguous()
            verb, noun, pad_rows = self.verb, self.noun, self.pad_rows
            if self.world > 1:
                txt, vid, verb, noun, pad_rows = parallel.all_gather_packed([txt, vid, verb, noun, pad_rows])
            pad = pad_rows[:, None].expand(-1, vid.shape[0]).contiguous()
            nce, _ = loss.EgoNCE()(metric.sim_matrix(txt, vid), metric.sim_matrix(verb, verb), metric.sim_matrix(noun, noun),
                                   multi_pad_mask=pad, strict_mask=True)
            lh, _ = box_utils.compute_box_loss('hand_boxes', self.crit, mo, self.px[:, :2].clone(), None, self.sizes, n_queries=12)
            lo_, _ = box_utils.compute_box_loss('obj_boxes', self.crit, mo, self.px[:, 2:].clone(), None, self.sizes, n_queries=12)
            word = loss.WordContrastiveLoss()(self.model.txt_proj(self.noun_feats), emb[:, :-1].contiguous(), self.inds)
        total = nce + lh + lo_ + 0.5 * word
        self.outputs = {"loss": total, "video_embed": vid, "text_embed": txt, "pred_boxes": mo["pred_boxes"],
                        "pred_logits": mo["pred_logits"]}
        if ev:
            ev[3].record()
        with around("backward"):
            total.backward()
        if ev:
            ev[4].record()
        self.opt.step()
        self.opt.zero_grad(set_to_none=True)
        if ev:
            ev[5].record()
            torch.cuda.synchronize()
            names = ["backbone_fwd_ms", "decoder_fwd_train_ms", "heads_losses_ms", "backward_ms", "optimizer_ms"]
            self.marks = {nm: ev[i].elapsed_time(ev[i + 1]) for i, nm in enumerate(names)}
        return total


# ---------------------------------------------------------------------------------------------- extras of the default line
def gpu_eager_baseline(T, nq, pred_traj, dev, clips=16):
    """SURVEY section 8(d) 'GPU baseline to beat': the reference's algorithm as plain torch ops (cuBLAS / ATen kernels;
    the oracle restatement -- /root/reference does not exist on the GPU box) on the SAME GPU, fp32 and bf16 autocast."""
    from oracle import hh_oracle as O            # baseline leg only: never on the product path
    vsd = O.synth_state_dict(O.encoder_param_shapes(1024, 24, 14, 256, T), 0)
    dsd = O.synth_state_dict(O.decoder_param_shapes(512, nq + 1, 256, T, 1024, 22048, layers=6, ffn=2048, pred_traj=pred_traj), 1)
    vsd = {k: v.to(dev) for k, v in vsd.items()}
    dsd = {k: v.to(dev) for k, v in dsd.items()}
    video = torch.randn(clips, T, 3, 224, 224, device=dev)
    text = torch.randn(nq + 1, 256, device=dev)

    def step():
        _, fmap = O.encoder_forward(video, vsd, 16)
        _, hs, _, _ = O.decoder_forward(fmap[:, 1:].unflatten(1, (T, 256)).float(), dsd, heads=8, pred_traj=pred_traj)
        vid = O.obj_proj(hs[-1], dsd)[:, -1]
        return O.sim_matrix(text, vid.float()).argmax(-1)

    res = {"what": "oracle restatement of the reference as torch-eager CUDA ops on this GPU", "clips_per_step": clips,
           "frames": T, "nq": nq}
    tf32 = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        for name, ctx in (("fp32", torch.autocast("cuda", enabled=False)),
                          ("bf16_autocast", torch.autocast("cuda", dtype=torch.bfloat16))):
            with torch.no_grad(), ctx:
                ms = gpu_ms(step, iters=3, warm=2)
            res[name] = {"ms_per_step": ms, "clips_per_s": clips / ms * 1e3}
    finally:
        torch.backends.cuda.matmul.allow_tf32 = tf32
    return res


def extra_c3_sim(dev, peaks, rows=9728):
    """EPIC-MIR scoring alone (BASELINE configs[3]): sim_matrix of [rows,256] text x [rows,256] video embeddings -> fp32
    [rows, rows].  Output-write bound: algorithmic bytes = 2 * rows * 256 * 4 in + rows^2 * 4 out."""
    from helping_hand_for_egocentric_videos_b200 import ops
    a = torch.randn(rows, 256, generator=torch.Generator().manual_seed(7)).to(dev)
    b = torch.randn(rows, 256, generator=torch.Generator().manual_seed(8)).to(dev)
    ms = gpu_ms(lambda: ops.sim_matrix(a, b), iters=10, warm=3)
    nbytes = 2.0 * rows * 256 * 4 + float(rows) * rows * 4
    tms = gpu_ms(lambda: torch.nn.functional.normalize(a, dim=-1) @ torch.nn.functional.normalize(b, dim=-1).t(), iters=10, warm=3)
    return {"ms": ms, "rows": rows, "algorithmic_bytes": nbytes, "achieved_GBps": nbytes / ms / 1e6,
            "hbm_peak_GBps": peaks["hbm"], "frac_of_hbm": nbytes / ms / 1e6 / peaks["hbm"],
            "floor_ms_at_hbm_peak": nbytes / peaks["hbm"] / 1e6, "torch_eager_fp32_ms": tms}


def extra_egomcq_question(dev):
    """The reference's real EgoMCQ call shape (run/test_EgoMCQ.py:215,266): one question = 5 candidate clips x 4 frames
    against 1 caption embedding, result read back per question.  Wall-clock latency, the engines' summed kernel time,
    and the torch-eager restatement beside it."""
    from helping_hand_for_egocentric_videos_b200 import ops
    from helping_hand_for_egocentric_videos_b200.model import metric
    T, nq = 4, 4
    vis, dec = build_modules(T, nq, seed=10, pred_traj=True, device=dev)
    video = torch.randn(5, T, 3, 224, 224, device=dev)
    text = torch.randn(1, 256, device=dev)

    def question():
        _, fmap = vis.forward_features(video)
        _, hs, _, _ = dec(fmap[:, 1:].unflatten(1, (T, 256)))
        vid = dec.obj_proj(hs[-1])[:, -1]
        return int(ops.row_argmax(metric.sim_matrix(text, vid)).item())          # host reads the choice
    for _ in range(5):
        question()
    torch.cuda.synchronize()
    n = 20
    t0 = time.perf_counter()
    for _ in range(n):
        question()
    wall = (time.perf_counter() - t0) / n * 1e3
    vis.set_profile(True)
    dec.set_profile(True)
    vis.profile(), dec.profile()
    for _ in range(n):
        question()
    prof = {}
    prof.update(vis.profile())
    prof.update(dec.profile())
    vis.set_profile(False)
    dec.set_profile(False)
    kernel_ms = sum(v[0] for v in prof.values()) / n
    launches = vis.last_launches() + dec.last_launches() + 4
    res = {"clips": 5, "frames": T, "nq": nq, "wall_ms": wall, "sum_kernel_ms": kernel_ms,
           "kernel_share_of_wall": kernel_ms / wall if wall > 0 else None, "launches": launches,
           "graph": bool(getattr(vis, "uses_graph", lambda: False)())}
    del vis, dec
    try:
        from oracle import hh_oracle as O        # baseline leg only
        vsd = {k: v.to(dev) for k, v in O.synth_state_dict(O.encoder_param_shapes(1024, 24, 14, 256, T), 0).items()}
        dsd = {k: v.to(dev) for k, v in O.synth_state_dict(
            O.decoder_param_shapes(512, nq + 1, 256, T, 1024, 22048, layers=6, ffn=2048, pred_traj=True), 1).items()}

        def eager():
            with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
                _, fmap = O.encoder_forward(video, vsd, 16)
                _, hs, _, _ = O.decoder_forward(fmap[:, 1:].unflatten(1, (T, 256)).float(), dsd, heads=8, pred_traj=True)
                v = O.obj_proj(hs[-1], dsd)[:, -1]
                return int(O.sim_matrix(text, v.float()).argmax(-1).item())
        for _ in range(3):
            eager()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(10):
            eager()
        res["torch_eager_bf16_wall_ms"] = (time.perf_counter() - t0) / 10 * 1e3
    except Exception as e:   # noqa: BLE001 -- a baseline leg must not take the headline line down
        res["torch_eager_error"] = repr(e)[:200]
    return res


def extra_c4(dev):
    ts = TrainShare(64, dev)
    for _ in range(2):
        ts.step()
    ms = gpu_ms(lambda: ts.step(), iters=3, warm=0)
    ts.step(timed_parts=True)
    res = {"ms": ms, "clips_per_s": 64 / ms * 1e3, "clips": 64, "frames": 4, "captions": 320, "parts": ts.marks,
           "what": "one GPU's share of BASELINE configs[4] (see --config c4)"}
    del ts
    return res


# ---------------------------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=None, help="clips per GPU per step (default: the configuration's)")
    ap.add_argument("--frames", type=int, default=None)
    ap.add_argument("--nq", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip gpu_eager_baseline and the extra.* measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (rank 0; outputs "
                         "of more than 2^20 elements as a fixed, seeded sample of their elements)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    cfg = dict(CONFIGS[args.config])
    for k in ("batch", "frames", "nq"):
        if getattr(args, k) is not None:
            cfg[k] = getattr(args, k)

    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    # inputs the configurations draw from torch's default generators (c3's embedding bank) and the decoder's dropout
    # stream in train() mode (c4) follow this seed: the same arguments give the same computation in every run
    torch.manual_seed(rank)
    # stdout carries exactly one JSON line: while the benchmark runs, file descriptor 1 points at stderr, so that
    # anything a C library prints there (NCCL's "NCCL version ..." banner when the box sets NCCL_DEBUG) cannot end up in
    # front of it; the descriptor is restored for the final print
    sys.stdout.flush()
    stdout_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.dup2(stdout_fd, 1)
        print(json.dumps(line), flush=True)
    if args.impl == "reference":
        run_reference(args, cfg, rank, emit)
        return

    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py (b200 arm) needs a CUDA device; there is no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ctx = dict(args=args, cfg=cfg, rank=rank, world=world, local=local, dev=dev, emit=emit, dist=dist)
    if cfg.get("train"):
        run_train(ctx)
    else:
        run_forward(ctx)
    if world > 1:
        dist.destroy_process_group()


def make_timers(ctx):
    dist, world, dev = ctx["dist"], ctx["world"], ctx["dev"]

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps):
        """K steps bracketed by barrier + synchronize; returns (max over ranks, this rank's, all ranks') milliseconds."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        own = e0.elapsed_time(e1)               # this rank's own device time, before anyone waits for the slowest
        barrier()
        ms = torch.tensor([own], device=dev)
        per_rank = [own]
        if world > 1:
            allms = [torch.zeros_like(ms) for _ in range(world)]
            dist.all_gather(allms, ms)
            per_rank = [t.item() for t in allms]
        return max(per_rank), own, per_rank
    return barrier, timed


def rank_spread(per_rank_total_ms, steps):
    v = sorted(t / steps for t in per_rank_total_ms)
    return {"min": v[0], "median": v[len(v) // 2], "max": v[-1], "all": [round(t, 3) for t in v]}


def run_forward(ctx):
    """c1 / c2 / c3: throughput of the forward path."""
    args, cfg, rank, world, dev, emit, dist = (ctx[k] for k in ("args", "cfg", "rank", "world", "dev", "emit", "dist"))
    from helping_hand_for_egocentric_videos_b200 import ops, parallel, synthetic
    from helping_hand_for_egocentric_videos_b200.model import metric
    barrier, timed = make_timers(ctx)
    warmup = max(3, args.warmup)
    B, T, nq = cfg["batch"], cfg["frames"], cfg["nq"]
    mir_rows = cfg.get("mir_rows", 0)

    vis_cpu, dec_cpu = build_modules(T, nq, pred_traj=cfg["pred_traj"])
    cpu_sd = None
    if rank == 0 and not args.no_cpu_baseline:
        cpu_sd = ({k: v.detach().clone() for k, v in vis_cpu.state_dict().items()},
                  {k: v.detach().clone() for k, v in dec_cpu.state_dict().items()})
    vis, dec = vis_cpu.to(dev), dec_cpu.to(dev)

    host_video = synthetic.synthetic_clips(B, T, 224, seed=1234 + rank, pinned=True)   # 616 MB at B=64, T=16: > L2 (126 MB)
    video = host_video.to(dev, non_blocking=True)
    text = torch.randn(nq + 1, 256, generator=torch.Generator().manual_seed(7)).to(dev)  # caption embeddings (text tower
    #                                                                                      is outside the measured path)
    # c3: this rank's rows of the 9728-row banks (video embeddings written by the forward, text embeddings given)
    state = {"i": 0, "pending": None, "last": None}
    if mir_rows:
        rows_local = mir_rows // world
        bank = torch.nn.functional.normalize(torch.randn(rows_local, 256, device=dev), dim=-1)
        text_bank = torch.randn(rows_local, 256, generator=torch.Generator().manual_seed(8 + rank)).to(dev)

    def embed(v, u8=None):
        if u8 is not None:
            _, fmap = vis.forward_features_u8(v, *u8)
        else:
            _, fmap = vis.forward_features(v)
        grid = fmap[:, 1:].unflatten(1, (T, 256))
        _, hs, _, _ = dec(grid)
        return dec.obj_proj(hs[-1])[:, -1]

    def step(v, u8=None):
        """One step.  world > 1: the all-gather of THIS step's embeddings is issued on a side stream and consumed by the
        NEXT step (its scores lag one step; finish() drains the last one), so no rank's compute stream ever waits for
        the slowest rank inside a step.  Every step issues exactly one collective and scores exactly one gathered set."""
        vid = embed(v, u8)
        i = state["i"]
        state["i"] = i + 1
        if mir_rows:
            lo = (i * B) % max(1, rows_local - B + 1)
            bank[lo:lo + B].copy_(vid)
            mine = [bank]
        else:
            mine = [vid]
        if world > 1:
            prev = state["pending"]
            state["pending"] = parallel.all_gather_packed_async(mine, slot=i % 2)
            if prev is None:
                return None
            (allv,) = prev.wait()
        else:
            (allv,) = mine
        if mir_rows:
            res = ops.row_argmax(metric.sim_matrix(text_bank, allv))
        else:
            res = ops.row_argmax(metric.sim_matrix(text, allv))
        state["last"] = (allv, res)
        return res

    def finish():
        if world > 1 and state["pending"] is not None:
            (allv,) = state["pending"].wait()
            state["pending"] = None
            src = text_bank if mir_rows else text
            state["last"] = (allv, ops.row_argmax(metric.sim_matrix(src, allv)))

    for _ in range(warmup):
        step(video)
    finish()
    flops_clip = vis.flops_per_clip() + dec.flops_per_clip(T)
    launches_step = vis.last_launches() + dec.last_launches() + 4 + (1 if world > 1 else 0) + (1 if mir_rows else 0)

    # ---- the collective, checked on the GPUs (outside the timed region): the gathered block must hold every rank's
    # embeddings at that rank's offset -- own rows bit-equal, the other ranks' rows by their fp64 checksums
    gather_check = None
    if world > 1:
        vid = embed(video)
        (allv,) = parallel.all_gather_packed([vid])
        n = vid.shape[0]
        assert allv.shape[0] == world * n, (allv.shape, world, n)
        assert torch.equal(allv[rank * n:(rank + 1) * n], vid), "gathered block differs from the rank-local embeddings"
        sums = torch.stack([vid.double().sum(), vid.double().abs().sum()])
        all_sums = [torch.zeros_like(sums) for _ in range(world)]
        dist.all_gather(all_sums, sums)
        for r in range(world):
            blk = allv[r * n:(r + 1) * n].double()
            got = torch.stack([blk.sum(), blk.abs().sum()])
            assert torch.equal(got, all_sums[r]), "gathered rows of rank %d do not match that rank's checksum" % r
        gather_check = {"own_rows_bit_equal": True, "all_ranks_checksums_equal": True, "rows": world * n}

    # ---- device-resident throughput (value), with per-kernel CUDA-event timing and clock sampling
    vis.set_profile(True)
    dec.set_profile(True)
    vis.profile(), dec.profile()
    sampler = ClockSampler(ctx["local"])
    if rank == 0:
        sampler.start()

    def timed_steps():
        step(video)
    ms_total, _, per_rank = timed(lambda: timed_steps(), args.steps)
    finish()
    clocks = sampler.stop() if rank == 0 else None
    prof = {}
    prof.update(vis.profile())
    prof.update(dec.profile())
    vis.set_profile(False)
    dec.set_profile(False)
    ms_step = ms_total / args.steps
    value = world * B / (ms_step * 1e-3)
    if args.dump_outputs and rank == 0:
        # the e2e measurements below take more steps: the timed path's last outputs are written now.  The step keeps
        # only its embeddings and choices; the scores it ranked are recomputed from them by the same kernel
        allv, res = state["last"]
        sim = metric.sim_matrix(text_bank if mir_rows else text, allv)
        write_outputs(args.dump_outputs, {"video_embed": allv, "sim": sim, "choice": res})

    # ---- end to end through the public modules with host buffers: pinned H2D of the clips + D2H of the choices
    e2e = e2e_u8 = None
    if not args.no_e2e:
        # Input pipeline: every step's clips cross PCIe from pinned host memory into one of two device buffers on a
        # copy stream, issued while the previous step computes (standard double buffering); the step waits for
        # its own copy, and its result is read back to the host before the next step starts.
        copy_stream = torch.cuda.Stream(device=dev)
        n_out = (mir_rows // world) if mir_rows else (nq + 1)

        def measure_e2e(host, run_step):
            bufs = [torch.empty_like(host, device=dev), torch.empty_like(host, device=dev)]
            ready = [torch.cuda.Event(), torch.cuda.Event()]
            free = [torch.cuda.Event(), torch.cuda.Event()]
            for ev in free:
                ev.record()
            st = {"i": 0}

            def issue_copy(i):
                with torch.cuda.stream(copy_stream):
                    copy_stream.wait_event(free[i % 2])
                    bufs[i % 2].copy_(host, non_blocking=True)
                    ready[i % 2].record(copy_stream)

            issue_copy(0)

            def e2e_step():
                i = st["i"]
                torch.cuda.current_stream().wait_event(ready[i % 2])
                issue_copy(i + 1)
                res = run_step(bufs[i % 2])
                free[i % 2].record()
                st["i"] = i + 1
                return res.cpu() if res is not None else None
            for _ in range(2):
                e2e_step()
            ms = timed(e2e_step, args.steps)[0] / args.steps
            finish()
            torch.cuda.synchronize()
            return {"value": world * B / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms,
                    "h2d_bytes_per_step": host.numel() * host.element_size(), "d2h_bytes_per_step": n_out * 8}

        e2e = measure_e2e(host_video, step)
        # same step fed with raw uint8 frames [B,T,224,224,3] (what the video decoder produces): the loader's
        # /255 + mean/std normalisation is fused into the patch loader (hh_encoder_forward_u8), a quarter of the H2D bytes
        g8 = torch.Generator().manual_seed(4321 + rank)
        host_u8 = torch.randint(0, 256, (B, T, 224, 224, 3), generator=g8, dtype=torch.uint8).pin_memory()
        mean = [108.3272985 / 255, 116.7460125 / 255, 104.09373615000001 / 255]
        std = [68.5005327 / 255, 66.6321579 / 255, 70.32316305 / 255]
        e2e_u8 = measure_e2e(host_u8, lambda frames: step(frames, (mean, std)))

    if rank != 0:
        return

    peaks = load_peaks()
    # dominant kernel = the tcgen05 GEMM (qkv / proj / fc1 / fc2 launches of the encoder)
    M = B * (1 + T * 256)
    gemm_flops = {"gemm_qkv": 2.0 * M * 3072 * 1024, "gemm_proj": 2.0 * M * 1024 * 1024,
                  "gemm_fc1": 2.0 * M * 4096 * 1024, "gemm_fc2": 2.0 * M * 1024 * 4096}
    g_ms = sum(prof[k][0] for k in gemm_flops if k in prof)
    g_fl = sum(gemm_flops[k] * prof[k][1] for k in gemm_flops if k in prof)
    gemm_tflops = g_fl / (g_ms * 1e-3) / 1e12 if g_ms > 0 else 0.0
    per_class = {k: {"ms_per_step": v[0] / args.steps, "launches_per_step": v[1] / args.steps} for k, v in prof.items()}
    # algorithmic bytes per launch of each GEMM class (A + W + output in bf16; with the LayerNorm folded in, the proj / fc2
    # launches also carry the fp32 residual stream: proj = time-proj (x read) and space-proj (x read + written) alternating,
    # fc2 = x read + written): the producers are co-bound by HBM, so both roofline fractions are reported per class
    fused_ln = os.environ.get("HH_LN_UNFUSED", "0") in ("", "0")
    D_, H_ = 1024, 4096
    res_extra = {"gemm_proj": 6.0 * M * D_, "gemm_fc2": 8.0 * M * D_} if fused_ln else {}
    gemm_bytes = {"gemm_qkv": 2.0 * (M * D_ + 3 * D_ * D_ + M * 3 * D_), "gemm_proj": 2.0 * (M * D_ + D_ * D_ + M * D_),
                  "gemm_fc1": 2.0 * (M * D_ + H_ * D_ + M * H_), "gemm_fc2": 2.0 * (M * H_ + D_ * H_ + M * D_)}
    for k in gemm_flops:
        if k in prof and prof[k][0] > 0:
            sec = prof[k][0] * 1e-3 / prof[k][1]
            per_class[k]["tflops"] = gemm_flops[k] / sec / 1e12
            per_class[k]["frac_of_sustained_bf16"] = gemm_flops[k] / sec / 1e12 / peaks["sustained"]
            nbytes = gemm_bytes[k] + res_extra.get(k, 0.0)
            per_class[k]["algorithmic_GB_per_launch"] = nbytes / 1e9
            per_class[k]["frac_of_hbm"] = nbytes / sec / 1e9 / peaks["hbm"]
    # DRAM traffic of the dominant kernel per launch: from the committed `ncu --set full` capture at these very shapes
    # (profiles/*_gemm_traffic.json, newest round first), averaged over the launches of one step like `achieved`.
    traffic, traffic_detail = None, None
    for tname in ("r2_gemm_traffic.json", "r1_gemm_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", tname)
        if os.path.isfile(tpath) and B == 64 and T == 16:
            with open(tpath) as f:
                tj = json.load(f)
            tk = tj["kernels"]
            per_step = {"qkv": 48, "proj": 48, "fc1": 24, "fc2": 24}
            traffic = sum(tk[k]["dram_bytes_per_launch"] * c for k, c in per_step.items()) / 144   # bytes per launch
            traffic_detail = {"avg_dram_bytes_per_launch": traffic,
                              "avg_algorithmic_bytes_per_launch": sum(tk[k]["algorithmic_bytes"] * c for k, c in per_step.items()) / 144,
                              "source": tj.get("source", "profiles/" + tname + " (ncu --set full, dram__bytes_read.sum + "
                                                                               "dram__bytes_write.sum)")}
            break
    path_tflops = value / world * flops_clip / 1e12
    line = {
        "metric": metric_name(T, nq), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": workload_string(cfg), "name": args.config,
                   "clips_per_gpu": B, "frames": T, "nq": nq, "l2": "inputs larger than L2 (%.0f MB clips/step)" % (
                       host_video.numel() * 4 / 1e6), "parallelism": "dp%d" % world,
                   "flops_per_clip": flops_clip, "path_tflops_per_gpu": path_tflops,
                   "path_frac_of_sustained_peak": path_tflops / peaks["sustained"],
                   "path_frac_of_burst_peak": path_tflops / peaks["burst"],
                   "kernel_ms_per_step": per_class},
        "roofline": {"bound": "tensor", "kernel": "gemm_kernel (tcgen05, encoder qkv/proj/fc1/fc2 launches)",
                     "achieved": gemm_tflops, "peak": peaks["sustained"], "unit": "TFLOP/s",
                     "frac": gemm_tflops / peaks["sustained"], "peak_source": peaks["source"] + " sustained bf16",
                     "share_of_step": g_ms / args.steps / ms_step if ms_step > 0 else None, "traffic": traffic,
                     "traffic_detail": traffic_detail,
                     "note": ("LayerNorm and the residual adds run INSIDE these launches (norm1/2/3 folded into the qkv / fc1 "
                              "epilogues, fp32 residual stream read / rewritten by the proj / fc2 epilogues): `achieved` counts "
                              "only the 2MNK flops of launches that also move the 20 B per element per layer of the residual "
                              "stream; per-class tensor and HBM fractions are in config.kernel_ms_per_step "
                              "(HH_LN_UNFUSED=1 gives the round-1 split: GEMMs at ~0.97 + 30 ms of LayerNorm kernels, a 3 % "
                              "slower step)") if fused_ln else None},
        "clocks": clocks, "gpu_launches": launches_step * args.steps,
        "rank_ms_per_step": rank_spread(per_rank, args.steps),
    }
    if world > 1:
        line["collective"] = {"what": "one packed ncclAllGather of the [B,256] video embeddings per step, issued on a side "
                                      "stream and consumed by the next step (scores lag one step)",
                              "check": gather_check}
    if e2e:
        line["e2e"] = e2e
        line["e2e_u8"] = e2e_u8
    if cpu_sd is not None:
        cores = os.cpu_count() or 1
        cpu_forward_clips(cpu_sd[0], cpu_sd[1], T, 1, cores, nq, cfg["pred_traj"])   # warm the host thread pool / allocator
        dt = cpu_forward_clips(cpu_sd[0], cpu_sd[1], T, 4, cores, nq, cfg["pred_traj"])
        line["cpu_baseline"] = {"value": 4.0 / dt, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": "4 clips (same L/14, %d-frame, nq=%d path) through oracle/hh_oracle.py (a port of "
                                          "the reference's algorithm), fp32 torch CPU, %.1f s" % (T, nq, dt)}
    if world == 1 and not args.no_extras:
        del video, host_video
        torch.cuda.empty_cache()

        def guarded(fn, *a):
            try:
                return fn(*a)
            except Exception as e:   # noqa: BLE001 -- an extra must not take the headline line down
                return {"error": repr(e)[:300]}
        line["gpu_eager_baseline"] = guarded(gpu_eager_baseline, T, nq, cfg["pred_traj"], dev)
        geb = line["gpu_eager_baseline"]
        if "bf16_autocast" in geb:
            geb["speedup_vs_bf16_autocast"] = value / geb["bf16_autocast"]["clips_per_s"]
            geb["speedup_vs_fp32"] = value / geb["fp32"]["clips_per_s"]
        torch.cuda.empty_cache()
        extra = {"c3_sim_9728": guarded(extra_c3_sim, dev, peaks)}
        extra["c3_sim_9728_ms"] = extra["c3_sim_9728"].get("ms")
        if args.config == "c2":
            del vis, dec
            torch.cuda.empty_cache()
            extra["egomcq_question"] = guarded(extra_egomcq_question, dev)
            extra["egomcq_question_ms"] = extra["egomcq_question"].get("wall_ms")
            torch.cuda.empty_cache()
            extra["c4_train_step"] = guarded(extra_c4, dev)
            extra["c4_train_step_ms"] = extra["c4_train_step"].get("ms")
        line["extra"] = extra
    emit(line)


def run_train(ctx):
    """c4: one GPU's share of the pre-training step."""
    args, cfg, rank, world, dev, emit, dist = (ctx[k] for k in ("args", "cfg", "rank", "world", "dev", "emit", "dist"))
    barrier, timed = make_timers(ctx)
    warmup = max(3, args.warmup)
    B, T, nq = cfg["batch"], cfg["frames"], cfg["nq"]
    assert T == 4 and nq == 12, "c4 is defined at 4 frames, nq = 12"
    ts = TrainShare(B, dev, world=world, rank=rank, on_device_init=False)
    for _ in range(warmup):
        ts.step()
    sampler = ClockSampler(ctx["local"])
    if rank == 0:
        sampler.start()
    ms_total, _, per_rank = timed(lambda: ts.step(), args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        params = torch.cat([p.detach().flatten() for p in ts.model.parameters()])    # after the last optimizer step
        write_outputs(args.dump_outputs, dict(ts.outputs, decoder_params=params))
    ms_step = ms_total / args.steps
    value = world * B / (ms_step * 1e-3)
    ts.step(timed_parts=True)
    parts = dict(ts.marks)

    e2e = None
    if not args.no_e2e:
        buf = torch.empty_like(ts.host_video, device=dev)

        def e2e_step():
            buf.copy_(ts.host_video, non_blocking=True)
            return float(ts.step(buf).item())             # the loss is read back every step (run/train.py logs it)
        for _ in range(2):
            e2e_step()
        ms = timed(e2e_step, args.steps)[0] / args.steps
        e2e = {"value": world * B / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms,
               "h2d_bytes_per_step": ts.host_video.numel() * 4, "d2h_bytes_per_step": 4}
    vis, dec = ts.clip.visual, ts.model
    # the dominant kernel is still the backbone's tcgen05 GEMM; its per-class times come from one profiled step.  EVERY rank
    # takes this step: at world > 1 it contains the packed all-gather (rank 0 stepping alone would wait for its peers forever)
    if rank == 0:
        vis.set_profile(True)
        vis.profile()
    ts.step()
    torch.cuda.synchronize()
    if rank != 0:
        return
    prof = vis.profile()
    vis.set_profile(False)
    peaks = load_peaks()
    flops_clip = ts.flops_per_clip()
    M = B * (1 + T * 256)
    gemm_flops = {"gemm_qkv": 2.0 * M * 3072 * 1024, "gemm_proj": 2.0 * M * 1024 * 1024,
                  "gemm_fc1": 2.0 * M * 4096 * 1024, "gemm_fc2": 2.0 * M * 1024 * 4096}
    g_ms = sum(prof[k][0] for k in gemm_flops if k in prof)
    g_fl = sum(gemm_flops[k] * prof[k][1] for k in gemm_flops if k in prof)
    gemm_tflops = g_fl / (g_ms * 1e-3) / 1e12 if g_ms > 0 else 0.0
    line = {
        "metric": metric_name(T, nq) + " training step", "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": workload_string(cfg), "name": args.config, "clips_per_gpu": B, "frames": T, "nq": nq,
                   "captions_per_gpu": B * 5, "l2": "inputs larger than L2 (%.0f MB clips/step)" % (ts.host_video.numel() * 4 / 1e6),
                   "parallelism": "dp%d" % world, "forward_flops_per_clip": flops_clip,
                   "forward_tflops_per_gpu": value / world * flops_clip / 1e12, "parts_ms": parts,
                   "kernel_ms_per_step": {k: {"ms_per_step": v[0], "launches_per_step": v[1]} for k, v in prof.items()}},
        "roofline": {"bound": "tensor", "kernel": "gemm_kernel (tcgen05, frozen backbone's qkv/proj/fc1/fc2 launches)",
                     "achieved": gemm_tflops, "peak": peaks["sustained"], "unit": "TFLOP/s",
                     "frac": gemm_tflops / peaks["sustained"], "peak_source": peaks["source"] + " sustained bf16",
                     "share_of_step": g_ms / ms_step if ms_step > 0 else None, "traffic": None},
        "clocks": clocks, "gpu_launches": (vis.last_launches() + dec.last_launches()) * args.steps,
        "rank_ms_per_step": rank_spread(per_rank, args.steps),
    }
    if e2e:
        line["e2e"] = e2e
    emit(line)


if __name__ == "__main__":
    main()
