"""Measures clips built from decoded videos on the device (x3d_video_clips_u8, video.py).

    python tools/video_bench.py [--out profiles] [--quick]

Writes <out>/r03_video_{kernel,eval_e2e,train,cpu_baseline}.json, each with the card name and power
limit read in the same run:
  kernel        kernel time per batch (CUDA events around >= 50 launches after a warm-up) and achieved
                GB/s = (output bytes + distinct source bytes) / time, for X3D-M eval (10 views, S=256,
                12 videos of 300 frames at 360x480), X3D-M train (batch 32, jitter 256-320, crop 224) and
                X3D-L eval (10 views, S=356, 4 videos of 300 frames at 480x640); every batch's sources
                exceed the 126 MB L2;
  eval_e2e      X3D.evaluate clips/s at the headline shape (X3D-M bf16, 16x256^2, 10 views, 12 videos
                per step) from pre-cropped pinned uint8 clips and from VideoBatches, alternating in one
                run, with the computed host->device bytes per step of each and the host time to pack
                one VideoBatch (not part of the timed loop: both inputs are prepared ahead);
  train         training step time (X3D-M fp32, batch 32, crop 224) from VideoBatches and from
                pre-cropped pinned uint8 clips, alternating;
  cpu_baseline  the same eval resize + crops with torch on the CPU (F.interpolate bilinear,
                align_corners=False, all host threads): what building the clips costs without this path.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from x3d_tf_b200 import ops, video as V                      # noqa: E402
from x3d_tf_b200.arch import build_arch                      # noqa: E402
from x3d_tf_b200.config import get_config                    # noqa: E402
from x3d_tf_b200.synth import synthetic_weights              # noqa: E402


def card() -> dict:
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [s.strip() for s in q.split(",")]
        info.update(card=name, power_limit=power, max_sm_clock=clk)
    except Exception as e:                                  # recorded, not hidden
        info.update(card=info["device"], power_limit=f"not read ({type(e).__name__})")
    return info


def write(out_dir, name, rec):
    rec = dict(card(), **rec)
    path = os.path.join(out_dir, f"r03_video_{name}.json")
    with open(path, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec))


class Frames:
    """A decoded video of F frames whose frames come from a shared pool of random frames (frame f of
    video k is pool[(7 * k + f) % len(pool)]): the packed buffer holds F distinct frame copies as a
    real video would, without generating gigabytes of random host data."""
    def __init__(self, pool, F, k):
        self.pool, self.k = pool, k
        self.shape, self.dtype = (F,) + pool.shape[1:], pool.dtype

    def __getitem__(self, f):
        return self.pool[(7 * self.k + int(f)) % len(self.pool)]


def videos(n, F, H, W, seed):
    pool = np.random.default_rng(seed).integers(0, 256, size=(61, H, W, 3), dtype=np.uint8)
    return [Frames(pool, F, k) for k in range(n)]


def kernel_case(name, vids, plan, launches):
    t0 = time.perf_counter()
    b = V.pack(vids, plan)
    pack_s = time.perf_counter() - t0
    dev = torch.device("cuda")
    frames, off, desc = b.frames.to(dev), b.frame_off.to(dev), b.desc.to(dev)
    out = torch.empty(b.shape, dtype=torch.uint8, device=dev)
    for _ in range(5):
        ops.video_clips_u8(frames, off, desc, b.shape[1], b.shape[2], out=out)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(launches):
        ops.video_clips_u8(frames, off, desc, b.shape[1], b.shape[2], out=out)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / launches
    moved = out.numel() + b.frames.numel()
    return {"case": name, "clips_shape": list(b.shape), "launches": launches, "ms_per_batch": ms,
            "output_bytes": out.numel(), "distinct_source_bytes": b.frames.numel(),
            "achieved_GBps": moved / ms / 1e6, "host_pack_ms": pack_s * 1e3}


def eval_cfg(variant, views, S, T=16):
    cfg = get_config(variant, freeze=False)
    cfg.TEST.NUM_TEMPORAL_VIEWS, cfg.TEST.NUM_SPATIAL_CROPS = views, 1
    cfg.DATA.TEMP_DURATION, cfg.DATA.TEST_CROP_SIZE = T, S
    cfg.freeze()
    return cfg


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--quick", action="store_true", help="fewer steps (a rehearsal, not a measurement)")
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    if not torch.cuda.is_available():
        raise SystemExit("video_bench needs a CUDA device")
    torch.cuda.set_device(0)
    launches = 10 if a.quick else 60

    # ---- kernel
    cases = []
    vm = videos(12, 300, 360, 480, 1)
    cases.append(kernel_case("X3D-M eval 10 views S=256, 12 videos 300x360x480",
                             vm, V.eval_plan([v.shape for v in vm], 16, 10, 1, 256), launches))
    vt = videos(32, 300, 360, 480, 2)
    cases.append(kernel_case("X3D-M train batch 32 jitter 256-320 crop 224, 300x360x480",
                             vt, V.train_plan([v.shape for v in vt], 16, 5, (256, 320), 224, V.train_rng(0)),
                             launches))
    del vt
    vl = videos(4, 300, 480, 640, 3)
    cases.append(kernel_case("X3D-L eval 10 views S=356, 4 videos 300x480x640",
                             vl, V.eval_plan([v.shape for v in vl], 16, 10, 1, 356), launches))
    del vl
    write(a.out, "kernel", {"what": "x3d_video_clips_u8 kernel time per batch (CUDA events)", "cases": cases})

    # ---- evaluate end to end: pre-cropped pinned uint8 clips vs VideoBatch, alternating
    from x3d_tf_b200 import model as M
    M.reset_block_counters()
    cfg = eval_cfg("X3D_M", 10, 256)
    m = M.X3D(cfg, dtype="bfloat16").compile()
    m.set_weights_dict(synthetic_weights(build_arch(cfg)))
    groups = [vm, videos(12, 300, 360, 480, 4)]
    labels = np.arange(12, dtype=np.int32)
    vbs = []
    t0 = time.perf_counter()
    for g in groups:
        vbs.append(V.eval_batch(g, cfg))
    pack_ms = (time.perf_counter() - t0) * 1e3 / len(groups)
    clips = []
    for b in vbs:                                 # the same clips, built once and kept pinned on the host
        clips.append(b.clips("cuda").cpu().pin_memory())
    del groups, vm
    steps = 4 if a.quick else 20
    res = {"u8_clips": [], "video_batch": []}

    def run(kind, n):
        src = clips if kind == "u8_clips" else vbs
        data = [(src[i % 2], labels) for i in range(n)]
        torch.cuda.synchronize()
        t = time.perf_counter()
        m.evaluate(data)
        torch.cuda.synchronize()
        return time.perf_counter() - t

    run("u8_clips", 3); run("video_batch", 3)                      # graphs, staging buffers, pinned pools
    for _ in range(2):
        for kind in ("u8_clips", "video_batch"):
            res[kind].append(120 * steps / run(kind, steps))
    write(a.out, "eval_e2e", {
        "what": "X3D.evaluate clips/s, X3D-M bf16 16x256^2, 10 views, 12 videos (120 clips) per step, "
                "host clock around evaluate (ends in a device synchronise); two alternating rounds per input",
        "steps_per_round": steps,
        "u8_clips_clips_per_s": res["u8_clips"], "video_batch_clips_per_s": res["video_batch"],
        "h2d_bytes_per_step_u8_clips": int(clips[0].numel()),
        "h2d_bytes_per_step_video_batch": int(vbs[0].h2d_bytes),
        "source_videos": "300 frames, 360x480", "host_pack_ms_per_step": pack_ms})
    del m, clips, vbs
    torch.cuda.empty_cache()

    # ---- training step
    from x3d_tf_b200.training import X3DTrainer
    M.reset_block_counters()
    tcfg = get_config("X3D_M")
    tr = X3DTrainer(tcfg).load(synthetic_weights(build_arch(tcfg)))
    vt = videos(32, 300, 360, 480, 5)
    rng = V.train_rng(1)
    tvb = [V.train_batch(vt, tcfg, rng) for _ in range(2)]
    tclips = [b.clips("cuda").cpu().pin_memory() for b in tvb]
    del vt
    lab = torch.arange(32, dtype=torch.int32, device="cuda")
    mean, std = tuple(tcfg.DATA.MEAN), tuple(tcfg.DATA.STD)

    def step(kind, i):
        x = tvb[i % 2].clips("cuda") if kind == "video_batch" else tclips[i % 2].to("cuda", non_blocking=True)
        return tr.step(ops.normalize_u8(x, mean, std, torch.float32), lab, 0.0)

    tsteps = 2 if a.quick else 8
    times = {"u8_clips": [], "video_batch": []}
    for kind in ("u8_clips", "video_batch"):
        step(kind, 0)
    for _ in range(2):
        for kind in ("u8_clips", "video_batch"):
            torch.cuda.synchronize()
            t = time.perf_counter()
            for i in range(tsteps):
                step(kind, i)
            torch.cuda.synchronize()
            times[kind].append((time.perf_counter() - t) * 1e3 / tsteps)
    write(a.out, "train", {
        "what": "X3DTrainer.step ms (X3D-M fp32, batch 32, crop 224, lr 0) including the input's H2D copy and "
                "normalisation; host clock around steps ending in a device synchronise; two alternating rounds",
        "steps_per_round": tsteps, "u8_clips_ms_per_step": times["u8_clips"],
        "video_batch_ms_per_step": times["video_batch"],
        "h2d_bytes_per_step_u8_clips": int(tclips[0].numel()), "h2d_bytes_per_step_video_batch": int(tvb[0].h2d_bytes)})
    del tr, tvb, tclips
    torch.cuda.empty_cache()

    # ---- CPU baseline: the eval resize + crop of one video with torch on the host
    import torch.nn.functional as Fn
    torch.set_num_threads(os.cpu_count() or 1)
    v = videos(1, 300, 360, 480, 6)[0]
    plan = V.eval_plan([v.shape], 16, 10, 1, 256)
    reps = 1 if a.quick else 3
    t = time.perf_counter()
    for _ in range(reps):
        idx = np.unique(plan.frames)
        x = torch.from_numpy(np.stack([v[f] for f in idx])).permute(0, 3, 1, 2).float()
        _, _, rh, rw, y0, x0, _ = plan.desc[0]
        r = Fn.interpolate(x, size=(int(rh), int(rw)), mode="bilinear", align_corners=False)
        r = r.clamp_(0, 255).to(torch.uint8).permute(0, 2, 3, 1)
        pos = {f: i for i, f in enumerate(idx.tolist())}
        sel = torch.as_tensor([pos[f] for f in plan.frames.reshape(-1).tolist()])
        clips_cpu = r[sel][:, y0:y0 + 256, x0:x0 + 256].contiguous()
    sec = (time.perf_counter() - t) / reps
    write(a.out, "cpu_baseline", {
        "what": "torch CPU F.interpolate(bilinear, align_corners=False) of the 160 sampled frames of one "
                "300x360x480 video to 256x341, then the 10 centre-cropped views (X3D-M eval)",
        "threads": torch.get_num_threads(), "cpu_count": os.cpu_count(), "seconds_per_video": sec,
        "videos_per_s": 1.0 / sec, "clips_per_s": 10.0 / sec, "clips_shape": list(clips_cpu.shape)})


if __name__ == "__main__":
    main()
