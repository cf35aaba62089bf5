#!/usr/bin/env python
"""Benchmark of the X3D forward path (BASELINE.json metric: X3D-M clips/sec at 1/2/4/8 B200).

    python bench.py --gpus N --steps K --warmup W                      # our CUDA path
    python bench.py --impl reference --gpus N --steps K --warmup W     # CPU reference arm
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...   # one rank per GPU
    python bench.py ... --dump-outputs DIR     # also write the last timed step's outputs as DIR/*.npy

A "step" = one forward pass over one batch of synthetic clips of the workload's shape
(default workload: BASELINE.json configs[2], X3D-M 10-view eval at 16x256x256, bf16,
12 videos = 120 clips per GPU per step).  Prints ONE JSON line on rank 0; its headline fields are
the m256x10 workload, and `configs` carries the other BASELINE configs (X3D-S 13x182^2, X3D-M
16x224^2, X3D-L 16x356^2 forward; the X3D-M training step) measured in the same run, >= 10 timed
steps each, at the same number of ranks.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOADS = {
    # name: (variant, T, S, views, default clips/GPU/step, dtype)
    "xs160": ("X3D_XS", 4, 160, 1, 8, "float32"),          # BASELINE configs[0]
    "s182": ("X3D_S", 13, 182, 1, 64, "bfloat16"),          # configs[1]
    # 12 videos per step: measured 7503 / 7982 / 8157 / 8300 / 8462 / 8488 clips/s at 40 / 60 / 80 / 100 / 120 / 160
    # clips per step (fixed per-launch costs of the 97 kernels; BASELINE configs[2] does not fix the batch)
    "m256x10": ("X3D_M", 16, 256, 10, 120, "bfloat16"),     # configs[2]  (metric config)
    "m224": ("X3D_M", 16, 224, 1, 64, "bfloat16"),          # north_star target shape
    "l356": ("X3D_L", 16, 356, 1, 32, "bfloat16"),          # configs[3]
    "train_m224": ("X3D_M", 16, 224, 1, 32, "float32"),     # configs[4]: one training step
}
METRIC = "X3D-M clips/sec"
DUMP_LIMIT_BYTES = 64 << 20      # --dump-outputs writes at most this much
FFMA2_PEAK_TMACS = 34.9          # measured packed-FFMA2 rate of this part, profiles/r01_microbench_fma_copy.txt


def workload_name(workload):
    """The `config.workload` string: identical for the repo arm and the reference arm (the
    driver compares them), batch sizes are separate keys."""
    variant, T, S, views, _, _ = WORKLOADS[workload]
    if workload.startswith("train"):
        return f"{variant} training step {T}x{S}x{S}"
    return f"{variant} {T}x{S}x{S}, {views}-view eval"
FALLBACK_HBM_GBS, FALLBACK_BF16_TFLOPS = 6650.0, 1590.0


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d["hbm_gbs"], d.get("bf16_tflops_sustained", d["bf16_tflops"]), "measured"
    return FALLBACK_HBM_GBS, FALLBACK_BF16_TFLOPS, "fallback"


def algorithmic_work(arch, T, H, W, esize):
    """Compulsory bytes and MACs per clip and per kernel class, TRUE channel counts
    (SURVEY.md section 8d / Appendix D: each kernel's logical input read once + output written
    once; weights excluded).  Classes follow the launches this build issues."""
    from x3d_tf_b200.arch import plan_shapes
    plan = plan_shapes(arch, T, H, W)
    c1 = arch.stem_channels
    out = {k: {"bytes": 0.0, "macs": 0.0} for k in
           ("stem", "a", "b", "ab", "c", "shortcut", "conv5", "head")}
    out["stem"]["bytes"] = (plan.input.P * 3 + plan.stem.P * c1) * esize
    out["stem"]["macs"] = plan.stem.P * c1 * (27 + arch.temp_filter)
    level = plan.stem
    for b in arch.blocks:
        p_in = level.P
        p_out = plan.stages[b.stage].P
        out["a"]["bytes"] += (b.cin + b.cinner) * p_in * esize
        out["a"]["macs"] += b.cin * b.cinner * p_in
        out["b"]["bytes"] += b.cinner * (p_in + p_out) * esize
        out["b"]["macs"] += 27 * b.cinner * p_out
        # fused expand+channelwise launch: only the block input and the channelwise output touch HBM
        out["ab"]["bytes"] += (b.cin * p_in + b.cinner * p_out) * esize
        out["ab"]["macs"] += b.cin * b.cinner * p_in + 27 * b.cinner * p_out
        out["c"]["bytes"] += (b.cinner + 2 * b.cout) * p_out * esize      # in + residual + out
        out["c"]["macs"] += b.cinner * b.cout * p_out
        if b.has_shortcut:
            out["shortcut"]["bytes"] += (b.cin + b.cout) * p_out * esize
            out["shortcut"]["macs"] += b.cin * b.cout * p_out
        level = plan.stages[b.stage]
    cl, c5 = arch.blocks[-1].cout, arch.conv5_channels
    out["conv5"]["bytes"] = (cl + c5) * level.P * esize
    out["conv5"]["macs"] = cl * c5 * level.P
    out["head"]["bytes"] = c5 * level.P * esize
    out["head"]["macs"] = c5 * arch.fc1_channels + arch.fc1_channels * arch.num_classes
    return out


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap",
               0x8: "hw_slowdown", 0x10: "sync_boost", 0x20: "sw_thermal_slowdown",
               0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown",
               0x100: "display_clock_setting"}

    def __init__(self, index: int, period: float = 0.05):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.sm, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        while not self._stop_evt.is_set():
            try:
                self.sm.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                mask = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) \
                    if hasattr(self.nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if mask & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def finish(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml_unavailable"]}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.sm)}


def physical_gpu_index(local_rank: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


def build_model(workload, graph=True):
    from x3d_tf_b200 import model as M
    from x3d_tf_b200.arch import build_arch
    from x3d_tf_b200.config import get_config
    from x3d_tf_b200.synth import synthetic_weights
    variant, T, S, views, clips, dtype = WORKLOADS[workload]
    cfg = get_config(variant, freeze=False)
    cfg.TEST.NUM_TEMPORAL_VIEWS, cfg.TEST.NUM_SPATIAL_CROPS = views, 1
    cfg.freeze()
    M.reset_block_counters()
    m = M.X3D(cfg, dtype=dtype, use_cuda_graph=graph)
    arch = build_arch(cfg)
    W = synthetic_weights(arch, seed=1111)
    m.set_weights_dict(W)
    return m, cfg, arch, W


def device_clips(n, T, S, cfg, dtype, device, seed):
    """Synthetic normalised clips generated on the device (uniform u8 pixels -> (x/255-mean)/std)."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    u8 = torch.randint(0, 256, (n, T, S, S, 3), generator=g, device=device, dtype=torch.uint8)
    mean = torch.tensor(cfg.DATA.MEAN, device=device, dtype=torch.float32)
    std = torch.tensor(cfg.DATA.STD, device=device, dtype=torch.float32)
    out = torch.empty((n, T, S, S, 3), device=device, dtype=dtype)
    for i in range(n):          # clip by clip: bounded temporary memory
        out[i] = ((u8[i].float() / 255.0 - mean) / std).to(dtype)
    return out


def cpu_reference_clips_per_s(workload, steps, warmup, budget_s, clips_per_step=None):
    """The reference's algorithm on the host cores: the torch-CPU fp32 restatement in oracle/
    (TensorFlow itself cannot be installed here -- DESIGN.md).  Returns (clips/s, info)."""
    from oracle import x3d_oracle as O
    from x3d_tf_b200.arch import build_arch
    from x3d_tf_b200.config import get_config
    from x3d_tf_b200.synth import synthetic_clips, synthetic_weights
    variant, T, S, views, _, _ = WORKLOADS[workload]
    cfg = get_config(variant)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    spec = O.OracleSpec.from_cfg(cfg, )
    spec.num_preds = 1
    W = synthetic_weights(build_arch(cfg), seed=1111)
    one = synthetic_clips(1, T, S, S, cfg.DATA.MEAN, cfg.DATA.STD, seed=1)
    t0 = time.perf_counter()
    O.forward(W, spec, one, torch.float32, channels_last=True)
    t1 = time.perf_counter() - t0            # includes first-touch cost; upper bound per clip
    if clips_per_step is None:
        clips_per_step = int(max(1, min(8, budget_s / max(t1, 1e-3) / max(steps + warmup, 1))))
    x = synthetic_clips(clips_per_step, T, S, S, cfg.DATA.MEAN, cfg.DATA.STD, seed=2)
    # BASELINE.md section 3 protocol: all host threads, inference_mode, channels_last_3d
    for _ in range(warmup):
        O.forward(W, spec, x, torch.float32, channels_last=True)
    t0 = time.perf_counter()
    for _ in range(steps):
        O.forward(W, spec, x, torch.float32, channels_last=True)
    dt = time.perf_counter() - t0
    return clips_per_step * steps / dt, {
        "cores": cores, "kind": "port", "clips_per_step": clips_per_step,
        "sample": f"{steps} steps x {clips_per_step} clips of {variant} {T}x{S}x{S} fp32 "
                  f"(torch-CPU restatement of model.py, {cores} threads, inference_mode, "
                  f"channels_last_3d), {warmup} warm-up",
        "ms_per_step": dt / steps * 1e3}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    variant, T, S, views, clips, dtype = WORKLOADS[args.workload]
    v, info = cpu_reference_clips_per_s(args.workload, args.steps, args.warmup, budget_s=150.0)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "clips/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": info["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(args.workload),
                       "clips_per_step": info["clips_per_step"],
                       "note": "CPU restatement of the reference (TensorFlow unavailable); each step is a "
                               "bounded sample of the workload's clips"},
            "cpu_baseline": {"value": v, "unit": "clips/s", "cores": info["cores"],
                             "kind": info["kind"], "sample": info["sample"]},
            "e2e": {"value": v, "unit": "clips/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def _dist_env():
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    return world, rank, local_rank


def _max_over_ranks(ms: float, device, world: int) -> float:
    import torch.distributed as dist
    t = torch.tensor([ms], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def _barrier(world: int):
    import torch.distributed as dist
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def kernel_traffic(kernel: str, workload: str, clips: int):
    """DRAM bytes per launch (read + write, averaged over the launches of one step) of `kernel`
    from a committed ncu capture of this workload -- only when the capture was taken from the
    kernel source that is in the tree NOW (sha256 of the .cu file), so the figure cannot go stale
    silently; null otherwise."""
    import hashlib
    tp = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if not os.path.exists(tp):
        return None, "no committed capture"
    with open(tp) as f:
        entries = json.load(f)
    for e in entries:
        if e.get("kernel") != kernel or e.get("workload") != workload or e.get("clips") != clips:
            continue
        srcs = [os.path.join(ROOT, x) for x in e.get("source", "").split(",")]
        if not all(os.path.exists(x) for x in srcs):
            continue
        h = hashlib.sha256()
        for x in srcs:
            with open(x, "rb") as f:
                h.update(f.read())
        if h.hexdigest() != e.get("source_sha256"):
            return None, f"capture {e.get('capture')} predates the current {e.get('source')}"
        return e["bytes_per_launch"], e.get("capture")
    return None, "no capture for this kernel/workload"


def dump_outputs(outdir, arrays):
    """Writes each array as `outdir/<name>.npy` in float32, so that two builds can be compared output
    for output on the same seeded inputs."""
    arrays = {k: np.ascontiguousarray(v, dtype=np.float32) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs would write {total / 2**20:.1f} MB "
                         f"(limit {DUMP_LIMIT_BYTES >> 20} MB): lower --clips")
    os.makedirs(outdir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(outdir, name + ".npy"), a)


def measure_forward(workload, clips, steps, warmup, device, world, rank, want_model=False, want_outputs=False):
    """Device-resident throughput of one forward workload (CUDA-graph replays on the captured
    input buffer, CUDA events, max over ranks) + per-kernel-class attribution of one eager pass.
    `want_outputs`: res["outputs"] holds what the last timed step returned (probabilities, and the
    logits the model exposes as `last_logits`), copied to the host after the timed region."""
    from x3d_tf_b200 import ops
    variant, T, S, views, dclips, dtype_name = WORKLOADS[workload]
    clips = clips or dclips
    clips -= clips % views
    tdt = torch.bfloat16 if dtype_name == "bfloat16" else torch.float32
    esize = 2 if tdt == torch.bfloat16 else 4
    model, cfg, arch, _ = build_model(workload, graph=True)
    x = device_clips(clips, T, S, cfg, tdt, device, seed=1111 + rank)
    model(x, copy=False)                       # eager warm-up + capture
    static_in = model.static_input(x.shape, tdt)
    static_in.copy_(x)
    del x
    for _ in range(warmup):
        probs = model(static_in, copy=False)
    _barrier(world)
    ops.Profiler.launches = 0
    sampler = ClockSampler(physical_gpu_index(device.index))
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        probs = model(static_in, copy=False)
    e1.record()
    _barrier(world)
    clocks = sampler.finish()
    ms_max = _max_over_ranks(e0.elapsed_time(e1), device, world)
    value = clips * world * steps / (ms_max / 1e3)
    # the graph's output buffers: copied now, before any later pass can overwrite them
    outputs = {"probs": probs.float().cpu().numpy(),
               "logits": model.last_logits.float().cpu().numpy()} if want_outputs else None

    # ---- per-class attribution: one eager, event-bracketed pass over the same batch
    model._use_graph = False
    ops.Profiler.start()
    model(static_in)
    recs = ops.Profiler.stop()
    model._use_graph = True
    work = algorithmic_work(arch, T, S, S, esize)
    hbm, tflops, peak_kind = peaks()
    classes = {}
    for tag, name, dt_ms in recs:
        if tag.startswith("head_"):
            sub = classes.setdefault("head_parts", {})
            sub[tag] = round(sub.get(tag, 0.0) + dt_ms, 4)
            tag = "head"
        c = classes.setdefault(tag, {"ms": 0.0, "launches": 0})
        c["ms"] += dt_ms
        c["launches"] += 1
    for tag, c in classes.items():
        if tag == "head_parts":
            continue
        if tag in work:
            c["GBps"] = work[tag]["bytes"] * clips / (c["ms"] * 1e-3) / 1e9
            c["hbm_frac"] = c["GBps"] / hbm
            c["tflops"] = 2 * work[tag]["macs"] * clips / (c["ms"] * 1e-3) / 1e12
        c["ms"] = round(c["ms"], 4)
    fused = "ab" in classes
    stencil_macs = work["b"]["macs"] * clips
    if fused:
        b = dict(classes["ab"])
        b_bytes = work["ab"]["bytes"] * clips
        kernel, src = "ab_persist_kernel", "x3d_tf_b200/csrc/x3d_ab_persist.cu"
        kname = ("ab_persist_kernel (expand 1x1x1 + BN + ReLU -> channelwise 3x3x3 + BN + swish / SE sums; "
                 "external bytes only: block input read + channelwise output written)")
        if "b" in classes:                     # layers without a fused tile plan ran the two kernels
            b["note"] = f"{classes['b']['launches']} layers ran unfused (no tile plan)"
    else:
        b = classes.get("b", {"ms": float("nan"), "launches": 0})
        b_bytes = work["b"]["bytes"] * clips
        kernel, src = "dw_tma_kernel,dw_planar_kernel", "x3d_tf_b200/csrc/x3d_dw_tma.cu,x3d_tf_b200/csrc/x3d_dw_planar.cu"
        kname = ("channelwise 3x3x3 + BN + swish / SE sums, all launches of the step: dw_planar_kernel on the "
                 "stride-1 layers it tiles without waste, dw_tma_kernel on the rest")
    achieved = b_bytes / (b["ms"] * 1e-3) / 1e9
    traffic, traffic_src = kernel_traffic(kernel, workload, clips)
    fma_tmacs = stencil_macs / (b["ms"] * 1e-3) / 1e12
    roofline = {"kernel": kname,
                # the 27-tap stencil runs on the fp32 FMA pipe (packed FFMA2): at bf16 it needs
                # 27 MACs per 3.2 bytes unfused (FMA floor ~ HBM floor) and per ~1.2 external bytes
                # fused, so the binding resource is the FMA pipe first, HBM second
                "bound": "fma+hbm" if not fused else "fma (hbm second)",
                "achieved": achieved, "peak": hbm, "unit": "GB/s", "frac": achieved / hbm,
                "fma_tmacs": fma_tmacs, "fma_peak_tmacs": FFMA2_PEAK_TMACS,
                "fma_frac": fma_tmacs / FFMA2_PEAK_TMACS,
                "fma_peak_source": "measured packed-FFMA2 rate, profiles/r01_microbench_fma_copy.txt",
                "traffic": traffic, "traffic_source": traffic_src,
                "algorithmic_bytes_per_launch": b_bytes / max(b["launches"], 1),
                "peak_source": f"{peak_kind} (MEASURED_PEAKS.json hbm_gbs)",
                "launches_per_step": b["launches"],
                "algorithmic_bytes_per_step": b_bytes,
                "avg_launch_ms": b["ms"] / max(b["launches"], 1),
                "how": "CUDA events around each launch of one eager pass over the timed batch"}
    if fused:
        roofline["unfused_equivalent_GBps"] = (work["a"]["bytes"] + work["b"]["bytes"]) * clips / (b["ms"] * 1e-3) / 1e9
    total_bytes = sum(w["bytes"] for k, w in work.items() if k != "ab") * clips
    pw_macs = (work["a"]["macs"] + work["c"]["macs"]) * clips
    pw_ms = classes.get("a", classes.get("ab", {"ms": 0}))["ms"] + classes.get("c", {"ms": 0})["ms"]
    res = {"workload": workload, "name": workload_name(workload), "clips": clips, "views": views,
           "T": T, "S": S, "tdt": tdt, "esize": esize, "value": value, "ms_max": ms_max,
           "steps": steps, "clocks": clocks, "launches_per_step": len(recs), "roofline": roofline,
           "classes": classes,
           "whole_model_hbm_frac_layerwise": total_bytes / (ms_max / steps * 1e-3) / 1e9 / hbm,
           "pointwise_tensor_pipe_util": (2 * pw_macs / (pw_ms * 1e-3) / 1e12 / tflops) if pw_ms else None,
           "outputs": outputs}
    if want_model:
        res.update(model=model, static_in=static_in, probs=probs, cfg=cfg)
    return res


def config_entry(r):
    """One element of the line's `configs` array (a BASELINE config measured beside the headline)."""
    rf = r["roofline"]
    return {"workload": r["name"], "clips_per_gpu_per_step": r["clips"], "value": r["value"], "unit": "clips/s",
            "ms_per_step": r["ms_max"] / r["steps"], "steps": r["steps"],
            "dtype": "bf16" if r["tdt"] == torch.bfloat16 else "f32",
            "stencil_kernel": rf["kernel"].split(" ")[0], "stencil_ms": rf["avg_launch_ms"] * rf["launches_per_step"],
            "stencil_hbm_frac": rf["frac"], "stencil_fma_frac": rf["fma_frac"],
            "whole_model_hbm_frac_layerwise": r["whole_model_hbm_frac_layerwise"],
            "pointwise_tensor_pipe_util": r["pointwise_tensor_pipe_util"],
            "gpu_launches_per_step": r["launches_per_step"], "clocks_sm_mhz": r["clocks"].get("sm_mhz")}


def run_b200(args):
    import torch.distributed as dist

    world, rank, local_rank = _dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU path; use --impl reference)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
    warmup = max(args.warmup, 3)               # the contract's minimum; the line reports what ran

    r = measure_forward(args.workload, args.clips, args.steps, warmup, device, world, rank, want_model=True,
                        want_outputs=bool(args.dump_outputs))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, r["outputs"])
    model, static_in, probs, cfg = r.pop("model"), r.pop("static_in"), r.pop("probs"), r.pop("cfg")
    clips, T, S, views, tdt, esize = r["clips"], r["T"], r["S"], r["views"], r["tdt"], r["esize"]
    extra = {"whole_model_hbm_frac_layerwise": r["whole_model_hbm_frac_layerwise"],
             "pointwise_tensor_pipe_util": r["pointwise_tensor_pipe_util"],
             "kernel_classes": r["classes"]}

    def e2e_measure(host_in, want, n_e2e, api):
        # public API: X3D.predict(iterable of HOST batches) -> host probabilities; every step
        # copies its clips host->device (pinned, copy stream, overlapped with the previous
        # step's forward) and its probabilities device->host inside the timed region
        got = None
        for got in model.predict(host_in for _ in range(3)):
            pass
        if not torch.allclose(got, want, rtol=0, atol=1e-6):
            raise SystemExit("bench.py: predict() result differs from the device-resident result")
        _barrier(world)
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for _ in model.predict(host_in for _ in range(n_e2e)):
            pass
        s1.record()
        _barrier(world)
        te = _max_over_ranks(s0.elapsed_time(s1), device, world)
        return {"value": clips * world * n_e2e / (te / 1e3), "unit": "clips/s",
                "h2d_bytes_per_step": host_in.numel() * host_in.element_size(),
                "d2h_bytes_per_step": want.numel() * 4, "steps": n_e2e, "api": api}

    # ---- end to end through the public API with HOST buffers (pinned), copies inside the region.
    # Headline: decoded uint8 frames, the format the reference's input pipeline delivers before
    # utils.normalize (dataloader.py:93-121, utils.py:42-72); the normalisation runs on the device.
    e2e = None
    if not args.no_e2e:
        n_e2e = max(3, min(args.steps, 30))      # (the first step's copy is not overlapped: more steps amortise it)
        if tdt == torch.bfloat16:
            g8 = torch.Generator()
            g8.manual_seed(2222 + rank)
            host_u8 = torch.randint(0, 256, (clips, T, S, S, 3), dtype=torch.uint8, generator=g8).pin_memory()
            want8 = model(host_u8.to(device)).float().cpu()
            e2e = e2e_measure(host_u8, want8, n_e2e,
                              "X3D.predict on pinned-host uint8 frames: per step H2D copy (copy stream, overlapped "
                              "with the previous step's forward), utils.normalize on the device, forward, D2H of "
                              "the probabilities")
            del host_u8
        host_in = torch.empty((clips, T, S, S, 3), dtype=tdt).pin_memory()
        host_in.copy_(static_in.cpu())
        want = probs.float().cpu()
        e2e_f = e2e_measure(host_in, want, n_e2e,
                            "X3D.predict on pinned-host, host-normalised clips in the compute dtype")
        del host_in
        if e2e is None:
            e2e = e2e_f
        else:
            extra["e2e_bf16_clips"] = e2e_f

    # ---- the other BASELINE configs, measured beside the headline at the same number of ranks
    configs = []
    if not args.no_configs and args.workload == "m256x10":
        del model, static_in, probs
        torch.cuda.empty_cache()
        for wl in ("s182", "m224", "l356"):
            rr = measure_forward(wl, 0, max(args.config_steps, 10), warmup, device, world, rank)
            configs.append(config_entry(rr))
            torch.cuda.empty_cache()
        tr = measure_train("train_m224", 0, max(args.config_steps, 10), warmup, device, world, rank)
        configs.append({k: tr[k] for k in ("workload", "clips_per_gpu_per_step", "value", "unit", "ms_per_step", "steps",
                                           "dtype", "allreduce_ms", "allreduce_bytes", "gpu_launches_per_step",
                                           "hbm_frac_of_3x_forward_bytes")})

    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            v, info = cpu_reference_clips_per_s(args.workload, steps=2, warmup=1, budget_s=20.0)
            cpu = {"value": v, "unit": "clips/s", "cores": info["cores"], "kind": info["kind"],
                   "sample": info["sample"]}
        line = {"metric": METRIC, "value": r["value"], "unit": "clips/s", "n_gpus": world,
                "steps": args.steps, "warmup": warmup,
                "ms_per_step": r["ms_max"] / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "bf16" if tdt == torch.bfloat16 else "f32",
                "data": "synthetic",
                "config": {"workload": workload_name(args.workload),
                           "clips_per_gpu_per_step": clips, "videos_per_gpu_per_step": clips // views,
                           "weights": "synthetic (checkpoint names/shapes; data shards absent)",
                           "l2": f"inputs larger than L2: the clip batch is "
                                 f"{clips * T * S * S * 3 * esize / 1e6:.0f} MB and every "
                                 "intermediate tensor is larger",
                           "cuda_graph": True, "parallelism": f"dp{world} (videos sharded, no collective)"},
                "clocks": r["clocks"], "e2e": e2e, "gpu_launches": r["launches_per_step"] * args.steps,
                "roofline": r["roofline"], "cpu_baseline": cpu, **extra}
        if configs:
            line["configs"] = configs
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def measure_train(workload, clips, steps, warmup, device, world, rank, want_outputs=False):
    """BASELINE configs[4]: one X3D-M training step (forward, backward, NCCL gradient all-reduce,
    SGD-Nesterov) per bench step; batch 32 per GPU, 16x224x224, fp32 (the reference's default
    precision; train.py:85-152).  value = clips trained per second over all ranks.
    `want_outputs`: res["outputs"] holds the per-clip losses the last timed step returned."""
    import torch.distributed as dist
    from x3d_tf_b200 import _lib
    from x3d_tf_b200.arch import build_arch
    from x3d_tf_b200.config import get_config
    from x3d_tf_b200.synth import synthetic_weights
    from x3d_tf_b200.training import X3DTrainer, lr_schedule

    variant, T, S, _, dclips, _ = WORKLOADS[workload]
    clips = clips or dclips
    cfg = get_config(variant)
    arch = build_arch(cfg)
    tr = X3DTrainer(cfg, device=device, world=world, rank=rank).load(synthetic_weights(arch, seed=1111))
    x = device_clips(clips, T, S, cfg, torch.float32, device, seed=1111 + rank)
    g = torch.Generator(device=device)
    g.manual_seed(7 + rank)
    labels = torch.randint(0, cfg.NETWORK.NUM_CLASSES, (clips,), generator=g, device=device, dtype=torch.int32)
    lr = lr_schedule(cfg, 0)

    for _ in range(warmup):
        loss = tr.step(x, labels, lr)
    _barrier(world)
    c0 = _lib.calls
    sampler = ClockSampler(physical_gpu_index(device.index))
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = tr.step(x, labels, lr)
    e1.record()
    _barrier(world)
    clocks = sampler.finish()
    launches = _lib.calls - c0
    ms_max = _max_over_ranks(e0.elapsed_time(e1), device, world)
    value = clips * world * steps / (ms_max / 1e3)
    outputs = {"loss": loss.float().cpu().numpy()} if want_outputs else None

    # the exchange step alone: the same flat fp32 gradient arena, summed over the ranks
    ar_ms = 0.0
    if world > 1:
        for _ in range(3):
            dist.all_reduce(tr.g, op=dist.ReduceOp.SUM)
        _barrier(world)
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(10):
            dist.all_reduce(tr.g, op=dist.ReduceOp.SUM)
        a1.record()
        _barrier(world)
        ar_ms = _max_over_ranks(a0.elapsed_time(a1), device, world) / 10

    # end to end: clips and labels come from pinned host memory every step, the loss goes back
    host_x = torch.empty(x.shape, dtype=torch.float32).pin_memory()
    host_x.copy_(x.cpu())
    host_l = labels.cpu().pin_memory()
    n_e2e = max(3, min(steps, 5))
    _barrier(world)
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    for _ in range(n_e2e):
        x.copy_(host_x, non_blocking=True)
        labels.copy_(host_l, non_blocking=True)
        host_loss = tr.step(x, labels, lr).float().cpu()
    s1.record()
    _barrier(world)
    te = _max_over_ranks(s0.elapsed_time(s1), device, world)
    hbm, _, peak_kind = peaks()
    work = algorithmic_work(arch, T, S, S, 4)
    fwd_bytes = sum(w["bytes"] for k, w in work.items() if k != "ab") * clips
    frac = 3 * fwd_bytes / (ms_max / steps * 1e-3) / 1e9 / hbm
    res = {"workload": workload_name(workload), "clips_per_gpu_per_step": clips, "value": value, "unit": "clips/s",
           "ms_per_step": ms_max / steps, "steps": steps, "dtype": "f32", "clocks": clocks,
           "allreduce_ms": ar_ms, "allreduce_bytes": tr.layout.size * 4 if world > 1 else 0,
           "gpu_launches": launches, "gpu_launches_per_step": launches // max(steps, 1),
           "hbm_frac_of_3x_forward_bytes": frac, "hbm": hbm, "peak_kind": peak_kind,
           "e2e": {"value": clips * world * n_e2e / (te / 1e3), "unit": "clips/s",
                   "h2d_bytes_per_step": host_x.numel() * 4 + host_l.numel() * 4,
                   "d2h_bytes_per_step": host_loss.numel() * 4, "steps": n_e2e,
                   "api": "X3DTrainer.step on clips/labels copied from pinned host memory, per-clip losses read back"},
           "momentum": tr.momentum, "dropout": tr.dropout, "x_bytes": x.numel() * 4,
           "loss_mean": float(loss.float().mean().item()), "outputs": outputs}
    del tr, x, host_x
    torch.cuda.empty_cache()
    return res


def run_train(args):
    import torch.distributed as dist
    world, rank, local_rank = _dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU path)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
    warmup = max(args.warmup, 3)
    r = measure_train(args.workload, args.clips, args.steps, warmup, device, world, rank,
                      want_outputs=bool(args.dump_outputs))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, r["outputs"])
    if rank == 0:
        line = {"metric": "X3D-M training clips/sec", "value": r["value"], "unit": "clips/s", "n_gpus": world,
                "steps": args.steps, "warmup": warmup, "ms_per_step": r["ms_per_step"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": {"workload": r["workload"], "clips_per_gpu_per_step": r["clips_per_gpu_per_step"],
                           "optimizer": f"SGD-Nesterov momentum {r['momentum']}, L2, dropout {r['dropout']}, batch-statistics BN",
                           "exchange": ("one NCCL sum all-reduce of the flat fp32 gradient arena "
                                        f"({r['allreduce_bytes'] / 1e6:.2f} MB, {r['allreduce_ms']:.3f} ms alone)"
                                        if world > 1 else "single rank: no exchange"),
                           "l2": f"inputs larger than L2: the clip batch is {r['x_bytes'] / 1e6:.0f} MB",
                           "parallelism": f"dp{world}"},
                "clocks": r["clocks"], "gpu_launches": r["gpu_launches"], "e2e": r["e2e"],
                "roofline": {"kernel": "whole training step", "bound": "hbm",
                             "achieved": r["hbm_frac_of_3x_forward_bytes"] * r["hbm"], "peak": r["hbm"],
                             "unit": "GB/s", "frac": r["hbm_frac_of_3x_forward_bytes"],
                             "traffic": None, "peak_source": f"{r['peak_kind']} (MEASURED_PEAKS.json hbm_gbs)",
                             "how": "3 x the forward pass's algorithmic fp32 bytes (SURVEY.md 8d estimate) / step time"},
                "cpu_baseline": None, "loss_mean": r["loss_mean"]}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="m256x10", choices=list(WORKLOADS))
    ap.add_argument("--clips", type=int, default=0, help="clips per GPU per step (override)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the `configs` array (the other BASELINE configs)")
    ap.add_argument("--config-steps", type=int, default=10, help="timed steps of each `configs` entry (>= 10)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (float32; rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the CUDA path's outputs; the reference arm has none to write")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload.startswith("train"):
        run_train(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
