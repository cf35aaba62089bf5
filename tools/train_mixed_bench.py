"""Training step time under the 'float32' and 'mixed_bfloat16' policies (X3D-M, batch 32, 16 x 224^2
by default), and the device time of the two pointwise-GEMM classes of each step.

    python tools/train_mixed_bench.py [--out_dir profiles] [--rounds 6] [--steps 10]

Writes `r07_train_mixed_step.json` (ms per step: after warm-up the policies alternate, `--steps`
steps each per round, CUDA events around each run of steps) and `r07_train_mixed_kernels.json`
(one profiled step per policy in a separate pass: torch.profiler's CUDA kernel times, summed per
GEMM class).  The card's name, power limit and maximum SM clock are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
from collections import defaultdict

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

# kernel-name patterns of the two GEMM classes (both policies): forward + backward-data (with the
# weight preparation and the shortcut's row gather / legacy path), and backward-filter
CLASSES = {
    "pw_fwd_dgrad": r"pw_tf32_tc_kernel|pw_bf16_train_tc_kernel|tf32_split_kernel|bf16_round_kernel|gather_rows|pw_fwd_kernel|pw_kernel",
    "pw_wgrad": r"pw_wgrad",
}


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else ""
    return {"device": torch.cuda.get_device_name(), "nvidia_smi": line}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--variant", default="X3D_M")
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--frames", type=int, default=16)
    ap.add_argument("--size", type=int, default=224)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out_dir", default="profiles")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    from x3d_tf_b200.arch import build_arch
    from x3d_tf_b200.config import get_config
    from x3d_tf_b200.synth import synthetic_weights
    from x3d_tf_b200.training import X3DTrainer
    torch.cuda.set_device(0)
    cfg = get_config(a.variant)
    W = synthetic_weights(build_arch(cfg), seed=1)
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(a.batch, a.frames, a.size, a.size, 3, device="cuda", generator=g)
    y = torch.randint(0, cfg.NETWORK.NUM_CLASSES, (a.batch,), device="cuda", dtype=torch.int32, generator=g)
    pols = ("float32", "mixed_bfloat16")
    tr = {p: X3DTrainer(cfg, precision=p).load(W) for p in pols}
    lr = 1e-4
    for p in pols:
        for _ in range(a.warmup):
            tr[p].step(x, y, lr)
    torch.cuda.synchronize()
    ms = defaultdict(list)
    for _ in range(a.rounds):
        for p in pols:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.steps):
                tr[p].step(x, y, lr)
            e1.record()
            e1.synchronize()
            ms[p].append(e0.elapsed_time(e1) / a.steps)
    info = card()
    step = {"what": f"training step ms, {a.variant} batch {a.batch} x {a.frames} x {a.size}^2, SGD, one GPU; "
                    f"policies alternate, {a.steps} steps per run, {a.rounds} runs each after {a.warmup} warm-up steps",
            **info, "ms_per_step": {p: {"median": float(np.median(v)), "min": float(np.min(v)),
                                        "max": float(np.max(v)), "runs": v} for p, v in ms.items()}}
    step["speedup_median"] = step["ms_per_step"]["float32"]["median"] / step["ms_per_step"]["mixed_bfloat16"]["median"]

    from torch.profiler import ProfilerActivity, profile
    kern = {}
    for p in pols:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            tr[p].step(x, y, lr)
            torch.cuda.synchronize()
        per = defaultdict(float)
        for ev in prof.events():
            if ev.device_type.name == "CUDA":
                per[ev.name] += ev.device_time / 1000.0          # us -> ms
        total = sum(per.values())
        cls = {c: sum(t for n, t in per.items() if re.search(pat, n)) for c, pat in CLASSES.items()}
        top = sorted(per.items(), key=lambda kv: -kv[1])[:25]
        kern[p] = {"kernel_ms_total": total, "class_ms": cls,
                   "class_share": {c: v / total for c, v in cls.items()},
                   "top_kernels_ms": {n: t for n, t in top}}
    kernels = {"what": "device kernel time of one profiled step per policy (torch.profiler, separate pass); "
                       "classes by kernel name: " + json.dumps(CLASSES), **info, "policies": kern}
    os.makedirs(a.out_dir, exist_ok=True)
    for name, obj in (("r07_train_mixed_step.json", step), ("r07_train_mixed_kernels.json", kernels)):
        with open(os.path.join(a.out_dir, name), "w") as f:
            json.dump(obj, f, indent=1)
    print(json.dumps({"ms_per_step": {p: step["ms_per_step"][p]["median"] for p in pols},
                      "class_ms": {p: kern[p]["class_ms"] for p in pols}, **info}))


if __name__ == "__main__":
    main()
