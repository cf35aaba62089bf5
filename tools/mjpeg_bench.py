"""Measures the Motion-JPEG AVI input path (avi.py, jpeg.parse(mjpeg=True), x3d_jpeg_entropy_rst).

    python tools/mjpeg_bench.py [--out profiles] [--quick]

Synthetic, seeded, video-like 360x480 frames encoded by Pillow at q90 4:2:0 (tools/jpeg_bench.py's
frame pool), with one restart interval per MCU row as ffmpeg's sliced MJPEG encoder writes them, or
without one.  Writes <out>/r06_mjpeg_{entropy,host,eval_e2e}.json, each with the card name, power
limit and maximum SM clock read in the same run:
  entropy   kernel time (CUDA events around >= 20 launches after a warm-up) of the entropy stage per
            X3D-M eval batch of 12 videos x 10 views (600 distinct frames): x3d_jpeg_entropy_rst on the
            restart-interval frames against x3d_jpeg_entropy on the same frames without restart
            intervals; per one-video batch (50 frames) too
  host      host time per 12-video X3D-M eval batch from 300-frame AVI files on disk: walking the
            chunks (cache cleared), reading the sampled frames and pack_jpeg, one thread; with shared
            Huffman tables (Pillow's standard tables) and with per-frame tables (Pillow optimize=True,
            every header made distinct by a COM segment, so the header cache never hits)
  eval_e2e  X3D.evaluate clips/s, X3D-M bf16 16x256^2 10 views, 12 videos per step: from AVI files
            read and packed in the loop (the eval driver's path), and from batches packed ahead
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import jpeg_bench as JB                                        # noqa: E402
from avi_writer import write_avi                               # noqa: E402
from x3d_tf_b200 import avi, ops, video as V                  # noqa: E402
from x3d_tf_b200 import jpeg as J                             # noqa: E402
from x3d_tf_b200.arch import build_arch                       # noqa: E402
from x3d_tf_b200.synth import synthetic_weights               # noqa: E402


def write(out_dir, name, rec):
    rec = dict(JB.card(), **rec)
    with open(os.path.join(out_dir, f"r06_mjpeg_{name}.json"), "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec))


def pool(n, H, W, seed, **kw):
    """n encoded frames (jpeg_bench's content) with Pillow options `kw`."""
    import io
    from PIL import Image
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:H, 0:W].astype(np.float32)
    ph = rng.uniform(0, 6.28, 3)
    out = []
    for f in range(n):
        t = f / 10.0
        img = np.stack([128 + 100 * np.sin(x / (17 + 5 * c) + y / (23 + 3 * c) + t + ph[c]) for c in range(3)], -1)
        y0, x0 = int(H / 3 * (1 + np.sin(t))), int(W / 3 * (1 + np.cos(t)))
        img[y0:y0 + H // 4, x0:x0 + W // 4] = rng.uniform(0, 255, 3)
        img += rng.normal(0, 8.0, img.shape)
        b = io.BytesIO()
        Image.fromarray(np.clip(img, 0, 255).astype(np.uint8)).save(b, "JPEG", quality=90, subsampling=2, **kw)
        out.append(b.getvalue())
    return out


class PoolVideo(JB.PoolVideo):
    mjpeg = True


def entropy_times(vb, reps):
    enc = vb.encoded
    scratch = {}
    _, status = enc.decode(torch.device("cuda"), scratch)
    torch.cuda.synchronize()
    enc.check(status.cpu().numpy())
    d, fr, tb, coef = scratch["jpeg_data"], scratch["jpeg_frames"], scratch["jpeg_tables"], scratch["jpeg_coef"]
    if enc.nintervals:
        iv = scratch["jpeg_intervals"]
        fn = lambda: ops.jpeg_entropy_rst(d, fr, tb, iv, enc.nintervals, coef, status, 0, enc.nframes)  # noqa: E731
    else:
        fn = lambda: ops.jpeg_entropy(d, fr, tb, enc.nframes, coef, status)                          # noqa: E731
    for _ in range(3):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    assert not status.any()
    return {"entropy_ms": e0.elapsed_time(e1) / reps, "frames": enc.nframes, "intervals": enc.nintervals,
            "entropy_coded_bytes": int(enc.data.numel())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--quick", action="store_true", help="fewer steps (a rehearsal, not a measurement)")
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    if not torch.cuda.is_available():
        raise SystemExit("mjpeg_bench needs a CUDA device")
    torch.cuda.set_device(0)
    reps = 5 if a.quick else 20
    H, W, F = 360, 480, 300
    n = 24 if a.quick else 120
    cfg = JB.eval_cfg()
    plain, rows = pool(n, H, W, 1), pool(n, H, W, 1, restart_marker_rows=1)

    # ---- entropy stage: one restart interval per MCU row against none, same frames
    res = {}
    for name, p in (("no_restart_x3d_jpeg_entropy", plain), ("restart_per_row_x3d_jpeg_entropy_rst", rows)):
        vids = [PoolVideo(p, F, k, H, W) for k in range(12)]
        res[name] = {"eval_batch_12_videos": entropy_times(V.eval_batch(vids, cfg, "INTEGER_FAST"), reps),
                     "one_video": entropy_times(V.eval_batch(vids[:1], cfg, "INTEGER_FAST"), reps)}
    write(a.out, "entropy", {
        "what": "entropy-stage kernel time per batch (CUDA events, mean of launches after warm-up), X3D-M eval "
                "10 views T=16, synthetic q90 4:2:0 360x480 frames, with one restart interval per MCU row "
                "(23 per frame) or none", **res})

    # ---- host: AVI walk + read + pack, shared and per-frame Huffman tables
    host = {}
    with tempfile.TemporaryDirectory() as tmp:
        kinds = {"shared_tables": rows,
                 "per_frame_tables": pool(n, H, W, 2, restart_marker_rows=1, optimize=True)}
        files = {}
        for kind, p in kinds.items():
            files[kind] = []
            for k in range(12):
                frames = [p[(7 * k + f) % len(p)] for f in range(F)]
                if kind == "per_frame_tables":                       # a distinct header per frame
                    frames = [fr[:2] + J._segment(0xFE, b"frame %d %d" % (k, f)) + fr[2:]
                              for f, fr in enumerate(frames)]
                path = os.path.join(tmp, f"{kind}_{k}.avi")
                write_avi(path, frames, W, H, audio=True)
                files[kind].append((path, k))
        for kind, items in files.items():
            size = sum(os.path.getsize(p) for p, _ in items)
            avi._tables.clear()
            J._mjpeg_cache.clear()
            t0 = time.perf_counter()
            vids = avi.open_videos(items)
            t1 = time.perf_counter()
            vb = V.eval_batch(vids, cfg, "INTEGER_FAST")
            t2 = time.perf_counter()
            host[kind] = {"file_bytes": size, "entropy_coded_bytes_packed": int(vb.encoded.data.numel()),
                          "distinct_frames": vb.encoded.nframes, "walk_ms": (t1 - t0) * 1e3,
                          "read_and_pack_ms": (t2 - t1) * 1e3, "host_ms_per_batch": (t2 - t0) * 1e3}
    write(a.out, "host", {"what": "host time per 12-video X3D-M eval batch from 300-frame MJPEG AVI files "
                                  "(one restart interval per MCU row): chunk walk (cache cleared), reading the "
                                  "sampled frames and pack_jpeg, one thread", **host})

    # ---- evaluate end to end from AVI files
    from x3d_tf_b200 import model as M
    from x3d_tf_b200.eval import mjpeg_batches
    with tempfile.TemporaryDirectory() as tmp:
        items = []
        for k in range(12):
            path = os.path.join(tmp, f"v{k}.avi")
            write_avi(path, [rows[(7 * k + f) % len(rows)] for f in range(F)], W, H)
            items.append((path, k))
        M.reset_block_counters()
        m = M.X3D(cfg, dtype="bfloat16").compile()
        m.set_weights_dict(synthetic_weights(build_arch(cfg)))
        steps = 4 if a.quick else 20
        labels = np.arange(12, dtype=np.int32)
        ahead = [(V.eval_batch(avi.open_videos(items), cfg, "INTEGER_FAST"), labels)]

        def run(kind, nsteps):
            data = (mjpeg_batches(items * nsteps, 12, cfg) if kind == "from_files"
                    else [ahead[0]] * nsteps)
            torch.cuda.synchronize()
            t = time.perf_counter()
            m.evaluate(data)
            torch.cuda.synchronize()
            return time.perf_counter() - t
        out = {"from_files": [], "packed_ahead": []}
        for k in out:
            run(k, 2)
        for _ in range(2):
            for k in out:
                out[k].append(10 * 12 * steps / run(k, steps))
    write(a.out, "eval_e2e", {
        "what": "X3D.evaluate clips/s, X3D-M bf16 16x256^2, 10 views, 12 videos per step, IFAST; host clock "
                "around evaluate (ends in a device synchronise); from_files reads and packs each batch from "
                "the AVI files in the loop (chunk tables cached after the first pass, files in the page "
                "cache), packed_ahead reuses one prepared batch; two alternating rounds",
        "steps_per_round": steps, **{f"{k}_clips_per_s": v for k, v in out.items()}})


if __name__ == "__main__":
    main()
