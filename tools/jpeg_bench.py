"""Measures the TFRecord / JPEG input path (tfrecord.py, jpeg.py, x3d_jpeg_* kernels, video.pack_jpeg).

    python tools/jpeg_bench.py [--out profiles] [--quick]

Synthetic, seeded, video-like frames (moving colour gradients, a moving hard-edged rectangle, noise),
360x480, encoded by Pillow at q90 4:2:0; videos of 300 frames (frame f of video k is one of a pool of
120 encoded frames, so the batch holds as many distinct frame copies as real videos would without
encoding 3600 frames).  Writes <out>/r04_jpeg_{stages,eval_e2e,host,cpu_baseline}.json, each with the
card name and power limit read in the same run:
  stages        JPEG bytes per frame; kernel time of each decode stage (CUDA events around >= 20
                launches after a warm-up) per X3D-M eval batch (12 videos, 10 views: 600 distinct frames)
                and per one-video batch (50 frames: the entropy stage's per-frame latency), for both IDCTs;
                H2D bytes per step of the TFRecord batch against the raw VideoBatch of the same frames
  eval_e2e      X3D.evaluate clips/s, X3D-M bf16 16x256^2 10 views, from TFRecord batches, raw
                VideoBatches and pre-cropped pinned uint8 clips, alternating in one run, at 12 videos per
                step and at cfg.TEST.BATCH_SIZE (one video per step); the batches are prepared ahead
  host          host time per 12-video batch: inflate + CRC + parse the records of a GZIP TFRecord
                file (read_videos) and pack_jpeg; compared with the device time per batch
  cpu_baseline  Pillow (libjpeg-turbo) decoding the same 600 frames on all host threads, frames/s
"""
from __future__ import annotations

import argparse
import gzip
import io
import json
import os
import struct
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from x3d_tf_b200 import ops, tfrecord, video as V             # noqa: E402
from x3d_tf_b200.arch import build_arch                       # noqa: E402
from x3d_tf_b200.config import get_config                     # noqa: E402
from x3d_tf_b200.synth import synthetic_weights               # noqa: E402
from x3d_tf_b200.tf_bundle import crc32c, mask_crc            # noqa: E402


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
    with open(os.path.join(out_dir, f"r04_jpeg_{name}.json"), "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec))


def frame_pool(n, H, W, seed):
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
        Image.fromarray(np.clip(img, 0, 255).astype(np.uint8)).save(b, "JPEG", quality=90, subsampling=2)
        out.append(b.getvalue())
    return out


class PoolVideo:
    """A video of F JPEG frames taken from a shared pool (frame f of video k = pool[(7k + f) % len])."""
    dtype = np.uint8

    def __init__(self, pool, F, k, H, W):
        self.pool, self.k, self.shape, self.name, self.label = pool, k, (F, H, W, 3), f"video {k}", k

    def jpeg(self, f):
        return self.pool[(7 * self.k + int(f)) % len(self.pool)]


def sequence_example(frames, label) -> bytes:
    """A minimal serialiser of the reference's SequenceExample (for the host-time measurement)."""
    def ld(field, payload):
        n, out = len(payload), bytearray([field << 3 | 2])
        while True:
            b = n & 0x7F
            n >>= 7
            out.append(b | (0x80 if n else 0))
            if not n:
                return bytes(out) + payload

    def varint(v):
        out = bytearray()
        while True:
            b = v & 0x7F
            v >>= 7
            out.append(b | (0x80 if v else 0))
            if not v:
                return bytes(out)

    def int_feature(v):
        return ld(3, ld(1, varint(v)))

    ctx = b"".join(ld(1, ld(1, k.encode()) + ld(2, int_feature(v)))
                   for k, v in (("video/num_frames", len(frames)), ("video/class/label", label)))
    fl = ld(1, ld(1, b"video") + ld(2, b"".join(ld(1, ld(1, ld(1, f))) for f in frames)))
    return ld(1, ctx) + ld(2, fl)


def stage_times(vb, reps):
    enc, dev = vb.encoded, torch.device("cuda")
    scratch = {}
    frames, status = enc.decode(dev, scratch)                  # warm-up, buffers
    torch.cuda.synchronize()
    enc.check(status.cpu().numpy())
    d, fr, tb = scratch["jpeg_data"], scratch["jpeg_frames"], scratch["jpeg_tables"]
    coef, planes = scratch["jpeg_coef"], scratch["jpeg_planes"]
    calls = {
        "entropy": lambda: ops.jpeg_entropy(d, fr, tb, enc.nframes, coef, status),
        "idct_islow": lambda: ops.jpeg_idct(coef, fr, tb, enc.nframes, enc.max_blocks, 0, planes),
        "idct_ifast": lambda: ops.jpeg_idct(coef, fr, tb, enc.nframes, enc.max_blocks, 1, planes),
        "color": lambda: ops.jpeg_color(planes, fr, enc.nframes, enc.max_pixels, frames),
    }
    out = {}
    for name, fn in calls.items():
        for _ in range(3):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        out[name + "_ms"] = e0.elapsed_time(e1) / reps
    out.update(frames=enc.nframes, coef_bytes=enc.coef_blocks * 128, plane_bytes=enc.plane_bytes,
               decoded_bytes=enc.out_bytes, entropy_coded_bytes=int(enc.data.numel()))
    return out


def eval_cfg(views=10, S=256, T=16):
    cfg = get_config("X3D_M", freeze=False)
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
        raise SystemExit("jpeg_bench needs a CUDA device")
    torch.cuda.set_device(0)
    reps = 5 if a.quick else 20
    H, W, F = 360, 480, 300
    pool = frame_pool(24 if a.quick else 120, H, W, 1)
    cfg = eval_cfg()
    vids = [PoolVideo(pool, F, k, H, W) for k in range(12)]

    # ---- stages and bytes
    jb = V.eval_batch(vids, cfg, "INTEGER_FAST")
    one = V.eval_batch(vids[:1], cfg, "INTEGER_FAST")
    frames_dev, _ = jb.encoded.decode("cuda", {})
    decoded0 = frames_dev[:H * W * 3].cpu().numpy().reshape(H, W, 3)       # frame 0 of the batch (out_off 0)
    plan = V.eval_plan([v.shape for v in vids], cfg.DATA.TEMP_DURATION, 10, 1, 256)

    class Raw:                                                # the decoded frames as a raw video
        def __init__(self, k):
            self.shape, self.dtype, self.k = (F, H, W, 3), np.uint8, k

        def __getitem__(self, f):
            return decoded0
    rb = V.pack([Raw(k) for k in range(12)], plan)
    write(a.out, "stages", {
        "what": "x3d_jpeg_* kernel time per batch (CUDA events), X3D-M eval 10 views T=16: 12 videos "
                "(distinct frames below) and one video; synthetic q90 4:2:0 360x480 frames",
        "jpeg_bytes_per_frame_mean": float(np.mean([len(p) for p in pool])),
        "raw_bytes_per_frame": H * W * 3,
        "h2d_bytes_per_step_tfrecord": int(jb.h2d_bytes), "h2d_bytes_per_step_raw_video_batch": int(rb.h2d_bytes),
        "eval_batch_12_videos": stage_times(jb, reps), "one_video": stage_times(one, reps)})

    # ---- host: inflate + parse + pack of a GZIP TFRecord file
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "videos.tfrecord.gz")
        with gzip.open(path, "wb", compresslevel=6) as f:
            for k, v in enumerate(vids):
                r = sequence_example([v.jpeg(i) for i in range(F)], k)
                head = struct.pack("<Q", len(r))
                f.write(head + struct.pack("<I", mask_crc(crc32c(head))) + r + struct.pack("<I", mask_crc(crc32c(r))))
        size = os.path.getsize(path)
        t0 = time.perf_counter()
        recs_read = list(tfrecord.read_videos(path))
        read_s = time.perf_counter() - t0
        t0 = time.perf_counter()
        V.eval_batch(recs_read, cfg, "INTEGER_FAST")
        pack_s = time.perf_counter() - t0
    write(a.out, "host", {
        "what": "host time per 12-video X3D-M eval batch (300-frame records): inflate + CRC + parse "
                "(tfrecord.read_videos) and pack_jpeg, one thread",
        "file_bytes": size, "read_parse_ms": read_s * 1e3, "pack_ms": pack_s * 1e3,
        "host_ms_per_batch": (read_s + pack_s) * 1e3})

    # ---- Pillow on all host threads
    from PIL import Image
    segs = [vids[int(k >> 32)].jpeg(int(k & 0xffffffff)) for k in
            np.unique((plan.video[:, None] * (1 << 32) + plan.frames).reshape(-1))]

    def dec(b):
        return np.asarray(Image.open(io.BytesIO(b)).convert("RGB"))
    threads = os.cpu_count() or 1
    with ThreadPoolExecutor(threads) as ex:
        list(ex.map(dec, segs[:threads]))
        t0 = time.perf_counter()
        list(ex.map(dec, segs))
        pil_s = time.perf_counter() - t0
    write(a.out, "cpu_baseline", {"what": "Pillow decode of the eval batch's distinct frames, all host threads",
                                  "threads": threads, "frames": len(segs), "frames_per_s": len(segs) / pil_s})

    # ---- evaluate end to end
    from x3d_tf_b200 import model as M
    res = {}
    for vpb in (12, max(cfg.TEST.BATCH_SIZE // 10, 1)):
        M.reset_block_counters()
        m = M.X3D(cfg, dtype="bfloat16").compile()
        m.set_weights_dict(synthetic_weights(build_arch(cfg)))
        groups = [vids[:vpb], vids[12 - vpb:]]
        labels = np.arange(vpb, dtype=np.int32)
        plans = [V.eval_plan([v.shape for v in g], cfg.DATA.TEMP_DURATION, 10, 1, 256) for g in groups]
        tf = [V.pack_jpeg(g, p) for g, p in zip(groups, plans)]
        raw = [V.pack([Raw(v.k) for v in g], p) for g, p in zip(groups, plans)]
        clips = [b.clips("cuda").cpu().pin_memory() for b in raw]
        steps = (4 if a.quick else 20) * (12 // vpb)
        src = {"tfrecord": tf, "raw_video_batch": raw, "u8_clips": clips}
        out = {k: [] for k in src}

        def run(kind, n):
            data = [(src[kind][i % 2], labels) for i in range(n)]
            torch.cuda.synchronize()
            t = time.perf_counter()
            m.evaluate(data)
            torch.cuda.synchronize()
            return time.perf_counter() - t
        for k in src:
            run(k, 3)
        for _ in range(2):
            for k in src:
                out[k].append(10 * vpb * steps / run(k, steps))
        res[f"{vpb}_videos_per_step"] = {f"{k}_clips_per_s": v for k, v in out.items()}
        res[f"{vpb}_videos_per_step"]["steps_per_round"] = steps
        del m, clips, tf, raw
        torch.cuda.empty_cache()
    write(a.out, "eval_e2e", {
        "what": "X3D.evaluate clips/s, X3D-M bf16 16x256^2, 10 views; host clock around evaluate (ends in a "
                "device synchronise); batches prepared ahead; two alternating rounds per input; IFAST", **res})


if __name__ == "__main__":
    main()
