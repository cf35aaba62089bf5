"""Measures the device JPEG encoder (x3d_jpeg_fdct / _enc_bits / _enc_emit / _enc_stuff) and the TFRecord
writing driver (x3d_tf_b200.create_tfrecords).

    python tools/jpeg_encode_bench.py [--out profiles] [--quick]

Synthetic, seeded, video-like frames (tests/tfrecord_writer.video_frames), 360x480, q90 4:2:0.  Writes
<out>/r05_jpeg_encode_{stages,cpu_baseline,driver}.json, each with the card name and power limit read in
the same run:
  stages        kernel time of each encode stage (CUDA events around >= 20 launches after a warm-up) for
                one 600-frame batch already on the device, and encode_frames end to end from pinned host
                frames (H2D, four stages, the result read-back and the D2H of the segments)
  cpu_baseline  Pillow (libjpeg-turbo) encoding the same 600 frames on all host threads, frames/s
  driver        create_tfrecords on 48 videos of 150 frames (.npy, memory-mapped; each video is the first
                150 of the frames above in its own rotation), 32 videos per file (2 files) and 4 per file
                (12 files), gzip levels 6, 1 and 0: videos/s end to end, with the device encode time (on
                the main thread) and the serialise and gzip + write time summed over the thread pool
"""
from __future__ import annotations

import argparse
import io
import json
import os
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tests.tfrecord_writer import video_frames                 # noqa: E402
from tools.jpeg_bench import card                              # noqa: E402
from x3d_tf_b200 import jpeg as J                              # noqa: E402
from x3d_tf_b200 import ops                                    # noqa: E402


def write(out_dir, name, rec):
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, f"r05_jpeg_encode_{name}.json"), "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec))


def frames_600(quick):
    """600 distinct frames: 20 seeded videos of 30 frames."""
    n = 60 if quick else 600
    return np.concatenate([video_frames(30, 360, 480, 1000 + k) for k in range(n // 30)])


def stage_times(frames, reps):
    scratch = {}
    dev = torch.from_numpy(frames).cuda()
    J.encode_frames(dev, 90, "420", scratch)                    # sizes the buffers, warms up
    names = ["x3d_jpeg_fdct", "x3d_jpeg_enc_bits", "x3d_jpeg_enc_emit", "x3d_jpeg_enc_stuff"]
    acc = {k: [] for k in names}
    for _ in range(reps):
        ops.Profiler.start()
        J.encode_frames(dev, 90, "420", scratch)
        for _, name, ms in ops.Profiler.stop():
            acc[name].append(ms)
    host = torch.from_numpy(frames).pin_memory()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        out = J.encode_frames(host, 90, "420", scratch)
    e2e = (time.perf_counter() - t0) / reps
    return {k: float(np.median(v)) for k, v in acc.items()}, e2e, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--quick", action="store_true")
    a = ap.parse_args()
    info = card()
    frames = frames_600(a.quick)
    F = len(frames)
    ms, e2e, jpegs = stage_times(frames, 5 if a.quick else 20)
    write(a.out, "stages", dict(info, frames=F, H=360, W=480, quality=90, chroma="420",
                                stage_ms=ms, device_ms_total=sum(ms.values()),
                                device_frames_per_s=F / (sum(ms.values()) / 1e3),
                                encode_frames_e2e_ms=e2e * 1e3, encode_frames_e2e_frames_per_s=F / e2e,
                                jpeg_bytes_per_frame=float(np.mean([len(j) for j in jpegs])),
                                raw_bytes_per_frame=360 * 480 * 3))

    from PIL import Image

    def pil(img):
        b = io.BytesIO()
        Image.fromarray(img).save(b, "JPEG", quality=90, subsampling=2, dpi=(300, 300))
        return b.getvalue()

    threads = os.cpu_count() or 1
    with ThreadPoolExecutor(threads) as pool:
        list(pool.map(pil, frames[:threads]))
        t0 = time.perf_counter()
        ref = list(pool.map(pil, frames))
        dt = time.perf_counter() - t0
    write(a.out, "cpu_baseline", dict(info, frames=F, threads=threads, seconds=dt, frames_per_s=F / dt,
                                      identical_to_device=ref == jpegs))

    from x3d_tf_b200 import create_tfrecords as C
    nv, nf = (6, 30) if a.quick else (48, 150)
    pool_frames = np.concatenate([frames, frames[::-1]])[:nf]
    with tempfile.TemporaryDirectory() as tmp:
        lines = []
        for k in range(nv):
            np.save(os.path.join(tmp, f"v{k}.npy"), np.roll(pool_frames, 7 * k, axis=0))    # distinct order
            lines.append(f"v{k}.npy {k % 400}")
        with open(os.path.join(tmp, "list.txt"), "w") as f:
            f.write("\n".join(lines) + "\n")
        args = ["--file_list", os.path.join(tmp, "list.txt"), "--out_dir", os.path.join(tmp, "out"),
                "--threads", str(min(16, threads))]
        C.run(args + ["--out_dir", os.path.join(tmp, "warm"), "--max_frames", "2"])
        runs = []
        # one gzip stream per file: the files in flight bound how many threads compress
        for vpf, level in ((32, 6), (4, 6), (4, 6), (4, 1), (4, 0)):
            r = C.run(args + ["--videos_per_file", str(vpf), "--gzip_level", str(level)])
            runs.append(dict(r, videos_per_file=vpf, gzip_level=level))
    write(a.out, "driver", dict(info, videos=nv, frames_per_video=nf, H=360, W=480, quality=90, chroma="420",
                                runs=runs, threads=min(16, threads), host_cpus=threads))


if __name__ == "__main__":
    main()
