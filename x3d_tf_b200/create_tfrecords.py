"""Writes the reference's TFRecord datasets from decoded videos (the counterpart of the reference's
datasets/create_tfrecords.py), with the JPEG frames encoded on the GPU:

    python -m x3d_tf_b200.create_tfrecords --file_list videos.txt --out_dir DIR [--videos_per_file 32]
        [--quality 90] [--chroma 420|444] [--max_frames K] [--gzip_level 6] [--threads 16]

`--file_list` is the `<video.npy> <label>` list `eval.py` / `train.py --decoded_videos` read (decoded
[F, H, W, 3] uint8 videos, memory-mapped).  Each video becomes one SequenceExample (context
`video/num_frames`, `video/class/label`; feature list `video` of one JPEG per frame, what
tf.io.encode_jpeg(frame, quality) writes) in GZIP TFRecord files of `--videos_per_file` videos each,
in list order: DIR/shard-00000-of-0000N.tfrecord.gz, ...  `eval.py --tfrecord` and
`train.py --use_tfrecord` read them with `--test_file_pattern` / the train pattern 'DIR/*.tfrecord.gz'.
`--max_frames` keeps the first K frames of each video (the reference cuts its videos at 10 seconds;
decoded `.npy` videos carry no frame rate).

With `--mjpeg_videos` the list names Motion-JPEG `.avi` files instead (avi.py).  The frames of a
shard are decoded on the device (x3d_jpeg_*, IDCT by `--dct_method`, INTEGER_FAST by default as in
the other drivers) into the packed RGB buffer the decoder writes, and that buffer goes straight to the
encoder: a transcode from AVI to TFRecords never leaves the device between the two codecs.

The frames of a shard are encoded on the device in one batch and staged through pinned memory; the
records are serialised, compressed and written on a thread pool while the next shard is encoded.
At most 2 x `--threads` encoded shards wait for the pool (the oldest is awaited before the next one is
encoded), so host memory stays bounded when compression is slower than encoding.
"""
from __future__ import annotations

import argparse
import os
import time
from collections import deque
from concurrent.futures import ThreadPoolExecutor
from typing import List, Optional

from . import jpeg as J
from . import tfrecord as R
from .eval import read_file_list
from .video import load_video


def shard_name(out_dir: str, i: int, n: int) -> str:
    return os.path.join(out_dir, f"shard-{i:05d}-of-{n:05d}.tfrecord.gz")


def _write(path: str, jpegs: List[List[bytes]], labels: List[int], level: int):
    t0 = time.perf_counter()
    recs = [R.serialize_sequence_example(j, lab) for j, lab in zip(jpegs, labels)]
    t1 = time.perf_counter()
    raw = R.write_records(path, recs, level)
    return t1 - t0, time.perf_counter() - t1, raw


def _decode_mjpeg(part, max_frames: int, dct_method: str, scratch: dict):
    """(frames per video, [H, W, 3] uint8 device views of every frame in order) of the Motion-JPEG
    videos `part`, decoded on the current device in one batch."""
    import torch
    from . import avi, video
    vids = avi.open_videos(part)
    counts = [min(len(v), max_frames) if max_frames > 0 else len(v) for v in vids]
    pairs = [(i, f) for i, n in enumerate(counts) for f in range(n)]
    enc, out_off = video.encoded_frames(vids, pairs, dct_method=dct_method)
    dec = scratch.setdefault("decode", {})
    out, status = enc.decode(torch.device("cuda", torch.cuda.current_device()), dec)
    enc.check(status.cpu().numpy())
    frames = []
    for (i, _), o in zip(pairs, out_off):
        _, H, W, _ = vids[i].shape
        frames.append(out[int(o):int(o) + H * W * 3].view(H, W, 3))
    return counts, frames


def run(argv: Optional[List[str]] = None) -> dict:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--file_list", required=True, help="text file: '<video.npy> <label>' per video")
    ap.add_argument("--out_dir", required=True)
    ap.add_argument("--videos_per_file", type=int, default=32)
    ap.add_argument("--quality", type=int, default=90)
    ap.add_argument("--chroma", default="420", choices=sorted(J.CHROMA))
    ap.add_argument("--max_frames", type=int, default=0, help="keep the first K frames of each video (0: all)")
    ap.add_argument("--gzip_level", type=int, default=6)
    ap.add_argument("--threads", type=int, default=min(16, os.cpu_count() or 1))
    ap.add_argument("--mjpeg_videos", action="store_true", help="list lines name Motion-JPEG .avi videos")
    ap.add_argument("--dct_method", default="INTEGER_FAST", choices=["INTEGER_FAST", "INTEGER_ACCURATE"],
                    help="IDCT of the JPEG decoder for --mjpeg_videos (tf.io.decode_jpeg's names)")
    a = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("create_tfrecords encodes on a CUDA device and none is available")
    if a.videos_per_file < 1 or a.threads < 1 or not 0 <= a.gzip_level <= 9:
        raise SystemExit("--videos_per_file and --threads must be >= 1, --gzip_level 0..9")
    items = read_file_list(a.file_list)
    if not items:
        raise SystemExit(f"{a.file_list}: no videos")
    os.makedirs(a.out_dir, exist_ok=True)
    nshards = -(-len(items) // a.videos_per_file)
    scratch: dict = {}
    t0 = time.perf_counter()
    encode_s = 0.0
    frames = jpeg_bytes = 0
    max_pending = 2 * a.threads               # shards encoded and waiting for (or in) the pool
    pending: deque = deque()
    done = []
    with ThreadPoolExecutor(a.threads) as pool:
        for s in range(nshards):
            while len(pending) >= max_pending:
                done.append(pending.popleft().result())
            part = items[s * a.videos_per_file:(s + 1) * a.videos_per_file]
            t1 = time.perf_counter()
            if a.mjpeg_videos:
                counts, frame_list = _decode_mjpeg(part, a.max_frames, a.dct_method, scratch)
            else:
                videos = [load_video(p) for p, _ in part]
                if a.max_frames > 0:
                    videos = [v[:a.max_frames] for v in videos]
                counts, frame_list = [len(v) for v in videos], [f for v in videos for f in v]
            flat = J.encode_frames(frame_list, a.quality, a.chroma, scratch)
            encode_s += time.perf_counter() - t1
            jpegs, k = [], 0
            for n in counts:
                jpegs.append(flat[k:k + n])
                k += n
            frames += len(flat)
            jpeg_bytes += sum(len(b) for b in flat)
            pending.append(pool.submit(_write, shard_name(a.out_dir, s, nshards), jpegs, [lab for _, lab in part],
                                       a.gzip_level))
        while pending:
            done.append(pending.popleft().result())
    wall = time.perf_counter() - t0
    out = {"videos": len(items), "frames": frames, "files": nshards, "jpeg_bytes": jpeg_bytes,
           "wall_s": wall, "encode_s": encode_s, "serialize_s": sum(d[0] for d in done),
           "gzip_write_s": sum(d[1] for d in done), "videos_per_s": len(items) / wall}
    print(out)
    return out


if __name__ == "__main__":
    run()
