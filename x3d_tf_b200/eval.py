"""Evaluation driver: the caller of the forward path, reference `eval.py:26-91`.

    python -m x3d_tf_b200.eval --cfg X3D_M --model_folder models/X3D-M --test_file_pattern list.txt [--gpus N]
    torchrun --nnodes=1 --nproc-per-node N -m x3d_tf_b200.eval ... --gpus N      # one rank per GPU

Same flags and flow as the reference: build the config, construct `X3D(cfg)`, `compile` it with
the loss / metrics of `eval.py:62-70`, find the newest checkpoint of `--model_folder` through its
`checkpoint` file (`tf.train.latest_checkpoint`), `load_weights(...).expect_partial()` (optimizer
slots in the bundle are ignored) and `evaluate` the test set.  Multi-GPU: videos are split in
contiguous blocks over the ranks (`shard.shard_range`; the reference's MirroredStrategy splits
every batch, `utils.py:160-167`), the four metric sums are all-reduced at the end.

Video decoding (`dataloader.py`, `transforms.py`) is outside this path.  `--test_file_pattern`
names a text file with one `<path> <label>` line per video as in the reference, where <path> is
a `.npy` file of already decoded and cropped uint8 clips `[num_preds, T, H, W, 3]` (normalised on
the device, `utils.py:42-72`) or float32 clips (already normalised).  With `--decoded_videos` the
lines name decoded videos `[F, H, W, 3]` uint8 of any frame count and size instead: the short-side
resize, temporal views and crops of `transforms.py` run on the device (`video.py`,
x3d_video_clips_u8), and only the frames the views sample are read and copied.  With `--tfrecord`
(the reference's flag) `--test_file_pattern` is a glob of the reference's GZIP TFRecord files
(`tfrecord.py`; taken in sorted order, ranks get contiguous blocks of files, records are read in
file order): the JPEG frames the views sample are decoded on the device (x3d_jpeg_*) and then go
through the same clip kernel.  `--dct_method` picks the IDCT as TF's decode_jpeg names it:
INTEGER_FAST (TF 2.4's default for dct_method='') or INTEGER_ACCURATE.  With `--mjpeg_videos` the
list lines name Motion-JPEG `.avi` files, the reference's default `<video> <label>` lists (`avi.py`):
the same plans and sharding as `--decoded_videos`, and only the JPEG frames the views sample are read
from the files and decoded on the device.  `--synthetic V` evaluates V
seeded random videos instead (no files needed).
"""
from __future__ import annotations

import argparse
import glob
import os
import sys
from typing import Iterator, List, Optional, Tuple

import numpy as np
import torch

from . import shard
from .config import get_config, get_default_config
from .tf_bundle import latest_checkpoint


def read_file_list(path: str) -> List[Tuple[str, int]]:
    """`<path> <label>` per line (`dataloader.py:60-75` reads the same layout)."""
    base = os.path.dirname(os.path.abspath(path))
    out = []
    with open(path) as f:
        for ln, line in enumerate(f, 1):
            line = line.strip()
            if not line or line.startswith("#"):
                continue
            parts = line.rsplit(None, 1)
            if len(parts) != 2:
                raise ValueError(f"{path}:{ln}: expected '<path> <label>'")
            p = parts[0] if os.path.isabs(parts[0]) else os.path.join(base, parts[0])
            out.append((p, int(parts[1])))
    return out


def file_batches(items: List[Tuple[str, int]], videos_per_batch: int, num_preds: int
                 ) -> Iterator[Tuple[np.ndarray, np.ndarray]]:
    for i in range(0, len(items), videos_per_batch):
        chunk = items[i:i + videos_per_batch]
        clips = []
        for path, _ in chunk:
            a = np.load(path)
            if a.ndim == 4:
                a = a[None]
            if a.ndim != 5 or a.shape[0] != num_preds:
                raise ValueError(f"{path}: expected [{num_preds}, T, H, W, C] clips, got {a.shape}")
            clips.append(a)
        yield np.concatenate(clips, 0), np.asarray([lab for _, lab in chunk], np.int32)


def video_batches(items: List[Tuple[str, int]], videos_per_batch: int, cfg):
    """Batches of decoded videos (`.npy` [F, H, W, 3] uint8, memory-mapped) as video.VideoBatch."""
    from . import video
    for i in range(0, len(items), videos_per_batch):
        chunk = items[i:i + videos_per_batch]
        yield (video.eval_batch([video.load_video(p) for p, _ in chunk], cfg),
               np.asarray([lab for _, lab in chunk], np.int32))


def mjpeg_batches(items: List[Tuple[str, int]], videos_per_batch: int, cfg, dct_method: str = "INTEGER_FAST"):
    """Batches of Motion-JPEG AVI videos as video.VideoBatch of JPEG frames."""
    from . import avi, video
    for i in range(0, len(items), videos_per_batch):
        chunk = items[i:i + videos_per_batch]
        yield (video.eval_batch(avi.open_videos(chunk), cfg, dct_method),
               np.asarray([lab for _, lab in chunk], np.int32))


def tfrecord_files(pattern: str) -> List[str]:
    """The GZIP TFRecord files a glob names, sorted."""
    files = sorted(glob.glob(pattern))
    if not files:
        raise FileNotFoundError(f"no TFRecord files match {pattern!r}")
    return files


def tfrecord_batches(files: List[str], videos_per_batch: int, cfg, dct_method: str = "INTEGER_FAST"):
    """Batches of the videos in `files` (read in file order) as video.VideoBatch of JPEG frames."""
    from . import tfrecord, video
    chunk = []
    for path in files:
        for v in tfrecord.read_videos(path):
            chunk.append(v)
            if len(chunk) == videos_per_batch:
                yield video.eval_batch(chunk, cfg, dct_method), np.asarray([c.label for c in chunk], np.int32)
                chunk = []
    if chunk:
        yield video.eval_batch(chunk, cfg, dct_method), np.asarray([c.label for c in chunk], np.int32)


def synthetic_batches(lo: int, hi: int, videos_per_batch: int, num_preds: int, T: int, S: int,
                      num_classes: int) -> Iterator[Tuple[np.ndarray, np.ndarray]]:
    """Seeded per VIDEO (not per rank), so any sharding evaluates the same set."""
    for i in range(lo, hi, videos_per_batch):
        ids = range(i, min(i + videos_per_batch, hi))
        clips = np.concatenate([np.random.default_rng(1111 + v).integers(
            0, 256, size=(num_preds, T, S, S, 3), dtype=np.uint8) for v in ids], 0)
        labels = np.asarray([(v * 7919) % num_classes for v in ids], np.int32)
        yield clips, labels


def load_cfg(name_or_path: str):
    if name_or_path.endswith(".yaml"):
        cfg = get_default_config()
        cfg.merge_from_file(name_or_path)
        cfg.freeze()
        return cfg
    return get_config(name_or_path)


def run(argv: Optional[List[str]] = None) -> Optional[dict]:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--cfg", required=True, help="config .yaml (reference layout) or a variant name, e.g. X3D_M")
    ap.add_argument("--test_file_pattern", default=None, help="text file: '<clips.npy> <label>' per video")
    ap.add_argument("--model_folder", required=True, help="directory with a TF `checkpoint` file")
    ap.add_argument("--decoded_videos", action="store_true",
                    help="list lines name decoded videos [F,H,W,3] uint8 (.npy, any size): clips are built on the device")
    ap.add_argument("--tfrecord", action="store_true",
                    help="--test_file_pattern is a glob of GZIP TFRecord files (JPEG frames, decoded on the device)")
    ap.add_argument("--mjpeg_videos", action="store_true",
                    help="list lines name Motion-JPEG .avi videos (JPEG frames decoded on the device)")
    ap.add_argument("--dct_method", default="INTEGER_FAST", choices=["INTEGER_FAST", "INTEGER_ACCURATE"],
                    help="IDCT of the JPEG decoder (tf.io.decode_jpeg's names; INTEGER_FAST is its default)")
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--synthetic", type=int, default=0, help="evaluate this many seeded random videos")
    ap.add_argument("--dtype", default=None, choices=["bfloat16", "float32"],
                    help="activation storage; default: the --mixed_precision policy")
    ap.add_argument("--mixed_precision", action="store_true", default=True,
                    help="utils.get_precision: 16-bit activations (bfloat16 here, see runtime.py); --no_mixed_precision for fp32")
    ap.add_argument("--no_mixed_precision", dest="mixed_precision", action="store_false")
    ap.add_argument("--allow_random_init", action="store_true",
                    help="run with freshly initialised weights when the folder has no checkpoint data")
    a = ap.parse_args(argv)
    if not a.test_file_pattern and not a.synthetic:
        ap.error("one of --test_file_pattern / --synthetic is required")
    if a.tfrecord + a.decoded_videos + a.mjpeg_videos > 1:
        ap.error("--tfrecord, --decoded_videos and --mjpeg_videos are mutually exclusive")
    cfg = load_cfg(a.cfg)
    if not os.path.isdir(a.model_folder):
        raise NotADirectoryError(a.model_folder)          # eval.py:36-37

    import torch.distributed as dist
    world, rank = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0"))
    if world != max(a.gpus, 1):
        raise SystemExit(f"--gpus {a.gpus} needs {a.gpus} ranks (torchrun --nproc-per-node {a.gpus}); WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise RuntimeError("no CUDA device: the X3D path has no CPU implementation")
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl")

    from .model import X3D, reset_block_counters
    reset_block_counters()
    from .runtime import get_precision, policy_dtype
    model = X3D(cfg, dtype=a.dtype or policy_dtype(get_precision(a.mixed_precision))).compile(top_k=5)
    ckpt = latest_checkpoint(a.model_folder)
    if ckpt:
        print(f"Found checkpoint {ckpt}", file=sys.stderr)
        try:
            model.load_weights(ckpt).expect_partial()
        except FileNotFoundError:
            if not a.allow_random_init:
                raise
            print("checkpoint data shards are missing: evaluating freshly initialised weights", file=sys.stderr)
    elif not a.allow_random_init:
        print("No checkpoint found!", file=sys.stderr)     # eval.py:90-91
        return None

    num_preds = cfg.TEST.NUM_TEMPORAL_VIEWS * cfg.TEST.NUM_SPATIAL_CROPS
    vpb = max(cfg.TEST.BATCH_SIZE // num_preds, 1)
    if a.synthetic:
        lo, hi = shard.shard_range(a.synthetic, world, rank)
        data = synthetic_batches(lo, hi, vpb, num_preds, cfg.DATA.TEMP_DURATION, cfg.DATA.TEST_CROP_SIZE,
                                 cfg.NETWORK.NUM_CLASSES)
    elif a.tfrecord:
        files = tfrecord_files(a.test_file_pattern)
        lo, hi = shard.shard_range(len(files), world, rank)
        data = tfrecord_batches(files[lo:hi], vpb, cfg, a.dct_method)
    else:
        items = read_file_list(a.test_file_pattern)
        lo, hi = shard.shard_range(len(items), world, rank)
        if a.mjpeg_videos:
            data = mjpeg_batches(items[lo:hi], vpb, cfg, a.dct_method)
        elif a.decoded_videos:
            data = video_batches(items[lo:hi], vpb, cfg)
        else:
            data = file_batches(items[lo:hi], vpb, num_preds)
    res = model.evaluate(data, verbose=1 if rank == 0 else 0)
    if rank == 0:
        print(f"\nloss: {res['loss']:.4f} - acc: {res['acc']:.4f} - top_5_acc: {res['top_5_acc']:.4f} "
              f"({res['videos']} videos, {world} GPU{'s' if world > 1 else ''})")
    if world > 1:
        dist.destroy_process_group()
    return res


if __name__ == "__main__":
    run()
