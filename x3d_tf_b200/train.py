"""Training driver: the caller of the training step, reference `train.py:37-155` + `utils.py:110-142`.

    python -m x3d_tf_b200.train --config X3D_M --train_file_pattern train.txt --model_dir out/ [--val_file_pattern val.txt]
    torchrun --nnodes=1 --nproc-per-node N -m x3d_tf_b200.train ... --num_gpus N          # one rank per GPU

Same flags and flow as the reference: build the config, create the model / SGD-Nesterov optimizer
(`train.py:85-92`), resume from the newest `ckpt-{epoch}` of `--model_dir` (epoch parsed from the
file name, `train.py:131-136`) or start from `--pretrained_ckpt`, then for every epoch set the
learning rate from the schedule of `train.py:114-125` (Keras `LearningRateScheduler`: once per
epoch), run `DATASET_SIZE // BATCH_SIZE` steps, evaluate `--val_file_pattern` (Keras `fit`'s
validation pass) and write `ckpt-{epoch}` with the optimizer slots (`ModelCheckpoint`,
`utils.py:128-132`).  The global batch `TRAIN.BATCH_SIZE` is split over the ranks as
MirroredStrategy does (`utils.py:160-167`); gradients are summed by one NCCL all-reduce per step
(`training.py`), BN moving statistics are averaged over ranks when a checkpoint is written.

Out of scope here as in eval.py's driver: video decoding and augmentation (`dataloader.py`,
`transforms.py`).  File lists name `.npy` arrays of already decoded and cropped uint8 clips
`[T, H, W, 3]` (or `[k, T, H, W, 3]`: k training clips of one video) with an integer label, or,
with `--decoded_videos`, decoded videos `[F, H, W, 3]` uint8 of any size: then every global-batch
slot draws one random clip of its video (temporal start, short-side scale jitter, crop, flip;
`video.train_plan`) and the resize / crop / flip run on the device (x3d_video_clips_u8); or, with
`--use_tfrecord` (the reference's flag), globs of the reference's GZIP TFRecord files: the file list
is shuffled per epoch with the epoch seed (the same on every rank), rank r reads files r::world,
records stream through a shuffle buffer of 16 x the per-rank batch (dataloader.py:158-159) and
repeat as needed, and the sampled JPEG frames are decoded on the device (x3d_jpeg_*); or, with
`--mjpeg_videos`, lists of Motion-JPEG `.avi` files (the reference's default `<video> <label>` lists,
`avi.py`), drawn as with `--decoded_videos`, whose sampled JPEG frames are read and decoded on the
device;
`--synthetic N` trains on N seeded random clips per epoch instead.  W&B / TensorBoard callbacks are
not reproduced; the per-epoch log line carries the same quantities Keras prints.
"""
from __future__ import annotations

import argparse
import os
import sys
import time
from typing import Iterator, List, Optional, Tuple

import numpy as np
import torch

from .config import get_config, get_default_config
from .eval import read_file_list
from .tf_bundle import latest_checkpoint


def lr_for_epoch(cfg, epoch: int) -> float:
    from .training import lr_schedule
    return lr_schedule(cfg, epoch)


def epoch_of_checkpoint(path: str) -> int:
    """`int(os.path.basename(ckpt_path).split('-')[1])`, train.py:133."""
    return int(os.path.basename(path).split("-")[1])


def global_batch_indices(n_items: int, gbatch: int, steps: int, seed: int) -> Iterator[np.ndarray]:
    """Exactly `steps` global batches of `gbatch` item indices, identical on every rank (the seed
    holds no rank): the list is reshuffled and repeated when it is shorter than `steps * gbatch`,
    as Keras `fit(steps_per_epoch=...)` does on a repeating dataset.  Every rank therefore runs
    the same number of steps whatever the list length -- the per-step gradient all-reduce of one
    rank can never pair with another rank's end-of-epoch reduction."""
    if n_items <= 0:
        raise ValueError("empty training list")
    rng = np.random.default_rng(seed)
    pool = np.empty(0, np.int64)
    for _ in range(steps):
        while pool.size < gbatch:
            pool = np.concatenate([pool, rng.permutation(n_items)])
        yield pool[:gbatch]
        pool = pool[gbatch:]


def file_clip_batches(items: List[Tuple[str, int]], gbatch: int, steps: int, seed: int, rank: int = 0,
                      world: int = 1) -> Iterator[Tuple[np.ndarray, np.ndarray]]:
    """This rank's slice of every global batch (one clip per listed file; a `[k,...]` file
    contributes a random one of its k clips)."""
    batch = gbatch // world
    pick = np.random.default_rng(seed + 104729 * (rank + 1))
    for idx in global_batch_indices(len(items), gbatch, steps, seed):
        clips, labels = [], []
        for j in idx[rank * batch:(rank + 1) * batch]:
            a = np.load(items[j][0])
            if a.ndim == 5:
                a = a[pick.integers(a.shape[0])]
            clips.append(a)
            labels.append(items[j][1])
        yield np.stack(clips), np.asarray(labels, np.int32)


def video_clip_batches(items: List[Tuple[str, int]], gbatch: int, steps: int, seed: int, cfg, rank: int = 0,
                       world: int = 1, crop_size: int = 0, mjpeg: bool = False, dct_method: str = "INTEGER_FAST"):
    """This rank's slice of every global batch as a video.VideoBatch: one random clip per listed
    decoded video (`mjpeg`: Motion-JPEG AVI video), the random numbers from video.train_rng(seed,
    rank) (per epoch and rank)."""
    from . import avi, video
    batch = gbatch // world
    rng = video.train_rng(seed, rank)
    for idx in global_batch_indices(len(items), gbatch, steps, seed):
        mine = idx[rank * batch:(rank + 1) * batch]
        vids = (avi.open_videos([items[j] for j in mine]) if mjpeg
                else [video.load_video(items[j][0]) for j in mine])
        vb = video.train_batch(vids, cfg, rng, crop_size, dct_method)
        yield vb, np.asarray([items[j][1] for j in mine], np.int32)


def tfrecord_rank_files(files: List[str], seed: int, rank: int = 0, world: int = 1) -> List[str]:
    """This rank's files of an epoch: the list shuffled with the epoch seed (identically on every
    rank), then every world-th file from position `rank`."""
    if len(files) < world:
        raise ValueError(f"{len(files)} TFRecord files for {world} ranks: every rank needs at least one")
    order = np.random.default_rng(seed).permutation(len(files))
    return [files[i] for i in order[rank::world]]


def tfrecord_clip_batches(files: List[str], gbatch: int, steps: int, seed: int, cfg, rank: int = 0,
                          world: int = 1, crop_size: int = 0, dct_method: str = "INTEGER_FAST"):
    """Exactly `steps` batches of this rank's share of the global batch as video.VideoBatch of JPEG
    frames: the records of tfrecord_rank_files(...) in file order, repeated as needed, through a
    shuffle buffer of 16 x the per-rank batch; one random clip per video, the clip draws from
    video.train_rng(seed, rank).  The buffer holds whole parsed records (every JPEG frame of each
    video, a few MB per 300-frame record), so its host memory grows with the batch: about 16 x batch
    x the record size, as with tf.data's shuffle buffer in the reference."""
    from . import tfrecord, video
    batch = gbatch // world
    mine = tfrecord_rank_files(files, seed, rank, world)
    rng = video.train_rng(seed, rank)
    pick = np.random.default_rng((int(seed), int(rank), 1))           # the shuffle buffer's draws

    def records():
        while True:
            n = 0
            for path in mine:
                for v in tfrecord.read_videos(path):
                    n += 1
                    yield v
            if n == 0:
                raise ValueError(f"rank {rank}: its TFRecord files hold no records")

    src, pool = records(), []
    for _ in range(steps):
        chosen = []
        while len(chosen) < batch:
            while len(pool) < 16 * batch:
                pool.append(next(src))
            j = int(pick.integers(0, len(pool)))
            chosen.append(pool[j])
            pool[j] = pool[-1]
            pool.pop()
        yield (video.train_batch(chosen, cfg, rng, crop_size, dct_method),
               np.asarray([v.label for v in chosen], np.int32))


def synthetic_clip_batches(steps: int, batch: int, T: int, S: int, num_classes: int, seed: int
                           ) -> Iterator[Tuple[np.ndarray, np.ndarray]]:
    rng = np.random.default_rng(seed)
    for _ in range(steps):
        yield (rng.integers(0, 256, size=(batch, T, S, S, 3), dtype=np.uint8),
               rng.integers(0, num_classes, size=batch).astype(np.int32))


def build_parser() -> argparse.ArgumentParser:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--config", required=True, help="config .yaml (reference layout) or a variant name")
    ap.add_argument("--train_file_pattern", default=None)
    ap.add_argument("--val_file_pattern", default=None)
    ap.add_argument("--decoded_videos", action="store_true",
                    help="list lines name decoded videos [F,H,W,3] uint8 (.npy, any size): clips are built on the device")
    ap.add_argument("--use_tfrecord", action="store_true",
                    help="the file patterns are globs of GZIP TFRecord files (JPEG frames, decoded on the device)")
    ap.add_argument("--mjpeg_videos", action="store_true",
                    help="list lines name Motion-JPEG .avi videos (JPEG frames decoded on the device)")
    ap.add_argument("--dct_method", default="INTEGER_FAST", choices=["INTEGER_FAST", "INTEGER_ACCURATE"],
                    help="IDCT of the JPEG decoder (tf.io.decode_jpeg's names; INTEGER_FAST is its default)")
    ap.add_argument("--model_dir", required=True)
    ap.add_argument("--pretrained_ckpt", default=None)
    ap.add_argument("--num_gpus", type=int, default=1)
    ap.add_argument("--synthetic", type=int, default=0, help="train on this many seeded random clips per epoch")
    ap.add_argument("--epochs", type=int, default=0, help="override cfg.TRAIN.EPOCHS (smoke runs)")
    ap.add_argument("--steps_per_epoch", type=int, default=0, help="override DATASET_SIZE // BATCH_SIZE")
    ap.add_argument("--batch_size", type=int, default=0, help="override cfg.TRAIN.BATCH_SIZE (global batch)")
    ap.add_argument("--crop_size", type=int, default=0, help="override cfg.DATA.TRAIN_CROP_SIZE (synthetic data)")
    ap.add_argument("--mixed_precision", action="store_true",
                    help="train.py:26,72-74,99-100: the 'mixed_bfloat16' policy -- every 1x1x1 conv and Dense "
                         "layer multiplies bf16 operands with fp32 accumulation (BatchNorm, softmax, the master "
                         "weights and the optimizer stay fp32); validation runs the bf16 inference engine")
    return ap


def run(argv: Optional[List[str]] = None) -> Optional[dict]:
    ap = build_parser()
    a = ap.parse_args(argv)
    if not a.train_file_pattern and not a.synthetic:
        ap.error("one of --train_file_pattern / --synthetic is required")
    if a.use_tfrecord + a.decoded_videos + a.mjpeg_videos > 1:
        ap.error("--use_tfrecord, --decoded_videos and --mjpeg_videos are mutually exclusive")
    if a.config.endswith(".yaml"):
        cfg = get_default_config(); cfg.merge_from_file(a.config); cfg.freeze()
    else:
        cfg = get_config(a.config)
    if cfg.TRAIN.OPTIMIZER.lower() not in ("sgd", "adam"):
        raise NotImplementedError(f"{cfg.TRAIN.OPTIMIZER} not supported")          # train.py:96-97
    os.makedirs(a.model_dir, exist_ok=True)

    import torch.distributed as dist
    world, rank = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0"))
    if world != max(a.num_gpus, 1):
        raise SystemExit(f"--num_gpus {a.num_gpus} needs {a.num_gpus} ranks (torchrun); WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise RuntimeError("no CUDA device: the X3D path has no CPU implementation")
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=dev)

    from . import ops
    from .arch import build_arch
    from .model import X3D, keras_default_weights, reset_block_counters
    from .training import X3DTrainer
    from .eval import file_batches, mjpeg_batches, tfrecord_batches, tfrecord_files, video_batches
    from .video import VideoBatch

    from .runtime import get_precision, policy_dtype
    precision = get_precision(a.mixed_precision)
    tr = X3DTrainer(cfg, device=dev, world=world, rank=rank, precision=precision)
    # a from-scratch run starts where `X3D(cfg)` starts in the reference (train.py:128): Keras default
    # initialisers -- Glorot-uniform kernels, zero biases, BN gamma=1 / beta=0 / mean=0 / variance=1
    tr.load(keras_default_weights(cfg, seed=1111))
    current_epoch = 0
    ckpt = latest_checkpoint(a.model_dir)
    if ckpt:
        current_epoch = epoch_of_checkpoint(ckpt)
        print(f"Found checkpoint {ckpt} at epoch {current_epoch}", file=sys.stderr)
        tr.load_checkpoint(ckpt)
    elif a.pretrained_ckpt:
        src = latest_checkpoint(a.pretrained_ckpt) if os.path.isdir(a.pretrained_ckpt) else a.pretrained_ckpt
        print(f"Loading model from pretrained weights at {src}", file=sys.stderr)
        tr.load_checkpoint(src)
        tr.iteration = 0

    gbatch = a.batch_size or cfg.TRAIN.BATCH_SIZE
    if gbatch % world:
        raise SystemExit(f"global batch {gbatch} is not divisible by {world} ranks")
    batch = gbatch // world
    epochs = a.epochs or cfg.TRAIN.EPOCHS
    steps = a.steps_per_epoch or max(cfg.TRAIN.DATASET_SIZE // gbatch, 1)
    T, S = cfg.DATA.TEMP_DURATION, a.crop_size or cfg.DATA.TRAIN_CROP_SIZE
    read_list = tfrecord_files if a.use_tfrecord else read_file_list
    items = read_list(a.train_file_pattern) if a.train_file_pattern else None
    if a.synthetic:
        steps = min(steps, max(a.synthetic // gbatch, 1))
    val_items = read_list(a.val_file_pattern) if a.val_file_pattern else None
    mean, std = tuple(cfg.DATA.MEAN), tuple(cfg.DATA.STD)
    history = []
    for epoch in range(current_epoch, epochs):
        lr = lr_for_epoch(cfg, epoch)
        if rank == 0:
            print(f"\nEpoch {epoch + 1}/{epochs}\nEpoch {epoch + 1:05d}: LearningRateScheduler setting learning rate to {lr}.")
        # every rank runs exactly `steps` steps (rank-independent count; short lists repeat)
        if items is not None and a.use_tfrecord:
            data = tfrecord_clip_batches(items, gbatch, steps, 1111 + 7919 * epoch, cfg, rank, world, a.crop_size,
                                         a.dct_method)
        elif items is not None and (a.decoded_videos or a.mjpeg_videos):
            data = video_clip_batches(items, gbatch, steps, 1111 + 7919 * epoch, cfg, rank, world, a.crop_size,
                                      a.mjpeg_videos, a.dct_method)
        else:
            data = (file_clip_batches(items, gbatch, steps, 1111 + 7919 * epoch, rank, world) if items is not None
                    else synthetic_clip_batches(steps, batch, T, S, cfg.NETWORK.NUM_CLASSES,
                                                1111 + 7919 * epoch + rank))
        t0, n, loss_sum = time.time(), 0, torch.zeros((), dtype=torch.float64, device=dev)
        for clips, labels in data:
            x = clips.clips(dev) if isinstance(clips, VideoBatch) else torch.from_numpy(clips).to(dev, non_blocking=True)
            if x.dtype == torch.uint8:
                x = ops.normalize_u8(x, mean, std, torch.float32)           # utils.normalize on the device
            loss = tr.step(x.float(), torch.from_numpy(labels).to(dev), lr)
            loss_sum += loss.double().sum()
            n += 1
            if n >= steps:
                break
        stats = torch.stack([loss_sum, torch.tensor(float(n * batch), dtype=torch.float64, device=dev)])
        if world > 1:
            dist.all_reduce(stats)
            from .exchange import average_
            average_(tr.moving.values(), world)                              # SURVEY 8e: average at save time
        log = {"epoch": epoch + 1, "policy": precision, "lr": lr, "loss": float(stats[0] / max(float(stats[1]), 1.0)),
               "steps": n, "seconds": time.time() - t0}
        if val_items is not None:
            reset_block_counters()
            m = X3D(cfg, dtype=policy_dtype(precision)).compile()
            m.set_weights_dict(tr.weights())
            num_preds = cfg.TEST.NUM_TEMPORAL_VIEWS * cfg.TEST.NUM_SPATIAL_CROPS
            from .shard import shard_range
            lo, hi = shard_range(len(val_items), world, rank)
            vpb = max(cfg.TEST.BATCH_SIZE // num_preds, 1)
            if a.use_tfrecord:
                val = tfrecord_batches(val_items[lo:hi], vpb, cfg, a.dct_method)
            elif a.mjpeg_videos:
                val = mjpeg_batches(val_items[lo:hi], vpb, cfg, a.dct_method)
            elif a.decoded_videos:
                val = video_batches(val_items[lo:hi], vpb, cfg)
            else:
                val = file_batches(val_items[lo:hi], vpb, num_preds)
            res = m.evaluate(val)
            log.update(val_loss=res["loss"], val_acc=res["acc"], val_top_5_acc=res["top_5_acc"])
            del m
        if rank == 0:
            tr.save_checkpoint(os.path.join(a.model_dir, f"ckpt-{epoch + 1}"), lr)
            print(" - ".join(f"{k}: {v:.4f}" if isinstance(v, float) else f"{k}: {v}" for k, v in log.items()))
            print(f"Epoch {epoch + 1:05d}: saving model to {os.path.join(a.model_dir, f'ckpt-{epoch + 1}')}")
        history.append(log)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return {"history": history, "iteration": tr.iteration}


if __name__ == "__main__":
    run()
