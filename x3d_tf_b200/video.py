"""Clips from decoded videos, built on the device: the host-side rules of the reference's
`transforms.py` (temporal sampling, short-side resize extent, crop offsets, flip) and the packing of
the frames those rules select.  The per-pixel work (bilinear resize, crop, flip) is one launch of
`x3d_video_clips_u8` over a whole ragged batch of videos (`ops.video_clips_u8`).

Every rule lives in exactly one function here, so that a correction lands in one place:

  resized_extent   short side -> `size`, long side -> floor(long * size / short) (integer arithmetic)
  eval_plan        transforms.py:48-65, 149-222: frame ((view*T + t) * max(1, F // T)) mod F of the
                   video; the frame resized so that its short side is `size` (TEST_CROP_SIZE); centre
                   crop, or left / centre / right along the longer side (offsets ceil((dim - S) / 2),
                   0, dim - S); clips in [crop][view] order (dataloader.py:107-116); no flip
  train_plan       transforms.py:15-47, 112-147, 192-206, one clip per video, random numbers drawn
                   from the generator in this order per clip:
                     t0    ~ U{0 .. F-1}          frame i = (t0 + i * FRAME_RATE) mod F
                     short ~ U{jitter[0] .. jitter[1]}   (inclusive)
                     y0    ~ U{0 .. rh - S},  x0 ~ U{0 .. rw - S}
                   and flip = 1 always: the reference applies flip_left_right unconditionally
                   (transforms.py:205-206), which this follows
  train_rng        the generator of one epoch and rank: numpy default_rng((seed, rank))

The resize is TF 2.4's ResizeBilinear with half_pixel_centers (what `tf.image.resize(method=
"bilinear")` runs) followed by the cast back to uint8; include/x3d_b200.h states the arithmetic.
Parity of these rules with TensorFlow is unpinned (TensorFlow is not available to this project's
tests); they are restated from the reference's source.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

# x3d_clip_desc (include/x3d_b200.h): seven int32 fields
DESC_FIELDS = ("H", "W", "rh", "rw", "y0", "x0", "flip")


def resized_extent(H: int, W: int, size: int) -> Tuple[int, int]:
    """(rh, rw) of an H x W frame whose short side is resized to `size`."""
    if H <= 0 or W <= 0 or size <= 0:
        raise ValueError(f"resized_extent: bad sizes H={H} W={W} size={size}")
    if H <= W:
        return size, (W * size) // H
    return (H * size) // W, size


@dataclass
class ClipPlan:
    """Which frames every clip reads and how it resizes and crops them.
    video  [N] int64: index of the clip's source video in the list the plan was made for;
    frames [N, T] int64: frame index within that video of each output frame;
    desc   [N, 7] int32: x3d_clip_desc (H, W, rh, rw, y0, x0, flip) of each clip;
    S      output crop size."""
    video: np.ndarray
    frames: np.ndarray
    desc: np.ndarray
    S: int

    @property
    def shape(self) -> Tuple[int, int, int, int, int]:
        return (self.frames.shape[0], self.frames.shape[1], self.S, self.S, 3)


def _check_shape(shape) -> Tuple[int, int, int]:
    if len(shape) != 4 or shape[3] != 3:
        raise ValueError(f"a decoded video is [F, H, W, 3], got {tuple(shape)}")
    F, H, W = (int(v) for v in shape[:3])
    if F <= 0 or H <= 0 or W <= 0:
        raise ValueError(f"empty video of shape {tuple(shape)}")
    return F, H, W


def uniform_crop_offsets(rh: int, rw: int, S: int, spatial_idx: int) -> Tuple[int, int]:
    """transforms.py:149-190: centre offsets ceil((dim - S) / 2); index 0 / 2 moves the crop to the
    start / end of the longer side."""
    y0, x0 = (rh - S + 1) // 2, (rw - S + 1) // 2
    if rh > rw:
        y0 = {0: 0, 1: y0, 2: rh - S}[spatial_idx]
    else:
        x0 = {0: 0, 1: x0, 2: rw - S}[spatial_idx]
    return y0, x0


def eval_plan(shapes: Sequence[Sequence[int]], T: int, views: int, crops: int, size: int) -> ClipPlan:
    """crops * views clips per video (shapes: [F, H, W, 3] of each), resized to short side `size`
    and cropped to `size` x `size`."""
    if crops not in (1, 3) or views <= 0 or T <= 0:
        raise ValueError(f"eval_plan: T={T} views={views} crops={crops}")
    vid, frames, desc = [], [], []
    for v, shape in enumerate(shapes):
        F, H, W = _check_shape(shape)
        rh, rw = resized_extent(H, W, size)
        rate = max(1, F // T)
        idx = ((np.arange(views * T, dtype=np.int64) * rate) % F).reshape(views, T)
        for c in range(crops):
            y0, x0 = uniform_crop_offsets(rh, rw, size, c % 3 if crops > 1 else 1)
            for view in range(views):
                vid.append(v)
                frames.append(idx[view])
                desc.append((H, W, rh, rw, y0, x0, 0))
    return _plan(vid, frames, desc, size, T)


def train_rng(seed: int, rank: int = 0) -> np.random.Generator:
    return np.random.default_rng((int(seed), int(rank)))


def train_plan(shapes: Sequence[Sequence[int]], T: int, frame_rate: int, jitter: Sequence[int], S: int,
               rng: np.random.Generator) -> ClipPlan:
    """One random training clip per video (order of the draws: module docstring)."""
    lo, hi = int(jitter[0]), int(jitter[1])
    if lo > hi or lo <= 0:
        raise ValueError(f"train_plan: jitter scales {lo}..{hi}")
    if S > lo:
        raise ValueError(f"train_plan: crop {S} is larger than the smallest short side {lo}")
    vid, frames, desc = [], [], []
    for v, shape in enumerate(shapes):
        F, H, W = _check_shape(shape)
        t0 = int(rng.integers(0, F))
        short = int(rng.integers(lo, hi + 1))
        rh, rw = resized_extent(H, W, short)
        y0 = int(rng.integers(0, rh - S + 1))
        x0 = int(rng.integers(0, rw - S + 1))
        vid.append(v)
        frames.append((t0 + np.arange(T, dtype=np.int64) * frame_rate) % F)
        desc.append((H, W, rh, rw, y0, x0, 1))
    return _plan(vid, frames, desc, S, T)


def _plan(vid, frames, desc, S: int, T: int) -> ClipPlan:
    if not vid:
        raise ValueError("a clip plan needs at least one video")
    return ClipPlan(np.asarray(vid, np.int64), np.asarray(frames, np.int64).reshape(len(vid), T),
                    np.asarray(desc, np.int32).reshape(len(vid), 7), int(S))


def validate(plan: ClipPlan, shapes: Sequence[Sequence[int]]) -> None:
    """What x3d_video_clips_u8 takes as preconditions (its descriptors are device data and are
    not checked there): raises ValueError for a crop outside the resized frame, S larger than the
    resized short side, a frame index outside its video or a descriptor that disagrees with it."""
    S = plan.S
    if not 0 < S <= 2048:
        raise ValueError(f"crop size {S} outside 1..2048")
    if plan.frames.ndim != 2 or plan.desc.shape != (plan.frames.shape[0], 7) or plan.video.shape != plan.frames.shape[:1]:
        raise ValueError("malformed clip plan")
    dims = [_check_shape(s) for s in shapes]
    for n in range(plan.frames.shape[0]):
        v = int(plan.video[n])
        if not 0 <= v < len(dims):
            raise ValueError(f"clip {n}: video {v} of {len(dims)}")
        F, H, W = dims[v]
        h, w, rh, rw, y0, x0, flip = (int(x) for x in plan.desc[n])
        if (h, w) != (H, W):
            raise ValueError(f"clip {n}: descriptor says {h}x{w}, the video is {H}x{W}")
        if S > min(rh, rw):
            raise ValueError(f"clip {n}: crop {S} is larger than the resized short side {min(rh, rw)}")
        if not (0 <= y0 <= rh - S and 0 <= x0 <= rw - S):
            raise ValueError(f"clip {n}: crop at ({y0}, {x0}) leaves the {rh}x{rw} resized frame")
        if flip not in (0, 1):
            raise ValueError(f"clip {n}: flip={flip}")
        f = plan.frames[n]
        if f.min() < 0 or f.max() >= F:
            raise ValueError(f"clip {n}: frame index outside 0..{F - 1}")


@dataclass
class VideoBatch:
    """Everything one x3d_video_clips_u8 launch needs, on the host: the distinct frames the plan
    reads, packed (pinned when a CUDA device is present, so the copy to the device is
    asynchronous), the byte offset of each output frame's source and the clip descriptors.
    `shape` is the shape of the uint8 clips it produces, [N, T, S, S, 3]."""
    frames: torch.Tensor        # [bytes] uint8
    frame_off: torch.Tensor     # [N*T] int64
    desc: torch.Tensor          # [N, 7] int32
    shape: Tuple[int, int, int, int, int]

    @property
    def h2d_bytes(self) -> int:
        return self.frames.numel() + self.frame_off.numel() * 8 + self.desc.numel() * 4

    def clips(self, device=None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Copy to `device` and build the clips there (current stream)."""
        from . import ops
        device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        frames = self.frames.to(device, non_blocking=True)
        off = self.frame_off.to(device, non_blocking=True)
        desc = self.desc.to(device, non_blocking=True)
        return ops.video_clips_u8(frames, off, desc, self.shape[1], self.shape[2], out=out)


def pack(videos: Sequence[np.ndarray], plan: ClipPlan, pin: Optional[bool] = None) -> VideoBatch:
    """Reads only the frames `plan` uses (each distinct frame once; a memory-mapped `.npy` video is
    read frame by frame) into one packed buffer.  A video is anything with `shape`, `dtype` and
    `video[f]` -> [H, W, 3] uint8 frame (a numpy array or memmap, or a frame reader)."""
    shapes = [np.shape(v) for v in videos]
    validate(plan, shapes)
    for i, v in enumerate(videos):
        if getattr(v, "dtype", None) != np.uint8:
            raise ValueError(f"video {i}: decoded frames must be uint8")
    N, T = plan.frames.shape
    keys = plan.video[:, None] * (1 << 32) + plan.frames                  # (video, frame) pairs
    uniq, inv = np.unique(keys.reshape(-1), return_inverse=True)
    sizes = np.asarray([shapes[int(k >> 32)][1] * shapes[int(k >> 32)][2] * 3 for k in uniq], np.int64)
    starts = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int64)
    total = int(sizes.sum())
    if pin is None:
        pin = torch.cuda.is_available()
    buf = torch.empty(total, dtype=torch.uint8, pin_memory=bool(pin))
    host = buf.numpy()
    for k, s, n in zip(uniq, starts, sizes):
        v, f = int(k >> 32), int(k & 0xffffffff)
        host[s:s + n] = np.ascontiguousarray(videos[v][f]).reshape(-1)
    off = torch.from_numpy(starts[inv].reshape(N * T).astype(np.int64))
    desc = torch.from_numpy(np.ascontiguousarray(plan.desc, np.int32))
    if pin:
        off, desc = off.pin_memory(), desc.pin_memory()
    return VideoBatch(buf, off, desc, plan.shape)


def load_video(path: str) -> np.ndarray:
    """A decoded video `.npy` [F, H, W, 3] uint8, memory-mapped (packing reads the sampled frames only)."""
    v = np.load(path, mmap_mode="r")
    _check_shape(v.shape)
    if v.dtype != np.uint8:
        raise ValueError(f"{path}: decoded frames must be uint8, got {v.dtype}")
    return v


def eval_batch(videos: List[np.ndarray], cfg) -> VideoBatch:
    """The evaluation clips of `videos` for cfg.DATA / cfg.TEST."""
    plan = eval_plan([v.shape for v in videos], cfg.DATA.TEMP_DURATION, cfg.TEST.NUM_TEMPORAL_VIEWS,
                     cfg.TEST.NUM_SPATIAL_CROPS, cfg.DATA.TEST_CROP_SIZE)
    return pack(videos, plan)


def train_batch(videos: List[np.ndarray], cfg, rng: np.random.Generator, crop_size: int = 0) -> VideoBatch:
    """One random training clip per video for cfg.DATA."""
    plan = train_plan([v.shape for v in videos], cfg.DATA.TEMP_DURATION, cfg.DATA.FRAME_RATE,
                      cfg.DATA.TRAIN_JITTER_SCALES, crop_size or cfg.DATA.TRAIN_CROP_SIZE, rng)
    return pack(videos, plan)
