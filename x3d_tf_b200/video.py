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

Videos read from the reference's TFRecords (tfrecord.TFRecordVideo, JPEG frames) or from Motion-JPEG
AVI files (avi.MJPEGVideo) are packed by `pack_jpeg` instead of `pack`: the batch then carries the
entropy-coded segments of the distinct frames and their headers' tables (EncodedFrames), and the
frames are decoded on the device (x3d_jpeg_entropy / _entropy_rst / _idct / _color) into the packed
buffer the clip kernel reads.
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


DCT_METHODS = {"INTEGER_FAST": 1, "INTEGER_ACCURATE": 0}          # X3D_JPEG_IFAST / X3D_JPEG_ISLOW
STATUS_TEXT = {1: "invalid Huffman code", 2: "run of coefficients past coefficient 63",
               3: "premature end of the entropy-coded data"}


def _align16(n: int) -> int:
    return (n + 15) & ~15


@dataclass
class EncodedFrames:
    """The JPEG frames of a VideoBatch, on the host (pinned when a CUDA device is present):
    `data` the entropy-coded segments of the distinct frames, `frames` / `tables` their
    x3d_jpeg_frame / x3d_jpeg_tables records (raw bytes), the sizes of the device buffers the
    three decode stages use, the IDCT (`method`, DCT_METHODS) and a name per frame for messages.
    Frames with a restart interval (Motion-JPEG only) come last, from frame `nplain` on; their
    entropy stage is x3d_jpeg_entropy_rst over `intervals` (x3d_jpeg_interval records, raw bytes,
    empty for TFRecord batches)."""
    data: torch.Tensor          # [bytes] uint8
    frames: torch.Tensor        # [nframes * 64] uint8
    tables: torch.Tensor        # [ntables * 4200] uint8
    nframes: int
    coef_blocks: int
    plane_bytes: int
    out_bytes: int
    max_blocks: int
    max_pixels: int
    method: int
    names: List[str]
    intervals: Optional[torch.Tensor] = None   # [nintervals * 24] uint8
    nintervals: int = 0
    nplain: Optional[int] = None               # frames without a restart interval (None: all)

    @property
    def h2d_bytes(self) -> int:
        iv = self.intervals.numel() if self.intervals is not None else 0
        return self.data.numel() + self.frames.numel() + self.tables.numel() + iv

    def decode(self, device, scratch: dict) -> Tuple[torch.Tensor, torch.Tensor]:
        """Copy to `device` and decode on the current stream into buffers kept in `scratch` (grown
        as needed, reused while large enough).  Returns (decoded frames uint8, status int32
        [nframes]); the status words are only valid once the stream has reached them."""
        from . import ops

        def buf(name, n, dtype):
            t = scratch.get(name)
            if t is None or t.numel() < n:
                t = scratch[name] = torch.empty(max(n, 1), dtype=dtype, device=device)
            return t[:max(n, 1)]

        data, frames, tables = (buf(f"jpeg_{k}", v.numel(), torch.uint8) for k, v in
                                (("data", self.data), ("frames", self.frames), ("tables", self.tables)))
        data.copy_(self.data, non_blocking=True)
        frames.copy_(self.frames, non_blocking=True)
        tables.copy_(self.tables, non_blocking=True)
        coef = buf("jpeg_coef", self.coef_blocks * 64, torch.int16)
        planes = buf("jpeg_planes", self.plane_bytes, torch.uint8)
        out = buf("frames", self.out_bytes, torch.uint8)
        status = buf("jpeg_status", self.nframes, torch.int32)
        nplain = self.nframes if self.nplain is None else self.nplain
        if nplain:
            ops.jpeg_entropy(data, frames, tables, nplain, coef, status)
        if self.nintervals:
            iv = buf("jpeg_intervals", self.intervals.numel(), torch.uint8)
            iv.copy_(self.intervals, non_blocking=True)
            ops.jpeg_entropy_rst(data, frames, tables, iv, self.nintervals, coef, status, nplain, self.nframes)
        ops.jpeg_idct(coef, frames, tables, self.nframes, self.max_blocks, self.method, planes)
        ops.jpeg_color(planes, frames, self.nframes, self.max_pixels, out)
        return out, status

    def check(self, status) -> None:
        """Raises ValueError naming the record and frame of the first nonzero status word (TF's
        decode_jpeg with try_recover_truncated=False fails on such a frame too)."""
        st = np.asarray(status).reshape(-1)[:self.nframes]
        bad = np.flatnonzero(st)
        if bad.size:
            i = int(bad[0])
            raise ValueError(f"{self.names[i]}: JPEG decoding failed: {STATUS_TEXT.get(int(st[i]), int(st[i]))}")


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
    encoded: Optional[EncodedFrames] = None   # JPEG frames (pack_jpeg): `frames` is empty, and
                                              # frame_off points into the frames they decode to

    @property
    def h2d_bytes(self) -> int:
        enc = self.encoded.h2d_bytes if self.encoded is not None else 0
        return self.frames.numel() + self.frame_off.numel() * 8 + self.desc.numel() * 4 + enc

    def clips(self, device=None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Copy to `device` and build the clips there (current stream).  JPEG frames are decoded
        first; their status words are checked before this returns (a synchronisation), so a
        corrupt frame raises ValueError here."""
        from . import ops
        device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        if self.encoded is not None:
            frames, status = self.encoded.decode(device, {})
            self.encoded.check(status.cpu().numpy())
        else:
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


def pack_jpeg(videos: Sequence, plan: ClipPlan, pin: Optional[bool] = None,
              dct_method: str = "INTEGER_FAST") -> VideoBatch:
    """`pack` for videos of JPEG frames (tfrecord.TFRecordVideo, avi.MJPEGVideo, or anything with
    `shape` and `jpeg(f)` -> bytes): the entropy-coded segment of each distinct (video, frame) pair
    the plan reads, once, in one buffer; a table set per distinct header; the frame descriptors and
    the offsets of the decoded frames (16-byte aligned) that frame_off points at.  Headers are parsed
    and checked here (jpeg.parse; with mjpeg=True for videos whose `mjpeg` attribute is true), so an
    unsupported or mis-sized frame raises ValueError naming its video and frame before anything
    reaches the device.  `dct_method`: TF's decode_jpeg names, INTEGER_FAST (its default) or
    INTEGER_ACCURATE."""
    shapes = [tuple(int(x) for x in v.shape) for v in videos]
    validate(plan, shapes)
    N, T = plan.frames.shape
    keys = plan.video[:, None] * (1 << 32) + plan.frames
    uniq, inv = np.unique(keys.reshape(-1), return_inverse=True)
    enc, out_off = encoded_frames(videos, [(int(k >> 32), int(k & 0xffffffff)) for k in uniq], pin, dct_method)
    off = torch.from_numpy(out_off[inv].reshape(N * T).astype(np.int64))
    desc = torch.from_numpy(np.ascontiguousarray(plan.desc, np.int32))
    if enc.frames.is_pinned():
        off, desc = off.pin_memory(), desc.pin_memory()
    return VideoBatch(torch.empty(0, dtype=torch.uint8), off, desc, plan.shape, enc)


def encoded_frames(videos: Sequence, pairs: Sequence[Tuple[int, int]], pin: Optional[bool] = None,
                  dct_method: str = "INTEGER_FAST") -> Tuple[EncodedFrames, np.ndarray]:
    """The EncodedFrames of the (video, frame) `pairs` (distinct), and the byte offset in the
    decoded buffer of each pair's [H, W, 3] frame.  Frames without a restart interval come first in
    the batch (x3d_jpeg_entropy), then those with one (an x3d_jpeg_interval per interval)."""
    from . import jpeg as J
    from . import _lib
    if dct_method not in DCT_METHODS:
        raise ValueError(f"dct_method {dct_method!r}: INTEGER_FAST or INTEGER_ACCURATE")
    parsed = []
    for v, f in pairs:
        name = f"{getattr(videos[v], 'name', f'video {v}')} frame {f}"
        buf = videos[v].jpeg(f)
        try:
            fr = J.parse(buf, mjpeg=bool(getattr(videos[v], "mjpeg", False)))
        except ValueError as e:
            raise ValueError(f"{name}: {e}") from None
        h = fr.header
        shape = tuple(int(x) for x in videos[v].shape)
        if (h.H, h.W) != shape[1:3]:
            raise ValueError(f"{name}: {h.H}x{h.W}, but frame 0 of its video is {shape[1]}x{shape[2]}")
        parsed.append((name, buf, fr))
    order = sorted(range(len(parsed)), key=lambda n: parsed[n][2].header.ri != 0)     # stable
    recs = np.zeros(len(parsed), J.FRAME_DTYPE)
    out_off = np.zeros(len(parsed), np.int64)
    table_index, table_recs, segs, names, ivs = {}, [], [], [], []
    seg_off = coef = plane = out = 0
    max_blocks = max_pixels = 0
    nplain = 0
    for n, p in enumerate(order):
        name, buf, fr = parsed[p]
        h = fr.header
        t = table_index.get(id(h))
        if t is None:
            t = table_index[id(h)] = len(table_recs)
            table_recs.append(h)
        blocks = h.mcus * (h.hs * h.vs + 2)
        recs[n] = (seg_off, coef, plane, out, fr.seg_len, h.H, h.W, h.hs, h.vs, t, n, 0)
        if h.ri:
            iv = np.zeros(len(fr.intervals), J.INTERVAL_DTYPE)
            iv["off"] = fr.intervals[:, 0] - fr.seg_off + seg_off
            iv["len"] = fr.intervals[:, 1]
            iv["frame"] = n
            iv["mcu0"] = np.arange(len(iv)) * h.ri
            iv["nmcu"] = np.minimum(h.ri, h.mcus - iv["mcu0"])
            ivs.append(iv)
        else:
            nplain = n + 1
        segs.append(memoryview(buf)[fr.seg_off:fr.seg_off + fr.seg_len])
        names.append(name)
        out_off[p] = out
        seg_off += fr.seg_len
        coef += blocks
        plane += blocks * 64
        out += _align16(h.H * h.W * 3)
        max_blocks, max_pixels = max(max_blocks, blocks), max(max_pixels, h.H * h.W)
    if pin is None:
        pin = torch.cuda.is_available()
    data = torch.empty(max(seg_off, 1), dtype=torch.uint8, pin_memory=bool(pin))
    host = data.numpy()
    for r, sg in zip(recs, segs):
        host[r["seg_off"]:r["seg_off"] + len(sg)] = np.frombuffer(sg, np.uint8)
    tables = np.stack([h.tables for h in table_recs])
    frames_t = torch.from_numpy(recs.view(np.uint8).copy())
    tables_t = torch.from_numpy(tables.view(np.uint8).reshape(-1).copy())
    iv = np.concatenate(ivs) if ivs else np.zeros(0, J.INTERVAL_DTYPE)
    iv_t = torch.from_numpy(iv.view(np.uint8).copy())
    if pin:
        frames_t, tables_t, iv_t = (t.pin_memory() for t in (frames_t, tables_t, iv_t))
    enc = EncodedFrames(data, frames_t, tables_t, len(parsed), coef, plane, out, max_blocks, max_pixels,
                        DCT_METHODS[dct_method], names, iv_t, len(iv), nplain if ivs else None)
    return enc, out_off


def _pack(videos, plan: ClipPlan, dct_method: str) -> VideoBatch:
    return pack_jpeg(videos, plan, dct_method=dct_method) if hasattr(videos[0], "jpeg") else pack(videos, plan)


def load_video(path: str) -> np.ndarray:
    """A decoded video `.npy` [F, H, W, 3] uint8, memory-mapped (packing reads the sampled frames only)."""
    v = np.load(path, mmap_mode="r")
    _check_shape(v.shape)
    if v.dtype != np.uint8:
        raise ValueError(f"{path}: decoded frames must be uint8, got {v.dtype}")
    return v


def eval_batch(videos: List[np.ndarray], cfg, dct_method: str = "INTEGER_FAST") -> VideoBatch:
    """The evaluation clips of `videos` (decoded, or of JPEG frames) for cfg.DATA / cfg.TEST."""
    plan = eval_plan([v.shape for v in videos], cfg.DATA.TEMP_DURATION, cfg.TEST.NUM_TEMPORAL_VIEWS,
                     cfg.TEST.NUM_SPATIAL_CROPS, cfg.DATA.TEST_CROP_SIZE)
    return _pack(videos, plan, dct_method)


def train_batch(videos: List[np.ndarray], cfg, rng: np.random.Generator, crop_size: int = 0,
                dct_method: str = "INTEGER_FAST") -> VideoBatch:
    """One random training clip per video (decoded, or of JPEG frames) for cfg.DATA."""
    plan = train_plan([v.shape for v in videos], cfg.DATA.TEMP_DURATION, cfg.DATA.FRAME_RATE,
                      cfg.DATA.TRAIN_JITTER_SCALES, crop_size or cfg.DATA.TRAIN_CROP_SIZE, rng)
    return _pack(videos, plan, dct_method)
