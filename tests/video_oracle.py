"""numpy restatement of the clips built from decoded videos (x3d_tf_b200/video.py + x3d_video_clips_u8),
for the tests only.  Parity with TensorFlow is unpinned: the rules are restated from TF 2.4's
ResizeBilinear (half_pixel_centers=True, what tf.image.resize(method="bilinear") runs) and the
reference's transforms.py, and pinned here by hand-worked values (tests/test_video.py).

  resize_bilinear_u8  per channel, fp32, every operation rounded on its own (numpy never fuses):
                        scale = H / rh;  in = (y + 0.5) * scale - 0.5;  lo = max(floor(in), 0)
                        hi = min(ceil(in), H - 1);  l = in - floor(in)
                        top = tl + (tr - tl) * lx;  bottom = bl + (br - bl) * lx
                        v = top + (bottom - top) * ly;  out = uint8(trunc(v))  (tf.cast)
  resized_extent      short side -> size, long side -> floor(long * size / short)
  eval_clips          resize to short side TEST_CROP_SIZE, then io_oracle.eval_views (temporal views,
                      uniform crops, [crop][view] order)
  train_clip          the frames, resize, crop and flip of one clip of a plan
"""
from __future__ import annotations

import numpy as np

from oracle import io_oracle

f32 = np.float32


def resized_extent(H: int, W: int, size: int):
    if H <= W:
        return size, W * size // H
    return H * size // W, size


def _axis(n_in: int, n_out: int):
    scale = f32(n_in) / f32(n_out)
    p = (np.arange(n_out, dtype=f32) + f32(0.5)) * scale - f32(0.5)
    fl = np.floor(p)
    lo = np.maximum(fl, 0).astype(np.int64)
    hi = np.minimum(np.ceil(p), n_in - 1).astype(np.int64)
    return lo, hi, (p - fl).astype(f32)


def resize_bilinear_u8(frames: np.ndarray, rh: int, rw: int) -> np.ndarray:
    """[..., H, W, C] uint8 -> [..., rh, rw, C] uint8."""
    H, W = frames.shape[-3], frames.shape[-2]
    ylo, yhi, ly = _axis(H, rh)
    xlo, xhi, lx = _axis(W, rw)
    x = frames.astype(f32)
    top, bot = x[..., ylo, :, :], x[..., yhi, :, :]
    tl, tr, bl, br = top[..., xlo, :], top[..., xhi, :], bot[..., xlo, :], bot[..., xhi, :]
    lx = lx[:, None]
    ly = ly[:, None, None]
    t = tl + (tr - tl) * lx
    b = bl + (br - bl) * lx
    v = t + (b - t) * ly
    assert v.dtype == f32
    return np.trunc(v).astype(np.uint8)


def eval_clips(video: np.ndarray, T: int, views: int, crops: int, size: int) -> np.ndarray:
    rh, rw = resized_extent(video.shape[1], video.shape[2], size)
    return io_oracle.eval_views(resize_bilinear_u8(video, rh, rw), T, views, crops, size)


def train_clip(video: np.ndarray, frames, desc, S: int) -> np.ndarray:
    """One clip of a plan: `frames` [T] frame indices, `desc` (H, W, rh, rw, y0, x0, flip)."""
    H, W, rh, rw, y0, x0, flip = (int(v) for v in desc)
    assert video.shape[1:3] == (H, W)
    r = resize_bilinear_u8(np.asarray(video)[np.asarray(frames)], rh, rw)
    clip = r[:, y0:y0 + S, x0:x0 + S, :]
    return np.ascontiguousarray(clip[:, :, ::-1, :] if flip else clip)
