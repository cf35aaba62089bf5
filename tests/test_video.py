"""Host side of the clips built from decoded videos (x3d_tf_b200/video.py), the numpy restatement
the GPU tests compare against (tests/video_oracle.py) and the C layout of x3d_clip_desc.  No GPU."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import io_oracle
from tests import video_oracle as VO
from x3d_tf_b200 import video as V

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _row(vals):
    return np.asarray(vals, np.uint8).reshape(1, -1, 1)


def test_oracle_hand_worked_values():
    assert VO.resize_bilinear_u8(_row([0, 255]), 1, 3).ravel().tolist() == [0, 127, 255]
    assert VO.resize_bilinear_u8(_row([10, 20, 30, 41]), 1, 2).ravel().tolist() == [15, 35]   # 35.5 truncated
    x = np.random.default_rng(0).integers(0, 256, size=(3, 17, 23, 3), dtype=np.uint8)
    assert np.array_equal(VO.resize_bilinear_u8(x, 17, 23), x)
    # the same rows as columns
    assert VO.resize_bilinear_u8(_row([0, 255]).reshape(2, 1, 1), 3, 1).ravel().tolist() == [0, 127, 255]


def test_resized_extent():
    assert V.resized_extent(360, 480, 256) == (256, 341)          # landscape: 480 * 256 / 360 = 341.33
    assert V.resized_extent(480, 360, 256) == (341, 256)          # portrait
    assert V.resized_extent(300, 300, 224) == (224, 224)          # square
    assert V.resized_extent(256, 340, 256) == (256, 340)          # already sized: identity
    assert V.resized_extent(100, 140, 320) == (320, 448)          # upscale
    for H, W, s in ((360, 480, 256), (481, 359, 182), (7, 9, 5)):
        assert V.resized_extent(H, W, s) == VO.resized_extent(H, W, s)
    with pytest.raises(ValueError):
        V.resized_extent(0, 10, 5)


@pytest.mark.parametrize("F,H,W,T,views,crops,S", [(40, 20, 28, 4, 2, 3, 20), (7, 33, 21, 4, 3, 3, 21),
                                                   (100, 16, 16, 13, 1, 1, 16), (5, 24, 19, 16, 10, 1, 19)])
def test_eval_plan_identity_reproduces_eval_views(F, H, W, T, views, crops, S):
    """With the short side already at the crop size the plan is an identity resize, and gathering
    its frames and crops reproduces io_oracle.eval_views."""
    video = np.random.default_rng(F + H).integers(0, 256, size=(F, H, W, 3), dtype=np.uint8)
    plan = V.eval_plan([video.shape], T, views, crops, S)
    assert plan.shape == (crops * views, T, S, S, 3)
    assert (plan.desc[:, 2] == H).all() and (plan.desc[:, 3] == W).all() and (plan.desc[:, 6] == 0).all()
    got = np.stack([VO.train_clip(video, plan.frames[n], plan.desc[n], S) for n in range(plan.frames.shape[0])])
    assert np.array_equal(got, io_oracle.eval_views(video, T, views, crops, S))


def test_eval_plan_resized_matches_oracle_eval_clips():
    video = np.random.default_rng(3).integers(0, 256, size=(9, 30, 41, 3), dtype=np.uint8)
    plan = V.eval_plan([video.shape], 4, 2, 3, 24)
    got = np.stack([VO.train_clip(video, plan.frames[n], plan.desc[n], 24) for n in range(6)])
    assert np.array_equal(got, VO.eval_clips(video, 4, 2, 3, 24))


def _shapes():
    return [(50, 360, 480, 3), (7, 100, 140, 3), (300, 481, 359, 3)]


def test_train_plan_deterministic_per_seed_and_rank():
    a = V.train_plan(_shapes(), 16, 5, (256, 320), 224, V.train_rng(11, 0))
    b = V.train_plan(_shapes(), 16, 5, (256, 320), 224, V.train_rng(11, 0))
    c = V.train_plan(_shapes(), 16, 5, (256, 320), 224, V.train_rng(11, 1))
    d = V.train_plan(_shapes(), 16, 5, (256, 320), 224, V.train_rng(12, 0))
    assert np.array_equal(a.frames, b.frames) and np.array_equal(a.desc, b.desc)
    assert not np.array_equal(a.desc, c.desc) or not np.array_equal(a.frames, c.frames)
    assert not np.array_equal(a.desc, d.desc) or not np.array_equal(a.frames, d.frames)


def test_train_plan_bounds_flip_and_wrap():
    rng = V.train_rng(3, 2)
    for _ in range(50):
        p = V.train_plan(_shapes(), 16, 5, (256, 320), 224, rng)
        V.validate(p, _shapes())
        for n, (F, H, W, _) in enumerate(_shapes()):
            h, w, rh, rw, y0, x0, flip = p.desc[n]
            assert (h, w) == (H, W) and flip == 1
            assert 256 <= min(rh, rw) <= 320 and (rh, rw) == V.resized_extent(H, W, min(rh, rw))
            assert 0 <= y0 <= rh - 224 and 0 <= x0 <= rw - 224
            f = p.frames[n]
            assert ((f - f[0]) % F == (np.arange(16) * 5) % F).all() and f.max() < F
    # the 7-frame video loops: 16 frames at stride 5 must wrap
    assert len(set(p.frames[1].tolist())) <= 7


def test_pack_keeps_distinct_frames_only():
    rng = np.random.default_rng(1)
    videos = [rng.integers(0, 256, size=s, dtype=np.uint8) for s in ((5, 12, 16, 3), (3, 9, 7, 3))]
    plan = V.eval_plan([v.shape for v in videos], 4, 2, 3, 6)            # 4*2 = 8 frames of 5 and of 3: loops
    b = V.pack(videos, plan, pin=False)
    assert b.shape == (12, 4, 6, 6, 3)
    assert b.frames.numel() == 5 * 12 * 16 * 3 + 3 * 9 * 7 * 3             # every frame once, no repeats
    host = b.frames.numpy()
    off = b.frame_off.numpy().reshape(12, 4)
    for n in range(12):
        v = videos[plan.video[n]]
        for t in range(4):
            o = off[n, t]
            got = host[o:o + v[0].size].reshape(v.shape[1:])
            assert np.array_equal(got, v[plan.frames[n, t]])
    assert np.array_equal(b.desc.numpy(), plan.desc)


def test_pack_reads_memory_mapped_npy(tmp_path):
    v = np.random.default_rng(2).integers(0, 256, size=(20, 10, 14, 3), dtype=np.uint8)
    np.save(tmp_path / "v.npy", v)
    m = V.load_video(str(tmp_path / "v.npy"))
    assert isinstance(m, np.memmap)
    plan = V.eval_plan([m.shape], 4, 1, 1, 10)
    b = V.pack([m], plan, pin=False)
    assert b.frames.numel() == 4 * 10 * 14 * 3
    np.save(tmp_path / "bad.npy", v.astype(np.float32))
    with pytest.raises(ValueError):
        V.load_video(str(tmp_path / "bad.npy"))


def test_bad_plans_raise_value_error():
    shapes = [(10, 30, 40, 3)]
    plan = V.eval_plan(shapes, 4, 1, 1, 24)
    V.validate(plan, shapes)
    bad = V.ClipPlan(plan.video, plan.frames, plan.desc.copy(), plan.S)
    bad.desc[0, 5] = bad.desc[0, 3] - 23                                  # crop leaves the resized frame
    with pytest.raises(ValueError, match="leaves"):
        V.validate(bad, shapes)
    big = V.ClipPlan(plan.video, plan.frames, plan.desc, 25)              # S larger than the short side
    with pytest.raises(ValueError, match="larger"):
        V.validate(big, shapes)
    frames = plan.frames.copy(); frames[0, 0] = 10
    with pytest.raises(ValueError, match="frame index"):
        V.validate(V.ClipPlan(plan.video, frames, plan.desc, 24), shapes)
    flip = plan.desc.copy(); flip[0, 6] = 2
    with pytest.raises(ValueError, match="flip"):
        V.validate(V.ClipPlan(plan.video, plan.frames, flip, 24), shapes)
    with pytest.raises(ValueError, match="larger"):
        V.train_plan(shapes, 4, 5, (200, 240), 224, V.train_rng(0))
    for s in ((0, 30, 40, 3), (10, 0, 40, 3), (10, 30, 40), (10, 30, 40, 1)):
        with pytest.raises(ValueError):
            V.eval_plan([s], 4, 1, 1, 24)
    with pytest.raises(ValueError):
        V.eval_plan([], 4, 1, 1, 24)
    with pytest.raises(ValueError):
        V.pack([np.zeros((10, 30, 40, 3), np.float32)], plan, pin=False)


def test_clip_desc_layout_matches_header(tmp_path):
    """x3d_clip_desc as gcc lays it out == the ctypes structure and the [N, 7] int32 rows video.py uploads."""
    from x3d_tf_b200 import _lib
    ct = _lib.ClipDesc
    lines = ['#include <stddef.h>', '#include <stdio.h>', '#include "x3d_b200.h"', 'int main(void) {',
             '  printf("size %zu\\n", sizeof(x3d_clip_desc));']
    lines += [f'  printf("{f} %zu\\n", offsetof(x3d_clip_desc, {f}));' for f, _ in ct._fields_]
    lines += ['  return 0;', '}']
    (tmp_path / "probe.c").write_text("\n".join(lines))
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(tmp_path / "probe.c")], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert int(got["size"]) == ctypes.sizeof(ct) == 7 * 4
    assert [f for f, _ in ct._fields_] == list(V.DESC_FIELDS)
    for i, (f, _) in enumerate(ct._fields_):
        assert int(got[f]) == getattr(ct, f).offset == 4 * i


def _cuobjdump():
    for c in (os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump"), shutil.which("cuobjdump")):
        if c and os.path.exists(c):
            return c
    return None


@pytest.mark.skipif(_cuobjdump() is None, reason="cuobjdump not installed")
def test_interpolation_has_no_fma():
    """Every interpolation is rounded per operation: after the table phase (the barrier) the clip
    kernel's main body has no FFMA (the correctly rounded division of the table phase keeps its own)."""
    from x3d_tf_b200 import _lib, build
    build.build()
    sass = subprocess.run([_cuobjdump(), "-sass", _lib.LIB_PATH], check=True, capture_output=True, text=True).stdout
    funcs = [f for f in sass.split("Function : ")[1:] if f.startswith("_ZN3x3d2io21video_clips_u8_kernel")]
    assert len(funcs) == 2                                                # device-array plan and by-value plan
    for f in funcs:
        body = f[f.index("BAR.SYNC"):]
        body = body[:body.rindex(" EXIT ;")]
        assert "FFMA" not in body and "FMUL" in body and "FADD" in body
