"""Motion-JPEG AVI input on the device: x3d_jpeg_entropy_rst and the 4:2:2 paths against Pillow
(libjpeg-turbo) and the numpy restatement (tests/mjpeg_oracle.py), corrupt intervals, and the drivers
(eval.py / X3D.fit / create_tfrecords with --mjpeg_videos) against the same frames decoded by Pillow.
Every decode case writes >= 100 kB."""
import os

import numpy as np
import pytest
import torch

from tests import avi_writer as AW
from tests import mjpeg_oracle as M
from tests import tfrecord_writer as TW
from x3d_tf_b200 import avi
from x3d_tf_b200 import jpeg as J
from x3d_tf_b200 import ops
from x3d_tf_b200 import tfrecord as R
from x3d_tf_b200 import video as V
from x3d_tf_b200.arch import build_arch
from x3d_tf_b200.config import get_config
from x3d_tf_b200.synth import synthetic_weights

pytestmark = pytest.mark.gpu


def _avi(path, jpegs):
    h = J.parse_header(jpegs[0], mjpeg=True)
    AW.write_avi(str(path), jpegs, h.W, h.H, audio=True)
    return avi.MJPEGVideo(str(path))


def _decode(vb):
    frames, status = vb.encoded.decode("cuda", {})
    torch.cuda.synchronize()
    return frames.cpu().numpy(), status.cpu().numpy()


def _by_pair(vb, flat, pairs_shape):
    """Decoded frames in plan order (frame_off), [N*T] of [H, W, 3]."""
    H, W = pairs_shape
    return [flat[o:o + H * W * 3].reshape(H, W, 3) for o in vb.frame_off.numpy()]


CASES = [("420_rst_1mcu", 2, {"restart_marker_blocks": 1}, (360, 480)),
         ("420_rst_row", 2, {"restart_marker_rows": 1}, (360, 480)),
         ("420_rst_uneven", 2, {"restart_marker_blocks": 7}, (241, 179)),
         ("420_rst_row_1080p", 2, {"restart_marker_rows": 1}, (1080, 1920)),
         ("420_rst_1mcu_8x8", 2, {"restart_marker_blocks": 1}, (8, 8)),
         ("422_plain", 1, {}, (241, 179)),
         ("422_rst_row", 1, {"restart_marker_rows": 1}, (360, 480)),
         ("422_rst_uneven_odd", 1, {"restart_marker_blocks": 5}, (37, 53)),
         ("422_rst_1mcu_1080p", 1, {"restart_marker_blocks": 1}, (1080, 1920)),
         ("444_rst_uneven", 0, {"restart_marker_blocks": 3}, (37, 53))]


def _case_jpegs(sub, kw, hw, seed):
    H, W = hw
    F = max(2, -(-100_000 // (H * W * 3)))
    return [TW.encode(f, quality=90, subsampling=sub, **kw) for f in TW.video_frames(F, H, W, seed, noise=2.0)]


@pytest.mark.parametrize("case", [c[0] for c in CASES])
def test_decode_islow_byte_identical_to_pillow(tmp_path, case):
    _, sub, kw, hw = next(c for c in CASES if c[0] == case)
    jpegs = _case_jpegs(sub, kw, hw, len(case))
    v = _avi(tmp_path / "v.avi", jpegs)
    vb = V.pack_jpeg([v], V.eval_plan([v.shape], len(jpegs), 1, 1, min(hw)), dct_method="INTEGER_ACCURATE")
    flat, status = _decode(vb)
    assert not status.any()
    got = _by_pair(vb, flat, hw)
    assert sum(g.nbytes for g in got) >= 100_000
    for g, j in zip(got, jpegs):
        want = TW.pil_decode(j)
        assert np.array_equal(g, want), f"{(g != want).sum()} of {g.size} bytes differ"


def test_ragged_batch_mixes_restart_422_and_tfrecord_frames(tmp_path):
    """AVI videos of every case and TFRecord-style videos in one batch: one launch per stage, the
    restart-interval frames through x3d_jpeg_entropy_rst; every frame == Pillow."""
    videos, want = [], []
    for i, (name, sub, kw, hw) in enumerate(CASES):
        jpegs = _case_jpegs(sub, kw, hw, 200 + i)[:2]
        videos.append(_avi(tmp_path / f"{name}.avi", jpegs))
        want.append(jpegs)
    for i, hw in enumerate([(180, 240), (37, 53)]):
        jpegs = [TW.encode(f) for f in TW.video_frames(2, *hw, 300 + i)]
        videos.append(R.parse_sequence_example(TW.sequence_example(jpegs, 0), f"rec{i}"))
        want.append(jpegs)
    plan = V.eval_plan([v.shape for v in videos], 2, 1, 1, 8)
    vb = V.pack_jpeg(videos, plan, dct_method="INTEGER_ACCURATE")
    assert 0 < vb.encoded.nplain < vb.encoded.nframes and vb.encoded.nintervals > 0
    before = ops.Profiler.launches
    flat, status = _decode(vb)
    assert ops.Profiler.launches - before == 4 and not status.any()
    offs = vb.frame_off.numpy()
    total = 0
    for n in range(len(videos)):
        for t in range(2):
            j = want[n][plan.frames[n, t]]
            w = TW.pil_decode(j)
            g = flat[offs[n * 2 + t]:offs[n * 2 + t] + w.size].reshape(w.shape)
            assert np.array_equal(g, w), (n, t)
            total += w.nbytes
    assert total >= 100_000


def test_ifast_equals_mjpeg_oracle(tmp_path):
    jpegs = [TW.encode(f, quality=q, subsampling=s, **kw) for f, q, s, kw in
             zip(TW.video_frames(4, 200, 176, 4), (90, 50, 100, 75), (2, 1, 1, 0),
                 ({"restart_marker_rows": 1}, {"restart_marker_blocks": 3}, {}, {"restart_marker_blocks": 1}))]
    v = _avi(tmp_path / "v.avi", jpegs)
    vb = V.pack_jpeg([v], V.eval_plan([v.shape], 4, 1, 1, 176), dct_method="INTEGER_FAST")
    flat, status = _decode(vb)
    assert not status.any()
    got = _by_pair(vb, flat, (200, 176))
    assert sum(g.nbytes for g in got) >= 100_000
    for g, j in zip(got, jpegs):
        assert np.array_equal(g, M.decode(j, "INTEGER_FAST"))


def _corrupt(good):
    """(an interval cut short, a bad Huffman code inside an interval) of a restart-interval frame."""
    fr = J.parse(good, mjpeg=True)
    (o, n) = (int(x) for x in fr.intervals[3])
    short = good[:o + n // 3] + good[o + n:]
    mid = o + n // 2
    while good[mid - 1] == 0xFF or good[mid + 7] == 0xFF:
        mid += 1
    bad = good[:mid] + b"\xff\x00" * 8 + good[mid + 8:]
    return short, bad


def test_corrupt_intervals_set_status_and_stay_in_bounds(tmp_path):
    img = TW.video_frames(1, 240, 320, 9)[0]
    good = TW.encode(img, restart_marker_rows=1)
    short, bad = _corrupt(good)
    v = _avi(tmp_path / "c.avi", [good, short, bad, good])
    vb = V.pack_jpeg([v], V.eval_plan([v.shape], 4, 1, 1, 240), dct_method="INTEGER_ACCURATE")
    enc = vb.encoded
    G = 4096
    sizes = {"jpeg_coef": (enc.coef_blocks * 64, torch.int16), "jpeg_planes": (enc.plane_bytes, torch.uint8),
             "frames": (enc.out_bytes, torch.uint8), "jpeg_status": (enc.nframes, torch.int32)}
    scratch = {k: torch.full((n + G,), 0x5A, dtype=dt, device="cuda") for k, (n, dt) in sizes.items()}
    flat, status = enc.decode("cuda", scratch)
    torch.cuda.synchronize()
    st = status.cpu().numpy()
    assert list(st) == [0, 3, 1, 0]                               # frames in file order (all have intervals)
    for k, (n, _) in sizes.items():
        assert bool((scratch[k][n:] == 0x5A).all()), k
    got = _by_pair(vb, flat.cpu().numpy(), (240, 320))
    assert np.array_equal(got[0], TW.pil_decode(good)) and np.array_equal(got[3], TW.pil_decode(good))
    with pytest.raises(ValueError, match=r"c\.avi frame 1: JPEG decoding failed: premature end"):
        enc.check(st)


def test_corrupt_interval_writes_only_its_own_blocks(tmp_path):
    """The coefficient blocks of the MCUs after a failed interval's error (and of no other frame) are
    left as they were: every block outside the corrupt frame equals a clean decode, and the corrupt
    frame's blocks of the intervals before and after the bad one equal the clean decode too."""
    img = TW.video_frames(2, 240, 320, 10)
    good = [TW.encode(f, restart_marker_rows=1) for f in img]
    _, bad = _corrupt(good[1])
    clean = V.pack_jpeg([_avi(tmp_path / "a.avi", good)], V.eval_plan([(2, 240, 320, 3)], 2, 1, 1, 240))
    dirty = V.pack_jpeg([_avi(tmp_path / "b.avi", [good[0], bad])], V.eval_plan([(2, 240, 320, 3)], 2, 1, 1, 240))
    sa, sb = {}, {}
    clean.encoded.decode("cuda", sa)
    n = dirty.encoded.coef_blocks * 64
    sb["jpeg_coef"] = torch.full((n,), 0x5A5A, dtype=torch.int16, device="cuda")
    _, status = dirty.encoded.decode("cuda", sb)
    torch.cuda.synchronize()
    assert list(status.cpu().numpy()) == [0, 1]
    ca, cb = sa["jpeg_coef"][:n].cpu().numpy().reshape(-1, 64), sb["jpeg_coef"][:n].cpu().numpy().reshape(-1, 64)
    recs = dirty.encoded.frames.numpy().view(J.FRAME_DTYPE)
    f1 = int(recs["coef_off"][1])
    assert np.array_equal(ca[:f1], cb[:f1])                       # frame 0 untouched by frame 1's failure
    differ = np.flatnonzero((ca[f1:] != cb[f1:]).any(1))
    assert differ.size and (cb[f1:][differ] == 0x5A5A).all(1).mean() > 0.5     # mostly blocks left unwritten
    # 240x320 4:2:0: luma 40 x 30 blocks, chroma 20 x 15 each; interval 3 is MCU row 3 = luma block
    # rows 6 and 7, chroma block row 3
    luma, chroma = differ[differ < 1200], (differ[differ >= 1200] - 1200) % 300
    assert set((luma // 40).tolist()) <= {6, 7} and set((chroma // 20).tolist()) <= {3}


# ------------------------------------------------------------------------------------------ drivers
def _model_dir(tmp_path, cfg, seed):
    from x3d_tf_b200 import model as M_
    M_.reset_block_counters()
    m = M_.X3D(cfg, dtype="bfloat16")
    m.set_weights_dict(synthetic_weights(build_arch(cfg), seed=seed))
    m.save_weights(str(tmp_path / "ckpt-1"))
    (tmp_path / "checkpoint").write_text('model_checkpoint_path: "ckpt-1"\nall_model_checkpoint_paths: "ckpt-1"\n')


def _avi_and_npy(tmp_path, shapes, seed, kinds):
    """AVI files of Pillow-encoded frames (restart intervals / 4:2:2 per `kinds`), .npy files of the
    same frames decoded by Pillow, and the two lists."""
    avis, npys = [], []
    for i, ((F, H, W), (sub, kw)) in enumerate(zip(shapes, kinds)):
        jpegs = [TW.encode(f, subsampling=sub, **kw) for f in TW.video_frames(F, H, W, seed + i)]
        AW.write_avi(str(tmp_path / f"v{i}.avi"), jpegs, W, H, rec=i % 2 == 1)
        np.save(tmp_path / f"v{i}.npy", np.stack([TW.pil_decode(j) for j in jpegs]))
        avis.append(f"v{i}.avi")
        npys.append(f"v{i}.npy")
    return avis, npys


KINDS = [(2, {"restart_marker_rows": 1}), (1, {}), (1, {"restart_marker_blocks": 5}), (2, {})]


def test_eval_driver_mjpeg_equals_decoded_videos(tmp_path):
    from x3d_tf_b200 import eval as E
    cfg = get_config("X3D_XS")
    _model_dir(tmp_path, cfg, 77)
    avis, npys = _avi_and_npy(tmp_path, [(24, 180, 240), (9, 240, 180), (15, 161, 163), (12, 120, 160)], 12, KINDS)
    labels = [3, 200, 17, 5]
    (tmp_path / "avi.txt").write_text("".join(f"{p} {l}\n" for p, l in zip(avis, labels)))
    (tmp_path / "npy.txt").write_text("".join(f"{p} {l}\n" for p, l in zip(npys, labels)))
    base = ["--cfg", "X3D_XS", "--model_folder", str(tmp_path)]
    want = E.run(base + ["--test_file_pattern", str(tmp_path / "npy.txt"), "--decoded_videos"])
    got = E.run(base + ["--test_file_pattern", str(tmp_path / "avi.txt"), "--mjpeg_videos",
                        "--dct_method", "INTEGER_ACCURATE"])
    assert got == want and got["videos"] == 4


def test_fit_from_avi_equals_fit_from_decodes(tmp_path):
    from x3d_tf_b200 import model as M_
    from x3d_tf_b200.train import video_clip_batches
    cfg = get_config("X3D_XS", freeze=False)
    cfg.NETWORK.DROPOUT_RATE = 0.0
    cfg.freeze()
    avis, npys = _avi_and_npy(tmp_path, [(30, 240, 320), (16, 200, 150), (20, 180, 180), (12, 160, 224)], 40, KINDS)
    labels = [7, 311, 2, 100]
    items_a = [(str(tmp_path / p), l) for p, l in zip(avis, labels)]
    items_n = [(str(tmp_path / p), l) for p, l in zip(npys, labels)]
    W = synthetic_weights(build_arch(cfg), seed=5)
    hists = []
    for items, mj in ((items_a, True), (items_n, False)):
        data = list(video_clip_batches(items, 2, 2, 1234, cfg, mjpeg=mj, dct_method="INTEGER_ACCURATE"))
        M_.reset_block_counters()
        m = M_.X3D(cfg)
        m.set_weights_dict(W)
        hists.append((m.fit(data, epochs=1, lr_schedule=lambda e: 0.01), m.named_variables()))
    (ha, wa), (hn, wn) = hists
    assert ha["loss"] == hn["loss"]
    assert all(np.array_equal(wa[k], wn[k]) for k in wa)


def test_create_tfrecords_from_avi_equals_from_decodes(tmp_path):
    from x3d_tf_b200 import create_tfrecords as C
    avis, npys = _avi_and_npy(tmp_path, [(12, 180, 240), (9, 120, 160), (7, 97, 131)], 60, KINDS)
    (tmp_path / "avi.txt").write_text("".join(f"{p} {i}\n" for i, p in enumerate(avis)))
    (tmp_path / "npy.txt").write_text("".join(f"{p} {i}\n" for i, p in enumerate(npys)))
    common = ["--videos_per_file", "2", "--max_frames", "8", "--threads", "2"]
    C.run(["--file_list", str(tmp_path / "npy.txt"), "--out_dir", str(tmp_path / "npy")] + common)
    C.run(["--file_list", str(tmp_path / "avi.txt"), "--out_dir", str(tmp_path / "avi"), "--mjpeg_videos",
           "--dct_method", "INTEGER_ACCURATE"] + common)
    names = sorted(os.listdir(tmp_path / "npy"))
    assert names == sorted(os.listdir(tmp_path / "avi")) and len(names) == 2
    for n in names:
        a = list(R.read_records(str(tmp_path / "avi" / n)))
        b = list(R.read_records(str(tmp_path / "npy" / n)))
        assert [bytes(x) for x in a] == [bytes(x) for x in b]
