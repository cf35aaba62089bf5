"""The device JPEG decoder (x3d_jpeg_entropy / _idct / _color) against Pillow (libjpeg-turbo) and the
numpy restatement (tests/jpeg_oracle.py), corrupt data, the clips of TFRecord batches, and every
consumer (X3D.evaluate, the eval driver with --tfrecord, X3D.fit).  Every decode case writes >= 100 kB."""
import numpy as np
import pytest
import torch

from tests import jpeg_oracle as O
from tests import tfrecord_writer as TW
from x3d_tf_b200 import jpeg as J
from x3d_tf_b200 import tfrecord as R
from x3d_tf_b200 import video as V
from x3d_tf_b200.arch import build_arch
from x3d_tf_b200.config import get_config
from x3d_tf_b200.synth import synthetic_weights

pytestmark = pytest.mark.gpu


def _content(kind, F, H, W, seed):
    if kind == "noise":
        return np.random.default_rng(seed).integers(0, 256, (F, H, W, 3), dtype=np.uint8)
    return TW.video_frames(F, H, W, seed, noise=2.0)


def _video(jpegs, name="rec"):
    return R.parse_sequence_example(TW.sequence_example(jpegs, 0), name)


def _decode(vb):
    frames, status = vb.encoded.decode("cuda", {})
    torch.cuda.synchronize()
    return frames.cpu().numpy(), status.cpu().numpy()


def _frames_of(vb, flat):
    recs = vb.encoded.frames.numpy().view(J.FRAME_DTYPE)
    return [flat[r["out_off"]:r["out_off"] + r["H"] * r["W"] * 3].reshape(r["H"], r["W"], 3) for r in recs]


CASES = [("420_q90_smooth", 2, 90, {}, (360, 480), "smooth"),
         ("444_q90_noise", 0, 90, {}, (241, 179), "noise"),
         ("420_q50_noise", 2, 50, {}, (37, 53), "noise"),
         ("420_q100_smooth", 2, 100, {}, (8, 8), "smooth"),
         ("444_q100_noise", 0, 100, {}, (37, 53), "noise"),
         ("420_optimize", 2, 90, {"optimize": True}, (241, 179), "smooth"),
         ("444_q50_smooth", 0, 50, {}, (360, 480), "smooth"),
         ("420_1080p", 2, 90, {}, (1080, 1920), "smooth"),
         ("444_8x8_noise", 0, 90, {}, (8, 8), "noise")]


def _case(name, sub, q, kw, hw, kind, seed):
    H, W = hw
    F = max(1, -(-100_000 // (H * W * 3)))
    imgs = _content(kind, F, H, W, seed)
    return [TW.encode(f, quality=q, subsampling=sub, **kw) for f in imgs]


@pytest.mark.parametrize("case", [c[0] for c in CASES])
def test_decode_islow_byte_identical_to_pillow(case):
    c = next(c for c in CASES if c[0] == case)
    jpegs = _case(*c, seed=len(case))
    v = _video(jpegs)
    vb = V.pack_jpeg([v], V.eval_plan([v.shape], len(jpegs), 1, 1, min(c[4])), dct_method="INTEGER_ACCURATE")
    flat, status = _decode(vb)
    assert not status.any()
    got = _frames_of(vb, flat)
    assert sum(g.nbytes for g in got) >= 100_000
    for g, j in zip(got, jpegs):
        want = TW.pil_decode(j)
        assert np.array_equal(g, want), f"{(g != want).sum()} of {g.size} bytes differ"


def test_ragged_batch_one_launch_per_stage():
    """Every case above in one batch (one launch per stage) == Pillow."""
    videos, jpeg_lists = [], []
    for i, c in enumerate(CASES):
        jpegs = _case(*c, seed=100 + i)[:3]
        jpeg_lists.append(jpegs)
        videos.append(_video(jpegs, c[0]))
    plans = V.eval_plan([v.shape for v in videos], 3, 1, 1, 8)
    vb = V.pack_jpeg(videos, plans, dct_method="INTEGER_ACCURATE")
    from x3d_tf_b200 import ops
    before = ops.Profiler.launches
    flat, status = _decode(vb)
    assert ops.Profiler.launches - before == 3 and not status.any()
    got = _frames_of(vb, flat)
    want = [TW.pil_decode(j) for js in jpeg_lists for j in js]
    assert sum(g.nbytes for g in got) >= 100_000
    assert all(np.array_equal(g, w) for g, w in zip(got, want))


def test_ifast_idct_equals_numpy_restatement():
    """INTEGER_FAST: the device IDCT of the device's coefficients == jpeg_oracle.idct_ifast, byte for
    byte (and the device's coefficients == the numpy entropy decoder's).  Parity with TF's own IFAST
    build is not pinned."""
    jpegs = [TW.encode(f, quality=q, subsampling=s) for f, q, s in
             zip(TW.video_frames(3, 200, 176, 4), (90, 50, 100), (2, 0, 2))]
    vb = V.pack_jpeg([_video(jpegs)], V.eval_plan([(3, 200, 176, 3)], 3, 1, 1, 176), dct_method="INTEGER_FAST")
    scratch = {}
    vb.encoded.decode("cuda", scratch)
    torch.cuda.synchronize()
    coef = scratch["jpeg_coef"][:vb.encoded.coef_blocks * 64].cpu().numpy().reshape(-1, 64)
    planes = scratch["jpeg_planes"][:vb.encoded.plane_bytes].cpu().numpy()
    recs = vb.encoded.frames.numpy().view(J.FRAME_DTYPE)
    total = 0
    for r, j in zip(recs, jpegs):
        h = J.parse_header(j)
        _, _, dims = O.grid(h)
        nb = sum(bw * bh for bw, bh in dims)
        c = coef[r["coef_off"]:r["coef_off"] + nb]
        assert np.array_equal(c, O.entropy(j))
        want = O.idct(j, c, "INTEGER_FAST")
        off = r["plane_off"]
        for p in want:
            got = planes[off:off + p.size].reshape(p.shape)
            assert np.array_equal(got, p)
            off += p.size
            total += p.size
    assert total >= 100_000


def _corrupt_cases():
    img = TW.video_frames(2, 240, 320, 9)
    good = TW.encode(img[0])
    fr = J.parse(good)
    seg = good[fr.seg_off:fr.seg_off + fr.seg_len]
    truncated = good[:fr.seg_off] + seg[:len(seg) // 3] + b"\xff\xd9"
    mid = len(seg) // 2
    while seg[mid - 1] == 0xFF or seg[mid + 7] == 0xFF:           # splice between whole bytes, not inside FF 00
        mid += 1
    bad_code = good[:fr.seg_off] + seg[:mid] + b"\xff\x00" * 8 + seg[mid + 8:] + b"\xff\xd9"
    return good, truncated, bad_code


def test_corrupt_frames_set_status_and_stay_in_bounds():
    good, truncated, bad_code = _corrupt_cases()
    v = _video([good, truncated, bad_code, good], "rec5")
    vb = V.pack_jpeg([v], V.eval_plan([v.shape], 4, 1, 1, 240), dct_method="INTEGER_ACCURATE")
    enc = vb.encoded
    G = 4096
    sizes = {"jpeg_coef": (enc.coef_blocks * 64, torch.int16), "jpeg_planes": (enc.plane_bytes, torch.uint8),
             "frames": (enc.out_bytes, torch.uint8), "jpeg_status": (enc.nframes, torch.int32)}
    scratch = {k: torch.full((n + G,), 0x5A, dtype=dt, device="cuda") for k, (n, dt) in sizes.items()}
    flat, status = enc.decode("cuda", scratch)
    torch.cuda.synchronize()
    st = status.cpu().numpy()
    assert st[0] == 0 and st[3] == 0
    assert st[1] == 3 and st[2] == 1                                  # short data, bad Huffman code
    for k, (n, _) in sizes.items():
        assert bool((scratch[k][n:] == 0x5A).all()), k                 # guards after every buffer
    got = _frames_of(vb, flat.cpu().numpy())
    assert np.array_equal(got[0], TW.pil_decode(good)) and np.array_equal(got[3], TW.pil_decode(good))
    with pytest.raises(ValueError, match=r"rec5 frame 1: JPEG decoding failed: premature end"):
        enc.check(st)


def _model(dtype, views=2):
    from x3d_tf_b200 import model as M
    M.reset_block_counters()
    cfg = get_config("X3D_XS", freeze=False)
    cfg.TEST.NUM_TEMPORAL_VIEWS, cfg.TEST.NUM_SPATIAL_CROPS = views, 1
    cfg.freeze()
    m = M.X3D(cfg, dtype=dtype)
    m.set_weights_dict(synthetic_weights(build_arch(cfg), seed=21))
    return m.compile(top_k=5), cfg


def test_predict_raises_on_corrupt_frame():
    m, cfg = _model("bfloat16")
    good, truncated, _ = _corrupt_cases()
    ok = _video([good] * 8, "recA")
    bad = _video([good, good, truncated, good, good, good, good, good], "recB")     # the views read frames 0, 2, 4, 6
    batches = [V.eval_batch([ok], cfg, "INTEGER_ACCURATE"), V.eval_batch([bad], cfg, "INTEGER_ACCURATE")]
    with pytest.raises(ValueError, match="recB frame 2"):
        list(m.predict(batches))


def _tf_videos(shapes, seed, q=90):
    """TFRecord videos of Pillow-encoded frames, and the same frames decoded by Pillow."""
    vids, dec = [], []
    for i, (F, H, W) in enumerate(shapes):
        jpegs = [TW.encode(f, quality=q) for f in TW.video_frames(F, H, W, seed + i)]
        vids.append(_video(jpegs, f"video{i}"))
        dec.append(np.stack([TW.pil_decode(j) for j in jpegs]))
    return vids, dec


@pytest.mark.parametrize("kind", ["eval", "train"])
def test_clips_equal_pack_of_pillow_frames(kind):
    vids, dec = _tf_videos([(20, 180, 240), (7, 100, 140), (13, 241, 179)], 3)
    shapes = [v.shape for v in vids]
    if kind == "eval":
        plan = V.eval_plan(shapes, 8, 2, 3, 96)
    else:
        plan = V.train_plan(shapes, 8, 5, (100, 130), 96, V.train_rng(4, 0))
    got = V.pack_jpeg(vids, plan, dct_method="INTEGER_ACCURATE").clips("cuda").cpu().numpy()
    want = V.pack(dec, plan).clips("cuda").cpu().numpy()
    assert got.nbytes >= 100_000 and np.array_equal(got, want)


@pytest.mark.parametrize("dtype", ["float32", "bfloat16"])
def test_evaluate_tfrecord_batches_equals_raw_batches(dtype):
    m, cfg = _model(dtype)
    rng = np.random.default_rng(2)
    tb, raw = [], []
    for i, shapes in enumerate([[(20, 120, 160), (9, 200, 170)], [(12, 181, 163), (16, 144, 256)]]):
        vids, dec = _tf_videos(shapes, 50 + 10 * i)
        labels = rng.integers(0, 400, size=len(shapes)).astype(np.int32)
        tb.append((V.eval_batch(vids, cfg, "INTEGER_ACCURATE"), labels))
        raw.append((V.eval_batch(dec, cfg), labels))
    assert m.evaluate(tb) == m.evaluate(raw)


def test_eval_driver_tfrecord(tmp_path):
    from x3d_tf_b200 import eval as E
    from x3d_tf_b200 import model as M
    cfg = get_config("X3D_XS")
    M.reset_block_counters()
    m = M.X3D(cfg, dtype="bfloat16")
    m.set_weights_dict(synthetic_weights(build_arch(cfg), seed=77))
    m.save_weights(str(tmp_path / "ckpt-1"))
    (tmp_path / "checkpoint").write_text('model_checkpoint_path: "ckpt-1"\nall_model_checkpoint_paths: "ckpt-1"\n')
    vids, dec = _tf_videos([(24, 180, 240), (9, 240, 180), (15, 161, 163)], 12)
    labels = [3, 200, 17]
    jp = [[v.jpeg(f) for f in range(v.shape[0])] for v in vids]
    TW.write_tfrecord(tmp_path / "b.tfrecord.gz", [TW.sequence_example(jp[2], labels[2])])
    TW.write_tfrecord(tmp_path / "a.tfrecord.gz", [TW.sequence_example(jp[i], labels[i]) for i in range(2)])
    vpb = max(cfg.TEST.BATCH_SIZE // (cfg.TEST.NUM_TEMPORAL_VIEWS * cfg.TEST.NUM_SPATIAL_CROPS), 1)
    want = m.compile().evaluate([(V.eval_batch(dec[i:i + vpb], cfg), np.asarray(labels[i:i + vpb], np.int32))
                                 for i in range(0, 3, vpb)])
    got = E.run(["--cfg", "X3D_XS", "--model_folder", str(tmp_path), "--test_file_pattern",
                 str(tmp_path / "*.tfrecord.gz"), "--tfrecord", "--dct_method", "INTEGER_ACCURATE"])
    assert got == want and got["videos"] == 3


def test_fit_on_tfrecord_batches_equals_trainer_on_raw_clips():
    from x3d_tf_b200 import model as M
    from x3d_tf_b200 import ops
    from x3d_tf_b200.training import X3DTrainer
    cfg = get_config("X3D_XS", freeze=False)
    cfg.NETWORK.DROPOUT_RATE = 0.0
    cfg.TEST.NUM_TEMPORAL_VIEWS, cfg.TEST.NUM_SPATIAL_CROPS = 1, 1
    cfg.freeze()
    W = synthetic_weights(build_arch(cfg), seed=5)
    rng = V.train_rng(31, 0)
    data, raw = [], []
    for step in range(2):
        vids, dec = _tf_videos([(30, 240, 320), (6, 200, 150)], 40 + step)
        plan = V.train_plan([v.shape for v in vids], cfg.DATA.TEMP_DURATION, cfg.DATA.FRAME_RATE,
                            cfg.DATA.TRAIN_JITTER_SCALES, cfg.DATA.TRAIN_CROP_SIZE, rng)
        labels = np.array([7 + step, 311 - step], np.int32)
        data.append((V.pack_jpeg(vids, plan, dct_method="INTEGER_ACCURATE"), labels))
        raw.append((V.pack(dec, plan), labels))
    M.reset_block_counters()
    m = M.X3D(cfg)
    m.set_weights_dict(W)
    hist = m.fit(data, epochs=1, lr_schedule=lambda e: 0.01)
    tr = X3DTrainer(cfg).load(W)
    tot = torch.zeros((), dtype=torch.float64, device="cuda")
    for vb, l in raw:
        x = ops.normalize_u8(vb.clips("cuda"), tuple(cfg.DATA.MEAN), tuple(cfg.DATA.STD), torch.float32)
        tot += tr.step(x, torch.from_numpy(l).cuda(), 0.01).double().mean()
    torch.cuda.synchronize()
    assert hist["loss"][0] == float(tot / 2)
    Wt, Wm = tr.weights(), m.named_variables()
    assert all(np.array_equal(Wt[k], Wm[k]) for k in Wt)
