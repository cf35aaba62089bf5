"""The device JPEG encoder (x3d_jpeg_fdct / _enc_bits / _enc_emit / _enc_stuff, jpeg.encode_frames)
against Pillow (libjpeg-turbo) and the numpy restatement (tests/jpeg_enc_oracle.py), its output
through the device decoder, and the TFRecord writing driver through the eval driver."""
import numpy as np
import pytest
import torch

from tests import jpeg_enc_oracle as E
from tests import tfrecord_writer as TW
from tests.test_jpeg_encode import canonical
from x3d_tf_b200 import jpeg as J
from x3d_tf_b200 import tfrecord as R
from x3d_tf_b200 import video as V

pytestmark = pytest.mark.gpu

SUB = {"420": 2, "444": 0}
SIZES = [(8, 8), (1, 1), (7, 9), (17, 33), (31, 47), (241, 179), (360, 480), (1080, 1920)]


def _content(kind, F, H, W, seed):
    if kind == "noise":
        return np.random.default_rng(seed).integers(0, 256, (F, H, W, 3), dtype=np.uint8)
    return TW.video_frames(F, H, W, seed, noise=2.0)


def _pil(img, q, chroma):
    return TW.encode(img, quality=q, subsampling=SUB[chroma], dpi=(300, 300))


def _first_diff(a, b):
    n = min(len(a), len(b))
    d = np.flatnonzero(np.frombuffer(a[:n], np.uint8) != np.frombuffer(b[:n], np.uint8))
    return int(d[0]) if d.size else n


@pytest.mark.parametrize("q", [10, 90, 100])
@pytest.mark.parametrize("chroma", ["420", "444"])
@pytest.mark.parametrize("kind", ["noise", "smooth"])
def test_encode_byte_identical_to_pillow(q, chroma, kind):
    """Every size, from device memory, whole file == Pillow's."""
    for i, (H, W) in enumerate(SIZES):
        F = 1 if H * W > 200_000 else 3
        imgs = _content(kind, F, H, W, 10 * i + q)
        got = J.encode_frames(torch.from_numpy(imgs).cuda(), q, chroma)
        for f, g in enumerate(got):
            want = _pil(imgs[f], q, chroma)
            assert g == want, f"{H}x{W} frame {f}: {len(g)} vs {len(want)} bytes, first difference at {_first_diff(g, want)}"


def test_ragged_batch_one_launch_per_stage():
    """Every size, both contents, from pinned host memory, in one call: four stage calls, == Pillow."""
    from x3d_tf_b200 import ops
    imgs = [_content(kind, 1, H, W, i)[0] for i, (H, W) in enumerate(SIZES) for kind in ("noise", "smooth")]
    frames = [torch.from_numpy(f).pin_memory() for f in imgs]
    before = ops.Profiler.launches
    got = J.encode_frames(frames, 100, "420")
    assert ops.Profiler.launches - before == 4
    for f, g in zip(imgs, got):
        assert g == _pil(f, 100, "420"), f.shape


@pytest.mark.parametrize("chroma", ["420", "444"])
def test_stage_a_coefficients_equal_oracle(chroma):
    """Coefficients (dummy blocks included) == jpeg_enc_oracle.coefficients, in the decoder's layout."""
    imgs = [_content("noise", 1, H, W, 7)[0] for H, W in [(17, 33), (31, 47), (241, 179), (360, 480)]]
    scratch = {}
    J.encode_frames(imgs, 90, chroma, scratch)
    coef = scratch["enc_coef_group"].cpu().numpy().reshape(-1, 64)
    recs = scratch["enc_frames"].cpu().numpy().view(J.ENC_FRAME_DTYPE)
    for img, r in zip(imgs, recs):
        want = E.coefficients(img, 90, chroma)
        got = coef[r["coef_off"]:r["coef_off"] + len(want)]
        assert np.array_equal(got, want), f"{img.shape}: {(got != want).sum()} coefficients differ"


def test_device_decode_of_device_output_equals_pillow_decode():
    imgs = _content("smooth", 4, 241, 179, 5)
    jpegs = J.encode_frames(imgs, 90, "420")
    v = R.parse_sequence_example(R.serialize_sequence_example(jpegs, 0), "enc")
    vb = V.pack_jpeg([v], V.eval_plan([v.shape], 4, 1, 1, 179), dct_method="INTEGER_ACCURATE")
    flat, status = vb.encoded.decode("cuda", {})
    flat, status = flat.cpu().numpy(), status.cpu().numpy()
    assert not status.any()
    recs = vb.encoded.frames.numpy().view(J.FRAME_DTYPE)
    for r, j in zip(recs, jpegs):
        got = flat[r["out_off"]:r["out_off"] + r["H"] * r["W"] * 3].reshape(r["H"], r["W"], 3)
        assert np.array_equal(got, TW.pil_decode(j))


def test_driver_then_eval_tfrecord_equals_decoded_videos(tmp_path):
    """create_tfrecords on a .npy list, then eval.py --tfrecord on its files == eval.py
    --decoded_videos on the Pillow round trip of the same frames; the records (decompressed) equal
    those of a writer built on Pillow and google.protobuf."""
    import glob
    from x3d_tf_b200 import create_tfrecords as C
    from x3d_tf_b200 import eval as EV
    from x3d_tf_b200 import model as M
    from x3d_tf_b200.arch import build_arch
    from x3d_tf_b200.config import get_config
    from x3d_tf_b200.synth import synthetic_weights
    cfg = get_config("X3D_XS")
    M.reset_block_counters()
    m = M.X3D(cfg, dtype="bfloat16")
    m.set_weights_dict(synthetic_weights(build_arch(cfg), seed=78))
    m.save_weights(str(tmp_path / "ckpt-1"))
    (tmp_path / "checkpoint").write_text('model_checkpoint_path: "ckpt-1"\nall_model_checkpoint_paths: "ckpt-1"\n')
    shapes, labels = [(24, 180, 240), (30, 241, 179), (15, 161, 163)], [3, 200, 17]
    lines, rt_lines, want_recs = [], [], []
    for i, ((F, H, W), lab) in enumerate(zip(shapes, labels)):
        v = TW.video_frames(F, H, W, 40 + i)
        np.save(tmp_path / f"v{i}.npy", v)
        lines.append(f"v{i}.npy {lab}")
        K = min(F, 20)
        jp = [_pil(f, 90, "420") for f in v[:K]]
        want_recs.append(TW.sequence_example(jp, lab))
        np.save(tmp_path / f"rt{i}.npy", np.stack([TW.pil_decode(j) for j in jp]))
        rt_lines.append(f"rt{i}.npy {lab}")
    (tmp_path / "videos.txt").write_text("\n".join(lines) + "\n")
    (tmp_path / "rt.txt").write_text("\n".join(rt_lines) + "\n")
    out = tmp_path / "records"
    summary = C.run(["--file_list", str(tmp_path / "videos.txt"), "--out_dir", str(out), "--videos_per_file", "2",
                     "--max_frames", "20", "--threads", "2"])
    assert summary["videos"] == 3 and summary["files"] == 2 and summary["frames"] == 55
    files = sorted(glob.glob(str(out / "*.tfrecord.gz")))
    assert [r for f in files for r in R.read_records(f)] == [canonical(r) for r in want_recs]
    common = ["--cfg", "X3D_XS", "--model_folder", str(tmp_path)]
    got = EV.run(common + ["--test_file_pattern", str(out / "*.tfrecord.gz"), "--tfrecord",
                           "--dct_method", "INTEGER_ACCURATE"])
    want = EV.run(common + ["--test_file_pattern", str(tmp_path / "rt.txt"), "--decoded_videos"])
    assert got == want and got["videos"] == 3


def _overflow_setup(imgs):
    """The device buffers of one encode_frames call, for the stages to be run again by hand."""
    scratch = {}
    J.encode_frames(imgs, 90, "420", scratch)
    recs = scratch["enc_frames"].cpu().numpy().view(J.ENC_FRAME_DTYPE).copy()
    tables = torch.from_numpy(J.enc_tables(90).reshape(1).view(np.uint8).copy()).cuda()
    nblocks = int(recs["coef_off"][-1]) + J.enc_blocks(*imgs[-1].shape[:2], 2)
    return scratch["enc_coef_group"], recs, tables, nblocks


def _res(res):
    return res.cpu().numpy().view(J.ENC_RESULT_DTYPE)


def test_word_cap_overflow_sets_status_and_writes_nothing():
    """A frame whose bits exceed its word_cap gets X3D_JPEG_OVERFLOW from x3d_jpeg_enc_bits; the emit and
    stuffing stages then write none of its words or bytes and leave its len as it was.  The other
    frame of the batch is encoded as usual."""
    from x3d_tf_b200 import _lib, ops
    imgs = [_content("noise", 1, 16, 16, 1)[0], _content("noise", 1, 64, 64, 2)[0]]
    coef, recs, tables, nblocks = _overflow_setup(imgs)
    recs["word_cap"][1] = 4                                   # far fewer words than 64x64 noise needs
    frames = torch.from_numpy(recs.view(np.uint8).copy()).cuda()
    boff = torch.empty(nblocks, dtype=torch.int64, device="cuda")
    res = torch.full((2 * J.ENC_RESULT_DTYPE.itemsize,), 0xAB, dtype=torch.uint8, device="cuda")
    words = torch.full((int(recs["word_off"][1] + recs["word_cap"][1]),), 0x5A5A5A5A, dtype=torch.int32, device="cuda")
    out = torch.full((1 << 16,), 0xEE, dtype=torch.uint8, device="cuda")
    ops.jpeg_enc_bits(coef, frames, tables, 2, boff, res, words)
    ops.jpeg_enc_emit(coef, frames, tables, 2, J.enc_blocks(64, 64, 2), boff, res, words)
    ops.jpeg_enc_stuff(words, frames, 2, res, out)
    r = _res(res)
    assert r["status"].tolist() == [0, _lib.X3D_JPEG_OVERFLOW]
    assert r["bits"][1] > 32 * 4                               # the real bit count is still reported
    assert r["len"][1] == np.full(1, 0xAB, np.uint8).repeat(8).view(np.int64)[0]
    w = words.cpu().numpy()
    assert (w[int(recs["word_off"][1]):] == 0x5A5A5A5A).all()
    o = out.cpu().numpy()
    seg0 = _pil(imgs[0], 90, "420")[len(J.encoder_header(16, 16)):-2]
    assert o[r["out_off"][0]:r["out_off"][0] + r["len"][0]].tobytes() == seg0
    assert (o[r["out_off"][1]:] == 0xEE).all()


def test_out_cap_overflow_sets_status_and_writes_nothing():
    """A frame whose output region ends past out_cap gets X3D_JPEG_OVERFLOW from x3d_jpeg_enc_stuff and
    none of its bytes are written; the frame before it, which fits, is written."""
    from x3d_tf_b200 import _lib, ops
    imgs = [_content("noise", 1, 16, 16, 1)[0], _content("noise", 1, 64, 64, 2)[0]]
    coef, recs, tables, nblocks = _overflow_setup(imgs)
    frames = torch.from_numpy(recs.view(np.uint8).copy()).cuda()
    boff = torch.empty(nblocks, dtype=torch.int64, device="cuda")
    res = torch.full((2 * J.ENC_RESULT_DTYPE.itemsize,), 0xAB, dtype=torch.uint8, device="cuda")
    words = torch.empty(int(recs["word_off"][1] + recs["word_cap"][1]), dtype=torch.int32, device="cuda")
    ops.jpeg_enc_bits(coef, frames, tables, 2, boff, res, words)
    ops.jpeg_enc_emit(coef, frames, tables, 2, J.enc_blocks(64, 64, 2), boff, res, words)
    bits = _res(res)["bits"]
    bound0 = 2 * ((int(bits[0]) + 7) // 8)
    cap = bound0 + (int(bits[1]) + 7) // 8                    # frame 1's region needs 2x its bytes
    buf = torch.full((cap + 64,), 0xEE, dtype=torch.uint8, device="cuda")
    ops.jpeg_enc_stuff(words, frames, 2, res, buf[:cap])
    r = _res(res)
    assert r["status"].tolist() == [0, _lib.X3D_JPEG_OVERFLOW]
    assert r["out_off"].tolist() == [0, bound0]
    assert r["len"][1] == np.full(1, 0xAB, np.uint8).repeat(8).view(np.int64)[0]
    o = buf.cpu().numpy()
    assert o[:r["len"][0]].tobytes() == _pil(imgs[0], 90, "420")[len(J.encoder_header(16, 16)):-2]
    assert (o[bound0:] == 0xEE).all()
