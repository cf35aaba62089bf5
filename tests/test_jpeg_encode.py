"""Encoder side of the JPEG / TFRecord format without a GPU: quantisation tables and headers against
Pillow (libjpeg-turbo), the numpy restatement of the encoder (tests/jpeg_enc_oracle.py) against
Pillow byte for byte and against hand-worked blocks, the record writer against google.protobuf and
the reader, the encoder's C-ABI structs probed with gcc, and argument checks of the entry points."""
import ctypes
import gzip
import io
import os
import subprocess

import numpy as np
import pytest

from tests import jpeg_enc_oracle as E
from tests import tfrecord_writer as TW
from x3d_tf_b200 import jpeg as J
from x3d_tf_b200 import tfrecord as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SUB = {"420": 2, "444": 0}


def _pil(img, q, chroma):
    return TW.encode(img, quality=q, subsampling=SUB[chroma], dpi=(300, 300))


def canonical(rec: bytes) -> bytes:
    """google.protobuf's deterministic serialisation of a SequenceExample (map entries in key order;
    its default order is not stable from one process to the next)."""
    cls = TW._classes()["SequenceExample"]
    return cls.FromString(rec).SerializeToString(deterministic=True)


@pytest.mark.parametrize("q", [10, 50, 75, 90, 95, 100])
@pytest.mark.parametrize("chroma", ["420", "444"])
@pytest.mark.parametrize("hw", [(1, 1), (8, 8), (17, 33), (360, 480), (1080, 1920)])
def test_header_and_quant_tables_equal_pillow(q, chroma, hw):
    H, W = hw
    img = np.full((H, W, 3), 77, np.uint8)
    want = _pil(img, q, chroma)
    hdr = J.encoder_header(H, W, q, chroma)
    assert want[:len(hdr)] == hdr
    h = J.parse_header(want)                       # the decoder's parse: natural order
    assert np.array_equal(h.qtables[:2], J.quant_tables(q))
    assert (h.hs, h.vs) == J.CHROMA[chroma] and h.scan_off == len(hdr)


def test_quant_tables_scaling():
    """jcparam.c: q 50 is the Annex K table itself; q 100 all ones; q 10 clamped to 255 (force_baseline)."""
    assert np.array_equal(J.quant_tables(50), J.STD_QUANT)
    assert (J.quant_tables(100) == 1).all()
    t = J.quant_tables(10)
    assert t.max() == 255 and t[0, 0] == 80 and t[1, 63] == 255


def test_huffman_codes_annex_k():
    """ITU T.81 table K.3 (luminance DC) and K.5 (luminance AC) entries."""
    co, si = J.huff_codes(*J.STD_HUFF[0])
    assert [(int(si[s]), int(co[s])) for s in (0, 1, 5, 11)] == [(2, 0b00), (3, 0b010), (3, 0b110), (9, 0b111111110)]
    co, si = J.huff_codes(*J.STD_HUFF[1])
    assert (int(si[0x00]), int(co[0x00])) == (4, 0b1010)            # EOB
    assert (int(si[0xF0]), int(co[0xF0])) == (11, 0b11111111001)    # ZRL
    assert (int(si[0x01]), int(co[0x01])) == (2, 0b00)


def test_bad_arguments():
    with pytest.raises(ValueError, match="subsampling"):
        J.encoder_header(8, 8, 90, "422")
    with pytest.raises(ValueError, match="65535"):
        J.encoder_header(70000, 8)
    with pytest.raises(ValueError, match="chroma"):
        J.encode_frames(np.zeros((1, 8, 8, 3), np.uint8), 90, "422")
    with pytest.raises(ValueError, match="quality"):
        J.encode_frames(np.zeros((1, 8, 8, 3), np.uint8), 0)


def test_fdct_hand_worked_block():
    """A block of constant 138 (10 above the level shift): only DC, 64 * 10 = 640 (jpeg_fdct_islow's
    output is 8x the orthonormal DCT: 8 * 80); quantised by q 16 (divisor 128) to 5.  A horizontal ramp
    0..7 above 128: DC 8 * 28 = 224, the first horizontal frequency worked by hand below, and every
    vertical frequency 0 because the block is constant down its columns."""
    blk = np.full((1, 64), 138)
    d = E.fdct_islow(blk)
    assert d[0, 0] == 640 and not d[0, 1:].any()
    assert E.quantize(d, np.full(64, 16))[0, 0] == 5
    ramp = np.tile(np.arange(128, 136), 8)[None]
    d = E.fdct_islow(ramp).reshape(8, 8)
    assert d[0, 0] == 224 and not d[1:].any()
    # pass 1 on the row 128..135 - 128 = 0..7: tmp7 = -7, tmp5 + tmp7 = -10, tmp4 + tmp7 = -8,
    # tmp4 + tmp6 = -6; z5 = (-6 - 10) * 9633; out[1] = DESCALE(tmp7 * 12299 + z1 + z4, CONST_BITS -
    # PASS1_BITS = 11) with z1 = -8 * -7373, z4 = -10 * -3196 + z5: -148253 / 2048 -> -73.  Pass 2 on 8
    # equal rows keeps only its DC term: DESCALE(8 * -73, PASS1_BITS) = -146 (the orthonormal DCT's
    # -18.2, times 8)
    z5 = (-6 - 10) * 9633
    out1 = (-7 * 12299 + (-8 * -7373) + (-10 * -3196 + z5) + (1 << 10)) >> 11
    assert out1 == -73 and d[0, 1] == (8 * out1 + 2) >> 2 == -146
    assert E.quantize(d.reshape(1, 64), np.full(64, 11))[0, 1] == -2          # divisor 88: -146 / 88 = -1.66


def test_quantize_by_reciprocal():
    """jcdctmgr.c compute_reciprocal / quantize, worked by hand: q 8 (divisor 64, a power of two):
    recip 2^21 / 64 halved to 32768, corr 32, shift 21; q 3 (divisor 24): 2^20 / 24 = 43690 rem 16 >
    12, so recip 43691, corr 12, shift 20.  Over every quantiser 1..255 and every |x| the FDCT can
    produce (< 9000), the result equals round-half-up division, floor((|x| + d/2) / d), with the sign
    of x: checked here rather than assumed."""
    r, c, s = E.reciprocals(np.array([8, 3]))
    assert (r.tolist(), c.tolist(), (s + 16).tolist()) == ([32768, 43691], [32, 12], [21, 20])
    assert E.quantize(np.array([20, 32, -32, 31]), np.full(4, 8)).tolist() == [0, 1, -1, 0]
    assert E.quantize(np.array([12, 11, -12]), np.full(3, 3)).tolist() == [1, 0, -1]
    x = np.arange(-9000, 9001)
    for q in range(1, 256):
        d = 8 * q
        want = np.sign(x) * ((np.abs(x) + d // 2) // d)
        assert np.array_equal(E.quantize(x, np.full(x.size, q)), want), q


def _content(kind, H, W, seed):
    if kind == "noise":
        return np.random.default_rng(seed).integers(0, 256, (H, W, 3), dtype=np.uint8)
    return TW.video_frames(1, H, W, seed, noise=2.0)[0]


@pytest.mark.parametrize("hw", [(1, 1), (7, 9), (17, 33), (31, 47), (360, 480)])
@pytest.mark.parametrize("kind", ["noise", "smooth"])
@pytest.mark.parametrize("chroma", ["420", "444"])
def test_oracle_byte_identical_to_pillow(hw, kind, chroma):
    H, W = hw
    img = _content(kind, H, W, H * 31 + W)
    qs = (90,) if H * W > 10_000 else (10, 50, 90, 100)
    for q in qs:
        assert E.encode(img, q, chroma) == _pil(img, q, chroma), q


def test_oracle_coefficients_decode_back():
    """The oracle's coefficients are those the existing numpy decoder reads from Pillow's file."""
    from tests import jpeg_oracle as D
    for hw, chroma in (((17, 33), "420"), ((31, 47), "444"), ((9, 40), "420")):
        img = _content("noise", *hw, 3)
        assert np.array_equal(E.coefficients(img, 90, chroma), D.entropy(_pil(img, 90, chroma)))


def test_records_equal_protobuf_and_read_back(tmp_path):
    rng = np.random.default_rng(0)
    vids = []
    for i, F in enumerate((1, 5, 12)):
        frames = [_pil(f, 90, "420") for f in TW.video_frames(F, 24 + i, 40, i)]
        vids.append((frames, int(rng.integers(0, 400))))
    recs = [R.serialize_sequence_example(f, lab) for f, lab in vids]
    assert recs == [canonical(TW.sequence_example(f, lab)) for f, lab in vids]
    p = str(tmp_path / "x.tfrecord.gz")
    R.write_records(p, recs)
    assert list(R.read_records(p)) == recs
    assert gzip.open(p).read() == TW.frame_records(recs)
    for (frames, lab), v in zip(vids, R.read_videos(p)):
        assert v.label == lab and [v.jpeg(f) for f in range(len(v))] == frames
    # a flipped byte inside the first record's data is caught by its CRC
    raw = bytearray(gzip.open(p).read())
    raw[40] ^= 1
    bad = str(tmp_path / "bad.tfrecord.gz")
    with gzip.open(bad, "wb") as f:
        f.write(bytes(raw))
    with pytest.raises(ValueError, match="record 0: data CRC mismatch"):
        list(R.read_records(bad))


def test_gzip_level_changes_only_compression(tmp_path):
    recs = [R.serialize_sequence_example([b"\xff\xd8" + bytes(range(256)) * 4], 1)]
    for level in (0, 1, 9):
        p = str(tmp_path / f"l{level}.gz")
        R.write_records(p, recs, level)
        assert list(R.read_records(p)) == recs


def test_encoder_struct_layouts_match_header(tmp_path):
    from x3d_tf_b200 import _lib
    structs = {"x3d_jpeg_enc_frame": _lib.JpegEncFrame, "x3d_jpeg_enc_tables": _lib.JpegEncTables,
               "x3d_jpeg_enc_result": _lib.JpegEncResult}
    lines = ['#include <stddef.h>', '#include <stdio.h>', '#include "x3d_b200.h"', 'int main(void) {']
    for cname, ct in structs.items():
        lines.append(f'  printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in ct._fields_:
            lines.append(f'  printf("{cname}.{fname} %zu\\n", offsetof({cname}, {fname}));')
    lines.append('  printf("overflow %d\\n", X3D_JPEG_OVERFLOW);')
    lines += ['  return 0;', '}']
    src = tmp_path / "probe.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    for cname, ct in structs.items():
        assert int(got[cname]) == ctypes.sizeof(ct), cname
        for fname, _ in ct._fields_:
            assert int(got[f"{cname}.{fname}"]) == getattr(ct, fname).offset, f"{cname}.{fname}"
    assert int(got["overflow"]) == _lib.X3D_JPEG_OVERFLOW
    assert J.enc_tables(90).nbytes == ctypes.sizeof(_lib.JpegEncTables)


def test_entry_points_reject_bad_arguments_without_gpu():
    from x3d_tf_b200 import _lib
    from x3d_tf_b200 import build as b
    b.build()
    h = _lib.lib()
    assert h.x3d_jpeg_fdct(None, None, None, 1, 1, None, None) == -1 and b"null" in h.x3d_last_error()
    assert h.x3d_jpeg_enc_bits(1, 8, 2, 0, 8, 8, 4, None) == -1 and b"nframes" in h.x3d_last_error()
    assert h.x3d_jpeg_enc_emit(1, 8, 2, 1, 1, 8, 8, 3, None) == -1 and b"aligned" in h.x3d_last_error()
    assert h.x3d_jpeg_enc_stuff(4, 8, 1, 8, 1, -1, None) == -1 and b"out_cap" in h.x3d_last_error()


def test_driver_bounds_the_shards_waiting_for_the_pool(tmp_path, monkeypatch):
    """create_tfrecords with a writer much slower than the encoder: at most 2 x --threads encoded
    shards are ever held (waiting for or inside the pool), every shard is still written, in order.
    The device encoder is replaced by a stand-in, so no GPU is needed."""
    import threading
    import time
    import torch
    from x3d_tf_b200 import create_tfrecords as C
    lock = threading.Lock()
    state = {"encoded": 0, "written": 0, "max_held": 0}
    written = []

    def fake_encode(frames, quality, chroma, scratch):
        with lock:
            state["encoded"] += 1
            state["max_held"] = max(state["max_held"], state["encoded"] - state["written"])
        return [b"\xff\xd8frame\xff\xd9"] * len(frames)

    def slow_write(path, jpegs, labels, level):
        time.sleep(0.05)
        with lock:
            state["written"] += 1
            written.append(os.path.basename(path))
        return 0.0, 0.05, 0

    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    monkeypatch.setattr(C.J, "encode_frames", fake_encode)
    monkeypatch.setattr(C, "_write", slow_write)
    monkeypatch.setattr(C, "load_video", lambda p: np.zeros((3, 8, 8, 3), np.uint8))
    (tmp_path / "list.txt").write_text("".join(f"v{i}.npy {i}\n" for i in range(12)))
    for threads in (1, 3):
        state.update(encoded=0, written=0, max_held=0)
        written.clear()
        out = C.run(["--file_list", str(tmp_path / "list.txt"), "--out_dir", str(tmp_path / f"o{threads}"),
                     "--videos_per_file", "1", "--threads", str(threads)])
        assert out["files"] == 12 and out["frames"] == 36 and state["written"] == 12
        # held = the shard being encoded + those submitted and not yet written
        assert state["max_held"] <= 2 * threads + 1, (threads, state)
        if threads == 1:
            assert written == [C.shard_name("", i, 12) for i in range(12)]
