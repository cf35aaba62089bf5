"""Motion-JPEG input without a GPU: the AVI reader (x3d_tf_b200/avi.py) on files written by
tests/avi_writer.py, the opt-in JPEG parsing of restart intervals, 4:2:2 and DHT-less frames, the
numpy restatement (tests/mjpeg_oracle.py) against a hand-worked row and Pillow, the x3d_jpeg_interval
layout probed with gcc, and pack_jpeg of mixed batches."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from tests import avi_writer as AW
from tests import mjpeg_oracle as M
from tests import tfrecord_writer as TW
from x3d_tf_b200 import avi
from x3d_tf_b200 import jpeg as J
from x3d_tf_b200 import video as V

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _jpegs(F=6, H=40, W=56, seed=0, **kw):
    return [TW.encode(f, **kw) for f in TW.video_frames(F, H, W, seed)]


def strip_dht(buf: bytes) -> bytes:
    """The frame without its DHT segments (what Motion-JPEG writers store)."""
    out, pos = bytearray(buf[:2]), 2
    while True:
        m, n = buf[pos + 1], (buf[pos + 2] << 8) | buf[pos + 3]
        if m != 0xC4:
            out += buf[pos:pos + 2 + n]
        pos += 2 + n
        if m == 0xDA:
            return bytes(out) + buf[pos:]


# ------------------------------------------------------------------------------------------- AVI
@pytest.mark.parametrize("kind", ["idx1", "no_idx1", "rec_junk_audio", "avix", "repeat", "audio_first",
                                  "lowercase_handler"])
def test_avi_reader_returns_every_frame_in_order(tmp_path, kind):
    frames = _jpegs(7, seed=1)
    kw = {"idx1": {}, "no_idx1": {"idx1": False}, "rec_junk_audio": {"rec": True, "junk": True, "audio": True},
          "avix": {"avix": True, "audio": True}, "repeat": {"repeat": (2, 3, 6)},
          "audio_first": {"audio_first": True, "junk": True},
          "lowercase_handler": {"handler": b"mjpg", "compression": b"mjpg"}}[kind]
    p = str(tmp_path / f"{kind}.avi")
    want = AW.write_avi(p, frames, 56, 40, **kw)
    v = avi.MJPEGVideo(p, label=5)
    assert v.shape == (7, 40, 56, 3) and v.label == 5 and v.name == p and v.mjpeg
    assert [v.jpeg(f) for f in range(7)] == want


def test_avi_chunk_table_is_cached(tmp_path, monkeypatch):
    p = str(tmp_path / "a.avi")
    AW.write_avi(p, _jpegs(3), 56, 40)
    avi.MJPEGVideo(p)
    calls = []
    monkeypatch.setattr(avi, "_walk", lambda path: calls.append(path))
    assert avi.MJPEGVideo(p).shape[0] == 3 and not calls


@pytest.mark.parametrize("kind,match", [("truncated", "truncated"), ("not_mjpeg", "not Motion-JPEG"),
                                        ("leading_empty", "first video chunk is empty"),
                                        ("no_video", "no video stream"), ("not_avi", "not an AVI")])
def test_avi_reader_errors_name_the_file(tmp_path, kind, match):
    frames = _jpegs(4)
    p = str(tmp_path / f"{kind}.avi")
    if kind == "truncated":
        AW.write_avi(p, frames, 56, 40, idx1=False, truncate=-len(frames[-1]) // 2)
    elif kind == "not_mjpeg":
        AW.write_avi(p, frames, 56, 40, handler=b"H264", compression=b"H264")
    elif kind == "leading_empty":
        AW.write_avi(p, frames, 56, 40, repeat=(0,))
    elif kind == "no_video":
        AW.write_avi(p, frames, 56, 40)
        raw = bytearray(open(p, "rb").read())
        i = raw.find(b"vids")
        raw[i:i + 4] = b"txts"
        open(p, "wb").write(bytes(raw))
    else:
        open(p, "wb").write(b"RIFX" + bytes(40))
    with pytest.raises(ValueError, match=match) as e:
        avi.MJPEGVideo(p)
    assert p in str(e.value)


# ----------------------------------------------------------------------------------------- parsing
def _iv_reference(buf, fr):
    """Interval ranges found by a plain byte walk (stuffing kept, fill bytes and marker dropped)."""
    out, start, i = [], fr.seg_off, fr.seg_off
    while True:
        if buf[i] == 0xFF and buf[i + 1] not in (0x00, 0xFF):
            end = i
            while buf[end - 1] == 0xFF:
                end -= 1
            out.append((start, end - start))
            if buf[i + 1] == 0xD9:
                return out
            start = i = i + 2
        else:
            i += 1


@pytest.mark.parametrize("kw", [{"restart_marker_blocks": 1}, {"restart_marker_rows": 1},
                                {"restart_marker_blocks": 7}, {"restart_marker_rows": 2, "subsampling": 1},
                                {"restart_marker_blocks": 3, "subsampling": 0}])
def test_restart_intervals_are_found(kw):
    img = TW.video_frames(1, 37, 91, 3)[0]
    buf = TW.encode(img, **kw)
    fr = J.parse(buf, mjpeg=True)
    h = fr.header
    assert h.ri > 0 and len(fr.intervals) == -(-h.mcus // h.ri)
    assert [tuple(map(int, r)) for r in fr.intervals] == _iv_reference(buf, fr)
    with pytest.raises(ValueError, match="restart interval"):
        J.parse(buf)


def _markers(buf, fr):
    return [int(o + n) for o, n in fr.intervals[:-1]]


def test_reordered_or_dropped_restart_marker_raises():
    buf = TW.encode(TW.video_frames(1, 128, 64, 4)[0], restart_marker_rows=1)
    fr = J.parse(buf, mjpeg=True)
    pos = _markers(buf, fr)
    swapped = bytearray(buf)
    swapped[pos[1] + 1], swapped[pos[2] + 1] = buf[pos[2] + 1], buf[pos[1] + 1]
    with pytest.raises(ValueError, match="RST1"):
        J.parse(bytes(swapped), mjpeg=True)
    dropped = buf[:pos[3]] + buf[pos[3] + 2:]
    with pytest.raises(ValueError, match="restart markers"):
        J.parse(dropped, mjpeg=True)


def test_dht_less_frame_gets_annex_k_tables():
    buf = TW.encode(TW.video_frames(1, 40, 56, 5)[0])
    bare = strip_dht(buf)
    assert b"\xff\xc4" not in bare[:J.parse(buf).seg_off]
    h, h0 = J.parse_header(bare, mjpeg=True), J.parse_header(buf)
    for a, b in zip(h.dc + h.ac, h0.dc + h0.ac):
        for f in ("maxcode", "valoffset", "lookup", "huffval"):
            assert np.array_equal(getattr(a, f), getattr(b, f))
    assert h.tables.tobytes() == h0.tables.tobytes()
    with pytest.raises(ValueError, match="Huffman table not defined"):
        J.parse(bare)


def test_422_only_under_the_opt_in():
    buf = TW.encode(TW.video_frames(1, 40, 56, 6)[0], subsampling=1)
    h = J.parse(buf, mjpeg=True).header
    assert (h.hs, h.vs, h.ri) == (2, 1, 0)
    with pytest.raises(ValueError, match="4:2:2"):
        J.parse(buf)


# ------------------------------------------------------------------------------------------ oracle
def test_h2v1_fancy_hand_worked_row():
    # samples 10 20 40 80 -> 10, (3*10+20+2)>>2=13, (3*20+10+1)>>2=17, (3*20+40+2)>>2=25, (3*40+20+1)>>2=35,
    # (3*40+80+2)>>2=50, (3*80+40+1)>>2=70, 80
    p = np.array([[10, 20, 40, 80]], np.uint8)
    assert M.h2v1_fancy(p, 1, 8).tolist() == [[10, 13, 17, 25, 35, 50, 70, 80]]
    assert M.h2v1_fancy(p, 1, 7).tolist() == [[10, 13, 17, 25, 35, 50, 70]]
    assert M.h2v1_fancy(p[:, :2], 1, 4).tolist() == [[10, 10, 20, 20]]             # box filter, width <= 2


ORACLE_CASES = [(sub, hw, kw) for sub in (2, 1) for hw in ((8, 8), (37, 53), (61, 90))
                for kw in ({}, {"restart_marker_blocks": 1}, {"restart_marker_rows": 1},
                           {"restart_marker_blocks": 5})] + [(0, (37, 53), {"restart_marker_blocks": 5})]


@pytest.mark.parametrize("sub,hw,kw", ORACLE_CASES)
def test_oracle_byte_identical_to_pillow(sub, hw, kw):
    img = TW.video_frames(1, *hw, 7 + sub)[0]
    buf = TW.encode(img, subsampling=sub, **kw)
    assert np.array_equal(M.decode(buf), TW.pil_decode(buf))
    bare = strip_dht(buf)
    assert np.array_equal(M.decode(bare), TW.pil_decode(bare))


# ---------------------------------------------------------------------------------------- packing
def test_interval_struct_layout_matches_header(tmp_path):
    from x3d_tf_b200 import _lib
    ct = _lib.JpegInterval
    lines = ['#include <stddef.h>', '#include <stdio.h>', '#include "x3d_b200.h"', 'int main(void) {',
             '  printf("size %zu\\n", sizeof(x3d_jpeg_interval));']
    lines += [f'  printf("{f} %zu\\n", offsetof(x3d_jpeg_interval, {f}));' for f, _ in ct._fields_]
    lines += ['  return 0;', '}']
    (tmp_path / "probe.c").write_text("\n".join(lines))
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(tmp_path / "probe.c")], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert int(got["size"]) == ctypes.sizeof(ct) == J.INTERVAL_DTYPE.itemsize
    for f, _ in ct._fields_:
        assert int(got[f]) == getattr(ct, f).offset, f


def test_pack_mixed_batch_orders_plain_frames_first(tmp_path):
    img = TW.video_frames(4, 48, 64, 8)
    kinds = [{"restart_marker_rows": 1}, {}, {"subsampling": 1, "restart_marker_blocks": 3}, {"subsampling": 1}]
    jpegs = [TW.encode(f, **kw) for f, kw in zip(img, kinds)]
    p = str(tmp_path / "mixed.avi")
    AW.write_avi(p, jpegs, 64, 48)
    v = avi.MJPEGVideo(p)
    vb = V.pack_jpeg([v], V.eval_plan([v.shape], 4, 1, 1, 48), pin=False)
    enc = vb.encoded
    recs = enc.frames.numpy().view(J.FRAME_DTYPE)
    assert enc.nplain == 2 and enc.nframes == 4
    assert [n.split()[-1] for n in enc.names] == ["1", "3", "0", "2"]
    assert list(recs["status"]) == [0, 1, 2, 3]
    iv = enc.intervals.numpy().view(J.INTERVAL_DTYPE)
    frs = [J.parse(jpegs[0], mjpeg=True), J.parse(jpegs[2], mjpeg=True)]
    assert enc.nintervals == len(iv) == sum(len(f.intervals) for f in frs)
    for fidx, fr in zip((2, 3), frs):
        mine = iv[iv["frame"] == fidx]
        h = fr.header
        assert list(mine["len"]) == list(fr.intervals[:, 1])
        assert list(mine["off"] - recs["seg_off"][fidx]) == list(fr.intervals[:, 0] - fr.seg_off)
        assert list(mine["mcu0"]) == list(range(0, h.mcus, h.ri)) and mine["nmcu"].sum() == h.mcus
    # frame_off points each output frame at its own decode, whatever the order
    outs = recs["out_off"]
    assert list(vb.frame_off.numpy()) == [outs[2], outs[0], outs[3], outs[1]]


def test_tfrecord_style_batch_has_no_intervals():
    jpegs = _jpegs(3)
    from x3d_tf_b200 import tfrecord as R
    v = R.parse_sequence_example(TW.sequence_example(jpegs, 0), "rec")
    enc = V.pack_jpeg([v], V.eval_plan([v.shape], 3, 1, 1, 40), pin=False).encoded
    assert enc.nintervals == 0 and enc.nplain is None and enc.intervals.numel() == 0


def test_drivers_reject_two_input_kinds():
    from x3d_tf_b200 import eval as E
    from x3d_tf_b200 import train as T
    with pytest.raises(SystemExit):
        E.run(["--cfg", "X3D_XS", "--model_folder", ".", "--test_file_pattern", "x", "--mjpeg_videos", "--tfrecord"])
    with pytest.raises(SystemExit):
        T.run(["--config", "X3D_XS", "--model_dir", "/nonexistent", "--train_file_pattern", "x", "--mjpeg_videos",
               "--decoded_videos"])
