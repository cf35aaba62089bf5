"""TFRecord / SequenceExample reading, JPEG header parsing and rejection, pack_jpeg, the C layout of
x3d_jpeg_frame / x3d_jpeg_tables, and the numpy decoder restatement the GPU tests compare against
(tests/jpeg_oracle.py).  No GPU."""
import ctypes
import gzip
import os
import subprocess

import numpy as np
import pytest

from tests import jpeg_oracle as O
from tests import tfrecord_writer as TW
from x3d_tf_b200 import jpeg as J
from x3d_tf_b200 import tfrecord as R
from x3d_tf_b200 import video as V

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _frames(F=4, H=40, W=56, seed=0, **kw):
    return [TW.encode(f, **kw) for f in TW.video_frames(F, H, W, seed)]


# ------------------------------------------------------------------------------------------ TFRecord
def test_tfrecord_round_trip(tmp_path):
    recs = [TW.sequence_example(_frames(3, seed=i), label=i) for i in range(3)]
    p = tmp_path / "a.tfrecord.gz"
    TW.write_tfrecord(p, recs)
    assert [bytes(r) for r in R.read_records(str(p))] == recs
    vids = list(R.read_videos(str(p)))
    assert [v.label for v in vids] == [0, 1, 2] and all(v.shape == (3, 40, 56, 3) for v in vids)


@pytest.mark.parametrize("where", ["data", "length_crc", "truncated", "gzip"])
def test_tfrecord_corruption_raises(tmp_path, where):
    recs = [TW.sequence_example(_frames(2), label=1), TW.sequence_example(_frames(2, seed=1), label=2)]
    raw = bytearray(TW.frame_records(recs))
    p = tmp_path / "bad.tfrecord.gz"
    second = len(recs[0]) + 16                                   # start of record 1
    if where == "data":
        raw[second + 12 + 40] ^= 0x10
    elif where == "length_crc":
        raw[second + 9] ^= 0x01
    if where == "truncated":
        raw = raw[:second + 12 + 100]
    data = gzip.compress(bytes(raw))
    if where == "gzip":
        data = data[:10] + bytes(b ^ 0x5A for b in data[10:60]) + data[60:]
    p.write_bytes(data)
    with pytest.raises(ValueError) as e:
        list(R.read_records(str(p)))
    assert str(p) in str(e.value) and "record" in str(e.value)
    if where != "gzip":
        assert "record 1" in str(e.value)


@pytest.mark.parametrize("packed", [True, False])
def test_sequence_example_parses(packed):
    fr = _frames(5)
    v = R.parse_sequence_example(TW.sequence_example(fr, label=42, packed=packed))
    assert v.label == 42 and v.shape == (5, 40, 56, 3) and v.dtype == np.uint8
    assert [v.jpeg(i) for i in range(5)] == fr


def test_sequence_example_mismatch_and_missing_keys():
    fr = _frames(3)
    with pytest.raises(ValueError, match="num_frames"):
        R.parse_sequence_example(TW.sequence_example(fr, 1, num_frames=4))
    for key in ("video/num_frames", "video/class/label", "video"):
        with pytest.raises(ValueError, match="missing"):
            R.parse_sequence_example(TW.sequence_example(fr, 1, drop=(key,)))


# ------------------------------------------------------------------------------------------- headers
@pytest.mark.parametrize("sub,q", [(2, 90), (0, 90), (2, 50), (0, 100)])
def test_header_matches_pillow(sub, q):
    from PIL import Image
    import io
    img = TW.video_frames(1, 37, 53, 3)[0]
    buf = TW.encode(img, quality=q, subsampling=sub)
    h = J.parse_header(buf)
    im = Image.open(io.BytesIO(buf))
    assert (h.H, h.W) == (37, 53)
    assert [(c[1], c[2]) for c in im.layer] == [(h.hs, h.vs), (1, 1), (1, 1)]
    assert h.hs == (2 if sub == 2 else 1)
    for i, t in im.quantization.items():
        assert np.array_equal(h.qtables[i], np.asarray(t))
    assert [c[3] for c in im.layer] == list(h.comp_q)
    fr = J.parse(buf)
    assert fr.seg_off == h.scan_off and buf[fr.seg_off + fr.seg_len:] == b"\xff\xd9"


def test_header_cache_shares_tables():
    a, b = _frames(2)
    assert J.parse_header(a) is J.parse_header(b)


def test_derived_tables_annex_k():
    """ITU T.81 Annex K.3 table K.3 (luminance DC) and K.5 (luminance AC)."""
    dc_bits = [0, 0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0]
    t = J.derive_table(dc_bits, bytes(range(12)), True)
    # codes: 00 -> 0 (len 2), 010..110 -> 1..5 (len 3), 1110 -> 6, 11110 -> 7, ..., 111111110 -> 11 (len 9)
    assert t.lookup[0b00000000] == (2 << 8) | 0 and t.lookup[0b00111111] == (2 << 8) | 0
    assert t.lookup[0b01000000] == (3 << 8) | 1 and t.lookup[0b11000000] == (3 << 8) | 5
    assert t.lookup[0b11100000] == (4 << 8) | 6 and t.lookup[0b11111110] == (8 << 8) | 10
    assert t.lookup[0b11111111] == 9 << 8                                  # code 11 is 9 bits long
    assert t.maxcode[2] == 0 and t.maxcode[3] == 6 and t.maxcode[9] == 0b111111110 and t.maxcode[1] == -1
    assert t.valoffset[3] == 1 - 2 and t.valoffset[9] == 11 - 0b111111110 and t.maxcode[17] == 0xFFFFF
    ac_bits = [0, 0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7D]
    ac_vals = bytes([0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07])
    t = J.derive_table(ac_bits, ac_vals + bytes(162 - len(ac_vals)), False)
    assert t.lookup[0b00000000] == (2 << 8) | 0x01 and t.lookup[0b01000000] == (2 << 8) | 0x02
    assert t.lookup[0b10000000] == (3 << 8) | 0x03 and t.lookup[0b10100000] == (4 << 8) | 0x00   # EOB = 1010
    assert t.lookup[0b11110000] == (7 << 8) | 0x06 and t.lookup[0b11110110] == (7 << 8) | 0x61   # 1111000, 1111011
    assert t.maxcode[15] == 0b111111111000000 and t.maxcode[16] == 0xFFFE and t.maxcode[14] == -1
    assert t.lookup[0b11111111] == 9 << 8


def _patch_marker(buf: bytes, marker: int, new: int) -> bytes:
    i = buf.index(bytes([0xFF, marker]))
    return buf[:i + 1] + bytes([new]) + buf[i + 2:]


def test_unsupported_jpegs_raise():
    img = TW.video_frames(1, 32, 48, 0)[0]
    cases = {
        "progressive": TW.encode(img, progressive=True),
        "4:2:2": TW.encode(img, subsampling=1),
        "grey": None,
        "restart": TW.encode(img, restart_marker_blocks=4),
        "arithmetic": _patch_marker(TW.encode(img), 0xC0, 0xC9),
    }
    from PIL import Image
    import io
    b = io.BytesIO()
    Image.fromarray(img[..., 0]).save(b, "JPEG", quality=90)
    cases["grey"] = b.getvalue()
    reasons = {"progressive": "progressive", "4:2:2": "4:2:2", "grey": "grey", "restart": "restart",
               "arithmetic": "arithmetic"}
    for k, buf in cases.items():
        with pytest.raises(ValueError, match=reasons[k]):
            J.parse(buf)


def test_mixed_frame_sizes_raise():
    a = TW.encode(TW.video_frames(1, 32, 48, 0)[0])
    b = TW.encode(TW.video_frames(1, 40, 48, 0)[0])
    v = R.parse_sequence_example(TW.sequence_example([a, b, a], 3), "rec7")
    plan = V.eval_plan([v.shape], 3, 1, 1, 32)
    with pytest.raises(ValueError, match="rec7 frame 1"):
        V.pack_jpeg([v], plan, pin=False)


# ------------------------------------------------------------------------------------------ packing
def test_pack_jpeg_stores_each_frame_and_header_once():
    fr1, fr2 = _frames(6, seed=0), _frames(4, H=48, W=40, seed=1, quality=70)
    v1 = R.parse_sequence_example(TW.sequence_example(fr1, 0), "a")
    v2 = R.parse_sequence_example(TW.sequence_example(fr2, 1), "b")
    plan = V.eval_plan([v1.shape, v2.shape], 4, 2, 3, 32)                  # frames repeat over views/crops
    vb = V.pack_jpeg([v1, v2], plan, pin=False)
    enc = vb.encoded
    pairs = {(int(v), int(f)) for v, fs in zip(plan.video, plan.frames) for f in fs}
    assert enc.nframes == len(pairs)
    assert enc.tables.numel() == 2 * J.TABLES_DTYPE.itemsize                   # two encoder settings
    recs = enc.frames.numpy().view(J.FRAME_DTYPE)
    segs = {bytes(enc.data.numpy()[r["seg_off"]:r["seg_off"] + r["seg_len"]]) for r in recs}
    assert len(segs) == enc.nframes
    assert enc.data.numel() == sum(int(r["seg_len"]) for r in recs)
    assert np.all(recs["out_off"] % 16 == 0) and np.all(recs["status"] == np.arange(enc.nframes))
    # frame_off points at the decoded frame of each (clip, t)
    off = vb.frame_off.numpy().reshape(plan.frames.shape)
    for n in range(plan.frames.shape[0]):
        for t in range(plan.frames.shape[1]):
            r = recs[recs["out_off"] == off[n, t]][0]
            src = (fr1 if plan.video[n] == 0 else fr2)[plan.frames[n, t]]
            s = J.parse(src)
            assert bytes(enc.data.numpy()[r["seg_off"]:r["seg_off"] + r["seg_len"]]) == src[s.seg_off:s.seg_off + s.seg_len]
    assert vb.frames.numel() == 0 and vb.shape == plan.shape


def test_jpeg_struct_layouts_match_header(tmp_path):
    """x3d_jpeg_frame / x3d_jpeg_huff / x3d_jpeg_tables as gcc lays them out == the ctypes structures
    the host packs the descriptors with."""
    from x3d_tf_b200 import _lib
    structs = {"x3d_jpeg_frame": _lib.JpegFrame, "x3d_jpeg_huff": _lib.JpegHuff, "x3d_jpeg_tables": _lib.JpegTables}
    lines = ['#include <stddef.h>', '#include <stdio.h>', '#include "x3d_b200.h"', 'int main(void) {']
    for cname, ct in structs.items():
        lines.append(f'  printf("{cname} %zu\\n", sizeof({cname}));')
        lines += [f'  printf("{cname}.{f} %zu\\n", offsetof({cname}, {f}));' for f, _ in ct._fields_]
    lines += ['  return 0;', '}']
    (tmp_path / "probe.c").write_text("\n".join(lines))
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(tmp_path / "probe.c")], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    for cname, ct in structs.items():
        assert int(got[cname]) == ctypes.sizeof(ct), cname
        for f, _ in ct._fields_:
            assert int(got[f"{cname}.{f}"]) == getattr(ct, f).offset, f"{cname}.{f}"
    assert ctypes.sizeof(_lib.JpegFrame) == 64 and ctypes.sizeof(_lib.JpegTables) == 4200


# ------------------------------------------------------------------------------------ IDCT oracles
def test_idct_dc_only():
    """DC only: every sample = range_limit(DESCALE(DESCALE(dc*q << 13, 11) << 13, 18)) = 128 + round(dc*q/8)."""
    coef = np.zeros((1, 64), np.int16)
    coef[0, 0] = 10
    q = np.full(64, 4)
    assert np.all(O.idct_islow(coef, q) == 128 + 5)                    # 40 / 8 = 5
    # IFAST: multiplier (4 * 16384 + 2048) >> 12 = 16; pass 2 (160 >> 5) = 5
    assert np.all(O.idct_ifast(coef, q) == 128 + 5)
    coef[0, 0] = -3
    assert np.all(O.idct_islow(coef, np.ones(64)) == 128 + 0)          # (-3*4 + 16) >> 5 = 0
    assert np.all(O.idct_ifast(coef, np.ones(64)) == 128 - 1)          # mult 4: -12 >> 5 = -1


def test_idct_one_ac_term():
    """Coefficient (0, 1) = 8, q = 1: ISLOW row values DESCALE(8 * 4 * c_k * 8192 ... ) worked by hand:
    pass 1 puts 8 << 2 = 32 in row 0 of column 1 of the workspace (the other columns are 0); pass 2 on
    row 0: z from wsptr[1] = 32 gives tmp3 = 32 * 12299 + 32 * (-3196 + 9633) ... -> outputs
    DESCALE(+-32 * {11363, 9633, 6437, 2260}, 18) + 128 for columns 0..7, rows all equal."""
    coef = np.zeros((1, 64), np.int16)
    coef[0, 1] = 8
    got = O.idct_islow(coef, np.ones(64))[0]
    c = np.array([11363, 9633, 6437, 2260])                   # 8192 * sqrt(2) * cos(k pi / 16), rounded as libjpeg's sums
    exp = np.concatenate([(32 * c + (1 << 17)) >> 18, (-32 * c[::-1] + (1 << 17)) >> 18]) + 128
    assert np.array_equal(got, np.tile(exp, (8, 1)))
    assert np.array_equal(got[:, :4], np.array([[129, 129, 129, 128]] * 8))


def test_idct_ifast_one_ac_term():
    """Coefficient (0, 1) = 8, q = 1: the IFAST multiplier is (22725 + 2048) >> 12 = 6, so pass 1 leaves
    48 in column 1 of every workspace row.  Pass 2 on a row with only wsptr[1] = 48 (odd part only):
    z11 = z12 = 48, tmp7 = 48, tmp11 = (48*362) >> 8 = 67, z5 = (48*473) >> 8 = 88,
    tmp10 = ((48*277) >> 8) - 88 = 51 - 88 = -37, tmp12 = 88, tmp6 = 88 - 48 = 40, tmp5 = 67 - 40 = 27,
    tmp4 = -37 + 27 = -10; outputs [0..7] = tmp7, tmp6, tmp5, -tmp4, tmp4, -tmp5, -tmp6, -tmp7
    = 48, 40, 27, 10, -10, -27, -40, -48, shifted right by 5 (no rounding) = 1, 1, 0, 0, -1, -1, -2, -2.
    The transposed coefficient (1, 0) runs the same odd part in pass 1 and gives the transposed block."""
    coef = np.zeros((1, 64), np.int16)
    coef[0, 1] = 8
    assert O.ifast_multipliers(np.ones(64))[1] == 6
    got = O.idct_ifast(coef, np.ones(64))[0]
    assert np.array_equal(got, np.tile(128 + np.array([1, 1, 0, 0, -1, -1, -2, -2]), (8, 1)))
    coef_t = np.zeros((1, 64), np.int16)
    coef_t[0, 8] = 8
    assert np.array_equal(O.idct_ifast(coef_t, np.ones(64))[0], got.T)


def test_idct_range_mask_wrap():
    """A saturating block: DC 1023 with q 255 descales to x = 32608; libjpeg's IDCT_range_limit takes
    x & RANGE_MASK = 864, which lies in the table's negative-clamp part: every sample is 0, not 255."""
    coef = np.zeros((1, 64), np.int16)
    coef[0, 0] = 1023
    got = O.idct_islow(coef, np.full(64, 255))
    x = (1023 * 255 * 4 * 8192 + (1 << 17)) >> 18                      # DESCALE of the DC path
    assert x == 32608 and (x & 1023) == 864
    assert np.all(got == 0)
    assert np.array_equal(O.range_limit(np.array([0, 127, 128, 511, 512, 895, 896, 1023, 1024 + 5])),
                          np.array([128, 255, 255, 255, 0, 0, 0, 127, 133]))


def test_oracle_decode_matches_pillow():
    """The numpy restatement of the whole chain (ISLOW) is byte-identical to Pillow (libjpeg-turbo)."""
    for (H, W) in [(8, 8), (37, 53), (3, 5), (2, 9)]:
        for sub in (0, 2):
            for q in (50, 90, 100):
                img = TW.video_frames(1, H, W, H * W + q)[0]
                buf = TW.encode(img, quality=q, subsampling=sub)
                assert np.array_equal(O.decode(buf), TW.pil_decode(buf)), (H, W, sub, q)
    buf = TW.encode(TW.video_frames(1, 24, 40, 5)[0], optimize=True)
    assert np.array_equal(O.decode(buf), TW.pil_decode(buf))


# ------------------------------------------------------------------------------------------ sharding
def _shard_worker(rank, world, port, root, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from x3d_tf_b200 import eval as E
        from x3d_tf_b200 import shard
        from x3d_tf_b200 import train as T
        from x3d_tf_b200.config import get_config
        cfg = get_config("X3D_XS")
        files = E.tfrecord_files(os.path.join(root, "*.tfrecord.gz"))
        lo, hi = shard.shard_range(len(files), world, rank)
        eval_labels = [int(l) for _, labels in E.tfrecord_batches(files[lo:hi], 2, cfg) for l in labels]
        mine = T.tfrecord_rank_files(files, 77, rank, world)
        steps = [labels.tolist() for _, labels in T.tfrecord_clip_batches(files, 4, 3, 77, cfg, rank, world)]
        out = [None] * world
        dist.all_gather_object(out, (eval_labels, mine, steps))
        if rank == 0:
            q.put(out)
    finally:
        dist.destroy_process_group()


def test_tfrecord_sharding_gloo_world2(tmp_path):
    """eval: ranks take contiguous blocks of the sorted files and together see every record once;
    train: every rank gets its own files r::world of the epoch's shuffled list (the same list on
    both ranks) and runs exactly `steps` steps of its share of the global batch."""
    import multiprocessing as mp
    labels = iter(range(100))
    for i in range(5):
        recs = [TW.sequence_example(_frames(2, H=16, W=16, seed=10 * i + k), next(labels)) for k in range(i % 2 + 1)]
        TW.write_tfrecord(tmp_path / f"f{i}.tfrecord.gz", recs)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() + 7) % 2000
    procs = [ctx.Process(target=_shard_worker, args=(r, 2, port, str(tmp_path), q)) for r in range(2)]
    for p in procs:
        p.start()
    out = q.get(timeout=240)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    (e0, m0, s0), (e1, m1, s1) = out
    assert e0 + e1 == list(range(7))                                   # file order, contiguous blocks
    assert sorted(m0 + m1) == sorted(str(p) for p in tmp_path.glob("*.tfrecord.gz")) and not set(m0) & set(m1)
    assert len(s0) == len(s1) == 3 and all(len(b) == 2 for b in s0 + s1)
    own = {0: set(), 1: set()}
    for r, m in ((0, m0), (1, m1)):
        for f in m:
            own[r] |= {v.label for v in R.read_videos(f)}
    assert all(set(b) <= own[0] for b in s0) and all(set(b) <= own[1] for b in s1)
