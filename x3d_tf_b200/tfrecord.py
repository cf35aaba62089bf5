"""The reference's TFRecord datasets on the host: GZIP TFRecord files of `tf.train.SequenceExample`s,
one video per record, with one JPEG per frame (datasets/create_tfrecords.py:48-83, 100-103, read by
dataloader.py:66-91, 150-174 behind `eval.py --tfrecord` / `train.py --use_tfrecord`).

  read_records(path)          the records of one GZIP TFRecord file, both CRCs checked
  parse_sequence_example(buf) one record -> TFRecordVideo (label, shape, JPEG bytes of each frame)
  serialize_sequence_example  JPEG frames + label -> one record (the reference's keys)
  write_records(path, recs)   one GZIP TFRecord file, both CRCs written

A TFRecordVideo has what video.eval_plan / train_plan need (`shape`) and what video.pack_jpeg reads
(`jpeg(f)`); its frames are decoded on the device.
"""
from __future__ import annotations

import gzip
import struct
import zlib
from typing import Iterator, List

import numpy as np

from . import jpeg as J
from .tf_bundle import BundleError, _get_varint, _pb_fields, _signed64, crc32c, mask_crc, unmask_crc

CONTEXT_FRAMES = "video/num_frames"
CONTEXT_LABEL = "video/class/label"
FRAMES_KEY = "video"


def _native_crc() -> None:
    # the C-ABI library installs its CRC-32C into tf_bundle when it loads (a record is megabytes)
    try:
        from . import _lib
        _lib.lib()
    except Exception:
        pass


def read_records(path: str) -> Iterator[bytes]:
    """Records of a GZIP TFRecord file.  Framing per record: uint64 length, uint32 masked
    crc32c(length), the data, uint32 masked crc32c(data).  A bad CRC, a truncated record or a bad
    gzip stream raises ValueError naming the file and the record index."""
    _native_crc()
    i = 0
    try:
        with gzip.open(path, "rb") as f:
            while True:
                head = f.read(12)
                if not head:
                    return
                if len(head) < 12:
                    raise ValueError(f"{path}: record {i}: truncated length field")
                length, lcrc = struct.unpack("<QI", head)
                if unmask_crc(lcrc) != crc32c(head[:8]):
                    raise ValueError(f"{path}: record {i}: length CRC mismatch")
                data = f.read(length)
                foot = f.read(4)
                if len(data) < length or len(foot) < 4:
                    raise ValueError(f"{path}: record {i}: truncated record")
                if unmask_crc(struct.unpack("<I", foot)[0]) != crc32c(data):
                    raise ValueError(f"{path}: record {i}: data CRC mismatch")
                yield data
                i += 1
    except (OSError, EOFError, zlib.error) as e:
        raise ValueError(f"{path}: record {i}: bad gzip stream ({e})") from None


def _features(buf) -> dict:
    """Features / FeatureLists: {1: map entry {1: key, 2: value}} -> {key: value bytes}."""
    out = {}
    for fno, _, entry in _pb_fields(buf):
        if fno != 1:
            continue
        key, val = None, b""
        for f2, _, v in _pb_fields(entry):
            if f2 == 1:
                key = bytes(v).decode("utf-8")
            elif f2 == 2:
                val = v
        if key is not None:
            out[key] = val
    return out


def _int64s(feature) -> List[int]:
    """Feature{3: Int64List{1: repeated int64, packed or not}}."""
    vals: List[int] = []
    found = False
    for fno, _, v in _pb_fields(feature):
        if fno != 3:
            continue
        found = True
        for f2, wt, x in _pb_fields(v):
            if f2 != 1:
                continue
            if wt == 0:
                vals.append(_signed64(x))
            elif wt == 2:
                pos = 0
                while pos < len(x):
                    u, pos = _get_varint(x, pos)
                    vals.append(_signed64(u))
    if not found:
        raise ValueError("feature is not an Int64List")
    return vals


def _bytes(feature) -> List[memoryview]:
    """Feature{1: BytesList{1: repeated bytes}}."""
    out: List[memoryview] = []
    found = False
    for fno, _, v in _pb_fields(feature):
        if fno == 1:
            found = True
            out += [x for f2, _, x in _pb_fields(v) if f2 == 1]
    if not found:
        raise ValueError("feature is not a BytesList")
    return out


class TFRecordVideo:
    """One parsed record: `label`, `shape` = (F, H, W, 3) (H and W from frame 0's header), `dtype`
    uint8 and `jpeg(f)` -> the JPEG bytes of frame f.  `name` identifies the record in messages."""
    dtype = np.uint8

    def __init__(self, label: int, frames: List[memoryview], name: str = "record"):
        self.label, self._frames, self.name = int(label), frames, name
        h = J.parse_header(frames[0])
        self.shape = (len(frames), h.H, h.W, 3)

    def jpeg(self, f: int) -> bytes:
        return bytes(self._frames[f])

    def __len__(self) -> int:
        return self.shape[0]


def parse_sequence_example(buf, name: str = "record") -> TFRecordVideo:
    """SequenceExample{1: context Features, 2: feature_lists FeatureLists} with the reference's keys:
    context `video/num_frames`, `video/class/label`; feature list `video` of one-entry BytesLists
    (one JPEG per frame).  F is the length of that list; a `video/num_frames` that disagrees or a
    missing key raises ValueError."""
    mv = memoryview(buf)
    try:
        context, lists = b"", b""
        for fno, _, v in _pb_fields(mv):
            if fno == 1:
                context = v
            elif fno == 2:
                lists = v
        ctx, fl = _features(context), _features(lists)
        for key in (CONTEXT_FRAMES, CONTEXT_LABEL):
            if key not in ctx:
                raise ValueError(f"{name}: context feature '{key}' missing")
        if FRAMES_KEY not in fl:
            raise ValueError(f"{name}: feature list '{FRAMES_KEY}' missing")
        frames = []
        for fno, _, feat in _pb_fields(fl[FRAMES_KEY]):
            if fno == 1:
                b = _bytes(feat)
                if len(b) != 1:
                    raise ValueError(f"{name}: frame {len(frames)} holds {len(b)} byte strings, not one JPEG")
                frames.append(b[0])
        nf, lab = _int64s(ctx[CONTEXT_FRAMES]), _int64s(ctx[CONTEXT_LABEL])
        if len(nf) != 1 or len(lab) != 1:
            raise ValueError(f"{name}: '{CONTEXT_FRAMES}' / '{CONTEXT_LABEL}' must hold one value each")
    except (BundleError, struct.error, IndexError) as e:
        raise ValueError(f"{name}: malformed SequenceExample ({e})") from None
    if not frames:
        raise ValueError(f"{name}: no frames")
    if nf[0] != len(frames):
        raise ValueError(f"{name}: video/num_frames = {nf[0]} but the record holds {len(frames)} frames")
    try:
        return TFRecordVideo(lab[0], frames, name)
    except ValueError as e:
        raise ValueError(f"{name}: frame 0: {e}") from None


def read_videos(path: str) -> Iterator[TFRecordVideo]:
    """The videos of one TFRecord file, in file order."""
    for i, rec in enumerate(read_records(path)):
        yield parse_sequence_example(rec, f"{path}:{i}")


# ---- writing (the reference's datasets/create_tfrecords.py:48-83, 100-103)

def _varint(n: int) -> bytes:
    n &= (1 << 64) - 1
    out = bytearray()
    while True:
        b = n & 0x7F
        n >>= 7
        if n:
            out.append(b | 0x80)
        else:
            out.append(b)
            return bytes(out)


def _ld(field: int, payload: bytes) -> bytes:
    """A length-delimited protobuf field."""
    return _varint(field << 3 | 2) + _varint(len(payload)) + payload


def _entry(key: str, value: bytes) -> bytes:
    """One map<string, message> entry of Features / FeatureLists (field 1)."""
    return _ld(1, _ld(1, key.encode("utf-8")) + _ld(2, value))


def _int64_feature(v: int) -> bytes:
    return _ld(3, _ld(1, _varint(int(v))))                   # Feature{int64_list{packed value}}


def serialize_sequence_example(frames, label: int) -> bytes:
    """The reference's record: context `video/num_frames` and `video/class/label` (Int64List), feature
    list `video` with one BytesList of one JPEG per frame, serialised as protobuf does (map entries in
    key order, as its deterministic serialisation writes them)."""
    context = _entry(CONTEXT_LABEL, _int64_feature(label)) + _entry(CONTEXT_FRAMES, _int64_feature(len(frames)))
    video = b"".join(_ld(1, _ld(1, _ld(1, bytes(f)))) for f in frames)
    return _ld(1, context) + _ld(2, _entry(FRAMES_KEY, video))


def write_records(path: str, records, level: int = 6) -> int:
    """Writes a GZIP TFRecord file (TFRecordWriter with options "GZIP"): per record the uint64 length,
    its masked CRC-32C, the data and its masked CRC-32C.  Returns the uncompressed bytes written."""
    _native_crc()
    n = 0
    with gzip.open(path, "wb", compresslevel=level) as f:
        for r in records:
            head = struct.pack("<Q", len(r))
            f.write(head + struct.pack("<I", mask_crc(crc32c(head))))
            f.write(r)
            f.write(struct.pack("<I", mask_crc(crc32c(r))))
            n += len(r) + 16
    return n
