"""Test-side writer of the reference's TFRecord videos, independent of the reader under test:
`tf.train.SequenceExample` messages are built at run time from `feature.proto` / `example.proto`
definitions with `descriptor_pb2` and serialised by `google.protobuf`; the TFRecord framing and GZIP
are written here.  Also synthetic video-like frames and their JPEG encoding with Pillow."""
from __future__ import annotations

import gzip
import io
import struct

import numpy as np

from x3d_tf_b200.tf_bundle import crc32c, mask_crc

_CLASSES = None


def _classes():
    global _CLASSES
    if _CLASSES is None:
        from google.protobuf import descriptor_pb2, descriptor_pool, message_factory
        F = descriptor_pb2.FieldDescriptorProto
        fd = descriptor_pb2.FileDescriptorProto(name="x3d_test_example.proto", package="x3dtest", syntax="proto3")

        def msg(name, fields, nested=()):
            m = fd.message_type.add(name=name)
            for n in nested:
                m.nested_type.add().CopyFrom(n)
            for fname, num, typ, label, tname, packed in fields:
                f = m.field.add(name=fname, number=num, type=typ, label=label)
                if tname:
                    f.type_name = tname
                if packed is not None:
                    f.options.packed = packed
            return m

        R, O = F.LABEL_REPEATED, F.LABEL_OPTIONAL
        msg("BytesList", [("value", 1, F.TYPE_BYTES, R, None, None)])
        msg("Int64List", [("value", 1, F.TYPE_INT64, R, None, True)])
        msg("Int64ListUnpacked", [("value", 1, F.TYPE_INT64, R, None, False)])
        msg("Feature", [("bytes_list", 1, F.TYPE_MESSAGE, O, ".x3dtest.BytesList", None),
                        ("int64_list", 3, F.TYPE_MESSAGE, O, ".x3dtest.Int64List", None)])
        msg("FeatureUnpacked", [("bytes_list", 1, F.TYPE_MESSAGE, O, ".x3dtest.BytesList", None),
                                ("int64_list", 3, F.TYPE_MESSAGE, O, ".x3dtest.Int64ListUnpacked", None)])
        for feat in ("Feature", "FeatureUnpacked"):
            entry = descriptor_pb2.DescriptorProto(name="FeatureEntry", options=descriptor_pb2.MessageOptions(map_entry=True))
            entry.field.add(name="key", number=1, type=F.TYPE_STRING, label=O)
            entry.field.add(name="value", number=2, type=F.TYPE_MESSAGE, label=O, type_name=f".x3dtest.{feat}")
            m = msg(f"Features{feat[7:]}", [], [entry])
            m.field.add(name="feature", number=1, type=F.TYPE_MESSAGE, label=R,
                        type_name=f".x3dtest.Features{feat[7:]}.FeatureEntry")
            msg(f"FeatureList{feat[7:]}", [("feature", 1, F.TYPE_MESSAGE, R, f".x3dtest.{feat}", None)])
            entry = descriptor_pb2.DescriptorProto(name="FeatureListEntry", options=descriptor_pb2.MessageOptions(map_entry=True))
            entry.field.add(name="key", number=1, type=F.TYPE_STRING, label=O)
            entry.field.add(name="value", number=2, type=F.TYPE_MESSAGE, label=O, type_name=f".x3dtest.FeatureList{feat[7:]}")
            m = msg(f"FeatureLists{feat[7:]}", [], [entry])
            m.field.add(name="feature_list", number=1, type=F.TYPE_MESSAGE, label=R,
                        type_name=f".x3dtest.FeatureLists{feat[7:]}.FeatureListEntry")
            msg(f"SequenceExample{feat[7:]}", [("context", 1, F.TYPE_MESSAGE, O, f".x3dtest.Features{feat[7:]}", None),
                                              ("feature_lists", 2, F.TYPE_MESSAGE, O, f".x3dtest.FeatureLists{feat[7:]}", None)])
        pool = descriptor_pool.DescriptorPool()
        pool.Add(fd)
        _CLASSES = {n: message_factory.GetMessageClass(pool.FindMessageTypeByName(f"x3dtest.{n}"))
                    for n in ("SequenceExample", "SequenceExampleUnpacked")}
    return _CLASSES


def sequence_example(frames, label: int, num_frames=None, packed: bool = True, drop=()) -> bytes:
    """The reference's record (create_tfrecords.py:48-83): context video/num_frames and
    video/class/label, feature list `video` with one JPEG per frame.  `drop` omits keys."""
    se = _classes()["SequenceExample" if packed else "SequenceExampleUnpacked"]()
    ctx = {"video/num_frames": len(frames) if num_frames is None else num_frames, "video/class/label": label}
    for k, v in ctx.items():
        if k not in drop:
            se.context.feature[k].int64_list.value.append(int(v))
    if "video" not in drop:
        fl = se.feature_lists.feature_list["video"]
        for f in frames:
            fl.feature.add().bytes_list.value.append(bytes(f))
    return se.SerializeToString()


def frame_records(records) -> bytes:
    out = bytearray()
    for r in records:
        head = struct.pack("<Q", len(r))
        out += head + struct.pack("<I", mask_crc(crc32c(head))) + r + struct.pack("<I", mask_crc(crc32c(r)))
    return bytes(out)


def write_tfrecord(path, records) -> None:
    with gzip.open(path, "wb") as f:
        f.write(frame_records(records))


def video_frames(F: int, H: int, W: int, seed: int, noise: float = 8.0) -> np.ndarray:
    """Video-like uint8 frames: moving colour gradients, a moving rectangle with hard edges and some
    noise, seeded."""
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:H, 0:W].astype(np.float32)
    ph = rng.uniform(0, 6.28, 3)
    out = np.empty((F, H, W, 3), np.uint8)
    for f in range(F):
        t = f / 10.0
        base = np.stack([128 + 100 * np.sin(x / (17 + 5 * c) + y / (23 + 3 * c) + t + ph[c]) for c in range(3)], -1)
        y0, x0 = int((H / 3) * (1 + np.sin(t))), int((W / 3) * (1 + np.cos(t)))
        base[y0:y0 + H // 4, x0:x0 + W // 4] = rng.uniform(0, 255, 3)
        base += rng.normal(0, noise, base.shape)
        out[f] = np.clip(base, 0, 255).astype(np.uint8)
    return out


def encode(img: np.ndarray, quality: int = 90, subsampling: int = 2, **kw) -> bytes:
    """Pillow JPEG (libjpeg-turbo); subsampling 2 = 4:2:0, 0 = 4:4:4."""
    from PIL import Image
    b = io.BytesIO()
    Image.fromarray(img).save(b, "JPEG", quality=quality, subsampling=subsampling, **kw)
    return b.getvalue()


def pil_decode(buf: bytes) -> np.ndarray:
    from PIL import Image
    return np.asarray(Image.open(io.BytesIO(buf)).convert("RGB"))
