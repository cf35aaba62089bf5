"""Test-side writer of Motion-JPEG AVI files, independent of the reader under test (x3d_tf_b200/avi.py):
RIFF 'AVI ' with hdrl (avih, one strl per stream: strh + strf), a movi list of '00dc' chunks and,
optionally, an idx1 index, 'rec ' lists, JUNK chunks, an interleaved audio stream ('01wb'), an OpenDML
'AVIX' extension holding the second half of the frames, zero-length (repeat) chunks and odd-sized
chunks with their pad byte."""
from __future__ import annotations

import struct
from typing import List, Optional, Sequence


def chunk(cid: bytes, body: bytes) -> bytes:
    return cid + struct.pack("<I", len(body)) + body + (b"\0" if len(body) & 1 else b"")


def lst(kind: bytes, body: bytes, cid: bytes = b"LIST") -> bytes:
    return cid + struct.pack("<I", len(body) + 4) + kind + body


def _strl(typ: bytes, handler: bytes, compression: bytes, W: int, H: int) -> bytes:
    strh = typ + handler + struct.pack("<IHHIIIIIIIIhhhh", 0, 0, 0, 0, 1, 25, 0, 0, 0, 0xFFFFFFFF, 0, 0, 0, W, H)
    if typ == b"vids":
        strf = struct.pack("<IiiHH4sIiiII", 40, W, H, 1, 24, compression, W * H * 3, 0, 0, 0, 0)
    else:
        strf = struct.pack("<HHIIHH", 1, 1, 8000, 16000, 2, 16)
    return lst(b"strl", chunk(b"strh", strh) + chunk(b"strf", strf))


def write_avi(path, frames: Sequence[bytes], W: int = 0, H: int = 0, idx1: bool = True, rec: bool = False,
              junk: bool = False, audio: bool = False, avix: bool = False, repeat: Sequence[int] = (),
              handler: bytes = b"MJPG", compression: bytes = b"MJPG", audio_first: bool = False,
              truncate: Optional[int] = None) -> List[bytes]:
    """Writes `frames` (JPEG bytes) as stream 0 ('00dc' chunks; with audio_first the audio is stream 0
    and the video '01dc').  `repeat`: frame numbers written as zero-length chunks instead (they repeat
    the previous frame).  Returns the frames a reader must give back, in order."""
    vs = 1 if audio_first else 0
    vid = b"%02ddc" % vs
    aud = b"%02dwb" % (1 - vs)
    strls = [_strl(b"vids", handler, compression, W, H)]
    if audio or audio_first:
        strls.append(_strl(b"auds", b"\0\0\0\0", b"", 0, 0))
        if audio_first:
            strls.reverse()
    avih = struct.pack("<IIIIIIIIIIIIII", 40000, 0, 0, 0x10, len(frames), 0, len(strls), 0, W, H, 0, 0, 0, 0)
    hdrl = lst(b"hdrl", chunk(b"avih", avih) + b"".join(strls))
    expect, items = [], []
    for i, f in enumerate(frames):
        body = b"" if i in repeat else bytes(f)
        expect.append((expect[-1] if expect else None) if i in repeat else bytes(f))
        c = chunk(vid, body)
        if audio or audio_first:
            c += chunk(aud, bytes(range(7)) * (i + 1))          # odd sizes: pad bytes
        if junk and i % 3 == 1:
            c += chunk(b"JUNK", b"\0" * 5)
        if rec:
            c = lst(b"rec ", c)
        items.append(c)
    half = len(items) // 2 if avix else len(items)
    movi = lst(b"movi", b"".join(items[:half]))
    idx = b""
    if idx1:
        entries, pos = b"", 4
        for c in items[:half]:
            entries += struct.pack("<4sIII", vid, 0x10, pos, 0)
            pos += len(c)
        idx = chunk(b"idx1", entries)
    junk_top = chunk(b"JUNK", b"\0" * 12) if junk else b""
    out = lst(b"AVI ", hdrl + junk_top + movi + idx, cid=b"RIFF")
    if avix:
        out += lst(b"AVIX", lst(b"movi", b"".join(items[half:])), cid=b"RIFF")
    if truncate is not None:
        out = out[:truncate]
    with open(path, "wb") as f:
        f.write(out)
    return expect
