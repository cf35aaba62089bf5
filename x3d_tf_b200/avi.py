"""Motion-JPEG AVI files: the video files the reference's default input path reads with
decord.VideoReader (dataloader.py:29-63), in the one codec this project decodes on the device.
Any video converts to one with

    ffmpeg -i in.mp4 -an -c:v mjpeg -pix_fmt yuvj420p -q:v 3 out.avi

The file is walked chunk header by chunk header over an mmap (RIFF 'AVI ', then any RIFF 'AVIX'
extensions of OpenDML files over 1 GB).  The video stream is the first stream whose `strh` has type
'vids' and whose handler or `strf` compression is 'MJPG' (either case); its frames are the 'NNdc' /
'NNdb' chunks of that stream number inside the 'movi' lists (nested 'rec ' lists included), in file
order.  'JUNK', 'ix##' and the chunks of other streams are skipped.  The 'idx1' / 'indx' indexes are
not read: their offsets are relative to the file or to 'movi' depending on the writer, and walking the
headers is cheap.  A zero-length video chunk repeats the previous frame (a leading one is an error).

Only the chunk table (offset and length of every frame) is kept, cached per file, so an epoch does not
re-walk its files and a batch reads only the frames its clips sample.  The frames are JPEG images with
the Motion-JPEG variants jpeg.parse(mjpeg=True) accepts: restart intervals, 4:2:2, no DHT.
"""
from __future__ import annotations

import mmap
import os
import struct
from typing import Dict, List, Sequence, Tuple

import numpy as np

from . import jpeg as J

_tables: Dict[Tuple[str, int, int], Tuple[np.ndarray, np.ndarray]] = {}


def _fourcc(b) -> str:
    return bytes(b).decode("latin-1")


def _stream_of(cid: bytes) -> int:
    """Stream number of a 'NNxx' chunk id, or -1."""
    return int(cid[:2]) if cid[:2].isdigit() else -1


def chunk_table(path: str) -> Tuple[np.ndarray, np.ndarray]:
    """(offsets, lengths) int64 of every video frame of `path` (zero-length chunks already resolved
    to the frame they repeat).  Cached by path, size and modification time."""
    st = os.stat(path)
    key = (os.path.abspath(path), st.st_size, st.st_mtime_ns)
    t = _tables.get(key)
    if t is None:
        t = _walk(path)
        if len(_tables) > 65536:
            _tables.clear()
        _tables[key] = t
    return t


def _walk(path: str) -> Tuple[np.ndarray, np.ndarray]:
    with open(path, "rb") as f:
        size = os.fstat(f.fileno()).st_size
        if size < 12:
            raise ValueError(f"{path}: not an AVI file (too short)")
        with mmap.mmap(f.fileno(), 0, access=mmap.ACCESS_READ) as m:
            return _walk_map(path, m, size)


def _walk_map(path: str, m, size: int) -> Tuple[np.ndarray, np.ndarray]:
    streams: List[Tuple[str, str, str]] = []           # (type, handler, strf compression) per strl
    video = [-1]
    off: List[int] = []
    ln: List[int] = []

    def header(pos, end):
        if pos + 8 > end:
            raise ValueError(f"{path}: truncated chunk header at byte {pos}")
        cid, n = bytes(m[pos:pos + 4]), struct.unpack_from("<I", m, pos + 4)[0]
        if pos + 8 + n > end:
            raise ValueError(f"{path}: chunk '{_fourcc(cid)}' at byte {pos} is truncated "
                             f"({n} bytes, {end - pos - 8} left)")
        return cid, n

    def find_video():
        for i, (typ, handler, comp) in enumerate(streams):
            if typ == "vids":
                if "MJPG" not in (handler.upper(), comp.upper()):
                    raise ValueError(f"{path}: video stream {i} is '{handler or comp}', not Motion-JPEG (MJPG)")
                return i
        raise ValueError(f"{path}: no video stream")

    def walk(pos, end, where):
        while pos + 8 <= end:
            cid, n = header(pos, end)
            body = pos + 8
            if cid in (b"LIST", b"RIFF"):
                if n < 4:
                    raise ValueError(f"{path}: malformed '{_fourcc(cid)}' at byte {pos}")
                kind = bytes(m[body:body + 4])
                if cid == b"RIFF" and where != "top":
                    raise ValueError(f"{path}: nested RIFF chunk at byte {pos}")
                if kind == b"strl":
                    streams.append(("", "", ""))
                if kind == b"movi" and video[0] < 0:
                    video[0] = find_video()
                if kind in (b"AVI ", b"AVIX", b"hdrl", b"strl", b"movi", b"rec "):
                    walk(body + 4, body + n, kind.decode("latin-1").strip())
            elif where == "strl" and cid == b"strh" and n >= 8:
                typ, handler = _fourcc(m[body:body + 4]), _fourcc(m[body + 4:body + 8]).strip("\0 ")
                streams[-1] = (typ, handler, streams[-1][2])
            elif where == "strl" and cid == b"strf" and n >= 20:
                streams[-1] = (streams[-1][0], streams[-1][1], _fourcc(m[body + 16:body + 20]).strip("\0 "))
            elif where in ("movi", "rec") and cid[2:] in (b"dc", b"db") and _stream_of(cid) == video[0]:
                if n == 0:
                    if not off:
                        raise ValueError(f"{path}: the first video chunk is empty (it can repeat no frame)")
                    off.append(off[-1])
                    ln.append(ln[-1])
                else:
                    off.append(body)
                    ln.append(n)
            pos = body + n + (n & 1)                          # chunks are padded to even sizes
        if pos < end and where == "top" and any(m[pos:end]):
            raise ValueError(f"{path}: truncated chunk header at byte {pos}")

    if bytes(m[0:4]) != b"RIFF" or bytes(m[8:12]) != b"AVI ":
        raise ValueError(f"{path}: not an AVI file (no RIFF 'AVI ' header)")
    walk(0, size, "top")
    if video[0] < 0:
        find_video()                                          # raises: no stream, or not MJPEG
        raise ValueError(f"{path}: no 'movi' list")
    if not off:
        raise ValueError(f"{path}: the video stream has no frames")
    return np.asarray(off, np.int64), np.asarray(ln, np.int64)


class MJPEGVideo:
    """The frames of one Motion-JPEG AVI file: `shape` = (F, H, W, 3) (H and W from frame 0's SOF),
    `dtype` uint8, `jpeg(f)` -> the JPEG bytes of frame f (read from the file on demand), `name`
    (the path) and `label`.  `mjpeg` tells video.pack_jpeg to parse with jpeg.parse(mjpeg=True)."""
    dtype = np.uint8
    mjpeg = True

    def __init__(self, path: str, label: int = 0):
        self.name, self.label = path, int(label)
        self._off, self._len = chunk_table(path)
        try:
            h = J.parse_header(self.jpeg(0), mjpeg=True)
        except ValueError as e:
            raise ValueError(f"{path} frame 0: {e}") from None
        self.shape = (len(self._off), h.H, h.W, 3)

    def jpeg(self, f: int) -> bytes:
        with open(self.name, "rb") as fh:
            return os.pread(fh.fileno(), int(self._len[f]), int(self._off[f]))

    def __len__(self) -> int:
        return self.shape[0]


def open_videos(items: Sequence[Tuple[str, int]]) -> List[MJPEGVideo]:
    """MJPEGVideo of each `(path, label)` of a `<video> <label>` list."""
    return [MJPEGVideo(p, lab) for p, lab in items]
