"""JPEG headers on the host: everything the device decoder (x3d_jpeg_entropy / _idct / _color,
include/x3d_b200.h) needs for one frame, and the rejection of everything it does not decode.

Supported input is exactly what TF 2.4's `tf.io.encode_jpeg` writes for RGB frames (the reference's
`datasets/create_tfrecords.py:48-83`): baseline sequential Huffman (SOF0), 8-bit samples and
quantisation tables, three components in one interleaved scan, luma sampling 2x2 (4:2:0, TF's
default `chroma_downsampling=True`) or 1x1 (4:4:4), chroma 1x1, no restart interval.  APPn and COM
segments are skipped.  Anything else raises ValueError with the reason before anything reaches the
device.

The frames of one encoder run share their header, so `parse` caches the parsed tables by the header
bytes (everything before the entropy-coded segment); a batch then carries one table set per distinct
header.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, Tuple

import numpy as np

from . import _lib

# zigzag position -> natural (row-major) index, ITU T.81 figure A.6
ZIGZAG = np.array([
    0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14,
    21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60,
    61, 54, 47, 55, 62, 63], np.int64)

LOOKAHEAD = 8
TABLES_DTYPE = np.dtype(_lib.JpegTables)
FRAME_DTYPE = np.dtype(_lib.JpegFrame)

_SOF_REASON = {0xC1: "extended sequential (SOF1)", 0xC2: "progressive (SOF2)", 0xC3: "lossless (SOF3)",
               0xC5: "hierarchical (SOF5)", 0xC6: "hierarchical progressive (SOF6)",
               0xC7: "hierarchical lossless (SOF7)", 0xC9: "arithmetic coding (SOF9)",
               0xCA: "arithmetic progressive (SOF10)", 0xCB: "arithmetic lossless (SOF11)",
               0xCD: "arithmetic hierarchical (SOF13)", 0xCE: "arithmetic hierarchical progressive (SOF14)",
               0xCF: "arithmetic hierarchical lossless (SOF15)"}


@dataclass(frozen=True)
class DerivedTable:
    """libjpeg's jpeg_make_d_derived_tbl (jdhuff.c) of one Huffman table: maxcode[18], valoffset[18]
    (index 1..16 used, maxcode[17] = 0xFFFFF), lookup[256] = (length << 8) | symbol of the code the
    next 8 bits start with (9 << 8 when that code is longer) and huffval[256]."""
    maxcode: np.ndarray
    valoffset: np.ndarray
    lookup: np.ndarray
    huffval: np.ndarray


@dataclass(frozen=True)
class JpegHeader:
    H: int
    W: int
    hs: int                                # luma sampling factors (chroma is 1x1)
    vs: int
    qtables: np.ndarray                    # [4, 64] uint16, natural order, by table id (unused ids zero)
    comp_q: Tuple[int, int, int]           # quantisation table id of component 0, 1, 2
    comp_dc: Tuple[int, int, int]          # DC / AC Huffman table id of each component
    comp_ac: Tuple[int, int, int]
    dc: Tuple[DerivedTable, ...]           # derived DC / AC tables by id (None where undefined)
    ac: Tuple[DerivedTable, ...]
    scan_off: int                          # offset of the entropy-coded segment = header length
    tables: np.ndarray                     # the x3d_jpeg_tables record the device reads


@dataclass(frozen=True)
class JpegFrame:
    header: JpegHeader
    seg_off: int                           # the entropy-coded segment (byte stuffing included)
    seg_len: int


def derive_table(bits, huffval, is_dc: bool) -> DerivedTable:
    """jdhuff.c jpeg_make_d_derived_tbl: bits[1..16] code counts (bits[0] ignored), huffval symbols."""
    bits = [int(b) for b in bits]
    n = sum(bits[1:17])
    if n > 256 or len(huffval) < n:
        raise ValueError("bad Huffman table: more than 256 codes")
    sizes = [l for l in range(1, 17) for _ in range(bits[l])]
    codes, code, si, p = [], 0, sizes[0] if sizes else 0, 0
    while p < n:
        while p < n and sizes[p] == si:
            codes.append(code)
            code += 1
            p += 1
        if code >= (1 << si):
            raise ValueError("bad Huffman table: code lengths overflow")
        code <<= 1
        si += 1
    maxcode = np.full(18, -1, np.int32)
    valoffset = np.zeros(18, np.int32)
    p = 0
    for l in range(1, 17):
        if bits[l]:
            valoffset[l] = p - codes[p]
            p += bits[l]
            maxcode[l] = codes[p - 1]
    maxcode[17] = 0xFFFFF
    lookup = np.full(1 << LOOKAHEAD, (LOOKAHEAD + 1) << LOOKAHEAD, np.uint16)
    p = 0
    for l in range(1, LOOKAHEAD + 1):
        for _ in range(bits[l]):
            look = codes[p] << (LOOKAHEAD - l)
            lookup[look:look + (1 << (LOOKAHEAD - l))] = (l << LOOKAHEAD) | huffval[p]
            p += 1
    hv = np.zeros(256, np.uint8)
    hv[:n] = np.frombuffer(bytes(huffval[:n]), np.uint8)
    if is_dc and n and int(hv[:n].max()) > 15:
        raise ValueError("bad Huffman table: DC symbol above 15")
    return DerivedTable(maxcode, valoffset, lookup, hv)


def _u16(buf, pos: int) -> int:
    if pos + 2 > len(buf):
        raise ValueError("truncated JPEG header")
    return (buf[pos] << 8) | buf[pos + 1]


def _header_end(buf) -> int:
    """Offset of the first entropy-coded byte: the end of the first SOS segment."""
    if len(buf) < 4 or buf[0] != 0xFF or buf[1] != 0xD8:
        raise ValueError("not a JPEG stream (no SOI marker)")
    pos = 2
    while True:
        if pos + 4 > len(buf) or buf[pos] != 0xFF:
            raise ValueError("truncated or malformed JPEG header")
        while buf[pos + 1] == 0xFF:                          # fill bytes before a marker
            pos += 1
            if pos + 4 > len(buf):
                raise ValueError("truncated JPEG header")
        m, ln = buf[pos + 1], _u16(buf, pos + 2)
        if m == 0xD9:
            raise ValueError("JPEG stream ends before its scan")
        pos += 2 + ln
        if m == 0xDA:
            if pos > len(buf):
                raise ValueError("truncated JPEG header")
            return pos


def _parse_header(hdr) -> JpegHeader:
    q: Dict[int, np.ndarray] = {}
    huff: Dict[Tuple[int, int], DerivedTable] = {}
    sof = scan = None
    adobe = jfif = False
    pos = 2
    while pos < len(hdr):
        while hdr[pos + 1] == 0xFF:
            pos += 1
        m, ln = hdr[pos + 1], _u16(hdr, pos + 2)
        seg = hdr[pos + 4:pos + 2 + ln]
        pos += 2 + ln
        if ln < 2 or len(seg) != ln - 2:
            raise ValueError(f"truncated JPEG segment (marker 0x{m:02X})")
        if 0xE0 <= m <= 0xEF or m == 0xFE:
            if m == 0xE0 and bytes(seg[:5]) == b"JFIF\0":
                jfif = True
            if m == 0xEE and bytes(seg[:5]) == b"Adobe" and len(seg) >= 12:
                adobe = True
                if seg[11] != 1:
                    raise ValueError(f"Adobe colour transform {seg[11]} (only YCbCr, 1, is supported)")
        elif m == 0xDB:
            i = 0
            while i < len(seg):
                pq, tq = seg[i] >> 4, seg[i] & 15
                if pq != 0:
                    raise ValueError("16-bit quantisation table (only 8-bit tables are supported)")
                if tq > 3 or i + 65 > len(seg):
                    raise ValueError("malformed DQT segment")
                t = np.zeros(64, np.uint16)
                t[ZIGZAG] = np.frombuffer(bytes(seg[i + 1:i + 65]), np.uint8)
                q[tq] = t
                i += 65
        elif m == 0xC4:
            i = 0
            while i < len(seg):
                tc, th = seg[i] >> 4, seg[i] & 15
                if tc > 1 or th > 1:
                    raise ValueError(f"Huffman table class {tc} id {th} (baseline allows ids 0 and 1)")
                bits = [0] + list(seg[i + 1:i + 17])
                n = sum(bits)
                if len(bits) != 17 or i + 17 + n > len(seg):
                    raise ValueError("malformed DHT segment")
                huff[(tc, th)] = derive_table(bits, bytes(seg[i + 17:i + 17 + n]), tc == 0)
                i += 17 + n
        elif m == 0xC0:
            if len(seg) < 6:
                raise ValueError("malformed SOF0 segment")
            P, H, W, nf = seg[0], _u16(seg, 1), _u16(seg, 3), seg[5]
            if P != 8:
                raise ValueError(f"{P}-bit samples (only 8-bit baseline is supported)")
            if nf == 1:
                raise ValueError("grey (one-component) JPEG: only three-component YCbCr is supported")
            if nf != 3 or len(seg) < 6 + 3 * nf:
                raise ValueError(f"{nf} components: only three-component YCbCr is supported")
            if H == 0 or W == 0:
                raise ValueError("JPEG with a zero height or width (DNL) is not supported")
            comps = [(seg[6 + 3 * k], seg[7 + 3 * k] >> 4, seg[7 + 3 * k] & 15, seg[8 + 3 * k]) for k in range(3)]
            sof = (H, W, comps)
        elif m in _SOF_REASON:
            raise ValueError(f"{_SOF_REASON[m]} JPEG: only baseline sequential (SOF0) is supported")
        elif m == 0xCC:
            raise ValueError("arithmetic coding conditioning (DAC): only Huffman coding is supported")
        elif m == 0xDD:
            if len(seg) < 2 or _u16(seg, 0) != 0:
                raise ValueError("restart interval (DRI != 0) is not supported")
        elif m == 0xDA:
            ns = seg[0] if seg else 0
            if ns != 3:
                raise ValueError(f"non-interleaved scan ({ns} of 3 components): one interleaved scan is required")
            if len(seg) < 1 + 2 * ns + 3:
                raise ValueError("malformed SOS segment")
            sel = [(seg[1 + 2 * k], seg[2 + 2 * k] >> 4, seg[2 + 2 * k] & 15) for k in range(ns)]
            ss, se, ahl = seg[1 + 2 * ns], seg[2 + 2 * ns], seg[3 + 2 * ns]
            if (ss, se, ahl) != (0, 63, 0):
                raise ValueError("scan is not a baseline sequential scan (Ss, Se, Ah/Al)")
            scan = sel
        else:
            raise ValueError(f"unsupported JPEG marker 0x{m:02X}")
    if sof is None:
        raise ValueError("JPEG without a frame header (SOF0) before its scan")
    H, W, comps = sof
    ids = [c[0] for c in comps]
    if not jfif and not adobe and ids == [82, 71, 66]:
        raise ValueError("RGB-coded JPEG (component ids 'R', 'G', 'B'): only YCbCr is supported")
    (hs, vs), chroma = comps[0][1:3], [c[1:3] for c in comps[1:]]
    if any(c != (1, 1) for c in chroma):
        raise ValueError(f"chroma sampling {chroma}: only 1x1 chroma is supported")
    if (hs, vs) == (2, 1) or (hs, vs) == (1, 2):
        raise ValueError(f"4:2:2 / 4:4:0 JPEG (luma sampling {hs}x{vs}): only 4:2:0 and 4:4:4 are supported")
    if (hs, vs) not in ((1, 1), (2, 2)):
        raise ValueError(f"luma sampling {hs}x{vs}: only 2x2 (4:2:0) and 1x1 (4:4:4) are supported")
    if [s[0] for s in scan] != ids:
        raise ValueError("the scan's components are not the frame's in frame order")
    comp_q = tuple(int(c[3]) for c in comps)
    comp_dc = tuple(int(s[1]) for s in scan)
    comp_ac = tuple(int(s[2]) for s in scan)
    for k in range(3):
        if comp_q[k] not in q:
            raise ValueError(f"component {k}: quantisation table {comp_q[k]} is not defined")
        if (0, comp_dc[k]) not in huff or (1, comp_ac[k]) not in huff:
            raise ValueError(f"component {k}: Huffman table not defined")
    qt = np.zeros((4, 64), np.uint16)
    for i, t in q.items():
        qt[i] = t
    dc = tuple(huff.get((0, i)) for i in range(2))
    ac = tuple(huff.get((1, i)) for i in range(2))
    rec = np.zeros((), TABLES_DTYPE)
    for name, tabs in (("dc", dc), ("ac", ac)):
        for i, t in enumerate(tabs):
            if t is not None:
                for f in ("maxcode", "valoffset", "lookup", "huffval"):
                    rec[name][f][i] = getattr(t, f)
    rec["q"] = qt
    rec["comp_q"], rec["comp_dc"], rec["comp_ac"] = comp_q, comp_dc, comp_ac
    return JpegHeader(H, W, hs, vs, qt, comp_q, comp_dc, comp_ac, dc, ac, len(hdr), rec)


_cache: Dict[bytes, JpegHeader] = {}


def parse_header(buf) -> JpegHeader:
    """The header of one JPEG frame (cached by its bytes)."""
    end = _header_end(buf)
    key = bytes(buf[:end])
    h = _cache.get(key)
    if h is None:
        h = _parse_header(key)
        if len(_cache) > 4096:
            _cache.clear()
        _cache[key] = h
    return h


def parse(buf) -> JpegFrame:
    """Header and entropy-coded segment of one frame.  The segment runs up to the first marker
    (0xFF followed by a byte other than 0x00), which must be EOI: restart markers, a second scan or
    a DNL are rejected."""
    h = parse_header(buf)
    a = np.frombuffer(buf, np.uint8)[h.scan_off:]
    ff = np.flatnonzero(a[:-1] == 0xFF)
    ff = ff[a[ff + 1] != 0]
    if ff.size == 0:
        raise ValueError("JPEG entropy-coded segment without an end marker")
    end = int(ff[0])
    while end + 1 < a.size and a[end + 1] == 0xFF:         # fill bytes before the marker
        end += 1
    marker = int(a[end + 1])
    if 0xD0 <= marker <= 0xD7:
        raise ValueError("restart marker in the scan: restart intervals are not supported")
    if marker != 0xD9:
        raise ValueError(f"marker 0x{marker:02X} after the scan: only one scan followed by EOI is supported")
    return JpegFrame(h, h.scan_off, int(ff[0]))
