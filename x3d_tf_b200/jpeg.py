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

`parse(buf, mjpeg=True)` is the opt-in for the frames of Motion-JPEG videos (avi.py; TFRecord reading
never uses it).  It accepts, on top of the above:
  - a restart interval (DRI != 0): the RSTn markers must cycle RST0..RST7 and there must be exactly
    ceil(MCUs / Ri) - 1 of them before EOI; JpegFrame.intervals gives each interval's byte range
    (byte stuffing included, fill bytes and the marker excluded), which the device decodes in parallel
    (x3d_jpeg_entropy_rst);
  - luma sampling 2x1 (4:2:2), chroma 1x1;
  - no DHT segment: the missing Huffman tables of ids 0 and 1 are the standard (Annex K) ones, as
    libjpeg-turbo's decompressor sets them for Motion-JPEG (jstdhuff.c std_huff_tables).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, Optional, Tuple

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
INTERVAL_DTYPE = np.dtype(_lib.JpegInterval)

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
    ri: int = 0                            # restart interval in MCUs (0: none; mjpeg parsing only)

    @property
    def mcus(self) -> int:
        return -(-self.W // (8 * self.hs)) * -(-self.H // (8 * self.vs))


@dataclass(frozen=True)
class JpegFrame:
    header: JpegHeader
    seg_off: int                           # the entropy-coded segment (byte stuffing included)
    seg_len: int
    intervals: Optional[np.ndarray] = None   # [n, 2] int64 (offset in buf, length) of each restart
                                             # interval when header.ri != 0, else None


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


def _parse_header(hdr, mjpeg: bool = False) -> JpegHeader:
    q: Dict[int, np.ndarray] = {}
    ri = 0
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
            if len(seg) < 2:
                raise ValueError("malformed DRI segment")
            if _u16(seg, 0) != 0 and not mjpeg:
                raise ValueError("restart interval (DRI != 0) is not supported")
            ri = _u16(seg, 0)
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
    if mjpeg and (hs, vs) == (2, 1):
        pass                                                  # 4:2:2, Motion-JPEG frames only
    elif (hs, vs) == (2, 1) or (hs, vs) == (1, 2):
        raise ValueError(f"4:2:2 / 4:4:0 JPEG (luma sampling {hs}x{vs}): only 4:2:0 and 4:4:4 are supported")
    elif (hs, vs) not in ((1, 1), (2, 2)):
        raise ValueError(f"luma sampling {hs}x{vs}: only 2x2 (4:2:0) and 1x1 (4:4:4) are supported")
    if [s[0] for s in scan] != ids:
        raise ValueError("the scan's components are not the frame's in frame order")
    comp_q = tuple(int(c[3]) for c in comps)
    comp_dc = tuple(int(s[1]) for s in scan)
    comp_ac = tuple(int(s[2]) for s in scan)
    if mjpeg:
        for k, (bits, vals) in enumerate(STD_HUFF):       # DC0, AC0, DC1, AC1 where the frame has none
            key = (k & 1, k >> 1)
            if key not in huff:
                huff[key] = _std_table(k)
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
    return JpegHeader(H, W, hs, vs, qt, comp_q, comp_dc, comp_ac, dc, ac, len(hdr), rec, ri)


_cache: Dict[bytes, JpegHeader] = {}
_mjpeg_cache: Dict[bytes, JpegHeader] = {}
_std_tables: Dict[int, DerivedTable] = {}


def _std_table(k: int) -> DerivedTable:
    """STD_HUFF[k] derived (k: 0 DC0, 1 AC0, 2 DC1, 3 AC1)."""
    t = _std_tables.get(k)
    if t is None:
        bits, vals = STD_HUFF[k]
        t = _std_tables[k] = derive_table([0] + bits, bytes(vals), k % 2 == 0)
    return t


def parse_header(buf, mjpeg: bool = False) -> JpegHeader:
    """The header of one JPEG frame (cached by its bytes; `mjpeg`: module docstring)."""
    end = _header_end(buf)
    key = bytes(buf[:end])
    cache = _mjpeg_cache if mjpeg else _cache
    h = cache.get(key)
    if h is None:
        h = _parse_header(key, mjpeg)
        if len(cache) > 4096:
            cache.clear()
        cache[key] = h
    return h


def _intervals(a: np.ndarray, h: JpegHeader, base: int) -> Tuple[int, np.ndarray]:
    """(segment length up to EOI's fill bytes, [n, 2] (offset, length) of each restart interval) of
    the entropy-coded bytes `a` (starting at offset `base` of the frame)."""
    n = -(-h.mcus // h.ri)
    pos = np.flatnonzero((a[:-1] == 0xFF) & (a[1:] != 0x00) & (a[1:] != 0xFF))     # a marker at each
    codes = a[pos[:n] + 1]
    if pos.size < n or codes[-1] != 0xD9:
        found = int(np.count_nonzero((codes >= 0xD0) & (codes <= 0xD7)))
        raise ValueError(f"{found} restart markers before the end of the scan: "
                         f"{n - 1} expected ({h.mcus} MCUs, restart interval {h.ri})")
    want = 0xD0 + np.arange(n - 1) % 8
    bad = np.flatnonzero(codes[:-1] != want)
    if bad.size:
        i = int(bad[0])
        raise ValueError(f"marker 0x{int(codes[i]):02X} where RST{i % 8} (restart interval {i + 1} of {n}) "
                         "was expected")
    ends = pos[:n].copy()
    for i in np.flatnonzero(a[np.maximum(ends - 1, 0)] == 0xFF):           # fill bytes before a marker
        while ends[i] > 0 and a[ends[i] - 1] == 0xFF:
            ends[i] -= 1
    starts = np.concatenate([[0], pos[:n - 1] + 2])
    if (ends < starts).any():
        raise ValueError("malformed restart interval")
    iv = np.stack([starts + base, ends - starts], 1).astype(np.int64)
    return int(ends[-1]), iv


def parse(buf, mjpeg: bool = False) -> JpegFrame:
    """Header and entropy-coded segment of one frame.  The segment runs up to the first marker
    (0xFF followed by a byte other than 0x00), which must be EOI: restart markers, a second scan or
    a DNL are rejected.  With `mjpeg` (module docstring), a frame with a restart interval has its
    segment up to EOI and the byte range of every interval."""
    h = parse_header(buf, mjpeg)
    a = np.frombuffer(buf, np.uint8)[h.scan_off:]
    if h.ri:
        if a.size < 2:
            raise ValueError("JPEG entropy-coded segment without an end marker")
        seg_len, iv = _intervals(a, h, h.scan_off)
        return JpegFrame(h, h.scan_off, seg_len, iv)
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


# ---- Encoder side: the tables and headers libjpeg-turbo's compressor writes with tf.io.encode_jpeg's
# settings (the reference's datasets/create_tfrecords.py:48-83): baseline, JDCT_ISLOW, standard
# Huffman tables, jpeg_set_quality(q, force_baseline=TRUE), no restart interval, JFIF 1.01 APP0 with
# 300x300 dpi.  The entropy-coded segments come from the device (x3d_jpeg_fdct / _enc_bits / _emit /
# _stuff, include/x3d_b200.h).

# jcparam.c std_luminance_quant_tbl / std_chrominance_quant_tbl (ITU T.81 Annex K.1), natural order
STD_QUANT = np.array([
    [16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55, 14, 13, 16, 24, 40, 57, 69, 56,
     14, 17, 22, 29, 51, 87, 80, 62, 18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113, 92,
     49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99],
    [17, 18, 24, 47] + [99] * 4 + [18, 21, 26, 66] + [99] * 4 + [24, 26, 56] + [99] * 5 + [47, 66] + [99] * 38],
    np.int64)

# jcparam.c std_huff_tables (Annex K.3): (bits[1..16], huffval) of DC luma, AC luma, DC chroma, AC chroma
STD_HUFF = (
    ([0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0], list(range(12))),
    ([0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7D], [
        0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07,
        0x22, 0x71, 0x14, 0x32, 0x81, 0x91, 0xA1, 0x08, 0x23, 0x42, 0xB1, 0xC1, 0x15, 0x52, 0xD1, 0xF0,
        0x24, 0x33, 0x62, 0x72, 0x82, 0x09, 0x0A, 0x16, 0x17, 0x18, 0x19, 0x1A, 0x25, 0x26, 0x27, 0x28,
        0x29, 0x2A, 0x34, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3A, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49,
        0x4A, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5A, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69,
        0x6A, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7A, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89,
        0x8A, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9A, 0xA2, 0xA3, 0xA4, 0xA5, 0xA6, 0xA7,
        0xA8, 0xA9, 0xAA, 0xB2, 0xB3, 0xB4, 0xB5, 0xB6, 0xB7, 0xB8, 0xB9, 0xBA, 0xC2, 0xC3, 0xC4, 0xC5,
        0xC6, 0xC7, 0xC8, 0xC9, 0xCA, 0xD2, 0xD3, 0xD4, 0xD5, 0xD6, 0xD7, 0xD8, 0xD9, 0xDA, 0xE1, 0xE2,
        0xE3, 0xE4, 0xE5, 0xE6, 0xE7, 0xE8, 0xE9, 0xEA, 0xF1, 0xF2, 0xF3, 0xF4, 0xF5, 0xF6, 0xF7, 0xF8,
        0xF9, 0xFA]),
    ([0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0], list(range(12))),
    ([0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77], [
        0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71,
        0x13, 0x22, 0x32, 0x81, 0x08, 0x14, 0x42, 0x91, 0xA1, 0xB1, 0xC1, 0x09, 0x23, 0x33, 0x52, 0xF0,
        0x15, 0x62, 0x72, 0xD1, 0x0A, 0x16, 0x24, 0x34, 0xE1, 0x25, 0xF1, 0x17, 0x18, 0x19, 0x1A, 0x26,
        0x27, 0x28, 0x29, 0x2A, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3A, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48,
        0x49, 0x4A, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5A, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68,
        0x69, 0x6A, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7A, 0x82, 0x83, 0x84, 0x85, 0x86, 0x87,
        0x88, 0x89, 0x8A, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9A, 0xA2, 0xA3, 0xA4, 0xA5,
        0xA6, 0xA7, 0xA8, 0xA9, 0xAA, 0xB2, 0xB3, 0xB4, 0xB5, 0xB6, 0xB7, 0xB8, 0xB9, 0xBA, 0xC2, 0xC3,
        0xC4, 0xC5, 0xC6, 0xC7, 0xC8, 0xC9, 0xCA, 0xD2, 0xD3, 0xD4, 0xD5, 0xD6, 0xD7, 0xD8, 0xD9, 0xDA,
        0xE2, 0xE3, 0xE4, 0xE5, 0xE6, 0xE7, 0xE8, 0xE9, 0xEA, 0xF2, 0xF3, 0xF4, 0xF5, 0xF6, 0xF7, 0xF8,
        0xF9, 0xFA]),
)

CHROMA = {"420": (2, 2), "444": (1, 1)}                 # encode_jpeg chroma_downsampling True / False
ENC_FRAME_DTYPE = np.dtype(_lib.JpegEncFrame)
ENC_RESULT_DTYPE = np.dtype(_lib.JpegEncResult)
EOI = b"\xff\xd9"


def quant_tables(quality: int) -> np.ndarray:
    """[2, 64] uint16 luma / chroma quantisation tables, natural order: jcparam.c jpeg_set_quality
    (jpeg_quality_scaling, then jpeg_add_quant_table with force_baseline = TRUE)."""
    q = min(max(int(quality), 1), 100)
    scale = 5000 // q if q < 50 else 200 - 2 * q
    t = (STD_QUANT * scale + 50) // 100
    return np.clip(t, 1, 255).astype(np.uint16)


def huff_codes(bits, huffval):
    """jchuff.c jpeg_make_c_derived_tbl: (ehufco[256], ehufsi[256]) code and length by symbol."""
    co, si = np.zeros(256, np.uint32), np.zeros(256, np.uint8)
    code, p = 0, 0
    for l in range(1, 17):
        for _ in range(bits[l - 1]):
            co[huffval[p]], si[huffval[p]] = code, l
            code += 1
            p += 1
        code <<= 1
    return co, si


def _segment(marker: int, body: bytes) -> bytes:
    return bytes([0xFF, marker]) + (len(body) + 2).to_bytes(2, "big") + body


def encoder_header(H: int, W: int, quality: int = 90, subsampling: str = "420") -> bytes:
    """Everything before the entropy-coded segment, as libjpeg-turbo writes it (jcmarker.c): SOI,
    JFIF 1.01 APP0 with 300x300 dpi, DQT luma, DQT chroma (zigzag order), SOF0, DHT DC0, AC0, DC1,
    AC1, SOS of the three components."""
    if subsampling not in CHROMA:
        raise ValueError(f"subsampling {subsampling!r}: '420' or '444'")
    if not (1 <= H <= 65535 and 1 <= W <= 65535):
        raise ValueError(f"frame size {H}x{W}: 1..65535 each")
    hs, vs = CHROMA[subsampling]
    qt = quant_tables(quality)
    out = b"\xff\xd8" + _segment(0xE0, b"JFIF\0\x01\x01\x01" + (300).to_bytes(2, "big") * 2 + b"\0\0")
    for i in range(2):
        out += _segment(0xDB, bytes([i]) + bytes(qt[i][ZIGZAG].astype(np.uint8)))
    out += _segment(0xC0, bytes([8]) + H.to_bytes(2, "big") + W.to_bytes(2, "big") +
                    bytes([3, 1, hs << 4 | vs, 0, 2, 0x11, 1, 3, 0x11, 1]))
    for cls_id, (bits, vals) in zip((0x00, 0x10, 0x01, 0x11), STD_HUFF):
        out += _segment(0xC4, bytes([cls_id] + bits + vals))
    return out + _segment(0xDA, bytes([3, 1, 0x00, 2, 0x11, 3, 0x11, 0, 63, 0]))


ENC_TABLES_DTYPE = np.dtype(_lib.JpegEncTables)
WORDS_PER_BLOCK = 52            # a block codes to at most 11 + 11 + 63 * (16 + 10) = 1660 bits
# blocks per launch group, which bounds the device scratch: per block 128 B of coefficients, 8 B of bit
# offset, 52 words of bits (208 B) and 416 B of output bound, 760 B in all: 3.2 GB at 2^22 blocks (a
# 600-frame 360x480 4:2:0 batch is 2.4 M blocks), plus the frames themselves
MAX_LAUNCH_BLOCKS = 1 << 22

_enc_tables: Dict[int, np.ndarray] = {}
_headers: Dict[Tuple[int, int, int, str], bytes] = {}


def enc_tables(quality: int) -> np.ndarray:
    """The x3d_jpeg_enc_tables record of `quality`: quant_tables and the standard Huffman codes."""
    t = _enc_tables.get(quality)
    if t is None:
        t = np.zeros((), ENC_TABLES_DTYPE)
        t["q"] = quant_tables(quality)
        for i, (bits, vals) in enumerate(STD_HUFF):
            t["code"][i], t["size"][i] = huff_codes(bits, vals)
        _enc_tables[quality] = t
    return t


def enc_blocks(H: int, W: int, hs: int) -> int:
    """Coefficient blocks of an H x W frame with luma sampling hs x hs (dummy blocks included)."""
    mcux, mcuy = -(-W // (8 * hs)), -(-H // (8 * hs))
    return mcux * mcuy * (hs * hs + 2)


def _as_frames(frames):
    """A list of [H, W, 3] uint8 frames: torch tensors (on the device or the host) or numpy arrays
    (memory-mapped ones are read once, into the pinned staging buffer)."""
    import torch
    if isinstance(frames, (list, tuple)):
        items = list(frames)
    else:
        if frames.ndim == 3:
            frames = frames[None]
        if frames.ndim != 4:
            raise ValueError(f"frames must be [F, H, W, 3] or [H, W, 3], got {tuple(frames.shape)}")
        items = list(frames)
    for i, f in enumerate(items):
        dtype_ok = f.dtype == (torch.uint8 if isinstance(f, torch.Tensor) else np.uint8)
        if not dtype_ok or f.ndim != 3 or f.shape[2] != 3:
            raise ValueError(f"frame {i}: need uint8 [H, W, 3], got {f.dtype} {tuple(f.shape)}")
        if not (1 <= f.shape[0] <= 65535 and 1 <= f.shape[1] <= 65535):
            raise ValueError(f"frame {i}: size {f.shape[0]}x{f.shape[1]} (1..65535 each)")
    return items


def _on_device(f) -> bool:
    return getattr(f, "is_cuda", False)


def encode_frames(frames, quality: int = 90, chroma: str = "420", scratch: dict = None) -> list:
    """Complete JPEG files of uint8 RGB frames, encoded on the current CUDA device exactly as
    tf.io.encode_jpeg(frame, quality, chroma_downsampling=chroma == "420") (libjpeg-turbo) writes
    them.  `frames`: [F, H, W, 3] or a ragged list of [H, W, 3], on the device or on the host
    (pinned host memory is copied asynchronously).  `scratch` keeps the device buffers between
    calls (grown as needed); after the call it also holds the last launch group's buffers."""
    import torch
    if chroma not in CHROMA:
        raise ValueError(f"chroma {chroma!r}: '420' or '444'")
    if not 1 <= int(quality) <= 100:
        raise ValueError(f"quality {quality}: 1..100")
    quality = int(quality)
    hs = CHROMA[chroma][0]
    items = _as_frames(frames)
    scratch = {} if scratch is None else scratch
    device = torch.device("cuda", torch.cuda.current_device())
    out: list = []
    i = 0
    while i < len(items):
        j, blocks = i, 0
        while j < len(items) and (j == i or blocks + enc_blocks(*items[j].shape[:2], hs) <= MAX_LAUNCH_BLOCKS):
            blocks += enc_blocks(*items[j].shape[:2], hs)
            j += 1
        out += _encode_group(items[i:j], quality, chroma, hs, scratch, device)
        i = j
    return out


def _encode_group(items, quality, chroma, hs, scratch, device) -> list:
    import torch
    from . import ops

    def buf(name, n, dtype, pin=False):
        t = scratch.get(name)
        if t is None or t.numel() < n:
            t = scratch[name] = (torch.empty(max(n, 1), dtype=dtype, pin_memory=True) if pin else
                                 torch.empty(max(n, 1), dtype=dtype, device=device))
        return t[:max(n, 1)]

    n = len(items)
    recs = np.zeros(n, ENC_FRAME_DTYPE)
    in_off = coef = word = 0
    max_blocks = 0
    for k, f in enumerate(items):
        H, W = int(f.shape[0]), int(f.shape[1])
        nb = enc_blocks(H, W, hs)
        cap = nb * WORDS_PER_BLOCK + 1
        recs[k] = (in_off, coef, word, cap, H, W, hs, hs, 0, 0)
        in_off += H * W * 3
        coef += nb
        word += cap
        max_blocks = max(max_blocks, nb)
    # the frames, packed on the device (host frames through the pinned staging buffer)
    if all(_on_device(f) for f in items):
        rgb = torch.cat([f.reshape(-1) for f in items]) if len(items) > 1 else items[0].reshape(-1).contiguous()
    else:
        stage = buf("enc_rgb_host", in_off, torch.uint8, pin=True)
        host = stage.numpy()
        for k, f in enumerate(items):
            o, size = int(recs[k]["in_off"]), int(np.prod(f.shape))
            if isinstance(f, torch.Tensor):
                stage[o:o + size].copy_(f.reshape(-1))
            else:
                host[o:o + size] = np.asarray(f).reshape(-1)
        rgb = buf("enc_rgb", in_off, torch.uint8)
        rgb.copy_(stage, non_blocking=True)
    frames_t = torch.from_numpy(recs.view(np.uint8).copy()).to(device, non_blocking=False)
    tables_t = torch.from_numpy(enc_tables(quality).reshape(1).view(np.uint8).copy()).to(device)
    coef_t = buf("enc_coef", coef * 64, torch.int16)
    boff = buf("enc_boff", coef, torch.int64)
    res = buf("enc_res", n * ENC_RESULT_DTYPE.itemsize, torch.uint8)
    words = buf("enc_words", word, torch.int32)
    seg = buf("enc_out", word * 8, torch.uint8)
    ops.jpeg_fdct(rgb, frames_t, tables_t, n, max_blocks, coef_t)
    ops.jpeg_enc_bits(coef_t, frames_t, tables_t, n, boff, res, words)
    ops.jpeg_enc_emit(coef_t, frames_t, tables_t, n, max_blocks, boff, res, words)
    ops.jpeg_enc_stuff(words, frames_t, n, res, seg)
    scratch.update(enc_frames=frames_t, enc_coef_group=coef_t, enc_res_group=res, enc_out_group=seg)
    r = res.cpu().numpy().view(ENC_RESULT_DTYPE)            # synchronises
    bad = np.flatnonzero(r["status"] != 0)
    if bad.size:
        raise RuntimeError(f"JPEG encoding of frame {int(bad[0])} failed with status {int(r['status'][bad[0]])}")
    end = int((r["out_off"] + r["len"]).max())
    out_host = buf("enc_out_host", end, torch.uint8, pin=True)
    out_host.copy_(seg[:end])
    mv = memoryview(out_host.numpy())
    files = []
    for k, f in enumerate(items):
        key = (int(f.shape[0]), int(f.shape[1]), quality, chroma)
        hdr = _headers.get(key)
        if hdr is None:
            if len(_headers) > 4096:
                _headers.clear()
            hdr = _headers[key] = encoder_header(*key)
        o = int(r["out_off"][k])
        files.append(b"".join((hdr, mv[o:o + int(r["len"][k])], EOI)))
    return files
