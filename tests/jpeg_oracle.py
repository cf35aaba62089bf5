"""numpy restatement of the device JPEG decoder (x3d_tf_b200/csrc/x3d_jpeg.cu), stage by stage, from
libjpeg-turbo's sources in their default libjpeg-6b mode:

  entropy      jdhuff.c decode_mcu: coefficient blocks int16 [blocks][64] (natural order), the
               device's block layout (component after component, each block grid row-major)
  idct_islow   jidctint.c jpeg_idct_islow (CONST_BITS 13, PASS1_BITS 2, JLONG = int64)
  idct_ifast   jidctfst.c jpeg_idct_ifast (DCTELEM = int32, multiplier table of jddctmgr.c)
  color        jdsample.c h2v2_fancy_upsample / h2v2_upsample + jdcolor.c ycc_rgb_convert

`decode(buf, method)` chains them.  The IDCTs are pinned by hand-worked blocks (tests/test_jpeg.py);
the whole chain with ISLOW is pinned against Pillow (libjpeg-turbo) there too.
"""
from __future__ import annotations

import numpy as np

from x3d_tf_b200 import jpeg as J

AANSCALES = np.array([
    16384, 22725, 21407, 19266, 16384, 12873, 8867, 4520, 22725, 31521, 29692, 26722, 22725, 17855, 12299, 6270,
    21407, 29692, 27969, 25172, 21407, 16819, 11585, 5906, 19266, 26722, 25172, 22654, 19266, 15137, 10426, 5315,
    16384, 22725, 21407, 19266, 16384, 12873, 8867, 4520, 12873, 17855, 16819, 15137, 12873, 10114, 6967, 3552,
    8867, 12299, 11585, 10426, 8867, 6967, 4799, 2446, 4520, 6270, 5906, 5315, 4520, 3552, 2446, 1247], np.int64)


def range_limit(x):
    """IDCT_range_limit(cinfo)[x & RANGE_MASK] (jdmaster.c prepare_range_limit_table)."""
    v = ((np.asarray(x, np.int64) + 512) & 1023) - 512 + 128
    return np.clip(v, 0, 255).astype(np.uint8)


def _descale(x, n):
    return (x + (1 << (n - 1))) >> n


def _islow_1d(d, n):
    """d: [..., 8] int64 -> [..., 8] int64 descaled by n."""
    z2, z3 = d[..., 2], d[..., 6]
    z1 = (z2 + z3) * 4433
    tmp2, tmp3 = z1 + z3 * -15137, z1 + z2 * 6270
    z2, z3 = d[..., 0], d[..., 4]
    tmp0, tmp1 = (z2 + z3) << 13, (z2 - z3) << 13
    tmp10, tmp13, tmp11, tmp12 = tmp0 + tmp3, tmp0 - tmp3, tmp1 + tmp2, tmp1 - tmp2
    tmp0, tmp1, tmp2, tmp3 = d[..., 7], d[..., 5], d[..., 3], d[..., 1]
    z1, z2, z3, z4 = tmp0 + tmp3, tmp1 + tmp2, tmp0 + tmp2, tmp1 + tmp3
    z5 = (z3 + z4) * 9633
    tmp0, tmp1, tmp2, tmp3 = tmp0 * 2446, tmp1 * 16819, tmp2 * 25172, tmp3 * 12299
    z1, z2, z3, z4 = z1 * -7373, z2 * -20995, z3 * -16069 + z5, z4 * -3196 + z5
    tmp0, tmp1, tmp2, tmp3 = tmp0 + z1 + z3, tmp1 + z2 + z4, tmp2 + z2 + z3, tmp3 + z1 + z4
    out = [tmp10 + tmp3, tmp11 + tmp2, tmp12 + tmp1, tmp13 + tmp0,
           tmp13 - tmp0, tmp12 - tmp1, tmp11 - tmp2, tmp10 - tmp3]
    return np.stack([_descale(o, n) for o in out], -1)


def idct_islow(coef, q):
    """coef [N, 64] int16 (natural order), q [N, 64] or [64] quantisation table -> [N, 8, 8] uint8."""
    d = (np.asarray(coef, np.int64) * np.asarray(q, np.int64)).reshape(-1, 8, 8)
    ws = _islow_1d(np.swapaxes(d, 1, 2), 13 - 2).astype(np.int32).astype(np.int64)   # columns
    ws = np.swapaxes(ws, 1, 2)                                                           # [N, row, col]
    return range_limit(_islow_1d(ws, 13 + 2 + 3))


def _w32(x):
    return np.asarray(x, np.int64).astype(np.int32).astype(np.int64)             # C int wrap-around


def _fmul(v, c):
    return _w32((v * c) >> 8)


def _ifast_1d(d):
    t0, t1, t2, t3 = d[..., 0], d[..., 2], d[..., 4], d[..., 6]
    t10, t11, t13 = _w32(t0 + t2), _w32(t0 - t2), _w32(t1 + t3)
    t12 = _w32(_fmul(_w32(t1 - t3), 362) - t13)
    t0, t3, t1, t2 = _w32(t10 + t13), _w32(t10 - t13), _w32(t11 + t12), _w32(t11 - t12)
    t4, t5, t6, t7 = d[..., 1], d[..., 3], d[..., 5], d[..., 7]
    z13, z10, z11, z12 = _w32(t6 + t5), _w32(t6 - t5), _w32(t4 + t7), _w32(t4 - t7)
    t7 = _w32(z11 + z13)
    t11 = _fmul(_w32(z11 - z13), 362)
    z5 = _fmul(_w32(z10 + z12), 473)
    t10 = _w32(_fmul(z12, 277) - z5)
    t12 = _w32(_fmul(z10, -669) + z5)
    t6 = _w32(t12 - t7)
    t5 = _w32(t11 - t6)
    t4 = _w32(t10 + t5)
    out = [t0 + t7, t1 + t6, t2 + t5, t3 - t4, t3 + t4, t2 - t5, t1 - t6, t0 - t7]
    return np.stack([_w32(o) for o in out], -1)


def ifast_multipliers(q):
    """jddctmgr.c: DESCALE(quantval * aanscales, CONST_BITS - IFAST_SCALE_BITS = 12), natural order."""
    return (np.asarray(q, np.int64) * AANSCALES + (1 << 11)) >> 12


def idct_ifast(coef, q):
    d = _w32(np.asarray(coef, np.int64) * ifast_multipliers(q)).reshape(-1, 8, 8)
    ws = np.swapaxes(_ifast_1d(np.swapaxes(d, 1, 2)), 1, 2)
    return range_limit(_ifast_1d(ws) >> 5)


# ---------------------------------------------------------------------------------- entropy decoding
class _Bits:
    def __init__(self, seg: bytes):
        self.data = seg.replace(b"\xff\x00", b"\xff")       # in-segment FF is always stuffed
        self.pos = 0                                        # bit position

    def peek(self, n):
        v = 0
        for k in range(n):
            i = self.pos + k
            byte = self.data[i >> 3] if (i >> 3) < len(self.data) else 0
            v = (v << 1) | ((byte >> (7 - (i & 7))) & 1)
        return v

    def get(self, n):
        v = self.peek(n)
        self.pos += n
        return v


def _decode_sym(br, t: J.DerivedTable):
    look = int(t.lookup[br.peek(8)])
    if look >> 8 <= 8:
        br.pos += look >> 8
        return look & 0xFF
    l = 9
    while l <= 16 and br.peek(l) > int(t.maxcode[l]):
        l += 1
    if l > 16:
        raise ValueError("bad Huffman code")
    code = br.get(l)
    return int(t.huffval[(code + int(t.valoffset[l])) & 0xFF])


def _extend(r, s):
    return r - (1 << s) + 1 if r < (1 << (s - 1)) else r


def grid(h: J.JpegHeader):
    """(mcux, mcuy, [(bw, bh)] per component)."""
    mcux, mcuy = -(-h.W // (8 * h.hs)), -(-h.H // (8 * h.vs))
    return mcux, mcuy, [(mcux * h.hs, mcuy * h.vs), (mcux, mcuy), (mcux, mcuy)]


def entropy(buf: bytes):
    """Coefficients [blocks, 64] int16 of one frame in the device layout."""
    fr = J.parse(buf)
    h = fr.header
    mcux, mcuy, dims = grid(h)
    planes = [np.zeros((bh, bw, 64), np.int16) for bw, bh in dims]
    br = _Bits(bytes(buf[fr.seg_off:fr.seg_off + fr.seg_len]))
    pred = [0, 0, 0]
    for my in range(mcuy):
        for mx in range(mcux):
            for c in range(3):
                hs, vs = (h.hs, h.vs) if c == 0 else (1, 1)
                for by in range(vs):
                    for bx in range(hs):
                        blk = planes[c][my * vs + by, mx * hs + bx]
                        s = _decode_sym(br, h.dc[h.comp_dc[c]])
                        if s:
                            s = _extend(br.get(s), s)
                        pred[c] = int(np.int32(np.int64(pred[c]) + s))
                        blk[0] = np.int64(pred[c]).astype(np.int16)
                        k = 1
                        while k < 64:
                            s = _decode_sym(br, h.ac[h.comp_ac[c]])
                            r, s = s >> 4, s & 15
                            if s:
                                k += r
                                if k > 63:
                                    raise ValueError("run past coefficient 63")
                                blk[J.ZIGZAG[k]] = _extend(br.get(s), s)
                            else:
                                if r != 15:
                                    break
                                k += 15
                                if k > 63:
                                    raise ValueError("run past coefficient 63")
                            k += 1
    if br.pos > len(br.data) * 8:
        raise ValueError("premature end of data")
    return np.concatenate([p.reshape(-1, 64) for p in planes])


def idct(buf: bytes, coef, method: str = "INTEGER_ACCURATE"):
    """Sample planes [bh*8, bw*8] uint8 of the three components."""
    h = J.parse_header(buf)
    _, _, dims = grid(h)
    fn = idct_islow if method == "INTEGER_ACCURATE" else idct_ifast
    out, b = [], 0
    for c, (bw, bh) in enumerate(dims):
        blocks = fn(coef[b:b + bw * bh], h.qtables[h.comp_q[c]])
        b += bw * bh
        out.append(blocks.reshape(bh, bw, 8, 8).transpose(0, 2, 1, 3).reshape(bh * 8, bw * 8))
    return out


def _fancy(p, H, W):
    """h2v2_fancy_upsample of plane p to H x W (edges at the downsampled extent)."""
    dh, dw = -(-H // 2), -(-W // 2)
    p = p[:dh, :dw].astype(np.int64)
    y, x = np.arange(H), np.arange(W)
    i, j = y >> 1, x >> 1
    far = np.where(y & 1, np.minimum(i + 1, dh - 1), np.maximum(i - 1, 0))
    cs = 3 * p[i] + p[far]                                            # [H, dw] column sums
    if dw <= 2:                                                       # libjpeg uses the box filter
        return p[i][:, j]
    jn = np.where(x & 1, np.minimum(j + 1, dw - 1), np.maximum(j - 1, 0))
    return np.where(x & 1, (3 * cs[:, j] + cs[:, jn] + 7) >> 4, (3 * cs[:, j] + cs[:, jn] + 8) >> 4)


def color(buf: bytes, planes):
    h = J.parse_header(buf)
    H, W = h.H, h.W
    Y = planes[0][:H, :W].astype(np.int64)
    if h.hs == 2:
        cb, cr = _fancy(planes[1], H, W), _fancy(planes[2], H, W)
    else:
        cb, cr = planes[1][:H, :W].astype(np.int64), planes[2][:H, :W].astype(np.int64)
    cb, cr = cb - 128, cr - 128
    r = Y + ((91881 * cr + 32768) >> 16)
    g = Y + ((-22554 * cb + 32768 - 46802 * cr) >> 16)
    b = Y + ((116130 * cb + 32768) >> 16)
    return np.clip(np.stack([r, g, b], -1), 0, 255).astype(np.uint8)


def decode(buf: bytes, method: str = "INTEGER_ACCURATE"):
    return color(buf, idct(buf, entropy(buf), method))
