"""numpy restatement of the Motion-JPEG additions to the device decoder, built on tests/jpeg_oracle.py:

  entropy   jdhuff.c decode_mcu with restart intervals (each interval an independent bit stream whose
            DC predictors start at 0, process_restart), 2x1 MCUs (two luma blocks side by side, then
            Cb, then Cr), missing DHT tables taken from Annex K (jstdhuff.c)
  color     jdsample.c h2v1_fancy_upsample (h2v1_upsample when ceil(W/2) <= 2) for 2x1 frames,
            jpeg_oracle.color otherwise

`decode(buf, method)` chains them with jpeg_oracle.idct.  Pinned by a hand-worked h2v1 row and
against Pillow (libjpeg-turbo) in tests/test_mjpeg.py.
"""
from __future__ import annotations

import numpy as np

from tests import jpeg_oracle as O
from x3d_tf_b200 import jpeg as J


def _decode_block(br, h, c, pred, blk):
    s = O._decode_sym(br, h.dc[h.comp_dc[c]])
    if s:
        s = O._extend(br.get(s), s)
    pred[c] = int(np.int32(np.int64(pred[c]) + s))
    blk[0] = np.int64(pred[c]).astype(np.int16)
    k = 1
    while k < 64:
        s = O._decode_sym(br, h.ac[h.comp_ac[c]])
        r, s = s >> 4, s & 15
        if s:
            k += r
            if k > 63:
                raise ValueError("run past coefficient 63")
            blk[J.ZIGZAG[k]] = O._extend(br.get(s), s)
        else:
            if r != 15:
                break
            k += 15
            if k > 63:
                raise ValueError("run past coefficient 63")
        k += 1


def entropy(buf: bytes):
    """Coefficients [blocks, 64] int16 of one frame in the device layout."""
    fr = J.parse(buf, mjpeg=True)
    h = fr.header
    mcux, mcuy, dims = O.grid(h)
    planes = [np.zeros((bh, bw, 64), np.int16) for bw, bh in dims]
    ri = h.ri or mcux * mcuy
    ranges = fr.intervals if h.ri else [(fr.seg_off, fr.seg_len)]
    for i, (off, ln) in enumerate(ranges):
        br = O._Bits(bytes(buf[off:off + ln]))
        pred = [0, 0, 0]
        for m in range(i * ri, min((i + 1) * ri, mcux * mcuy)):
            my, mx = divmod(m, mcux)
            for c in range(3):
                hs, vs = (h.hs, h.vs) if c == 0 else (1, 1)
                for by in range(vs):
                    for bx in range(hs):
                        _decode_block(br, h, c, pred, planes[c][my * vs + by, mx * hs + bx])
        if br.pos > len(br.data) * 8:
            raise ValueError("premature end of data")
    return np.concatenate([p.reshape(-1, 64) for p in planes])


def h2v1_fancy(p, H, W):
    """h2v1_fancy_upsample of plane p to H x W (edges at the downsampled width ceil(W/2))."""
    dw = -(-W // 2)
    p = p[:H, :dw].astype(np.int64)
    x = np.arange(W)
    j = x >> 1
    if dw <= 2:                                                   # libjpeg uses the box filter
        return p[:, j]
    left, right = p[:, np.maximum(j - 1, 0)], p[:, np.minimum(j + 1, dw - 1)]
    even = np.where(j == 0, p[:, j], (3 * p[:, j] + left + 1) >> 2)
    odd = np.where(j == dw - 1, p[:, j], (3 * p[:, j] + right + 2) >> 2)
    return np.where(x & 1, odd, even)


def color(buf: bytes, planes):
    h = J.parse_header(buf, mjpeg=True)
    return _color(h, planes, h2v1_fancy if (h.hs, h.vs) == (2, 1) else None)


def _color(h, planes, up):
    H, W = h.H, h.W
    Y = planes[0][:H, :W].astype(np.int64)
    if up is not None:
        cb, cr = up(planes[1], H, W), up(planes[2], H, W)
    elif h.hs == 2:
        cb, cr = O._fancy(planes[1], H, W), O._fancy(planes[2], H, W)
    else:
        cb, cr = planes[1][:H, :W].astype(np.int64), planes[2][:H, :W].astype(np.int64)
    cb, cr = cb - 128, cr - 128
    r = Y + ((91881 * cr + 32768) >> 16)
    g = Y + ((-22554 * cb + 32768 - 46802 * cr) >> 16)
    b = Y + ((116130 * cb + 32768) >> 16)
    return np.clip(np.stack([r, g, b], -1), 0, 255).astype(np.uint8)


def idct(buf: bytes, coef, method: str = "INTEGER_ACCURATE"):
    """Sample planes [bh*8, bw*8] uint8 of the three components (jpeg_oracle's IDCTs)."""
    h = J.parse_header(buf, mjpeg=True)
    _, _, dims = O.grid(h)
    fn = O.idct_islow if method == "INTEGER_ACCURATE" else O.idct_ifast
    out, b = [], 0
    for c, (bw, bh) in enumerate(dims):
        blocks = fn(coef[b:b + bw * bh], h.qtables[h.comp_q[c]])
        b += bw * bh
        out.append(blocks.reshape(bh, bw, 8, 8).transpose(0, 2, 1, 3).reshape(bh * 8, bw * 8))
    return out


def decode(buf: bytes, method: str = "INTEGER_ACCURATE"):
    return color(buf, idct(buf, entropy(buf), method))
