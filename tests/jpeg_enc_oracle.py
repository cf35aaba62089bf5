"""numpy restatement of libjpeg-turbo's baseline compressor with tf.io.encode_jpeg's settings (JDCT_ISLOW,
standard Huffman tables, no restart interval), the reference for the device encoder:

  color_planes  jccolor.c rgb_ycc_convert, jcprepct.c / jcsample.c edge expansion and h2v2_downsample
  fdct_islow    jfdctint.c jpeg_fdct_islow (CONST_BITS 13, PASS1_BITS 2)
  quantize      jcdctmgr.c compute_reciprocal / quantize with the 16-bit DCTELEM of the SIMD build
  coefficients  jccoefct.c compress_data, dummy blocks included, in the decoder's coefficient layout
  entropy       jchuff.c encode_one_block + flush_bits (byte stuffing, 1-bit padding)
  encode        encoder_header + entropy + EOI: the whole file
"""
from __future__ import annotations

import numpy as np

from x3d_tf_b200 import jpeg as J

SCALEBITS = 16
ONE_HALF = 1 << (SCALEBITS - 1)
CBCR_OFFSET = 128 << SCALEBITS


def FIX(x):
    return int(x * (1 << SCALEBITS) + 0.5)


def rgb_ycc(rgb):
    """[..., 3] uint8 -> Y, Cb, Cr int64 (jccolor.c: 16-bit fixed point, Cb/Cr with ONE_HALF - 1)."""
    r, g, b = (rgb[..., k].astype(np.int64) for k in range(3))
    y = (FIX(0.29900) * r + FIX(0.58700) * g + FIX(0.11400) * b + ONE_HALF) >> SCALEBITS
    cb = (-FIX(0.16874) * r - FIX(0.33126) * g + FIX(0.50000) * b + CBCR_OFFSET + ONE_HALF - 1) >> SCALEBITS
    cr = (FIX(0.50000) * r - FIX(0.41869) * g - FIX(0.08131) * b + CBCR_OFFSET + ONE_HALF - 1) >> SCALEBITS
    return y, cb, cr


def grid(H, W, hs):
    mcux, mcuy = -(-W // (8 * hs)), -(-H // (8 * hs))
    return mcux, mcuy, [(mcux * hs, mcuy * hs), (mcux, mcuy), (mcux, mcuy)]


def color_planes(img, hs):
    """The three sample planes the DCT reads, [bh*8, bw*8] each: full-resolution components with the
    last column / row replicated (expand_right_edge, expand_bottom_edge), chroma of 4:2:0 by
    h2v2_downsample (bias 1, 2 alternating by output column) and its last row replicated to the
    iMCU height.  Blocks of the luma grid past ceil(W/8) x ceil(H/8) are dummy blocks (not read)."""
    H, W, _ = img.shape
    _, _, dims = grid(H, W, hs)
    ycc = rgb_ycc(img)
    out = []
    for c, (bw, bh) in enumerate(dims):
        p = ycc[c]
        if c > 0 and hs == 2:
            cols = np.minimum(np.arange(bw * 16), W - 1)
            dh = -(-H // 2)
            rows = np.minimum(np.arange(2 * dh), H - 1)
            q = p[rows][:, cols]
            bias = 1 + (np.arange(bw * 8) & 1)
            d = (q[0::2, 0::2] + q[0::2, 1::2] + q[1::2, 0::2] + q[1::2, 1::2] + bias) >> 2
            out.append(d[np.minimum(np.arange(bh * 8), dh - 1)])
        else:
            out.append(p[np.minimum(np.arange(bh * 8), H - 1)][:, np.minimum(np.arange(bw * 8), W - 1)])
    return out


def _descale(x, n):
    return (x + (1 << (n - 1))) >> n


def _fdct_1d(d, pass2):
    """One pass of jpeg_fdct_islow over the last axis of d [..., 8] (int64)."""
    CB, P1 = 13, 2
    tmp0, tmp7 = d[..., 0] + d[..., 7], d[..., 0] - d[..., 7]
    tmp1, tmp6 = d[..., 1] + d[..., 6], d[..., 1] - d[..., 6]
    tmp2, tmp5 = d[..., 2] + d[..., 5], d[..., 2] - d[..., 5]
    tmp3, tmp4 = d[..., 3] + d[..., 4], d[..., 3] - d[..., 4]
    tmp10, tmp13, tmp11, tmp12 = tmp0 + tmp3, tmp0 - tmp3, tmp1 + tmp2, tmp1 - tmp2
    out = np.empty_like(d)
    if pass2:
        out[..., 0], out[..., 4] = _descale(tmp10 + tmp11, P1), _descale(tmp10 - tmp11, P1)
        n = CB + P1
    else:
        out[..., 0], out[..., 4] = (tmp10 + tmp11) << P1, (tmp10 - tmp11) << P1
        n = CB - P1
    z1 = (tmp12 + tmp13) * 4433
    out[..., 2] = _descale(z1 + tmp13 * 6270, n)
    out[..., 6] = _descale(z1 + tmp12 * -15137, n)
    z1, z2, z3, z4 = tmp4 + tmp7, tmp5 + tmp6, tmp4 + tmp6, tmp5 + tmp7
    z5 = (z3 + z4) * 9633
    tmp4, tmp5, tmp6, tmp7 = tmp4 * 2446, tmp5 * 16819, tmp6 * 25172, tmp7 * 12299
    z1, z2, z3, z4 = z1 * -7373, z2 * -20995, z3 * -16069 + z5, z4 * -3196 + z5
    out[..., 7] = _descale(tmp4 + z1 + z3, n)
    out[..., 5] = _descale(tmp5 + z2 + z4, n)
    out[..., 3] = _descale(tmp6 + z2 + z3, n)
    out[..., 1] = _descale(tmp7 + z1 + z4, n)
    return out


def fdct_islow(blocks):
    """[n, 64] samples (0..255, natural order) -> [n, 64] int64 FDCT output (scaled up by 8)."""
    d = blocks.reshape(-1, 8, 8).astype(np.int64) - 128
    d = _fdct_1d(d, False)                                           # rows
    d = _fdct_1d(d.transpose(0, 2, 1), True).transpose(0, 2, 1)      # columns
    return d.reshape(-1, 64)


def reciprocals(q):
    """jcdctmgr.c compute_reciprocal(q << 3) with a 16-bit DCTELEM: (recip, corr, shift) per entry."""
    q = np.asarray(q, np.int64).reshape(-1)
    recip, corr, shift = (np.zeros(q.size, np.int64) for _ in range(3))
    for i, qq in enumerate(q):
        d = int(qq) << 3
        b = d.bit_length() - 1
        r = 16 + b
        fq, fr, c = (1 << r) // d, (1 << r) % d, d // 2
        if fr == 0:
            fq >>= 1
            r -= 1
        elif fr <= d // 2:
            c += 1
        else:
            fq += 1
        recip[i], corr[i], shift[i] = fq, c, r - 16
    return recip, corr, shift


def quantize(dct, q):
    """jcdctmgr.c quantize: sign(x) * (((|x| + corr) * recip) >> (shift + 16))."""
    recip, corr, shift = reciprocals(q)
    a = np.abs(dct)
    v = ((a + corr) * recip) >> (shift + 16)
    return np.where(dct < 0, -v, v)


def coefficients(img, quality=90, chroma="420"):
    """Quantised coefficients [blocks, 64] int16 (natural order) in the decoder's layout: component
    after component, each block grid row-major, dummy blocks of the right and bottom MCUs included
    (AC zero, DC of the block before them in jccoefct.c's order)."""
    hs = J.CHROMA[chroma][0]
    H, W, _ = img.shape
    mcux, mcuy, dims = grid(H, W, hs)
    qt = J.quant_tables(quality)
    out = []
    for c, (p, (bw, bh)) in enumerate(zip(color_planes(img, hs), dims)):
        blocks = p.reshape(bh, 8, bw, 8).transpose(0, 2, 1, 3).reshape(bh, bw, 64)
        coef = quantize(fdct_islow(blocks.reshape(-1, 64)), qt[min(c, 1)]).reshape(bh, bw, 64)
        if c == 0 and hs == 2:
            wib, hib = -(-W // 8), -(-H // 8)
            for by in range(bh):
                for bx in range(bw):
                    if bx >= wib or by >= hib:
                        coef[by, bx] = 0
                        coef[by, bx, 0] = coef[min(by, hib - 1), min(bx | 1, wib - 1), 0]
        out.append(coef.reshape(-1, 64))
    return np.concatenate(out).astype(np.int16)


class _BitWriter:
    def __init__(self):
        self.bits = []

    def put(self, code, n):
        code, n = int(code), int(n)
        self.bits += [(code >> (n - 1 - i)) & 1 for i in range(n)]

    def flush(self):
        """flush_bits: pad with 1-bits to a byte, then stuff a 0x00 after every 0xFF."""
        self.bits += [1] * (-len(self.bits) % 8)
        raw = np.packbits(np.array(self.bits, np.uint8)).tobytes() if self.bits else b""
        return raw.replace(b"\xff", b"\xff\x00")


def scan_order(H, W, hs):
    """Block indices (into the coefficient layout) in scan order with their component."""
    mcux, mcuy, dims = grid(H, W, hs)
    n0, n1 = dims[0][0] * dims[0][1], mcux * mcuy
    order = []
    for my in range(mcuy):
        for mx in range(mcux):
            for by in range(hs):
                for bx in range(hs):
                    order.append(((my * hs + by) * dims[0][0] + mx * hs + bx, 0))
            order.append((n0 + my * mcux + mx, 1))
            order.append((n0 + n1 + my * mcux + mx, 2))
    return order


def entropy(coef, H, W, chroma="420"):
    """jchuff.c encode_one_block over the blocks in scan order: the stuffed entropy-coded segment."""
    hs = J.CHROMA[chroma][0]
    tabs = [J.huff_codes(*t) for t in J.STD_HUFF]                   # dc0, ac0, dc1, ac1
    bw = _BitWriter()
    last = [0, 0, 0]
    for b, c in scan_order(H, W, hs):
        blk = coef[b].astype(np.int64)[J.ZIGZAG]
        dco, dsi = tabs[0 if c == 0 else 2]
        aco, asi = tabs[1 if c == 0 else 3]
        t = int(blk[0]) - last[c]
        last[c] = int(blk[0])
        nb = abs(t).bit_length()
        bw.put(dco[nb], dsi[nb])
        if nb:
            bw.put((t - 1 if t < 0 else t) & ((1 << nb) - 1), nb)
        run = 0
        for k in range(1, 64):
            v = int(blk[k])
            if v == 0:
                run += 1
                continue
            while run > 15:
                bw.put(aco[0xF0], asi[0xF0])
                run -= 16
            nb = abs(v).bit_length()
            s = (run << 4) + nb
            bw.put(aco[s], asi[s])
            bw.put((v - 1 if v < 0 else v) & ((1 << nb) - 1), nb)
            run = 0
        if run:
            bw.put(aco[0], asi[0])
    return bw.flush()


def encode(img, quality=90, chroma="420"):
    """The whole JPEG file of one [H, W, 3] uint8 frame."""
    H, W, _ = img.shape
    seg = entropy(coefficients(img, quality, chroma), H, W, chroma)
    return J.encoder_header(H, W, quality, chroma) + seg + J.EOI
