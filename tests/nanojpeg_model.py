"""An independent integer model of NanoJPEG's decoder, and a baseline JPEG writer for crafted files (TEST INFRASTRUCTURE).

The decoder promises NanoJPEG's pixels bit for bit.  Its recorded answers (tests/golden/ref_digests.json) cover only the
files the tests had when they were made, and every other check compares the GPU with the CPU run of the same source
(jpeg_decode.cuh).  This module states NanoJPEG's algorithm a second time, from jpeg_dec.h (the line numbers are the
ones the decoder source quotes) and T.81, on whole planes in numpy:

  geometry   njDecodeSOF (:520-571): component size (W * ssx + ssxmax - 1) / ssxmax, padded stride mbwidth * ssx * 8, a
             single component forced to 1x1, and the rejections (ncomp, precision, sampling factors, narrow planes)
  IDCT       dequantise (:666), njRowIDCT (:350-396) and njColIDCT (:398-442) in int64, every intermediate asserted to
             fit in int32 (the reference is C: a wider value would be undefined behaviour there, so tests must avoid it)
  upsample   njUpsampleH (:736-763) with its read of the last three samples at the END OF THE PADDED ROW, njUpsampleV
             (:765-790), in njConvert's order (:817-836): per plane, H pass if too narrow then V pass if too short
  colour     njConvert's 8-bit YCbCr -> RGB (:838-852); gray drops the stride (:853-866)

It imports neither `oracle` nor `imagecodecs_b200`; it reads files through tests/jpeg_model.parse().
"""
import numpy as np

from tests import jpeg_model as jm

NJ_OK, NJ_NO_JPEG, NJ_UNSUPPORTED, NJ_OUT_OF_MEM, NJ_INTERNAL_ERR, NJ_SYNTAX_ERROR = range(6)

W1, W2, W3, W5, W6, W7 = 2841, 2676, 2408, 1609, 1108, 565       # 2048 * sqrt(2) * cos(k * pi / 16) (:343-348)


class Int32Overflow(AssertionError):
    """An IDCT intermediate left int32: NanoJPEG's result is undefined for this input, so no test may use it."""


def _i32(v):
    if v.size and (v.min() < -(1 << 31) or v.max() > (1 << 31) - 1):
        raise Int32Overflow("IDCT intermediate out of int32: [%d, %d]" % (v.min(), v.max()))
    return v


def _clip(v):                                          # njClip (:339-341)
    return np.clip(v, 0, 255)


def _butterfly(x0, x1, x2, x3, x4, x5, x6, x7, k):
    """The second stage both passes share; returns the eight sums before their final shift."""
    x8 = k(x0 + x1); x0 = k(x0 - x1)
    x1 = k(x4 + x6); x4 = k(x4 - x6); x6 = k(x5 + x7); x5 = k(x5 - x7)
    x7 = k(x8 + x3); x8 = k(x8 - x3); x3 = k(x0 + x2); x0 = k(x0 - x2)
    x2 = k(k(181 * k(x4 + x5)) + 128) >> 8
    x4 = k(k(181 * k(x4 - x5)) + 128) >> 8
    return [k(x7 + x1), k(x3 + x2), k(x0 + x4), k(x8 + x6), k(x8 - x6), k(x0 - x4), k(x3 - x2), k(x7 - x1)]


def _row_idct(b):
    """njRowIDCT on every row of b (int64 [n, 8]); rows keep 3 fraction bits."""
    k = _i32
    x1 = k(b[:, 4] << 11)
    flat = (x1 | b[:, 6] | b[:, 2] | b[:, 1] | b[:, 7] | b[:, 5] | b[:, 3]) == 0
    out = np.repeat(b[:, :1] << 3, 8, 1)
    r = b[~flat]
    x1, x2, x3, x4, x5, x6, x7 = r[:, 4] << 11, r[:, 6], r[:, 2], r[:, 1], r[:, 7], r[:, 5], r[:, 3]
    x0 = k(k(r[:, 0] << 11) + 128)
    x8 = k(W7 * k(x4 + x5))
    x4 = k(x8 + k((W1 - W7) * x4)); x5 = k(x8 - k((W1 + W7) * x5))
    x8 = k(W3 * k(x6 + x7))
    x6 = k(x8 - k((W3 - W5) * x6)); x7 = k(x8 - k((W3 + W5) * x7))
    x1_ = k(W6 * k(x3 + x2))
    x2 = k(x1_ - k((W2 + W6) * x2)); x3 = k(x1_ + k((W2 - W6) * x3))
    out[~flat] = np.stack(_butterfly(x0, x1, x2, x3, x4, x5, x6, x7, k), 1) >> 8
    return out


def _col_idct(b):
    """njColIDCT on every column of b (int64 [n, 8], a column per row of b) -> uint8 values, + 128 and clipped."""
    k = _i32
    x1 = k(b[:, 4] << 8)
    flat = (x1 | b[:, 6] | b[:, 2] | b[:, 1] | b[:, 7] | b[:, 5] | b[:, 3]) == 0
    out = np.repeat(_clip((k(b[:, :1] + 32) >> 6) + 128), 8, 1)
    r = b[~flat]
    x1, x2, x3, x4, x5, x6, x7 = r[:, 4] << 8, r[:, 6], r[:, 2], r[:, 1], r[:, 7], r[:, 5], r[:, 3]
    x0 = k(k(r[:, 0] << 8) + 8192)
    x8 = k(k(W7 * k(x4 + x5)) + 4)
    x4 = k(x8 + k((W1 - W7) * x4)) >> 3; x5 = k(x8 - k((W1 + W7) * x5)) >> 3
    x8 = k(k(W3 * k(x6 + x7)) + 4)
    x6 = k(x8 - k((W3 - W5) * x6)) >> 3; x7 = k(x8 - k((W3 + W5) * x7)) >> 3
    x1_ = k(k(W6 * k(x3 + x2)) + 4)
    x2 = k(x1_ - k((W2 + W6) * x2)) >> 3; x3 = k(x1_ + k((W2 - W6) * x3)) >> 3
    out[~flat] = _clip((np.stack(_butterfly(x0, x1, x2, x3, x4, x5, x6, x7, k), 1) >> 14) + 128)
    return out


def idct_plane(grid, qt):
    """Padded plane (uint8 [8 * rows, 8 * cols]) of one component: grid is int [rows, cols, 64] quantised coefficients in
    zigzag order, qt the component's table in stored (zigzag) order.  Coefficient k lands at natural index njZZ[k]."""
    rows, cols = grid.shape[:2]
    z = grid.reshape(-1, 64).astype(np.int64) * np.asarray(qt, np.int64)
    nat = z[:, jm.ZZ]                                  # natural index i holds zigzag position ZZ[i]
    rowpass = _row_idct(nat.reshape(-1, 8)).reshape(-1, 8, 8)
    cols_ = _col_idct(rowpass.transpose(0, 2, 1).reshape(-1, 8)).reshape(-1, 8, 8).transpose(0, 2, 1)
    return cols_.reshape(rows, cols, 8, 8).transpose(0, 2, 1, 3).reshape(8 * rows, 8 * cols).astype(np.uint8)


def _cf(v):                                            # CF(x) = njClip(((x) + 64) >> 7) (:722-734)
    return _clip((v + 64) >> 7)


def upsample_h(plane, w):
    """njUpsampleH: plane is [h, stride] (stride >= w); returns [h, 2w].  The last three outputs read the last three
    bytes of the PADDED row (lin += stride, then lin[-1..-3])."""
    l = plane.astype(np.int64)
    out = np.empty((l.shape[0], 2 * w), np.int64)
    out[:, 0] = _cf(139 * l[:, 0] - 11 * l[:, 1])
    out[:, 1] = _cf(104 * l[:, 0] + 27 * l[:, 1] - 3 * l[:, 2])
    out[:, 2] = _cf(28 * l[:, 0] + 109 * l[:, 1] - 9 * l[:, 2])
    n = w - 3
    a, b, c, d = l[:, 0:n], l[:, 1:n + 1], l[:, 2:n + 2], l[:, 3:n + 3]
    out[:, 3:2 * n + 3:2] = _cf(-9 * a + 111 * b + 29 * c - 3 * d)
    out[:, 4:2 * n + 4:2] = _cf(-3 * a + 29 * b + 111 * c - 9 * d)
    t1, t2, t3 = l[:, -1], l[:, -2], l[:, -3]
    out[:, 2 * w - 3] = _cf(28 * t1 + 109 * t2 - 9 * t3)
    out[:, 2 * w - 2] = _cf(104 * t1 + 27 * t2 - 3 * t3)
    out[:, 2 * w - 1] = _cf(139 * t1 - 11 * t2)
    return out.astype(np.uint8)


def upsample_v(plane, w, h):
    """njUpsampleV: rows 0..h-1 of plane ([>= h, stride]), columns 0..w-1; returns [2h, w].  The last three outputs read
    the last LOGICAL rows."""
    r = plane[:h, :w].astype(np.int64)
    out = np.empty((2 * h, w), np.int64)
    out[0] = _cf(139 * r[0] - 11 * r[1])
    out[1] = _cf(104 * r[0] + 27 * r[1] - 3 * r[2])
    out[2] = _cf(28 * r[0] + 109 * r[1] - 9 * r[2])
    n = h - 3
    a, b, c, d = r[0:n], r[1:n + 1], r[2:n + 2], r[3:n + 3]
    out[3:2 * n + 3:2] = _cf(-9 * a + 111 * b + 29 * c - 3 * d)
    out[4:2 * n + 4:2] = _cf(-3 * a + 29 * b + 111 * c - 9 * d)
    out[2 * h - 3] = _cf(28 * r[h - 1] + 109 * r[h - 2] - 9 * r[h - 3])
    out[2 * h - 2] = _cf(104 * r[h - 1] + 27 * r[h - 2] - 3 * r[h - 3])
    out[2 * h - 1] = _cf(139 * r[h - 1] - 11 * r[h - 2])
    return out.astype(np.uint8)


def geometry(width, height, factors, precision=8, marker=0xC0):
    """njDecodeSOF's verdict and geometry.  factors: [(ssx, ssy)] as declared.  Returns an NJ_* error code, or a dict with
    mbwidth, mbheight and per component ssx, ssy (after the 1x1 rule for one component), width, height, stride, and the
    block grid (rows, cols)."""
    if marker != 0xC0:
        return NJ_UNSUPPORTED                          # njDecode's marker loop: only SOF0 (:891-905)
    if precision != 8:
        return NJ_UNSUPPORTED
    if not width or not height:
        return NJ_SYNTAX_ERROR
    if len(factors) not in (1, 3):
        return NJ_UNSUPPORTED
    for ssx, ssy in factors:                           # checked in this order per component
        if not ssx:
            return NJ_SYNTAX_ERROR
        if ssx & (ssx - 1):
            return NJ_UNSUPPORTED
        if not ssy:
            return NJ_SYNTAX_ERROR
        if ssy & (ssy - 1):
            return NJ_UNSUPPORTED
    if len(factors) == 1:
        factors = [(1, 1)]
    sxm, sym = max(f[0] for f in factors), max(f[1] for f in factors)
    mbw, mbh = -(-width // (8 * sxm)), -(-height // (8 * sym))
    comps = []
    for ssx, ssy in factors:
        cw, ch = (width * ssx + sxm - 1) // sxm, (height * ssy + sym - 1) // sym
        if (cw < 3 and ssx != sxm) or (ch < 3 and ssy != sym):
            return NJ_UNSUPPORTED
        comps.append(dict(ssx=ssx, ssy=ssy, width=cw, height=ch, stride=mbw * ssx * 8, grid=(mbh * ssy, mbw * ssx)))
    return dict(mbwidth=mbw, mbheight=mbh, comps=comps)


def decode_blocks(width, height, factors, qtabs, grids, precision=8, marker=0xC0):
    """NanoJPEG's pixels (uint8 [h, w, 3] or [h, w]) or its NJ_* error code, from coefficients and geometry.

    grids[c]: int [rows, cols, 64] quantised coefficients of component c in zigzag order, DC already un-differenced, over
    its padded block grid (geometry()['comps'][c]['grid']); qtabs[c]: its quantiser table in stored (zigzag) order."""
    g = geometry(width, height, factors, precision, marker)
    if not isinstance(g, dict):
        return g
    planes = []
    for k, grid, qt in zip(g["comps"], grids, qtabs):
        assert tuple(grid.shape) == k["grid"] + (64,), (grid.shape, k["grid"])
        p, w, h = idct_plane(grid, qt), k["width"], k["height"]
        while w < width or h < height:                 # njConvert (:817-836)
            if w < width:
                p = upsample_h(p[:h], w)
                w *= 2
            if h < height:
                p = upsample_v(p, w, h)
                h *= 2
        planes.append(p[:height, :width].astype(np.int64))
    if len(planes) == 1:
        return planes[0].astype(np.uint8)
    y, cb, cr = planes[0] << 8, planes[1] - 128, planes[2] - 128
    rgb = [(y + 359 * cr + 128) >> 8, (y - 88 * cb - 183 * cr + 128) >> 8, (y + 454 * cb + 128) >> 8]
    return _clip(np.stack(rgb, -1)).astype(np.uint8)


def grids_of(parsed):
    """Per-component coefficient grids (decode_blocks' layout) from jm.parse() output (stream order)."""
    sof = parsed["sof"]
    comps = sof["comps"]
    if len(comps) == 1:
        cols, rows = -(-sof["width"] // 8), -(-sof["height"] // 8)
        return [parsed["coefs"].reshape(rows, cols, 64)]
    hmax, vmax = max(c[1] for c in comps), max(c[2] for c in comps)
    mbw, mbh = -(-sof["width"] // (8 * hmax)), -(-sof["height"] // (8 * vmax))
    out = []
    for ci, (_, h, v, _) in enumerate(comps):
        b = parsed["coefs"][parsed["comp"] == ci].reshape(mbh, mbw, v, h, 64)
        out.append(b.transpose(0, 2, 1, 3, 4).reshape(mbh * v, mbw * h, 64))
    return out


def decode_parsed(parsed):
    """decode_blocks() of a file read by jm.parse() (which only reads 8-bit SOF0 files)."""
    sof = parsed["sof"]
    comps = sof["comps"]
    factors = [(c[1], c[2]) for c in comps]
    g = geometry(sof["width"], sof["height"], factors, sof["precision"])
    if not isinstance(g, dict):
        return g
    return decode_blocks(sof["width"], sof["height"], factors, [parsed["dqt"][c[3]] for c in comps], grids_of(parsed))


def decode(jpeg):
    """The model's pixels for a well-formed baseline file (fill bits are not checked: NanoJPEG ignores them)."""
    return decode_parsed(jm.parse(jpeg, padding=None))


# ---------------------------------------------------------------------------------------------------------------
# A baseline writer for crafted files: any sampling factors, component count, precision byte and SOF marker
# ---------------------------------------------------------------------------------------------------------------
def _complete_table(n_symbols, length):
    bits = [0] * 16
    bits[length - 1] = n_symbols
    return bytes(bits)


# A complete custom table pair: every DC category 0..15 (5-bit codes) and every AC symbol with categories 1..15, plus EOB
# and ZRL (8-bit codes).  Neither has an all-ones code.  jm.parse() stops at DC 11 / AC 10, the K.3 limits.
_AC_ALL = bytes([0x00, 0xF0] + [(r << 4) | s for r in range(16) for s in range(1, 16)])
HUFFMAN_FULL = {(0, 0): (_complete_table(16, 5), bytes(range(16))), (0, 1): (_complete_table(16, 5), bytes(range(16))),
                (1, 0): (_complete_table(len(_AC_ALL), 8), _AC_ALL), (1, 1): (_complete_table(len(_AC_ALL), 8), _AC_ALL)}


def _codes(bits, vals):
    """symbol -> (code, length) of a canonical Huffman table (T.81 C.2)."""
    out, code, k = {}, 0, 0
    for l in range(1, 17):
        for _ in range(bits[l - 1]):
            out[vals[k]] = (code, l)
            code += 1
            k += 1
        code <<= 1
    return out


class _Bits:
    def __init__(self):
        self.out = bytearray()
        self.acc = 0
        self.n = 0

    def put(self, v, n):
        self.acc = (self.acc << n) | (v & ((1 << n) - 1))
        self.n += n
        while self.n >= 8:
            self.n -= 8
            b = (self.acc >> self.n) & 0xFF
            self.out.append(b)
            if b == 0xFF:
                self.out.append(0)                     # byte stuffing (T.81 F.1.2.3)
        self.acc &= (1 << self.n) - 1

    def flush(self):                                   # fill with 1-bits to the byte boundary
        if self.n:
            self.put((1 << (8 - self.n)) - 1, 8 - self.n)


def _category(v):
    return int(abs(int(v))).bit_length()


def stream_order(width, height, factors, grids):
    """[blocks, 64] in scan order (one component: raster; several: MCU by MCU, component by component, ssy x ssx each)."""
    if len(grids) == 1:
        return grids[0].reshape(-1, 64)
    hmax, vmax = max(f[0] for f in factors), max(f[1] for f in factors)
    mbw, mbh = -(-width // (8 * hmax)), -(-height // (8 * vmax))
    parts = [g.reshape(mbh, v, mbw, h, 64).transpose(0, 2, 1, 3, 4).reshape(mbh, mbw, h * v, 64)
             for g, (h, v) in zip(grids, factors)]
    return np.concatenate(parts, 2).reshape(-1, 64)


def write(width, height, factors, qtabs, grids, dri=0, tables=None, precision=8, marker=0xC0):
    """A baseline JPEG file: SOI, DQT, SOFn, DHT, [DRI], SOS, byte-stuffed scan with RSTm every `dri` MCUs (1-bit fill
    before each), EOI.  Component c has id c + 1, quantiser table c, Huffman tables 0 (c == 0) or 1.  grids as in
    decode_blocks(); a component with a zero factor contributes no blocks.  tables: jm.HUFFMAN_K3 (default) or
    HUFFMAN_FULL."""
    tables = tables or jm.HUFFMAN_K3
    nc = len(factors)
    f = bytearray(b"\xff\xd8")
    for c in range(nc):
        f += b"\xff\xdb\x00\x43" + bytes([c]) + bytes(int(q) for q in qtabs[c])
    f += bytes([0xFF, marker]) + (8 + 3 * nc).to_bytes(2, "big") + bytes([precision]) + height.to_bytes(2, "big") + width.to_bytes(2, "big")
    f += bytes([nc]) + b"".join(bytes([c + 1, (h << 4) | v, c]) for c, (h, v) in enumerate(factors))
    for (tc, th), (bits, vals) in sorted(tables.items()):
        f += b"\xff\xc4" + (19 + len(vals)).to_bytes(2, "big") + bytes([(tc << 4) | th]) + bits + vals
    if dri:
        f += b"\xff\xdd\x00\x04" + dri.to_bytes(2, "big")
    f += b"\xff\xda" + (6 + 2 * nc).to_bytes(2, "big") + bytes([nc])
    f += b"".join(bytes([c + 1, 0x00 if c == 0 else 0x11]) for c in range(nc)) + b"\x00\x3f\x00"
    codes = {k: _codes(*v) for k, v in tables.items()}
    if nc == 1:
        units, n_mcus = [0], grids[0].shape[0] * grids[0].shape[1]
    else:
        units = [c for c, (h, v) in enumerate(factors) for _ in range(h * v)]
        hmax, vmax = max(x[0] for x in factors), max(x[1] for x in factors)
        n_mcus = -(-width // (8 * hmax)) * -(-height // (8 * vmax))
    blocks = stream_order(width, height, factors, grids) if nc != 1 else grids[0].reshape(-1, 64)
    assert len(blocks) == n_mcus * len(units)
    bw = _Bits()
    pred = [0] * nc
    blk = 0
    for m in range(n_mcus):
        if dri and m and m % dri == 0:
            bw.flush()
            bw.out += bytes([0xFF, 0xD0 + (m // dri - 1) % 8])
            pred = [0] * nc
        for c in units:
            dc_codes, ac_codes = codes[(0, min(c, 1))], codes[(1, min(c, 1))]
            z = [int(v) for v in blocks[blk]]
            blk += 1
            diff = z[0] - pred[c]
            pred[c] = z[0]
            s = _category(diff)
            bw.put(*dc_codes[s])
            if s:
                bw.put(diff if diff > 0 else diff + (1 << s) - 1, s)
            run = 0
            for k in range(1, 64):
                v = z[k]
                if v == 0:
                    run += 1
                    continue
                while run > 15:
                    bw.put(*ac_codes[0xF0])
                    run -= 16
                s = _category(v)
                bw.put(*ac_codes[(run << 4) | s])
                bw.put(v if v > 0 else v + (1 << s) - 1, s)
                run = 0
            if run:
                bw.put(*ac_codes[0x00])
    bw.flush()
    return bytes(f + bw.out + b"\xff\xd9")
