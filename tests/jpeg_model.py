"""An independent float64 model of the encoder, and a strict baseline-JPEG reader (TEST INFRASTRUCTURE).

The oracle (oracle/jpeg_oracle.c) restates the kernels' float32 arithmetic operation for operation, so a rule that both
state wrongly (a table, the IJG scale, a colour constant, the 2x2 chroma mean, edge replication, block order, zigzag)
passes every kernel-against-oracle test.  This module states the same transform a second way, from the definitions:
edge-replicated MCUs, RGB->YCbCr in float64, an orthonormal DCT-II as a matrix product, division by the quantiser.  Its
coefficients are exact up to float64 rounding; the kernels' float32 AAN DCT lands on the same integers except next to a
.5 boundary (check_quantised).

It imports neither `oracle` nor `imagecodecs_b200`: only the tables below, typed in from their sources.
"""
import numpy as np

# ---------------------------------------------------------------------------------------------------------------
# Tables
# ---------------------------------------------------------------------------------------------------------------
# ZZ[natural index] = position in the zigzag scan (jpeg_enc.h:376-386)
ZZ = np.array([0, 1, 5, 6, 14, 15, 27, 28, 2, 4, 7, 13, 16, 26, 29, 42,
               3, 8, 12, 17, 25, 30, 41, 43, 9, 11, 18, 24, 31, 40, 44, 53,
               10, 19, 23, 32, 39, 45, 52, 54, 20, 22, 33, 38, 46, 51, 55, 60,
               21, 34, 37, 47, 50, 56, 59, 61, 35, 36, 48, 49, 57, 58, 62, 63])
# The reference's two base tables in the order it stores them (= DQT order; DESIGN.md section 2).  Luma is Annex K.1;
# chroma is the reference's "from paper" table (jpeg_enc.h:294-305), not Annex K.2.
BASE_LUMA = np.array([16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55,
                      14, 13, 16, 24, 40, 57, 69, 56, 14, 17, 22, 29, 51, 87, 80, 62,
                      18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113, 92,
                      49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99])
BASE_CHROMA = np.array([16, 12, 14, 14, 18, 24, 49, 72, 11, 10, 16, 24, 40, 51, 61, 12,
                        13, 17, 22, 35, 64, 92, 14, 16, 22, 37, 55, 78, 95, 19, 24, 29,
                        56, 64, 87, 98, 26, 40, 51, 68, 81, 103, 112, 58, 57, 87, 109, 104,
                        121, 100, 60, 69, 80, 103, 113, 120, 103, 55, 56, 62, 77, 92, 101, 99])

# ITU-T T.81 Annex K.3: the typical Huffman tables as (BITS, HUFFVAL), keyed by (table class, destination).
_AC_LUMA_VALS = bytes.fromhex(
    "01020300041105122131410613516107227114328191a1082342b1c11552d1f0"
    "2433627282090a161718191a25262728292a3435363738393a434445464748494a"
    "535455565758595a636465666768696a737475767778797a838485868788898a"
    "92939495969798999aa2a3a4a5a6a7a8a9aab2b3b4b5b6b7b8b9bac2c3c4c5c6"
    "c7c8c9cad2d3d4d5d6d7d8d9dae1e2e3e4e5e6e7e8e9eaf1f2f3f4f5f6f7f8f9fa")
_AC_CHROMA_VALS = bytes.fromhex(
    "0001020311040521310612415107617113223281081442" "91a1b1c109233352f0"
    "156272d10a162434e125f11718191a262728292a35363738393a434445464748"
    "494a535455565758595a636465666768696a737475767778797a828384858687"
    "88898a92939495969798999aa2a3a4a5a6a7a8a9aab2b3b4b5b6b7b8b9bac2c3"
    "c4c5c6c7c8c9cad2d3d4d5d6d7d8d9dae2e3e4e5e6e7e8e9eaf2f3f4f5f6f7f8f9fa")
HUFFMAN_K3 = {
    (0, 0): (bytes([0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0]), bytes(range(12))),
    (0, 1): (bytes([0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0]), bytes(range(12))),
    (1, 0): (bytes([0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d]), _AC_LUMA_VALS),
    (1, 1): (bytes([0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77]), _AC_CHROMA_VALS),
}

QMODE_TJE, QMODE_IJG = 0, 1
SUB_444, SUB_420 = 0, 1


def quant_tables(qmode, quality):
    """(luma, chroma) quantiser tables in stored (zigzag, DQT) order, from the rules of DESIGN.md section 2.

    tje quality 3: all ones; 2: base // 10; 1: the base tables (zeros raised to 1).  IJG quality Q:
    s = 5000 // Q below 50, else 200 - 2Q; entry = clamp((base * s + 50) // 100, 1, 255)."""
    if qmode == QMODE_TJE:
        if quality not in (1, 2, 3):
            raise ValueError("tje quality is 1..3")
        if quality == 3:
            return np.ones(64, np.int64), np.ones(64, np.int64)
        d = 10 if quality == 2 else 1
        return np.maximum(BASE_LUMA // d, 1), np.maximum(BASE_CHROMA // d, 1)
    if not 1 <= quality <= 100:
        raise ValueError("IJG quality is 1..100")
    s = 5000 // quality if quality < 50 else 200 - 2 * quality
    return tuple(np.clip((b * s + 50) // 100, 1, 255) for b in (BASE_LUMA, BASE_CHROMA))


# ---------------------------------------------------------------------------------------------------------------
# Forward model
# ---------------------------------------------------------------------------------------------------------------
_k = np.arange(8)
# orthonormal DCT-II: F = D x D^T, x = D^T F D
DCT = np.cos((2 * _k[None, :] + 1) * _k[:, None] * np.pi / 16) * np.where(_k == 0, np.sqrt(0.125), 0.5)[:, None]


def _blocks(plane):
    """[H, W] (multiples of 8) -> [H/8, W/8, 8, 8]."""
    H, W = plane.shape
    return plane.reshape(H // 8, 8, W // 8, 8).transpose(0, 2, 1, 3)


def _fdct_quantise(plane, qt):
    """Unrounded quantised coefficients of every block of `plane`: [by, bx, 64] in zigzag order."""
    F = DCT @ _blocks(plane) @ DCT.T
    v = F.reshape(F.shape[:2] + (64,)) / qt[ZZ]          # natural index i is quantised by qt[zz[i]]
    z = np.empty_like(v)
    z[..., ZZ] = v                                        # and lands at zigzag position zz[i]
    return z


def exact_coefficients(img, qmode, quality, sub=SUB_444):
    """float64 [blocks, 64]: the unrounded quantised coefficients of `img` (uint8 [h,w] / [h,w,1|3|4]), zigzag order,
    blocks in stream order (4:4:4: Y Cb Cr per MCU; 4:2:0: Y00 Y01 Y10 Y11 Cb Cr; gray: Y).  Alpha is ignored."""
    img = np.asarray(img)
    if img.ndim == 2:
        img = img[..., None]
    h, w, nc = img.shape
    sub = sub if nc != 1 else SUB_444
    mcu = 16 if sub == SUB_420 else 8
    H, W = -(-h // mcu) * mcu, -(-w // mcu) * mcu
    p = np.pad(img[..., :3].astype(np.float64), ((0, H - h), (0, W - w), (0, 0)), mode="edge")   # edge replication
    ql, qc = quant_tables(qmode, quality)
    if nc == 1:
        return _fdct_quantise(p[..., 0] - 128.0, ql).reshape(-1, 64)
    r, g, b = p[..., 0], p[..., 1], p[..., 2]
    y = 0.299 * r + 0.587 * g + 0.114 * b - 128.0      # the reference's constants (jpeg_enc.h:1118-1120)
    cb = -0.1687 * r - 0.3313 * g + 0.5 * b
    cr = 0.5 * r - 0.4187 * g - 0.0813 * b
    if sub == SUB_420:
        cb, cr = [(c[0::2, 0::2] + c[0::2, 1::2] + c[1::2, 0::2] + c[1::2, 1::2]) / 4.0 for c in (cb, cr)]
    zy, zcb, zcr = _fdct_quantise(y, ql), _fdct_quantise(cb, qc), _fdct_quantise(cr, qc)
    if sub == SUB_444:
        return np.stack([zy, zcb, zcr], 2).reshape(-1, 64)
    my, mx = zcb.shape[:2]
    zy = zy.reshape(my, 2, mx, 2, 64).transpose(0, 2, 1, 3, 4).reshape(my, mx, 4, 64)
    return np.concatenate([zy, zcb[:, :, None], zcr[:, :, None]], 2).reshape(-1, 64)


def check_quantised(got, exact, delta=1e-3, what=""):
    """Assert that integer coefficients `got` are `exact` rounded half up, except next to a .5 boundary.

    The kernels (and the oracle) compute a float32 AAN DCT, multiply by a float32 reciprocal quantiser and round
    (v + 1024) + 0.5 with two float roundings, so a value that lies within their float32 error of k + .5 may land on
    either k or k + 1.  (v + 1024) alone is rounded to a float32 step of 1.2e-4 between 1024 and 2048, so at unit
    quantisers a disagreement up to ~6e-5 from .5 is expected from that rounding, plus the AAN error.  Measured: over
    3.8 M coefficients (4:4:4 tje-3 noise, gray, 4:2:0 q75..q100, 1080p) the largest distance from .5 at which the
    float32 result and the float64 rounding differ was 6.3e-5 (delta = 1e-3 is x16 that); over the 72 M coefficients
    of tests/test_model.py's grid plus ten 1080p photo / noise images in every layout, 1.1e-4 (x9).  Everywhere else
    the two must agree exactly: a wrong table, constant or sample rule moves coefficients by whole steps at distances
    far from .5."""
    got = np.asarray(got, dtype=np.float64).reshape(-1, 64)
    exact = np.asarray(exact, dtype=np.float64).reshape(-1, 64)
    assert got.shape == exact.shape, "%s: %s coefficients against %s" % (what, got.shape, exact.shape)
    lo = np.floor(exact)
    dist = np.abs(exact - lo - 0.5)
    ok = (got == np.floor(exact + 0.5)) | ((dist < delta) & ((got == lo) | (got == lo + 1)))
    if ok.all():
        return
    bad = np.argwhere(~ok)
    first = ", ".join("(%d,%d): got %d want %.4f" % (b, k, got[b, k], exact[b, k]) for b, k in bad[:6])
    raise AssertionError("%s: %d of %d coefficients off; nearest to .5 at %.3g; worst |got-exact| %.3g; first %s"
                         % (what, len(bad), got.size, dist[~ok].min(), np.abs(got - exact)[~ok].max(), first))


# ---------------------------------------------------------------------------------------------------------------
# Strict baseline-JPEG reader
# ---------------------------------------------------------------------------------------------------------------
class JpegSyntaxError(ValueError):
    pass


def _huff_lut(bits, vals):
    """16-bit look-ahead table of a canonical Huffman code (T.81 Annex C): lut[w] = (symbol, length); length 0 marks a
    window that starts with no code of the table."""
    sym = np.full(1 << 16, -1, np.int32)
    ln = np.zeros(1 << 16, np.int32)
    code, k = 0, 0
    for l in range(1, 17):
        for _ in range(bits[l - 1]):
            if code >= (1 << l):
                raise JpegSyntaxError("over-subscribed Huffman table")
            lo = code << (16 - l)
            sym[lo:lo + (1 << (16 - l))] = vals[k]
            ln[lo:lo + (1 << (16 - l))] = l
            code += 1
            k += 1
        code <<= 1
    return sym, ln


def _unstuff(data, pos, expect_rst):
    """Entropy-coded bytes from `pos` up to the next marker.  Returns (bytes, position of the marker).  0xFF must be
    followed by 00 (a stuffed data byte), the expected RSTm, or EOI."""
    out = bytearray()
    n = len(data)
    while True:
        j = data.find(b"\xff", pos)
        if j < 0 or j + 1 >= n:
            raise JpegSyntaxError("entropy-coded data runs off the end of the file")
        out += data[pos:j]
        nxt = data[j + 1]
        if nxt == 0:
            out.append(0xFF)
            pos = j + 2
            continue
        if nxt == 0xD9 or (expect_rst is not None and nxt == 0xD0 + expect_rst):
            return bytes(out), j
        raise JpegSyntaxError("0xFF %02X at offset %d inside entropy-coded data (expected 00%s or EOI)"
                              % (nxt, j, "" if expect_rst is None else ", RST%d" % expect_rst))


def parse(jpeg, padding="ours"):
    """Read a baseline sequential JPEG (SOF0, one scan) completely and strictly.

    Returns a dict with
      markers  list of marker codes in file order (0xD8 SOI ... 0xD9 EOI; RSTm included)
      dqt      {table id: int array [64], stored (zigzag) order}
      dht      {(class, id): (BITS bytes[16], HUFFVAL bytes)}
      sof      dict(precision, height, width, comps=[(id, h, v, tq)])
      sos      dict(comps=[(id, td, ta)], ss, se, ahal)
      dri      restart interval in MCUs (0 without DRI)
      coefs    int32 [blocks, 64], zigzag order, stream order, DC un-differenced
      comp     int32 [blocks], the SOF index of each block's component
      pads     list of (nbits, value) of the fill bits that end each interval
    padding: "ours" -- with DRI every interval is padded with 1-bits, without DRI the last byte with 0-bits (what this
    encoder, the oracle and the reference write); "ones" -- every interval with 1-bits (T.81 F.1.2.3, libjpeg); None --
    not checked.  Raises JpegSyntaxError on anything else."""
    d = bytes(jpeg)
    if d[:2] != b"\xff\xd8":
        raise JpegSyntaxError("no SOI")
    res = dict(markers=[0xD8], dqt={}, dht={}, sof=None, sos=None, dri=0, pads=[])
    pos = 2
    while True:
        if pos + 4 > len(d) or d[pos] != 0xFF:
            raise JpegSyntaxError("expected a marker at offset %d" % pos)
        m = d[pos + 1]
        ln = (d[pos + 2] << 8) | d[pos + 3]
        seg = d[pos + 4:pos + 2 + ln]
        if ln < 2 or len(seg) != ln - 2:
            raise JpegSyntaxError("segment %02X runs off the end" % m)
        res["markers"].append(m)
        pos += 2 + ln
        if m == 0xDB:
            k = 0
            while k < len(seg):
                if seg[k] >> 4:
                    raise JpegSyntaxError("16-bit DQT in a baseline file")
                res["dqt"][seg[k] & 15] = np.frombuffer(seg[k + 1:k + 65], np.uint8).astype(np.int64)
                k += 65
            if k != len(seg):
                raise JpegSyntaxError("DQT length")
        elif m == 0xC4:
            k = 0
            while k < len(seg):
                tc, th = seg[k] >> 4, seg[k] & 15
                bits = seg[k + 1:k + 17]
                nv = sum(bits)
                res["dht"][(tc, th)] = (bytes(bits), bytes(seg[k + 17:k + 17 + nv]))
                k += 17 + nv
            if k != len(seg):
                raise JpegSyntaxError("DHT length")
        elif m == 0xC0:
            nc = seg[5]
            if seg[0] != 8 or len(seg) != 6 + 3 * nc:
                raise JpegSyntaxError("SOF0")
            comps = [(seg[6 + 3 * i], seg[7 + 3 * i] >> 4, seg[7 + 3 * i] & 15, seg[8 + 3 * i]) for i in range(nc)]
            res["sof"] = dict(precision=seg[0], height=(seg[1] << 8) | seg[2], width=(seg[3] << 8) | seg[4], comps=comps)
        elif 0xC1 <= m <= 0xCF and m not in (0xC4, 0xC8, 0xCC):
            raise JpegSyntaxError("not a baseline file (SOF%d)" % (m - 0xC0))
        elif m == 0xDD:
            if len(seg) != 2:
                raise JpegSyntaxError("DRI length")
            res["dri"] = (seg[0] << 8) | seg[1]
        elif m == 0xDA:
            ns = seg[0]
            if len(seg) != 4 + 2 * ns:
                raise JpegSyntaxError("SOS length")
            res["sos"] = dict(comps=[(seg[1 + 2 * i], seg[2 + 2 * i] >> 4, seg[2 + 2 * i] & 15) for i in range(ns)],
                              ss=seg[1 + 2 * ns], se=seg[2 + 2 * ns], ahal=seg[3 + 2 * ns])
            break
        elif not (0xE0 <= m <= 0xEF or m == 0xFE):
            raise JpegSyntaxError("unexpected marker %02X before the scan" % m)
    sof, sos = res["sof"], res["sos"]
    if sof is None:
        raise JpegSyntaxError("scan before SOF0")
    if (sos["ss"], sos["se"], sos["ahal"]) != (0, 63, 0):
        raise JpegSyntaxError("not a sequential scan")

    # geometry of the scan (T.81 A.2)
    W, H = sof["width"], sof["height"]
    hmax = max(c[1] for c in sof["comps"]); vmax = max(c[2] for c in sof["comps"])
    index = {c[0]: i for i, c in enumerate(sof["comps"])}
    units = []                                    # per MCU: (component index, dc lut, ac lut) for each data unit
    luts = {}

    def lut(cls, tid):
        if (cls, tid) not in luts:
            if (cls, tid) not in res["dht"]:
                raise JpegSyntaxError("scan uses undefined Huffman table %d/%d" % (cls, tid))
            luts[(cls, tid)] = _huff_lut(*res["dht"][(cls, tid)])
        return luts[(cls, tid)]
    for cid, td, ta in sos["comps"]:
        if cid not in index:
            raise JpegSyntaxError("scan component %d not in SOF" % cid)
        ci = index[cid]
        if sof["comps"][ci][3] not in res["dqt"]:
            raise JpegSyntaxError("component %d uses an undefined quantiser table" % cid)
        n = sof["comps"][ci][1] * sof["comps"][ci][2] if len(sos["comps"]) > 1 else 1
        units += [(ci, lut(0, td), lut(1, ta))] * n
    if len(sos["comps"]) > 1:
        total = (-(-W // (8 * hmax))) * (-(-H // (8 * vmax)))
    else:
        c = sof["comps"][index[sos["comps"][0][0]]]
        total = (-(-(-(-W * c[1] // hmax)) // 8)) * (-(-(-(-H * c[2] // vmax)) // 8))
    interval = res["dri"] or total

    coefs = np.zeros((total * len(units), 64), np.int32)
    comp = np.tile(np.array([u[0] for u in units], np.int32), total)
    mcu = 0
    blk = 0
    while mcu < total:
        k = mcu // interval
        last = mcu + interval >= total
        data, mpos = _unstuff(d, pos, None if last else k & 7)
        end_marker = d[mpos + 1]
        if last != (end_marker == 0xD9):
            raise JpegSyntaxError("scan ends after %d of %d MCUs" % (mcu + interval if not last else mcu, total)
                                  if end_marker == 0xD9 else "RST after the last interval")
        # zero bits after the data: one block reads at most 64 * (16 + 11) bits, checked after each block
        nbits = 8 * len(data)
        bits = np.unpackbits(np.frombuffer(data + bytes(260), np.uint8)).astype(np.uint32)
        win = np.zeros(nbits + 2048, np.uint32)
        for b in range(16):
            win += bits[b:b + nbits + 2048] << (15 - b)
        win = win.tolist()
        p = 0
        pred = [0] * len(sof["comps"])
        for _ in range(min(interval, total - mcu)):
            for ci, (dsym, dlen), (asym, alen) in units:
                w_ = win[p]
                t, l = int(dsym[w_]), int(dlen[w_])
                if l == 0:
                    raise JpegSyntaxError("DC code not in the table at bit %d of interval %d" % (p, k))
                if t > 11:
                    raise JpegSyntaxError("DC category %d" % t)
                p += l
                diff = 0
                if t:
                    v = win[p] >> (16 - t)
                    diff = v if v >> (t - 1) else v - (1 << t) + 1
                    p += t
                pred[ci] += diff
                row = coefs[blk]
                row[0] = pred[ci]
                z = 1
                while z < 64:
                    w_ = win[p]
                    rs, l = int(asym[w_]), int(alen[w_])
                    if l == 0:
                        raise JpegSyntaxError("AC code not in the table at bit %d of interval %d" % (p, k))
                    p += l
                    r, s = rs >> 4, rs & 15
                    if s == 0:
                        if r == 15:
                            z += 16
                            if z > 64:
                                raise JpegSyntaxError("ZRL runs past position 63")
                            continue
                        if r:
                            raise JpegSyntaxError("AC symbol %02X" % rs)
                        break                                     # EOB
                    if s > 10:
                        raise JpegSyntaxError("AC category %d" % s)
                    z += r
                    if z > 63:
                        raise JpegSyntaxError("AC run past position 63")
                    v = win[p] >> (16 - s)
                    row[z] = v if v >> (s - 1) else v - (1 << s) + 1
                    p += s
                    z += 1
                if p > nbits:
                    raise JpegSyntaxError("entropy-coded data ends inside MCU %d" % mcu)
                blk += 1
            mcu += 1
        fill = nbits - p
        if fill > 7:
            raise JpegSyntaxError("%d bits after the last MCU of interval %d" % (fill, k))
        val = int(win[p] >> (16 - fill)) if fill else 0
        res["pads"].append((fill, val))
        if fill and padding is not None:
            ones = (padding == "ones") or res["dri"] > 0
            if val != ((1 << fill) - 1 if ones else 0):
                raise JpegSyntaxError("interval %d padded with %s (%d bits), want %s" % (k, bin(val), fill, "ones" if ones else "zeros"))
        res["markers"].append(end_marker)
        pos = mpos + 2
    if pos != len(d):
        raise JpegSyntaxError("%d bytes after EOI" % (len(d) - pos))
    res["coefs"], res["comp"] = coefs, comp
    return res


# ---------------------------------------------------------------------------------------------------------------
# Inverse model
# ---------------------------------------------------------------------------------------------------------------
def reconstruct(parsed):
    """float64 pixels of a parsed 4:4:4 or gray file: exact IDCT of the dequantised coefficients, each plane + 128
    clipped to [0, 255], then JFIF YCbCr->RGB (T.871), clipped.  Returns [h, w] (one component) or [h, w, 3]."""
    sof = parsed["sof"]
    comps = sof["comps"]
    if any((c[1], c[2]) != (1, 1) for c in comps) or len(comps) not in (1, 3):
        raise ValueError("reconstruct() is for 4:4:4 and gray files")
    W, H = sof["width"], sof["height"]
    bw, bh = -(-W // 8), -(-H // 8)
    planes = []
    for ci, c in enumerate(comps):
        z = parsed["coefs"][parsed["comp"] == ci].astype(np.float64) * parsed["dqt"][c[3]]
        nat = z[:, ZZ].reshape(bh, bw, 8, 8)                         # natural index i holds zigzag position zz[i]
        f = DCT.T @ nat @ DCT
        planes.append(np.clip(f.transpose(0, 2, 1, 3).reshape(8 * bh, 8 * bw)[:H, :W] + 128.0, 0.0, 255.0))
    if len(planes) == 1:
        return planes[0]
    y, cb, cr = planes[0], planes[1] - 128.0, planes[2] - 128.0
    rgb = np.stack([y + 1.402 * cr, y - 0.344136 * cb - 0.714136 * cr, y + 1.772 * cb], -1)
    return np.clip(rgb, 0.0, 255.0)
