"""CPU: the encoder's extended modes (IJG quality, 4:2:0, gray, restart intervals) and the decoder on files nobody
recorded, against the independent float64 model of tests/jpeg_model.py.

The other CPU tests compare the kernel source with oracle/jpeg_oracle.c, a restatement of the same float32 arithmetic;
these compare both of them with the definitions (DCT-II, the quantiser rule, the colour transform, the chroma mean),
so a rule that the kernels and the oracle state the same wrong way fails here."""
import io
import json
import os

import numpy as np
import pytest

import oracle
from tests import jpeg_model as jm
from tests.emu.emu import emu_decode, emu_encode
from tests.helpers import REF_DIGESTS, sha

QUALITIES = [(0, 1), (0, 2), (0, 3)] + [(1, q) for q in (1, 5, 10, 25, 49, 50, 51, 75, 90, 97, 99, 100)]
LAYOUTS = {"444rgb": (3, 0), "444rgba": (4, 0), "420rgb": (3, 1), "420rgba": (4, 1), "gray": (1, 0)}
SIZES = [(1, 1), (7, 9), (8, 8), (15, 17), (16, 16), (17, 15), (33, 47), (203, 117)]
CONTENTS = ("photo", "noise", "flat", "check1", "check2", "check8", "primaries")

# 16x16 patches of black / white / yellow / blue / cyan / red / green / magenta: neighbours that flip the luma DC by the
# whole range (DC difference 2040, category 11, at quantiser 1) and the largest |Cb| and |Cr| there are, in 4:2:0 too
_PRIMARIES = np.array([[0, 0, 0], [255, 255, 255], [255, 255, 0], [0, 0, 255], [0, 255, 255], [255, 0, 0], [0, 255, 0],
                       [255, 0, 255]], np.uint8)


def content(kind, w, h, nc, n=0):
    """uint8 [h, w, nc] test image.  Alpha (nc == 4) is noise: the encoder must ignore it."""
    if kind in ("photo", "noise"):
        img = oracle.synth_image(w, h, nc, n=n, kind=kind)
    else:
        yy, xx = np.mgrid[0:h, 0:w]
        if kind == "flat":
            img = np.full((h, w, nc), 77 + 13 * np.arange(nc), np.uint8)
        elif kind.startswith("check"):
            p = int(kind[5:])
            img = np.repeat((((xx // p + yy // p) % 2) * 255).astype(np.uint8)[..., None], nc, 2)
        else:
            img = _PRIMARIES[(xx // 16 + 3 * (yy // 16)) % 8]
            img = img[..., :1] if nc == 1 else img
            if nc == 4:
                img = np.concatenate([img, np.zeros((h, w, 1), np.uint8)], 2)
    if nc == 4:
        img = img.copy()
        img[..., 3] = oracle.synth_image(w, h, 1, n=n + 1, kind="noise")[..., 0]
    return np.ascontiguousarray(img)


def _recorded_decodes():
    with open(REF_DIGESTS) as fh:
        return json.load(fh)["decode"]


# ---------------------------------------------------------------------------------------------------------------
# 1. the model against independent data
# ---------------------------------------------------------------------------------------------------------------
def _pil(img, **kw):
    from PIL import Image
    b = io.BytesIO()
    Image.fromarray(img).save(b, "JPEG", **kw)
    return b.getvalue()


def _cv2(img, quality, sampling=None, rst=0):
    import cv2
    params = [cv2.IMWRITE_JPEG_QUALITY, quality, cv2.IMWRITE_JPEG_RST_INTERVAL, rst]
    if sampling is not None:
        params += [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, sampling]
    ok, enc = cv2.imencode(".jpg", img, params)
    assert ok
    return enc.tobytes()


def test_parser_reads_other_encoders_files():
    """PIL and OpenCV (libjpeg) files: optimised Huffman tables, 4:2:2, 4:1:1, 4:4:0, gray, restart intervals 1 / 7 / 16.
    Sampling factors, restart counts and fill bits come out as written; 4:4:4 and gray reconstruct() within +-2 of
    libjpeg's own decode (its integer IDCT and 8-bit planes: |d| <= 1.92 measured)."""
    import cv2
    src = oracle.synth_image(211, 97, 3)
    gray = np.ascontiguousarray(src[..., 0])
    files = [(_pil(src, subsampling=0, quality=90), (1, 1)), (_pil(src, subsampling=1, quality=80), (2, 1)),
             (_pil(src, subsampling=2, quality=30, optimize=True), (2, 2)), (_pil(src, subsampling=0, quality=95, optimize=True), (1, 1)),
             (_pil(gray, quality=85), None), (_pil(gray, quality=95, optimize=True), None)]
    for rst in (0, 1, 7, 16):
        for ss, hv in ((cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444, (1, 1)), (cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422, (2, 1)),
                       (cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411, (4, 1)), (cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440, (1, 2))):
            files.append((_cv2(src, 85, ss, rst), hv))
        files.append((_cv2(gray, 90, None, rst), None))
    for f, hv in files:
        p = jm.parse(f, padding="ones")
        comps = p["sof"]["comps"]
        if hv is None:
            assert len(comps) == 1
        else:
            assert [c[1:3] for c in comps] == [hv, (1, 1), (1, 1)]
        mcus = -(-211 // (8 * (hv or (1, 1))[0])) * -(-97 // (8 * (hv or (1, 1))[1]))
        assert len(p["pads"]) == (-(-mcus // p["dri"]) if p["dri"] else 1)
        assert p["markers"].count(0xDA) == 1 and p["markers"][-1] == 0xD9
        assert sum(0xD0 <= m <= 0xD7 for m in p["markers"]) == len(p["pads"]) - 1
        if hv in (None, (1, 1)):
            want = cv2.imdecode(np.frombuffer(f, np.uint8), cv2.IMREAD_UNCHANGED if hv is None else cv2.IMREAD_COLOR)
            want = want if hv is None else want[..., ::-1]
            assert np.abs(jm.reconstruct(p) - want).max() <= 2.0


def test_parser_rejects_damaged_streams():
    img = oracle.synth_image(40, 24, 3)
    f = oracle.oracle_encode(img, 1, 75, 0)
    r = oracle.oracle_encode(img, 1, 75, 0, restart=2)
    sos = f.index(b"\xff\xda")
    body = sos + 2 + ((f[sos + 2] << 8) | f[sos + 3])
    rs = r.index(b"\xff\xda")
    rbody = rs + 2 + ((r[rs + 2] << 8) | r[rs + 3])
    rst0 = r.index(b"\xff\xd0", rbody)
    bad = {
        "bytes after EOI": f + b"\0",
        "0xFF not followed by 00": f[:body + 3] + b"\xff\x12" + f[body + 3:],
        "RST out of sequence": r[:rst0] + b"\xff\xd1" + r[rst0 + 2:],
        "RST without DRI": f[:body + 3] + b"\xff\xd0" + f[body + 3:],
        "zero padding in restart mode": r[:-3] + bytes([r[-3] & 0xF0]) + r[-2:] if r[-3] & 0x0F == 0x0F else None,
        "ones padding without restarts": f[:-3] + bytes([f[-3] | ((1 << jm.parse(f)["pads"][-1][0]) - 1)]) + f[-2:],
        "truncated scan": f[:body + 20] + b"\xff\xd9",
        "progressive": _pil(img, progressive=True),
    }
    assert jm.parse(f)["pads"][-1][0] > 0
    for what, data in bad.items():
        if data is None:
            continue
        with pytest.raises(jm.JpegSyntaxError):
            jm.parse(data)
    # a code that no table defines: all-ones 16-bit window (the luma AC table leaves 1111111111111111 unassigned)
    with pytest.raises(jm.JpegSyntaxError):
        jm.parse(f[:body] + b"\xff\x00\xff\x00\xff\x00" + f[body:])


@pytest.mark.parametrize("layout", sorted(LAYOUTS))
def test_quant_tables_equal_the_emitted_dqt(jg, layout):
    """quant_tables() against the DQT bytes the host emitter writes, every IJG quality and tje 1-3; the DHT segments
    against T.81 Annex K.3."""
    nc, sub = LAYOUTS[layout]
    for qm, q in [(0, 1), (0, 2), (0, 3)] + [(1, q) for q in range(1, 101)]:
        hdr = jg.emit_headers(33, 17, nc, qm, q, sub)
        ql, qc = jm.quant_tables(qm, q)
        dqt = _segments(hdr, 0xDB)
        assert [s[0] for s in dqt] == ([0] if nc == 1 else [0, 1]), (qm, q)
        assert np.array_equal(np.frombuffer(dqt[0][1:], np.uint8), ql), (layout, qm, q)
        if nc != 1:
            assert np.array_equal(np.frombuffer(dqt[1][1:], np.uint8), qc), (layout, qm, q)
    dht = {(s[0] >> 4, s[0] & 15): (s[1:17], s[17:]) for s in _segments(hdr, 0xC4)}
    assert dht == {k: v for k, v in jm.HUFFMAN_K3.items() if nc != 1 or k[1] == 0}


def _segments(hdr, marker):
    out, pos = [], 2
    while pos < len(hdr) and hdr[pos + 1] != 0xDA:
        ln = (hdr[pos + 2] << 8) | hdr[pos + 3]
        if hdr[pos + 1] == marker:
            out.append(hdr[pos + 4:pos + 2 + ln])
        pos += 2 + ln
    return out


# ---------------------------------------------------------------------------------------------------------------
# 2. the oracle against the model
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", sorted(LAYOUTS))
@pytest.mark.parametrize("qm,q", QUALITIES)
def test_oracle_coefficients_match_the_model(layout, qm, q):
    """Every size and content of the grid: oracle_stages() coefficients == the float64 model rounded half up (except
    within delta of .5), and parse() of the oracle's file, with and without restart intervals, gives the same
    coefficients bit for bit."""
    nc, sub = LAYOUTS[layout]
    for n, (w, h) in enumerate(SIZES):
        for kind in CONTENTS:
            img = content(kind, w, h, nc, n)
            st = oracle.oracle_stages(img, qm, q, sub)
            what = "%s %dx%d %s q%d/%d" % (layout, w, h, kind, qm, q)
            jm.check_quantised(st["coefs"], jm.exact_coefficients(img, qm, q, sub), what=what)
            if kind in ("photo", "noise", "primaries") or w * h < 300:
                assert np.array_equal(jm.parse(st["jpeg"])["coefs"], st["coefs"]), what
                ri = oracle.restart_interval(nc, sub) if n % 2 else 1 + n
                p = jm.parse(oracle.oracle_encode(img, qm, q, sub, restart=ri))
                assert p["dri"] == ri and np.array_equal(p["coefs"], st["coefs"]), what


def test_oracle_1080p_matches_the_model():
    for nc, sub, qm, q in ((3, 1, 1, 75), (4, 0, 1, 90), (1, 0, 1, 85)):
        img = oracle.synth_image(1920, 1080, nc, n=5)
        st = oracle.oracle_stages(img, qm, q, sub)
        jm.check_quantised(st["coefs"], jm.exact_coefficients(img, qm, q, sub), what="1080p nc=%d sub=%d q%d" % (nc, sub, q))


# ---------------------------------------------------------------------------------------------------------------
# 3. the kernel source (split pipeline, run on the CPU) against the model
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", sorted(LAYOUTS))
def test_emulated_kernel_coefficients_match_the_model(layout):
    nc, sub = LAYOUTS[layout]
    for qm, q in [(0, 1), (0, 3), (1, 5), (1, 50), (1, 75), (1, 97)]:
        for w, h in [(1, 1), (15, 17), (33, 47), (203, 117)]:
            batch = np.stack([content(k, w, h, nc, i) for i, k in enumerate(("photo", "noise", "primaries", "check1"))])
            _, _, status, coefs, _ = emu_encode(batch, qm, q, sub, stages=True)
            assert (status == 0).all()
            for i in range(len(batch)):
                jm.check_quantised(coefs[i], jm.exact_coefficients(batch[i], qm, q, sub), what="%s %dx%d #%d q%d/%d" % (layout, w, h, i, qm, q))


def test_emulated_kernel_swizzles_match_the_model():
    """FLAG_SWAP_RB and bottom-up rows: the model applied to the swizzled pixels."""
    img = content("primaries", 45, 38, 3)
    img = np.ascontiguousarray(np.where(oracle.synth_image(45, 38, 3, kind="noise") < 64, oracle.synth_image(45, 38, 3), img))
    for sub in (0, 1):
        for flags, bottom_up in ((1, False), (0, True), (1, True)):
            view = img[:, :, ::-1] if flags else img
            view = view[::-1] if bottom_up else view
            src = np.ascontiguousarray(img[::-1]) if bottom_up else img          # the array holds the rows last-to-first
            _, _, status, coefs, _ = emu_encode(src, 1, 80, sub, stages=True, flags=flags, bottom_up=bottom_up)
            assert (status == 0).all()
            jm.check_quantised(coefs[0], jm.exact_coefficients(np.ascontiguousarray(view[::-1] if bottom_up else view), 1, 80, sub),
                               what="flags=%d bottom_up=%s sub=%d" % (flags, bottom_up, sub))


# ---------------------------------------------------------------------------------------------------------------
# 4. the decoder source against the model, on files that have no recorded answer
# ---------------------------------------------------------------------------------------------------------------
# NanoJPEG (and so the decoder) works in integers: a fixed-point IDCT, planes rounded to 8 bits, and colour conversion
# with 8-bit constants (359, 88, 183, 454 / 256 against JFIF's 1.402, 0.344136, 0.714136, 1.772).  A plane is within
# ~0.6 of the exact IDCT + clip (0.5 of it the rounding to 8 bits); gray carries that straight through (bound 1.0,
# 0.57 measured).  R and B add 1.402 and 1.772 times the chroma plane's error, the constants' offset (<= 0.18 at
# |Cb| = 128) and the final rounding: at most 0.6 + 1.772 * 0.6 + 0.18 + 0.5 = 2.35 (bound 2.5, 1.93 measured over
# the cases below, noise at tje quality 3 the worst).  The mean error over a photo or noise image of 1000 pixels or
# more stays within +-0.25 (0.16 measured): no bias.  (Flat patches can sit on a .5 everywhere and round one way.)  A wrong table, zigzag, upsampling or colour rule is off by tens.
DECODE_BOUND_GRAY = 1.0
DECODE_BOUND_444 = 2.5


def _decode_cases():
    cases = []
    for i, (w, h) in enumerate([(1, 1), (9, 7), (61, 37), (130, 90), (203, 117), (257, 129)]):
        for nc in (1, 3, 4):
            for kind in ("photo", "noise", "primaries"):
                qm, q = [(1, 5), (0, 3), (1, 63), (1, 85), (0, 2), (1, 97)][(i + nc + len(kind)) % 6]
                cases.append((w, h, nc, kind, qm, q, i % 2))
    return cases


def test_emulated_decoder_matches_the_model_on_unrecorded_files():
    recorded = _recorded_decodes()
    worst = {1: 0.0, 3: 0.0}
    for (w, h, nc, kind, qm, q, rst) in _decode_cases():
        img = content(kind, w, h, nc, w)
        f = oracle.oracle_encode(img, qm, q, 0, restart=oracle.restart_interval(nc, 0) if rst else 0)
        assert sha(f) not in recorded
        got = emu_decode(f)
        assert isinstance(got, np.ndarray), (w, h, nc, kind, got)
        d = got.astype(np.float64) - jm.reconstruct(jm.parse(f))
        bound = DECODE_BOUND_GRAY if nc == 1 else DECODE_BOUND_444
        assert np.abs(d).max() <= bound and (w * h < 1000 or kind == "primaries" or abs(d.mean()) < 0.25), (w, h, nc, kind, qm, q, np.abs(d).max(), d.mean())
        worst[1 if nc == 1 else 3] = max(worst[1 if nc == 1 else 3], np.abs(d).max())
    assert worst[1] > 0.3 and worst[3] > 1.0          # the bounds are not vacuous: the integer decoder does differ


def test_emulated_decoder_rejects_narrow_subsampled_images():
    """NanoJPEG's rule: a subsampled component narrower or shorter than 3 samples is NJ_UNSUPPORTED (2).  Our 4:2:0
    files are rejected exactly when the image is at most 4 pixels wide or high, and decoded otherwise."""
    recorded = _recorded_decodes()
    for w, h in [(1, 1), (1, 17), (17, 1), (2, 2), (4, 40), (40, 4), (5, 5), (6, 33), (33, 6)]:
        f = oracle.oracle_encode(oracle.synth_image(w, h, 3), 1, 90, 1)
        assert sha(f) not in recorded
        got = emu_decode(f)
        if min(w, h) <= 4:
            assert got == 2, (w, h, got)
        else:
            assert isinstance(got, np.ndarray) and got.shape == (h, w, 3), (w, h)


def test_emulated_decoder_reads_440_files():
    """OpenCV 4:4:0 (vertical-only subsampling) with and without restart intervals: every decode path the library picks
    gives the same pixels, close to libjpeg's."""
    import cv2
    src = oracle.synth_image(97, 61, 3)
    for rst in (0, 1, 3):
        f = _cv2(src, 90, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440, rst)
        outs = [emu_decode(f, s) for s in (-1, 0, 3)]
        assert all(isinstance(o, np.ndarray) and np.array_equal(o, outs[0]) for o in outs), rst
        want = cv2.imdecode(np.frombuffer(f, np.uint8), cv2.IMREAD_COLOR)[..., ::-1]
        assert np.mean(np.abs(outs[0].astype(np.float64) - want)) < 2.0
