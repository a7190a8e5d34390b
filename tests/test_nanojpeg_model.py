"""CPU: the decoder source (jpeg_decode.cuh / jpeg_decode_host.cpp run on the CPU) against the independent integer model of
NanoJPEG in tests/nanojpeg_model.py, bit for bit.

The model is first anchored to the only NanoJPEG answers there are: the committed pixels of data/test.jpg and the
recorded decode digests of the files the decoder tests generate.  Then it stands in for NanoJPEG on files nobody
recorded: the encoder grid, 4:2:0 / 4:2:2 / 4:4:0 at every size residue, and crafted files with sampling layouts no
encoder in the tests writes (luma below chroma, Cb != Cr, vertical factor 4, MCUs of more than 10 and 16 blocks).
tests/test_gpu_nanojpeg_model.py runs the same files through the GPU's plane kernels and batch planner."""
import functools
import io
import os

import numpy as np
import pytest

import oracle
from tests import jpeg_model as jm
from tests import nanojpeg_model as nm
from tests.emu.emu import emu_decode, emu_set_round_order
from tests.helpers import pixel_digest, ref_decoded, sha
from tests.test_model import _cv2, _decode_cases, _pil, _recorded_decodes, content

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _same(got, want):
    """Pixels equal bit for bit, or the same NJ_* code."""
    if isinstance(want, np.ndarray):
        return isinstance(got, np.ndarray) and got.shape == want.shape and np.array_equal(got, want)
    return not isinstance(got, np.ndarray) and got == want


# ---------------------------------------------------------------------------------------------------------------
# 1. the model against NanoJPEG's own answers
# ---------------------------------------------------------------------------------------------------------------
def test_model_reproduces_the_committed_nanojpeg_pixels(fixture_pixels):
    jpeg = open(os.path.join(GOLDEN, "data_test.jpg"), "rb").read()
    assert np.array_equal(nm.decode(jpeg), fixture_pixels["testjpg"])


def recorded_files():
    """The files of test_decoder.py whose NanoJPEG answers are recorded, rebuilt with the same generator calls."""
    import cv2
    from PIL import Image, ImageFile
    files = []
    for (w, h, nc, qm, q, sub, rst) in [(200, 120, 3, 0, 3, 0, 0), (200, 120, 3, 1, 75, 1, 0), (130, 70, 1, 1, 85, 0, 0),
                                        (201, 123, 3, 1, 75, 1, 4), (64, 64, 3, 0, 2, 0, 8), (17, 13, 3, 0, 1, 0, 0),
                                        (333, 77, 3, 1, 50, 1, 4), (96, 96, 1, 1, 90, 0, 24), (8, 8, 3, 0, 3, 0, 0)]:
        img = oracle.synth_image(w, h, nc, kind="noise" if (w, h) == (64, 64) else "photo")
        files.append(oracle.oracle_encode(img, qm, q, sub, restart=rst))
    for (w, h, nc, qm, q, sub) in [(640, 360, 3, 1, 75, 1)]:          # the one subsequence case not already above
        files.append(oracle.oracle_encode(oracle.synth_image(w, h, nc, kind="photo"), qm, q, sub))
    rgb = Image.fromarray(oracle.synth_image(211, 97, 3))
    gray = Image.fromarray(oracle.synth_image(150, 61, 1)[:, :, 0])
    for im, kw in [(rgb, dict(subsampling=0)), (rgb, dict(subsampling=1)), (rgb, dict(subsampling=2)), (rgb, dict(subsampling=2, quality=30, optimize=True)),
                   (gray, dict(quality=85)), (gray, dict(quality=95, optimize=True)), (rgb, dict(subsampling=0, quality=95)),
                   (rgb, dict(subsampling="4:1:1", quality=80))]:
        b = io.BytesIO(); im.save(b, "JPEG", **kw)
        files.append(b.getvalue())
    img = oracle.synth_image(211, 97, 3)
    for rst in (1, 7, 16):
        for ss in (cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422,
                   cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411):
            files.append(_cv2(img, 85, ss, rst))
    files.append(_cv2(img[:, :, 0].copy(), 90, None, 5))
    # test_subsequence_decode_random_differential: the same random sequence, draws included
    ImageFile.MAXBLOCK = 1 << 24
    rng = np.random.default_rng(20261018)
    for it in range(200):
        w, h = int(rng.integers(8, 400)), int(rng.integers(8, 300))
        kind = "noise" if rng.random() < 0.25 else "photo"
        if rng.random() < 0.5:
            nc = 1 if rng.random() < 0.25 else 3
            qm = int(rng.integers(0, 2))
            q = int(rng.integers(1, 4)) if qm == 0 else int(rng.integers(5, 101))
            sub = 0 if (qm == 0 or nc == 1) else int(rng.integers(0, 2))
            f = oracle.oracle_encode(oracle.synth_image(w, h, nc, n=it, kind=kind), qm, q, sub)
        else:
            img = oracle.synth_image(w, h, 3, n=it, kind=kind)
            kw = dict(quality=int(rng.integers(5, 101)), optimize=bool(rng.random() < 0.5))
            b = io.BytesIO()
            if rng.random() < 0.2:
                Image.fromarray(img[:, :, 0]).save(b, "JPEG", **kw)
            else:
                Image.fromarray(img).save(b, "JPEG", subsampling=[0, 1, 2, "4:1:1"][int(rng.integers(0, 4))], **kw)
            f = b.getvalue()
        files.append(f)
        if ref_decoded(f) is not None:
            rng.integers(0, 4); rng.integers(2, 8)     # the round order and piece size that test draws
    return files


def test_model_reproduces_every_recorded_decode():
    """If the model disagrees with one of these, the model is wrong: they are NanoJPEG's answers."""
    checked = rejected = 0
    for i, f in enumerate(recorded_files()):
        want = ref_decoded(f)
        assert pixel_digest(nm.decode(f)) == want, i
        checked += 1
        rejected += want is None
    assert checked >= 230 and checked - rejected >= 150


# ---------------------------------------------------------------------------------------------------------------
# 2. files nobody recorded: the decoder source against the model
# ---------------------------------------------------------------------------------------------------------------
def _all_paths(f, want, what):
    """Every path emu_decode can take: the library's choice, the interval path, subsequences of 8 and 128 bytes with the
    threads of a round in each order."""
    try:
        for order in (0, 1, 2, 3):
            emu_set_round_order(order)
            for sub_log2 in ((-1, 0, 3, 7) if order == 0 else (3, 7)):
                assert _same(emu_decode(f, sub_log2), want), (what, order, sub_log2)
    finally:
        emu_set_round_order(0)


@functools.lru_cache(maxsize=None)
def unrecorded_files():
    """(name, file) pairs: the encoder grid of test_model.py, 4:2:0 and 4:2:2 at widths and heights of every residue
    mod 16, OpenCV 4:4:0 with and without restart intervals."""
    out = []
    for (w, h, nc, kind, qm, q, rst) in _decode_cases():
        img = content(kind, w, h, nc, w)
        out.append(("grid %dx%d nc%d %s q%d/%d rst%d" % (w, h, nc, kind, qm, q, rst),
                    oracle.oracle_encode(img, qm, q, 0, restart=oracle.restart_interval(nc, 0) if rst else 0)))
    for k in range(16):
        w, h = 32 + k, 17 + (5 * k + 3) % 16
        img = content("photo" if k % 2 else "noise", w, h, 3, k)
        out.append(("420 %dx%d" % (w, h), oracle.oracle_encode(img, 1, 60 + 2 * k, 1, restart=(0, 1, 3, 4)[k % 4])))
        out.append(("422 %dx%d" % (h + 20, w - 12), _pil(content("photo", h + 20, w - 12, 3, k), subsampling=1, quality=70 + k)))
    import cv2
    for w, h in ((97, 61), (40, 37)):
        for rst in (0, 1, 3):
            out.append(("440 %dx%d rst%d" % (w, h, rst), _cv2(oracle.synth_image(w, h, 3), 90, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440, rst)))
    return tuple(out)


def test_decoder_source_matches_the_model_on_unrecorded_files():
    recorded = _recorded_decodes()
    files = unrecorded_files()
    for name, f in files:
        assert sha(f) not in recorded, name
        want = nm.decode(f)
        assert isinstance(want, np.ndarray), name
        if name.startswith("grid"):
            assert _same(emu_decode(f), want), name
        else:
            _all_paths(f, want, name)
    assert len(files) == 92


# ---------------------------------------------------------------------------------------------------------------
# 3. crafted files: sampling layouts no encoder in the tests writes
# ---------------------------------------------------------------------------------------------------------------
# (Y, Cb, Cr) sampling factors (h, v)
LAYOUTS = {
    "Y11.C22.C22": [(1, 1), (2, 2), (2, 2)],        # luma below chroma: the luma plane is upsampled
    "Y22.Cb11.Cr21": [(2, 2), (1, 1), (2, 1)],      # Cb != Cr, one vertical pass each: fused
    "Y14.C11.C11": [(1, 4), (1, 1), (1, 1)],        # vertical factor 4: two V rounds, the last one fused
    "Y14.Cb12.Cr11": [(1, 4), (1, 2), (1, 1)],      # chroma planes of different heights: no fusion
    "Y42.C11.C11": [(4, 2), (1, 1), (1, 1)],        # 10 blocks per MCU
    "Y42.Cb22.Cr11": [(4, 2), (2, 2), (1, 1)],      # 13 blocks
    "Y44.C11.C11": [(4, 4), (1, 1), (1, 1)],        # 18 blocks: over the subsequence decode's 16
    "Y24.Cb24.Cr11": [(2, 4), (2, 4), (1, 1)],      # 17 blocks
    "Y21.C12.C12": [(2, 1), (1, 2), (1, 2)],
    "Y12.Cb11.Cr12": [(1, 2), (1, 1), (1, 2)],
    "Y11.C44.C44": [(1, 1), (4, 4), (4, 4)],        # 33 blocks; luma through four passes
    "Y22.Cb22.Cr11": [(2, 2), (2, 2), (1, 1)],
    "gray declared 22": [(2, 2)],                   # one component: NanoJPEG treats it as 1x1
}
# width and height of each layout's smallest component: 3, 4, 5 samples and each residue mod 4
MIN_SIZES = [(3, 4), (4, 5), (5, 3), (13, 7), (22, 14), (131, 9)]
DRIS = (0, 1, 3, 7)


def _coefficients(rng, rows, cols, mode):
    """Quantised coefficients of a padded block grid.  "photo": IJG q75 tables, moderate values; "saturate": quantiser
    255, values that drive the planes to 0 and 255; "fine": quantiser 1, DC over the whole 8-bit range.  Kept where no
    IDCT intermediate leaves int32 (the model asserts it)."""
    z = np.zeros((rows, cols, 64), np.int64)
    ac = rng.random((rows, cols, 63)) < (0.1 if mode == "saturate" else 0.15)
    lim = {"photo": (60, 5), "saturate": (12, 1), "fine": (1016, 40)}[mode]
    z[..., 0] = rng.integers(-lim[0], lim[0] + 1, (rows, cols))
    z[..., 1:] = np.where(ac, rng.integers(-lim[1], lim[1] + 1, (rows, cols, 63)), 0)
    return z


def _tables(mode, nc):
    ql, qc = jm.quant_tables(1, 75)
    if mode == "photo":
        return [ql] + [qc] * (nc - 1)
    return [np.full(64, 255 if mode == "saturate" else 1, np.int64)] * nc


def _size_for(factors, cw, ch):
    """An image size whose smallest component is cw x ch samples (ceil(W * ssx / ssxmax) = cw)."""
    dx = max(f[0] for f in factors) // min(f[0] for f in factors)
    dy = max(f[1] for f in factors) // min(f[1] for f in factors)
    if len(factors) == 1:
        dx = dy = 1
    return cw * dx - (cw % dx), ch * dy - ((ch + 1) % dy)


@functools.lru_cache(maxsize=None)
def crafted_files():
    """(name, file, factors, want) of every crafted layout at every size; want = the model's pixels."""
    rng = np.random.default_rng(20261021)
    out = []
    for li, (name, factors) in enumerate(LAYOUTS.items()):
        for si, (cw, ch) in enumerate(MIN_SIZES):
            W, H = _size_for(factors, cw, ch)
            g = nm.geometry(W, H, factors)
            assert isinstance(g, dict), (name, W, H, g)
            mode = ("photo", "saturate", "fine")[(li + si) % 3]
            grids = tuple(_coefficients(rng, *k["grid"], mode) for k in g["comps"])
            qt = _tables(mode, len(factors))
            dri = DRIS[(li + si) % 4]
            f = nm.write(W, H, factors, qt, grids, dri=dri)
            out.append(("%s %dx%d %s dri%d" % (name, W, H, mode, dri), f, tuple(factors), nm.decode_blocks(W, H, factors, qt, grids), grids))
    return tuple(out)


def test_writer_round_trips_through_the_strict_reader():
    for name, f, factors, _, grids in crafted_files():
        p = jm.parse(f, padding="ones")
        W, H = p["sof"]["width"], p["sof"]["height"]
        assert [c[1:3] for c in p["sof"]["comps"]] == list(factors), name
        assert np.array_equal(p["coefs"], nm.stream_order(W, H, factors, grids)), name


def test_crafted_layouts_cover_the_sizes_and_the_clip():
    """Every layout's smallest component is 3, 4 and 5 samples wide and high somewhere, every component width and height
    meets each residue mod 4, and the saturating files reach both ends of the clip."""
    seen_small, residues, lo, hi = set(), set(), 0, 0
    for name, f, factors, want, _ in crafted_files():
        p = jm.parse(f, padding="ones")
        g = nm.geometry(p["sof"]["width"], p["sof"]["height"], factors)
        for k in g["comps"]:
            seen_small |= {k["width"], k["height"]} & {3, 4, 5}
            residues |= {k["width"] % 4, k["height"] % 4}
        if "saturate" in name:
            lo += int((want == 0).any()); hi += int((want == 255).any())
    assert seen_small == {3, 4, 5} and residues == {0, 1, 2, 3}
    assert lo >= 10 and hi >= 10


def test_decoder_source_matches_the_model_on_crafted_layouts():
    for name, f, _, want, _ in crafted_files():
        _all_paths(f, want, name)


def test_decoder_source_matches_the_model_with_large_categories():
    """A complete custom Huffman table: DC differences and AC values of categories 12-15, beyond K.3 (quantiser 1,
    within int32 in the IDCT)."""
    rng = np.random.default_rng(7)
    for factors, (W, H) in (([(2, 2), (1, 1), (1, 1)], (61, 45)), ([(1, 1)], (70, 33)), ([(1, 2), (1, 1), (1, 1)], (40, 64))):
        g = nm.geometry(W, H, factors)
        grids = []
        for k in g["comps"]:
            z = np.zeros(k["grid"] + (64,), np.int64)
            z[..., 0] = rng.integers(-16000, 16001, k["grid"])
            big = rng.random(z.shape[:2] + (63,)) < 0.05
            z[..., 1:] = np.where(big, rng.integers(-6000, 6001, big.shape), 0)
            for r, c in np.ndindex(z.shape[:2]):          # an odd-frequency value this large leaves int32: keep such blocks DC-only
                try:
                    nm.idct_plane(z[r:r + 1, c:c + 1], np.ones(64, np.int64))
                except nm.Int32Overflow:
                    z[r, c, 1:] = 0
            grids.append(z)
        assert sum((np.abs(z[..., 1:]) >= 2048).sum() for z in grids) >= 3
        assert (np.abs(np.diff(grids[0][..., 0].ravel())) >= 2048).any()
        qt = [np.ones(64, np.int64)] * len(factors)
        f = nm.write(W, H, factors, qt, grids, dri=(0, 2)[len(factors) % 2], tables=nm.HUFFMAN_FULL)
        want = nm.decode_blocks(W, H, factors, qt, grids)
        assert isinstance(want, np.ndarray)
        _all_paths(f, want, factors)


def rejection_cases():
    """(what, file, the model's verdict) for files NanoJPEG rejects at the frame header."""
    out = []
    for what, W, H, factors, prec, marker in [
            ("factor 3", 40, 16, [(3, 1), (1, 1), (1, 1)], 8, 0xC0), ("vertical factor 3", 40, 48, [(1, 1), (1, 3), (1, 1)], 8, 0xC0),
            ("gray factor 3", 24, 24, [(3, 1)], 8, 0xC0), ("factor 0", 16, 16, [(1, 1), (0, 1), (1, 1)], 8, 0xC0),
            ("ncomp 2", 16, 16, [(1, 1), (1, 1)], 8, 0xC0), ("ncomp 4", 16, 16, [(1, 1)] * 4, 8, 0xC0),
            ("chroma 2 wide", 4, 16, [(2, 2), (1, 1), (1, 1)], 8, 0xC0), ("chroma 2 high", 16, 4, [(2, 2), (1, 1), (1, 1)], 8, 0xC0),
            ("luma 2 wide", 8, 16, [(1, 1), (4, 1), (4, 1)], 8, 0xC0), ("Cr 2 high", 24, 8, [(1, 4), (1, 4), (1, 1)], 8, 0xC0),
            ("precision 12", 16, 16, [(1, 1), (1, 1), (1, 1)], 12, 0xC0), ("SOF1", 16, 16, [(1, 1), (1, 1), (1, 1)], 8, 0xC1),
            ("SOF2", 16, 16, [(1, 1), (1, 1), (1, 1)], 8, 0xC2)]:
        hmax, vmax = max(f[0] for f in factors), max(f[1] for f in factors)
        mbw, mbh = -(-W // (8 * hmax)), -(-H // (8 * vmax))
        grids = [np.zeros((mbh * v, mbw * h, 64), np.int64) for h, v in factors]
        qt = [np.ones(64, np.int64)] * len(factors)
        out.append((what, nm.write(W, H, factors, qt, grids, precision=prec, marker=marker), nm.decode_blocks(W, H, factors, qt, grids, prec, marker)))
    # the same rule one sample later: accepted
    for W, H, factors in ((5, 16, [(2, 2), (1, 1), (1, 1)]), (16, 5, [(2, 2), (1, 1), (1, 1)]), (9, 16, [(1, 1), (4, 1), (4, 1)])):
        g = nm.geometry(W, H, factors)
        grids = [np.zeros(k["grid"] + (64,), np.int64) for k in g["comps"]]
        out.append(("accepted %dx%d" % (W, H), nm.write(W, H, factors, [np.ones(64, np.int64)] * 3, grids),
                    nm.decode_blocks(W, H, factors, [np.ones(64, np.int64)] * 3, grids)))
    return out


def test_rejections_match_the_model_code_for_code():
    verdicts = {}
    for what, f, want in rejection_cases():
        verdicts[what] = want if not isinstance(want, np.ndarray) else "pixels"
        assert _same(emu_decode(f), want), (what, emu_decode(f), want)
    assert verdicts == {"factor 3": 2, "vertical factor 3": 2, "gray factor 3": 2, "factor 0": 5, "ncomp 2": 2, "ncomp 4": 2,
                        "chroma 2 wide": 2, "chroma 2 high": 2, "luma 2 wide": 2, "Cr 2 high": 2, "precision 12": 2,
                        "SOF1": 2, "SOF2": 2, "accepted 5x16": "pixels", "accepted 16x5": "pixels", "accepted 9x16": "pixels"}


# ---------------------------------------------------------------------------------------------------------------
# 4. the two documented deviations on malformed streams (DESIGN.md section 7d)
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.xfail(strict=True, reason="DESIGN 7d: the DC predictor is kept in 16 bits with the coefficients; NanoJPEG's is an int")
def test_dc_predictor_beyond_16_bits():
    """Legal syntax: 40 gray blocks whose DC climbs by 2000 each (category 11), to 80000 at quantiser 1."""
    grid = np.zeros((1, 40, 64), np.int64)
    grid[0, :, 0] = 2000 * np.arange(1, 41)
    f = nm.write(320, 8, [(1, 1)], [np.ones(64, np.int64)], [grid])
    want = nm.decode(f)
    assert (want == 255).all()
    assert _same(emu_decode(f), want)


@pytest.mark.xfail(strict=True, reason="DESIGN 7d: a byte other than 00, FF, RSTn or D9 after an FF in the scan is swallowed; "
                                        "njShowBits raises NJ_SYNTAX_ERROR")
def test_marker_byte_inside_the_scan():
    """A stuffed FF 00 of a valid file turned into FF 01: NanoJPEG reads the FF as data and fails on the 01."""
    for _, g, _, _, _ in crafted_files():
        sos = g.index(b"\xff\xda")
        at = g.find(b"\xff\x00", sos + 2)
        if 0 < at < len(g) - 4:
            break
    else:
        raise AssertionError("no stuffed byte in the crafted files")
    bad = g[:at + 1] + b"\x01" + g[at + 2:]
    with pytest.raises(jm.JpegSyntaxError):
        jm.parse(bad, padding=None)
    assert isinstance(emu_decode(g), np.ndarray)
    assert emu_decode(bad, 0) == nm.NJ_SYNTAX_ERROR
