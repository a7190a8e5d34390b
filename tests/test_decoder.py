"""The decoder (SURVEY 8f rank 1): the product's decoder SOURCE (jpeg_decode.cuh / jpeg_decode_host.cpp) run on the
CPU, where one loop iteration is what one GPU thread executes, against the reference's NanoJPEG (its recorded answers,
tests/golden/ref_digests.json) and the committed fixture.  Bit-exact pixels are the bar.  The GPU run of the same code is in test_gpu_parity.py."""
import io
import os

import numpy as np
import pytest

import oracle
from tests.emu.emu import emu_decode, emu_set_round_order
from tests.helpers import pixel_digest, ref_decoded

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_reference_fixture_decodes_to_the_committed_pixels():
    """data/test.jpg of the reference (what tests.cpp reads first) -> exactly njDecode's pixels (tests/golden/fixture_pixels.npz)."""
    jpeg = open(os.path.join(GOLDEN, "data_test.jpg"), "rb").read()
    want = np.load(os.path.join(GOLDEN, "fixture_pixels.npz"))["testjpg"]
    got = emu_decode(jpeg)
    assert isinstance(got, np.ndarray) and np.array_equal(got, want)


@pytest.mark.parametrize("w,h,nc,qm,q,sub,rst", [(200, 120, 3, 0, 3, 0, 0), (200, 120, 3, 1, 75, 1, 0), (130, 70, 1, 1, 85, 0, 0),
                                                 (201, 123, 3, 1, 75, 1, 4), (64, 64, 3, 0, 2, 0, 8), (17, 13, 3, 0, 1, 0, 0),
                                                 (333, 77, 3, 1, 50, 1, 4), (96, 96, 1, 1, 90, 0, 24), (8, 8, 3, 0, 3, 0, 0)])
def test_decodes_our_own_streams_like_the_reference_decoder(w, h, nc, qm, q, sub, rst):
    img = oracle.synth_image(w, h, nc, kind="noise" if (w, h) == (64, 64) else "photo")
    jpeg = oracle.oracle_encode(img, qm, q, sub, restart=rst)
    want = ref_decoded(jpeg)
    got = emu_decode(jpeg)
    assert want is not None and pixel_digest(got) == want


def test_decodes_other_encoders_files():
    """Files of another encoder (PIL / libjpeg): 4:4:4, 4:2:2, 4:2:0, gray, custom Huffman tables, restart-free."""
    from PIL import Image
    rgb = Image.fromarray(oracle.synth_image(211, 97, 3))
    gray = Image.fromarray(oracle.synth_image(150, 61, 1)[:, :, 0])
    for im, kw in [(rgb, dict(subsampling=0)), (rgb, dict(subsampling=1)), (rgb, dict(subsampling=2)), (rgb, dict(subsampling=2, quality=30, optimize=True)),
                   (gray, dict(quality=85)), (gray, dict(quality=95, optimize=True))]:
        b = io.BytesIO(); im.save(b, "JPEG", **kw)
        want = ref_decoded(b.getvalue())
        got = emu_decode(b.getvalue())
        assert want is not None and pixel_digest(got) == want, kw


def test_rejects_what_the_reference_rejects():
    from PIL import Image
    assert emu_decode(b"\x00\x01\x02\x03") == 1                                    # NJ_NO_JPEG
    b = io.BytesIO(); Image.fromarray(oracle.synth_image(64, 48, 3)).save(b, "JPEG", progressive=True)
    assert ref_decoded(b.getvalue()) is None and emu_decode(b.getvalue()) == 2    # progressive: NJ_UNSUPPORTED
    good = oracle.oracle_encode(oracle.synth_image(40, 40, 3), 0, 3, 0)
    assert emu_decode(good[:300]) == 5                                             # truncated in the tables: NJ_SYNTAX_ERROR


def test_decodes_foreign_restart_streams_and_411():
    """libjpeg (OpenCV) files with restart intervals of 1 / 7 / 16 MCUs in 4:4:4, 4:2:0, 4:2:2 and 4:1:1 (two horizontal
    filter passes), gray with restarts, PIL 4:1:1: the parallel path on streams this encoder did not write."""
    import cv2
    from PIL import Image
    img = oracle.synth_image(211, 97, 3)
    files = []
    for rst in (1, 7, 16):
        for ss in (cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422,
                   cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411):
            ok, enc = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, 85, cv2.IMWRITE_JPEG_RST_INTERVAL, rst, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, ss])
            assert ok
            files.append(enc.tobytes())
    ok, enc = cv2.imencode(".jpg", img[:, :, 0].copy(), [cv2.IMWRITE_JPEG_QUALITY, 90, cv2.IMWRITE_JPEG_RST_INTERVAL, 5])
    files.append(enc.tobytes())
    b = io.BytesIO(); Image.fromarray(img).save(b, "JPEG", subsampling="4:1:1", quality=80)
    files.append(b.getvalue())
    for i, f in enumerate(files):
        want = ref_decoded(f)
        got = emu_decode(f)
        assert want is not None and pixel_digest(got) == want, i


# ---- restart-free scans: the subsequence (self-synchronising) decode --------------------------------------------

@pytest.mark.parametrize("w,h,nc,qm,q,sub", [(200, 120, 3, 0, 3, 0), (200, 120, 3, 1, 75, 1), (130, 70, 1, 1, 85, 0), (17, 13, 3, 0, 1, 0),
                                             (333, 77, 3, 1, 50, 1), (64, 64, 3, 0, 3, 0), (8, 8, 3, 0, 3, 0), (640, 360, 3, 1, 75, 1)])
def test_subsequence_decode_equals_the_reference_decoder(w, h, nc, qm, q, sub):
    """A scan without restart markers, cut into subsequences of 4 ... 128 bytes (4 bytes: shorter than one symbol can be,
    threads that have nothing to decode, stuffed bytes on the cuts): same pixels as njDecode, whatever the size."""
    img = oracle.synth_image(w, h, nc, kind="noise" if (w, h) == (64, 64) else "photo")
    jpeg = oracle.oracle_encode(img, qm, q, sub)
    want = ref_decoded(jpeg)
    assert want is not None
    try:
        for order in (0, 1, 2, 3):               # the threads of a round in different orders / racing host threads (records are updated in place)
            emu_set_round_order(order)
            for sub_log2 in (2, 3, 5, 7):
                got, rounds = emu_decode(jpeg, sub_log2, want_rounds=True)
                assert pixel_digest(got) == want, (order, sub_log2)
                assert rounds >= 2
    finally:
        emu_set_round_order(0)
    assert pixel_digest(emu_decode(jpeg, 0)) == want              # and the one-thread path still agrees


def test_subsequence_decode_is_the_default_for_restart_free_files():
    """The library's own policy: a restart-free scan of 512 bytes or more goes through subsequences (rounds > 0), restart
    streams and tiny scans through the interval path (rounds == 0); the reference's data/test.jpg is such a file."""
    jpeg = open(os.path.join(GOLDEN, "data_test.jpg"), "rb").read()
    got, rounds = emu_decode(jpeg, want_rounds=True)
    assert rounds > 0 and np.array_equal(got, np.load(os.path.join(GOLDEN, "fixture_pixels.npz"))["testjpg"])
    img = oracle.synth_image(201, 123, 3)
    assert emu_decode(oracle.oracle_encode(img, 1, 75, 1, restart=4), want_rounds=True)[1] == 0
    assert emu_decode(oracle.oracle_encode(oracle.synth_image(8, 8, 3), 0, 3, 0), want_rounds=True)[1] == 0


def test_subsequence_decode_of_other_encoders_files():
    """libjpeg files: optimised Huffman tables, 4:2:2 / 4:2:0 / 4:1:1 (six blocks per MCU in another order), gray."""
    from PIL import Image
    rgb = Image.fromarray(oracle.synth_image(211, 97, 3))
    gray = Image.fromarray(oracle.synth_image(150, 61, 1)[:, :, 0])
    for im, kw in [(rgb, dict(subsampling=0, quality=95)), (rgb, dict(subsampling=1)), (rgb, dict(subsampling=2, quality=30, optimize=True)),
                   (rgb, dict(subsampling="4:1:1", quality=80)), (gray, dict(quality=95, optimize=True))]:
        b = io.BytesIO(); im.save(b, "JPEG", **kw)
        want = ref_decoded(b.getvalue())
        for sub_log2 in (3, 5, -1):
            got = emu_decode(b.getvalue(), sub_log2)
            assert want is not None and pixel_digest(got) == want, (kw, sub_log2)


def test_subsequence_decode_of_damaged_scans_agrees_with_the_one_thread_path():
    """Truncated scans, flipped bits, marker bytes inside the scan: whatever the one-thread decode (NanoJPEG's loop) makes
    of the file -- pixels or NJ_SYNTAX_ERROR -- the subsequence decode makes of it too."""
    rng = np.random.default_rng(5)
    good = bytearray(oracle.oracle_encode(oracle.synth_image(160, 96, 3), 1, 80, 1))
    scan0 = 700
    cases = [bytes(good[:n]) + b"\xff\xd9" for n in (len(good) // 2, len(good) - 40, scan0 + 600)]
    for _ in range(40):
        b = bytearray(good)
        for _ in range(int(rng.integers(1, 4))):
            at = int(rng.integers(scan0, len(b) - 2))
            b[at] ^= 1 << int(rng.integers(0, 8))
        cases.append(bytes(b))
    seen_error = seen_pixels = 0
    for f in cases:
        one = emu_decode(f, 0)
        for sub_log2 in (3, 5):
            par = emu_decode(f, sub_log2)
            if isinstance(one, np.ndarray):
                assert isinstance(par, np.ndarray) and np.array_equal(par, one)
                seen_pixels += 1
            else:
                assert par == one
                seen_error += 1
    assert seen_error and seen_pixels


def test_irregular_marker_bytes_in_the_scan_stay_on_the_one_thread_path():
    """A scan in which an 0xFF is followed by something other than 00 has no canonical bit positions: such files are not cut
    into subsequences (rounds == 0) -- they decode, or fail, exactly as before."""
    good = bytearray(oracle.oracle_encode(oracle.synth_image(160, 96, 3), 1, 80, 1))
    at = 700 + next(i for i in range(len(good) - 1400) if good[700 + i] != 0xFF and good[699 + i] != 0xFF and good[701 + i] != 0xFF)
    good[at], good[at + 1] = 0xFF, 0x01
    res, rounds = emu_decode(bytes(good), 5, want_rounds=True)
    assert rounds == 0
    one = emu_decode(bytes(good), 0)
    assert (isinstance(res, np.ndarray) and np.array_equal(res, one)) or res == one


def test_subsequence_decode_random_differential():
    """200 random files (this encoder's oracle and libjpeg via PIL: sizes, qualities, samplings, gray, optimised tables, noise),
    random subsequence sizes of 4 ... 128 bytes and thread orders: every one decodes to the reference decoder's pixels."""
    from PIL import Image, ImageFile
    ImageFile.MAXBLOCK = 1 << 24
    rng = np.random.default_rng(20261018)
    checked = 0
    try:
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
            want = ref_decoded(f)
            if want is None:
                continue
            emu_set_round_order(int(rng.integers(0, 4)))
            sub_log2 = int(rng.integers(2, 8))
            got = emu_decode(f, sub_log2)
            assert pixel_digest(got) == want, (it, w, h, sub_log2)
            checked += 1
    finally:
        emu_set_round_order(0)
    assert checked > 150
