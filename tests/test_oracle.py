"""CPU: the oracle (oracle/jpeg_oracle.c) against the reference's pins.

The reference ships no golden JPEGs (SURVEY.md section 4), so the pins are (a) the SHA-256
known answers produced by compiling the unmodified jpeg_enc.h (tests/golden/kat.json, same
values as SURVEY.md 8c), (b) the reference's own output bytes for tiny inputs
(tests/golden/ref_*.jpg) and (c) the compiled reference's answers on further inputs, recorded as
digests (tests/golden/ref_digests.json).
"""
import hashlib
import io
import os

import numpy as np
import pytest

import oracle
from tests.helpers import kat_image, psnr, ref_encoded, sha


def test_known_answers(kat, fixture_pixels):
    for e in kat:
        img = kat_image(e, fixture_pixels)
        got = oracle.oracle_encode(img, oracle.QMODE_TJE, e["tje_quality"])
        assert len(got) == e["bytes"], e["name"]
        assert sha(got) == e["sha256"], e["name"]


def test_golden_reference_files(kat, fixture_pixels, golden_dir):
    n = 0
    for e in kat:
        if "file" not in e:
            continue
        want = open(os.path.join(golden_dir, e["file"]), "rb").read()
        assert sha(want) == e["sha256"]
        assert oracle.oracle_encode(kat_image(e, fixture_pixels), oracle.QMODE_TJE, e["tje_quality"]) == want
        n += 1
    assert n >= 7


def test_codecs_h_write_path_config1(kat, fixture_pixels):
    """BASELINE config 1: data/cat.bmp -> readBmp (BGR kept) -> writeJpg (quality 3)."""
    e = [k for k in kat if k["name"] == "cat_bgr" and k["tje_quality"] == 3][0]
    got = oracle.oracle_encode(fixture_pixels["cat_bgr"], oracle.QMODE_TJE, 3)
    assert len(got) == 152466 and sha(got) == e["sha256"]
    assert got[:2] == b"\xff\xd8" and got[-2:] == b"\xff\xd9"
    # 655 header bytes, scan follows (SURVEY 8c)
    assert got[:655] == oracle.oracle_headers(395, 348, 3, oracle.SUB_444, oracle.QMODE_TJE, 3)


def test_against_compiled_reference_random_shapes():
    rng = np.random.default_rng(7)
    for k in range(24):
        w, h = int(rng.integers(1, 90)), int(rng.integers(1, 70))
        nc = int(rng.choice([3, 4]))
        q = int(rng.integers(1, 4))
        img = rng.integers(0, 256, size=(h, w, nc), dtype=np.uint8)
        if k % 3 == 0:
            img[:] = rng.integers(0, 256)          # flat image: DC-only blocks, long zero runs
        ref = ref_encoded(img, q)
        assert ref is not None
        assert sha(oracle.oracle_encode(img, oracle.QMODE_TJE, q)) == ref, (w, h, nc, q)


def test_reference_rejects_what_survey_says():
    img = oracle.synth_image(16, 16, 3)
    assert ref_encoded(img, 90) is None and ref_encoded(img, 0) is None                 # jpeg_enc.h:1223
    assert ref_encoded(oracle.synth_image(16, 16, 1), 3) is None                        # :954
    assert oracle.oracle_encode(img, oracle.QMODE_TJE, 4) is None
    assert oracle.oracle_encode(img, oracle.QMODE_IJG, 101) is None
    assert oracle.oracle_encode(oracle.synth_image(16, 16, 1), oracle.QMODE_TJE, 3, oracle.SUB_420) is None


def test_extended_modes_collapse_to_native():
    for shape in [(64, 48, 3), (17, 13, 4)]:
        img = oracle.synth_image(*shape)
        assert oracle.oracle_encode(img, oracle.QMODE_IJG, 50) == oracle.oracle_encode(img, oracle.QMODE_TJE, 1)
        assert oracle.oracle_encode(img, oracle.QMODE_IJG, 100) == oracle.oracle_encode(img, oracle.QMODE_TJE, 3)


def test_stage_dumps_are_consistent():
    img = oracle.synth_image(50, 30, 3, kind="noise")
    st = oracle.oracle_stages(img, oracle.QMODE_TJE, 2)
    assert st["coefs"].shape == (7 * 4 * 3, 64)
    assert int(st["block_bits"].sum()) == st["raw_bits"]
    # re-stuff the raw scan by hand and compare with the file
    raw = st["raw"]
    stuffed = bytearray()
    for b in raw.tobytes():
        stuffed.append(b)
        if b == 0xFF:
            stuffed.append(0)
    assert bytes(st["jpeg"][655:-2]) == bytes(stuffed)


@pytest.mark.parametrize("qm,q,sub,nc,floor", [
    (oracle.QMODE_IJG, 75, oracle.SUB_420, 3, 30.0), (oracle.QMODE_IJG, 90, oracle.SUB_444, 3, 38.0),
    (oracle.QMODE_IJG, 85, oracle.SUB_444, 1, 36.0), (oracle.QMODE_IJG, 50, oracle.SUB_420, 4, 28.0),
    (oracle.QMODE_TJE, 3, oracle.SUB_420, 3, 40.0), (oracle.QMODE_IJG, 95, oracle.SUB_420, 3, 34.0)])
def test_extended_modes_decode_with_independent_decoders(qm, q, sub, nc, floor):
    """Extended modes are unpinned by the reference: validate with PIL, OpenCV and NanoJPEG."""
    from PIL import Image
    import cv2
    yy, xx = np.mgrid[0:117, 0:203]
    smooth = np.stack([xx, yy * 2, (xx + yy) // 2, np.full_like(xx, 255)], -1).astype(np.uint8)[..., :max(nc, 1)]
    if nc == 1:
        smooth = smooth[..., :1]
    jpg = oracle.oracle_encode(smooth, qm, q, sub)
    want = smooth[..., 0] if nc == 1 else smooth[..., :3]
    pil = np.array(Image.open(io.BytesIO(jpg)))
    assert pil.shape == want.shape
    assert psnr(pil, want) > floor
    cvd = cv2.imdecode(np.frombuffer(jpg, np.uint8), cv2.IMREAD_UNCHANGED)
    cvd = cvd if nc == 1 else cvd[..., ::-1]
    assert psnr(cvd, want) > floor
    if oracle.have_ref():
        nj = oracle.ref_decode(jpg)
        assert nj is not None and psnr(nj, want) > floor - 1.0


def test_read_bmp_keeps_bgr_order(fixture_pixels):
    """SURVEY section 0 item 5: the codecs.h path encodes B,G,R bytes as if they were R,G,B."""
    from PIL import Image
    cat = fixture_pixels["cat_bgr"]
    jpg = oracle.oracle_encode(cat, oracle.QMODE_TJE, 3)
    dec = np.array(Image.open(io.BytesIO(jpg)).convert("RGB"))
    assert psnr(dec, cat) > 45.0                 # decodes to the BGR-as-RGB pixels ...
    assert psnr(dec, cat[..., ::-1]) < 20.0      # ... not to the true colours
