"""Shared helpers of the test-suite."""
import hashlib
import json
import os

import numpy as np

REF_DIGESTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_digests.json")
_ref_digests = None


def kat_image(entry, fixture_pixels):
    """Materialise the input image of a known-answer entry."""
    import oracle
    gen = entry["gen"]
    if "fixture" in gen:
        return fixture_pixels[gen["fixture"]]
    w, h, c, n, kind = gen["synth"]
    return oracle.synth_image(w, h, c, n, kind)


def sha(b):
    return hashlib.sha256(b).hexdigest()


def psnr(a, b):
    m = np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2)
    return 99.0 if m == 0 else 10 * np.log10(255.0 ** 2 / m)


def pixel_digest(px):
    """Shape and SHA-256 of decoded pixels; None for anything else (a rejected file)."""
    if not isinstance(px, np.ndarray):
        return None
    return "%s:%s" % ("x".join(str(d) for d in px.shape), sha(np.ascontiguousarray(px).tobytes()))


def _recorded(table, key, compute, what):
    """The reference's answer for `key` from tests/golden/ref_digests.json.

    The reference (jpeg_enc.h / jpeg_dec.h, see oracle/Makefile) is not part of this repository, so its answers for the
    inputs the tests use are stored as digests.  With JPEG_REF_RECORD=<path> set and the reference compiled into
    oracle/_ref, answers missing from the golden file are computed with it and the merged table is written to <path>."""
    global _ref_digests
    if _ref_digests is None:
        with open(REF_DIGESTS) as fh:
            _ref_digests = json.load(fh)
    entries = _ref_digests[table]
    if key not in entries:
        out = os.environ.get("JPEG_REF_RECORD")
        assert out, "no recorded reference answer for this %s (tests/golden/ref_digests.json; see tests/helpers.py)" % what
        entries[key] = compute()
        with open(out, "w") as fh:
            json.dump(_ref_digests, fh, indent=0, sort_keys=True)
    return entries[key]


def ref_decoded(jpeg):
    """pixel_digest() of what the reference decoder (NanoJPEG, jpeg_dec.h) makes of `jpeg`; None where it rejects it."""
    import oracle
    return _recorded("decode", sha(jpeg), lambda: pixel_digest(oracle.ref_decode(jpeg)), "%d-byte file" % len(jpeg))


def ref_encoded(img, quality):
    """SHA-256 of the file the reference encoder (jpeg_enc.h, tje_encode_with_func) writes for `img` at `quality`;
    None where it rejects the call."""
    import oracle
    img = np.ascontiguousarray(img, dtype=np.uint8)
    key = "%s:q%d:%s" % ("x".join(str(d) for d in img.shape), quality, sha(img.tobytes()))

    def compute():
        rc, data = oracle.ref_encode(img, quality)
        return sha(data) if rc == 1 else None
    return _recorded("encode", key, compute, "%s image at quality %d" % (img.shape, quality))
