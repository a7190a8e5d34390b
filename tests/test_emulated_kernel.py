"""CPU: the product's kernel SOURCE (imagecodecs_b200/csrc/jpeg_kernel.cuh) compiled with g++
against tests/emu/cuda_emu.h (one OS thread per CUDA thread, several CTAs in flight) and
compared with the oracle.  This checks the kernel's logic -- tile bookkeeping, scans, packing,
stuffing, look-back -- where no GPU exists; the GPU parity tests (-m gpu) check the real thing."""
import numpy as np
import pytest

import oracle
from tests.emu.emu import emu_encode, emu_ticket_map
from tests.helpers import ref_decoded

CASES = [
    # label, (n, w, h, c, kind), qmode, quality, sub, window words, CTAs
    ("edge-clamped single MCU row", (1, 17, 13, 3, "photo"), 0, 3, 0, 0, 1),
    ("rgba, alpha ignored", (1, 17, 13, 4, "photo"), 0, 1, 0, 0, 1),
    ("two images, several tiles, 3 CTAs", (2, 200, 120, 3, "photo"), 0, 2, 0, 0, 3),
    ("unaligned pitch (byte loader)", (1, 131, 67, 3, "photo"), 0, 3, 0, 0, 2),
    ("noise: dense symbols, many 0xFF", (1, 96, 96, 3, "noise"), 0, 3, 0, 0, 2),
    ("forced tiny window: multi-group tiles", (1, 96, 64, 3, "noise"), 0, 3, 0, 64, 2),
    ("forced tiny window, sparse 4:2:0 (short last groups)", (2, 104, 56, 3, "photo"), 1, 50, 1, 8, 2),
    ("forced tiny window, gray", (1, 72, 40, 1, "photo"), 1, 85, 0, 4, 1),
    ("4:2:0 q75", (2, 120, 72, 3, "photo"), 1, 75, 1, 0, 2),
    ("4:2:0 edge + rgba", (1, 33, 47, 4, "photo"), 1, 90, 1, 0, 2),
    ("gray q85", (2, 200, 130, 1, "photo"), 1, 85, 0, 0, 2),
    ("gray single block", (1, 8, 8, 1, "photo"), 1, 85, 0, 0, 1),
]


@pytest.mark.parametrize("label,shape,qm,q,sub,win,ctas", CASES, ids=[c[0] for c in CASES])
def test_emulated_kernel_matches_oracle(label, shape, qm, q, sub, win, ctas):
    n, w, h, c, kind = shape
    batch = oracle.synth_batch(n, w, h, c, kind)
    scans, sizes, status, coefs, bits = emu_encode(batch, qm, q, sub, win_words=win, n_ctas=ctas, stages=True)
    for i in range(n):
        st = oracle.oracle_stages(batch[i], qm, q, sub)
        hdr = oracle.oracle_headers(w, h, 1 if c == 1 else 3, sub, qm, q)
        assert np.array_equal(coefs[i], st["coefs"]), "quantised coefficients differ"
        assert np.array_equal(bits[i], st["block_bits"]), "block bit lengths differ"
        assert hdr + scans[i] == st["jpeg"], "entropy-coded segment differs"
        assert status[i] == 0


def test_emulated_kernel_vector_load_paths():
    """16-byte (4:2:0, pitch % 16 == 0), 8-byte (pitch % 8 == 0) and 4-byte pixel loads."""
    for (w, h, nc, qm, q, sub) in [(64, 32, 3, 1, 75, 1), (40, 24, 3, 0, 3, 0), (44, 24, 3, 0, 2, 0), (32, 16, 4, 1, 90, 1), (48, 16, 1, 1, 85, 0)]:
        batch = oracle.synth_batch(1, w, h, nc, "photo")
        scans, sizes, status = emu_encode(batch, qm, q, sub, n_ctas=1)
        hdr = oracle.oracle_headers(w, h, 1 if nc == 1 else 3, sub, qm, q)
        assert hdr + scans[0] == oracle.oracle_encode(batch[0], qm, q, sub), (w, h, nc)


def test_emulated_kernel_reports_capacity_overflow():
    batch = oracle.synth_batch(1, 64, 64, 3, "noise")
    scans, sizes, status = emu_encode(batch, 0, 3, 0, n_ctas=1, cap=4096)
    want = len(oracle.oracle_encode(batch[0], 0, 3, 0)) - 655
    assert status[0] == 1 and int(sizes[0]) >= want      # flagged, nothing written past cap, a sufficient size reported


@pytest.mark.parametrize("tiles,force", [([5, 5, 5], False), ([5, 5, 5], True), ([1], False), ([7, 1, 3, 3, 12, 1], False),
                                         (list(np.random.default_rng(3).integers(1, 60, 150)), False)])
def test_ticket_schedule_is_a_round_robin_bijection(tiles, force):
    """Every tile gets exactly one ticket, a tile's predecessor in its image holds a smaller ticket
    (what makes the look-back deadlock-free), and consecutive tickets visit different images."""
    tiles = np.asarray(tiles)
    g, img = emu_ticket_map(tiles, force)
    first = np.concatenate([[0], np.cumsum(tiles)[:-1]])
    assert sorted(g.tolist()) == list(range(int(tiles.sum())))
    assert np.all((g >= first[img]) & (g < first[img] + tiles[img]))
    ticket_of = np.empty(len(g), np.int64); ticket_of[g] = np.arange(len(g))
    for i, t in enumerate(tiles):
        tk = ticket_of[first[i]:first[i] + t]
        assert np.all(np.diff(tk) > 0)
        # round-robin: between two tiles of one image every other still-active image got a ticket
        active_after = [(tiles > lt + 1).sum() for lt in range(t - 1)]
        assert np.all(np.diff(tk) >= np.maximum(1, np.asarray(active_after, dtype=np.int64))) if t > 1 else True


@pytest.mark.parametrize("qm,q,sub,ctas", [(1, 90, 1, 1), (1, 97, 0, 2), (0, 3, 0, 1), (1, 98, 0, 1), (1, 85, 0, 3)])
def test_emulated_kernel_sparse_dense_transitions(qm, q, sub, ctas):
    """Smooth / noise / smooth bands: the warps switch between half-region tiles (written two
    iterations later), whole-region tiles and the slow path, every combination of pending tiles."""
    w, h = 176, 240
    photo = oracle.synth_batch(1, w, h, 3, "photo")[0]
    noise = oracle.synth_batch(1, w, h, 3, "noise")[0]
    img = photo.copy()
    img[h // 3: 2 * h // 3] = noise[h // 3: 2 * h // 3]
    img[5 * h // 6:, : w // 2] = noise[5 * h // 6:, : w // 2]
    if qm == 1 and q == 98:
        img = img[:, :, :1].copy()
    nc_out = 1 if img.shape[2] == 1 else 3
    hdr = oracle.oracle_headers(w, h, nc_out, sub, qm, q)
    want = oracle.oracle_encode(img, qm, q, sub)
    scans, sizes, status = emu_encode(img[None], qm, q, sub, n_ctas=ctas)          # one image: the two-iteration (DEEP) kernel
    assert hdr + scans[0] == want and status[0] == 0
    if ctas == 1:
        scans, sizes, status = emu_encode(np.stack([img, img]), qm, q, sub, n_ctas=2)   # two images: the plain kernel
        assert hdr + scans[0] == want and hdr + scans[1] == want
    scans, sizes, status = emu_encode(np.stack([img, img[::-1].copy()]), qm, q, sub, n_ctas=2)
    assert hdr + scans[0] == want and hdr + scans[1] == oracle.oracle_encode(img[::-1].copy(), qm, q, sub)


@pytest.mark.parametrize("w,h,nc,qm,q,sub", [(45, 37, 3, 0, 3, 0), (64, 32, 3, 1, 75, 1), (33, 20, 4, 0, 2, 0), (40, 24, 4, 1, 90, 1)])
def test_emulated_kernel_load_time_swizzles(w, h, nc, qm, q, sub):
    """SWAP_RB and bottom-up rows (negative stride) give the bytes of swapBR() / flip() + writeJpg
    (codecs.cpp:162-251) without a host pass over the pixels -- vector and byte loaders."""
    img = oracle.synth_batch(1, w, h, nc, "photo")[0]
    hdr = oracle.oracle_headers(w, h, 3, sub, qm, q)
    want = oracle.oracle_encode(img, qm, q, sub)
    swapped = img.copy(); swapped[:, :, 0] = img[:, :, 2]; swapped[:, :, 2] = img[:, :, 0]
    scans, _, _ = emu_encode(swapped[None], qm, q, sub, n_ctas=1, flags=1)
    assert hdr + scans[0] == want
    scans, _, _ = emu_encode(np.ascontiguousarray(img[::-1])[None], qm, q, sub, n_ctas=1, bottom_up=True)
    assert hdr + scans[0] == want
    scans, _, _ = emu_encode(np.ascontiguousarray(swapped[::-1])[None], qm, q, sub, n_ctas=1, flags=1, bottom_up=True)
    assert hdr + scans[0] == want


@pytest.mark.parametrize("shape,qm,q,sub,ctas", [((1, 200, 120, 3), 0, 3, 0, 2), ((2, 120, 72, 3), 1, 75, 1, 2), ((1, 200, 130, 1), 1, 85, 0, 1),
                                                 ((1, 96, 96, 3), 0, 3, 0, 2), ((3, 64, 48, 4), 0, 2, 0, 1), ((1, 8, 8, 3), 0, 3, 0, 1)])
def test_emulated_kernel_restart_intervals(shape, qm, q, sub, ctas):
    """Opt-in restart mode (SURVEY 8f rank 3): every tile is a restart interval -- DRI header, 1-bit padding,
    RSTm markers inserted by the stuffing pass, DC prediction from 0.  Bytes == the oracle's restart mode,
    and the reference's decoder reads the same pixels as from the restart-free stream."""
    n, w, h, c = shape
    kind = "noise" if (w, h) == (96, 96) else "photo"       # noise: slow-path tiles + many 0xFF next to markers
    batch = oracle.synth_batch(n, w, h, c, kind)
    ri = oracle.restart_interval(c, sub)
    scans, sizes, status = emu_encode(batch, qm, q, sub, n_ctas=ctas, flags=2)
    hdr = oracle.oracle_headers(w, h, 1 if c == 1 else 3, sub, qm, q, restart=ri)
    for i in range(n):
        want = oracle.oracle_encode(batch[i], qm, q, sub, restart=ri)
        assert hdr + scans[i] == want and status[i] == 0
        plain = oracle.oracle_encode(batch[i], qm, q, sub)
        assert ref_decoded(want) is not None and ref_decoded(want) == ref_decoded(plain)


def test_emulated_stuffing_pass_over_many_chunks():
    """The stuffing pass's two-level scan (jpeg_stuff.cuh: 32 chunks of 8 KB per group, group totals scanned by one CTA):
    images of 62 and 38 chunks in one launch -- groups that straddle the image boundary, more than one group per image,
    ~2000 stuffed zeros per image -- and the same with restart markers."""
    imgs = np.stack([oracle.synth_batch(1, 384, 320, 3, "noise")[0], oracle.synth_batch(1, 384, 320, 3, "photo")[0]])
    hdr = oracle.oracle_headers(384, 320, 3, 0, 0, 3)
    scans, _, status = emu_encode(imgs, 0, 3, 0, n_ctas=3)
    for i in range(2):
        assert status[i] == 0 and hdr + scans[i] == oracle.oracle_encode(imgs[i], 0, 3, 0), i
    assert len(scans[0]) > 32 * 8192 and len(scans[1]) > 32 * 8192
    ri = oracle.restart_interval(3, 0)
    rhdr = oracle.oracle_headers(384, 320, 3, 0, 0, 3, restart=ri)
    rscans, _, status = emu_encode(imgs, 0, 3, 0, n_ctas=2, flags=2)
    for i in range(2):
        assert status[i] == 0 and rhdr + rscans[i] == oracle.oracle_encode(imgs[i], 0, 3, 0, restart=ri), i
