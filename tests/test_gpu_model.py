"""GPU (-m gpu): the B200's coefficients, files and decodes against the independent float64 model (tests/jpeg_model.py)
and, for the decoder, against the CPU run of its own source on files nobody recorded.

The parity tests compare the GPU with the oracle, which restates the same float32 arithmetic; these compare it with the
definitions, over every coefficient of the benchmark's workloads and on the paths the coefficient dump does not reach
(headers, restart markers, padding, the host-buffer and callback entry points)."""
import ctypes as C
import io

import numpy as np
import pytest
import torch

import oracle
from imagecodecs_b200.synth import synth_batch
from tests import jpeg_model as jm
from tests.emu.emu import emu_decode
from tests.test_model import CONTENTS, DECODE_BOUND_444, DECODE_BOUND_GRAY, LAYOUTS, QUALITIES, SIZES, content

pytestmark = pytest.mark.gpu

LAYOUT_OF = {(1, 0): [(1, 1)], (3, 0): [(1, 1)] * 3, (3, 1): [(2, 2), (1, 1), (1, 1)]}


def n_blocks(w, h, nc, sub):
    if nc == 1:
        return -(-w // 8) * -(-h // 8)
    return -(-w // 16) * -(-h // 16) * 6 if sub else -(-w // 8) * -(-h // 8) * 3


def run_plan(gpu, descs, keep, fetch=True):
    """Run a plan over `descs` with the coefficient dump attached.  Returns (files or None, device int16 [blocks, 64],
    first block of each image)."""
    torch.cuda.synchronize()             # the plan runs on the library's own stream: order it after torch's work
    plan = gpu.Plan(descs, device=0)
    plan._keep = keep
    nb = plan.num_blocks
    coefs = torch.zeros((nb, 64), dtype=torch.int16, device="cuda")
    bits = torch.zeros(nb, dtype=torch.int32, device="cuda")
    plan.attach_debug(coefs.data_ptr(), bits.data_ptr())
    for i, d in enumerate(descs):
        if not d.pixels_on_device:
            plan.upload(i, d.pixels)         # a plan copies host pixels only when asked (d.pixels is the top row)
    plan.run()
    files = plan.fetch() if fetch else None
    torch.cuda.synchronize()
    plan.close()
    first = np.cumsum([0] + [n_blocks(d.width, d.height, d.ncomp, d.subsampling) for d in descs])
    assert first[-1] == nb
    return files, coefs, first


def check_files(files, dump, first, modes, flags=None):
    """parse() of each file: its coefficients are the GPU's own dump; DQT, SOF sampling, DRI as the mode says."""
    for i, f in enumerate(files):
        nc, qm, q, sub = modes[i]
        p = jm.parse(f)
        ql, qc = jm.quant_tables(qm, q)
        assert np.array_equal(p["dqt"][0], ql) and (nc == 1 or np.array_equal(p["dqt"][1], qc)), (i, modes[i])
        assert [c[1:3] for c in p["sof"]["comps"]] == LAYOUT_OF[(1 if nc == 1 else 3, sub if nc != 1 else 0)], (i, modes[i])
        restart = flags is not None and flags[i] & 2
        assert p["dri"] == (oracle.restart_interval(nc, sub) if restart else 0), (i, modes[i])
        assert np.array_equal(p["coefs"], dump[first[i]:first[i + 1]]), (i, modes[i])


# ---------------------------------------------------------------------------------------------------------------
# 1. GPU coefficients against the model
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", sorted(LAYOUTS))
def test_grid_in_mixed_plans(gpu, layout):
    """The CPU grid (qualities x sizes x contents) in mixed plans, one per layout; every file also goes through
    parse(), half of them in restart mode."""
    nc, sub = LAYOUTS[layout]
    imgs, modes, descs, flags = [], [], [], []
    for j, (qm, q) in enumerate(QUALITIES):
        for n, (w, h) in enumerate(SIZES):
            for kind in CONTENTS:
                img = torch.from_numpy(content(kind, w, h, nc, n)).cuda()
                fl = gpu.FLAG_RESTART if (j + n) % 2 else 0
                imgs.append(img); modes.append((nc, qm, q, sub)); flags.append(fl)
                descs.append(gpu._describe(img, qm, q, sub, fl))
    torch.cuda.synchronize()
    files, coefs, first = run_plan(gpu, descs, imgs)
    dump = coefs.cpu().numpy()
    for i, img in enumerate(imgs):
        nc_, qm, q, sub_ = modes[i]
        jm.check_quantised(dump[first[i]:first[i + 1]], jm.exact_coefficients(img.cpu().numpy(), qm, q, sub_),
                           what="%s #%d %s q%d/%d" % (layout, i, tuple(img.shape), qm, q))
    check_files(files, dump, first, modes, flags)


def test_swizzles_and_restart_mode(gpu):
    """FLAG_SWAP_RB and bottom-up rows (described with a negative stride), host and device pixels, 4:4:4 and 4:2:0, with
    and without restarts: the model applied to the pixels the swizzle stands for."""
    base = [content("photo", 333, 201, 3, 1), content("primaries", 70, 45, 4, 2), content("noise", 129, 67, 3, 3)]
    descs, keep, want, modes, flags = [], [], [], [], []
    for k, img in enumerate(base):
        for swap in (0, 1):
            for bottom_up in (False, True):
                for sub in (0, 1):
                    fl = (gpu.FLAG_SWAP_RB if swap else 0) | (gpu.FLAG_RESTART if (k + sub + swap) % 2 else 0)
                    src = np.ascontiguousarray(img[::-1]) if bottom_up else img          # rows last-to-first
                    arr = torch.from_numpy(src).cuda() if (k + swap) % 2 else src
                    seen = img[..., [2, 1, 0] + ([3] if img.shape[2] == 4 else [])] if swap else img
                    q = (75, 90, 97, 50)[(k + sub) % 4]
                    descs.append(gpu._describe(arr, 1, q, sub, fl, bottom_up=bottom_up))
                    keep.append(arr); want.append(np.ascontiguousarray(seen)); modes.append((img.shape[2], 1, q, sub)); flags.append(fl)
    torch.cuda.synchronize()
    files, coefs, first = run_plan(gpu, descs, keep)
    dump = coefs.cpu().numpy()
    for i, seen in enumerate(want):
        nc, qm, q, sub = modes[i]
        jm.check_quantised(dump[first[i]:first[i + 1]], jm.exact_coefficients(seen, qm, q, sub), what="swizzle case %d" % i)
    check_files(files, dump, first, modes, flags)


def _check_plan_in_chunks(gpu, pixels, modes, chunk):
    """Every coefficient of every image of a device batch, copied back `chunk` images at a time."""
    n = pixels.shape[0]
    descs = [gpu._describe(pixels[i], *modes[i]) for i in range(n)]
    _, coefs, first = run_plan(gpu, descs, [pixels], fetch=False)
    for lo in range(0, n, chunk):
        hi = min(n, lo + chunk)
        dump = coefs[first[lo]:first[hi]].cpu().numpy()
        host = pixels[lo:hi].cpu().numpy()
        for i in range(lo, hi):
            jm.check_quantised(dump[first[i] - first[lo]:first[i + 1] - first[lo]], jm.exact_coefficients(host[i - lo], *modes[i]),
                               what="image %d %s" % (i, modes[i]))
    del coefs


def test_every_coefficient_of_config2_1080p_q75_420(gpu):
    """BASELINE configs[1], the benchmark's workload: 256 x 1920x1080, IJG q75, 4:2:0 -- all 801 M coefficients."""
    pixels = synth_batch(256, 1920, 1080, 3, "photo", seed=1, device="cuda")
    _check_plan_in_chunks(gpu, pixels, [(1, 75, 1)] * 256, 16)
    del pixels; torch.cuda.empty_cache()


def test_config3_4k_q90_444(gpu):
    """16 images of BASELINE configs[2]: 3840x2160, IJG q90, 4:4:4."""
    pixels = synth_batch(16, 3840, 2160, 3, "photo", seed=1, device="cuda")
    _check_plan_in_chunks(gpu, pixels, [(1, 90, 0)] * 16, 4)
    del pixels; torch.cuda.empty_cache()


def test_config5_sample_512_mixed_quality_420(gpu):
    """256 images spread evenly over the 16384 of BASELINE configs[4]: 512x512, IJG q by index % 3 in {50, 75, 95}, 4:2:0."""
    idx = np.linspace(0, 16383, 256).astype(int)
    pixels = torch.cat([synth_batch(1, 512, 512, 3, "photo", seed=1, first=int(i), device="cuda") for i in idx])
    _check_plan_in_chunks(gpu, pixels, [(1, (50, 75, 95)[i % 3], 1) for i in idx], 64)
    del pixels; torch.cuda.empty_cache()


def test_config4_16k_gray_q85_in_bands(gpu):
    """BASELINE configs[3]: one 16384x16384 gray image at IJG q85 (4.2 M blocks), checked 128 block rows at a time."""
    pixels = synth_batch(1, 16384, 16384, 1, "photo", seed=1, device="cuda", chunk=1)
    _, coefs, _ = run_plan(gpu, [gpu._describe(pixels[0], 1, 85, 0)], [pixels], fetch=False)
    coefs = coefs.view(2048, 2048, 64)
    for by in range(0, 2048, 128):
        band = pixels[0, 8 * by:8 * (by + 128)].cpu().numpy()
        jm.check_quantised(coefs[by:by + 128].cpu().numpy(), jm.exact_coefficients(band, 1, 85, 0), what="block rows %d.." % by)
    del coefs, pixels; torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------------------------
# 2. GPU files through parse()
# ---------------------------------------------------------------------------------------------------------------
def test_dqt_of_every_ijg_quality(gpu):
    """One batch per layout over IJG quality 1..100 (and tje 1..3): DQT == quant_tables(), SOF sampling factors, and the
    scan's coefficients against the model."""
    for layout, (nc, sub) in sorted(LAYOUTS.items()):
        qs = [(1, q) for q in range(1, 101)] + [(0, 1), (0, 2), (0, 3)]
        imgs = [content(("photo", "noise", "primaries")[k % 3], 40 + k % 9, 24 + k % 7, nc, k) for k in range(len(qs))]
        files, st = gpu.encode_batch(imgs, [m[0] for m in qs], [m[1] for m in qs], sub, device=0)
        assert st == [0] * len(imgs)
        for img, (qm, q), f in zip(imgs, qs, files):
            p = jm.parse(f)
            ql, qc = jm.quant_tables(qm, q)
            assert np.array_equal(p["dqt"][0], ql) and (nc == 1 or np.array_equal(p["dqt"][1], qc)), (layout, qm, q)
            assert [c[1:3] for c in p["sof"]["comps"]] == LAYOUT_OF[(1 if nc == 1 else 3, sub)], layout
            jm.check_quantised(p["coefs"], jm.exact_coefficients(img, qm, q, sub), what="%s q%d/%d" % (layout, qm, q))


def test_restart_files(gpu):
    """Restart mode: DRI is one tile in MCUs (8 / 4 / 24 for 4:4:4 / 4:2:0 / gray); parse() checks the RSTm sequence and
    the 1-bit padding of every interval; the coefficients are the model's."""
    for (w, h, nc, qm, q, sub) in [(641, 363, 3, 1, 75, 1), (500, 300, 1, 1, 85, 0), (640, 360, 4, 0, 3, 0), (97, 203, 3, 1, 10, 0),
                                   (1000, 17, 3, 1, 99, 1), (8, 8, 3, 0, 2, 0), (1, 1, 1, 1, 50, 0)]:
        img = content("photo", w, h, nc, w)
        files, st = gpu.encode_batch([img], qm, q, sub, device=0, flags=gpu.FLAG_RESTART, capacity=16 << 20)
        assert st == [0]
        p = jm.parse(files[0])
        ri = {(1, 0): 24, (3, 0): 8, (3, 1): 4}[(1 if nc == 1 else 3, sub)]
        mcus = n_blocks(w, h, nc, sub) // (1 if nc == 1 else (6 if sub else 3))
        assert p["dri"] == ri and len(p["pads"]) == -(-mcus // ri), (w, h, nc, sub)
        rst = [m for m in p["markers"] if 0xD0 <= m <= 0xD7]
        assert rst == [0xD0 + (k & 7) for k in range(len(rst))]
        jm.check_quantised(p["coefs"], jm.exact_coefficients(img, qm, q, sub), what="restart %dx%d" % (w, h))


def test_host_buffers_pitched_offset_and_chunked(gpu):
    """encode_batch with padded rows and a base pointer off alignment, and a host batch of more than one pipeline chunk
    (> 192 MB of pixels): the files parse, and their coefficients are the model's."""
    L = gpu.lib()
    for (w, h, nc, pad, shift, qm, q, sub) in [(1004, 64, 3, 0, 0, 1, 75, 1), (640, 48, 4, 64, 0, 1, 90, 1), (333, 41, 3, 7, 0, 1, 25, 0),
                                               (640, 48, 3, 0, 4, 1, 75, 1), (640, 48, 1, 24, 0, 1, 85, 0), (640, 48, 1, 0, 1, 1, 60, 0)]:
        img = content("photo", w, h, nc, w % 7)
        stride = w * nc + pad
        buf = np.zeros(shift + stride * h + 64, np.uint8)
        view = buf[shift:shift + stride * h].reshape(h, stride)
        view[:, :w * nc] = img.reshape(h, w * nc)
        view[:, w * nc:] = 0xAB
        desc = gpu.Image(buf.ctypes.data + shift, w, h, nc, stride, qm, q, sub, 0)
        cap = gpu.max_encoded_size(w, h, nc, sub)
        out = np.empty(cap, np.uint8)
        o = gpu.Output(out.ctypes.data, cap, 0, 0)
        assert L.jpeg_gpu_encode_batch(C.byref(desc), 1, C.byref(o), C.byref(gpu.BatchOpts(0, 0, None, 0))) == 1
        jm.check_quantised(jm.parse(out[:o.size].tobytes())["coefs"], jm.exact_coefficients(img, qm, q, sub),
                           what="pitched %dx%d nc=%d pad=%d shift=%d" % (w, h, nc, pad, shift))
    n = 40
    batch = synth_batch(n, 1920, 1080, 3, "photo", seed=1, first=7).numpy()     # 249 MB: two chunks
    files, st = gpu.encode_batch([batch[i] for i in range(n)], 1, [(50, 75, 95)[i % 3] for i in range(n)], 1, device=0)
    assert st == [0] * n
    for i in (0, 21, 39):
        jm.check_quantised(jm.parse(files[i])["coefs"], jm.exact_coefficients(batch[i], 1, (50, 75, 95)[i % 3], 1), what="chunked #%d" % i)


def test_encode_with_func_twin(gpu):
    L = gpu.lib()
    img = content("photo", 395, 348, 4, 4)
    chunks = []
    cb = gpu.WRITE_FUNC(lambda ctx, data, size: chunks.append(C.string_at(data, size)))
    for q in (1, 2, 3):
        chunks.clear()
        assert L.jpeg_gpu_encode_with_func(cb, None, q, 395, 348, 4, img.ctypes.data) == 1
        p = jm.parse(b"".join(chunks))
        assert np.array_equal(p["dqt"][0], jm.quant_tables(0, q)[0]) and p["dri"] == 0
        jm.check_quantised(p["coefs"], jm.exact_coefficients(img, 0, q, 0), what="encode_with_func q%d" % q)


# ---------------------------------------------------------------------------------------------------------------
# 3. the GPU decoder against the CPU run of its source, on unrecorded files
# ---------------------------------------------------------------------------------------------------------------
def _decoder_files(gpu):
    import cv2
    from PIL import Image
    rng = np.random.default_rng(20261020)
    files = []
    # this encoder, all layouts and qualities, with and without restarts; mostly small, some up to 2000x1500
    imgs, qm, q, sub, fl = [], [], [], [], []
    for k in range(72):
        big = k % 18 == 0
        w, h = (int(rng.integers(300, 2001)), int(rng.integers(200, 1501))) if big else (int(rng.integers(1, 260)), int(rng.integers(1, 200)))
        layout = sorted(LAYOUTS)[k % 5]
        nc, s = LAYOUTS[layout]
        mode = int(rng.integers(0, 2))
        imgs.append(content(CONTENTS[k % len(CONTENTS)], w, h, nc, k))
        qm.append(mode); q.append(int(rng.integers(1, 4)) if mode == 0 else int(rng.integers(1, 101))); sub.append(s)
        fl.append(gpu.FLAG_RESTART if k % 3 == 0 else 0)
    # tiny subsampled images: NanoJPEG rejects a chroma plane narrower or shorter than 3 samples
    for w, h in [(1, 1), (1, 17), (17, 1), (2, 2), (4, 9), (5, 5)]:
        imgs.append(content("photo", w, h, 3, w + h)); qm.append(1); q.append(90); sub.append(1); fl.append(0)
    out, st = gpu.encode_batch(imgs, qm, q, sub, device=0, flags=fl, capacity=24 << 20)
    assert st == [0] * len(imgs)
    files += out
    # other encoders: PIL (optimised tables), OpenCV 4:4:0 / 4:1:1 and restart intervals 1..16
    for k in range(24):
        w, h = int(rng.integers(1, 400)), int(rng.integers(1, 300))
        img = content(("photo", "noise", "check2")[k % 3], w, h, 3, k)
        if k % 2:
            b = io.BytesIO()
            if k % 6 == 5:
                Image.fromarray(img[..., 0]).save(b, "JPEG", quality=int(rng.integers(20, 98)), optimize=True)
            else:
                Image.fromarray(img).save(b, "JPEG", subsampling=(k // 2) % 3, quality=int(rng.integers(20, 98)), optimize=True)
            files.append(b.getvalue())
        else:
            ss = (cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420,
                  cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444)[(k // 2) % 4]
            ok, enc = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, int(rng.integers(30, 98)), cv2.IMWRITE_JPEG_SAMPLING_FACTOR, ss,
                                                 cv2.IMWRITE_JPEG_RST_INTERVAL, 1 + k % 16])
            assert ok
            files.append(enc.tobytes())
    ok, enc = cv2.imencode(".jpg", content("photo", 2000, 1500, 3, 9), [cv2.IMWRITE_JPEG_QUALITY, 80, cv2.IMWRITE_JPEG_SAMPLING_FACTOR,
                                                                       cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440, cv2.IMWRITE_JPEG_RST_INTERVAL, 9])
    files.append(enc.tobytes())
    return files


def test_gpu_decoder_matches_its_source_on_unrecorded_files(gpu):
    """decode_batch over >= 100 files in one host batch (the three-thread chunked pipeline) == emu_decode pixel for pixel,
    rejections included; the 4:4:4 and gray ones are also within the integer decoder's bounds of reconstruct()."""
    files = _decoder_files(gpu)
    assert len(files) >= 100
    got = gpu.decode_batch(files)
    rejected = 0
    for i, f in enumerate(files):
        want = emu_decode(f)
        if not isinstance(want, np.ndarray):
            rejected += 1
            assert got[i] is None, (i, want)
            continue
        assert got[i] is not None and got[i].shape == want.shape and np.array_equal(got[i], want), i
        p = jm.parse(f, padding=None)
        if all(c[1:3] == (1, 1) for c in p["sof"]["comps"]):
            d = np.abs(got[i].astype(np.float64) - jm.reconstruct(p)).max()
            assert d <= (DECODE_BOUND_GRAY if got[i].ndim == 2 else DECODE_BOUND_444), (i, d)
    assert rejected >= 5                 # at least the tiny 4:2:0 images up to 4 pixels wide or high
