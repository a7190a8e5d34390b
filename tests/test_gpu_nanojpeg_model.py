"""GPU (-m gpu): the B200 decoder against the independent integer model of NanoJPEG (tests/nanojpeg_model.py), bit for bit.

The CPU run of the decoder source covers decode_interval / decode_subsequence and the per-pixel device functions, but
not what only the GPU runs: idct_kernel's shared-memory tile, the word paths of upsample_h_kernel / upsample_v_kernel /
color_kernel, the vertical chroma pass fused into color_kernel, and the batch planner (jpeg_decode_api.cpp) that runs
the H and V rounds over all images of a call and decides per image when to fuse.  The crafted files of
test_nanojpeg_model.py send it down every kind of path: no fusion, fusion after zero or more rounds, two V rounds,
a luma plane upsampled four times, planes 3, 4 and 5 samples wide."""
import numpy as np
import pytest
import torch

from imagecodecs_b200.synth import synth_batch
from tests import jpeg_model as jm
from tests import nanojpeg_model as nm
from tests.test_nanojpeg_model import _same, crafted_files, rejection_cases, unrecorded_files

pytestmark = pytest.mark.gpu


def all_cases():
    """(name, file, want): crafted layouts, unrecorded encoder / PIL / OpenCV files, header rejections."""
    out = [(name, f, want) for name, f, _, want, _ in crafted_files()]
    out += [(name, f, nm.decode(f)) for name, f in unrecorded_files()]
    return out + list(rejection_cases())


def mixed_cases():
    """At most 63 files, so that an untimed decode_batch runs them as ONE call of the planner: every crafted layout at
    three sizes, 4:2:0 / 4:2:2 / 4:4:0 files, rejections."""
    crafted = [(name, f, want) for name, f, _, want, _ in crafted_files()][::2]
    other = [(name, f, nm.decode(f)) for name, f in unrecorded_files() if not name.startswith("grid")][::3]
    out = crafted + other + list(rejection_cases())[::2]
    assert len(out) <= 63
    return out


def planner_rounds(width, height, factors):
    """The planner's rule (jpeg_decode_api.cpp, fuse_now and the round loop) restated for one image: how many H / V rounds
    its planes take part in, and whether the last vertical chroma pass is fused into the colour kernel."""
    g = nm.geometry(width, height, factors)
    st = [[k["width"], k["height"]] for k in g["comps"]]
    rounds, fused = 0, False
    while not fused:
        moved = False
        for d in (0, 1):
            if d == 1 and len(st) == 3:
                (yw, yh), (aw, ah), (bw, bh) = st
                fused = aw >= width and bw >= width and ah == bh and ah < height and 2 * ah >= height and yh >= height and yw >= width
                if fused:
                    break
            todo = [p for p in st if (p[0] < width if d == 0 else p[1] < height)]
            for p in todo:
                p[d] *= 2
            rounds += bool(todo)
            moved = moved or bool(todo)
        if not moved:
            break
    return rounds, fused


def _geometry_of(f):
    """(width, height, declared factors) from the frame header."""
    sof = jm.parse(f, padding=None)["sof"]
    return sof["width"], sof["height"], [c[1:3] for c in sof["comps"]]


def test_mixed_batch_reaches_every_kind_of_planner_path():
    """Computed from the layouts: the one-piece batch holds images with 0, 1, 2 and 4 plane rounds, fused and not."""
    kinds = set()
    for name, f, want in mixed_cases():
        if isinstance(want, np.ndarray) and want.ndim == 3:
            kinds.add(planner_rounds(*_geometry_of(f)))
    assert {r for r, _ in kinds} >= {0, 1, 2, 4}
    assert {fz for _, fz in kinds} == {True, False}
    assert (2, False) in kinds and (1, True) in kinds and (0, True) in kinds     # two V rounds; fused after one; fused at once (4:4:0)


def test_one_decode_call_per_file(gpu):
    cases = all_cases()
    for name, f, want in cases:
        if isinstance(want, np.ndarray):
            got = gpu.decode(f)
            assert _same(got, want), name
        else:
            with pytest.raises(gpu.JpegGpuError):
                gpu.decode(f)
    assert len(cases) == 186


def _check_batch(got, cases):
    for (name, _, want), g in zip(cases, got):
        if isinstance(want, np.ndarray):
            assert _same(g, want), name
        else:
            assert g is None, name


def test_one_mixed_batch(gpu):
    cases = mixed_cases()
    _check_batch(gpu.decode_batch([f for _, f, _ in cases]), cases)


def test_whole_set_timed_in_one_piece(gpu):
    cases = all_cases()
    got, ms = gpu.decode_batch([f for _, f, _ in cases], timed=True)
    assert ms > 0
    _check_batch(got, cases)


def test_whole_set_chunked(gpu):
    """More than 64 files with host buffers: chunks of 32 on three host threads, each chunk its own planner call."""
    cases = all_cases()
    cases = cases + cases[:max(0, 64 - len(cases))]
    assert len(cases) >= 64
    _check_batch(gpu.decode_batch([f for _, f, _ in cases]), cases)


def test_pixels_on_device_with_guard_regions(gpu):
    """jpeg_gpu_decode_batch with pixels_on_device = 1 into torch buffers, base addresses off word alignment; every fifth
    image gets one byte too little capacity and must come back ERR_CAPACITY with its buffer untouched.  Every buffer sits
    between two guard regions that must keep their fill."""
    L = gpu.lib()
    cases = mixed_cases()
    n, G, FILL = len(cases), 256, 0xA5
    bufs = [np.frombuffer(f, np.uint8) for _, f, _ in cases]
    ins = (gpu.Stream * n)(*[gpu.Stream(b.ctypes.data, b.size) for b in bufs])
    outs = (gpu.Decoded * n)()
    dev, size, short = [], [], []
    for i, (_, _, want) in enumerate(cases):
        nbytes = want.size if isinstance(want, np.ndarray) else 16
        d = torch.full((2 * G + nbytes + 4,), FILL, dtype=torch.uint8, device="cuda")
        off = G + i % 4
        cap = nbytes - 1 if (i % 5 == 4 and isinstance(want, np.ndarray)) else nbytes
        outs[i] = gpu.Decoded(d.data_ptr() + off, cap, 0, 0, 0, 0)
        dev.append((d, off)); size.append(nbytes); short.append(cap < nbytes)
    torch.cuda.synchronize()
    done = L.jpeg_gpu_decode_batch(ins, n, outs, 1, None)
    torch.cuda.synchronize()
    ok = 0
    for i, (name, _, want) in enumerate(cases):
        host = dev[i][0].cpu().numpy()
        off = dev[i][1]
        assert (host[:off] == FILL).all() and (host[off + size[i]:] == FILL).all(), name
        if not isinstance(want, np.ndarray):
            assert outs[i].status == gpu.ERR_ARG, name
            assert (host == FILL).all(), name
        elif short[i]:
            assert outs[i].status == gpu.ERR_CAPACITY, name
            assert (host == FILL).all(), name
        else:
            assert outs[i].status == gpu.OK, name
            assert (outs[i].width, outs[i].height, outs[i].ncomp) == (want.shape[1], want.shape[0], 1 if want.ndim == 2 else 3)
            assert np.array_equal(host[off:off + size[i]], want.ravel()), name
            ok += 1
    assert done == ok and ok >= 30 and sum(short) >= 5


@pytest.mark.parametrize("restart", [True, False])
def test_headline_workload_1080p_q75_420(gpu, restart):
    """8 of the benchmark's 1920x1080 IJG q75 4:2:0 images (synth_batch seed 1), as files with one restart interval per
    tile and as ordinary restart-free files (the subsequence decode), in one call."""
    idx = [0, 37, 74, 111, 148, 185, 222, 255]
    pixels = torch.cat([synth_batch(1, 1920, 1080, 3, "photo", seed=1, first=i, device="cuda") for i in idx])
    files, st = gpu.encode_batch([pixels[k] for k in range(len(idx))], 1, 75, 1, device=0,
                                 flags=gpu.FLAG_RESTART if restart else 0)
    assert st == [0] * len(idx)
    got = gpu.decode_batch(files)
    for k, f in enumerate(files):
        want = nm.decode(f)
        assert want.shape == (1080, 1920, 3) and np.array_equal(got[k], want), idx[k]
