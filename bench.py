#!/usr/bin/env python
"""bench.py -- JPEG encode throughput of the B200 path (and of the CPU reference arm).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 1..5] [--dump-outputs DIR]

Headline workload (BASELINE.json configs[1] = SURVEY 8d config 2, the one the metric is quoted on; --config picks another):
    synthetic 1920x1080 RGB, batch of 256 per GPU, IJG quality 75, 4:2:0.
A step = one pass of the encode path over the whole batch: two memsets + transform kernel + entropy kernel + the four
kernels of the stuffing pass (chunk planner, 0xFF count, group scan, stuff) per quantiser group.  `value` is device-timed MP/s with pixels resident in HBM and the encoded scans left
in HBM; `e2e` is the same batch through ONE jpeg_gpu_encode_batch call with pinned HOST pixels in and HOST JPEG files out.
The line also carries every BASELINE configuration (`configs`: device-timed value, fraction of the HBM roofline, a parity
check against the CPU checker) with its byte-pinned native twin.

Under torchrun (N > 1) config 2 runs one 256-image shard per rank (weak scaling); configs 3 and 5 are partitioned by image
index over the ranks (strong scaling); there is no data-path collective (SURVEY.md 8e); times are the max over ranks.
"""
import argparse
import concurrent.futures as cf
import ctypes as C
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "jpeg_encode_mp_per_s"
UNIT = "MP/s"

# SURVEY 8(d) "Configs as concrete inputs": shape, count, requested mode, native (byte-pinned) twin, how N GPUs share it
CONFIGS = {
    1: dict(name="data/cat.bmp (395x348 BGR-as-RGB) through the codecs.h writeJpg path", w=395, h=348, nc=3, n=1,
            mode=lambda i: (0, 3, 0), twin=None, scaling="replicas", label="tje quality 3, 4:4:4 (what codecs.cpp:853 asks for)"),
    2: dict(name="1920x1080 RGB x 256 per GPU", w=1920, h=1080, nc=3, n=256, mode=lambda i: (1, 75, 1), twin=lambda i: (0, 2, 0),
            scaling="weak", label="IJG q=75, 4:2:0", twin_label="tje quality 2, 4:4:4"),
    3: dict(name="3840x2160 RGB x 128", w=3840, h=2160, nc=3, n=128, mode=lambda i: (1, 90, 0), twin=lambda i: (0, 3, 0),
            scaling="strong", label="IJG q=90, 4:4:4", twin_label="tje quality 3, 4:4:4"),
    4: dict(name="16384x16384 gray x 1", w=16384, h=16384, nc=1, n=1, mode=lambda i: (1, 85, 0), twin=lambda i: (0, 2, 0), twin_nc=3,
            scaling="replicas", label="IJG q=85, gray", twin_label="16384x16384 RGB, tje quality 2, 4:4:4"),
    5: dict(name="512x512 RGB x 16384", w=512, h=512, nc=3, n=16384, mode=lambda i: (1, (50, 75, 95)[i % 3], 1),
            twin=lambda i: (0, 1 + i % 3, 0), scaling="strong", label="IJG q by n%3 in {50,75,95}, 4:2:0",
            twin_label="tje quality by n%3 in {1,2,3}, 4:4:4"),
}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------
# CPU arms
# ------------------------------------------------------------------------------------------
def cpu_encode(img, qm, q, sub):
    """The CPU checker: oracle/_ref (compiled, unmodified jpeg_enc.h) where the reference has the mode, else the oracle port."""
    import oracle
    if qm == 0 and sub == 0 and img.shape[2] in (3, 4) and os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libtje_ref.so")):
        return oracle.ref_encode(img, q)[1], "reference"
    return oracle.oracle_encode(img, qm, q, sub), "port"


def cpu_encode_rate(images, qmode, quality, sub, threads, min_seconds=2.0, max_seconds=25.0):
    """MP/s of the CPU checker on `images` (list of HxWxC uint8), `threads` host threads.  Returns (mp_per_s, kind, n, seconds)."""
    import oracle
    oracle.build()
    kind = cpu_encode(images[0], qmode, quality, sub)[1]      # warm (page-in, table setup)
    mp = images[0].shape[0] * images[0].shape[1] / 1e6
    done, lock, t_end = [0], threading.Lock(), [0.0]
    start = time.perf_counter()

    def worker(k):
        i = k
        while True:
            now = time.perf_counter() - start
            if now > max_seconds or (now > min_seconds and i >= len(images)):
                break
            cpu_encode(images[i % len(images)], qmode, quality, sub)
            i += threads
            with lock:
                done[0] += 1
                t_end[0] = time.perf_counter() - start

    ths = [threading.Thread(target=worker, args=(k,)) for k in range(threads)]
    for t in ths: t.start()
    for t in ths: t.join()
    return done[0] * mp / t_end[0], kind, done[0], t_end[0]


def dump_outputs(out_dir, files, budget=64_000_000):
    """--dump-outputs: what a caller of the timed path receives, the JPEG files of its last step, for comparing two builds.
    encoded_sizes.npy holds every file's length (-1: not encoded); encoded_files.npy the byte values (float32) of whole files,
    taken in a fixed seeded order while everything fits `budget` bytes; encoded_files_index.npy which files those are."""
    os.makedirs(out_dir, exist_ok=True)
    sizes = np.array([len(f) if f is not None else -1 for f in files], np.float64)
    room = budget - sizes.nbytes
    pick = []
    for i in np.random.default_rng(0).permutation(len(files)):
        need = 4 * sizes[i] + 8
        if sizes[i] > 0 and need <= room:
            pick.append(int(i))
            room -= need
    pick.sort()
    data = np.frombuffer(b"".join(files[i] for i in pick), np.uint8).astype(np.float32)
    np.save(os.path.join(out_dir, "encoded_sizes.npy"), sizes)
    np.save(os.path.join(out_dir, "encoded_files_index.npy"), np.array(pick, np.float64))
    np.save(os.path.join(out_dir, "encoded_files.npy"), data)


def run_reference(args):
    """--impl reference: the CPU implementation of the path on this box's host cores (all of them), on the headline
    config; plus the byte-pinned native twin through the compiled reference itself."""
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    from oracle import synth_batch
    cfg = CONFIGS[args.config]
    cores = os.cpu_count() or 1
    n_img = max(1, min(cores, 16, cfg["n"])) if cfg["w"] * cfg["h"] < 50e6 else 1
    sample = synth_batch(n_img, cfg["w"], cfg["h"], cfg["nc"])
    imgs = [sample[i] for i in range(n_img)]
    qm, q, sub = cfg["mode"](0)
    for _ in range(args.warmup):
        cpu_encode_rate(imgs, qm, q, sub, cores, min_seconds=0.5, max_seconds=3.0)
    t0 = time.perf_counter()
    rates, n_total, kind = [], 0, "port"
    for _ in range(args.steps):
        r, kind, n, _ = cpu_encode_rate(imgs, qm, q, sub, cores, min_seconds=1.0, max_seconds=6.0)
        rates.append(r); n_total += n
    wall = time.perf_counter() - t0
    v = float(np.median(rates))
    twin = None
    if cfg["twin"] is not None and cfg.get("twin_nc", cfg["nc"]) == cfg["nc"]:
        tq = cfg["twin"](0)
        r2, kind2, n2, s2 = cpu_encode_rate(imgs, tq[0], tq[1], tq[2], cores, min_seconds=2.0, max_seconds=10.0)
        twin = {"workload": cfg["twin_label"], "value": round(r2, 3), "unit": UNIT, "cores": cores, "kind": kind2,
                "sample": "%d encodes in %.1f s on %d threads, jpeg_enc.h compiled -O2 -ffp-contract=off" % (n2, s2, cores)}
    why = "" if kind == "reference" else " (the reference has no such mode: jpeg_enc.h:1223,1038 -> oracle port of its algorithm)"
    sample_txt = "%d x %dx%dx%d synthetic photo images per step, cycled, on %d threads%s" % (len(imgs), cfg["w"], cfg["h"], cfg["nc"], cores, why)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": round(v, 3), "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * wall / max(args.steps, 1), 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "%s, %s (SURVEY 8d config %d), CPU sample" % (cfg["name"], cfg["label"], args.config),
                   "images_per_step": n_total // max(args.steps, 1)},
        "cpu_baseline": {"value": round(v, 3), "unit": UNIT, "cores": cores, "kind": kind, "sample": sample_txt},
        "e2e": {"value": round(v, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "native_twin": twin, "gpu_launches": 0,
    }))
    return 0


# ------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clock + throttle reasons of one GPU every 50 ms while `running`."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                 "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                 "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(0.05)

    def __enter__(self):
        if self.nv:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr:
            self._thr.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def bind_near_gpu(index, local, world):
    """Multi-GPU runs: keep this rank (and the pinned buffers it first-touches) on the CPUs NVML reports as local to its GPU;
    where several ranks share one CPU set (one NUMA node for all GPUs), give every rank its own slice of it."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        near = sorted({64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1} & os.sched_getaffinity(0))
        if near:
            per = max(2, len(near) // max(world, 1))
            mine = near[(local * per) % len(near):][:per] or near
            os.sched_setaffinity(0, set(mine))
            return len(mine)
    except Exception:
        pass
    return 0


# ------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import imagecodecs_b200 as jg
    import oracle
    from imagecodecs_b200.sharding import max_over_ranks as reduce_max, shard_range
    from imagecodecs_b200.synth import synth_batch

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    near_cpus = bind_near_gpu(local, local, world) if world > 1 else 0
    jg.init([local])
    dev = torch.device("cuda", local)
    stream = torch.cuda.Stream(device=dev)      # explicit stream: events and kernels share it
    torch.cuda.set_stream(stream)
    sptr = C.c_void_p(stream.cuda_stream)
    peak, peak_src = measured_peak()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(ms):
        return reduce_max(ms, device=dev)

    def sum_over_ranks(v):
        if world == 1:
            return float(v)
        t = torch.tensor([float(v)], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    def timed(plan, steps, warmup):
        for _ in range(warmup):
            plan.run(sptr)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            plan.run(sptr)
        e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        barrier()
        return max_over_ranks(ms) / steps

    def pass_times(plan, reps=5):
        plan.enable_timing(True)
        rows = []
        for _ in range(reps):
            plan.run(sptr); torch.cuda.synchronize()
            rows.append(plan.pass_times())
        plan.enable_timing(False)
        return [float(np.median([r[k] for r in rows])) for k in range(3)]

    def shard_of(cfg):
        """Images [lo, hi) of the synthetic sequence this rank encodes, and whether the rank takes part at all."""
        if cfg["scaling"] == "weak":
            return rank * cfg["n"], (rank + 1) * cfg["n"], True
        if cfg["scaling"] == "strong":
            lo, hi = shard_range(cfg["n"], world, rank)
            return lo, hi, hi > lo
        return 0, cfg["n"], rank == 0        # replicas / single image: rank 0 measures it

    def parity_sample(files, host_of, mode_of, idx):
        with cf.ThreadPoolExecutor(max_workers=min(16, os.cpu_count() or 4)) as ex:
            want = list(ex.map(lambda i: cpu_encode(host_of(i), *mode_of(i))[0], idx))
        return all(files[i] == w for i, w in zip(idx, want))

    def measure_config(k, steps, warmup, twin=False, check=4, keep=False):
        """Device-timed throughput of config k (or its native twin) on this rank's shard; max time over ranks."""
        cfg = CONFIGS[k]
        nc = cfg.get("twin_nc", cfg["nc"]) if twin else cfg["nc"]
        mode = cfg["twin"] if twin else cfg["mode"]
        lo, hi, active = shard_of(cfg)
        res = {"config": k, "workload": "%s, %s" % (cfg["name"], cfg["twin_label"] if twin else cfg["label"]), "scaling": cfg["scaling"]}
        plan = pixels = None
        ms = 0.0
        scan = px_bytes = 0
        mp = 0.0
        parity = None
        if active:
            if k == 1:
                px = torch.from_numpy(np.load(os.path.join(ROOT, "tests", "golden", "fixture_pixels.npz"))["cat_bgr"]).to(dev)
                pixels = px[None]
            else:
                pixels = synth_batch(hi - lo, cfg["w"], cfg["h"], nc, "photo", seed=1, first=lo, device=dev, chunk=1 if cfg["w"] > 8000 else (1024 if cfg["w"] <= 512 else 16))
            torch.cuda.synchronize()
            n = pixels.shape[0]
            modes = [mode(lo + i) for i in range(n)]
            plan = jg.Plan.for_arrays([pixels[i] for i in range(n)], [m[0] for m in modes], [m[1] for m in modes], [m[2] for m in modes], device=0)
            mp = n * cfg["w"] * cfg["h"] / 1e6
            px_bytes = n * cfg["w"] * cfg["h"] * nc
        if plan is not None:
            for _ in range(warmup): plan.run(sptr)
        barrier()
        if plan is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(steps): plan.run(sptr)
            e1.record(stream); torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
        barrier()
        if plan is not None:
            n = pixels.shape[0]
            sizes = [plan.encoded_size(i) for i in range(n)]
            scan = sum(sizes) - n * len(jg.emit_headers(cfg["w"], cfg["h"], nc, *modes[0]))     # (the header has the same length for every quality)
            if check and rank == 0:
                idx = sorted(set(int(x) for x in np.linspace(0, n - 1, min(check, n))))
                try:
                    files = plan.fetch(sptr)
                    if k == 4 and not twin:      # 268 MP through one CPU thread takes ~10 s: compare the file hash with the oracle's
                        parity = files[0] == cpu_encode(pixels[0].cpu().numpy(), *modes[0])[0]
                    elif k == 4:
                        parity = "checked in tests/test_gpu_parity.py::test_16k_rgb_native_twin (805 MB through one CPU thread)"
                    else:
                        parity = parity_sample(files, lambda i: pixels[i].cpu().numpy(), lambda i: modes[i], idx)
                    del files
                except Exception as e:
                    parity = "check failed: %r" % (e,)
        t = max_over_ranks(ms)
        tot_mp, tot_px, tot_scan = sum_over_ranks(mp), sum_over_ranks(px_bytes), sum_over_ranks(scan)
        used = max(1, int(sum_over_ranks(1 if active else 0)))
        res.update({"value": round(tot_mp / (t * 1e-3), 1) if t > 0 else None, "unit": UNIT, "ms_per_step": round(t, 4),
                    "roofline_frac": round((tot_px + tot_scan) / (t * 1e-3) / 1e9 / (peak * used), 4) if t > 0 else None,   # per GPU that took part
                    "out_bytes_per_px": round(tot_scan / (tot_mp * 1e6), 4) if tot_mp else None,
                    "images": int(sum_over_ranks(pixels.shape[0] if pixels is not None else 0)), "gpus_used": used if tot_mp else 0,
                    "parity_vs_cpu_checker": parity})
        if keep:
            return res, plan, pixels
        if plan is not None:
            plan.close()
        del pixels
        torch.cuda.empty_cache()
        return res

    # ---- device-timed headline ------------------------------------------------------------------
    K = args.config
    cfg = CONFIGS[K]
    with ClockSampler(local) as clk:
        head, plan, pixels = measure_config(K, args.steps, args.warmup, check=2, keep=True)
    if args.dump_outputs and plan is not None and rank == 0:
        dump_outputs(args.dump_outputs, plan.fetch(sptr))
    launches = plan.launches if plan is not None else 0     # per quantiser group: transform + entropy + plan_chunks + count_ff + scan_groups + stuff
    clocks = clk.summary()
    ms_step = head["ms_per_step"]
    value = head["value"]
    lo, hi, active = shard_of(cfg)
    n_img = pixels.shape[0] if pixels is not None else 0
    W, H, NC = cfg["w"], cfg["h"], cfg["nc"]
    modes = [cfg["mode"](lo + i) for i in range(n_img)]
    sizes = [plan.encoded_size(i) for i in range(n_img)] if plan is not None else []
    hdr_len = len(jg.emit_headers(W, H, NC, *modes[0])) if n_img else 0
    scan_bytes = sum(sizes) - n_img * hdr_len

    # roofline of pass 1 (transform + entropy kernels): their own launch durations from CUDA events the library records
    # around them on the launching stream; algorithmic bytes = pixels in + compressed scan out (SURVEY 8d)
    roofline = None
    if plan is not None and rank == 0:
        algo_bytes = n_img * W * H * NC + scan_bytes
        ta, tb, tc = pass_times(plan)
        dom = ("jg::transform_kernel", ta) if ta >= tb else ("jg::entropy_kernel", tb)
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
                traffic = json.load(fh)
        except Exception:
            pass
        coef_bytes = plan.num_blocks * 128
        roofline = {"bound": "hbm", "achieved": round(algo_bytes / ((ta + tb) * 1e-3) / 1e9, 2), "peak": peak, "unit": "GB/s",
                    "frac": round(algo_bytes / ((ta + tb) * 1e-3) / 1e9 / peak, 4),
                    "traffic": (traffic or {}).get("pass1_dram_bytes_per_launch_config2") if K == 2 else None, "peak_source": peak_src,
                    "kernel": "pass 1 = jg::transform_kernel + jg::entropy_kernel (the fused round-1 kernel split in two; the algorithmic bytes "
                              "-- pixels in, scan out -- enter the first and leave the second)",
                    "kernel_ms_per_launch": round(ta + tb, 4), "dominant_kernel": dom[0],
                    "kernels": {"transform": {"ms": round(ta, 4), "bytes": int(n_img * W * H * NC + coef_bytes), "what": "pixels read + coefficient plane written",
                                              "frac": round((n_img * W * H * NC + coef_bytes) / (ta * 1e-3) / 1e9 / peak, 4)},
                                "entropy": {"ms": round(tb, 4), "bytes": int(coef_bytes + scan_bytes), "what": "coefficient plane read + unstuffed scan written",
                                            "frac": round((coef_bytes + scan_bytes) / (tb * 1e-3) / 1e9 / peak, 4)},
                                "stuff": {"ms": round(tc, 4), "bytes": int(3 * scan_bytes), "what": "unstuffed scan read twice (count_ff, stuff) + final scan written",
                                          "frac": round(3 * scan_bytes / max(tc, 1e-6) / 1e-3 / 1e9 / peak, 4)}},
                    "kernel_share_of_step": round((ta + tb) / (ta + tb + tc), 4), "second_pass_ms": round(tc, 4),
                    "algorithmic_bytes_per_launch": int(algo_bytes),
                    "whole_step_frac": round(algo_bytes / (ms_step * 1e-3) / 1e9 / peak, 4),
                    "note": "a step = 2 memsets (state, results) + transform + entropy + plan_chunks + count_ff + scan_groups + stuff kernels; `achieved` = algorithmic bytes / "
                            "(transform + entropy CUDA-event durations); the coefficient plane between the two is extra traffic, counted in `kernels` only"}

    # ---- end to end: pinned host pixels -> ONE C-ABI call -> host JPEG files ----------------------
    L = jg.lib()

    def e2e_leg(px_dev, mode_list, steps, warm):
        n = px_dev.shape[0]
        nc = px_dev.shape[3]
        host_px = px_dev.cpu().pin_memory()
        cap = max(plan_sizes) + 4096
        host_out = torch.empty((n, cap), dtype=torch.uint8).pin_memory()
        e_imgs = (jg.Image * n)(*[jg.Image(host_px[i].data_ptr(), W, H, nc, 0, mode_list[i][0], mode_list[i][1], mode_list[i][2], 0) for i in range(n)])
        e_outs = (jg.Output * n)(*[jg.Output(host_out[i].data_ptr(), cap, 0, 0) for i in range(n)])
        e_opts = jg.BatchOpts(0, 0, None, 0)

        def step():
            ok = L.jpeg_gpu_encode_batch(e_imgs, n, e_outs, C.byref(e_opts))   # returns with the files in host memory
            if ok != n:
                raise RuntimeError("e2e step encoded %d of %d: %s" % (ok, n, jg.last_error()))

        for _ in range(warm): step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps): step()
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3 / steps
        barrier()
        ms = max_over_ranks(ms)
        d2h = int(sum(e_outs[i].size for i in range(n)))
        # what the box's link gives a bare pinned upload of the same pixels (no encoder), this rank, all ranks at once
        dst = torch.empty_like(px_dev)
        barrier()
        t0 = time.perf_counter()
        for _ in range(3):
            dst.copy_(host_px, non_blocking=True)
        torch.cuda.synchronize()
        probe_ms = max_over_ranks((time.perf_counter() - t0) * 1e3 / 3)
        barrier()
        first = bytes(host_out[0][:e_outs[0].size].numpy().tobytes())
        del dst, host_px, host_out
        return ms, d2h, probe_ms, first

    e2e = None
    twin = None
    if K in (2, 3, 5) and plan is not None:
        plan_sizes = sizes
        e2e_steps = max(2, min(args.steps, 10))
        e_ms, d2h, probe_ms, first_file = e2e_leg(pixels, modes, e2e_steps, max(1, min(args.warmup, 3)))
        tot_mp = sum_over_ranks(n_img * W * H / 1e6)
        h2d = n_img * W * H * NC
        e2e = {"value": round(tot_mp / (e_ms * 1e-3), 2), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "ms_per_step": round(e_ms, 3), "steps": e2e_steps,
               "api": "jpeg_gpu_encode_batch(%d host images) -> %d host JPEG files, pinned buffers, one call per step and rank" % (n_img, n_img),
               "h2d_probe": {"what": "bare pinned->device copy of the same pixels, all %d ranks at once, no encoder" % world,
                             "ms": round(probe_ms, 3), "gb_per_s_per_gpu": round(h2d / (probe_ms * 1e-3) / 1e9, 2),
                             "e2e_over_probe": round(e_ms / probe_ms, 3)}}
        if rank == 0 and head["parity_vs_cpu_checker"] is True:
            head["parity_vs_cpu_checker"] = first_file == cpu_encode(pixels[0].cpu().numpy(), *modes[0])[0]

    # ---- byte-pinned native twin of the headline shape: device-timed, per pass, and end to end --------
    if cfg["twin"] is not None and cfg.get("twin_nc", NC) == NC and plan is not None:
        plan.close(); plan = None
        tmodes = [cfg["twin"](lo + i) for i in range(n_img)]
        tplan = jg.Plan.for_arrays([pixels[i] for i in range(n_img)], [m[0] for m in tmodes], [m[1] for m in tmodes], [m[2] for m in tmodes], device=0)
        tsteps = max(3, min(args.steps, 10))
        tms = timed(tplan, tsteps, 3)
        tsizes = [tplan.encoded_size(i) for i in range(n_img)]
        tsz = sum(tsizes) - n_img * len(jg.emit_headers(W, H, NC, *tmodes[0]))
        tot_mp = sum_over_ranks(n_img * W * H / 1e6)
        twin = {"workload": "same pixels, %s (byte-identical to jpeg_enc.h)" % cfg["twin_label"], "value": round(tot_mp / (tms * 1e-3), 1),
                "unit": UNIT, "ms_per_step": round(tms, 3), "out_bytes_per_px": round(tsz / (n_img * W * H), 3)}
        if rank == 0:
            ta, tb, tc = pass_times(tplan)
            talgo = n_img * W * H * NC + tsz
            twin["roofline_native"] = {"bound": "hbm", "achieved": round(talgo / ((ta + tb) * 1e-3) / 1e9, 2), "peak": peak, "unit": "GB/s",
                                       "frac": round(talgo / ((ta + tb) * 1e-3) / 1e9 / peak, 4), "kernel": "pass 1 = jg::transform_kernel<444> + jg::entropy_kernel",
                                       "kernel_ms_per_launch": round(ta + tb, 4), "transform_ms": round(ta, 4), "entropy_ms": round(tb, 4), "stuff_ms": round(tc, 4),
                                       "algorithmic_bytes_per_launch": int(talgo), "whole_step_frac": round(talgo / (tms * 1e-3) / 1e9 / peak, 4)}
            files = tplan.fetch(sptr)
            idx = [0, n_img // 2, n_img - 1]
            twin["parity_vs_compiled_reference"] = parity_sample(files, lambda i: pixels[i].cpu().numpy(), lambda i: tmodes[i], idx)
            del files
        tplan.close()
        if K in (2, 3, 5):
            plan_sizes = tsizes
            t_ms, t_d2h, _, _ = e2e_leg(pixels, tmodes, max(2, min(args.steps, 5)), 1)
            twin["e2e"] = {"value": round(tot_mp / (t_ms * 1e-3), 2), "unit": UNIT, "ms_per_step": round(t_ms, 3),
                           "h2d_bytes_per_step": n_img * W * H * NC, "d2h_bytes_per_step": t_d2h}
    if plan is not None:
        plan.close()

    # ---- the other direction (SURVEY 8f rank 1): the headline batch decoded by jpeg_gpu_decode_batch ----------
    decode = None
    if rank == 0 and world == 1 and K == 2 and not args.no_twin:
        decode = {}
        for key, flags in (("restart", jg.FLAG_RESTART), ("restart_free", 0)):
            try:
                rplan = jg.Plan.for_arrays([pixels[i] for i in range(n_img)], 1, 75, 1, device=0, flags=flags)
                rplan.run(sptr); torch.cuda.synchronize()
                rfiles = rplan.fetch(sptr); rplan.close()
                jg.decode_batch(rfiles[:2])                               # module load, memory pool
                pinned = torch.empty(n_img * W * H * 3, dtype=torch.uint8).pin_memory().numpy()     # the caller's (pinned) pixel buffers
                used = [0]

                def alloc(nbytes):
                    a = pinned[used[0]:used[0] + nbytes]; used[0] += nbytes
                    return a

                t0 = time.perf_counter()
                dec_px, dec_ms = jg.decode_batch(rfiles, timed=True, alloc=alloc)       # first full-size call: grows the decoder's memory pool
                dec_first = (time.perf_counter() - t0) * 1e3
                used[0] = 0
                jg.decode_batch(rfiles, alloc=alloc)                                     # (the pipelined form's own pool growth)
                used[0] = 0
                t0 = time.perf_counter()
                dec_px = jg.decode_batch(rfiles, alloc=alloc)                            # untimed: chunks pipelined over three host threads
                dec_call = (time.perf_counter() - t0) * 1e3
                ok = all(np.array_equal(dec_px[i], oracle.ref_decode(rfiles[i])) for i in (0, n_img - 1)) if oracle.have_ref() else None
                decode[key] = {"workload": "the same %d images, IJG q75 4:2:0, %s" % (n_img, "one restart interval per 24 blocks" if flags else
                                                                                     "ordinary files (no restart markers): self-synchronising subsequences"),
                               "value": round(n_img * W * H / 1e6 / (dec_ms * 1e-3), 1), "unit": UNIT, "kernels_ms": round(dec_ms, 3),
                               "call_ms_host_files_to_host_pixels": round(dec_call, 1), "first_call_ms": round(dec_first, 1), "host_buffers": "files pageable, pixels pinned", "pixels_identical_to_reference_decoder": ok}
                del dec_px, pinned
            except Exception as e:
                decode[key] = {"error": repr(e)}

    # ---- CPU baseline on this box's host cores (rank 0, N=1 only; bounded sample) --------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu and pixels is not None and W * H < 50e6:
        sample = [pixels[i].cpu().numpy() for i in range(min(8, n_img))]
        qm, q, sub = modes[0]
        v1, kind, n1, s1 = cpu_encode_rate(sample, qm, q, sub, 1, min_seconds=2.0, max_seconds=10.0)
        cpu = {"value": round(v1, 3), "unit": UNIT, "cores": 1, "kind": kind,
               "sample": "%d encodes of %dx%d images (first %d of the batch, cycled) in %.1f s, 1 thread%s" % (
                   n1, W, H, len(sample), s1, "" if kind == "reference" else "; the reference has no such mode, so this is the oracle port of its algorithm")}
        if twin is not None:
            tq = cfg["twin"](0)
            v2, kind2, n2, s2 = cpu_encode_rate(sample, tq[0], tq[1], tq[2], 1, min_seconds=2.0, max_seconds=10.0)
            twin["cpu_baseline"] = {"value": round(v2, 3), "unit": UNIT, "cores": 1, "kind": kind2,
                                    "sample": "%d encodes in %.1f s, 1 thread, jpeg_enc.h compiled -O2 -ffp-contract=off" % (n2, s2)}
    del pixels
    torch.cuda.empty_cache()

    # ---- every BASELINE configuration + native twin, device-timed (few steps each) ------------------
    configs = None
    if not args.no_configs:
        configs = []
        for k in (1, 2, 3, 4, 5):
            if k == K:
                e = dict(head); e["note"] = "the headline of this line"
                configs.append(e)
            else:
                configs.append(measure_config(k, 5, 3))
            if CONFIGS[k]["twin"] is not None:
                t = measure_config(k, 5, 3, twin=True, check=3)
                t["native_twin_of"] = k
                configs.append(t)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": cfg["scaling"] if cfg["scaling"] != "replicas" else "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "%s, %s (SURVEY 8d config %d = BASELINE configs[%d])" % (cfg["name"], cfg["label"], K, K - 1),
                       "images_per_gpu": n_img, "l2_policy": "inputs + outputs larger than the 126 MB L2; no flush needed" if n_img * W * H * NC > 3e8 else "input smaller than L2",
                       "out_bytes_per_px": head["out_bytes_per_px"], "sharding": "image index, no collective",
                       "parity_spot_check": head["parity_vs_cpu_checker"], "cpus_bound_near_gpu": near_cpus,
                       "pipeline": os.environ.get("JPEG_GPU_PIPELINE", "split")},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "clocks": clocks,
            "gpu_launches": args.steps * launches,
            "native_twin": twin, "decode": decode, "configs": configs,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[1, 2, 3, 4, 5], help="SURVEY 8(d) configuration (2 = BASELINE configs[1], the default)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-twin", action="store_true", help="skip the decode legs")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-configuration table")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the JPEG files of the last timed step to DIR as .npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
