#!/usr/bin/env python
"""bench.py -- headline benchmark: fused gray -> 5x5 Gaussian -> Sobel on 4K RGB frames.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--no-extras] [--dump-outputs DIR]

One process per GPU (the driver launches N > 1 with torch.distributed.run).  Frames are
independent, so each rank owns whole frames (BASELINE config 4: 256 frames of 3840x2160 RGB8 over 8
GPUs = 32 frames per GPU); there is no data-path collective -- torch.distributed only supplies the
barrier and the max-over-ranks reduction of the device-timed duration.  Weak scaling: every rank
always processes 32 frames per step.

A "step" is one pass of the fused kernel over the rank's resident 32-frame batch (796 MB in +
265 MB out, far larger than the 126 MB L2, so every step streams from HBM).  `value` is
whole-job Mpixel/s with inputs resident in HBM; `e2e` is the same metric through the public
host-buffer API (rip_process_host: pinned host frames -> H2D -> kernel -> D2H every step).

After the two collective legs the process group is torn down, ranks > 0 exit, and rank 0 alone adds
the informational keys (so nothing spins in an NCCL barrier while the CPU oracle is timed):
  content   the same kernel on other frame content (smooth, letterboxed, half clipped, flat, black) with the
            fraction of pixels that took the exact replay -- the headline is iid noise, the friendliest case
  configs   BASELINE configs 1, 2, 3 (kernel time, Mpx/s, roofline fraction, oracle single-thread and all-core)
  config5   7680x4320: one frame as row bands over the run's N devices IN ONE PROCESS (rip_process_host_banded),
            a 16-frame batch sharded over the same N devices (rip_process_host), and the resident kernel
  e2e_nv12  the end-to-end leg with NV12 input (1.5 B/px in instead of 3)
  cpu_baseline  the oracle on the headline workload, all host threads, bounded sample

--dump-outputs DIR writes what the last timed step computed (see dump_outputs), so that two builds can be compared
output for output: the inputs are seeded and the same from run to run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the tree may be read-only and is left as it was: no __pycache__ from this run

W, H, CN = 3840, 2160, 3
FRAMES_PER_GPU = 32
KSIZE, SIGMA = 5, 1.0
ALGO_BYTES_PER_PX = 4  # 3 in (RGB8) + 1 out (u8)   -- SURVEY.md 8(d)
WORKLOAD = (f"fused gray->gauss{KSIZE}x{KSIZE}(sigma={SIGMA})->sobel, synthetic RGB8 {W}x{H}, "
            f"{FRAMES_PER_GPU} frames per GPU per step (BASELINE config 4 shard: 256 frames over 8 GPUs)")
DUMP_ROWS = 64  # rows per frame in --dump-outputs: 32 frames x 64 rows x 3840 px in float32 = 31.5 MB


def synth_batch(n: int, seed0: int) -> np.ndarray:
    """uniform iid u8 frames, seed = 0xB200 + 1000*config + frame (BASELINE.md section 2)."""
    out = np.empty((n, H, W, CN), np.uint8)
    for i in range(n):
        out[i] = np.random.default_rng(seed0 + i).integers(0, 256, (H, W, CN), dtype=np.uint8)
    return out


def dump_outputs(path: str, out: np.ndarray) -> None:
    """Write the fused output of the last timed step, (N, H, W) u8 as the caller receives it, to path/fused_rows.npy
    in float32.  A whole step is 265 MB of u8, so the file holds a fixed sample: the same DUMP_ROWS rows of every
    frame, namely the three top and three bottom rows (where the 5x5 blur and the Sobel clamp to the border) and rows
    drawn with a fixed seed."""
    h = out.shape[1]
    inner = np.random.default_rng(0xB200 + 99).choice(np.arange(3, h - 3), DUMP_ROWS - 6, replace=False)
    rows = np.sort(np.concatenate([[0, 1, 2, h - 3, h - 2, h - 1], inner]))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "fused_rows.npy"), out[:, rows].astype(np.float32))


def content_frame(kind: str, h: int = H, w: int = W) -> np.ndarray:
    """One RGB frame of the named content (the rows of the `content` key)."""
    rng = np.random.default_rng(0xB200 + 77)
    if kind == "smooth":      # natural-image-like: sinusoids + 2 LSB of noise, channels shifted against each other
        yy, xx = np.mgrid[0:h, 0:w]
        sm = (128 + 60 * np.sin(xx / 97.0) + 50 * np.cos(yy / 61.0) + rng.integers(-2, 3, (h, w))).clip(0, 255).astype(np.uint8)
        return np.ascontiguousarray(np.stack([sm, np.roll(sm, 7, 1), np.roll(sm, 13, 0)], -1))
    if kind in ("artemis_tiled", "tulips_tiled"):   # the reference's own images (decoded pixels from tests/golden), tiled to the frame size
        name = "Artemis_large1024.bgr" if kind == "artemis_tiled" else "Tulips_medium640.bgr"
        try:
            rgb = np.ascontiguousarray(dict(np.load(os.path.join(ROOT, "tests", "golden", "images.npz")))[name][..., ::-1])
        except Exception:
            return None
        reps = (-(-h // rgb.shape[0]), -(-w // rgb.shape[1]), 1)
        return np.ascontiguousarray(np.tile(rgb, reps)[:h, :w])
    one = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    if kind == "letterbox25":  # 25 % of the rows are black bars
        one[: h // 8] = 0
        one[-(h // 8):] = 0
    elif kind == "half_clipped":  # half of the frame is a clipped (constant 255) region
        one[:, : w // 2] = 255
    elif kind == "flat":
        one[:] = 77
    elif kind == "black":
        one[:] = 0
    return one


def measured_peak_gbs() -> tuple[float, str]:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def recorded_traffic_bytes():
    """dram__bytes_read.sum + dram__bytes_write.sum of one fused-kernel launch from the committed ncu
    capture of the shipped build (profiles/traffic.json), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get("fused_4k_32frames_dram_bytes_per_launch")
    except Exception:
        return None


def host_cores() -> int:
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def _oracle():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as O
    return O


def cpu_time(fn, budget_s: float = 3.0, max_reps: int = 20) -> float:
    """seconds per call of a CPU function: repeat until the budget is spent (at least once after one warm-up call)."""
    fn()
    t0 = time.perf_counter()
    n = 0
    while True:
        fn()
        n += 1
        dt = time.perf_counter() - t0
        if dt >= budget_s or n >= max_reps:
            return dt / n


def cpu_baseline(frames: np.ndarray, weights: np.ndarray, budget_s: float = 12.0) -> dict:
    """The oracle (CPU restatement of the reference's CPU paths) on a bounded sample, all host threads."""
    O = _oracle()
    cores = host_cores()   # passed explicitly: torchrun sets OMP_NUM_THREADS=1
    O.fused(frames[0], KSIZE, weights=weights, threads=cores)   # warm-up
    t0 = time.perf_counter()
    n = 0
    while True:   # the sample frames over and over until the budget is spent
        O.fused(frames[n % frames.shape[0]], KSIZE, weights=weights, threads=cores)
        n += 1
        dt = time.perf_counter() - t0
        if dt >= budget_s:
            break
    t0 = time.perf_counter()
    O.fused(frames[0], KSIZE, weights=weights, threads=1)
    t_single = time.perf_counter() - t0
    return {"value": n * W * H / dt / 1e6, "unit": "Mpixel/s", "cores": cores, "kind": "port",
            "sample": f"{n} passes over {frames.shape[0]} of the 32 4K frames of one step ({dt:.0f} s of CPU work), OpenMP over rows on "
                      f"{cores} threads ({dt / n * 1e3:.0f} ms per frame)",
            "single_thread_mpx_s": W * H / t_single / 1e6,
            "single_thread_note": "one frame, 1 thread: the reference's own CPU path is single-threaded"}


def run_reference(args, rank: int) -> None:
    """--impl reference: the reference's own CPU implementation of the path (oracle port; the reference
    needs OpenCV C++ + OpenCL and cannot be built here), all host threads, same config/metric."""
    if rank != 0:
        return
    O = _oracle()
    cores = host_cores()
    per_step = 2  # bounded sample: 2 of the 32 frames per step
    frames = synth_batch(per_step, 0xB200 + 4000)
    w = O.gauss_weights(KSIZE, SIGMA)
    for _ in range(args.warmup):
        O.fused(frames[0], KSIZE, weights=w, threads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        outs = [O.fused(frames[i], KSIZE, weights=w, threads=cores) for i in range(per_step)]
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, np.stack(outs))
    mpx = args.steps * per_step * W * H / dt / 1e6
    line = {"impl": "reference", "metric": "fused_4k_throughput", "value": mpx, "unit": "Mpixel/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "step_sample": f"{per_step} frames per step (bounded sample of the 32-frame step)"},
            "frames_per_s": mpx * 1e6 / (W * H),
            "cpu_baseline": {"value": mpx, "unit": "Mpixel/s", "cores": cores, "kind": "port",
                             "sample": f"{per_step} 4K frames per step x {args.steps} steps, OpenMP on {cores} threads"},
            "e2e": {"value": mpx, "unit": "Mpixel/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# rank-0 extras (after the process group is gone)
# ---------------------------------------------------------------------------------------------
def gpu_median_us(rip, fn, dev: int, stream, n: int = 7, warm: int = 2) -> float:
    """median device time of one call of fn (CUDA events on the stream the kernel is launched on)"""
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(n):
        e0, e1 = rip.Event(dev), rip.Event(dev)
        e0.record(stream); fn(); e1.record(stream); e1.sync()
        ts.append(e0.elapsed_ns(e1) / 1e3)
    return statistics.median(ts)


def content_rows(rip, dev, stream, d_in, d_out, weights, peak, n=FRAMES_PER_GPU) -> list:
    rows = []
    for kind in ("smooth", "artemis_tiled", "tulips_tiled", "letterbox25", "half_clipped", "flat", "black"):
        one = content_frame(kind)
        if one is None:
            continue
        for i in range(n):   # n shifted copies: every frame differs, constant regions stay constant
            d_in.upload(np.roll(one, 17 * i, axis=1), offset=i * one.nbytes)
        fn = lambda: rip.fused_dev(d_in.ptr, d_out.ptr, W, H, n, rip.FMT_RGB8, KSIZE, weights, device=dev, stream=stream)  # noqa: E731
        us = gpu_median_us(rip, fn, dev, stream)
        rip.slow_path_stats(True, dev)
        rip.fused_dev(d_in.ptr, d_out.ptr, W, H, 2, rip.FMT_RGB8, KSIZE, weights, device=dev, stream=stream)
        slow = rip.slow_path_stats(False, dev)
        rows.append({"content": kind, "us_per_step": us, "mpx_s": n * W * H / us,
                     "frac_of_hbm_peak": n * W * H * ALGO_BYTES_PER_PX / us / 1e3 / peak,
                     "guard_band_px_frac": slow / (2.0 * W * H)})
    return rows


def config_rows(rip, dev, stream, peak) -> list:
    """BASELINE configs 1-3 on this GPU next to the oracle on this host (single thread and all cores)."""
    O = _oracle()
    cores = host_cores()
    rows = []
    try:
        imgs = dict(np.load(os.path.join(ROOT, "tests", "golden", "images.npz")))
    except Exception:
        imgs = {}
    rng = np.random.default_rng(0xB200 + 1000)

    def add(name, px, bpp, us, t1, tn, extra=None):
        r = {"config": name, "kernel_us": us, "mpx_s": px / us, "frac_of_hbm_peak": px * bpp / us / 1e3 / peak,
             "algorithmic_bytes_per_px": bpp, "oracle_1thread_mpx_s": px / t1 / 1e6,
             f"oracle_{cores}threads_mpx_s": px / tn / 1e6, "cores": cores}
        if extra:
            r.update(extra)
        rows.append(r)

    # config 1: grayscale of Tulips_medium640 (RGBA upload as the reference does, (g,g,g,255) out); decoded pixels from tests/golden
    bgr = imgs.get("Tulips_medium640.bgr")
    if bgr is None:
        bgr = rng.integers(0, 256, (512, 640, 3), dtype=np.uint8)
    rgba = np.ascontiguousarray(np.concatenate([bgr[..., ::-1], np.full(bgr.shape[:2] + (1,), 255, np.uint8)], -1))
    h, w = rgba.shape[:2]
    d_i = rip.DeviceBuffer(rgba.nbytes, dev).upload(rgba)
    d_o = rip.DeviceBuffer(rgba.nbytes, dev)
    us = gpu_median_us(rip, lambda: rip.gray_dev(d_i.ptr, d_o.ptr, w, h, 1, rip.FMT_RGBA8, rip.GRAY_OUT_RGBA, device=dev, stream=stream), dev, stream, n=21)
    rgb = np.ascontiguousarray(rgba[..., :3])
    add(f"1: gray {w}x{h} RGBA -> (g,g,g,255), 1 frame (launch-bound)", w * h, 8, us,
        cpu_time(lambda: O.gray(rgb, threads=1), 1.0), cpu_time(lambda: O.gray(rgb, threads=cores), 1.0))
    # config 2: Gaussian 5x5 sigma 1.0 on Artemis_large1024 (683x1023 RGBA), and the reference's default 17x17 sigma 6
    bgr = imgs.get("Artemis_large1024.bgr")
    if bgr is None:
        bgr = rng.integers(0, 256, (1023, 683, 3), dtype=np.uint8)
    rgba = np.ascontiguousarray(np.concatenate([bgr[..., ::-1], np.full(bgr.shape[:2] + (1,), 255, np.uint8)], -1))
    h, w = rgba.shape[:2]
    d_i = rip.DeviceBuffer(rgba.nbytes, dev).upload(rgba)
    d_o = rip.DeviceBuffer(rgba.nbytes, dev)
    for k, s in ((5, 1.0), (17, 6.0)):
        wk = rip.gauss_weights(k, s)
        us = gpu_median_us(rip, lambda: rip.gauss_dev(d_i.ptr, d_o.ptr, w, h, 1, 4, k, wk, device=dev, stream=stream), dev, stream, n=21)
        add(f"2: Gaussian {k}x{k} sigma {s} on {w}x{h} RGBA, 1 frame", w * h, 8, us,
            cpu_time(lambda: O.blur(rgba, k, weights=wk, threads=1), 1.5, 5), cpu_time(lambda: O.blur(rgba, k, weights=wk, threads=cores), 1.0, 10))
    # the same two kernels at throughput size: 16 x 1080p RGBA frames with alpha = 255 (what the reference uploads, cv::COLOR_BGR2RGBA)
    nb, hb, wb = 16, 1080, 1920
    oneb = rng.integers(0, 256, (hb, wb, 4), dtype=np.uint8)
    oneb[..., 3] = 255
    d_i = rip.DeviceBuffer(nb * oneb.nbytes, dev)
    for i in range(nb):
        d_i.upload(np.roll(oneb, 29 * i, axis=1), offset=i * oneb.nbytes)
    d_o = rip.DeviceBuffer(nb * oneb.nbytes, dev)
    for k, s in ((5, 1.0), (17, 6.0)):
        wk = rip.gauss_weights(k, s)
        us = gpu_median_us(rip, lambda: rip.gauss_dev(d_i.ptr, d_o.ptr, wb, hb, nb, 4, k, wk, device=dev, stream=stream), dev, stream, n=9)
        t1 = cpu_time(lambda: O.blur(oneb[: hb // 8], k, weights=wk, threads=1), 1.0, 3) * 8
        tn = cpu_time(lambda: O.blur(oneb, k, weights=wk, threads=cores), 1.0, 5)
        add(f"2 (throughput): Gaussian {k}x{k} sigma {s} on {wb}x{hb} RGBA, alpha = 255, batch {nb}", nb * wb * hb, 8, us, t1 * nb, tn * nb,
            {"oracle_sample": "1 of the 16 frames on all cores; 1/8 of its rows on one thread; scaled"})
    d_i.free(); d_o.free()
    # config 3: Sobel on synthetic 1920x1080 RGB frames, batch 64
    n3, h, w = 64, 1080, 1920
    one = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    d_i = rip.DeviceBuffer(n3 * one.nbytes, dev)
    for i in range(n3):
        d_i.upload(np.roll(one, 13 * i, axis=1), offset=i * one.nbytes)
    d_o = rip.DeviceBuffer(n3 * h * w, dev)
    us = gpu_median_us(rip, lambda: rip.sobel_dev(d_i.ptr, d_o.ptr, w, h, n3, rip.FMT_RGB8, device=dev, stream=stream), dev, stream, n=11)
    t1 = cpu_time(lambda: O.sobel(O.gray(one, threads=1), threads=1), 1.5, 5)
    tn = cpu_time(lambda: O.sobel(O.gray(one, threads=cores), threads=cores), 1.0, 10)
    add(f"3: gray->Sobel {w}x{h} RGB8, batch {n3}", n3 * w * h, 4, us, t1 * n3, tn * n3, {"oracle_sample": "1 of the 64 frames, scaled"})
    return rows


def config5_rows(rip, n_dev: int, peak, weights) -> dict:
    """7680x4320 (BASELINE config 5) through ONE context over the run's N devices: row bands for a single frame,
    frame shards for a batch of 16; plus the resident kernel on device 0."""
    O = _oracle()
    cores = host_cores()
    w8, h8 = 7680, 4320
    one = np.random.default_rng(0xB200 + 5000).integers(0, 256, (h8, w8, 3), dtype=np.uint8)
    out = {"frame": f"{w8}x{h8} RGB8", "devices_in_one_context": n_dev}
    # resident kernel, 16 frames on device 0
    nb = 16
    d_i = rip.DeviceBuffer(nb * one.nbytes, 0)
    for i in range(nb):
        d_i.upload(np.roll(one, 17 * i, axis=1), offset=i * one.nbytes)
    d_o = rip.DeviceBuffer(nb * h8 * w8, 0)
    import ctypes as C
    st = C.c_void_p()
    rip.check(rip.lib().rip_stream_create(0, C.byref(st)))
    us = gpu_median_us(rip, lambda: rip.fused_dev(d_i.ptr, d_o.ptr, w8, h8, nb, rip.FMT_RGB8, KSIZE, weights, device=0, stream=st), 0, st, n=5)
    out["resident_batch16_1gpu"] = {"kernel_us": us, "mpx_s": nb * w8 * h8 / us, "frac_of_hbm_peak": nb * w8 * h8 * 4 / us / 1e3 / peak}
    us1 = gpu_median_us(rip, lambda: rip.fused_dev(d_i.ptr, d_o.ptr, w8, h8, 1, rip.FMT_RGB8, KSIZE, weights, device=0, stream=st), 0, st, n=11)
    out["resident_1frame_1gpu"] = {"kernel_us": us1, "mpx_s": w8 * h8 / us1, "note": "one frame (133 MB in + out) nearly fits the 126 MB L2"}
    d_i.free(); d_o.free()
    rip.lib().rip_stream_destroy(0, st)
    # host buffers end to end, one context over n_dev devices
    pin_in = rip.PinnedBuffer(nb * one.nbytes)
    src = pin_in.array.reshape(nb, h8, w8, 3)
    for i in range(nb):
        src[i] = np.roll(one, 17 * i, axis=1)
    pin_out = rip.PinnedBuffer(nb * h8 * w8)
    dst = pin_out.array.reshape(nb, h8, w8)
    ctx = rip.Context(list(range(n_dev)))
    for _ in range(3):
        ctx.process(src[0], rip.OP_FUSED, rip.FMT_RGB8, ksize=KSIZE, weights=weights, out=dst[:1], banded=True)
    ts = []
    for _ in range(9):
        t0 = time.perf_counter()
        ctx.process(src[0], rip.OP_FUSED, rip.FMT_RGB8, ksize=KSIZE, weights=weights, out=dst[:1], banded=True)
        ts.append((time.perf_counter() - t0) * 1e6)
    lat = statistics.median(ts)
    banded0 = dst[0].copy()
    out["banded_1frame_e2e"] = {"us_per_frame": lat, "mpx_s": w8 * h8 / lat, "bands": n_dev, "halo_rows": 3,
                                "api": "rip_process_host_banded, pinned host frame, H2D of band + halo / kernel / D2H per device"}
    for _ in range(2):
        ctx.process(src, rip.OP_FUSED, rip.FMT_RGB8, ksize=KSIZE, weights=weights, out=dst)
    t0 = time.perf_counter()
    reps = 3
    for _ in range(reps):
        ctx.process(src, rip.OP_FUSED, rip.FMT_RGB8, ksize=KSIZE, weights=weights, out=dst)
    dt = (time.perf_counter() - t0) / reps
    out["sharded_batch16_e2e"] = {"ms_per_batch": dt * 1e3, "mpx_s": nb * w8 * h8 / dt / 1e6, "frames_per_s": nb / dt,
                                  "api": "rip_process_host, 16 frames cut into contiguous blocks over the devices"}
    out["banded_equals_whole_frame"] = bool(np.array_equal(banded0, dst[0]))
    ctx.close()
    # the oracle on the same frame: all cores, and one thread on a 1/8 strip (scaled)
    tn = cpu_time(lambda: O.fused(one, KSIZE, weights=weights, threads=cores), 2.0, 3)
    strip = np.ascontiguousarray(one[: h8 // 8])
    t1 = cpu_time(lambda: O.fused(strip, KSIZE, weights=weights, threads=1), 2.0, 3) * 8
    out["oracle"] = {f"{cores}threads_mpx_s": w8 * h8 / tn / 1e6, "1thread_mpx_s": w8 * h8 / t1 / 1e6, "cores": cores,
                     "sample": "one 8K frame on all cores; 1/8 of its rows on one thread, scaled"}
    out["parity_spot_check"] = bool(np.array_equal(banded0[:64], O.fused(np.ascontiguousarray(one[:70]), KSIZE, weights=weights, threads=0)[:64]))
    pin_in.free(); pin_out.free()
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="headline + e2e legs only (no content / configs / config5 keys)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="steps of the host-buffer legs (default: --steps)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a fixed sample of the last step's output as DIR/fused_rows.npy "
                         "(float32; rank 0's frames when there are several ranks)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank)
        return

    import rip_b200 as rip
    if rip.device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device: librip_cuda has no CPU fallback")
    dev = local_rank % rip.device_count()

    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(dev)
        dist.init_process_group("nccl", device_id=torch.device("cuda", dev))

    def barrier():
        if dist is not None:
            dist.barrier()

    def max_over_ranks(x: float) -> float:
        if dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{dev}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # one process per GPU: host thread and pinned frame buffers on the GPU's own NUMA node (matters for the
    # end-to-end leg at 8 GPUs, where every rank streams 50 GB/s from host memory)
    numa = rip.bind_host_to_device_numa(dev) if world > 1 else {}

    L = rip.lib()
    weights = rip.gauss_weights(KSIZE, SIGMA)
    n = FRAMES_PER_GPU
    px_per_step_rank = n * W * H

    # ---- inputs: synthetic frames in pinned host memory, uploaded once for the resident leg ----
    pin_in = rip.PinnedBuffer(n * H * W * CN)
    pin_out = rip.PinnedBuffer(n * H * W)
    frames = pin_in.array.reshape(n, H, W, CN)
    frames[:] = synth_batch(n, 0xB200 + 4000 + 1000 * rank)
    d_in = rip.DeviceBuffer(frames.nbytes, dev).upload(frames)
    d_out = rip.DeviceBuffer(n * H * W, dev)
    import ctypes as C
    stream = C.c_void_p()
    rip.check(L.rip_stream_create(dev, C.byref(stream)))

    def step():
        rip.fused_dev(d_in.ptr, d_out.ptr, W, H, n, rip.FMT_RGB8, KSIZE, weights, device=dev, stream=stream)

    # ---- resident (kernel) leg ----
    # nvidia-smi samples every 100 ms and the timed region lasts milliseconds, so the sampler runs from
    # before the warm-up to the end of the end-to-end leg (the GPU is busy throughout that window)
    sampler = ClockSampler(dev)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        step()
    rip.check(L.rip_stream_sync(dev, stream))
    e0, e1 = rip.Event(dev), rip.Event(dev)
    launches0 = rip.launch_count()
    barrier()
    rip.check(L.rip_device_sync(dev))
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    e1.sync()
    rip.check(L.rip_device_sync(dev))
    barrier()
    launches = rip.launch_count() - launches0
    ms_local = e0.elapsed_ns(e1) / 1e6
    ms_total = max_over_ranks(ms_local)

    # correctness spot check outside the timed region: first frame of the resident output vs oracle
    out0 = d_out.download((H, W))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, d_out.download((n, H, W)))

    # ---- end-to-end leg: public host-buffer API, pinned host frames, H2D + kernel + D2H per step ----
    ctx = rip.Context([dev])
    e2e_steps = args.e2e_steps or args.steps
    out_host = pin_out.array.reshape(n, H, W)
    for _ in range(2):
        ctx.process(frames, rip.OP_FUSED, rip.FMT_RGB8, ksize=KSIZE, weights=weights, out=out_host)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        ctx.process(frames, rip.OP_FUSED, rip.FMT_RGB8, ksize=KSIZE, weights=weights, out=out_host)
    t_e2e_local = time.perf_counter() - t0
    barrier()
    t_e2e = max_over_ranks(t_e2e_local)
    e2e_ok = bool(np.array_equal(out_host[0], out0))

    # ---- the same leg with NV12 input (the reference's camera format): 1.5 bytes per pixel over PCIe instead of 3 ----
    nv = pin_in.array[: n * H * W * 3 // 2].reshape(n, H * 3 // 2, W)   # reuse the pinned input buffer: luma plane = the bytes that are there
    if not args.no_extras:
        for _ in range(2):
            ctx.process(nv, rip.OP_FUSED, rip.FMT_NV12, ksize=KSIZE, weights=weights, out=out_host)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            ctx.process(nv, rip.OP_FUSED, rip.FMT_NV12, ksize=KSIZE, weights=weights, out=out_host)
        t_nv_local = time.perf_counter() - t0
        barrier()
        t_nv = max_over_ranks(t_nv_local)
    ctx.close()
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None:
        clocks["window"] = "warm-up + timed steps + end-to-end legs (100 ms nvidia-smi samples)"

    # ---- the collective part is over: tear the process group down; ranks > 0 leave ----
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return

    mpx = world * px_per_step_rank * args.steps / (ms_total / 1e3) / 1e6
    ms_per_step = ms_total / args.steps
    peak, peak_src = measured_peak_gbs()
    achieved = px_per_step_rank * ALGO_BYTES_PER_PX / (ms_local / args.steps / 1e3) / 1e9  # this rank's kernel
    e2e_mpx = world * px_per_step_rank * e2e_steps / t_e2e / 1e6
    line = {
        "metric": "fused_4k_throughput", "value": mpx, "unit": "Mpixel/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "frames_per_gpu": n, "width": W, "height": H, "in_format": "RGB8",
                   "ksize": KSIZE, "sigma": SIGMA, "parallelism": f"frame-sharded x{world}, no collective",
                   "l2_policy": "batch (1.06 GB per step) larger than the 126 MB L2; no flush needed",
                   "dtype_note": "u8 in/out; gray in u32 integer arithmetic, blur/Sobel in fp32",
                   "content": "iid uniform noise (the friendliest content for the guard band; see the `content` key for others)"},
        "frames_per_s": mpx * 1e6 / (W * H),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": recorded_traffic_bytes(), "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": px_per_step_rank * ALGO_BYTES_PER_PX,
                     "frac_of_nominal_8TBs": achieved / 8000.0,
                     "note": "the kernel is issue / FMA-pipe bound, not HBM bound (profiles/README.md): frac is how far it is from the memory roofline"},
        "e2e": {"value": e2e_mpx, "unit": "Mpixel/s", "h2d_bytes_per_step": int(frames.nbytes) * world,
                "d2h_bytes_per_step": int(n * H * W) * world, "steps": e2e_steps,
                "frames_per_s": e2e_mpx * 1e6 / (W * H), "matches_resident_output": e2e_ok,
                "api": "rip_process_host (pinned host buffers, chunked H2D / kernel / D2H streams per device)",
                "host_numa_binding": numa or None},
        "gpu_launches": int(launches),
        "clocks": clocks,
    }
    if not args.no_extras:
        nv_mpx = world * px_per_step_rank * e2e_steps / t_nv / 1e6
        line["e2e_nv12"] = {"value": nv_mpx, "unit": "Mpixel/s", "h2d_bytes_per_step": int(nv.nbytes) * world,
                            "d2h_bytes_per_step": int(n * H * W) * world, "frames_per_s": nv_mpx * 1e6 / (W * H),
                            "note": "same leg, NV12 frames (luma plane + chroma plane uploaded, the kernel reads the luma plane)"}
        try:
            t0 = time.perf_counter()
            line["content"] = content_rows(rip, dev, stream, d_in, d_out, weights, peak)
            line["content"].insert(0, {"content": "iid_noise (headline)", "us_per_step": ms_local / args.steps * 1e3,
                                       "mpx_s": px_per_step_rank / (ms_local / args.steps * 1e3), "frac_of_hbm_peak": achieved / peak})
            d_in.free(); d_out.free()
            line["configs"] = config_rows(rip, dev, stream, peak)
            line["config5"] = config5_rows(rip, min(world, rip.device_count()), peak, weights)
            line["extras_seconds"] = time.perf_counter() - t0
        except Exception as e:  # noqa: BLE001 -- the headline must still be printed
            line["extras_error"] = f"{type(e).__name__}: {e}"
    if not args.no_cpu_baseline:
        fr = synth_batch(4, 0xB200 + 4000 + 1000 * rank)
        line["cpu_baseline"] = cpu_baseline(fr, weights)
        line["parity_spot_check"] = bool(np.array_equal(out0, _oracle().fused(fr[0], KSIZE, weights=weights, threads=0)))
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
