#!/usr/bin/env python
"""Times of the decoded camera formats: the NV12_COLOR, YUYV, UYVY and I420 decode kernels on device-resident data (the NV12_COLOR
legs are the same-session control for the others), the decode's share of GAUSSIAN, and the end-to-end host pipeline with
NV12_COLOR and YUYV against RGBA8 / BGR8 input.

    python tools/bench_nv12_color.py [--launches 21] > profiles/yuv_color_b200.txt

Kernel legs: CUDA events around each launch, 3 warm-up launches, the median of --launches (>= 20) launches; 32 x 3840x2160
frames are 398 MB of NV12 / I420 or 531 MB of YUYV / UYVY in and up to 1 GB out, far above the 126 MB L2.  Algorithmic bytes
per pixel: 1.5 (4:2:0) or 2 (4:2:2) in + the output's bytes per pixel out.  The share of peak is against the 6.55 TB/s device-to-device copy peak measured on a B200 (DESIGN.md).
End-to-end legs: rip_process_host from pinned host memory, wall clock over --e2e-steps blocking calls after 2 warm-up calls.
A sample of every timed output (first, middle and last frame) is checked against tests/nv12_ref.py / tests/yuv_ref.py and the C
oracle.
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import nv12_ref as R  # noqa: E402
import yuv_ref as YR  # noqa: E402
import oracle as O  # noqa: E402
import rip_b200 as rip  # noqa: E402

PEAK_GBS = 6550.0

ap = argparse.ArgumentParser()
ap.add_argument("--launches", type=int, default=21)
ap.add_argument("--e2e-steps", type=int, default=10)
a = ap.parse_args()
assert a.launches >= 20
if rip.device_count() < 1:
    sys.exit("bench_nv12_color.py needs a CUDA device (there is no CPU fallback)")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # noqa: BLE001
        q = f"nvidia-smi unavailable ({e})"
    return f"{rip.device_info(0).name.decode()}; nvidia-smi: {q}"


def timed(fn, n=a.launches, warm=3):
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(n):
        e0, e1 = rip.Event(), rip.Event()
        e0.record()
        fn()
        e1.record()
        e1.sync()
        ts.append(e0.elapsed_ns(e1) / 1e3)
    ts.sort()
    return ts[len(ts) // 2], ts[0]


def row(name, us, best, px, bpp, floor_note=True):
    gbs = px * bpp / us / 1e3
    floor = px * bpp / PEAK_GBS / 1e3
    extra = f"  floor {floor:7.1f} us  {100 * gbs / PEAK_GBS:5.1f} % of {PEAK_GBS:.0f} GB/s" if floor_note else ""
    print(f"{name:58s} {us:9.1f} us (best {best:8.1f})  {gbs:8.1f} GB/s ({bpp} B/px){extra}", flush=True)


def camera_like(n, h, w, seed):
    """Smooth luma + noise, slowly varying chroma (a decode is data-independent; the blur after it is not)."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    one = np.empty((h * 3 // 2, w), np.uint8)
    one[:h] = np.clip(120 + 90 * np.sin(0.01 * xx + 0.007 * yy) + rng.integers(-3, 4, (h, w)), 0, 255).astype(np.uint8)
    cy, cx = np.mgrid[0: h // 2, 0: w // 2].astype(np.float32)
    one[h:, 0::2] = np.clip(128 + 60 * np.sin(0.01 * cx), 0, 255).astype(np.uint8)
    one[h:, 1::2] = np.clip(128 + 60 * np.cos(0.013 * cy), 0, 255).astype(np.uint8)
    return np.stack([np.roll(one, 37 * i, axis=1) for i in range(n)])


def check(name, got, want):
    if not np.array_equal(got, want):
        raise SystemExit(f"{name}: timed output differs from the reference ({int((got != want).sum())} bytes)")


print(f"# {card()}")
print(f"# median of {a.launches} launches after 3 warm-up launches (CUDA events); copy peak {PEAK_GBS:.0f} GB/s", flush=True)

# ---- decode kernels, 32 x 4K --------------------------------------------------------------------------------------------------
N, H, W = 32, 2160, 3840
px = N * H * W
nv = camera_like(N, H, W, 1)
d_in = rip.DeviceBuffer(nv.nbytes).upload(nv)
d_out = rip.DeviceBuffer(px * 4)
sample = (0, N // 2, N - 1)
for order, fmt in (("rgba", rip.FMT_RGBA8), ("rgb", rip.FMT_RGB8)):
    us, best = timed(lambda: rip.convert_dev(d_in.ptr, d_out.ptr, W, H, N, rip.FMT_NV12_COLOR, fmt))
    row(f"rip_convert NV12_COLOR -> {order.upper()}8, {N} x {W}x{H}", us, best, px, 1.5 + len(order))
    fb = H * W * len(order)
    for i in sample:
        check(f"convert {order} frame {i}", d_out.download((H, W, len(order)), offset=i * fb), R.decode(nv[i], order))
for mode, bpp in ((rip.GRAY_OUT_U8, 1), (rip.GRAY_OUT_RGBA, 4)):
    us, best = timed(lambda: rip.gray_dev(d_in.ptr, d_out.ptr, W, H, N, rip.FMT_NV12_COLOR, mode))
    row(f"rip_gray NV12_COLOR -> {'u8' if bpp == 1 else '(g,g,g,255)'}, {N} x {W}x{H}", us, best, px, 1.5 + bpp)
    for i in sample:
        g = O.gray(R.decode(nv[i]), threads=0)
        got = d_out.download((H, W) if bpp == 1 else (H, W, 4), offset=i * H * W * bpp)
        check(f"gray frame {i}", got if bpp == 1 else got[..., 0], g)
del d_in


def packed_422(nv12, layout):
    """The camera-like NV12 frames as YUYV / UYVY: the same luma, each chroma row serving two luma rows."""
    out = np.empty((nv12.shape[0], H, W, 2), np.uint8)
    for i, f in enumerate(nv12):
        uv = np.repeat(f[H:].reshape(H // 2, W // 2, 2), 2, 0)
        out[i] = YR.packed_from_planes(f[:H], uv[..., 0], uv[..., 1], layout)
    return out


# ---- the other layouts, 32 x 4K: YUYV / UYVY (4:2:2, 2 B/px in) and I420 (4:2:0 planar, 1.5 B/px in) ---------------------------
LEGS = {"yuyv": (("rgba", "rgb"), True), "uyvy": (("rgba",), False), "i420": (("rgba",), True)}
for layout, (orders, with_gray) in LEGS.items():
    fmt = {"yuyv": rip.FMT_YUYV, "uyvy": rip.FMT_UYVY, "i420": rip.FMT_I420}[layout]
    src = np.stack([YR.i420_from_nv12(f) for f in nv]) if layout == "i420" else packed_422(nv, layout)
    in_b = src.nbytes / px
    d_in = rip.DeviceBuffer(src.nbytes).upload(src)
    for order in orders:
        ofmt = {"rgba": rip.FMT_RGBA8, "rgb": rip.FMT_RGB8}[order]
        us, best = timed(lambda: rip.convert_dev(d_in.ptr, d_out.ptr, W, H, N, fmt, ofmt))
        row(f"rip_convert {layout.upper()} -> {order.upper()}8, {N} x {W}x{H}", us, best, px, in_b + len(order))
        fb = H * W * len(order)
        for i in sample:
            check(f"convert {layout} {order} frame {i}", d_out.download((H, W, len(order)), offset=i * fb), YR.decode(src[i], layout, order))
    if with_gray:
        us, best = timed(lambda: rip.gray_dev(d_in.ptr, d_out.ptr, W, H, N, fmt, rip.GRAY_OUT_U8))
        row(f"rip_gray {layout.upper()} -> u8, {N} x {W}x{H}", us, best, px, in_b + 1)
        for i in sample:
            check(f"gray {layout} frame {i}", d_out.download((H, W), offset=i * H * W), O.gray(YR.decode(src[i], layout), threads=0))
    del d_in, src
del d_out

# ---- GAUSSIAN 5x5 on 16 x 1080p: decode + blur against the blur alone on RGBA8 ----------------------------------------------------
N, H, W = 16, 1080, 1920
px = N * H * W
nv = camera_like(N, H, W, 2)
wt = rip.gauss_weights(5, 1.0)
d_nv = rip.DeviceBuffer(nv.nbytes).upload(nv)
d_rgba = rip.DeviceBuffer(px * 4)
d_blur = rip.DeviceBuffer(px * 4)
rip.convert_dev(d_nv.ptr, d_rgba.ptr, W, H, N, rip.FMT_NV12_COLOR, rip.FMT_RGBA8)
us_blur, best = timed(lambda: rip.gauss_dev(d_rgba.ptr, d_blur.ptr, W, H, N, 4, 5, wt))
row(f"GAUSSIAN 5x5 blur alone, RGBA8, {N} x {W}x{H}", us_blur, best, px, 8)
us_dec, best = timed(lambda: rip.convert_dev(d_nv.ptr, d_rgba.ptr, W, H, N, rip.FMT_NV12_COLOR, rip.FMT_RGBA8))
row(f"decode NV12_COLOR -> RGBA8, {N} x {W}x{H}", us_dec, best, px, 5.5)


def both():
    rip.convert_dev(d_nv.ptr, d_rgba.ptr, W, H, N, rip.FMT_NV12_COLOR, rip.FMT_RGBA8)
    rip.gauss_dev(d_rgba.ptr, d_blur.ptr, W, H, N, 4, 5, wt)


us_both, best = timed(both)
row(f"decode + GAUSSIAN 5x5, NV12_COLOR, {N} x {W}x{H}", us_both, best, px, 5.5, floor_note=False)
print(f"  decode adds {us_both - us_blur:.1f} us = {100 * (us_both - us_blur) / us_blur:.1f} % of the blur alone", flush=True)
for i in (0, N - 1):
    check(f"blur frame {i}", d_blur.download((H, W, 4), offset=i * H * W * 4),
          O.blur(R.to_rgba(R.decode(nv[i])), 5, weights=wt, threads=0))
del d_nv, d_rgba, d_blur

# ---- end to end from pinned memory: NV12_COLOR against RGBA8 input -------------------------------------------------------------
ctx = rip.Context([0])
rgba = R.to_rgba(R.decode(nv))
print(f"# end to end, rip_process_host, pinned host buffers, {N} x {W}x{H}, wall clock over {a.e2e_steps} calls", flush=True)
yuyv = packed_422(nv, "yuyv")
bgr = R.decode(nv, "bgr")
NAMES = {rip.FMT_NV12_COLOR: "NV12_COLOR", rip.FMT_YUYV: "YUYV", rip.FMT_BGR8: "BGR8", rip.FMT_RGBA8: "RGBA8"}
for op, name, kw, inputs in ((rip.OP_GRAY, "GRAY", {}, ((rip.FMT_NV12_COLOR, nv), (rip.FMT_YUYV, yuyv), (rip.FMT_BGR8, bgr),
                                                        (rip.FMT_RGBA8, rgba))),
                             (rip.OP_GAUSSIAN, "GAUSSIAN 5x5", {"ksize": 5, "weights": wt}, ((rip.FMT_NV12_COLOR, nv), (rip.FMT_RGBA8, rgba)))):
    res = {}
    for fmt, src in inputs:
        h_in = rip.PinnedBuffer(src.nbytes)
        a_in = h_in.array.reshape(src.shape)
        a_in[...] = src
        out_bpp = 4 if op == rip.OP_GAUSSIAN else 1
        h_out = rip.PinnedBuffer(px * out_bpp)
        a_out = h_out.array.reshape((N, H, W, 4) if out_bpp == 4 else (N, H, W))
        for _ in range(2):
            ctx.process(a_in, op, fmt, out=a_out, **kw)
        t0 = time.perf_counter()
        for _ in range(a.e2e_steps):
            ctx.process(a_in, op, fmt, out=a_out, **kw)
        dt = (time.perf_counter() - t0) / a.e2e_steps
        res[fmt] = (dt, a_out.copy())
        in_b = src.nbytes / px
        print(f"  {name:13s} {NAMES[fmt]:10s} {dt * 1e3:8.2f} ms/call  "
              f"{px / dt / 1e9:6.2f} Gpx/s  ({in_b:.1f} B/px in, {out_bpp} B/px out)", flush=True)
        del a_in, a_out
        h_in.free()
        h_out.free()
    for fmt in res:
        check(f"e2e {name}: {NAMES[fmt]} vs RGBA8 of the decoded frames", res[fmt][1], res[rip.FMT_RGBA8][1])
    for fmt in [f for f in res if f not in (rip.FMT_RGBA8, rip.FMT_BGR8)]:
        for ref in [f for f in (rip.FMT_RGBA8, rip.FMT_BGR8) if f in res]:
            print(f"  {name}: {NAMES[fmt]} / {NAMES[ref]} speed {res[ref][0] / res[fmt][0]:.2f}x", flush=True)
ctx.close()
print("# every sampled output equal to the reference")
