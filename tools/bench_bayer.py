#!/usr/bin/env python
"""Times of the Bayer demosaic: the decode kernels on device-resident data, the decode's share of GAUSSIAN, and the end-to-end
host pipeline from Bayer against RGB8 and NV12_COLOR input.

    python tools/bench_bayer.py [--launches 21] > profiles/bayer_b200.txt
    python tools/bench_bayer.py --raw16 [--launches 21] > profiles/bayer16_b200.txt
    python tools/bench_bayer.py --packed [--launches 21] > profiles/bayer_packed_b200.txt

--raw16 times the 10- to 16-bit formats instead (2 bytes per pixel in): the kernel legs on 32 x 3840x2160 BAYER_RGGB12 and
BAYER_RGGB16, the demosaic's share of GAUSSIAN 5x5 on 16 x 1920x1080 BAYER_RGGB12, and the end-to-end legs from BAYER_RGGB12
against RGB8 of the same decoded image and against BAYER_RGGB8; outputs are checked against tests/bayer16_ref.py.

Kernel legs: CUDA events around each launch, 3 warm-up launches, the median of --launches (>= 20) launches; 32 x 3840x2160
Bayer frames are 265 MB in and up to 1.06 GB out, far above the 126 MB L2.  Algorithmic bytes per pixel: 1 in + the output's
bytes per pixel out.  The share of peak is against the 6.55 TB/s device-to-device copy peak measured on a B200 (DESIGN.md).
The gray leg is compared, in the same run, with the two-kernel route a caller has without it: rip_convert to RGB8, then
rip_gray on RGB8.
--packed times the packed 10- and 12-bit formats (MIPI CSI-2 and GenICam, 1.25 or 1.5 bytes per pixel in): the kernel legs on
32 x 3840x2160 RGGB in each layout beside the unpacked code of the same samples (BAYER_RGGB10 / 12), and the end-to-end legs
of 16 x 1920x1080 from each layout against BAYER_RGGB12 and BAYER_RGGB8.  Kernel legs: the first, middle and last frame of
every output against tests/bayer16_ref.py and the C oracle.  End-to-end legs: the first and last frame of every leg (packed or
not) against the oracle, and every packed leg in full against the unpacked code on the same samples.

End-to-end legs: rip_process_host from pinned host memory, wall clock over --e2e-steps blocking calls after 2 warm-up calls.
A sample of every timed output (first, middle and last frame) is checked against tests/bayer_ref.py and the C oracle.
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
import bayer16_ref as R16  # noqa: E402
import bayer_packed_ref as RP  # noqa: E402
import bayer_ref as R  # noqa: E402
import nv12_ref  # noqa: E402
import oracle as O  # noqa: E402
import rip_b200 as rip  # noqa: E402

PEAK_GBS = 6550.0

ap = argparse.ArgumentParser()
ap.add_argument("--launches", type=int, default=21)
ap.add_argument("--e2e-steps", type=int, default=10)
ap.add_argument("--raw16", action="store_true", help="time the 10- to 16-bit formats instead of the 8-bit ones")
ap.add_argument("--packed", action="store_true", help="time the packed 10- and 12-bit formats instead of the 8-bit ones")
a = ap.parse_args()
assert a.launches >= 20
if rip.device_count() < 1:
    sys.exit("bench_bayer.py needs a CUDA device (there is no CPU fallback)")


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
    """Raw frames of a smooth scene with sensor noise (a demosaic is data-independent; the blur after it is not)."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    one = np.clip(120 + 90 * np.sin(0.01 * xx + 0.007 * yy) + rng.integers(-3, 4, (h, w)), 0, 255).astype(np.uint8)
    return np.stack([np.roll(one, 37 * i, axis=1) for i in range(n)])


def check(name, got, want):
    if not np.array_equal(got, want):
        raise SystemExit(f"{name}: timed output differs from the reference ({int((got != want).sum())} bytes)")


def camera_like16(n, h, w, bits, seed):
    """camera_like at `bits` bits per sample: the same kind of scene, with the sensor noise of the deeper samples."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    top = (1 << bits) - 1
    one = np.clip(top * (0.47 + 0.35 * np.sin(0.01 * xx + 0.007 * yy)) + rng.integers(-3 << (bits - 8), 4 << (bits - 8), (h, w)),
                  0, top).astype(np.uint16)
    return np.stack([np.roll(one, 37 * i, axis=1) for i in range(n)])


def raw16_legs():
    # ---- decode kernels, 32 x 4K RGGB at 12 and at 16 bits: 2 B/px in --------------------------------------------------------
    N, H, W = 32, 2160, 3840
    px = N * H * W
    d_out = rip.DeviceBuffer(px * 4)
    d_rgb = rip.DeviceBuffer(px * 3)
    sample = (0, N // 2, N - 1)
    for bits in (12, 16):
        fmt, name = getattr(rip, f"FMT_BAYER_RGGB{bits}"), f"BAYER_RGGB{bits}"
        raw = camera_like16(N, H, W, bits, bits)
        d_in = rip.DeviceBuffer(raw.nbytes).upload(raw)
        want_rgb = {i: R16.decode(raw[i], "rggb", bits) for i in sample}
        for order, ofmt in (("rgba", rip.FMT_RGBA8), ("rgb", rip.FMT_RGB8)):
            us, best = timed(lambda: rip.convert_dev(d_in.ptr, d_out.ptr, W, H, N, fmt, ofmt))
            row(f"rip_convert {name} -> {order.upper()}8, {N} x {W}x{H}", us, best, px, 2 + len(order))
            fb = H * W * len(order)
            for i in sample:
                want = want_rgb[i] if order == "rgb" else np.concatenate([want_rgb[i], np.full((H, W, 1), 255, np.uint8)], -1)
                check(f"convert {name} {order} frame {i}", d_out.download((H, W, len(order)), offset=i * fb), want)
        want_gray = {i: O.gray(want_rgb[i], threads=0) for i in sample}
        us_gray, best = timed(lambda: rip.gray_dev(d_in.ptr, d_out.ptr, W, H, N, fmt, rip.GRAY_OUT_U8))
        row(f"rip_gray {name} -> u8, {N} x {W}x{H}", us_gray, best, px, 3)
        for i in sample:
            check(f"gray {name} frame {i}", d_out.download((H, W), offset=i * H * W), want_gray[i])

        def two_kernels():
            rip.convert_dev(d_in.ptr, d_rgb.ptr, W, H, N, fmt, rip.FMT_RGB8)
            rip.gray_dev(d_rgb.ptr, d_out.ptr, W, H, N, rip.FMT_RGB8, rip.GRAY_OUT_U8)

        us_two, best = timed(two_kernels)
        row(f"rip_convert -> RGB8, then rip_gray RGB8 -> u8, {name}", us_two, best, px, 3, floor_note=False)
        print(f"  rip_gray on {name} is {us_two / us_gray:.2f}x faster than the two-kernel route", flush=True)
        for i in sample:
            check(f"two-kernel gray {name} frame {i}", d_out.download((H, W), offset=i * H * W), want_gray[i])
        d_in.free()
        del raw
    d_out.free()
    d_rgb.free()

    # ---- GAUSSIAN 5x5 on 16 x 1080p: demosaic + blur against the blur alone on RGBA8 ------------------------------------------
    N, H, W = 16, 1080, 1920
    px = N * H * W
    fmt = rip.FMT_BAYER_RGGB12
    raw = camera_like16(N, H, W, 12, 2)
    wt = rip.gauss_weights(5, 1.0)
    d_raw = rip.DeviceBuffer(raw.nbytes).upload(raw)
    d_rgba = rip.DeviceBuffer(px * 4)
    d_blur = rip.DeviceBuffer(px * 4)
    rip.convert_dev(d_raw.ptr, d_rgba.ptr, W, H, N, fmt, rip.FMT_RGBA8)
    us_blur, best = timed(lambda: rip.gauss_dev(d_rgba.ptr, d_blur.ptr, W, H, N, 4, 5, wt))
    row(f"GAUSSIAN 5x5 blur alone, RGBA8, {N} x {W}x{H}", us_blur, best, px, 8)
    us_dec, best = timed(lambda: rip.convert_dev(d_raw.ptr, d_rgba.ptr, W, H, N, fmt, rip.FMT_RGBA8))
    row(f"demosaic BAYER_RGGB12 -> RGBA8, {N} x {W}x{H}", us_dec, best, px, 6)

    def both():
        rip.convert_dev(d_raw.ptr, d_rgba.ptr, W, H, N, fmt, rip.FMT_RGBA8)
        rip.gauss_dev(d_rgba.ptr, d_blur.ptr, W, H, N, 4, 5, wt)

    us_both, best = timed(both)
    row(f"demosaic + GAUSSIAN 5x5, BAYER_RGGB12, {N} x {W}x{H}", us_both, best, px, 6, floor_note=False)
    print(f"  demosaic adds {us_both - us_blur:.1f} us = {100 * (us_both - us_blur) / us_blur:.1f} % of the blur alone", flush=True)
    for i in (0, N - 1):
        check(f"blur frame {i}", d_blur.download((H, W, 4), offset=i * H * W * 4),
              O.blur(R16.decode(raw[i], "rggb", 12, "rgba"), 5, weights=wt, threads=0))
    d_raw.free()
    d_rgba.free()
    d_blur.free()

    # ---- end to end from pinned memory: BAYER_RGGB12 against RGB8 (the same decoded image) and BAYER_RGGB8 -------------------
    ctx = rip.Context([0])
    rgb = R16.decode(raw, "rggb", 12)
    raw8 = camera_like(N, H, W, 2)
    print(f"# end to end, rip_process_host, pinned host buffers, {N} x {W}x{H}, wall clock over {a.e2e_steps} calls", flush=True)
    names = {fmt: "BAYER_RGGB12", rip.FMT_RGB8: "RGB8", rip.FMT_BAYER_RGGB8: "BAYER_RGGB8"}
    for op, name, kw in ((rip.OP_GRAY, "GRAY", {}), (rip.OP_EDGE, "EDGE", {}), (rip.OP_FUSED, "FUSED 5x5", {"ksize": 5, "weights": wt})):
        res = {}
        for f, src in ((fmt, raw), (rip.FMT_RGB8, rgb), (rip.FMT_BAYER_RGGB8, raw8)):
            h_in = rip.PinnedBuffer(src.nbytes)
            a_in = h_in.array.view(src.dtype).reshape(src.shape)
            a_in[...] = src
            h_out = rip.PinnedBuffer(px)
            a_out = h_out.array.reshape((N, H, W))
            for _ in range(2):
                ctx.process(a_in, op, f, out=a_out, **kw)
            t0 = time.perf_counter()
            for _ in range(a.e2e_steps):
                ctx.process(a_in, op, f, out=a_out, **kw)
            dt = (time.perf_counter() - t0) / a.e2e_steps
            res[f] = (dt, a_out.copy())
            print(f"  {name:10s} {names[f]:12s} {dt * 1e3:8.2f} ms/call  {px / dt / 1e9:6.2f} Gpx/s  "
                  f"({src.nbytes / px:.1f} B/px in, 1 B/px out)", flush=True)
            del a_in, a_out
            h_in.free()
            h_out.free()
        check(f"e2e {name}: BAYER_RGGB12 vs RGB8 of the decoded frames", res[fmt][1], res[rip.FMT_RGB8][1])
        for ref in (rip.FMT_RGB8, rip.FMT_BAYER_RGGB8):
            print(f"  {name}: BAYER_RGGB12 / {names[ref]} speed {res[ref][0] / res[fmt][0]:.2f}x", flush=True)
    ctx.close()
    print("# every sampled output equal to the reference")


PACKED_FMT = {"mipi10": "10P_MIPI", "mipi12": "12P_MIPI", "genicam10": "10P_GENICAM", "genicam12": "12P_GENICAM"}


def packed_frames(n, h, w, layout, seed):
    """camera_like16 samples, packed: one frame packed, the others its rolls by 40 columns (a whole number of bytes in every
    layout), so that 32 4K frames need no packing pass of their own.  Returns (packed, samples)."""
    bits = RP.bits_of(layout)
    one = camera_like16(1, h, w, bits, seed)[0]
    p1 = RP.pack(one, layout)
    step = RP.row_bytes(layout, 40)
    packed = np.stack([np.roll(p1, step * i, axis=1) for i in range(n)])
    samples = np.stack([np.roll(one, 40 * i, axis=1) for i in range(n)])
    return packed, samples


def packed_legs():
    # ---- decode kernels, 32 x 4K RGGB in each layout, beside the unpacked code of the same samples ----------------------------
    N, H, W = 32, 2160, 3840
    px = N * H * W
    d_out = rip.DeviceBuffer(px * 4)
    sample = (0, N // 2, N - 1)
    for layout in RP.LAYOUTS:
        bits = RP.bits_of(layout)
        packed, samples = packed_frames(N, H, W, layout, bits)
        assert np.array_equal(RP.unpack(packed[N - 1], layout), samples[N - 1])
        fmt, name = getattr(rip, f"FMT_BAYER_RGGB{PACKED_FMT[layout]}"), f"BAYER_RGGB{PACKED_FMT[layout]}"
        u16, u16_name = getattr(rip, f"FMT_BAYER_RGGB{bits}"), f"BAYER_RGGB{bits}"
        d_in = rip.DeviceBuffer(packed.nbytes).upload(packed)
        d_u16 = rip.DeviceBuffer(samples.nbytes).upload(samples)
        bpp_in = bits / 8
        want_rgb = {i: R16.decode(samples[i], "rggb", bits) for i in sample}
        want_gray = {i: O.gray(want_rgb[i], threads=0) for i in sample}
        for order, ofmt in (("rgba", rip.FMT_RGBA8), ("rgb", rip.FMT_RGB8), ("gray", None)):
            nb = 1 if order == "gray" else len(order)
            res = {}
            for f, nm, src, b_in in ((fmt, name, d_in, bpp_in), (u16, u16_name, d_u16, 2)):
                if order == "gray":
                    us, best = timed(lambda: rip.gray_dev(src.ptr, d_out.ptr, W, H, N, f, rip.GRAY_OUT_U8))
                else:
                    us, best = timed(lambda: rip.convert_dev(src.ptr, d_out.ptr, W, H, N, f, ofmt))
                res[f] = us
                label = "rip_gray" if order == "gray" else "rip_convert"
                row(f"{label} {nm} -> {order.upper()}{'8' if order != 'gray' else ' u8'}, {N} x {W}x{H}", us, best, px, b_in + nb)
                for i in sample:
                    shape = (H, W) if order == "gray" else (H, W, nb)
                    got = d_out.download(shape, offset=i * H * W * nb)
                    if order == "gray":
                        want = want_gray[i]
                    else:
                        want = want_rgb[i] if order == "rgb" else np.concatenate([want_rgb[i], np.full((H, W, 1), 255, np.uint8)], -1)
                    check(f"{label} {nm} {order} frame {i}", got, want)
            print(f"  {order}: {name} / {u16_name} time {res[fmt] / res[u16]:.2f}", flush=True)
        d_in.free()
        d_u16.free()
        del packed, samples
    d_out.free()

    # ---- end to end from pinned memory, 16 x 1080p: each layout against BAYER_RGGB12 and BAYER_RGGB8 -------------------------
    N, H, W = 16, 1080, 1920
    px = N * H * W
    wt = rip.gauss_weights(5, 1.0)
    ctx = rip.Context([0])
    # (format, name, host frames, the unpacked code and samples of the same frames or None, decoded RGB of frame i)
    srcs = []
    for layout in RP.LAYOUTS:
        bits = RP.bits_of(layout)
        packed, samples = packed_frames(N, H, W, layout, 2)
        srcs.append((getattr(rip, f"FMT_BAYER_RGGB{PACKED_FMT[layout]}"), f"BAYER_RGGB{PACKED_FMT[layout]}", packed,
                     (getattr(rip, f"FMT_BAYER_RGGB{bits}"), samples),
                     lambda i, s=samples, b=bits: R16.decode(s[i], "rggb", b)))
    raw12, raw8 = camera_like16(N, H, W, 12, 2), camera_like(N, H, W, 2)
    srcs.append((rip.FMT_BAYER_RGGB12, "BAYER_RGGB12", raw12, None, lambda i: R16.decode(raw12[i], "rggb", 12)))
    srcs.append((rip.FMT_BAYER_RGGB8, "BAYER_RGGB8", raw8, None, lambda i: R.decode(raw8[i], "rggb")))
    print(f"# end to end, rip_process_host, pinned host buffers, {N} x {W}x{H}, wall clock over {a.e2e_steps} calls", flush=True)
    for op, name, kw in ((rip.OP_GRAY, "GRAY", {}), (rip.OP_EDGE, "EDGE", {}), (rip.OP_FUSED, "FUSED 5x5", {"ksize": 5, "weights": wt})):
        res = {}
        for f, nm, src, ref, rgb_of in srcs:
            h_in = rip.PinnedBuffer(src.nbytes)
            a_in = h_in.array.view(src.dtype).reshape(src.shape)
            a_in[...] = src
            h_out = rip.PinnedBuffer(px)
            a_out = h_out.array.reshape((N, H, W))
            for _ in range(2):
                ctx.process(a_in, op, f, out=a_out, **kw)
            t0 = time.perf_counter()
            for _ in range(a.e2e_steps):
                ctx.process(a_in, op, f, out=a_out, **kw)
            dt = (time.perf_counter() - t0) / a.e2e_steps
            res[nm] = dt
            print(f"  {name:10s} {nm:26s} {dt * 1e3:8.2f} ms/call  {px / dt / 1e9:6.2f} Gpx/s  "
                  f"({src.nbytes / px:.2f} B/px in, 1 B/px out)", flush=True)
            if ref is not None:
                check(f"e2e {name} {nm} vs the unpacked code", a_out, ctx.process(ref[1], op, ref[0], **kw))
            for i in (0, N - 1):
                rgb = rgb_of(i)
                want = O.gray(rgb, threads=0) if op == rip.OP_GRAY else \
                    O.sobel(O.gray(rgb, threads=0), threads=0) if op == rip.OP_EDGE else O.fused(rgb, 5, weights=wt, threads=0)
                check(f"e2e {name} {nm} frame {i} vs the oracle", a_out[i], want)
            del a_in, a_out
            h_in.free()
            h_out.free()
        for nm in [x[1] for x in srcs[:4]]:
            print(f"  {name}: {nm} speed against BAYER_RGGB12 {res['BAYER_RGGB12'] / res[nm]:.2f}x, "
                  f"against BAYER_RGGB8 {res['BAYER_RGGB8'] / res[nm]:.2f}x", flush=True)
    ctx.close()
    print("# every sampled output equal to the reference")


print(f"# {card()}")
print(f"# median of {a.launches} launches after 3 warm-up launches (CUDA events); copy peak {PEAK_GBS:.0f} GB/s", flush=True)
if a.raw16:
    raw16_legs()
    sys.exit(0)
if a.packed:
    packed_legs()
    sys.exit(0)

# ---- decode kernels, 32 x 4K RGGB ---------------------------------------------------------------------------------------------
N, H, W = 32, 2160, 3840
px = N * H * W
FMT = rip.FMT_BAYER_RGGB8
raw = camera_like(N, H, W, 1)
d_in = rip.DeviceBuffer(raw.nbytes).upload(raw)
d_out = rip.DeviceBuffer(px * 4)
d_rgb = rip.DeviceBuffer(px * 3)
sample = (0, N // 2, N - 1)
want_rgb = {i: R.decode(raw[i], "rggb") for i in sample}
for order, fmt in (("rgba", rip.FMT_RGBA8), ("rgb", rip.FMT_RGB8)):
    us, best = timed(lambda: rip.convert_dev(d_in.ptr, d_out.ptr, W, H, N, FMT, fmt))
    row(f"rip_convert BAYER_RGGB8 -> {order.upper()}8, {N} x {W}x{H}", us, best, px, 1 + len(order))
    fb = H * W * len(order)
    for i in sample:
        want = want_rgb[i] if order == "rgb" else np.concatenate([want_rgb[i], np.full((H, W, 1), 255, np.uint8)], -1)
        check(f"convert {order} frame {i}", d_out.download((H, W, len(order)), offset=i * fb), want)
want_gray = {i: O.gray(want_rgb[i], threads=0) for i in sample}
us_gray, best = timed(lambda: rip.gray_dev(d_in.ptr, d_out.ptr, W, H, N, FMT, rip.GRAY_OUT_U8))
row(f"rip_gray BAYER_RGGB8 -> u8, {N} x {W}x{H}", us_gray, best, px, 2)
for i in sample:
    check(f"gray frame {i}", d_out.download((H, W), offset=i * H * W), want_gray[i])


def two_kernels():
    rip.convert_dev(d_in.ptr, d_rgb.ptr, W, H, N, FMT, rip.FMT_RGB8)
    rip.gray_dev(d_rgb.ptr, d_out.ptr, W, H, N, rip.FMT_RGB8, rip.GRAY_OUT_U8)


us_two, best = timed(two_kernels)
row(f"rip_convert -> RGB8, then rip_gray RGB8 -> u8, {N} x {W}x{H}", us_two, best, px, 2, floor_note=False)
print(f"  rip_gray on Bayer is {us_two / us_gray:.2f}x faster than the two-kernel route", flush=True)
for i in sample:
    check(f"two-kernel gray frame {i}", d_out.download((H, W), offset=i * H * W), want_gray[i])
us, best = timed(lambda: rip.convert_dev(d_in.ptr, d_out.ptr, W, H, N, rip.FMT_BAYER_GBRG8, rip.FMT_RGBA8))
row(f"rip_convert BAYER_GBRG8 -> RGBA8, {N} x {W}x{H}", us, best, px, 5)
del d_in, d_out, d_rgb, raw

# ---- GAUSSIAN 5x5 on 16 x 1080p: demosaic + blur against the blur alone on RGBA8 ---------------------------------------------------
N, H, W = 16, 1080, 1920
px = N * H * W
raw = camera_like(N, H, W, 2)
wt = rip.gauss_weights(5, 1.0)
d_raw = rip.DeviceBuffer(raw.nbytes).upload(raw)
d_rgba = rip.DeviceBuffer(px * 4)
d_blur = rip.DeviceBuffer(px * 4)
rip.convert_dev(d_raw.ptr, d_rgba.ptr, W, H, N, FMT, rip.FMT_RGBA8)
us_blur, best = timed(lambda: rip.gauss_dev(d_rgba.ptr, d_blur.ptr, W, H, N, 4, 5, wt))
row(f"GAUSSIAN 5x5 blur alone, RGBA8, {N} x {W}x{H}", us_blur, best, px, 8)
us_dec, best = timed(lambda: rip.convert_dev(d_raw.ptr, d_rgba.ptr, W, H, N, FMT, rip.FMT_RGBA8))
row(f"demosaic BAYER_RGGB8 -> RGBA8, {N} x {W}x{H}", us_dec, best, px, 5)


def both():
    rip.convert_dev(d_raw.ptr, d_rgba.ptr, W, H, N, FMT, rip.FMT_RGBA8)
    rip.gauss_dev(d_rgba.ptr, d_blur.ptr, W, H, N, 4, 5, wt)


us_both, best = timed(both)
row(f"demosaic + GAUSSIAN 5x5, BAYER_RGGB8, {N} x {W}x{H}", us_both, best, px, 5, floor_note=False)
print(f"  demosaic adds {us_both - us_blur:.1f} us = {100 * (us_both - us_blur) / us_blur:.1f} % of the blur alone", flush=True)
for i in (0, N - 1):
    check(f"blur frame {i}", d_blur.download((H, W, 4), offset=i * H * W * 4),
          O.blur(R.decode(raw[i], "rggb", "rgba"), 5, weights=wt, threads=0))
del d_raw, d_rgba, d_blur

# ---- end to end from pinned memory: Bayer against RGB8 (the same decoded image) and NV12_COLOR --------------------------------------
ctx = rip.Context([0])
rgb = R.decode(raw, "rggb")
nv = np.empty((N, H * 3 // 2, W), np.uint8)
nv[:, :H] = raw
nv[:, H:] = 128   # neutral chroma; the NV12 leg is timed only
print(f"# end to end, rip_process_host, pinned host buffers, {N} x {W}x{H}, wall clock over {a.e2e_steps} calls", flush=True)
NAMES = {FMT: "BAYER_RGGB8", rip.FMT_RGB8: "RGB8", rip.FMT_NV12_COLOR: "NV12_COLOR"}
for op, name, kw in ((rip.OP_GRAY, "GRAY", {}), (rip.OP_EDGE, "EDGE", {}), (rip.OP_FUSED, "FUSED 5x5", {"ksize": 5, "weights": wt})):
    res = {}
    for fmt, src in ((FMT, raw), (rip.FMT_RGB8, rgb), (rip.FMT_NV12_COLOR, nv)):
        h_in = rip.PinnedBuffer(src.nbytes)
        a_in = h_in.array.reshape(src.shape)
        a_in[...] = src
        h_out = rip.PinnedBuffer(px)
        a_out = h_out.array.reshape((N, H, W))
        for _ in range(2):
            ctx.process(a_in, op, fmt, out=a_out, **kw)
        t0 = time.perf_counter()
        for _ in range(a.e2e_steps):
            ctx.process(a_in, op, fmt, out=a_out, **kw)
        dt = (time.perf_counter() - t0) / a.e2e_steps
        res[fmt] = (dt, a_out.copy())
        print(f"  {name:10s} {NAMES[fmt]:12s} {dt * 1e3:8.2f} ms/call  {px / dt / 1e9:6.2f} Gpx/s  "
              f"({src.nbytes / px:.1f} B/px in, 1 B/px out)", flush=True)
        del a_in, a_out
        h_in.free()
        h_out.free()
    check(f"e2e {name}: BAYER_RGGB8 vs RGB8 of the decoded frames", res[FMT][1], res[rip.FMT_RGB8][1])
    if op == rip.OP_GRAY:
        check("e2e GRAY NV12_COLOR", res[rip.FMT_NV12_COLOR][1][0], O.gray(nv12_ref.decode(nv[0]), threads=0))
    for ref in (rip.FMT_RGB8, rip.FMT_NV12_COLOR):
        print(f"  {name}: BAYER_RGGB8 / {NAMES[ref]} speed {res[ref][0] / res[FMT][0]:.2f}x", flush=True)
ctx.close()
print("# every sampled output equal to the reference")
