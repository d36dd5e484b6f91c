"""RIP_FMT_BAYER_RGGB8 / _BGGR8 / _GRBG8 / _GBRG8: 8-bit Bayer raw frames demosaiced exactly as OpenCV's default
cvtColor(COLOR_Bayer**2RGB) does, then the reference's chain on that colour image (GRAYSCALE its gray, GAUSSIAN the blur of
the RGBA image with alpha 255, EDGE / FUSED their result on its gray) -- the contract of the YUV formats, for raw sensors.

CPU tests pin the numpy restatement of the demosaic (tests/bayer_ref.py) to live cv2 and to the cv2 outputs recorded in
tests/golden/cv2_bayer.npz, and pin the pattern names against OpenCV's.  GPU tests compare every device path with that
restatement followed by the C oracle, bit for bit."""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np
import pytest

import bayer_ref as R
import rip_b200 as rip

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "opencl-development-real-time-image-processing_b200")
GOLDEN = os.path.join(ROOT, "tests", "golden", "cv2_bayer.npz")
FMT = {"rggb": rip.FMT_BAYER_RGGB8, "bggr": rip.FMT_BAYER_BGGR8, "grbg": rip.FMT_BAYER_GRBG8, "gbrg": rip.FMT_BAYER_GBRG8}
OUT_FMT = {"rgb": rip.FMT_RGB8, "bgr": rip.FMT_BGR8, "rgba": rip.FMT_RGBA8, "bgra": rip.FMT_BGRA8}


def _eq(got, want, what=""):
    if not np.array_equal(got, want):
        d = np.abs(got.astype(int) - want.astype(int))
        idx = np.argwhere(d > 0)
        raise AssertionError(f"{what}: {len(idx)} of {d.size} bytes differ, max abs {d.max()}, first at {idx[0].tolist()}")


def _noise(n, h, w, seed):
    return np.random.default_rng(seed).integers(0, 256, (n, h, w), dtype=np.uint8)


def _in_order(rgb, order):
    """An RGB image (.., 3) in another channel order (alpha 255)."""
    out = rgb[..., ::-1] if order.startswith("bgr") else rgb
    if len(order) == 4:
        out = np.concatenate([out, np.full(out.shape[:-1] + (1,), 255, np.uint8)], -1)
    return np.ascontiguousarray(out)


def _out_bytes(op, fmt, w, h, gray_out=rip.GRAY_OUT_U8):
    d = rip.OpDesc()
    d.op, d.in_format, d.gray_out = op, fmt, gray_out
    b = C.c_size_t(0)
    rip.check(rip.lib().rip_out_bytes_per_frame(C.byref(d), w, h, C.byref(b)))
    return b.value


# ---- CPU: the demosaic restatement, the pattern names, the host-side sizes and shapes ------------------------------------
SHAPES_CV2 = [(3, 3), (3, 4), (4, 3), (5, 5), (7, 9), (6, 9), (9, 6), (16, 24), (1023, 683)]   # (H, W)


@pytest.mark.parametrize("pattern", R.PATTERNS)
def test_reference_equals_cv2(pattern):
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(31)
    g = np.load(GOLDEN)
    frames = [rng.integers(0, 256, s, dtype=np.uint8) for s in SHAPES_CV2]
    frames += [f for k in g.files if k.endswith(".in") and k != "artemis.in" for f in g[k]]
    for f in frames:
        for order in R.ORDERS:
            _eq(R.decode(f, pattern, order), R.cv2_decode(f, pattern, order), f"{pattern} {order} {f.shape} vs cv2 {cv2.__version__}")


def test_reference_equals_recorded_cv2():
    g = np.load(GOLDEN)
    cases = [k[:-3] for k in g.files if k.endswith(".in") and k != "artemis.in"]
    assert {"noise3x3", "noise3x4", "noise4x3", "noise7x9", "noise6x9", "flat", "lattice", "impulse5x5", "hramp", "vramp"} <= set(cases)
    for case in cases:
        for pattern in R.PATTERNS:
            for order in ("rgb", "bgra"):
                _eq(R.decode(g[case + ".in"], pattern, order), g[f"{pattern}.{case}.{order}"], f"{pattern} {case} {order}")
    artemis = g["artemis.in"]
    assert artemis.shape == (1023, 683)
    for pattern in R.PATTERNS:
        for order in R.ORDERS:
            digest = hashlib.sha256(R.decode(artemis, pattern, order).tobytes()).digest()
            assert digest == g[f"{pattern}.artemis.{order}.sha256"].tobytes(), f"{pattern} {order} 683x1023"


def test_pattern_names_against_opencv():
    """Patterns are named by the top-left 2x2 (V4L2, GenICam); OpenCV names them by the 2x2 at (1, 1).  A frame that holds
    255 on the named red sites only must decode to pure red inside, on every pattern; and OpenCV's codes are pinned."""
    assert R.CV2_CODE == {"rggb": "BG", "bggr": "RG", "grbg": "GB", "gbrg": "GR"}
    yy, xx = np.mgrid[0:8, 0:10]
    for pattern, name in (("rggb", "RGGB"), ("bggr", "BGGR"), ("grbg", "GRBG"), ("gbrg", "GBRG")):
        f = np.zeros((8, 10), np.uint8)
        for i, ch in enumerate(name):   # R at its place in the 2x2, the rest 0
            if ch == "R":
                f[((yy & 1) == i // 2) & ((xx & 1) == i % 2)] = 255
        rgb = R.decode(f, pattern)
        assert (rgb[..., 0] > 0).all() and (rgb[..., 1:] == 0).all(), pattern
    cv2 = pytest.importorskip("cv2")
    for pattern, code in R.CV2_CODE.items():
        f = np.random.default_rng(5).integers(0, 256, (12, 14), dtype=np.uint8)
        _eq(R.decode(f, pattern), cv2.cvtColor(f, getattr(cv2, f"COLOR_Bayer{code}2RGB")), f"{pattern} = COLOR_Bayer{code}2RGB")


def test_output_sizes_of_the_bayer_formats():
    w, h = 683, 1023
    for fmt in FMT.values():
        assert _out_bytes(rip.OP_GAUSSIAN, fmt, w, h) == w * h * 4
        assert _out_bytes(rip.OP_GRAY, fmt, w, h) == w * h
        assert _out_bytes(rip.OP_GRAY, fmt, w, h, rip.GRAY_OUT_RGBA) == w * h * 4
        assert _out_bytes(rip.OP_EDGE, fmt, w, h) == w * h
        assert _out_bytes(rip.OP_FUSED, fmt, w, h) == w * h


def test_python_shapes_of_the_bayer_formats():
    """Context.process / submit take Bayer frames as (N, H, W) or (H, W): one raw byte per pixel."""
    c = object.__new__(rip.Context)   # the shape handling needs no device
    for fmt in FMT.values():
        assert rip.CHANNELS[fmt] == 1
        a, _, n, h, w, shape, out, squeeze = c._shapes(np.zeros((3, 5, 7), np.uint8), rip.OP_GAUSSIAN, fmt,
                                                        rip.GRAY_OUT_U8, 5, rip.gauss_weights(5, 1.0), None)
        assert (n, h, w, shape, out.shape, squeeze) == (3, 5, 7, (3, 5, 7, 4), (3, 5, 7, 4), False)
        a, _, n, h, w, shape, out, squeeze = c._shapes(np.zeros((5, 7), np.uint8), rip.OP_EDGE, fmt,
                                                        rip.GRAY_OUT_U8, 0, None, None)
        assert (a.shape, n, h, w, shape, squeeze) == ((1, 5, 7), 1, 5, 7, (1, 5, 7), True)
        a, _, n, h, w, shape, out, squeeze = c._shapes(np.zeros((2, 9, 10), np.uint8), rip.OP_GRAY, fmt,
                                                        rip.GRAY_OUT_RGBA, 0, None, None)
        assert (n, h, w, shape, squeeze) == (2, 9, 10, (2, 9, 10, 4), False)


@pytest.mark.skipif(rip.device_count() > 0, reason="only meaningful on a box without a GPU")
def test_bayer_fails_loudly_without_gpu():
    for fmt in FMT.values():
        with pytest.raises(rip.RipError, match="no CUDA device|no CPU fallback"):
            rip.convert_dev(16, 32, 4, 4, 1, fmt, rip.FMT_RGBA8)
        with pytest.raises(rip.RipError, match="no CUDA device|no CPU fallback"):
            rip.gray_dev(16, 32, 4, 4, 1, fmt)


def _build_dropin(tmp_path):
    exe = str(tmp_path / "bayer_dropin")
    cmd = ["/usr/bin/g++", "-O2", "-std=c++17", "-ffp-contract=off", "-I", os.path.join(PKG, "host"), "-I", os.path.join(ROOT, "include"),
           "-I", "/usr/local/cuda/include", os.path.join(ROOT, "tests", "cpp", "bayer_dropin.cpp"), "-o", exe, "-L", PKG, "-lrip_host",
           "-lrip_cuda", "-Wl,-rpath," + PKG, "-pthread"]
    subprocess.run(cmd, check=True)
    return exe


def test_cpp_driver_builds(tmp_path):
    exe = _build_dropin(tmp_path)
    res = subprocess.run([exe], capture_output=True, text=True)
    assert res.returncode == 2 and "usage" in res.stderr


# ---- GPU -------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    if rip.device_count() < 1:
        pytest.fail("GPU tests need a CUDA device: librip_cuda has no CPU fallback")
    c = rip.Context([0])
    yield c
    c.close()


def _convert(pattern, fr, order, in_off=0, out_off=0):
    n, h, w = fr.shape
    bpp = len(order)
    d_in = rip.DeviceBuffer(fr.nbytes + 16).upload(fr, offset=in_off)
    d_out = rip.DeviceBuffer(n * h * w * bpp + 16)
    rip.convert_dev(d_in.ptr + in_off, d_out.ptr + out_off, w, h, n, FMT[pattern], OUT_FMT[order])
    return d_out.download((n, h, w, bpp), offset=out_off)


def _gray_dev(pattern, fr, out_mode, in_off=0, out_off=0):
    n, h, w = fr.shape
    bpp = 4 if out_mode == rip.GRAY_OUT_RGBA else 1
    d_in = rip.DeviceBuffer(fr.nbytes + 16).upload(fr, offset=in_off)
    d_out = rip.DeviceBuffer(n * h * w * bpp + 16)
    rip.gray_dev(d_in.ptr + in_off, d_out.ptr + out_off, w, h, n, FMT[pattern], out_mode)
    return d_out.download((n, h, w, bpp) if bpp == 4 else (n, h, w), offset=out_off)


def _want_gray(oracle, pattern, fr):
    return np.stack([oracle.gray(R.decode(f, pattern), threads=0) for f in fr])


def _gray_rgba(g):
    return np.stack([g, g, g, np.full_like(g, 255)], -1)


# (n, h, w): W % 8 != 0 and odd W take the byte-granular kernel, W % 8 == 0 the wide one (also with odd H, H = 3 and H = 4,
# where every row pair is a border pair); odd W * H makes the frame stride odd, so every second frame is unaligned
SHAPES = [(1, 3, 3), (3, 3, 4), (2, 4, 3), (3, 5, 5), (2, 7, 9), (3, 6, 9), (2, 9, 6), (3, 3, 8), (2, 4, 8), (2, 9, 16),
          (3, 74, 76), (2, 75, 77), (1, 1023, 683), (2, 121, 1920), (1, 2160, 3840)]


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", R.PATTERNS)
@pytest.mark.parametrize("n,h,w", SHAPES)
def test_convert_shapes_and_batches(ctx, pattern, n, h, w):
    fr = _noise(n, h, w, 100 + h + w)
    rgb = R.decode(fr, pattern)
    for order in R.ORDERS:
        _eq(_convert(pattern, fr, order), _in_order(rgb, order), f"rip_convert {pattern} {order} {n}x{h}x{w}")


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", R.PATTERNS)
def test_convert_recorded_cases(ctx, pattern):
    """The adversarial frames of the golden file (flat, checkerboards, single-site lattices, impulses, ramps) through the device."""
    g = np.load(GOLDEN)
    for case in [k[:-3] for k in g.files if k.endswith(".in") and k != "artemis.in"]:
        fr = g[case + ".in"]
        for order in ("rgb", "bgra"):
            _eq(_convert(pattern, fr, order), g[f"{pattern}.{case}.{order}"], f"rip_convert {pattern} {case} {order} vs cv2")


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", R.PATTERNS)
@pytest.mark.parametrize("in_off,out_off", [(1, 0), (0, 1), (4, 12), (8, 8), (12, 4)])
def test_convert_and_gray_unaligned_buffers(ctx, oracle, pattern, in_off, out_off):
    """Offsets 4, 8 and 12 keep 4-byte alignment but break the 8- or 16-byte alignment the wide kernel needs."""
    fr = _noise(3, 6, 24, 7)
    rgb = R.decode(fr, pattern)
    for order in R.ORDERS:
        _eq(_convert(pattern, fr, order, in_off, out_off), _in_order(rgb, order), f"rip_convert {pattern} {order} offsets {in_off}/{out_off}")
    g = _want_gray(oracle, pattern, fr)
    _eq(_gray_dev(pattern, fr, rip.GRAY_OUT_U8, in_off, out_off), g, f"rip_gray {pattern} u8 unaligned")
    _eq(_gray_dev(pattern, fr, rip.GRAY_OUT_RGBA, in_off, out_off), _gray_rgba(g), f"rip_gray {pattern} rgba unaligned")


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", R.PATTERNS)
@pytest.mark.parametrize("n,h,w", [(1, 2160, 3840), (3, 74, 76), (2, 75, 77), (2, 3, 3), (2, 1080, 1920)])
def test_gray_dev_both_out_modes(ctx, oracle, pattern, n, h, w):
    fr = _noise(n, h, w, 5 + w)
    g = _want_gray(oracle, pattern, fr)
    _eq(_gray_dev(pattern, fr, rip.GRAY_OUT_U8), g, f"rip_gray {pattern} u8 {n}x{h}x{w}")
    _eq(_gray_dev(pattern, fr, rip.GRAY_OUT_RGBA), _gray_rgba(g), f"rip_gray {pattern} rgba {n}x{h}x{w}")


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", R.PATTERNS)
@pytest.mark.parametrize("h,w", [(64, 96), (9, 13)])
def test_gray_flat_frames_take_the_table(ctx, oracle, pattern, h, w):
    """A constant raw value gives r = g = b, so t = 1000 v and every pixel takes the (r, g) table path."""
    fr = np.stack([np.full((h, w), v, np.uint8) for v in range(256)])
    g = _want_gray(oracle, pattern, fr)
    _eq(_gray_dev(pattern, fr, rip.GRAY_OUT_U8), g, f"flat rip_gray {pattern} u8")
    _eq(_gray_dev(pattern, fr, rip.GRAY_OUT_RGBA), _gray_rgba(g), f"flat rip_gray {pattern} rgba")
    _eq(ctx.process(fr, rip.OP_GRAY, FMT[pattern]), g, f"flat GRAY {pattern}")


def _smooth(n, h, w, seed):
    """Camera-like raw frames: smooth content with noise and a flat black bar (the blur's constant windows)."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    out = []
    for _ in range(n):
        fx, fy, ph = rng.uniform(0.002, 0.03), rng.uniform(0.002, 0.03), rng.uniform(0, 6.28)
        f = np.clip(120 + 90 * np.sin(fx * xx + fy * yy + ph) + rng.integers(-3, 4, (h, w)), 0, 255).astype(np.uint8)
        f[: h // 8] = 0
        out.append(f)
    return np.stack(out)


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", R.PATTERNS)
@pytest.mark.parametrize("k,sigma", [(5, 1.5), (9, 2.5), (17, 6.0)])
@pytest.mark.parametrize("kernel", ["RIP_BLUR_STREAM", "RIP_BLUR_TILED"])
def test_pipeline_gaussian(ctx, oracle, opt, pattern, k, sigma, kernel):
    """Demosaic to RGBA, then the streaming or the tiled blur kernel, forced."""
    opt(kernel, 1)
    wt = rip.gauss_weights(k, sigma)
    for fr in (_smooth(2, 270, 480, k), _noise(2, 121, 163, k)):
        n, h, w = fr.shape
        got = ctx.process(fr, rip.OP_GAUSSIAN, FMT[pattern], ksize=k, weights=wt)
        assert got.shape == (n, h, w, 4)
        for i in range(n):
            want = oracle.blur(R.decode(fr[i], pattern, "rgba"), k, weights=wt, threads=0)
            _eq(got[i], want, f"GAUSSIAN {pattern} {k}x{k} {kernel} {h}x{w} frame {i}")


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", R.PATTERNS)
@pytest.mark.parametrize("n,h,w", [(3, 1080, 1920), (2, 75, 77), (3, 64, 128), (2, 3, 3)])
def test_pipeline_gray_edge_and_fused(ctx, oracle, pattern, n, h, w):
    fr = _noise(n, h, w, 3 + h)
    wt = rip.gauss_weights(5, 1.0)
    gray = ctx.process(fr, rip.OP_GRAY, FMT[pattern])
    gray_rgba = ctx.process(fr, rip.OP_GRAY, FMT[pattern], gray_out=rip.GRAY_OUT_RGBA)
    edge = ctx.process(fr, rip.OP_EDGE, FMT[pattern])
    fused = ctx.process(fr, rip.OP_FUSED, FMT[pattern], ksize=5, weights=wt)
    for i in range(n):
        rgb = R.decode(fr[i], pattern)
        g = oracle.gray(rgb, threads=0)
        _eq(gray[i], g, f"GRAY {pattern} {h}x{w} frame {i}")
        _eq(gray_rgba[i], _gray_rgba(g), f"GRAY rgba {pattern} {h}x{w} frame {i}")
        _eq(edge[i], oracle.sobel(g, threads=0), f"EDGE {pattern} {h}x{w} frame {i}")
        _eq(fused[i], oracle.fused(rgb, 5, weights=wt, threads=0), f"FUSED {pattern} {h}x{w} frame {i}")


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", R.PATTERNS)
def test_submit_collect_three_in_flight(ctx, oracle, pattern):
    fr = _noise(6, 270, 481, 44)
    wt = rip.gauss_weights(5, 1.5)
    want = [oracle.blur(R.decode(f, pattern, "rgba"), 5, weights=wt, threads=0) for f in fr]
    tickets, got = [], []
    for i in range(6):
        tickets.append(ctx.submit(fr[i], rip.OP_GAUSSIAN, FMT[pattern], ksize=5, weights=wt))
        if len(tickets) == 3:
            got.append(tickets.pop(0).collect())
    got += [t.collect() for t in tickets]
    for i in range(6):
        _eq(got[i], want[i], f"submit/collect {pattern} frame {i}")


@pytest.mark.gpu
def test_two_device_context(oracle):
    if rip.device_count() < 2:
        pytest.skip("needs two GPUs")
    wt = rip.gauss_weights(5, 1.0)
    c = rip.Context([0, 1])
    try:
        for pattern in R.PATTERNS:
            fr = _noise(5, 120, 161, 8)
            gray = c.process(fr, rip.OP_GRAY, FMT[pattern])
            blur = c.process(fr, rip.OP_GAUSSIAN, FMT[pattern], ksize=5, weights=wt)
            fused = c.process(fr, rip.OP_FUSED, FMT[pattern], ksize=5, weights=wt)
            for i in range(5):
                rgb = R.decode(fr[i], pattern)
                _eq(gray[i], oracle.gray(rgb), f"2-device GRAY {pattern} frame {i}")
                _eq(blur[i], oracle.blur(R.decode(fr[i], pattern, "rgba"), 5, weights=wt), f"2-device GAUSSIAN {pattern} frame {i}")
                _eq(fused[i], oracle.fused(rgb, 5, weights=wt), f"2-device FUSED {pattern} frame {i}")
    finally:
        c.close()


@pytest.mark.gpu
def test_rejections(ctx):
    wt = rip.gauss_weights(5, 1.0)
    # W or H below 3: the host pipeline, rip_convert and rip_gray, before any byte is read
    for pattern in R.PATTERNS:
        msg = f"BAYER_{pattern.upper()}8 frames need a width and height of at least 3"
        for h, w in ((2, 8), (8, 2), (1, 1), (2, 2)):
            raw = np.zeros(64, np.uint8)
            d_in, d_out = rip.DeviceBuffer(raw.nbytes), rip.DeviceBuffer(256)
            with pytest.raises(rip.RipError, match=msg):
                rip.convert_dev(d_in.ptr, d_out.ptr, w, h, 1, FMT[pattern], rip.FMT_RGBA8)
            with pytest.raises(rip.RipError, match=msg):
                rip.gray_dev(d_in.ptr, d_out.ptr, w, h, 1, FMT[pattern])
            for op in (rip.OP_GRAY, rip.OP_GAUSSIAN, rip.OP_EDGE, rip.OP_FUSED):
                d = ctx._desc(op, FMT[pattern], ksize=5, weights=wt)
                out = np.empty(h * w * 4, np.uint8)
                rc = rip.lib().rip_process_host(ctx.ptr, C.byref(d), raw.ctypes.data, out.ctypes.data, w, h, 1, None)
                assert rc == -1 and msg.encode() in rip.lib().rip_last_error_string()
    for pattern in R.PATTERNS:
        fr = _noise(1, 64, 64, 1)
        with pytest.raises(rip.RipError, match="rc=-4.*row-band"):
            ctx.process(fr, rip.OP_FUSED, FMT[pattern], ksize=5, weights=wt, banded=True)
        with pytest.raises(rip.RipError, match="rc=-4.*row-band"):
            ctx.process(fr, rip.OP_EDGE, FMT[pattern], banded=True)
        d_in, d_out = rip.DeviceBuffer(fr.nbytes).upload(fr), rip.DeviceBuffer(64 * 64 * 4)
        name = f"BAYER_{pattern.upper()}8"
        with pytest.raises(rip.RipError, match=f"rc=-4.*rip_sobel: RIP_FMT_{name} .*rip_gray"):
            rip.sobel_dev(d_in.ptr, d_out.ptr, 64, 64, 1, FMT[pattern])
        with pytest.raises(rip.RipError, match=f"rc=-4.*rip_fused: RIP_FMT_{name} .*rip_gray"):
            rip.fused_dev(d_in.ptr, d_out.ptr, 64, 64, 1, FMT[pattern], 5, wt)
        for out_fmt in (rip.FMT_GRAY8, rip.FMT_NV12, FMT[pattern]):
            with pytest.raises(rip.RipError, match="rc=-4"):
                rip.convert_dev(d_in.ptr, d_out.ptr, 64, 64, 1, FMT[pattern], out_fmt)


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", R.PATTERNS)
@pytest.mark.parametrize("n,h,w", [(2, 130, 248), (3, 75, 77), (3, 40, 1000), (2, 3, 8)])
def test_decode_stays_inside_its_output_buffer(oracle, pattern, n, h, w):
    """Every decode writes into the middle of a canary-filled buffer (256 KB on either side): the canaries must survive and the
    payload must equal the reference."""
    pad = 256 * 1024
    fr = _noise(n, h, w, 515)
    d_in = rip.DeviceBuffer(fr.nbytes).upload(fr)
    rgb = R.decode(fr, pattern)

    def run(name, out_bytes, launch, want):
        buf = rip.DeviceBuffer(out_bytes + 2 * pad)
        buf.upload(np.full(out_bytes + 2 * pad, 0xA5, np.uint8))
        launch(buf.ptr + pad)
        got = buf.download((out_bytes + 2 * pad,))
        assert (got[:pad] == 0xA5).all() and (got[pad + out_bytes:] == 0xA5).all(), f"{name} {n}x{h}x{w}: wrote outside its output"
        _eq(got[pad: pad + out_bytes].reshape(want.shape), want, f"{name} {n}x{h}x{w}")
        buf.free()

    for order in R.ORDERS:
        run(f"convert {pattern} {order}", n * h * w * len(order),
            lambda p: rip.convert_dev(d_in.ptr, p, w, h, n, FMT[pattern], OUT_FMT[order]), _in_order(rgb, order))
    g = _want_gray(oracle, pattern, fr)
    run(f"gray {pattern} u8", n * h * w, lambda p: rip.gray_dev(d_in.ptr, p, w, h, n, FMT[pattern], rip.GRAY_OUT_U8), g)
    run(f"gray {pattern} rgba", n * h * w * 4, lambda p: rip.gray_dev(d_in.ptr, p, w, h, n, FMT[pattern], rip.GRAY_OUT_RGBA),
        _gray_rgba(g))


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", R.PATTERNS)
def test_cpp_controller_drop_in(tmp_path, oracle, pattern):
    """PerformBatch / PerformFused / SubmitFrame + CollectFrame through the C++ Controller, and its rejection of short buffers
    and of frames narrower or shorter than 3, against bytes computed here through the oracle."""
    exe = _build_dropin(tmp_path)
    n, h, w = 3, 121, 163
    fr = _smooth(n, h, w, 12)
    fr.tofile(str(tmp_path / "in.raw"))
    res = subprocess.run([exe, str(tmp_path), str(FMT[pattern]), str(w), str(h), str(n)], capture_output=True, text=True)
    assert res.returncode == 0 and res.stdout.strip().endswith("OK"), res.stdout + res.stderr
    wt = oracle.gauss_weights(5, 1.5)
    rgb = R.decode(fr, pattern)
    gray = np.stack([oracle.gray(f) for f in rgb])
    want = {"batch_GRAYSCALE": gray,
            "batch_GAUSSIAN": np.stack([oracle.blur(R.decode(f, pattern, "rgba"), 5, weights=wt) for f in fr]),
            "batch_EDGE": np.stack([oracle.sobel(g) for g in gray]),
            "batch_FUSED": np.stack([oracle.fused(f, 5, weights=wt) for f in rgb]),
            "fused_frame0": oracle.fused(rgb[0], 5, weights=wt)}
    want["submit_GAUSSIAN"] = want["batch_GAUSSIAN"]
    for name, ref in want.items():
        got = np.fromfile(str(tmp_path / (name + ".raw")), np.uint8)
        _eq(got.reshape(ref.shape), ref, name)
