"""RIP_FMT_YUYV, RIP_FMT_UYVY and RIP_FMT_I420: camera and video frames decoded to colour exactly as OpenCV's cvtColor does,
then the reference's chain on that colour image (GRAYSCALE its gray, GAUSSIAN the blur of the RGBA image with alpha 255,
EDGE / FUSED their result on its gray) -- the same contract as RIP_FMT_NV12_COLOR, for the other common layouts.

CPU tests pin the numpy restatement of the decode (tests/yuv_ref.py) to cv2 on every (Y, U, V) triple of each layout and to
the recorded cv2 outputs in tests/golden/cv2_yuv.npz.  GPU tests compare every device path with that restatement followed by
the C oracle, bit for bit."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import nv12_ref
import rip_b200 as rip
import yuv_ref as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "opencl-development-real-time-image-processing_b200")
GOLDEN = os.path.join(ROOT, "tests", "golden", "cv2_yuv.npz")
FMT = {"yuyv": rip.FMT_YUYV, "uyvy": rip.FMT_UYVY, "i420": rip.FMT_I420}
OUT_FMT = {"rgb": rip.FMT_RGB8, "bgr": rip.FMT_BGR8, "rgba": rip.FMT_RGBA8, "bgra": rip.FMT_BGRA8}


def _eq(got, want, what=""):
    if not np.array_equal(got, want):
        d = np.abs(got.astype(int) - want.astype(int))
        idx = np.argwhere(d > 0)
        raise AssertionError(f"{what}: {len(idx)} of {d.size} bytes differ, max abs {d.max()}, first at {idx[0].tolist()}")


def _frame_shape(layout, h, w):
    return (h * 3 // 2, w) if layout == "i420" else (h, w, 2)


def _noise(layout, n, h, w, seed):
    return np.random.default_rng(seed).integers(0, 256, (n,) + _frame_shape(layout, h, w), dtype=np.uint8)


def _pack(layout, Y, U, V):
    """One frame from luma (H, W) and chroma planes: (H/2, W/2) each for I420, (H, W/2) for YUYV / UYVY."""
    if layout == "i420":
        h, w = Y.shape
        return np.concatenate([Y, np.concatenate([U.reshape(-1), V.reshape(-1)]).reshape(h // 2, w)], 0)
    return R.packed_from_planes(Y, U, V, layout)


def _chroma_shape(layout, h, w):
    return (h // 2, w // 2) if layout == "i420" else (h, w // 2)


def _smooth(layout, n, h, w, seed):
    """Camera-like frames: smooth luma with noise, slowly varying chroma, a flat letterbox bar (the blur's constant windows)."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    cy, cx = np.mgrid[0:_chroma_shape(layout, h, w)[0], 0:_chroma_shape(layout, h, w)[1]].astype(np.float32)
    out = []
    for _ in range(n):
        fx, fy, ph = rng.uniform(0.002, 0.03), rng.uniform(0.002, 0.03), rng.uniform(0, 6.28)
        Y = np.clip(120 + 90 * np.sin(fx * xx + fy * yy + ph) + rng.integers(-3, 4, (h, w)), 0, 255).astype(np.uint8)
        Y[: h // 8] = 16   # black bar
        U = np.clip(128 + 60 * np.sin(0.01 * cx + ph), 0, 255).astype(np.uint8)
        V = np.clip(128 + 60 * np.cos(0.013 * cy + ph), 0, 255).astype(np.uint8)
        out.append(_pack(layout, Y, U, V))
    return np.stack(out)


def _out_bytes(op, fmt, w, h, gray_out=rip.GRAY_OUT_U8):
    d = rip.OpDesc()
    d.op, d.in_format, d.gray_out = op, fmt, gray_out
    b = C.c_size_t(0)
    rip.check(rip.lib().rip_out_bytes_per_frame(C.byref(d), w, h, C.byref(b)))
    return b.value


# ---- CPU: the decode restatement, the host-side sizes and shapes -----------------------------------------------------
@pytest.mark.parametrize("layout", R.LAYOUTS)
def test_reference_decode_equals_cv2_on_every_triple(layout):
    cv2 = pytest.importorskip("cv2")
    frame = R.exhaustive_frame(layout)
    Y, U, V = R.unpack(frame, layout)
    assert len(np.unique((Y << 16 | U << 8 | V).reshape(-1))) == 1 << 24
    for order in R.ORDERS:
        _eq(R.decode(frame, layout, order), R.cv2_decode(frame, layout, order), f"{layout} {order} vs cv2 {cv2.__version__}")


def test_reference_decode_equals_recorded_cv2():
    g = np.load(GOLDEN)
    cases = [k[:-3] for k in g.files if k.endswith(".in")]
    for layout in R.LAYOUTS:
        assert len([c for c in cases if c.startswith(layout + ".")]) >= 6
    for case in cases:
        layout = case.split(".")[0]
        for order in ("rgb", "bgra"):
            _eq(R.decode(g[case + ".in"], layout, order), g[case + "." + order], f"{case} {order}")


def test_reference_agrees_with_nv12_restatement():
    nv = np.random.default_rng(9).integers(0, 256, (30, 22), dtype=np.uint8)   # 20 x 22: W/2 odd
    for order in R.ORDERS:
        _eq(R.decode(nv, "nv12", order), nv12_ref.decode(nv, order), f"nv12 {order}")
        _eq(R.decode(R.i420_from_nv12(nv), "i420", order), nv12_ref.decode(nv, order), f"i420 of the same image {order}")


def test_output_sizes_of_the_new_formats():
    w, h = 640, 481
    for fmt in FMT.values():
        assert _out_bytes(rip.OP_GAUSSIAN, fmt, w, h) == w * h * 4
        assert _out_bytes(rip.OP_GRAY, fmt, w, h) == w * h
        assert _out_bytes(rip.OP_GRAY, fmt, w, h, rip.GRAY_OUT_RGBA) == w * h * 4
        assert _out_bytes(rip.OP_EDGE, fmt, w, h) == w * h
        assert _out_bytes(rip.OP_FUSED, fmt, w, h) == w * h


def test_python_shapes_of_the_new_formats():
    """Context.process / submit take YUYV and UYVY as (N, H, W, 2) or (H, W, 2) and I420 as (N, H*3/2, W) or (H*3/2, W)."""
    c = object.__new__(rip.Context)   # the shape handling needs no device
    for layout in ("yuyv", "uyvy"):
        a, _, n, h, w, shape, out, squeeze = c._shapes(np.zeros((3, 5, 6, 2), np.uint8), rip.OP_GAUSSIAN, FMT[layout],
                                                        rip.GRAY_OUT_U8, 5, rip.gauss_weights(5, 1.0), None)
        assert (n, h, w, shape, out.shape, squeeze) == (3, 5, 6, (3, 5, 6, 4), (3, 5, 6, 4), False)
        a, _, n, h, w, shape, out, squeeze = c._shapes(np.zeros((5, 6, 2), np.uint8), rip.OP_GRAY, FMT[layout],
                                                        rip.GRAY_OUT_U8, 0, None, None)
        assert (a.shape, n, h, w, shape, squeeze) == ((1, 5, 6, 2), 1, 5, 6, (1, 5, 6), True)
        with pytest.raises(AssertionError, match="needs 2 channels"):
            c._shapes(np.zeros((1, 5, 6, 3), np.uint8), rip.OP_GRAY, FMT[layout], rip.GRAY_OUT_U8, 0, None, None)
    a, _, n, h, w, shape, out, squeeze = c._shapes(np.zeros((2, 9, 10), np.uint8), rip.OP_GRAY, rip.FMT_I420,
                                                    rip.GRAY_OUT_RGBA, 0, None, None)
    assert (n, h, w, shape, squeeze) == (2, 6, 10, (2, 6, 10, 4), False)
    a, _, n, h, w, shape, out, squeeze = c._shapes(np.zeros((9, 10), np.uint8), rip.OP_EDGE, rip.FMT_I420,
                                                    rip.GRAY_OUT_U8, 0, None, None)
    assert (a.shape, n, h, w, shape, squeeze) == ((1, 9, 10), 1, 6, 10, (1, 6, 10), True)


@pytest.mark.skipif(rip.device_count() > 0, reason="only meaningful on a box without a GPU")
def test_convert_fails_loudly_without_gpu():
    for fmt in FMT.values():
        with pytest.raises(rip.RipError, match="no CUDA device|no CPU fallback"):
            rip.convert_dev(16, 32, 4, 4, 1, fmt, rip.FMT_RGBA8)
        with pytest.raises(rip.RipError, match="no CUDA device|no CPU fallback"):
            rip.gray_dev(16, 32, 4, 4, 1, fmt)


def _build_dropin(tmp_path):
    exe = str(tmp_path / "yuv_color_dropin")
    cmd = ["/usr/bin/g++", "-O2", "-std=c++17", "-ffp-contract=off", "-I", os.path.join(PKG, "host"), "-I", os.path.join(ROOT, "include"),
           "-I", "/usr/local/cuda/include", os.path.join(ROOT, "tests", "cpp", "yuv_color_dropin.cpp"), "-o", exe, "-L", PKG, "-lrip_host",
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


def _convert(layout, fr, w, h, order, in_off=0, out_off=0):
    n = fr.shape[0]
    bpp = len(order)
    d_in = rip.DeviceBuffer(fr.nbytes + 16).upload(fr, offset=in_off)
    d_out = rip.DeviceBuffer(n * h * w * bpp + 16)
    rip.convert_dev(d_in.ptr + in_off, d_out.ptr + out_off, w, h, n, FMT[layout], OUT_FMT[order])
    return d_out.download((n, h, w, bpp), offset=out_off)


def _gray_dev(layout, fr, w, h, out_mode, in_off=0, out_off=0):
    n = fr.shape[0]
    bpp = 4 if out_mode == rip.GRAY_OUT_RGBA else 1
    d_in = rip.DeviceBuffer(fr.nbytes + 16).upload(fr, offset=in_off)
    d_out = rip.DeviceBuffer(n * h * w * bpp + 16)
    rip.gray_dev(d_in.ptr + in_off, d_out.ptr + out_off, w, h, n, FMT[layout], out_mode)
    return d_out.download((n, h, w, bpp) if bpp == 4 else (n, h, w), offset=out_off)


def _want_gray(oracle, layout, fr):
    return np.stack([oracle.gray(R.decode(f, layout), threads=0) for f in fr])


def _gray_rgba(g):
    return np.stack([g, g, g, np.full_like(g, 255)], -1)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", R.LAYOUTS)
def test_convert_every_triple(ctx, layout):
    fr = R.exhaustive_frame(layout)[None]
    for order in R.ORDERS:
        _eq(_convert(layout, fr, 4096, 4096, order)[0], R.decode(fr[0], layout, order), f"rip_convert {layout} {order}, all 2^24 triples")


RAGGED = {   # (n, h, w): widths that are not multiples of 8 take the byte-granular kernels; YUYV / UYVY also odd heights
    "i420": [(1, 2, 2), (3, 2, 6), (2, 6, 10), (2, 74, 76), (1, 682, 1022), (7, 2, 8), (5, 6, 24), (2, 120, 1920)],
    "yuyv": [(1, 1, 2), (3, 3, 6), (2, 5, 10), (2, 75, 76), (1, 683, 1022), (7, 1, 8), (5, 3, 24), (2, 121, 1920)],
}
RAGGED["uyvy"] = RAGGED["yuyv"]


@pytest.mark.gpu
@pytest.mark.parametrize("layout,n,h,w", [(lay, *s) for lay in R.LAYOUTS for s in RAGGED[lay]])
def test_convert_ragged_shapes_and_batches(ctx, layout, n, h, w):
    fr = _noise(layout, n, h, w, 100 + h + w)
    for order in R.ORDERS:
        _eq(_convert(layout, fr, w, h, order), R.decode(fr, layout, order), f"rip_convert {layout} {order} {n}x{h}x{w}")


@pytest.mark.gpu
@pytest.mark.parametrize("layout", R.LAYOUTS)
@pytest.mark.parametrize("in_off,out_off", [(1, 0), (0, 1), (4, 12), (8, 8), (12, 4)])
def test_convert_and_gray_unaligned_buffers(ctx, oracle, layout, in_off, out_off):
    """Offsets 4, 8 and 12 keep 4-byte alignment but break the 8- or 16-byte alignment the wide kernels need."""
    n, h, w = 3, 6, 24
    fr = _noise(layout, n, h, w, 7)
    for order in R.ORDERS:
        _eq(_convert(layout, fr, w, h, order, in_off, out_off), R.decode(fr, layout, order),
            f"rip_convert {layout} {order} offsets {in_off}/{out_off}")
    g = _want_gray(oracle, layout, fr)
    _eq(_gray_dev(layout, fr, w, h, rip.GRAY_OUT_U8, in_off, out_off), g, f"rip_gray {layout} u8 unaligned")
    _eq(_gray_dev(layout, fr, w, h, rip.GRAY_OUT_RGBA, in_off, out_off), _gray_rgba(g), f"rip_gray {layout} rgba unaligned")


@pytest.mark.gpu
@pytest.mark.parametrize("layout", R.LAYOUTS)
@pytest.mark.parametrize("n,h,w", [(1, 4096, 4096), (3, 74, 76), (2, 1080, 1920)])
def test_gray_dev_both_out_modes(ctx, oracle, layout, n, h, w):
    fr = R.exhaustive_frame(layout)[None] if h == 4096 else _noise(layout, n, h, w, 5 + w)
    g = _want_gray(oracle, layout, fr)
    _eq(_gray_dev(layout, fr, w, h, rip.GRAY_OUT_U8), g, f"rip_gray {layout} u8 {n}x{h}x{w}")
    _eq(_gray_dev(layout, fr, w, h, rip.GRAY_OUT_RGBA), _gray_rgba(g), f"rip_gray {layout} rgba {n}x{h}x{w}")


def _content_frames(layout, h, w):
    """Neutral chroma (U = V = 128: r = g = b on every pixel, the exact multiples of 1000 and the (r, g) table) over flat
    grey, black, white and a luma ramp, and the four saturating chroma corners over the ramp."""
    ch = _chroma_shape(layout, h, w)
    ramp = (np.arange(h * w) % 256).astype(np.uint8).reshape(h, w)
    frames = []
    for Y, u, v in [(np.full((h, w), yv, np.uint8), 128, 128) for yv in (128, 16, 0, 235, 255)] + \
                   [(ramp, 128, 128), (ramp, 0, 0), (ramp, 0, 255), (ramp, 255, 0), (ramp, 255, 255)]:
        frames.append(_pack(layout, Y, np.full(ch, u, np.uint8), np.full(ch, v, np.uint8)))
    return np.stack(frames)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", R.LAYOUTS)
def test_content_neutral_and_saturating_chroma(ctx, oracle, layout):
    h, w = 64, 96
    fr = _content_frames(layout, h, w)
    for order in R.ORDERS:
        _eq(_convert(layout, fr, w, h, order), R.decode(fr, layout, order), f"content rip_convert {layout} {order}")
    g = _want_gray(oracle, layout, fr)
    _eq(_gray_dev(layout, fr, w, h, rip.GRAY_OUT_U8), g, f"content rip_gray {layout}")
    _eq(ctx.process(fr, rip.OP_GRAY, FMT[layout]), g, f"content GRAY {layout}")
    _eq(ctx.process(fr, rip.OP_GRAY, FMT[layout], gray_out=rip.GRAY_OUT_RGBA), _gray_rgba(g), f"content GRAY rgba {layout}")


@pytest.mark.gpu
@pytest.mark.parametrize("layout", R.LAYOUTS)
@pytest.mark.parametrize("k,sigma", [(5, 1.5), (9, 2.5), (17, 6.0)])
def test_pipeline_gaussian(ctx, oracle, layout, k, sigma):
    """Decode to RGBA, then the blur kernels as they are chosen by size: 3 x 1080p (streaming) and 2 x 120x160 (tiled)."""
    wt = rip.gauss_weights(k, sigma)
    h_small = 121 if layout != "i420" else 120
    for fr, h, w in ((_smooth(layout, 3, 1080, 1920, k), 1080, 1920), (_noise(layout, 2, h_small, 160, k), h_small, 160)):
        n = fr.shape[0]
        got = ctx.process(fr, rip.OP_GAUSSIAN, FMT[layout], ksize=k, weights=wt)
        assert got.shape == (n, h, w, 4)
        for i in range(n):
            want = oracle.blur(R.decode(fr[i], layout, "rgba"), k, weights=wt, threads=0)
            _eq(got[i], want, f"GAUSSIAN {layout} {k}x{k} {h}x{w} frame {i}")


@pytest.mark.gpu
@pytest.mark.parametrize("layout", R.LAYOUTS)
@pytest.mark.parametrize("n,h,w", [(3, 1080, 1920), (2, 74, 76), (3, 64, 128)])
def test_pipeline_gray_edge_and_fused(ctx, oracle, layout, n, h, w):
    fr = _noise(layout, n, h, w, 3 + h)
    wt = rip.gauss_weights(5, 1.0)
    gray = ctx.process(fr, rip.OP_GRAY, FMT[layout])
    edge = ctx.process(fr, rip.OP_EDGE, FMT[layout])
    fused = ctx.process(fr, rip.OP_FUSED, FMT[layout], ksize=5, weights=wt)
    for i in range(n):
        rgb = R.decode(fr[i], layout)
        g = oracle.gray(rgb, threads=0)
        _eq(gray[i], g, f"GRAY {layout} {h}x{w} frame {i}")
        _eq(edge[i], oracle.sobel(g, threads=0), f"EDGE {layout} {h}x{w} frame {i}")
        _eq(fused[i], oracle.fused(rgb, 5, weights=wt, threads=0), f"FUSED {layout} {h}x{w} frame {i}")


@pytest.mark.gpu
@pytest.mark.parametrize("layout", R.LAYOUTS)
def test_submit_collect_three_in_flight(ctx, oracle, layout):
    h, w = 270, 480
    fr = _noise(layout, 6, h, w, 44)
    wt = rip.gauss_weights(5, 1.5)
    want = [oracle.blur(R.decode(f, layout, "rgba"), 5, weights=wt, threads=0) for f in fr]
    tickets, got = [], []
    for i in range(6):
        tickets.append(ctx.submit(fr[i], rip.OP_GAUSSIAN, FMT[layout], ksize=5, weights=wt))
        if len(tickets) == 3:
            got.append(tickets.pop(0).collect())
    got += [t.collect() for t in tickets]
    for i in range(6):
        _eq(got[i], want[i], f"submit/collect {layout} frame {i}")


@pytest.mark.gpu
def test_two_device_context(oracle):
    if rip.device_count() < 2:
        pytest.skip("needs two GPUs")
    wt = rip.gauss_weights(5, 1.0)
    c = rip.Context([0, 1])
    try:
        for layout in R.LAYOUTS:
            fr = _noise(layout, 5, 120, 160, 8)
            gray = c.process(fr, rip.OP_GRAY, FMT[layout])
            blur = c.process(fr, rip.OP_GAUSSIAN, FMT[layout], ksize=5, weights=wt)
            fused = c.process(fr, rip.OP_FUSED, FMT[layout], ksize=5, weights=wt)
            for i in range(5):
                rgb = R.decode(fr[i], layout)
                _eq(gray[i], oracle.gray(rgb), f"2-device GRAY {layout} frame {i}")
                _eq(blur[i], oracle.blur(R.decode(fr[i], layout, "rgba"), 5, weights=wt), f"2-device GAUSSIAN {layout} frame {i}")
                _eq(fused[i], oracle.fused(rgb, 5, weights=wt), f"2-device FUSED {layout} frame {i}")
    finally:
        c.close()


@pytest.mark.gpu
def test_rejections(ctx):
    wt = rip.gauss_weights(5, 1.0)
    # odd width (all three) or odd height (I420): the host pipeline, rip_convert and rip_gray, before any byte is read
    for layout, h, w, msg in (("yuyv", 6, 9, "YUYV frames need an even width"), ("uyvy", 5, 9, "UYVY frames need an even width"),
                              ("i420", 6, 9, "I420 frames need an even width and height"),
                              ("i420", 5, 8, "I420 frames need an even width and height")):
        raw = np.zeros(h * w * 2 + 64, np.uint8)
        d_in, d_out = rip.DeviceBuffer(raw.nbytes), rip.DeviceBuffer(h * w * 4 + 64)
        with pytest.raises(rip.RipError, match=msg):
            rip.convert_dev(d_in.ptr, d_out.ptr, w, h, 1, FMT[layout], rip.FMT_RGBA8)
        with pytest.raises(rip.RipError, match=msg):
            rip.gray_dev(d_in.ptr, d_out.ptr, w, h, 1, FMT[layout])
        for op in (rip.OP_GRAY, rip.OP_GAUSSIAN, rip.OP_EDGE, rip.OP_FUSED):
            d = ctx._desc(op, FMT[layout], ksize=5, weights=wt)
            out = np.empty(h * w * 4, np.uint8)
            rc = rip.lib().rip_process_host(ctx.ptr, C.byref(d), raw.ctypes.data, out.ctypes.data, w, h, 1, None)
            assert rc == -1 and msg.encode() in rip.lib().rip_last_error_string()
    for layout in R.LAYOUTS:
        fr = _noise(layout, 1, 64, 64, 1)
        with pytest.raises(rip.RipError, match="rc=-4.*row-band"):
            ctx.process(fr, rip.OP_FUSED, FMT[layout], ksize=5, weights=wt, banded=True)
        d_in, d_out = rip.DeviceBuffer(fr.nbytes).upload(fr), rip.DeviceBuffer(64 * 64 * 4)
        name = layout.upper()
        with pytest.raises(rip.RipError, match=f"rc=-4.*rip_sobel: RIP_FMT_{name} .*rip_gray"):
            rip.sobel_dev(d_in.ptr, d_out.ptr, 64, 64, 1, FMT[layout])
        with pytest.raises(rip.RipError, match=f"rc=-4.*rip_fused: RIP_FMT_{name} .*rip_gray"):
            rip.fused_dev(d_in.ptr, d_out.ptr, 64, 64, 1, FMT[layout], 5, wt)
        for out_fmt in (rip.FMT_GRAY8, rip.FMT_NV12, FMT[layout]):
            with pytest.raises(rip.RipError, match="rc=-4"):
                rip.convert_dev(d_in.ptr, d_out.ptr, 64, 64, 1, FMT[layout], out_fmt)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", R.LAYOUTS)
@pytest.mark.parametrize("n,h,w", [(2, 130, 248), (1, 74, 76), (3, 40, 1000)])
def test_decode_stays_inside_its_output_buffer(oracle, layout, n, h, w):
    """Every decode writes into the middle of a canary-filled buffer (256 KB on either side): the canaries must survive and the
    payload must equal the reference."""
    pad = 256 * 1024
    fr = _noise(layout, n, h, w, 515)
    d_in = rip.DeviceBuffer(fr.nbytes).upload(fr)

    def run(name, out_bytes, launch, want):
        buf = rip.DeviceBuffer(out_bytes + 2 * pad)
        buf.upload(np.full(out_bytes + 2 * pad, 0xA5, np.uint8))
        launch(buf.ptr + pad)
        got = buf.download((out_bytes + 2 * pad,))
        assert (got[:pad] == 0xA5).all() and (got[pad + out_bytes:] == 0xA5).all(), f"{name} {n}x{h}x{w}: wrote outside its output"
        _eq(got[pad: pad + out_bytes].reshape(want.shape), want, f"{name} {n}x{h}x{w}")
        buf.free()

    for order in R.ORDERS:
        run(f"convert {layout} {order}", n * h * w * len(order),
            lambda p: rip.convert_dev(d_in.ptr, p, w, h, n, FMT[layout], OUT_FMT[order]), R.decode(fr, layout, order))
    g = _want_gray(oracle, layout, fr)
    run(f"gray {layout} u8", n * h * w, lambda p: rip.gray_dev(d_in.ptr, p, w, h, n, FMT[layout], rip.GRAY_OUT_U8), g)
    run(f"gray {layout} rgba", n * h * w * 4, lambda p: rip.gray_dev(d_in.ptr, p, w, h, n, FMT[layout], rip.GRAY_OUT_RGBA),
        _gray_rgba(g))


@pytest.mark.gpu
@pytest.mark.parametrize("layout", R.LAYOUTS)
def test_cpp_controller_drop_in(tmp_path, oracle, layout):
    """PerformBatch / PerformFused / SubmitFrame + CollectFrame through the C++ Controller, and its rejection of short buffers,
    odd widths and odd I420 heights, against bytes computed here through the oracle."""
    exe = _build_dropin(tmp_path)
    n, h, w = 3, 120, 164
    fr = _smooth(layout, n, h, w, 12)
    fr.tofile(str(tmp_path / "in.raw"))
    res = subprocess.run([exe, str(tmp_path), str(FMT[layout]), str(w), str(h), str(n)], capture_output=True, text=True)
    assert res.returncode == 0 and res.stdout.strip().endswith("OK"), res.stdout + res.stderr
    wt = oracle.gauss_weights(5, 1.5)
    rgb = R.decode(fr, layout)
    gray = np.stack([oracle.gray(f) for f in rgb])
    want = {"batch_GRAYSCALE": gray,
            "batch_GAUSSIAN": np.stack([oracle.blur(R.decode(f, layout, "rgba"), 5, weights=wt) for f in fr]),
            "batch_EDGE": np.stack([oracle.sobel(g) for g in gray]),
            "batch_FUSED": np.stack([oracle.fused(f, 5, weights=wt) for f in rgb]),
            "fused_frame0": oracle.fused(rgb[0], 5, weights=wt)}
    want["submit_GAUSSIAN"] = want["batch_GAUSSIAN"]
    for name, ref in want.items():
        got = np.fromfile(str(tmp_path / (name + ".raw")), np.uint8)
        _eq(got.reshape(ref.shape), ref, name)
