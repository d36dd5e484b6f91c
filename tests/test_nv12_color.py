"""RIP_FMT_NV12_COLOR: NV12 camera frames decoded to colour exactly as OpenCV's cvtColor(COLOR_YUV2RGB_NV12) does, then the
reference's chain on that colour image (GRAYSCALE its gray, GAUSSIAN the blur of the RGBA image with alpha 255, EDGE / FUSED
their result on its gray).

CPU tests pin the numpy restatement of the decode (tests/nv12_ref.py) to cv2 on every (Y, U, V) triple and to the recorded cv2
outputs in tests/golden/cv2_nv12.npz.  GPU tests compare every device path with that restatement followed by the C oracle, bit
for bit."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import nv12_ref as R
import rip_b200 as rip

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "opencl-development-real-time-image-processing_b200")
GOLDEN = os.path.join(ROOT, "tests", "golden", "cv2_nv12.npz")
OUT_FMT = {"rgb": rip.FMT_RGB8, "bgr": rip.FMT_BGR8, "rgba": rip.FMT_RGBA8, "bgra": rip.FMT_BGRA8}


def _eq(got, want, what=""):
    if not np.array_equal(got, want):
        d = np.abs(got.astype(int) - want.astype(int))
        idx = np.argwhere(d > 0)
        raise AssertionError(f"{what}: {len(idx)} of {d.size} bytes differ, max abs {d.max()}, first at {idx[0].tolist()}")


def _noise(n, h, w, seed):
    return np.random.default_rng(seed).integers(0, 256, (n, h * 3 // 2, w), dtype=np.uint8)


def _out_bytes(op, fmt, w, h, gray_out=rip.GRAY_OUT_U8):
    d = rip.OpDesc()
    d.op, d.in_format, d.gray_out = op, fmt, gray_out
    b = C.c_size_t(0)
    rip.check(rip.lib().rip_out_bytes_per_frame(C.byref(d), w, h, C.byref(b)))
    return b.value


# ---- CPU: the decode restatement and the host-side sizes -------------------------------------------------------------
def test_reference_decode_equals_cv2_on_every_triple():
    cv2 = pytest.importorskip("cv2")
    frame = R.exhaustive_frame()
    for order in R.ORDERS:
        _eq(R.decode(frame, order), R.cv2_decode(frame, order), f"decode {order} vs cv2 {cv2.__version__}")


def test_reference_decode_equals_recorded_cv2():
    g = np.load(GOLDEN)
    cases = [k[:-5] for k in g.files if k.endswith(".nv12")]
    assert len(cases) >= 8
    for case in cases:
        for order in ("rgb", "bgra"):
            _eq(R.decode(g[case + ".nv12"], order), g[case + "." + order], f"{case} {order}")


def test_output_sizes_of_the_new_format():
    w, h = 640, 480
    assert _out_bytes(rip.OP_GAUSSIAN, rip.FMT_NV12_COLOR, w, h) == w * h * 4
    assert _out_bytes(rip.OP_GRAY, rip.FMT_NV12_COLOR, w, h) == w * h
    assert _out_bytes(rip.OP_GRAY, rip.FMT_NV12_COLOR, w, h, rip.GRAY_OUT_RGBA) == w * h * 4
    assert _out_bytes(rip.OP_EDGE, rip.FMT_NV12_COLOR, w, h) == w * h
    assert _out_bytes(rip.OP_FUSED, rip.FMT_NV12_COLOR, w, h) == w * h


@pytest.mark.skipif(rip.device_count() > 0, reason="only meaningful on a box without a GPU")
def test_convert_fails_loudly_without_gpu():
    with pytest.raises(rip.RipError, match="no CUDA device|no CPU fallback"):
        rip.convert_dev(16, 32, 4, 4, 1, rip.FMT_NV12_COLOR, rip.FMT_RGBA8)
    with pytest.raises(rip.RipError, match="no CUDA device|no CPU fallback"):
        rip.gray_dev(16, 32, 4, 4, 1, rip.FMT_NV12_COLOR)


def _build_dropin(tmp_path):
    exe = str(tmp_path / "nv12_color_dropin")
    cmd = ["/usr/bin/g++", "-O2", "-std=c++17", "-ffp-contract=off", "-I", os.path.join(PKG, "host"), "-I", os.path.join(ROOT, "include"),
           "-I", "/usr/local/cuda/include", os.path.join(ROOT, "tests", "cpp", "nv12_color_dropin.cpp"), "-o", exe, "-L", PKG, "-lrip_host",
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


def _convert(nv, w, h, order, in_off=0, out_off=0):
    n = nv.shape[0]
    bpp = len(order)
    d_in = rip.DeviceBuffer(nv.nbytes + 16).upload(nv, offset=in_off)
    d_out = rip.DeviceBuffer(n * h * w * bpp + 16)
    rip.convert_dev(d_in.ptr + in_off, d_out.ptr + out_off, w, h, n, rip.FMT_NV12_COLOR, OUT_FMT[order])
    return d_out.download((n, h, w, bpp), offset=out_off)


def _gray_dev(nv, w, h, out_mode, in_off=0, out_off=0):
    n = nv.shape[0]
    bpp = 4 if out_mode == rip.GRAY_OUT_RGBA else 1
    d_in = rip.DeviceBuffer(nv.nbytes + 16).upload(nv, offset=in_off)
    d_out = rip.DeviceBuffer(n * h * w * bpp + 16)
    rip.gray_dev(d_in.ptr + in_off, d_out.ptr + out_off, w, h, n, rip.FMT_NV12_COLOR, out_mode)
    return d_out.download((n, h, w, bpp) if bpp == 4 else (n, h, w), offset=out_off)


def _want_gray(oracle, nv):
    return np.stack([oracle.gray(R.decode(f), threads=0) for f in nv])


def _gray_rgba(g):
    return np.stack([g, g, g, np.full_like(g, 255)], -1)


@pytest.mark.gpu
def test_convert_every_triple(ctx):
    nv = R.exhaustive_frame()[None]
    for order in R.ORDERS:
        _eq(_convert(nv, 4096, 4096, order)[0], R.decode(nv[0], order), f"rip_convert {order}, all 2^24 triples")


@pytest.mark.gpu
@pytest.mark.parametrize("n,h,w", [(1, 2, 2), (3, 2, 6), (2, 6, 10), (2, 74, 76), (1, 682, 1022), (7, 2, 8), (5, 6, 24), (3, 16, 40),
                                   (2, 120, 1920)])
def test_convert_ragged_shapes_and_batches(ctx, n, h, w):
    """Widths that are not multiples of 8 take the byte-granular kernel; (7, 2, 8) and (5, 6, 24) are batches whose frame
    stride (24 and 216 bytes) is not a multiple of 16."""
    nv = _noise(n, h, w, 100 + h + w)
    for order in R.ORDERS:
        _eq(_convert(nv, w, h, order), R.decode(nv, order), f"rip_convert {order} {n}x{h}x{w}")


@pytest.mark.gpu
@pytest.mark.parametrize("in_off,out_off", [(1, 0), (0, 1), (8, 8), (4, 12)])
def test_convert_and_gray_unaligned_buffers(ctx, oracle, in_off, out_off):
    n, h, w = 3, 6, 24
    nv = _noise(n, h, w, 7)
    for order in R.ORDERS:
        _eq(_convert(nv, w, h, order, in_off, out_off), R.decode(nv, order), f"rip_convert {order} offsets {in_off}/{out_off}")
    g = _want_gray(oracle, nv)
    _eq(_gray_dev(nv, w, h, rip.GRAY_OUT_U8, in_off, out_off), g, "rip_gray u8 unaligned")
    _eq(_gray_dev(nv, w, h, rip.GRAY_OUT_RGBA, in_off, out_off), _gray_rgba(g), "rip_gray rgba unaligned")


@pytest.mark.gpu
@pytest.mark.parametrize("n,h,w", [(1, 4096, 4096), (3, 74, 76), (2, 1080, 1920)])
def test_gray_dev_both_out_modes(ctx, oracle, n, h, w):
    nv = R.exhaustive_frame()[None] if h == 4096 else _noise(n, h, w, 5 + w)
    g = _want_gray(oracle, nv)
    _eq(_gray_dev(nv, w, h, rip.GRAY_OUT_U8), g, f"rip_gray NV12_COLOR u8 {n}x{h}x{w}")
    _eq(_gray_dev(nv, w, h, rip.GRAY_OUT_RGBA), _gray_rgba(g), f"rip_gray NV12_COLOR rgba {n}x{h}x{w}")


def _content_frames(h, w):
    """Flat grey (U = V = 128: r = g = b on every pixel, the exact multiples of 1000), black, the four saturating chroma corners
    over a luma ramp, and white."""
    frames = []
    for yv, u, v in ((128, 128, 128), (16, 128, 128), (0, 128, 128), (235, 128, 128), (255, 128, 128)):
        f = np.empty((h * 3 // 2, w), np.uint8)
        f[:h] = yv
        f[h:, 0::2], f[h:, 1::2] = u, v
        frames.append(f)
    ramp = (np.arange(h * w) % 256).astype(np.uint8).reshape(h, w)
    for u, v in ((0, 0), (0, 255), (255, 0), (255, 255)):
        f = np.empty((h * 3 // 2, w), np.uint8)
        f[:h] = ramp
        f[h:, 0::2], f[h:, 1::2] = u, v
        frames.append(f)
    return np.stack(frames)


@pytest.mark.gpu
def test_content_flat_black_and_saturating_chroma(ctx, oracle):
    h, w = 64, 96
    nv = _content_frames(h, w)
    n = nv.shape[0]
    for order in R.ORDERS:
        _eq(_convert(nv, w, h, order), R.decode(nv, order), f"content rip_convert {order}")
    g = _want_gray(oracle, nv)
    _eq(ctx.process(nv, rip.OP_GRAY, rip.FMT_NV12_COLOR), g, "content GRAY")
    wt = rip.gauss_weights(5, 1.5)
    got = ctx.process(nv, rip.OP_GAUSSIAN, rip.FMT_NV12_COLOR, ksize=5, weights=wt)
    for i in range(n):
        _eq(got[i], oracle.blur(R.to_rgba(R.decode(nv[i])), 5, weights=wt, threads=0), f"content GAUSSIAN frame {i}")
        assert (got[i, ..., 3] == oracle.blur(np.full((4, 4), 255, np.uint8), 5, weights=wt)[0, 0]).all()
    got = ctx.process(nv, rip.OP_FUSED, rip.FMT_NV12_COLOR, ksize=5, weights=wt)
    for i in range(n):
        _eq(got[i], oracle.fused(R.decode(nv[i]), 5, weights=wt, threads=0), f"content FUSED frame {i}")


@pytest.mark.gpu
@pytest.mark.parametrize("n,h,w", [(3, 1080, 1920), (2, 74, 76), (1, 682, 1022)])
def test_pipeline_gray_both_out_modes(ctx, oracle, n, h, w):
    nv = _noise(n, h, w, 11 + w)
    g = _want_gray(oracle, nv)
    _eq(ctx.process(nv, rip.OP_GRAY, rip.FMT_NV12_COLOR), g, f"GRAY u8 {n}x{h}x{w}")
    _eq(ctx.process(nv, rip.OP_GRAY, rip.FMT_NV12_COLOR, gray_out=rip.GRAY_OUT_RGBA), _gray_rgba(g), f"GRAY rgba {n}x{h}x{w}")


def _smooth_nv12(n, h, w, seed):
    """Camera-like frames: smooth luma with noise, slowly varying chroma, a flat letterbox bar (the blur's constant windows)."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    out = np.empty((n, h * 3 // 2, w), np.uint8)
    for i in range(n):
        fx, fy, ph = rng.uniform(0.002, 0.03), rng.uniform(0.002, 0.03), rng.uniform(0, 6.28)
        luma = 120 + 90 * np.sin(fx * xx + fy * yy + ph) + rng.integers(-3, 4, (h, w))
        out[i, :h] = np.clip(luma, 0, 255).astype(np.uint8)
        out[i, : h // 8] = 16   # black bar
        cy, cx = np.mgrid[0: h // 2, 0: w // 2].astype(np.float32)
        out[i, h:, 0::2] = np.clip(128 + 60 * np.sin(0.01 * cx + ph), 0, 255).astype(np.uint8)
        out[i, h:, 1::2] = np.clip(128 + 60 * np.cos(0.013 * cy + ph), 0, 255).astype(np.uint8)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("k,sigma", [(5, 1.0), (5, 1.5), (9, 2.5), (17, 6.0)])
def test_pipeline_gaussian(ctx, oracle, k, sigma):
    """Decode to RGBA, then the blur kernels as they are chosen by size: 3 x 1080p (streaming), 2 x 120x160 (tiled), and for
    17x17 a 4K frame as well."""
    w = rip.gauss_weights(k, sigma)
    cases = [_smooth_nv12(3, 1080, 1920, k), _noise(2, 120, 160, k)]
    if k == 17:
        cases.append(_smooth_nv12(1, 2160, 3840, 99))
    for nv in cases:
        n, h3, wd = nv.shape
        h = h3 * 2 // 3
        got = ctx.process(nv, rip.OP_GAUSSIAN, rip.FMT_NV12_COLOR, ksize=k, weights=w)
        assert got.shape == (n, h, wd, 4)
        for i in range(n):
            _eq(got[i], oracle.blur(R.to_rgba(R.decode(nv[i])), k, weights=w, threads=0), f"GAUSSIAN {k}x{k} {h}x{wd} frame {i}")


@pytest.mark.gpu
@pytest.mark.parametrize("n,h,w", [(3, 1080, 1920), (2, 74, 76), (3, 64, 128)])
def test_pipeline_edge_and_fused_differ_from_luma(ctx, oracle, n, h, w):
    nv = _noise(n, h, w, 3 + h)
    wt = rip.gauss_weights(5, 1.0)
    edge = ctx.process(nv, rip.OP_EDGE, rip.FMT_NV12_COLOR)
    fused = ctx.process(nv, rip.OP_FUSED, rip.FMT_NV12_COLOR, ksize=5, weights=wt)
    for i in range(n):
        rgb = R.decode(nv[i])
        _eq(edge[i], oracle.sobel(oracle.gray(rgb, threads=0), threads=0), f"EDGE {h}x{w} frame {i}")
        _eq(fused[i], oracle.fused(rgb, 5, weights=wt, threads=0), f"FUSED {h}x{w} frame {i}")
    # the luma-only format on the same bytes gives a different image: that difference is the feature
    assert not np.array_equal(edge, ctx.process(nv, rip.OP_EDGE, rip.FMT_NV12))
    assert not np.array_equal(fused, ctx.process(nv, rip.OP_FUSED, rip.FMT_NV12, ksize=5, weights=wt))


@pytest.mark.gpu
def test_submit_collect_three_in_flight(ctx, oracle):
    h, w = 270, 480
    nv = _noise(6, h, w, 44)
    wt = rip.gauss_weights(5, 1.5)
    want = [oracle.blur(R.to_rgba(R.decode(f)), 5, weights=wt, threads=0) for f in nv]
    tickets, got = [], []
    for i in range(6):
        tickets.append(ctx.submit(nv[i], rip.OP_GAUSSIAN, rip.FMT_NV12_COLOR, ksize=5, weights=wt))
        if len(tickets) == 3:
            got.append(tickets.pop(0).collect())
    got += [t.collect() for t in tickets]
    for i in range(6):
        _eq(got[i], want[i], f"submit/collect frame {i}")


@pytest.mark.gpu
def test_two_device_context(oracle):
    if rip.device_count() < 2:
        pytest.skip("needs two GPUs")
    nv = _noise(5, 120, 160, 8)
    wt = rip.gauss_weights(5, 1.0)
    c = rip.Context([0, 1])
    try:
        gray = c.process(nv, rip.OP_GRAY, rip.FMT_NV12_COLOR)
        blur = c.process(nv, rip.OP_GAUSSIAN, rip.FMT_NV12_COLOR, ksize=5, weights=wt)
        fused = c.process(nv, rip.OP_FUSED, rip.FMT_NV12_COLOR, ksize=5, weights=wt)
    finally:
        c.close()
    for i in range(5):
        rgb = R.decode(nv[i])
        _eq(gray[i], oracle.gray(rgb), f"2-device GRAY frame {i}")
        _eq(blur[i], oracle.blur(R.to_rgba(rgb), 5, weights=wt), f"2-device GAUSSIAN frame {i}")
        _eq(fused[i], oracle.fused(rgb, 5, weights=wt), f"2-device FUSED frame {i}")


@pytest.mark.gpu
def test_rejections(ctx):
    wt = rip.gauss_weights(5, 1.0)
    # odd width or height: the host pipeline, rip_convert and rip_gray
    for h, w in ((6, 9), (5, 8)):
        raw = np.zeros((1, h * w * 3 // 2), np.uint8)
        d_in, d_out = rip.DeviceBuffer(raw.nbytes + 64), rip.DeviceBuffer(h * w * 4 + 64)
        with pytest.raises(rip.RipError, match="even width and height"):
            rip.convert_dev(d_in.ptr, d_out.ptr, w, h, 1, rip.FMT_NV12_COLOR, rip.FMT_RGBA8)
        with pytest.raises(rip.RipError, match="even width and height"):
            rip.gray_dev(d_in.ptr, d_out.ptr, w, h, 1, rip.FMT_NV12_COLOR)
        d = rip.OpDesc()
        d.op, d.in_format = rip.OP_GRAY, rip.FMT_NV12_COLOR
        out = np.empty(h * w, np.uint8)
        rc = rip.lib().rip_process_host(ctx.ptr, C.byref(d), raw.ctypes.data, out.ctypes.data, w, h, 1, None)
        assert rc == -1 and b"even width and height" in rip.lib().rip_last_error_string()
    nv = _noise(1, 64, 64, 1)
    with pytest.raises(rip.RipError, match="row-band"):
        ctx.process(nv, rip.OP_FUSED, rip.FMT_NV12_COLOR, ksize=5, weights=wt, banded=True)
    d_in, d_out = rip.DeviceBuffer(nv.nbytes).upload(nv), rip.DeviceBuffer(64 * 64 * 4)
    with pytest.raises(rip.RipError, match=r"rc=-4.*rip_gray"):
        rip.sobel_dev(d_in.ptr, d_out.ptr, 64, 64, 1, rip.FMT_NV12_COLOR)
    with pytest.raises(rip.RipError, match=r"rc=-4.*rip_gray"):
        rip.fused_dev(d_in.ptr, d_out.ptr, 64, 64, 1, rip.FMT_NV12_COLOR, 5, wt)
    with pytest.raises(rip.RipError, match="rc=-4"):
        rip.convert_dev(d_in.ptr, d_out.ptr, 64, 64, 1, rip.FMT_NV12_COLOR, rip.FMT_GRAY8)
    with pytest.raises(rip.RipError, match="rc=-4"):
        rip.convert_dev(d_in.ptr, d_out.ptr, 64, 64, 1, rip.FMT_NV12, rip.FMT_RGBA8)


@pytest.mark.gpu
@pytest.mark.parametrize("n,h,w", [(2, 130, 248), (1, 74, 76), (3, 40, 1000)])
def test_decode_stays_inside_its_output_buffer(oracle, n, h, w):
    """Every decode writes into the middle of a canary-filled buffer (256 KB on either side): the canaries must survive and the
    payload must equal the reference."""
    pad = 256 * 1024
    nv = _noise(n, h, w, 515)
    d_in = rip.DeviceBuffer(nv.nbytes).upload(nv)

    def run(name, out_bytes, launch, want):
        buf = rip.DeviceBuffer(out_bytes + 2 * pad)
        buf.upload(np.full(out_bytes + 2 * pad, 0xA5, np.uint8))
        launch(buf.ptr + pad)
        got = buf.download((out_bytes + 2 * pad,))
        assert (got[:pad] == 0xA5).all() and (got[pad + out_bytes:] == 0xA5).all(), f"{name} {n}x{h}x{w}: wrote outside its output"
        _eq(got[pad: pad + out_bytes].reshape(want.shape), want, f"{name} {n}x{h}x{w}")
        buf.free()

    for order in R.ORDERS:
        run(f"convert {order}", n * h * w * len(order),
            lambda p: rip.convert_dev(d_in.ptr, p, w, h, n, rip.FMT_NV12_COLOR, OUT_FMT[order]), R.decode(nv, order))
    g = _want_gray(oracle, nv)
    run("gray u8", n * h * w, lambda p: rip.gray_dev(d_in.ptr, p, w, h, n, rip.FMT_NV12_COLOR, rip.GRAY_OUT_U8), g)
    run("gray rgba", n * h * w * 4, lambda p: rip.gray_dev(d_in.ptr, p, w, h, n, rip.FMT_NV12_COLOR, rip.GRAY_OUT_RGBA), _gray_rgba(g))


@pytest.mark.gpu
def test_cpp_controller_drop_in(tmp_path, oracle):
    """PerformBatch / PerformFused / SubmitFrame + CollectFrame with RIP_FMT_NV12_COLOR through the C++ Controller, and its
    rejection of short buffers and odd widths, against bytes computed here through the oracle."""
    exe = _build_dropin(tmp_path)
    n, h, w = 3, 120, 164
    nv = _smooth_nv12(n, h, w, 12)
    nv.tofile(str(tmp_path / "in.nv12"))
    res = subprocess.run([exe, str(tmp_path), str(w), str(h), str(n)], capture_output=True, text=True)
    assert res.returncode == 0 and res.stdout.strip().endswith("OK"), res.stdout + res.stderr
    wt = oracle.gauss_weights(5, 1.5)
    rgb = R.decode(nv)
    gray = np.stack([oracle.gray(f) for f in rgb])
    want = {"batch_GRAYSCALE": gray,
            "batch_GAUSSIAN": np.stack([oracle.blur(R.to_rgba(f), 5, weights=wt) for f in rgb]),
            "batch_EDGE": np.stack([oracle.sobel(g) for g in gray]),
            "batch_FUSED": np.stack([oracle.fused(f, 5, weights=wt) for f in rgb]),
            "fused_frame0": oracle.fused(rgb[0], 5, weights=wt)}
    want["submit_GAUSSIAN"] = want["batch_GAUSSIAN"]
    for name, ref in want.items():
        got = np.fromfile(str(tmp_path / (name + ".raw")), np.uint8)
        _eq(got.reshape(ref.shape), ref, name)
