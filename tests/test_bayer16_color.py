"""RIP_FMT_BAYER_<pattern>10 / 12 / 14 / 16: Bayer raw frames of 10 to 16 bits per sample (one little-endian 16-bit word each)
decoded exactly as OpenCV's cvtColor(COLOR_Bayer**2RGB) on the CV_16U frame followed by convertTo(CV_8U, 1 / 2^(bits - 8)),
then the reference's chain on that 8-bit colour image -- the contract of the 8-bit Bayer formats.

CPU tests pin the numpy restatement (tests/bayer16_ref.py) to live cv2 and to the cv2 outputs recorded in
tests/golden/cv2_bayer16.npz, pin its reduction on every 16-bit input, and check the host-side sizes, shapes and dtypes.  GPU
tests compare every device path with that restatement followed by the C oracle, bit for bit."""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np
import pytest

import bayer16_ref as R
import rip_b200 as rip

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "opencl-development-real-time-image-processing_b200")
GOLDEN = os.path.join(ROOT, "tests", "golden", "cv2_bayer16.npz")
FMT = {(p, b): getattr(rip, f"FMT_BAYER_{p.upper()}{b}") for b in R.BITS for p in R.PATTERNS}
CODES = sorted(FMT)   # (pattern, bits)
OUT_FMT = {"rgb": rip.FMT_RGB8, "bgr": rip.FMT_BGR8, "rgba": rip.FMT_RGBA8, "bgra": rip.FMT_BGRA8}


def _eq(got, want, what=""):
    if not np.array_equal(got, want):
        d = np.abs(got.astype(int) - want.astype(int))
        idx = np.argwhere(d > 0)
        raise AssertionError(f"{what}: {len(idx)} of {d.size} bytes differ, max abs {d.max()}, first at {idx[0].tolist()}")


def _noise(n, h, w, bits, seed):
    return np.random.default_rng(seed).integers(0, 1 << bits, (n, h, w), dtype=np.uint16)


def _out_bytes(op, fmt, w, h, gray_out=rip.GRAY_OUT_U8):
    d = rip.OpDesc()
    d.op, d.in_format, d.gray_out = op, fmt, gray_out
    b = C.c_size_t(0)
    rip.check(rip.lib().rip_out_bytes_per_frame(C.byref(d), w, h, C.byref(b)))
    return b.value


def _golden_cases(g, bits):
    return sorted(k.split(".")[1] for k in g.files if k.startswith(f"{bits}.") and k.endswith(".in"))


# ---- CPU: the restatement, the reduction, the pattern names, the host-side sizes, shapes and dtypes ------------------------
def test_format_codes():
    """16 new codes after the 8-bit ones: depth-major, the pattern order of codes 12-15 within each depth."""
    assert [FMT[p, b] for b in R.BITS for p in R.PATTERNS] == list(range(16, 32))
    assert [getattr(rip, f"FMT_BAYER_{p.upper()}8") for p in R.PATTERNS] == [12, 13, 14, 15]
    assert rip.FMTS_U16 == frozenset(range(16, 32))


@pytest.mark.parametrize("bits", R.BITS)
def test_reference_equals_cv2(bits):
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(bits)
    g = np.load(GOLDEN)
    frames = [rng.integers(0, 1 << bits, s, dtype=np.uint16) for s in ((3, 3), (4, 5), (9, 16), (31, 17), (480, 641))]
    frames.append(rng.integers(0, 1 << 16, (33, 40), dtype=np.uint16))   # padding bits set
    frames += [f for case in _golden_cases(g, bits) for f in g[f"{bits}.{case}.in"][:8]]
    for f in frames:
        for pattern in R.PATTERNS:
            for order in R.ORDERS:
                _eq(R.decode(f, pattern, bits, order), R.cv2_decode(f, pattern, bits, order),
                    f"{pattern}{bits} {order} {f.shape} vs cv2 {cv2.__version__}")


def test_reference_equals_recorded_cv2():
    g = np.load(GOLDEN)
    for bits in R.BITS:
        cases = _golden_cases(g, bits)
        want = {"noise3x3", "noise3x4", "noise4x3", "noise7x9", "noise6x9", "noise9x6", "noise5x16", "flat", "ties", "tienoise",
                "impulse5x5", "hramp", "vramp"} | ({"padded"} if bits < 16 else set())
        assert set(cases) == want, (bits, cases)
        for case in cases:
            for pattern in R.PATTERNS:
                for order in ("rgb", "bgra"):
                    _eq(R.decode(g[f"{bits}.{case}.in"], pattern, bits, order), g[f"{pattern}{bits}.{case}.{order}"],
                        f"{pattern}{bits} {case} {order}")
        artemis = R.hash_noise(1023, 683, bits, bits)
        for pattern in R.PATTERNS:
            for order in R.ORDERS:
                digest = hashlib.sha256(R.decode(artemis, pattern, bits, order).tobytes()).digest()
                assert digest == g[f"{pattern}{bits}.artemis.{order}.sha256"].tobytes(), f"{pattern}{bits} {order} 683x1023"


def test_recorded_ties_have_both_quotient_parities():
    """The tie frames hold v = (q + 1/2) 2^s for every q: round half to even sends even q down and odd q up."""
    g = np.load(GOLDEN)
    for bits in R.BITS:
        s = bits - 8
        ties = g[f"{bits}.ties.in"][:, 0, 0].astype(np.int64)
        q = ties >> s
        assert ((ties & ((1 << s) - 1)) == 1 << (s - 1)).all() and sorted(q) == list(range(256))
        got = g[f"rggb{bits}.ties.rgb"][:, 1, 1, 0].astype(np.int64)
        assert (got == np.where(q & 1, np.minimum(q + 1, 255), q)).all(), bits


def test_reduction_on_every_input():
    """The reduction on all 65 536 inputs at every depth, against an independent statement of convertTo (float division,
    numpy's round half to even, saturation) and against cv2 when present.  Rounding half up, or truncating, fails here."""
    v = np.arange(1 << 16, dtype=np.int64)
    cv2 = None
    try:
        import cv2
    except ImportError:
        pass
    for bits in R.BITS:
        s = bits - 8
        want = np.minimum(255, np.round(v / float(1 << s))).astype(np.uint8)
        got = R.reduce(v, bits)
        _eq(got, want, f"reduce at {bits} bits")
        half_up = np.minimum(255, (v + (1 << (s - 1))) >> s)
        trunc = np.minimum(255, v >> s)
        assert (half_up != want).sum() == 128 and (trunc != want).sum() >= 128, bits
        assert got[(1 << bits) - 1] == 255 and got[(1 << s) * 255 + (1 << (s - 1))] == 255   # full scale; 255.5 -> 256 -> 255
        if cv2 is not None:
            _eq(cv2.convertScaleAbs(v.astype(np.uint16).reshape(256, 256), alpha=1.0 / (1 << s)).ravel(), want, f"cv2 at {bits}")


def test_demosaic_is_the_8_bit_one():
    """On 8-bit samples the 16-bit demosaic gives exactly bayer_ref's result: one set of formulas for every depth."""
    import bayer_ref as R8
    rng = np.random.default_rng(3)
    for shape in ((3, 3), (7, 10), (24, 17)):
        f = rng.integers(0, 256, shape, dtype=np.uint8)
        for pattern in R.PATTERNS:
            _eq(R.demosaic(f, pattern).astype(np.uint8), R8.decode(f, pattern), f"{pattern} {shape}")


def test_pattern_names_against_opencv():
    """A frame that holds full scale on the named red sites only decodes to pure red inside, at every depth; and OpenCV's
    code for each name gives the same colours on 16-bit input."""
    yy, xx = np.mgrid[0:8, 0:10]
    for bits in R.BITS:
        for pattern in R.PATTERNS:
            i = pattern.upper().index("R")
            f = np.where(((yy & 1) == i // 2) & ((xx & 1) == i % 2), (1 << bits) - 1, 0).astype(np.uint16)
            rgb = R.decode(f, pattern, bits)
            assert (rgb[..., 0] > 0).all() and (rgb[..., 1:] == 0).all(), (pattern, bits)
    cv2 = pytest.importorskip("cv2")
    for pattern, code in R.CV2_CODE.items():
        f = np.random.default_rng(5).integers(0, 1 << 16, (12, 14), dtype=np.uint16)
        _eq(R.decode(f, pattern, 16), cv2.convertScaleAbs(cv2.cvtColor(f, getattr(cv2, f"COLOR_Bayer{code}2RGB")), alpha=1 / 256),
            f"{pattern} = COLOR_Bayer{code}2RGB")


def test_output_sizes_of_the_16_bit_formats():
    w, h = 683, 1023
    for fmt in FMT.values():
        assert _out_bytes(rip.OP_GAUSSIAN, fmt, w, h) == w * h * 4
        assert _out_bytes(rip.OP_GRAY, fmt, w, h) == w * h
        assert _out_bytes(rip.OP_GRAY, fmt, w, h, rip.GRAY_OUT_RGBA) == w * h * 4
        assert _out_bytes(rip.OP_EDGE, fmt, w, h) == w * h
        assert _out_bytes(rip.OP_FUSED, fmt, w, h) == w * h


def test_python_shapes_and_dtypes():
    """Context.process / submit take 16-bit Bayer frames as (N, H, W) or (H, W) native little-endian uint16, and refuse uint8
    for them; every other format refuses uint16."""
    c = object.__new__(rip.Context)   # the shape handling needs no device
    wt = rip.gauss_weights(5, 1.0)
    for fmt in FMT.values():
        assert rip.CHANNELS[fmt] == 1
        a, _, n, h, w, shape, out, squeeze = c._shapes(np.zeros((3, 5, 7), np.uint16), rip.OP_GAUSSIAN, fmt,
                                                        rip.GRAY_OUT_U8, 5, wt, None)
        assert (n, h, w, shape, out.shape, out.dtype, squeeze) == (3, 5, 7, (3, 5, 7, 4), (3, 5, 7, 4), np.uint8, False)
        a, _, n, h, w, shape, out, squeeze = c._shapes(np.zeros((5, 7), np.uint16), rip.OP_EDGE, fmt, rip.GRAY_OUT_U8, 0, None, None)
        assert (a.shape, a.nbytes, n, h, w, shape, squeeze) == ((1, 5, 7), 70, 1, 5, 7, (1, 5, 7), True)
        a, _, n, h, w, shape, out, squeeze = c._shapes(np.zeros((2, 9, 10), np.uint16), rip.OP_GRAY, fmt,
                                                        rip.GRAY_OUT_RGBA, 0, None, None)
        assert (n, h, w, shape, squeeze) == (2, 9, 10, (2, 9, 10, 4), False)
        for bad in (np.zeros((2, 9, 10), np.uint8), np.zeros((2, 9, 10), ">u2"), np.zeros((2, 9, 10), np.int16)):
            with pytest.raises(AssertionError, match="little-endian uint16"):
                c._shapes(bad, rip.OP_GRAY, fmt, rip.GRAY_OUT_U8, 0, None, None)
    for fmt, shape in ((rip.FMT_BAYER_RGGB8, (2, 9, 10)), (rip.FMT_GRAY8, (9, 10)), (rip.FMT_RGB8, (9, 10, 3)),
                       (rip.FMT_NV12_COLOR, (12, 10))):
        with pytest.raises(AssertionError, match="takes uint8"):
            c._shapes(np.zeros(shape, np.uint16), rip.OP_GRAY if fmt != rip.FMT_GRAY8 else rip.OP_EDGE, fmt, rip.GRAY_OUT_U8, 0,
                      None, None)


@pytest.mark.skipif(rip.device_count() > 0, reason="only meaningful on a box without a GPU")
def test_16_bit_bayer_fails_loudly_without_gpu():
    for fmt in FMT.values():
        with pytest.raises(rip.RipError, match="no CUDA device|no CPU fallback"):
            rip.convert_dev(16, 32, 4, 4, 1, fmt, rip.FMT_RGBA8)
        with pytest.raises(rip.RipError, match="no CUDA device|no CPU fallback"):
            rip.gray_dev(16, 32, 4, 4, 1, fmt)


def _build_dropin(tmp_path):
    exe = str(tmp_path / "bayer16_dropin")
    cmd = ["/usr/bin/g++", "-O2", "-std=c++17", "-ffp-contract=off", "-I", os.path.join(PKG, "host"), "-I", os.path.join(ROOT, "include"),
           "-I", "/usr/local/cuda/include", os.path.join(ROOT, "tests", "cpp", "bayer16_dropin.cpp"), "-o", exe, "-L", PKG, "-lrip_host",
           "-lrip_cuda", "-Wl,-rpath," + PKG, "-pthread"]
    subprocess.run(cmd, check=True)
    return exe


def test_cpp_driver_builds(tmp_path):
    exe = _build_dropin(tmp_path)
    res = subprocess.run([exe], capture_output=True, text=True)
    assert res.returncode == 2 and "usage" in res.stderr
    res = subprocess.run([exe, str(tmp_path), str(rip.FMT_BAYER_GBRG8), "8", "8", "1"], capture_output=True, text=True)
    assert res.returncode == 2 and "not a 10- to 16-bit" in res.stderr


# ---- GPU -------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    if rip.device_count() < 1:
        pytest.fail("GPU tests need a CUDA device: librip_cuda has no CPU fallback")
    c = rip.Context([0])
    yield c
    c.close()


def _in_order(rgb, order):
    """An RGB image (.., 3) in another channel order (alpha 255)."""
    out = rgb[..., ::-1] if order.startswith("bgr") else rgb
    if len(order) == 4:
        out = np.concatenate([out, np.full(out.shape[:-1] + (1,), 255, np.uint8)], -1)
    return np.ascontiguousarray(out)


def _convert(fmt, fr, order, in_off=0, out_off=0):
    n, h, w = fr.shape
    bpp = len(order)
    d_in = rip.DeviceBuffer(fr.nbytes + 16).upload(fr, offset=in_off)
    d_out = rip.DeviceBuffer(n * h * w * bpp + 16)
    rip.convert_dev(d_in.ptr + in_off, d_out.ptr + out_off, w, h, n, fmt, OUT_FMT[order])
    return d_out.download((n, h, w, bpp), offset=out_off)


def _gray_dev(fmt, fr, out_mode, in_off=0, out_off=0):
    n, h, w = fr.shape
    bpp = 4 if out_mode == rip.GRAY_OUT_RGBA else 1
    d_in = rip.DeviceBuffer(fr.nbytes + 16).upload(fr, offset=in_off)
    d_out = rip.DeviceBuffer(n * h * w * bpp + 16)
    rip.gray_dev(d_in.ptr + in_off, d_out.ptr + out_off, w, h, n, fmt, out_mode)
    return d_out.download((n, h, w, bpp) if bpp == 4 else (n, h, w), offset=out_off)


def _want_gray(oracle, pattern, bits, fr):
    return np.stack([oracle.gray(R.decode(f, pattern, bits), threads=0) for f in fr])


def _gray_rgba(g):
    return np.stack([g, g, g, np.full_like(g, 255)], -1)


# (n, h, w): W % 8 != 0 and odd W take the byte-granular kernel, W % 8 == 0 the wide one (also with odd H, H = 3 and H = 4,
# where every row pair is a border pair); an odd W * H makes the frame stride 2 mod 4 bytes, so every second frame of the
# byte-granular kernel starts off a 4-byte boundary
SHAPES = [(1, 3, 3), (3, 3, 4), (2, 4, 3), (2, 7, 9), (3, 6, 9), (2, 9, 6), (3, 3, 8), (2, 4, 8), (2, 9, 16), (3, 74, 76),
          (2, 75, 77), (1, 1023, 683), (2, 121, 1920)]


@pytest.mark.gpu
@pytest.mark.parametrize("pattern,bits", CODES)
def test_convert_every_code(ctx, pattern, bits):
    for n, h, w in SHAPES:
        fr = _noise(n, h, w, bits, 100 + h + w)
        if (h, w) == (9, 16):
            fr |= np.uint16(0xffff ^ ((1 << bits) - 1))   # padding bits set: used as they are, so most channels saturate
        rgb = R.decode(fr, pattern, bits)
        for order in R.ORDERS:
            _eq(_convert(FMT[pattern, bits], fr, order), _in_order(rgb, order), f"rip_convert {pattern}{bits} {order} {n}x{h}x{w}")


@pytest.mark.gpu
@pytest.mark.parametrize("pattern,bits", CODES)
def test_convert_recorded_cases(ctx, pattern, bits):
    """The adversarial frames of the golden file (padding bits, flat and full-scale, ties, impulses, ramps) through the device."""
    g = np.load(GOLDEN)
    for case in _golden_cases(g, bits):
        fr = g[f"{bits}.{case}.in"]
        for order in ("rgb", "bgra"):
            _eq(_convert(FMT[pattern, bits], fr, order), g[f"{pattern}{bits}.{case}.{order}"],
                f"rip_convert {pattern}{bits} {case} {order} vs cv2")


@pytest.mark.gpu
@pytest.mark.parametrize("bits", R.BITS)
def test_convert_4k(ctx, bits):
    fr = np.stack([R.hash_noise(2160, 3840, bits, 7 + bits)])
    for pattern in R.PATTERNS:
        rgb = R.decode(fr, pattern, bits)
        for order in ("rgb", "bgra"):
            _eq(_convert(FMT[pattern, bits], fr, order), _in_order(rgb, order), f"rip_convert {pattern}{bits} {order} 4K")


@pytest.mark.gpu
@pytest.mark.parametrize("pattern,bits", CODES)
def test_gray_dev_both_out_modes(ctx, oracle, pattern, bits):
    shapes = [(3, 74, 76), (2, 75, 77), (2, 3, 3), (2, 4, 8), (2, 9, 6)]
    if bits in (12, 16):
        shapes.append((1, 2160, 3840))
    for n, h, w in shapes:
        fr = _noise(n, h, w, bits, 5 + w)
        g = _want_gray(oracle, pattern, bits, fr)
        _eq(_gray_dev(FMT[pattern, bits], fr, rip.GRAY_OUT_U8), g, f"rip_gray {pattern}{bits} u8 {n}x{h}x{w}")
        _eq(_gray_dev(FMT[pattern, bits], fr, rip.GRAY_OUT_RGBA), _gray_rgba(g), f"rip_gray {pattern}{bits} rgba {n}x{h}x{w}")


@pytest.mark.gpu
@pytest.mark.parametrize("bits", R.BITS)
@pytest.mark.parametrize("in_off,out_off", [(1, 0), (0, 1), (3, 5), (2, 0), (4, 12), (8, 8), (12, 4), (6, 2)])
def test_convert_and_gray_unaligned_buffers(ctx, oracle, bits, in_off, out_off):
    """Odd offsets put every sample on an odd byte address; 2, 4, 6, 8 and 12 keep 2-byte alignment but break the 16-byte
    input (or 8- and 16-byte output) alignment the wide kernel needs.  (3, 6, 24) is wide-kernel shaped, (3, 5, 13) has
    frame strides of 130 bytes."""
    for n, h, w in ((3, 6, 24), (3, 5, 13)):
        fr = _noise(n, h, w, bits, 7)
        for pattern in R.PATTERNS:
            fmt = FMT[pattern, bits]
            rgb = R.decode(fr, pattern, bits)
            for order in R.ORDERS:
                _eq(_convert(fmt, fr, order, in_off, out_off), _in_order(rgb, order),
                    f"rip_convert {pattern}{bits} {order} {h}x{w} offsets {in_off}/{out_off}")
            g = _want_gray(oracle, pattern, bits, fr)
            _eq(_gray_dev(fmt, fr, rip.GRAY_OUT_U8, in_off, out_off), g, f"rip_gray {pattern}{bits} u8 unaligned")
            _eq(_gray_dev(fmt, fr, rip.GRAY_OUT_RGBA, in_off, out_off), _gray_rgba(g), f"rip_gray {pattern}{bits} rgba unaligned")


@pytest.mark.gpu
@pytest.mark.parametrize("bits", R.BITS)
def test_gray_flat_frames_take_the_table(ctx, oracle, bits):
    """A constant raw sample gives r = g = b = q, so t = 1000 q and every pixel takes the (r, g) table path: one frame for
    every q (its tie value too, and the saturated values)."""
    s = bits - 8
    vals = [q << s for q in range(256)] + [(2 * q + 1) << (s - 1) for q in range(0, 256, 3)] + [(1 << bits) - 1, 0xffff]
    for pattern in R.PATTERNS:
        for h, w in ((64, 96), (9, 13)):
            fr = np.stack([np.full((h, w), v, np.uint16) for v in vals])
            assert sorted(set(R.decode(fr[:, :3, :3], pattern, bits)[:, 1, 1, 0])) == list(range(256))
            g = _want_gray(oracle, pattern, bits, fr)
            _eq(_gray_dev(FMT[pattern, bits], fr, rip.GRAY_OUT_U8), g, f"flat rip_gray {pattern}{bits} u8")
            _eq(_gray_dev(FMT[pattern, bits], fr, rip.GRAY_OUT_RGBA), _gray_rgba(g), f"flat rip_gray {pattern}{bits} rgba")
            _eq(ctx.process(fr, rip.OP_GRAY, FMT[pattern, bits]), g, f"flat GRAY {pattern}{bits}")


def _smooth(n, h, w, bits, seed):
    """Camera-like raw frames: smooth content with noise and a flat black bar (the blur's constant windows)."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    top = (1 << bits) - 1
    out = []
    for _ in range(n):
        fx, fy, ph = rng.uniform(0.002, 0.03), rng.uniform(0.002, 0.03), rng.uniform(0, 6.28)
        f = 0.47 * top * (1 + 0.75 * np.sin(fx * xx + fy * yy + ph)) + rng.integers(-3 << (bits - 8), 4 << (bits - 8), (h, w))
        f = np.clip(f, 0, top).astype(np.uint16)
        f[: h // 8] = 0
        out.append(f)
    return np.stack(out)


@pytest.mark.gpu
@pytest.mark.parametrize("k,sigma", [(5, 1.5), (9, 2.5), (17, 6.0)])
@pytest.mark.parametrize("kernel", ["RIP_BLUR_STREAM", "RIP_BLUR_TILED"])
def test_pipeline_gaussian(ctx, oracle, opt, k, sigma, kernel):
    """Demosaic to RGBA, then the streaming or the tiled blur kernel, forced; every pattern, the depths in turn."""
    opt(kernel, 1)
    wt = rip.gauss_weights(k, sigma)
    for i, pattern in enumerate(R.PATTERNS):
        bits = R.BITS[(i + k) % 4]
        for fr in (_smooth(2, 270, 480, bits, k), _noise(2, 121, 163, bits, k)):
            n, h, w = fr.shape
            got = ctx.process(fr, rip.OP_GAUSSIAN, FMT[pattern, bits], ksize=k, weights=wt)
            assert got.shape == (n, h, w, 4)
            for j in range(n):
                want = oracle.blur(R.decode(fr[j], pattern, bits, "rgba"), k, weights=wt, threads=0)
                _eq(got[j], want, f"GAUSSIAN {pattern}{bits} {k}x{k} {kernel} {h}x{w} frame {j}")


@pytest.mark.gpu
@pytest.mark.parametrize("pattern,bits", CODES)
def test_pipeline_gray_edge_and_fused(ctx, oracle, pattern, bits):
    wt = rip.gauss_weights(5, 1.0)
    shapes = [(2, 75, 77), (3, 64, 128), (2, 3, 3)] + ([(2, 1080, 1920)] if bits == 12 else [])
    for n, h, w in shapes:
        fr = _noise(n, h, w, bits, 3 + h)
        fmt = FMT[pattern, bits]
        gray = ctx.process(fr, rip.OP_GRAY, fmt)
        gray_rgba = ctx.process(fr, rip.OP_GRAY, fmt, gray_out=rip.GRAY_OUT_RGBA)
        edge = ctx.process(fr, rip.OP_EDGE, fmt)
        fused = ctx.process(fr, rip.OP_FUSED, fmt, ksize=5, weights=wt)
        for i in range(n):
            rgb = R.decode(fr[i], pattern, bits)
            g = oracle.gray(rgb, threads=0)
            _eq(gray[i], g, f"GRAY {pattern}{bits} {h}x{w} frame {i}")
            _eq(gray_rgba[i], _gray_rgba(g), f"GRAY rgba {pattern}{bits} {h}x{w} frame {i}")
            _eq(edge[i], oracle.sobel(g, threads=0), f"EDGE {pattern}{bits} {h}x{w} frame {i}")
            _eq(fused[i], oracle.fused(rgb, 5, weights=wt, threads=0), f"FUSED {pattern}{bits} {h}x{w} frame {i}")


@pytest.mark.gpu
@pytest.mark.parametrize("pattern,bits", [("rggb", 12), ("gbrg", 16)])
def test_pipeline_chunks_large_batches(ctx, oracle, pattern, bits):
    """14 frames of 1080p are 58 MB of 16-bit input: the pipeline moves them in two chunks (process and submit)."""
    fr = _smooth(14, 1080, 1920, bits, 77)
    fmt = FMT[pattern, bits]
    wt = rip.gauss_weights(5, 1.0)
    gray = ctx.process(fr, rip.OP_GRAY, fmt)
    fused = ctx.submit(fr, rip.OP_FUSED, fmt, ksize=5, weights=wt).collect()
    for i in range(len(fr)):
        rgb = R.decode(fr[i], pattern, bits)
        _eq(gray[i], oracle.gray(rgb, threads=0), f"chunked GRAY {pattern}{bits} frame {i}")
        _eq(fused[i], oracle.fused(rgb, 5, weights=wt, threads=0), f"chunked FUSED {pattern}{bits} frame {i}")


@pytest.mark.gpu
@pytest.mark.parametrize("bits", R.BITS)
def test_submit_collect_three_in_flight(ctx, oracle, bits):
    fr = _noise(6, 270, 481, bits, 44)
    wt = rip.gauss_weights(5, 1.5)
    pattern = R.PATTERNS[R.BITS.index(bits)]
    want = [oracle.blur(R.decode(f, pattern, bits, "rgba"), 5, weights=wt, threads=0) for f in fr]
    tickets, got = [], []
    for i in range(6):
        tickets.append(ctx.submit(fr[i], rip.OP_GAUSSIAN, FMT[pattern, bits], ksize=5, weights=wt))
        if len(tickets) == 3:
            got.append(tickets.pop(0).collect())
    got += [t.collect() for t in tickets]
    for i in range(6):
        _eq(got[i], want[i], f"submit/collect {pattern}{bits} frame {i}")


@pytest.mark.gpu
def test_rejections(ctx):
    wt = rip.gauss_weights(5, 1.0)
    for (pattern, bits), fmt in FMT.items():
        name = f"BAYER_{pattern.upper()}{bits}"
        # W or H below 3: the host pipeline, rip_convert and rip_gray, before any byte is read
        msg = f"{name} frames need a width and height of at least 3"
        raw = np.zeros(64, np.uint16)
        d_in, d_out = rip.DeviceBuffer(raw.nbytes), rip.DeviceBuffer(256)
        for h, w in ((2, 8), (8, 2), (1, 1), (2, 2)):
            with pytest.raises(rip.RipError, match=msg):
                rip.convert_dev(d_in.ptr, d_out.ptr, w, h, 1, fmt, rip.FMT_RGBA8)
            with pytest.raises(rip.RipError, match=msg):
                rip.gray_dev(d_in.ptr, d_out.ptr, w, h, 1, fmt)
            for op in (rip.OP_GRAY, rip.OP_GAUSSIAN, rip.OP_EDGE, rip.OP_FUSED):
                d = ctx._desc(op, fmt, ksize=5, weights=wt)
                out = np.empty(h * w * 4, np.uint8)
                rc = rip.lib().rip_process_host(ctx.ptr, C.byref(d), raw.ctypes.data, out.ctypes.data, w, h, 1, None)
                assert rc == -1 and msg.encode() in rip.lib().rip_last_error_string()
        fr = _noise(1, 64, 64, bits, 1)
        with pytest.raises(rip.RipError, match="rc=-4.*row-band"):
            ctx.process(fr, rip.OP_FUSED, fmt, ksize=5, weights=wt, banded=True)
        with pytest.raises(rip.RipError, match="rc=-4.*row-band"):
            ctx.process(fr, rip.OP_EDGE, fmt, banded=True)
        d_in, d_out = rip.DeviceBuffer(fr.nbytes).upload(fr), rip.DeviceBuffer(64 * 64 * 4)
        with pytest.raises(rip.RipError, match=f"rc=-4.*rip_sobel: RIP_FMT_{name} .*rip_gray"):
            rip.sobel_dev(d_in.ptr, d_out.ptr, 64, 64, 1, fmt)
        with pytest.raises(rip.RipError, match=f"rc=-4.*rip_fused: RIP_FMT_{name} .*rip_gray"):
            rip.fused_dev(d_in.ptr, d_out.ptr, 64, 64, 1, fmt, 5, wt)
        for out_fmt in (rip.FMT_GRAY8, rip.FMT_NV12, fmt):
            with pytest.raises(rip.RipError, match="rc=-4"):
                rip.convert_dev(d_in.ptr, d_out.ptr, 64, 64, 1, fmt, out_fmt)
        with pytest.raises(AssertionError, match="little-endian uint16"):
            ctx.process(fr.astype(np.uint8), rip.OP_GRAY, fmt)
    # the codes after the last Bayer format are not formats
    for bad in (32, 33, 1000):
        with pytest.raises(rip.RipError, match="rc=-4"):
            rip.convert_dev(d_in.ptr, d_out.ptr, 64, 64, 1, bad, rip.FMT_RGBA8)


@pytest.mark.gpu
@pytest.mark.parametrize("bits", R.BITS)
@pytest.mark.parametrize("n,h,w", [(2, 130, 248), (3, 75, 77), (3, 40, 1000), (2, 3, 8)])
def test_decode_stays_inside_its_output_buffer(oracle, bits, n, h, w):
    """Every decode writes into the middle of a canary-filled buffer (256 KB on either side): the canaries must survive and the
    payload must equal the reference."""
    pad = 256 * 1024
    fr = _noise(n, h, w, bits, 515)
    d_in = rip.DeviceBuffer(fr.nbytes).upload(fr)

    def run(name, out_bytes, launch, want):
        buf = rip.DeviceBuffer(out_bytes + 2 * pad)
        buf.upload(np.full(out_bytes + 2 * pad, 0xA5, np.uint8))
        launch(buf.ptr + pad)
        got = buf.download((out_bytes + 2 * pad,))
        assert (got[:pad] == 0xA5).all() and (got[pad + out_bytes:] == 0xA5).all(), f"{name} {n}x{h}x{w}: wrote outside its output"
        _eq(got[pad: pad + out_bytes].reshape(want.shape), want, f"{name} {n}x{h}x{w}")
        buf.free()

    for pattern in R.PATTERNS:
        fmt = FMT[pattern, bits]
        rgb = R.decode(fr, pattern, bits)
        for order in R.ORDERS:
            run(f"convert {pattern}{bits} {order}", n * h * w * len(order),
                lambda p: rip.convert_dev(d_in.ptr, p, w, h, n, fmt, OUT_FMT[order]), _in_order(rgb, order))
        g = _want_gray(oracle, pattern, bits, fr)
        run(f"gray {pattern}{bits} u8", n * h * w, lambda p: rip.gray_dev(d_in.ptr, p, w, h, n, fmt, rip.GRAY_OUT_U8), g)
        run(f"gray {pattern}{bits} rgba", n * h * w * 4, lambda p: rip.gray_dev(d_in.ptr, p, w, h, n, fmt, rip.GRAY_OUT_RGBA),
            _gray_rgba(g))


@pytest.mark.gpu
@pytest.mark.parametrize("pattern,bits", [("rggb", 10), ("bggr", 12), ("grbg", 14), ("gbrg", 16)])
def test_cpp_controller_drop_in(tmp_path, oracle, pattern, bits):
    """PerformBatch / PerformFused / SubmitFrame + CollectFrame through the C++ Controller, and its rejection of short buffers
    and of frames narrower or shorter than 3, against bytes computed here through the oracle."""
    exe = _build_dropin(tmp_path)
    n, h, w = 3, 121, 163
    fr = _smooth(n, h, w, bits, 12)
    fr.astype("<u2").tofile(str(tmp_path / "in.raw"))
    res = subprocess.run([exe, str(tmp_path), str(FMT[pattern, bits]), str(w), str(h), str(n)], capture_output=True, text=True)
    assert res.returncode == 0 and res.stdout.strip().endswith("OK"), res.stdout + res.stderr
    wt = oracle.gauss_weights(5, 1.5)
    rgb = R.decode(fr, pattern, bits)
    gray = np.stack([oracle.gray(f) for f in rgb])
    want = {"batch_GRAYSCALE": gray,
            "batch_GAUSSIAN": np.stack([oracle.blur(R.decode(f, pattern, bits, "rgba"), 5, weights=wt) for f in fr]),
            "batch_EDGE": np.stack([oracle.sobel(g) for g in gray]),
            "batch_FUSED": np.stack([oracle.fused(f, 5, weights=wt) for f in rgb]),
            "fused_frame0": oracle.fused(rgb[0], 5, weights=wt)}
    want["submit_GAUSSIAN"] = want["batch_GAUSSIAN"]
    for name, ref in want.items():
        got = np.fromfile(str(tmp_path / (name + ".raw")), np.uint8)
        _eq(got.reshape(ref.shape), ref, name)
