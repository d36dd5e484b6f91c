"""RIP_FMT_BAYER_<pattern>10P_MIPI / 12P_MIPI / 10P_GENICAM / 12P_GENICAM: packed 10- and 12-bit Bayer raw frames (MIPI CSI-2
RAW10 / RAW12 and GenICam's LSB-first bit streams), unpacked on the device in the demosaic kernel and decoded exactly as
RIP_FMT_BAYER_<pattern>10 / 12 decode the unpacked samples -- then the reference's chain on that 8-bit colour image.

CPU tests pin the numpy packers (tests/bayer_packed_ref.py) to hand-written byte vectors of the published layouts and to
each other's round trips, and check the codes, host-side sizes, shapes and dtypes.  GPU tests compare every device path bit
for bit with two references: the restatement followed by the C oracle, and the device output of the same samples through
the unpacked codes."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import bayer16_ref as R16
import bayer_packed_ref as P
import rip_b200 as rip

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "opencl-development-real-time-image-processing_b200")
SUFFIX = {"mipi10": "10P_MIPI", "mipi12": "12P_MIPI", "genicam10": "10P_GENICAM", "genicam12": "12P_GENICAM"}
FMT = {(p, lay): getattr(rip, f"FMT_BAYER_{p.upper()}{SUFFIX[lay]}") for lay in P.LAYOUTS for p in R16.PATTERNS}
CODES = sorted(FMT)   # (pattern, layout)
OUT_FMT = {"rgb": rip.FMT_RGB8, "bgr": rip.FMT_BGR8, "rgba": rip.FMT_RGBA8, "bgra": rip.FMT_BGRA8}


def _u16_fmt(pattern, layout):
    """The unpacked code of the same pattern and depth."""
    return getattr(rip, f"FMT_BAYER_{pattern.upper()}{P.bits_of(layout)}")


def _eq(got, want, what=""):
    if not np.array_equal(got, want):
        d = np.abs(got.astype(int) - want.astype(int))
        idx = np.argwhere(d > 0)
        raise AssertionError(f"{what}: {len(idx)} of {d.size} bytes differ, max abs {d.max()}, first at {idx[0].tolist()}")


def _noise(n, h, w, layout, seed):
    """Random packed bytes: every byte string is a valid packed frame."""
    return np.random.default_rng(seed).integers(0, 256, (n, h, P.row_bytes(layout, w)), dtype=np.uint8)


def _out_bytes(op, fmt, w, h, gray_out=rip.GRAY_OUT_U8):
    d = rip.OpDesc()
    d.op, d.in_format, d.gray_out = op, fmt, gray_out
    b = C.c_size_t(0)
    rip.check(rip.lib().rip_out_bytes_per_frame(C.byref(d), w, h, C.byref(b)))
    return b.value


# ---- CPU: the packers, the codes, the host-side sizes, shapes and dtypes ----------------------------------------------------
# one group per layout with distinct bits in every position, written out from the layout tables
KNOWN = [
    ("mipi10", [0x3FF, 0x001, 0x2AA, 0x155], "FF 00 AA 55 67"),
    ("genicam10", [0x3FF, 0x001, 0x2AA, 0x155], "FF 07 A0 6A 55"),
    ("mipi10", [0x001, 0x002, 0x004, 0x300], "00 00 01 C0 09"),
    ("genicam10", [0x001, 0x002, 0x004, 0x300], "01 08 40 00 C0"),
    ("mipi12", [0xABC, 0x123], "AB 12 3C"),
    ("genicam12", [0xABC, 0x123], "BC 3A 12"),
    ("mipi12", [0xFFF, 0x001], "FF 00 1F"),
    ("genicam12", [0xFFF, 0x001], "FF 1F 00"),
]


@pytest.mark.parametrize("layout,samples,hexbytes", KNOWN)
def test_known_answer_vectors(layout, samples, hexbytes):
    want = np.array([int(b, 16) for b in hexbytes.split()], np.uint8)
    s = np.array([samples], np.uint16)
    _eq(P.pack(s, layout)[0], want, f"pack {layout} {samples}")
    _eq(P.unpack(want[None], layout)[0], s[0], f"unpack {layout} {hexbytes}")


@pytest.mark.parametrize("layout", P.LAYOUTS)
def test_round_trip_of_random_bytes(layout):
    """pack(unpack(x)) == x: every byte string is a packed frame, and unpack loses nothing."""
    rng = np.random.default_rng(11)
    for w in (4, 12, 16, 20, 1000, 1920) + ((6, 1002) if P.bits_of(layout) == 12 else ()):
        x = rng.integers(0, 256, (2, 5, P.row_bytes(layout, w)), dtype=np.uint8)
        s = P.unpack(x, layout)
        assert s.shape == (2, 5, w) and s.dtype == np.uint16 and (s >> P.bits_of(layout) == 0).all()
        _eq(P.pack(s, layout), x, f"{layout} W={w}")


@pytest.mark.parametrize("layout", P.LAYOUTS)
def test_every_value_in_every_position(layout):
    """unpack(pack(s)) == s for all 2^b values at each pixel position of a group, the other positions random."""
    b = P.bits_of(layout)
    group = 4 if b == 10 else 2
    rng = np.random.default_rng(b)
    for i in range(group):
        s = rng.integers(0, 1 << b, (1 << b, 2 * group), dtype=np.uint16)
        s[:, i] = s[:, group + i] = np.arange(1 << b)
        _eq(P.unpack(P.pack(s, layout), layout), s, f"{layout} position {i}")


def test_mipi_and_genicam_differ_and_decode_alike():
    """The same samples in the two layouts of one depth are different bytes with the same decode."""
    rng = np.random.default_rng(4)
    for b in (10, 12):
        s = rng.integers(0, 1 << b, (9, 16), dtype=np.uint16)
        m, g = P.pack(s, f"mipi{b}"), P.pack(s, f"genicam{b}")
        assert m.shape == g.shape == (9, 2 * b) and not np.array_equal(m, g)
        for pattern in R16.PATTERNS:
            _eq(P.decode(m, pattern, f"mipi{b}"), R16.decode(s, pattern, b), f"mipi{b} {pattern}")
            _eq(P.decode(g, pattern, f"genicam{b}"), R16.decode(s, pattern, b), f"genicam{b} {pattern}")


def test_format_codes():
    """16 codes at 40-55: layout-major (MIPI 10, MIPI 12, GenICam 10, GenICam 12), the pattern order of codes 12-15 within
    each; 32-39 stay unassigned, and the 16-bit codes and their uint16 set are unchanged."""
    assert [FMT[p, lay] for lay in P.LAYOUTS for p in R16.PATTERNS] == list(range(40, 56))
    assert rip.FMTS_PACKED == frozenset(range(40, 56))
    assert rip.FMTS_U16 == frozenset(range(16, 32)) and not rip.FMTS_U16 & rip.FMTS_PACKED
    assert all(rip.CHANNELS[f] == 1 for f in rip.FMTS_PACKED)
    assert not any(v in range(32, 40) for k, v in vars(rip).items() if k.startswith("FMT_"))
    assert [rip.packed_bits(FMT[p, lay]) for lay in P.LAYOUTS for p in R16.PATTERNS] == [10] * 4 + [12] * 4 + [10] * 4 + [12] * 4
    header = open(os.path.join(ROOT, "include", "rip_cuda.h")).read()
    for (pattern, layout), code in FMT.items():
        assert f"RIP_FMT_BAYER_{pattern.upper()}{SUFFIX[layout]} = {code}" in header
    assert "Packed RAW10 / RAW12 are not taken" not in header


def test_output_sizes_of_the_packed_formats():
    w, h = 684, 1023
    for fmt in FMT.values():
        assert _out_bytes(rip.OP_GAUSSIAN, fmt, w, h) == w * h * 4
        assert _out_bytes(rip.OP_GRAY, fmt, w, h) == w * h
        assert _out_bytes(rip.OP_GRAY, fmt, w, h, rip.GRAY_OUT_RGBA) == w * h * 4
        assert _out_bytes(rip.OP_EDGE, fmt, w, h) == w * h
        assert _out_bytes(rip.OP_FUSED, fmt, w, h) == w * h


def test_python_shapes_and_dtypes():
    """Context.process / submit take packed frames as (N, H, row_bytes) or (H, row_bytes) uint8 and derive W; a row_bytes
    that is not a whole number of groups, and uint16 arrays, are refused."""
    c = object.__new__(rip.Context)   # the shape handling needs no device
    wt = rip.gauss_weights(5, 1.0)
    for (pattern, layout), fmt in FMT.items():
        b = P.bits_of(layout)
        group = 5 if b == 10 else 3
        for n, h, w in ((3, 5, 8), (2, 9, 12)) + (((1, 4, 6),) if b == 12 else ()):
            rb = w * b // 8
            a, _, n2, h2, w2, shape, out, squeeze = c._shapes(np.zeros((n, h, rb), np.uint8), rip.OP_GAUSSIAN, fmt,
                                                              rip.GRAY_OUT_U8, 5, wt, None)
            assert (a.shape, n2, h2, w2, shape, out.shape, out.dtype, squeeze) == \
                ((n, h, rb), n, h, w, (n, h, w, 4), (n, h, w, 4), np.uint8, False)
            a, _, n2, h2, w2, shape, out, squeeze = c._shapes(np.zeros((h, rb), np.uint8), rip.OP_EDGE, fmt, rip.GRAY_OUT_U8,
                                                              0, None, None)
            assert (a.shape, a.nbytes, n2, h2, w2, shape, squeeze) == ((1, h, rb), h * rb, 1, h, w, (1, h, w), True)
        for rb in (group + 1, 2 * group - 1, 7 if b == 10 else 8):
            with pytest.raises(AssertionError, match=f"multiple of {group} bytes"):
                c._shapes(np.zeros((2, 9, rb), np.uint8), rip.OP_GRAY, fmt, rip.GRAY_OUT_U8, 0, None, None)
        for bad in (np.zeros((2, 9, 10), np.uint16), np.zeros((2, 9, 10), np.int8)):
            with pytest.raises(AssertionError, match="takes uint8"):
                c._shapes(bad, rip.OP_GRAY, fmt, rip.GRAY_OUT_U8, 0, None, None)


@pytest.mark.skipif(rip.device_count() > 0, reason="only meaningful on a box without a GPU")
def test_packed_bayer_fails_loudly_without_gpu():
    for fmt in FMT.values():
        with pytest.raises(rip.RipError, match="no CUDA device|no CPU fallback"):
            rip.convert_dev(16, 32, 4, 4, 1, fmt, rip.FMT_RGBA8)
        with pytest.raises(rip.RipError, match="no CUDA device|no CPU fallback"):
            rip.gray_dev(16, 32, 4, 4, 1, fmt)


def _build_dropin(tmp_path):
    exe = str(tmp_path / "bayer_packed_dropin")
    cmd = ["/usr/bin/g++", "-O2", "-std=c++17", "-ffp-contract=off", "-I", os.path.join(PKG, "host"), "-I", os.path.join(ROOT, "include"),
           "-I", "/usr/local/cuda/include", os.path.join(ROOT, "tests", "cpp", "bayer_packed_dropin.cpp"), "-o", exe, "-L", PKG,
           "-lrip_host", "-lrip_cuda", "-Wl,-rpath," + PKG, "-pthread"]
    subprocess.run(cmd, check=True)
    return exe


def test_cpp_driver_builds(tmp_path):
    exe = _build_dropin(tmp_path)
    res = subprocess.run([exe], capture_output=True, text=True)
    assert res.returncode == 2 and "usage" in res.stderr
    res = subprocess.run([exe, str(tmp_path), str(rip.FMT_BAYER_GBRG12), "8", "8", "1"], capture_output=True, text=True)
    assert res.returncode == 2 and "not a packed" in res.stderr


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


def _gray_rgba(g):
    return np.stack([g, g, g, np.full_like(g, 255)], -1)


def _convert(fmt, fr, w, order, in_off=0, out_off=0):
    n, h = fr.shape[:2]
    bpp = len(order)
    d_in = rip.DeviceBuffer(fr.nbytes + 16).upload(fr, offset=in_off)
    d_out = rip.DeviceBuffer(n * h * w * bpp + 16)
    rip.convert_dev(d_in.ptr + in_off, d_out.ptr + out_off, w, h, n, fmt, OUT_FMT[order])
    return d_out.download((n, h, w, bpp), offset=out_off)


def _gray_dev(fmt, fr, w, out_mode, in_off=0, out_off=0):
    n, h = fr.shape[:2]
    bpp = 4 if out_mode == rip.GRAY_OUT_RGBA else 1
    d_in = rip.DeviceBuffer(fr.nbytes + 16).upload(fr, offset=in_off)
    d_out = rip.DeviceBuffer(n * h * w * bpp + 16)
    rip.gray_dev(d_in.ptr + in_off, d_out.ptr + out_off, w, h, n, fmt, out_mode)
    return d_out.download((n, h, w, bpp) if bpp == 4 else (n, h, w), offset=out_off)


def _want_gray(oracle, rgb):
    return np.stack([oracle.gray(f, threads=0) for f in rgb])


def _check_decodes(oracle, pattern, layout, fr, what, in_off=0, out_off=0, orders=R16.ORDERS):
    """rip_convert in `orders` and both rip_gray outputs of packed frames `fr`, against the restatement (+ the C oracle for
    gray) and against the same samples through the unpacked code."""
    fmt, u16 = FMT[pattern, layout], _u16_fmt(pattern, layout)
    samples = P.unpack(fr, layout)
    w = samples.shape[-1]
    rgb = R16.decode(samples, pattern, P.bits_of(layout))
    for order in orders:
        got = _convert(fmt, fr, w, order, in_off, out_off)
        _eq(got, _in_order(rgb, order), f"rip_convert {pattern} {layout} {order} {fr.shape} {what}")
        _eq(got, _convert(u16, samples, w, order), f"rip_convert {pattern} {layout} {order} {fr.shape} {what} vs unpacked")
    g = _want_gray(oracle, rgb)
    got = _gray_dev(fmt, fr, w, rip.GRAY_OUT_U8, in_off, out_off)
    _eq(got, g, f"rip_gray u8 {pattern} {layout} {fr.shape} {what}")
    _eq(got, _gray_dev(u16, samples, w, rip.GRAY_OUT_U8), f"rip_gray u8 {pattern} {layout} {fr.shape} {what} vs unpacked")
    _eq(_gray_dev(fmt, fr, w, rip.GRAY_OUT_RGBA, in_off, out_off), _gray_rgba(g), f"rip_gray rgba {pattern} {layout} {what}")


# (n, h, w): W % 16 == 0 takes the word-load kernel (16, 1920, and 4K below; odd H, H = 3 and H = 4, where every row pair is a
# border pair), every other width the byte-granular kernel (4, 12, 20, 1000 = 8 * 125; 6 and 1002 at 12 bits).  A frame of
# 3 x 4 at 10 bits is 15 bytes, so every second frame of a batch starts on an odd address.
SHAPES = [(1, 3, 4), (3, 3, 4), (3, 5, 12), (2, 4, 16), (3, 7, 16), (3, 3, 16), (2, 9, 20), (2, 33, 1000), (1, 61, 1920),
          (2, 6, 32)]
SHAPES12 = [(3, 5, 6), (3, 3, 6), (2, 7, 1002)]


@pytest.mark.gpu
@pytest.mark.parametrize("pattern,layout", CODES)
def test_convert_and_gray_every_code(ctx, oracle, pattern, layout):
    for n, h, w in SHAPES + (SHAPES12 if P.bits_of(layout) == 12 else []):
        _check_decodes(oracle, pattern, layout, _noise(n, h, w, layout, 100 + h + w), f"{n}x{h}x{w}")


@pytest.mark.gpu
@pytest.mark.parametrize("layout", P.LAYOUTS)
def test_convert_and_gray_4k(ctx, oracle, layout):
    fr = _noise(1, 2160, 3840, layout, 7)
    for pattern in ("rggb", "gbrg"):
        _check_decodes(oracle, pattern, layout, fr, "4K", orders=("rgb", "bgra"))


@pytest.mark.gpu
@pytest.mark.parametrize("layout", P.LAYOUTS)
@pytest.mark.parametrize("in_off,out_off", [(1, 0), (2, 0), (3, 0), (5, 0), (0, 1), (0, 2), (0, 3), (0, 5), (3, 5), (5, 3)])
def test_unaligned_buffers(ctx, oracle, layout, in_off, out_off):
    """Input offsets 1, 2, 3 and 5 break the word alignment of every row; output offsets break the 8- and 16-byte stores.
    (3, 6, 32) is word-kernel shaped, (3, 5, 12) byte-granular either way."""
    for n, h, w in ((3, 6, 32), (3, 5, 12)):
        fr = _noise(n, h, w, layout, 7 + in_off)
        for pattern in ("bggr", "grbg"):
            _check_decodes(oracle, pattern, layout, fr, f"offsets {in_off}/{out_off}", in_off, out_off)


def _bit_frames(layout, h, w):
    """Frames that put a distinct value in every bit position of a group: sample i of the row holds one set bit (or all
    but one) that walks through the b positions, so every byte of the packing carries a lone bit somewhere."""
    b = P.bits_of(layout)
    yy, xx = np.mgrid[0:h, 0:w]
    one = (1 << ((xx + 3 * yy) % b)).astype(np.uint16)
    return np.stack([P.pack(one, layout), P.pack(((1 << b) - 1) ^ one, layout)])


@pytest.mark.gpu
@pytest.mark.parametrize("layout", P.LAYOUTS)
def test_full_scale_flat_and_bit_position_frames(ctx, oracle, layout):
    b = P.bits_of(layout)
    s = b - 8
    vals = [(1 << b) - 1, 0] + [q << s for q in range(0, 256, 5)] + [(2 * q + 1) << (s - 1) for q in range(0, 256, 17)]
    for h, w in ((9, 16), (7, 12)):
        flat = np.stack([P.pack(np.full((h, w), v, np.uint16), layout) for v in vals])
        for pattern in R16.PATTERNS:
            full = P.decode(flat[0], pattern, layout)
            assert (full == 255).all()   # full scale 1023 / 4095 gives 255
            _check_decodes(oracle, pattern, layout, flat, "flat", orders=("rgb", "bgra"))
            _check_decodes(oracle, pattern, layout, _bit_frames(layout, h, w), "bit positions")
    fmt = FMT["rggb", layout]
    got = ctx.process(flat, rip.OP_GRAY, fmt)
    _eq(got, _want_gray(oracle, P.decode(flat, "rggb", layout)), f"flat GRAY {layout}")


def _smooth(n, h, w, layout, seed):
    """Camera-like packed frames: smooth content with noise and a flat black bar (the blur's constant windows)."""
    b = P.bits_of(layout)
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    top = (1 << b) - 1
    out = []
    for _ in range(n):
        fx, fy, ph = rng.uniform(0.002, 0.03), rng.uniform(0.002, 0.03), rng.uniform(0, 6.28)
        f = 0.47 * top * (1 + 0.75 * np.sin(fx * xx + fy * yy + ph)) + rng.integers(-3 << (b - 8), 4 << (b - 8), (h, w))
        f = np.clip(f, 0, top).astype(np.uint16)
        f[: h // 8] = 0
        out.append(P.pack(f, layout))
    return np.stack(out)


@pytest.mark.gpu
@pytest.mark.parametrize("k,sigma", [(5, 1.5), (9, 2.5), (17, 6.0)])
@pytest.mark.parametrize("kernel", ["RIP_BLUR_STREAM", "RIP_BLUR_TILED"])
def test_pipeline_gaussian(ctx, oracle, opt, k, sigma, kernel):
    """Demosaic to RGBA, then the streaming or the tiled blur kernel, forced; every layout, the patterns in turn."""
    opt(kernel, 1)
    wt = rip.gauss_weights(k, sigma)
    for i, layout in enumerate(P.LAYOUTS):
        pattern = R16.PATTERNS[(i + k) % 4]
        for fr in (_smooth(2, 270, 480, layout, k), _noise(2, 121, 164, layout, k)):
            n, h = fr.shape[:2]
            w = P.unpack(fr[:1, :1], layout).shape[-1]
            got = ctx.process(fr, rip.OP_GAUSSIAN, FMT[pattern, layout], ksize=k, weights=wt)
            assert got.shape == (n, h, w, 4)
            for j in range(n):
                want = oracle.blur(P.decode(fr[j], pattern, layout, "rgba"), k, weights=wt, threads=0)
                _eq(got[j], want, f"GAUSSIAN {pattern} {layout} {k}x{k} {kernel} {h}x{w} frame {j}")


@pytest.mark.gpu
@pytest.mark.parametrize("pattern,layout", CODES)
def test_pipeline_gray_edge_and_fused(ctx, oracle, pattern, layout):
    wt = rip.gauss_weights(5, 1.0)
    shapes = [(2, 75, 76), (3, 64, 128), (2, 3, 4)] + ([(2, 1080, 1920)] if pattern == "rggb" else [])
    for n, h, w in shapes:
        fr = _noise(n, h, w, layout, 3 + h)
        fmt = FMT[pattern, layout]
        gray = ctx.process(fr, rip.OP_GRAY, fmt)
        gray_rgba = ctx.process(fr, rip.OP_GRAY, fmt, gray_out=rip.GRAY_OUT_RGBA)
        edge = ctx.process(fr, rip.OP_EDGE, fmt)
        fused = ctx.process(fr, rip.OP_FUSED, fmt, ksize=5, weights=wt)
        assert gray.shape == edge.shape == fused.shape == (n, h, w)
        for i in range(n):
            rgb = P.decode(fr[i], pattern, layout)
            g = oracle.gray(rgb, threads=0)
            _eq(gray[i], g, f"GRAY {pattern} {layout} {h}x{w} frame {i}")
            _eq(gray_rgba[i], _gray_rgba(g), f"GRAY rgba {pattern} {layout} {h}x{w} frame {i}")
            _eq(edge[i], oracle.sobel(g, threads=0), f"EDGE {pattern} {layout} {h}x{w} frame {i}")
            _eq(fused[i], oracle.fused(rgb, 5, weights=wt, threads=0), f"FUSED {pattern} {layout} {h}x{w} frame {i}")


@pytest.mark.gpu
@pytest.mark.parametrize("pattern,layout,n", [("rggb", "mipi12", 20), ("gbrg", "genicam10", 24)])
def test_pipeline_chunks_large_batches(ctx, oracle, pattern, layout, n):
    """1080p frames are 2.6 MB (10-bit) or 3.1 MB (12-bit) packed: 24 / 20 of them are more than one 48 MiB chunk, so the
    pipeline sizes its chunks from the packed frame bytes (process and submit).  Every frame is checked against the unpacked
    code on the device, the chunk edges and the last frame against the oracle."""
    fr = _smooth(n, 1080, 1920, layout, 77)
    fmt, u16 = FMT[pattern, layout], _u16_fmt(pattern, layout)
    samples = P.unpack(fr, layout)
    wt = rip.gauss_weights(5, 1.0)
    gray = ctx.process(fr, rip.OP_GRAY, fmt)
    fused = ctx.submit(fr, rip.OP_FUSED, fmt, ksize=5, weights=wt).collect()
    _eq(gray, ctx.process(samples, rip.OP_GRAY, u16), f"chunked GRAY {pattern} {layout} vs unpacked")
    _eq(fused, ctx.process(samples, rip.OP_FUSED, u16, ksize=5, weights=wt), f"chunked FUSED {pattern} {layout} vs unpacked")
    per_chunk = (48 << 20) // fr[0].nbytes
    assert per_chunk < n
    for i in sorted({0, per_chunk - 1, per_chunk, n - 1}):
        rgb = P.decode(fr[i], pattern, layout)
        _eq(gray[i], oracle.gray(rgb, threads=0), f"chunked GRAY {pattern} {layout} frame {i}")
        _eq(fused[i], oracle.fused(rgb, 5, weights=wt, threads=0), f"chunked FUSED {pattern} {layout} frame {i}")


@pytest.mark.gpu
@pytest.mark.parametrize("layout", P.LAYOUTS)
def test_submit_collect_three_in_flight(ctx, oracle, layout):
    fr = _noise(6, 270, 480, layout, 44)
    wt = rip.gauss_weights(5, 1.5)
    pattern = R16.PATTERNS[P.LAYOUTS.index(layout)]
    want = [oracle.blur(P.decode(f, pattern, layout, "rgba"), 5, weights=wt, threads=0) for f in fr]
    tickets, got = [], []
    for i in range(6):
        tickets.append(ctx.submit(fr[i], rip.OP_GAUSSIAN, FMT[pattern, layout], ksize=5, weights=wt))
        if len(tickets) == 3:
            got.append(tickets.pop(0).collect())
    got += [t.collect() for t in tickets]
    for i in range(6):
        _eq(got[i], want[i], f"submit/collect {pattern} {layout} frame {i}")


@pytest.mark.gpu
def test_rejections(ctx):
    wt = rip.gauss_weights(5, 1.0)
    raw = np.zeros(256, np.uint8)
    d_in, d_out = rip.DeviceBuffer(4096), rip.DeviceBuffer(4096)
    for (pattern, layout), fmt in FMT.items():
        name = f"BAYER_{pattern.upper()}{SUFFIX[layout]}"
        b = P.bits_of(layout)
        per = 4 if b == 10 else 2
        msg = f"{name} frames need a width that is a multiple of {per} and at least 4, and a height of at least 3"
        bad_shapes = [(3, 2), (3, 3), (8, 5), (2, 8), (1, 4), (2, 2)] + ([(3, 6), (5, 10), (4, 1002)] if b == 10 else [(3, 7)])
        for h, w in bad_shapes:
            with pytest.raises(rip.RipError, match=msg) as e:
                rip.convert_dev(d_in.ptr, d_out.ptr, w, h, 1, fmt, rip.FMT_RGBA8)
            assert ("inside a byte" in str(e.value)) == (layout.startswith("genicam"))
            with pytest.raises(rip.RipError, match=msg):
                rip.gray_dev(d_in.ptr, d_out.ptr, w, h, 1, fmt)
            for op in (rip.OP_GRAY, rip.OP_GAUSSIAN, rip.OP_EDGE, rip.OP_FUSED):
                d = ctx._desc(op, fmt, ksize=5, weights=wt)
                out = np.empty(h * w * 4, np.uint8)
                rc = rip.lib().rip_process_host(ctx.ptr, C.byref(d), raw.ctypes.data, out.ctypes.data, w, h, 1, None)
                assert rc == -1 and msg.encode() in rip.lib().rip_last_error_string()
        fr = _noise(1, 64, 64, layout, 1)
        with pytest.raises(rip.RipError, match="rc=-4.*row-band"):
            ctx.process(fr, rip.OP_FUSED, fmt, ksize=5, weights=wt, banded=True)
        with pytest.raises(rip.RipError, match="rc=-4.*row-band"):
            ctx.process(fr, rip.OP_EDGE, fmt, banded=True)
        d_fr = rip.DeviceBuffer(fr.nbytes).upload(fr)
        with pytest.raises(rip.RipError, match=f"rc=-4.*rip_sobel: RIP_FMT_{name} .*rip_gray"):
            rip.sobel_dev(d_fr.ptr, d_out.ptr, 64, 64, 1, fmt)
        with pytest.raises(rip.RipError, match=f"rc=-4.*rip_fused: RIP_FMT_{name} .*rip_gray"):
            rip.fused_dev(d_fr.ptr, d_out.ptr, 64, 64, 1, fmt, 5, wt)
        for out_fmt in (rip.FMT_GRAY8, rip.FMT_NV12, fmt):
            with pytest.raises(rip.RipError, match="rc=-4"):
                rip.convert_dev(d_fr.ptr, d_out.ptr, 64, 64, 1, fmt, out_fmt)
        with pytest.raises(AssertionError, match="takes uint8"):
            ctx.process(P.unpack(fr, layout), rip.OP_GRAY, fmt)
        with pytest.raises(AssertionError, match="bytes"):
            ctx.process(np.ascontiguousarray(fr[..., :-1]), rip.OP_GRAY, fmt)
        d_fr.free()
    # the unassigned codes between the 16-bit and the packed formats are not formats
    for bad in range(32, 40):
        with pytest.raises(rip.RipError, match="rc=-4"):
            rip.convert_dev(d_in.ptr, d_out.ptr, 8, 8, 1, bad, rip.FMT_RGBA8)
        with pytest.raises(rip.RipError):
            rip.gray_dev(d_in.ptr, d_out.ptr, 8, 8, 1, bad)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", P.LAYOUTS)
@pytest.mark.parametrize("n,h,w", [(2, 130, 256), (3, 75, 76), (3, 40, 1000), (2, 3, 16), (3, 3, 4)])
def test_decode_stays_inside_its_output_buffer(oracle, layout, n, h, w):
    """Every decode writes into the middle of a canary-filled buffer (256 KB on either side): the canaries must survive and the
    payload must equal the reference."""
    pad = 256 * 1024
    fr = _noise(n, h, w, layout, 515)
    d_in = rip.DeviceBuffer(fr.nbytes).upload(fr)

    def run(name, out_bytes, launch, want):
        buf = rip.DeviceBuffer(out_bytes + 2 * pad)
        buf.upload(np.full(out_bytes + 2 * pad, 0xA5, np.uint8))
        launch(buf.ptr + pad)
        got = buf.download((out_bytes + 2 * pad,))
        assert (got[:pad] == 0xA5).all() and (got[pad + out_bytes:] == 0xA5).all(), f"{name} {n}x{h}x{w}: wrote outside its output"
        _eq(got[pad: pad + out_bytes].reshape(want.shape), want, f"{name} {n}x{h}x{w}")
        buf.free()

    for pattern in R16.PATTERNS:
        fmt = FMT[pattern, layout]
        rgb = P.decode(fr, pattern, layout)
        for order in R16.ORDERS:
            run(f"convert {pattern} {layout} {order}", n * h * w * len(order),
                lambda p: rip.convert_dev(d_in.ptr, p, w, h, n, fmt, OUT_FMT[order]), _in_order(rgb, order))
        g = _want_gray(oracle, rgb)
        run(f"gray {pattern} {layout} u8", n * h * w, lambda p: rip.gray_dev(d_in.ptr, p, w, h, n, fmt, rip.GRAY_OUT_U8), g)
        run(f"gray {pattern} {layout} rgba", n * h * w * 4, lambda p: rip.gray_dev(d_in.ptr, p, w, h, n, fmt, rip.GRAY_OUT_RGBA),
            _gray_rgba(g))


@pytest.mark.gpu
@pytest.mark.parametrize("pattern,layout", [("rggb", "mipi10"), ("bggr", "mipi12"), ("grbg", "genicam10"), ("gbrg", "genicam12")])
def test_cpp_controller_drop_in(tmp_path, oracle, pattern, layout):
    """PerformBatch / PerformFused / SubmitFrame + CollectFrame through the C++ Controller, and its rejection of short buffers
    and of frames too narrow, too short or of a width the packing cannot hold, against bytes computed here through the
    oracle."""
    exe = _build_dropin(tmp_path)
    n, h, w = 3, 121, 164
    fr = _smooth(n, h, w, layout, 12)
    fr.tofile(str(tmp_path / "in.raw"))
    res = subprocess.run([exe, str(tmp_path), str(FMT[pattern, layout]), str(w), str(h), str(n)], capture_output=True, text=True)
    assert res.returncode == 0 and res.stdout.strip().endswith("OK"), res.stdout + res.stderr
    wt = oracle.gauss_weights(5, 1.5)
    rgb = P.decode(fr, pattern, layout)
    gray = np.stack([oracle.gray(f) for f in rgb])
    want = {"batch_GRAYSCALE": gray,
            "batch_GAUSSIAN": np.stack([oracle.blur(P.decode(f, pattern, layout, "rgba"), 5, weights=wt) for f in fr]),
            "batch_EDGE": np.stack([oracle.sobel(g) for g in gray]),
            "batch_FUSED": np.stack([oracle.fused(f, 5, weights=wt) for f in rgb]),
            "fused_frame0": oracle.fused(rgb[0], 5, weights=wt)}
    want["submit_GAUSSIAN"] = want["batch_GAUSSIAN"]
    for name, ref in want.items():
        got = np.fromfile(str(tmp_path / (name + ".raw")), np.uint8)
        _eq(got.reshape(ref.shape), ref, name)
