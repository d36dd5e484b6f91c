"""GPU parity: every CUDA path against the CPU oracle, bit-exact, through the C ABI.

Run on a B200 with `pytest -m gpu`.  Sizes are chosen so the oracle finishes in seconds; the
BASELINE-size cases use all host threads for the oracle and size-independent properties
(frame independence, band/whole-frame equality)."""
import numpy as np
import pytest

import rip_b200 as rip
from conftest import bgr_to_rgba, synth_frame

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    if rip.device_count() < 1:
        pytest.fail("GPU tests need a CUDA device: librip_cuda has no CPU fallback")
    c = rip.Context([0])
    yield c
    c.close()


def _eq(got, want, what=""):
    if not np.array_equal(got, want):
        d = np.abs(got.astype(int) - want.astype(int))
        idx = np.argwhere(d > 0)
        raise AssertionError(f"{what}: {len(idx)} of {d.size} bytes differ, max abs {d.max()}, first at {idx[0].tolist()}")


# ---------------------------------------------------------------------------------------------
def test_native_library_loaded_and_counts_launches(ctx):
    before = rip.launch_count()
    ctx.process(np.zeros((8, 8, 3), np.uint8), rip.OP_GRAY, rip.FMT_RGB8)
    assert rip.launch_count() > before
    info = rip.device_info(0)
    assert info.cc_major == 10, f"expected a Blackwell sm_100 device, got cc {info.cc_major}.{info.cc_minor}"


def test_device_selftest_of_arithmetic_shortcuts():
    checked, bad = rip.selftest(0)
    assert checked > 4 * (1 << 24) and bad == 0, (checked, bad)


# ---- gray (config 1) -------------------------------------------------------------------------
def test_gray_all_16777216_triples(ctx, oracle):
    i = np.arange(1 << 24, dtype=np.uint32)
    rgb = np.stack([i & 255, (i >> 8) & 255, i >> 16], -1).astype(np.uint8).reshape(4096, 4096, 3)
    _eq(ctx.process(rgb, rip.OP_GRAY, rip.FMT_RGB8), oracle.gray(rgb, threads=0), "gray RGB exhaustive")


def test_gray_config1_tulips_medium640(ctx, oracle, golden_images):
    bgr = golden_images["Tulips_medium640.bgr"]
    rgba = bgr_to_rgba(bgr)
    want = oracle.gray(bgr, oracle.BGR)
    # drop-in container of Controller::PerformCLImageGrayscaling: (g,g,g,255) W*H*4
    got = ctx.process(rgba, rip.OP_GRAY, rip.FMT_RGBA8, gray_out=rip.GRAY_OUT_RGBA)
    assert got.shape == (512, 640, 4)
    for c in range(3):
        _eq(got[..., c], want, "gray RGBA->RGBA")
    assert (got[..., 3] == 255).all()
    _eq(ctx.process(rgba, rip.OP_GRAY, rip.FMT_RGBA8), want, "gray RGBA->u8")
    _eq(ctx.process(np.ascontiguousarray(bgr), rip.OP_GRAY, rip.FMT_BGR8), want, "gray BGR->u8")


@pytest.mark.parametrize("fmt,cn,order", [(rip.FMT_RGB8, 3, "RGB"), (rip.FMT_BGR8, 3, "BGR"),
                                          (rip.FMT_RGBA8, 4, "RGB"), (rip.FMT_BGRA8, 4, "BGR")])
@pytest.mark.parametrize("shape", [(1, 1), (3, 5), (7, 9), (75, 75), (33, 130)])
def test_gray_formats_and_ragged_sizes(ctx, oracle, fmt, cn, order, shape):
    img = synth_frame("uniform", shape[0], shape[1], 11, cn)
    img[0, 0, :3] = 1  # r=g=b=1 -> 0: the double-rounding case
    want = oracle.gray(img, oracle.BGR if order == "BGR" else oracle.RGB)
    _eq(ctx.process(img, rip.OP_GRAY, fmt), want, f"gray {order}{cn} {shape}")
    got4 = ctx.process(img, rip.OP_GRAY, fmt, gray_out=rip.GRAY_OUT_RGBA)
    _eq(got4[..., 1], want, "gray rgba container")


def test_gray_grey_images_take_the_double_path(ctx, oracle):
    v = np.arange(256, dtype=np.uint8)
    img = np.repeat(np.tile(v, 4)[None, :, None], 3, axis=2).repeat(8, axis=0).copy()  # r=g=b
    want = oracle.gray(img)
    assert (want != img[..., 0]).sum() > 0  # 65 of the 256 greys come out v-1
    _eq(ctx.process(img, rip.OP_GRAY, rip.FMT_RGB8), want, "grey ramp")


# ---- Gaussian blur (config 2) ----------------------------------------------------------------
@pytest.mark.parametrize("sigma", [1.0, 1.5])
def test_blur_config2_artemis_large1024(ctx, oracle, golden_images, sigma):
    rgba = bgr_to_rgba(golden_images["Artemis_large1024.bgr"])
    assert rgba.shape == (1023, 683, 4)
    w = rip.gauss_weights(5, sigma)
    got = ctx.process(rgba, rip.OP_GAUSSIAN, rip.FMT_RGBA8, ksize=5, weights=w)
    want = oracle.blur(rgba, 5, weights=oracle.gauss_weights(5, sigma), threads=0)
    _eq(got, want, f"blur RGBA 5x5 sigma {sigma}")  # bit-exact, i.e. max/mean abs error 0


@pytest.mark.parametrize("k,sigma", [(1, 1.0), (3, 0.8), (7, 2.0), (17, 6.0), (31, 9.5)])
def test_blur_generic_kernel_sizes(ctx, oracle, k, sigma):
    img = synth_frame("smooth", 61, 83, 5, 4)
    w = rip.gauss_weights(k, sigma)
    _eq(ctx.process(img, rip.OP_GAUSSIAN, rip.FMT_RGBA8, ksize=k, weights=w), oracle.blur(img, k, weights=w, threads=0),
        f"blur K={k}")
    g = np.ascontiguousarray(img[..., 0])
    _eq(ctx.process(g, rip.OP_GAUSSIAN, rip.FMT_GRAY8, ksize=k, weights=w), oracle.blur(g, k, weights=w, threads=0),
        f"blur gray K={k}")


def test_blur_flat_regions_sigma15_lose_one_level(ctx, oracle):
    flat = np.full((20, 24, 4), 255, np.uint8)
    got = ctx.process(flat, rip.OP_GAUSSIAN, rip.FMT_RGBA8, ksize=5, weights=rip.gauss_weights(5, 1.5))
    assert (got == 254).all()  # what the reference CPU path does (sum of float weights < 1)
    got = ctx.process(flat, rip.OP_GAUSSIAN, rip.FMT_RGBA8, ksize=5, weights=rip.gauss_weights(5, 1.0))
    assert (got == 255).all()


def _adversarial_rgba(h, w):
    """SURVEY.md 8(d)(iii): constants, ramps, 1-px checkerboard, bright corner pixels."""
    yy, xx = np.mgrid[0:h, 0:w]
    frames = [np.full((h, w), v, np.uint8) for v in (0, 255, 1, 2, 4, 254, 77)]
    frames += [(xx * 255 // max(w - 1, 1)).astype(np.uint8), (yy * 255 // max(h - 1, 1)).astype(np.uint8),
               (((xx + yy) & 1) * 255).astype(np.uint8)]
    corners = np.zeros((h, w), np.uint8)
    corners[0, 0] = corners[0, -1] = corners[-1, 0] = corners[-1, -1] = corners[h // 2, 0] = corners[0, w // 2] = 255
    frames.append(corners)
    return [np.ascontiguousarray(np.stack([f, f[::-1], f[:, ::-1], 255 - f], -1)) for f in frames]


@pytest.mark.parametrize("k,sigma", [(5, 1.0), (5, 1.5), (9, 2.5), (17, 6.0)])
def test_blur_separable_kernel_equals_exact_kernel_and_oracle(ctx, oracle, k, sigma, opt):
    """The separable guard-band kernel (default) and the reference-order kernel (RIP_BLUR_EXACT) must agree bit for bit."""
    w = rip.gauss_weights(k, sigma)
    imgs = [synth_frame("uniform", 70, 101, 3, 4), synth_frame("smooth", 33, 64, 4, 4)] + _adversarial_rgba(37, 45)
    for i, img in enumerate(imgs):
        want = oracle.blur(img, k, weights=w, threads=0)
        opt("RIP_BLUR_EXACT", 0)
        _eq(ctx.process(img, rip.OP_GAUSSIAN, rip.FMT_RGBA8, ksize=k, weights=w), want, f"separable blur K={k} frame {i}")
        g = np.ascontiguousarray(img[..., 0])
        _eq(ctx.process(g, rip.OP_GAUSSIAN, rip.FMT_GRAY8, ksize=k, weights=w), oracle.blur(g, k, weights=w, threads=0),
            f"separable blur gray K={k} frame {i}")
        opt("RIP_BLUR_EXACT", 1)
        _eq(ctx.process(img, rip.OP_GAUSSIAN, rip.FMT_RGBA8, ksize=k, weights=w), want, f"exact blur K={k} frame {i}")
        if k == 5:   # 5x5 RGBA has two guard-band kernels: streaming (large inputs) and tiled; force each
            opt("RIP_BLUR_EXACT", 0)
            for force in ("RIP_BLUR_TILED", "RIP_BLUR_STREAM"):
                opt(force, 1)
                _eq(ctx.process(img, rip.OP_GAUSSIAN, rip.FMT_RGBA8, ksize=k, weights=w), want, f"{force} blur frame {i}")
                opt(force, 0)


@pytest.mark.parametrize("shape", [(3, 130, 250), (2, 67, 61), (1, 40, 1000), (5, 33, 64)])
def test_blur_streaming_kernel_batches_and_ragged_widths(ctx, oracle, shape, opt):
    opt("RIP_BLUR_STREAM", 1)
    n, h, wd = shape
    for sigma in (1.0, 1.5):
        w = rip.gauss_weights(5, sigma)
        imgs = np.stack([synth_frame("uniform" if i % 2 == 0 else "smooth", h, wd, 40 + i, 4) for i in range(n)])
        got = ctx.process(imgs, rip.OP_GAUSSIAN, rip.FMT_RGBA8, ksize=5, weights=w)
        for i in range(n):
            _eq(got[i], oracle.blur(imgs[i], 5, weights=w, threads=0), f"streaming blur {shape} sigma {sigma} frame {i}")


def test_blur_guard_band_statistics_and_non_separable_weights(ctx, oracle):
    """The replay must trigger (flat frames: always) yet stay rare on noise; weights that are not a symmetric
    separable kernel must take the reference-order kernel and still match."""
    h, wd = 96, 160
    d_out = rip.DeviceBuffer(h * wd * 4)
    w = rip.gauss_weights(5, 1.0)
    # "flat": a constant tile takes its results from the constant-window table, no replay at all (every real RGBA frame has such a
    # channel: alpha); "speckled": constant but for one pixel per 16 x 16 block, so no tile is constant while nearly every window
    # still is -- those pixels sit inside the guard band and are replayed
    speck = np.full((h, wd, 4), 77, np.uint8)
    speck[5::16, 7::16] = 200
    for kind, lo, hi in (("uniform", 1e-5, 2e-2), ("flat", 0.0, 0.0), ("speckled", 0.5, 1.1)):
        img = synth_frame("uniform", h, wd, 72, 4) if kind == "uniform" else np.full((h, wd, 4), 77, np.uint8) if kind == "flat" else speck
        d_in = rip.DeviceBuffer(img.nbytes).upload(img)
        rip.slow_path_stats(True)
        rip.gauss_dev(d_in.ptr, d_out.ptr, wd, h, 1, 4, 5, w)
        frac = rip.slow_path_stats(False) / (h * wd)
        assert lo <= frac <= hi, (kind, frac)
        _eq(d_out.download((h, wd, 4)), oracle.blur(img, 5, weights=w), f"blur {kind}")
    rng = np.random.default_rng(5)
    wr = rng.random((5, 5)).astype(np.float32)
    wr /= wr.sum() * np.float32(1.001)
    img = synth_frame("uniform", 40, 52, 9, 4)
    rip.slow_path_stats(True)
    _eq(ctx.process(img, rip.OP_GAUSSIAN, rip.FMT_RGBA8, ksize=5, weights=wr), oracle.blur(img, 5, weights=wr, threads=0), "random weights")
    assert rip.slow_path_stats(False) == 0   # the separable kernel did not run


@pytest.mark.parametrize("k,sigma,stream", [(5, 1.0, 0), (5, 1.5, 0), (9, 2.5, 0), (17, 6.0, 0), (5, 1.0, 1), (5, 1.5, 1)])
def test_blur_constant_channels_take_the_table(ctx, oracle, k, sigma, stream, opt):
    """Real RGBA frames: alpha is 255 throughout, sky is black, highlights are clipped.  A constant channel's fast sum sits on an
    integer -- inside the guard band for every pixel -- so its result comes from the host-evaluated constant-window table
    (tile-wide in the tiled kernel, per lane neighbourhood in the streaming kernel); the other channels are untouched."""
    opt("RIP_BLUR_STREAM" if stream else "RIP_BLUR_TILED", 1)
    h, wd = 130, 200
    img = synth_frame("uniform", h, wd, 123, 4)
    img[..., 3] = 255                      # alpha
    img[: h // 3, :, :3] = 0               # black sky
    img[h // 3: h // 2, : wd // 2, 1] = 255  # one clipped channel in a region
    img[-20:, -70:] = (13, 13, 13, 255)    # a flat patch that ends at the image corner
    w = rip.gauss_weights(k, sigma)
    _eq(ctx.process(img, rip.OP_GAUSSIAN, rip.FMT_RGBA8, ksize=k, weights=w), oracle.blur(img, k, weights=w, threads=0), f"constant channels K={k}")
    g = np.ascontiguousarray(img[..., 1])
    _eq(ctx.process(g, rip.OP_GAUSSIAN, rip.FMT_GRAY8, ksize=k, weights=w), oracle.blur(g, k, weights=w, threads=0), f"constant regions, gray K={k}")


@pytest.mark.parametrize("k,sigma", [(9, 2.5), (17, 6.0), (17, 2.0)])
def test_blur_streaming_k_alpha_255_shortcut_is_exact(ctx, oracle, k, sigma, opt):
    """The same shortcut in the streaming KxK kernel (its chains run horizontal-first): near misses must not take it."""
    opt("RIP_BLUR_STREAM", 1)
    h, wd = 90, 200
    rng = np.random.default_rng(78)
    img = rng.integers(0, 256, (h, wd, 4), dtype=np.uint8)
    img[..., 3] = 255
    img[5::23, 7::31, 3] = 254
    img[40:70, 100:180, 3] = rng.integers(253, 256, (30, 80), dtype=np.uint8)
    img[60:, :40, :3] = 255
    w = rip.gauss_weights(k, sigma)
    _eq(ctx.process(img, rip.OP_GAUSSIAN, rip.FMT_RGBA8, ksize=k, weights=w), oracle.blur(img, k, weights=w, threads=0), f"alpha shortcut K={k} sigma {sigma}")


@pytest.mark.parametrize("k,sigma", [(9, 2.5), (17, 6.0)])
def test_blur_streaming_k_constant_value_is_the_complement_of_the_first_row(ctx, oracle, k, sigma, opt):
    """Regression (found by tests/soak.py): the cached table bytes of the constant-window shortcut were keyed on a sentinel ~(first row), so a
    channel that is 0 in the segment's first row and constant 255 further down took a stale 0."""
    opt("RIP_BLUR_STREAM", 1)
    h, wd = 120, 200
    rng = np.random.default_rng(79)
    img = rng.integers(0, 256, (h, wd, 4), dtype=np.uint8)   # (alpha is noise: nothing else refreshes the cache)
    img[:10, :, :3] = 0
    img[40:100, 30:150, :3] = 255
    img[50:90, 160:, 1] = 0
    w = rip.gauss_weights(k, sigma)
    _eq(ctx.process(img, rip.OP_GAUSSIAN, rip.FMT_RGBA8, ksize=k, weights=w), oracle.blur(img, k, weights=w, threads=0), f"complement K={k}")


@pytest.mark.parametrize("sigma", [1.0, 1.5, 0.6])
def test_blur_streaming_alpha_255_shortcut_is_exact(ctx, oracle, sigma, opt):
    """The streaming kernel takes alpha from the constant-window table when the fast sum equals that of an all-255 window (proved on
    the host to identify the all-255 window).  Near misses -- 254 specks, 255 runs shorter than the window, image borders -- must not."""
    opt("RIP_BLUR_STREAM", 1)
    h, wd = 97, 246
    rng = np.random.default_rng(77)
    img = rng.integers(0, 256, (h, wd, 4), dtype=np.uint8)
    img[..., 3] = 255
    img[3::7, 5::11, 3] = 254                       # specks one level below
    img[40:60, 100:180, 3] = rng.integers(253, 256, (20, 80), dtype=np.uint8)   # a region that hovers around 255
    img[70:, :30, :3] = 255                         # clipped colour channels next to the border
    w = rip.gauss_weights(5, sigma)
    _eq(ctx.process(img, rip.OP_GAUSSIAN, rip.FMT_RGBA8, ksize=5, weights=w), oracle.blur(img, 5, weights=w, threads=0), f"alpha shortcut sigma {sigma}")


@pytest.mark.parametrize("k,sigma", [(9, 2.5), (17, 6.0), (17, 3.0)])
@pytest.mark.parametrize("shape", [(2, 150, 250), (1, 67, 61), (3, 40, 33), (1, 300, 1000)])
def test_blur_streaming_k_kernel(ctx, oracle, k, sigma, shape, opt):
    """9x9 / 17x17 RGBA through the accumulate-form streaming kernel (forced on small inputs): noise, smooth content, real-frame
    content (alpha 255, black sky, a clipped channel, a flat patch at the corner), ragged widths, batches."""
    opt("RIP_BLUR_STREAM", 1)
    n, h, wd = shape
    w = rip.gauss_weights(k, sigma)
    imgs = np.stack([synth_frame("uniform" if i % 2 == 0 else "smooth", h, wd, 90 + i, 4) for i in range(n)])
    imgs[-1, ..., 3] = 255
    imgs[-1, : h // 3, :, :3] = 0
    imgs[-1, h // 3: h // 2, : wd // 2, 1] = 255
    imgs[-1, -20:, -25:] = (13, 13, 13, 255)
    got = ctx.process(imgs, rip.OP_GAUSSIAN, rip.FMT_RGBA8, ksize=k, weights=w)
    for i in range(n):
        _eq(got[i], oracle.blur(imgs[i], k, weights=w, threads=0), f"streaming {k}x{k} blur {shape} frame {i}")


def test_blur_streaming_k_kernel_1080p_default(ctx, oracle):
    """The reference's default blur (17x17, sigma 6) on 1080p frames takes the streaming kernel by size: several row segments per band."""
    rng = np.random.default_rng(17)
    imgs = rng.integers(0, 256, (3, 1080, 1920, 4), dtype=np.uint8)   # 6.2 Mpx: above the streaming kernel's threshold for 17x17
    imgs[1:, ..., 3] = 255
    imgs[1, 200:500, 300:900, :3] = 255
    w = rip.gauss_weights(17, 6.0)
    got = ctx.process(imgs, rip.OP_GAUSSIAN, rip.FMT_RGBA8, ksize=17, weights=w)
    for i in range(3):
        _eq(got[i], oracle.blur(imgs[i], 17, weights=w, threads=0), f"17x17 1080p frame {i}")


@pytest.mark.parametrize("k,sigma,stream", [(5, 1.0, 0), (5, 1.0, 1), (5, 1.5, 1), (9, 2.5, 1), (17, 6.0, 0), (17, 6.0, 1)])
def test_blur_black_sky_with_stars(ctx, oracle, k, sigma, stream, opt):
    """The reference's Artemis_* images: black sky that is not quite constant (a few dim pixels, a few stars), alpha = 255.  A channel whose
    fast value is 0 needs no replay (its true sum is >= 0 and below 1) -- but sums just below 1, 2, ... still do."""
    opt("RIP_BLUR_STREAM" if stream else "RIP_BLUR_TILED", 1)
    h, wd = 150, 260
    rng = np.random.default_rng(404)
    img = np.zeros((h, wd, 4), np.uint8)
    img[..., 3] = 255
    dim = rng.random((h, wd)) < 0.02
    img[dim, :3] = rng.integers(1, 4, (int(dim.sum()), 3), dtype=np.uint8)
    stars = rng.random((h, wd)) < 0.002
    img[stars, :3] = rng.integers(100, 256, (int(stars.sum()), 3), dtype=np.uint8)
    img[100:, 180:, :3] = rng.integers(0, 256, (50, 80, 3), dtype=np.uint8)   # the lit limb
    img[60:90, 40:120, 2] = 1                                                 # a faint flat glow: blurred sums sit on / just below 1
    w = rip.gauss_weights(k, sigma)
    _eq(ctx.process(img, rip.OP_GAUSSIAN, rip.FMT_RGBA8, ksize=k, weights=w), oracle.blur(img, k, weights=w, threads=0), f"black sky K={k} stream={stream}")
    g = np.ascontiguousarray(img[..., 2])
    _eq(ctx.process(g, rip.OP_GAUSSIAN, rip.FMT_GRAY8, ksize=k, weights=w), oracle.blur(g, k, weights=w, threads=0), f"black sky, gray K={k}")


@pytest.mark.parametrize("shape", [(2, 131, 248), (1, 75, 76), (3, 40, 1000)])
def test_device_ops_stay_inside_their_output_buffers(oracle, shape, opt):
    """compute-sanitizer is closed on this GPU pool, so the bounds check is our own: every device-API operation writes into the middle of
    a canary-filled buffer (256 KB on either side) -- the canaries must
    survive and the payload must equal the oracle's.  Covers the byte-granular patch stores of the deferred replays (streaming KxK
    kernel), the predicated stores of partial bands and the halo lanes of every streaming kernel."""
    n, h, wd = shape
    rng = np.random.default_rng(515)
    pad = 256 * 1024
    rgba = rng.integers(0, 256, (n, h, wd, 4), dtype=np.uint8)
    rgba[-1, ..., 3] = 255
    rgba[-1, : h // 2, : wd // 2, :3] = 0
    rgba[0, h // 3:, wd // 3:, :3] = 255
    rgb = np.ascontiguousarray(rgba[..., :3])
    d_rgba = rip.DeviceBuffer(rgba.nbytes).upload(rgba)
    d_rgb = rip.DeviceBuffer(rgb.nbytes).upload(rgb)

    def run(name, out_bytes, launch, want):
        buf = rip.DeviceBuffer(out_bytes + 2 * pad)
        buf.upload(np.full(out_bytes + 2 * pad, 0xA5, np.uint8))
        launch(buf.ptr + pad)
        got = buf.download((out_bytes + 2 * pad,))
        assert (got[:pad] == 0xA5).all() and (got[pad + out_bytes:] == 0xA5).all(), f"{name} {shape}: wrote outside its output"
        _eq(got[pad: pad + out_bytes].reshape(want.shape), want, f"{name} {shape}")
        buf.free()

    for k, sigma in ((5, 1.0), (9, 2.5), (17, 6.0)):
        w = rip.gauss_weights(k, sigma)
        want = np.stack([oracle.blur(rgba[i], k, weights=w, threads=0) for i in range(n)])
        for force in ("RIP_BLUR_STREAM", "RIP_BLUR_TILED"):
            opt(force, 1)
            run(f"gauss {k}x{k} {force}", rgba.nbytes, lambda p: rip.gauss_dev(d_rgba.ptr, p, wd, h, n, 4, k, w), want)
            opt(force, 0)
    w5 = rip.gauss_weights(5, 1.0)
    gray = np.stack([oracle.gray(rgb[i], threads=0) for i in range(n)])
    run("gray", n * h * wd, lambda p: rip.gray_dev(d_rgb.ptr, p, wd, h, n, rip.FMT_RGB8, rip.GRAY_OUT_U8), gray)
    run("sobel", n * h * wd, lambda p: rip.sobel_dev(d_rgb.ptr, p, wd, h, n, rip.FMT_RGB8), np.stack([oracle.sobel(gray[i]) for i in range(n)]))
    run("fused", n * h * wd, lambda p: rip.fused_dev(d_rgb.ptr, p, wd, h, n, rip.FMT_RGB8, 5, w5),
        np.stack([oracle.fused(rgb[i], 5, weights=w5, threads=0) for i in range(n)]))


def test_blur_rejects_bad_arguments(ctx):
    img = np.zeros((8, 8, 4), np.uint8)
    with pytest.raises(rip.RipError):
        ctx.process(img, rip.OP_GAUSSIAN, rip.FMT_RGBA8, ksize=4, weights=np.ones((4, 4), np.float32))
    with pytest.raises(rip.RipError):
        ctx.process(img, rip.OP_GAUSSIAN, rip.FMT_RGBA8, ksize=5, weights=None)


# ---- Sobel (config 3) ------------------------------------------------------------------------
def test_sobel_gray_input_matches_opencv_goldens(ctx, golden_cv2_sobel, golden_images):
    for k, v in golden_cv2_sobel.items():
        if k.startswith("syn.") and k.endswith(".in"):
            if min(v.shape) < 2:
                continue
            _eq(ctx.process(v, rip.OP_EDGE, rip.FMT_GRAY8), golden_cv2_sobel[k[:-3] + ".out"], k)
        elif not k.startswith("syn."):
            _eq(ctx.process(golden_images[k + ".imread_gray"], rip.OP_EDGE, rip.FMT_GRAY8), v, k)


@pytest.mark.parametrize("shape", [(2, 4), (2, 8), (5, 12), (37, 120), (37, 124), (64, 128), (33, 244), (75, 75), (19, 241),
                                   (2, 16), (31, 240), (17, 256), (40, 496)])
@pytest.mark.parametrize("fmt,cn,npx", [(rip.FMT_RGB8, 3, 8), (rip.FMT_RGBA8, 4, 8), (rip.FMT_BGR8, 3, 8), (rip.FMT_RGB8, 3, 4), (rip.FMT_RGBA8, 4, 4)])
def test_sobel_colour_input(ctx, oracle, shape, fmt, cn, npx, opt):
    opt("RIP_FUSED_NPX", npx)  # pixels per lane of the fused kernel (8 where the width allows it)
    img = synth_frame("uniform", shape[0], shape[1], 21, cn)
    g = oracle.gray(img, oracle.BGR if fmt == rip.FMT_BGR8 else oracle.RGB)
    _eq(ctx.process(img, rip.OP_EDGE, fmt), oracle.sobel(g), f"sobel colour {shape} cn={cn}")


@pytest.mark.parametrize("shape", [(2, 8), (5, 12), (37, 120), (64, 128), (33, 244), (75, 75), (40, 496), (70, 720)])
@pytest.mark.parametrize("npx", [8, 4])
def test_gray_and_nv12_input_edge_and_fused(ctx, oracle, shape, npx, opt):
    """GRAY8 frames, and NV12 frames whose luma plane is the image (SURVEY.md 8f-3): Sobel and blur->Sobel on the
    given gray, through the fused kernel where the shape allows it and the staged kernels elsewhere."""
    opt("RIP_FUSED_NPX", npx)
    h, w = shape
    n = 3
    rng = np.random.default_rng(77)
    gray = rng.integers(0, 256, (n, h, w), dtype=np.uint8)
    wts = rip.gauss_weights(5, 1.0)
    want_edge = np.stack([oracle.sobel(g) for g in gray])
    want_fused = np.stack([oracle.sobel(oracle.blur(g, 5, weights=wts, threads=0)) for g in gray])
    _eq(ctx.process(gray, rip.OP_EDGE, rip.FMT_GRAY8), want_edge, f"sobel GRAY8 {shape}")
    _eq(ctx.process(gray, rip.OP_FUSED, rip.FMT_GRAY8, ksize=5, weights=wts), want_fused, f"fused GRAY8 {shape}")
    if h % 2 == 0:
        nv12 = np.concatenate([gray, rng.integers(0, 256, (n, h // 2, w), dtype=np.uint8)], axis=1)   # chroma: noise, never read
        _eq(ctx.process(nv12, rip.OP_EDGE, rip.FMT_NV12), want_edge, f"sobel NV12 {shape}")
        _eq(ctx.process(nv12, rip.OP_FUSED, rip.FMT_NV12, ksize=5, weights=wts), want_fused, f"fused NV12 {shape}")
        with pytest.raises(rip.RipError):
            ctx.process(nv12, rip.OP_GRAY, rip.FMT_NV12)


def test_sobel_config3_1080p_batch(ctx, oracle):
    n = 8  # batch 64 in the bench; 8 distinct frames here, frame independence checked below
    frames = np.stack([synth_frame("uniform", 1080, 1920, 0xB200 + 3000 + i) for i in range(n)])
    got = ctx.process(frames, rip.OP_EDGE, rip.FMT_RGB8)
    for i in range(n):
        _eq(got[i], oracle.sobel(oracle.gray(frames[i], threads=0), threads=0), f"sobel 1080p frame {i}")
    rep = np.concatenate([frames[:2]] * 8)  # 16 frames, only 2 distinct
    out = ctx.process(rep, rip.OP_EDGE, rip.FMT_RGB8)
    for i in range(16):
        _eq(out[i], got[i % 2], "frame independence")


# ---- fused gray -> blur -> Sobel (configs 4, 5) ------------------------------------------------
# widths that are multiples of 8 run 8 pixels per lane, other multiples of 4 run 4 (RIP_FUSED_NPX=4 forces 4)
FUSED_SHAPES = [(2, 4), (3, 8), (7, 12), (16, 120), (40, 124), (9, 128), (70, 244), (130, 364), (300, 480), (64, 1920),
                (2, 16), (5, 16), (9, 32), (41, 240), (33, 256), (64, 496), (23, 272), (300, 16)]


@pytest.mark.parametrize("shape", FUSED_SHAPES)
@pytest.mark.parametrize("kind,npx", [("uniform", 8), ("smooth", 8), ("uniform", 4)])
def test_fused_single_kernel_path(ctx, oracle, shape, kind, npx, opt):
    opt("RIP_FUSED_NPX", npx)
    img = synth_frame(kind, shape[0], shape[1], 31)
    w = rip.gauss_weights(5, 1.0)
    _eq(ctx.process(img, rip.OP_FUSED, rip.FMT_RGB8, ksize=5, weights=w), oracle.fused(img, 5, weights=w, threads=0),
        f"fused {kind} {shape}")


@pytest.mark.parametrize("fmt,cn,order", [(rip.FMT_RGBA8, 4, "RGB"), (rip.FMT_BGR8, 3, "BGR"), (rip.FMT_BGRA8, 4, "BGR")])
@pytest.mark.parametrize("sigma,npx", [(1.0, 8), (1.5, 8), (1.5, 4)])
def test_fused_formats_and_sigmas(ctx, oracle, fmt, cn, order, sigma, npx, opt):
    opt("RIP_FUSED_NPX", npx)
    img = synth_frame("smooth", 97, 248, 41, cn)
    w = rip.gauss_weights(5, sigma)
    want = oracle.fused(img, 5, weights=w, order=oracle.BGR if order == "BGR" else oracle.RGB)
    _eq(ctx.process(img, rip.OP_FUSED, fmt, ksize=5, weights=w), want, f"fused {order}{cn} sigma {sigma}")


@pytest.mark.parametrize("shape", [(1, 1), (1, 9), (9, 1), (5, 5), (75, 75), (33, 241), (40, 683), (2, 2), (17, 33), (16, 32), (49, 97)])
def test_fused_odd_shapes_tile_kernel(ctx, oracle, shape):
    """Shapes the streaming kernel rejects run as one any-shape tile kernel (rip_fused_tile.cu); the streaming kernel takes
    the others, also in one launch."""
    img = synth_frame("uniform", shape[0], shape[1], 51)
    w = rip.gauss_weights(5, 1.0)
    before = rip.launch_count()
    _eq(ctx.process(img, rip.OP_FUSED, rip.FMT_RGB8, ksize=5, weights=w), oracle.fused(img, 5, weights=w), f"fused odd shape {shape}")
    assert rip.launch_count() - before == 1


def test_fused_reference_image_sizes_run_one_kernel(ctx, oracle, golden_images):
    """The reference's own JPEGs (75, 160, 240, 640, 683 wide -- /root/reference/images, decoded pixels in tests/golden):
    gray -> 5x5 -> Sobel is ONE launch on every one of them, whatever the width."""
    w = rip.gauss_weights(5, 1.0)
    for name, bgr in golden_images.items():
        if not name.endswith(".bgr"):
            continue
        before = rip.launch_count()
        got = ctx.process(np.ascontiguousarray(bgr), rip.OP_FUSED, rip.FMT_BGR8, ksize=5, weights=w)
        assert rip.launch_count() - before == 1, name
        _eq(got, oracle.fused(np.ascontiguousarray(bgr[..., ::-1]), 5, weights=w, threads=0), f"fused {name} {bgr.shape}")


@pytest.mark.parametrize("fmt,cn", [(rip.FMT_RGB8, 3), (rip.FMT_BGR8, 3), (rip.FMT_RGBA8, 4), (rip.FMT_BGRA8, 4), (rip.FMT_GRAY8, 1)])
def test_fused_tile_kernel_formats_batches_bands(ctx, oracle, fmt, cn, opt):
    """The tile kernel forced on a shape the streaming kernel would take: every format, a batch, row bands."""
    opt("RIP_FUSED_GENERIC", 1)
    h, wd, n = 61, 136, 3
    w = rip.gauss_weights(5, 1.5)
    rgb = [synth_frame("uniform" if i else "smooth", h, wd, 400 + i) for i in range(n)]
    if cn == 1:
        frames = np.stack([oracle.gray(f) for f in rgb])
        want = [oracle.sobel(oracle.blur(g, 5, weights=w)) for g in frames]
    else:
        order = slice(None, None, -1) if fmt in (rip.FMT_BGR8, rip.FMT_BGRA8) else slice(None)
        frames = np.stack([np.ascontiguousarray(f[..., order]) for f in rgb])
        if cn == 4:
            frames = np.ascontiguousarray(np.concatenate([frames, np.full(frames.shape[:3] + (1,), 200, np.uint8)], -1))
        want = [oracle.fused(f, 5, weights=w) for f in rgb]
    got = ctx.process(frames, rip.OP_FUSED, fmt, ksize=5, weights=w)
    for i in range(n):
        _eq(got[i], want[i], f"tile kernel fmt {fmt} frame {i}")
    # row bands of frame 0 through the device API
    d_out = rip.DeviceBuffer(h * wd)
    out = np.empty((h, wd), np.uint8)
    for nb in (2, 5):
        for i in range(nb):
            o0, o1 = h * i // nb, h * (i + 1) // nb
            i0, i1 = max(0, o0 - 3), min(h, o1 + 3)
            d_in = rip.DeviceBuffer((i1 - i0) * wd * cn).upload(frames[0][i0:i1])
            rip.fused_dev(d_in.ptr, d_out.ptr, wd, h, 1, fmt, 5, w, in_row0=i0, in_rows=i1 - i0, out_row0=o0, out_rows=o1 - o0)
            out[o0:o1] = d_out.download((o1 - o0, wd))
        _eq(out, want[0], f"tile kernel, {nb} row bands")


@pytest.mark.parametrize("k,sigma", [(1, 1.0), (3, 0.8), (7, 2.0), (17, 6.0), (31, 9.5)])
def test_fused_other_kernel_sizes(ctx, oracle, k, sigma):
    """Any odd K (17x17 sigma 6 is the reference's default, ProgramHandler.hpp:9): still one launch."""
    img = synth_frame("smooth", 90, 160, 61)
    w = rip.gauss_weights(k, sigma)
    before = rip.launch_count()
    _eq(ctx.process(img, rip.OP_FUSED, rip.FMT_RGB8, ksize=k, weights=w), oracle.fused(img, k, weights=w, threads=0), f"fused K={k}")
    assert rip.launch_count() - before == 1


def _adversarial(h, w):
    yy, xx = np.mgrid[0:h, 0:w]
    frames = {"zeros": np.zeros((h, w), np.uint8), "ones255": np.full((h, w), 255, np.uint8)}
    for v in (1, 2, 4, 127, 254):
        frames[f"flat{v}"] = np.full((h, w), v, np.uint8)
    frames["hramp"] = (xx % 256).astype(np.uint8)
    frames["vramp"] = (yy % 256).astype(np.uint8)
    frames["checker"] = (((xx + yy) & 1) * 255).astype(np.uint8)
    c = np.zeros((h, w), np.uint8)
    c[0, 0] = c[0, -1] = c[-1, 0] = c[-1, -1] = c[h // 2, 0] = c[0, w // 2] = 255
    frames["corners"] = c
    return {k: np.repeat(v[..., None], 3, axis=2).copy() for k, v in frames.items()}


@pytest.mark.parametrize("sigma", [1.0, 1.5])
def test_fused_adversarial_frames(ctx, oracle, sigma):
    w = rip.gauss_weights(5, sigma)
    for name, img in _adversarial(67, 252).items():
        _eq(ctx.process(img, rip.OP_FUSED, rip.FMT_RGB8, ksize=5, weights=w), oracle.fused(img, 5, weights=w), f"fused {name}")
    # colour ramps exercise gray values off the grey diagonal
    yy, xx = np.mgrid[0:67, 0:252]
    img = np.stack([(xx * 3) % 256, (yy * 5 + xx) % 256, (xx + 2 * yy) % 256], -1).astype(np.uint8)
    _eq(ctx.process(img, rip.OP_FUSED, rip.FMT_RGB8, ksize=5, weights=w), oracle.fused(img, 5, weights=w), "fused colour ramps")


def test_fused_8_and_4_pixel_kernels_agree(oracle, opt):
    """The 4-pixels-per-lane kernel (fallback for widths that are not multiples of 8) must match on an 8-capable shape too."""
    h, wd = 120, 496
    img = synth_frame("uniform", h, wd, 77)
    w = rip.gauss_weights(5, 1.0)
    want = oracle.fused(img, 5, weights=w, threads=0)
    d_in = rip.DeviceBuffer(img.nbytes).upload(img)
    d_out = rip.DeviceBuffer(h * wd)
    outs = []
    for npx in (8, 4):
        opt("RIP_FUSED_NPX", npx)
        rip.lib().rip_memset_device_async(0, d_out.ptr, 0, h * wd, None)
        rip.fused_dev(d_in.ptr, d_out.ptr, wd, h, 1, rip.FMT_RGB8, 5, w)
        outs.append(d_out.download((h, wd)))
    _eq(outs[0], want, "8 pixels per lane")
    _eq(outs[1], want, "4 pixels per lane")


@pytest.mark.parametrize("sigma", [1.0, 1.5])
def test_fused_flat_regions_are_exact(ctx, oracle, sigma):
    """Letterbox bars / clipped highlights: every pixel of a constant region lies inside the guard band and is
    replayed (sigma 1.5: 255 blurs to 254); results must be exact there and where a flat region meets texture."""
    w = rip.gauss_weights(5, sigma)
    h, wd = 96, 1024
    rng = np.random.default_rng(9)
    img = rng.integers(0, 256, (h, wd, 3), dtype=np.uint8)
    img[:30] = 0                      # black bar
    img[30:52] = 255                  # clipped white
    img[52:70, :600] = (200, 200, 200)  # a grey slab next to noise (every r=g=b triple is a multiple of 1000)
    img[70:, 300:] = (13, 200, 77)
    _eq(ctx.process(img, rip.OP_FUSED, rip.FMT_RGB8, ksize=5, weights=w), oracle.fused(img, 5, weights=w, threads=0), f"flat regions sigma {sigma}")
    g = np.ascontiguousarray(img[..., 1])
    _eq(ctx.process(g, rip.OP_FUSED, rip.FMT_GRAY8, ksize=5, weights=w), oracle.sobel(oracle.blur(g, 5, weights=w, threads=0)), "flat regions, gray input")


@pytest.mark.parametrize("sigma", [1.0, 1.5])
@pytest.mark.parametrize("npx", [8, 4])
def test_fused_plateaus_of_real_images(ctx, oracle, golden_images, sigma, npx, opt):
    """Decoded JPEGs (the reference's own images): dark plateaus a few pixels wide, where several pixels of a lane sit inside the guard
    band with constant 5x5 windows while the lane's neighbourhood as a whole is not constant -- the per-pixel constant-window pass of the
    cold path.  Also synthetic patches of every small size next to each other, and patches that differ by one level."""
    opt("RIP_FUSED_NPX", npx)
    w = rip.gauss_weights(5, sigma)
    for name in ("Artemis_large1024", "Tulips_medium640"):
        bgr = golden_images[name + ".bgr"]
        rgb = np.ascontiguousarray(bgr[:, : bgr.shape[1] // 8 * 8, ::-1])
        _eq(ctx.process(rgb, rip.OP_FUSED, rip.FMT_RGB8, ksize=5, weights=w), oracle.fused(rgb, 5, weights=w, threads=0), f"{name} sigma {sigma} npx {npx}")
    rng = np.random.default_rng(606)
    h, wd = 160, 512
    img = rng.integers(0, 256, (h, wd, 3), dtype=np.uint8)
    for i in range(60):   # plateaus of 3..14 pixels, grey (r = g = b: the gray stage's own cold path too) and coloured
        y, x, sy, sx = rng.integers(0, h - 16), rng.integers(0, wd - 16), rng.integers(3, 15), rng.integers(3, 15)
        v = int(rng.integers(1, 256))
        img[y: y + sy, x: x + sx] = (v, v, v) if i % 2 else tuple(int(t) for t in rng.integers(0, 256, 3))
    img[100:130, 200:300] = 7
    img[110:120, 230:260] = 8             # one level up inside a plateau
    gray_in = np.ascontiguousarray(img[..., 0])
    _eq(ctx.process(img, rip.OP_FUSED, rip.FMT_RGB8, ksize=5, weights=w), oracle.fused(img, 5, weights=w, threads=0), f"patches sigma {sigma} npx {npx}")
    _eq(ctx.process(gray_in, rip.OP_FUSED, rip.FMT_GRAY8, ksize=5, weights=w), oracle.sobel(oracle.blur(gray_in, 5, weights=w, threads=0)), "patches, gray input")


def test_fused_guard_band_statistics():
    """The exact replay must actually trigger (flat frames: always) yet stay rare on noise."""
    w = rip.gauss_weights(5, 1.0)
    h, wd = 256, 480
    d_out = rip.DeviceBuffer(h * wd)
    for kind, lo, hi in (("uniform", 1e-5, 5e-3), ("flat", 0.5, 1.5)):
        img = synth_frame("uniform", h, wd, 71) if kind == "uniform" else np.full((h, wd, 3), 77, np.uint8)
        d_in = rip.DeviceBuffer(img.nbytes).upload(img)
        rip.slow_path_stats(True)
        rip.fused_dev(d_in.ptr, d_out.ptr, wd, h, 1, rip.FMT_RGB8, 5, w)
        frac = rip.slow_path_stats(False) / (h * wd)
        assert lo <= frac <= hi, (kind, frac)


@pytest.mark.parametrize("wd,npx", [(364, 4), (368, 8), (368, 4)])
def test_fused_row_bands_equal_whole_frame(ctx, oracle, wd, npx, opt):
    opt("RIP_FUSED_NPX", npx)
    h = 200
    img = synth_frame("uniform", h, wd, 81)
    w = rip.gauss_weights(5, 1.0)
    whole = oracle.fused(img, 5, weights=w, threads=0)
    d_out = rip.DeviceBuffer(h * wd)
    for nb in (2, 3, 8):
        out = np.empty((h, wd), np.uint8)
        for i in range(nb):
            o0, o1 = h * i // nb, h * (i + 1) // nb
            i0, i1 = max(0, o0 - 3), min(h, o1 + 3)
            d_in = rip.DeviceBuffer((i1 - i0) * wd * 3).upload(img[i0:i1])
            rip.fused_dev(d_in.ptr, d_out.ptr, wd, h, 1, rip.FMT_RGB8, 5, w, in_row0=i0, in_rows=i1 - i0, out_row0=o0, out_rows=o1 - o0)
            out[o0:o1] = d_out.download((o1 - o0, wd))
        _eq(out, whole, f"{nb} row bands")
    # a band that does not cover its halo must be rejected, not silently clamped
    d_in = rip.DeviceBuffer(50 * wd * 3)
    with pytest.raises(rip.RipError, match="does not cover"):
        rip.fused_dev(d_in.ptr, d_out.ptr, wd, h, 1, rip.FMT_RGB8, 5, w, in_row0=50, in_rows=50, out_row0=50, out_rows=50)
    # banded host pipeline (one band per device of the context; 1 device -> 1 band)
    _eq(ctx.process(img, rip.OP_FUSED, rip.FMT_RGB8, ksize=5, weights=w, banded=True), whole, "process_host_banded")


def test_fused_config4_4k_frames(ctx, oracle):
    w = rip.gauss_weights(5, 1.0)
    distinct = [synth_frame("uniform", 2160, 3840, 0xB200 + 4000), synth_frame("smooth", 2160, 3840, 0xB200 + 4001)]
    want = [oracle.fused(f, 5, weights=w, threads=0) for f in distinct]
    frames = np.stack([distinct[i % 2] for i in range(6)])
    got = ctx.process(frames, rip.OP_FUSED, rip.FMT_RGB8, ksize=5, weights=w)
    for i in range(6):
        _eq(got[i], want[i % 2], f"fused 4K frame {i}")


def test_fused_config5_8k_row_bands(oracle):
    """8K frame as 8 row bands with 3-row halos through the device API (what 8 GPUs would each run)."""
    h, wd = 4320, 7680
    img = synth_frame("uniform", h, wd, 0xB200 + 5000)
    w = rip.gauss_weights(5, 1.0)
    want = oracle.fused(img, 5, weights=w, threads=0)
    out = np.empty((h, wd), np.uint8)
    nb = 8
    d_out = rip.DeviceBuffer((h // nb + 1) * wd)
    for i in range(nb):
        o0, o1 = h * i // nb, h * (i + 1) // nb
        i0, i1 = max(0, o0 - 3), min(h, o1 + 3)
        d_in = rip.DeviceBuffer((i1 - i0) * wd * 3).upload(img[i0:i1])
        rip.fused_dev(d_in.ptr, d_out.ptr, wd, h, 1, rip.FMT_RGB8, 5, w, in_row0=i0, in_rows=i1 - i0, out_row0=o0, out_rows=o1 - o0)
        out[o0:o1] = d_out.download((o1 - o0, wd))
        d_in.free()
    _eq(out, want, "8K in 8 bands")


def test_fused_non_separable_weights_fall_back_to_exact(ctx, oracle):
    rng = np.random.default_rng(5)
    w = rng.random((5, 5)).astype(np.float32)
    w /= w.sum() * 1.001
    img = synth_frame("uniform", 50, 120, 91)
    _eq(ctx.process(img, rip.OP_FUSED, rip.FMT_RGB8, ksize=5, weights=w), oracle.fused(img, 5, weights=w), "fused arbitrary weights")


# ---- host pipeline plumbing --------------------------------------------------------------------
def test_process_host_pinned_chunked_and_profiled(ctx, oracle):
    n, h, wd = 40, 540, 960  # 62 MB of input: more than one 48 MiB chunk
    pin = rip.PinnedBuffer(n * h * wd * 3)
    frames = pin.array.reshape(n, h, wd, 3)
    base = synth_frame("uniform", h, wd, 101)
    for i in range(n):
        frames[i] = np.roll(base, i, axis=1)
    w = rip.gauss_weights(5, 1.0)
    got, prof = ctx.process(frames, rip.OP_FUSED, rip.FMT_RGB8, ksize=5, weights=w, prof=True)
    for i in (0, 1, 17, 39):
        _eq(got[i], oracle.fused(np.ascontiguousarray(frames[i]), 5, weights=w, threads=0), f"chunked frame {i}")
    assert prof[0] == 0 and prof[1] <= prof[3] <= prof[5] and prof[5] > 0 and prof[2] == prof[1] and prof[4] == prof[3]
    pin.free()


def test_context_handles_mirror_the_opencl_objects(ctx):
    import ctypes as C
    L = rip.lib()
    mod, ker, op = C.c_void_p(), C.c_void_p(), C.c_int(-1)
    for variant, name, want in (("grayscale_base.cl", "grayscale", rip.OP_GRAY), ("gaussian_base.cl", "gaussian_blur", rip.OP_GAUSSIAN),
                                ("edge_base.cl", "sobel_edge_detection", rip.OP_EDGE), ("fused", "fused", rip.OP_FUSED)):
        rip.check(L.rip_module_load(ctx.ptr, variant.encode(), C.byref(mod)))
        rip.check(L.rip_kernel_get(mod, name.encode(), C.byref(ker)))
        rip.check(L.rip_kernel_op(ker, C.byref(op)))
        assert op.value == want
        L.rip_kernel_release(ker)
        L.rip_module_release(mod)
    rip.check(L.rip_module_load(ctx.ptr, b"grayscale_base.cl", C.byref(mod)))
    assert L.rip_kernel_get(mod, b"gaussian_blur", C.byref(ker)) != 0  # wrong entry point for the module
    assert L.rip_module_load(ctx.ptr, b"nonsense.cl", C.byref(ker)) != 0
    L.rip_module_release(mod)
