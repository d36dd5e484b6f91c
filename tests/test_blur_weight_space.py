"""The Gaussian and fused kernels across the weight space, bit for bit against the C oracle.

Every fast blur path evaluates a separable sum S~ and trusts floor(S~) outside a guard band that the host proves per weight
set (plan_sep_blur in rip_blur_sep.cu, plan_weights_band in rip_fused.cu); inside the band a pixel is replayed in the
reference's order (or takes the constant-window table, the alpha-255 proof, or the "fast value 0" rule).  Which kernel runs
depends on the weights:

* plan_sep_blur / plan_weights_band accept non-negative weights whose band is <= 0.05 (not only Gaussians);
* the streaming blur kernels (5x5, 9x9, 17x17 RGBA) and the 5x5 fused kernel also need every weight to be 0 or >= 2^-70,
  otherwise the tiled kernel (blur_sep_kernel) or fused_tile_kernel runs;
* weights that fail the band test take the reference-order kernels (blur_exact_kernel, fused_tile_kernel).

At the sigmas of everyday use hardly any sum lands near an integer, so a replay that is subtly wrong passes.  The weight
sets here are the ones that load the replay: the reference generator near the identity (sigma 0.2 .. 0.3: the centre weight
sits just below 1, so a pixel of value p sums to just below p) and box-like (sigma >= 1000: equal weights, every window
whose pixel sum is a multiple of K^2 sums to an integer), the 2^-70 route boundary of every K, and asymmetric sets (one
off-diagonal weight raised) whose band is wide, accepted and rejected.  The CPU tests prove that the frames make these sums
land near integers and decide the truncation; the GPU tests send every case through every route that can take it and
read the guard-band statistics to show which route ran.
"""
import math
import threading

import numpy as np
import pytest

import rip_b200 as rip

KSIZES = (3, 5, 7, 9, 11, 17, 31)
# The sigma below which the reference generator's KxK kernel holds a weight that is nonzero and below 2^-70, so that the
# streaming blur kernels and the 5x5 fused kernel hand it to the tiled kernel / fused_tile_kernel (bisection of
# rip_gauss_weights; test_route_boundary_sigmas checks both sides).  Well below it the corner weights underflow to 0.
TINY_WEIGHT_SIGMA = {3: 0.143562, 5: 0.287151, 7: 0.431829, 9: 0.578733, 11: 0.726852, 17: 1.174947, 31: 2.234216}
SIGMAS = (0.2, 0.25, 0.5, 1.0, 6.0, 20.0, 1e3, 1e4, 1e5)
TWO_M70 = np.float32(2.0 ** -70)


def sigma_grid(k):
    b = TINY_WEIGHT_SIGMA[k]
    return sorted(set(SIGMAS) | {round(0.99 * b, 6), round(1.01 * b, 6)})


# (K, sigma, raised weight (row, column), amount): the reference kernel with one off-diagonal weight raised -- asymmetric,
# and the separable fit's deviation widens the guard band to ~0.013 / ~0.04 (accepted: 3-8 % of the pixels replay) or
# past 0.05 (rejected: the reference-order kernels run)
PERTURBED = [(5, 1.0, (0, 1), 5e-5), (5, 1.0, (0, 1), 1.5e-4), (5, 1.0, (0, 1), 2.5e-4),
             (9, 2.5, (1, 6), 5e-5), (9, 2.5, (1, 6), 1.5e-4), (9, 2.5, (1, 6), 2.5e-4),
             (17, 6.0, (3, 11), 1e-4), (17, 6.0, (3, 11), 1.5e-4), (17, 6.0, (3, 11), 2.5e-4)]

CASES = [("gauss", k, s) for k in KSIZES for s in sigma_grid(k)] + [("perturbed",) + c for c in PERTURBED] + [("random", 5)]


def case_id(c):
    if c[0] == "gauss":
        return f"k{c[1]}-s{c[2]:g}"
    if c[0] == "perturbed":
        return f"k{c[1]}-s{c[2]:g}-w{c[3][0]}{c[3][1]}+{c[4]:g}"
    return "k5-random"


def case_weights(c, gen):
    """The float32 weights of a case; gen is rip.gauss_weights or oracle.gauss_weights (pinned equal below)."""
    if c[0] == "gauss":
        return gen(c[1], c[2])
    if c[0] == "perturbed":
        k, s, pos, d = c[1:]
        w = gen(k, s).copy()
        w[pos] = np.float32(w[pos] + np.float32(d))
        return w
    rng = np.random.default_rng(5)
    w = rng.random((5, 5)).astype(np.float32)
    return (w / (w.sum() * np.float32(1.001))).astype(np.float32)


# ---- the planner, restated (plan_sep_blur, rip_blur_sep.cu) ------------------------------------------------------------
def _hulp(x):
    return math.ldexp(1.0, math.floor(math.log2(x)) - 24) if x > 0 else 0.0


def sep_band(w):
    """plan_sep_blur's guard band for these weights, or None where it sends them to the reference-order kernel."""
    k = w.shape[0]
    wf = [float(v) for v in w.ravel()]
    if any(not (v >= 0.0) or not math.isfinite(v) for v in wf):
        return None
    up, s, b_ref = 1.0 + 1e-6, 0.0, 0.0
    for i, v in enumerate(wf):
        s += v
        b_ref += _hulp(255.0 * v * up)
        if i >= 1:
            b_ref += _hulp(255.0 * s + 1e-3)
    if not s > 0.0 or 255.0 * s >= 255.9:
        return None
    g = [float(np.float32(math.sqrt(wf[i * k + i]))) for i in range(k)]
    dev = sum(abs(wf[i * k + j] - g[i] * g[j]) for i in range(k) for j in range(k))
    gs = b_h = 0.0
    for i in range(k):
        gs += g[i]
        b_h += _hulp(255.0 * gs * up)
    band = (255.0 * dev + b_ref + b_h * gs + k * 2.0 ** -16) * 1.02 + 1e-6
    return band if band <= 0.05 else None


def scaled_ok(w):
    """Every weight 0 or >= 2^-70: the streaming kernels' and the 5x5 fused kernel's replay on integer bit patterns is exact."""
    return bool(((w == 0) | (w >= TWO_M70)).all())


# ---- frames -----------------------------------------------------------------------------------------------------------
BLUR_SHAPE = (2, 45, 77)    # ragged width (77: partial 32-column tiles, 60- and 32-column streaming bands), a batch
FUSED_SHAPE = (2, 40, 120)  # a width the fused kernel takes (8 pixels per lane by default, 4 forced)


def composite_rgba(h, w, seed):
    """A real frame's features: alpha 255, black sky with dim pixels, one clipped channel, a flat patch reaching a corner."""
    rng = np.random.default_rng(seed)
    img = rng.integers(0, 256, (h, w, 4), dtype=np.uint8)
    img[..., 3] = 255
    sky = img[: h // 3, :, :3]
    sky[...] = 0
    dim = rng.random(sky.shape[:2]) < 0.05
    sky[dim] = rng.integers(1, 4, (int(dim.sum()), 3), dtype=np.uint8)
    img[h // 3: h // 2, : w // 2, 1] = 255
    img[-(h // 3):, -(w // 3):] = (13, 13, 13, 255)
    return img


def blur_frames(shape=BLUR_SHAPE, seed=1):
    """RGBA batch: noise, then real-frame composites."""
    n, h, w = shape
    frames = [np.random.default_rng(seed).integers(0, 256, (h, w, 4), dtype=np.uint8)]
    frames += [composite_rgba(h, w, seed + i) for i in range(1, n)]
    return np.ascontiguousarray(np.stack(frames))


def ref_sums(img, w):
    """The reference's sum (GaussianBlur.cpp:236-258) restated in numpy float32: accumulator from 0, one rounded product and
    one rounded add per tap, ky-major / kx-minor, clamp-to-edge.  Returns it and the same sum in float64."""
    k = w.shape[0]
    r = k // 2
    h, wd = img.shape[:2]
    pad = np.pad(img, ((r, r), (r, r)) + ((0, 0),) * (img.ndim - 2), mode="edge")
    pad32, pad64 = pad.astype(np.float32), pad.astype(np.float64)
    s32 = np.zeros(img.shape, np.float32)
    s64 = np.zeros(img.shape, np.float64)
    for ky in range(k):
        for kx in range(k):
            s32 = s32 + pad32[ky:ky + h, kx:kx + wd] * w[ky, kx]   # (float32 * float32 scalar: a rounded product, then a rounded add)
            s64 += pad64[ky:ky + h, kx:kx + wd] * float(w[ky, kx])
    return s32, s64


# ---- CPU: the weights ---------------------------------------------------------------------------------------------------
def test_weights_equal_the_oracle_generator_over_the_grid(oracle):
    """rip_gauss_weights equals the oracle's restatement of the reference generator bit for bit at every sigma used here
    (test_ref_pins ties a few sigmas of both to the reference itself)."""
    for k in KSIZES:
        for s in sigma_grid(k):
            assert np.array_equal(rip.gauss_weights(k, s).view(np.uint32), oracle.gauss_weights(k, s).view(np.uint32)), (k, s)


def test_route_boundary_sigmas(oracle):
    """Just below the boundary the kernel holds a weight in (0, 2^-70); just above it does not."""
    for k, b in TINY_WEIGHT_SIGMA.items():
        lo, hi = oracle.gauss_weights(k, round(0.99 * b, 6)), oracle.gauss_weights(k, round(1.01 * b, 6))
        assert not scaled_ok(lo) and scaled_ok(hi), k
        assert sep_band(lo) is not None and sep_band(hi) is not None, k


def test_planner_accepts_and_rejects_the_cases_it_should(oracle):
    """Every reference kernel of the grid goes to a guard-band kernel; of the perturbed sets the two smaller raises are
    accepted with a wide band and the largest is rejected; the random set is rejected."""
    for c in CASES:
        w = case_weights(c, oracle.gauss_weights)
        band = sep_band(w)
        if c[0] == "gauss":
            assert band is not None, c
        elif c[0] == "perturbed":
            assert (band is not None) == (c[4] < 2e-4), (c, band)
            if band is not None:
                assert band > 0.01, (c, band)
        else:
            assert band is None


# ---- CPU: the frames are adversarial -------------------------------------------------------------------------------------
NEAR = 2.0 ** -14
# Least counts, on the noise frame of the blur batch (45 x 77 pixels x 4 channels = 13860 sums), of (a) sums within 2^-14 of an
# integer and (b) sums whose float32 truncation differs from that of the float64 sum: half of what the frame gives (rounded
# up for b).  The cases listed are the adversarial ones.  Near the identity a pixel of value p sums to just below p (at the
# K = 3 route boundary every sum does); with box-like weights every window whose pixel sum is a multiple of K^2 sums to an
# integer, fewer of them the larger K.  The other reference kernels of the grid put almost no sum there (0 to 9 of 13860).
MIN_COUNTS = {
    "k3-s0.142126": (6930, 0), "k3-s0.144998": (6930, 0), "k3-s0.2": (212, 13), "k3-s0.25": (7, 1), "k3-s1000": (781, 173),
    "k3-s10000": (781, 2), "k3-s100000": (781, 0), "k5-s0.2": (212, 13), "k5-s0.25": (7, 1), "k5-s1000": (256, 29),
    "k5-s10000": (262, 1), "k5-s100000": (262, 0), "k7-s0.2": (212, 13), "k7-s0.25": (7, 1), "k7-s1000": (129, 21),
    "k7-s10000": (137, 15), "k7-s100000": (139, 4), "k9-s0.2": (212, 13), "k9-s0.25": (7, 1), "k9-s1000": (60, 13),
    "k9-s10000": (58, 2), "k9-s100000": (85, 8), "k11-s0.2": (212, 13), "k11-s0.25": (7, 1), "k11-s1000": (38, 8),
    "k11-s100000": (63, 18), "k17-s0.2": (212, 13), "k17-s0.25": (7, 1), "k17-s1000": (10, 3), "k31-s0.2": (212, 13),
    "k31-s0.25": (7, 1)}
# the perturbed sets that the planner accepts: least share of the noise frame's sums within the guard band of an integer
# (what the kernels must replay; ~2 x band)
MIN_IN_BAND = 0.02


def adversarial(c):
    """The frames put sums inside the guard band for these weights: the kernel that takes them must replay."""
    return case_id(c) in MIN_COUNTS or c[0] == "perturbed"


def test_every_adversarial_case_is_in_the_grid():
    assert set(MIN_COUNTS) <= {case_id(c) for c in CASES}


@pytest.mark.parametrize("c", [c for c in CASES if adversarial(c) or c[0] == "random"], ids=case_id)
def test_frames_put_sums_where_the_rounding_decides(oracle, c):
    w = case_weights(c, oracle.gauss_weights)
    k = w.shape[0]
    frames = blur_frames()
    for f in frames:
        s32, _ = ref_sums(f, w)
        assert np.array_equal(np.clip(s32, 0, 255).astype(np.uint8), oracle.blur(f, k, weights=w, threads=0)), case_id(c)
    s32, s64 = ref_sums(frames[0], w)
    s = s32.astype(np.float64)
    dist = np.abs(s - np.rint(s))
    if case_id(c) in MIN_COUNTS:
        near, decided = int((dist < NEAR).sum()), int((np.floor(s) != np.floor(s64)).sum())
        min_near, min_decided = MIN_COUNTS[case_id(c)]
        assert near >= min_near and decided >= min_decided, (case_id(c), near, decided)
    elif sep_band(w) is not None:
        assert (dist < sep_band(w)).mean() >= MIN_IN_BAND, (case_id(c), sep_band(w))


# ---- GPU ---------------------------------------------------------------------------------------------------------------
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


def _counted(fn):
    """Run fn with the guard-band statistics on; returns (fn's result, the count)."""
    rip.slow_path_stats(True)
    try:
        out = fn()
    finally:
        n = rip.slow_path_stats(False)
    return out, n


def _check_count(n, must_run, limit, what):
    """must_run: a guard-band kernel takes these weights.  Every frame batch here puts sums inside its band (black sky with dim
    pixels and the edges of flat regions do at every sigma), so it must have replayed; the reference-order kernels count nothing."""
    if must_run:
        assert 0 < n <= limit, f"{what}: {n} replays counted (the guard-band kernel should run and replay, at most {limit})"
    else:
        assert n == 0, f"{what}: {n} replays counted, yet the weights should have gone to the reference-order kernel"


@pytest.mark.gpu
@pytest.mark.parametrize("c", CASES, ids=case_id)
def test_gaussian_every_route(ctx, oracle, c, opt):
    """rip_gauss on RGBA (default selection; streaming, tiled and exact kernels forced) and GRAY8.  On these small frames the
    default selection is the tiled kernel (blur_sep_kernel); RIP_BLUR_STREAM reaches blur_stream5_kernel for K = 5 and
    blur_streamk_kernel for K = 9, 17 when every weight is 0 or >= 2^-70, the tiled kernel otherwise.  The statistics count
    pixels with a replay (tiled, 5x5 streaming) or replayed (pixel, channel) entries (KxK streaming)."""
    w = case_weights(c, rip.gauss_weights)
    k = w.shape[0]
    frames = blur_frames()
    n_px = frames.shape[0] * frames.shape[1] * frames.shape[2]
    want = np.stack([oracle.blur(f, k, weights=w, threads=0) for f in frames])
    must_run = sep_band(w) is not None
    for force in (None, "RIP_BLUR_STREAM", "RIP_BLUR_TILED"):
        if force:
            opt(force, 1)
        got, n = _counted(lambda: ctx.process(frames, rip.OP_GAUSSIAN, rip.FMT_RGBA8, ksize=k, weights=w))
        if force:
            opt(force, 0)
        _eq(got, want, f"{case_id(c)} RGBA {force or 'default'}")
        per_entry = force == "RIP_BLUR_STREAM" and k in (9, 17) and scaled_ok(w)
        _check_count(n, must_run, n_px * (4 if per_entry else 1), f"{case_id(c)} RGBA {force or 'default'}")
    opt("RIP_BLUR_EXACT", 1)
    _eq(ctx.process(frames, rip.OP_GAUSSIAN, rip.FMT_RGBA8, ksize=k, weights=w), want, f"{case_id(c)} RGBA exact")
    opt("RIP_BLUR_EXACT", 0)
    gray = np.ascontiguousarray(frames[..., 1])
    got, n = _counted(lambda: ctx.process(gray, rip.OP_GAUSSIAN, rip.FMT_GRAY8, ksize=k, weights=w))
    _eq(got, np.stack([oracle.blur(g, k, weights=w, threads=0) for g in gray]), f"{case_id(c)} GRAY8")
    _check_count(n, must_run, n_px, f"{case_id(c)} GRAY8")


@pytest.mark.gpu
@pytest.mark.parametrize("c", CASES, ids=case_id)
def test_fused_every_route(ctx, oracle, c, opt):
    """rip_fused from RGB8 and GRAY8: default selection, 4 pixels per lane, and the tile kernel forced.  fused_x2_kernel takes
    5x5 weights its planner accepts when every weight is 0 or >= 2^-70; everything else runs fused_tile_kernel, which counts
    nothing.  The x2 kernel's statistics build is a separate instance: its count is taken in a call of its own, the bits are
    compared on the instance that ships."""
    w = case_weights(c, rip.gauss_weights)
    k = w.shape[0]
    rgb = np.ascontiguousarray(blur_frames(FUSED_SHAPE, seed=7)[..., :3])
    gray = np.ascontiguousarray(rgb[..., 1])
    want_rgb = np.stack([oracle.fused(f, k, weights=w, threads=0) for f in rgb])
    want_gray = np.stack([oracle.sobel(oracle.blur(g, k, weights=w, threads=0)) for g in gray])
    for name, value in (("default", 0), ("RIP_FUSED_NPX", 4), ("RIP_FUSED_GENERIC", 1)):
        if value:
            opt(name, value)
        _eq(ctx.process(rgb, rip.OP_FUSED, rip.FMT_RGB8, ksize=k, weights=w), want_rgb, f"{case_id(c)} fused RGB8 {name}")
        _eq(ctx.process(gray, rip.OP_FUSED, rip.FMT_GRAY8, ksize=k, weights=w), want_gray, f"{case_id(c)} fused GRAY8 {name}")
        if value:
            opt(name, 0)
    x2 = k == 5 and sep_band(w) is not None and scaled_ok(w)
    _, n = _counted(lambda: ctx.process(rgb, rip.OP_FUSED, rip.FMT_RGB8, ksize=k, weights=w))
    _check_count(n, x2, rgb.shape[0] * rgb.shape[1] * rgb.shape[2], f"{case_id(c)} fused RGB8")


def _pert(k, d):
    return next(c for c in CASES if c[0] == "perturbed" and c[1] == k and c[4] == d)


@pytest.mark.gpu
@pytest.mark.parametrize("k,shape,cases", [
    (5, (1, 480, 640), [_pert(5, 1.5e-4), ("gauss", 5, 1e3), ("gauss", 5, round(1.01 * TINY_WEIGHT_SIGMA[5], 6))]),
    (9, (2, 1080, 1440), [_pert(9, 1.5e-4), ("gauss", 9, 1e3)]),
    (17, (3, 1080, 1920), [_pert(17, 1.5e-4), ("gauss", 17, 1e4)])], ids=["k5-0.3Mpx", "k9-3.1Mpx", "k17-6.2Mpx"])
def test_default_selection_on_large_inputs_takes_the_streaming_kernel(ctx, oracle, k, shape, cases):
    """Inputs large enough for the default selection to pick blur_stream5_kernel (>= 0.3 Mpx) or blur_streamk_kernel (9x9:
    >= 3 Mpx, 17x17: >= 6 Mpx) without a switch: heavy replay (perturbed, 3-8 % of the pixels), box-like and near-identity
    weights."""
    assert shape[0] * shape[1] * shape[2] >= {5: 300000, 9: 3000000, 17: 6000000}[k]
    frames = blur_frames(shape, seed=11)
    for c in cases:
        w = case_weights(c, rip.gauss_weights)
        got, n = _counted(lambda: ctx.process(frames, rip.OP_GAUSSIAN, rip.FMT_RGBA8, ksize=k, weights=w))
        for i in range(shape[0]):
            _eq(got[i], oracle.blur(frames[i], k, weights=w, threads=0), f"{case_id(c)} {shape} frame {i}")
        assert n > 0, f"{case_id(c)}: no replays counted"


def _canary_run(name, out_bytes, launch, want, pad=256 * 1024):
    """Write into the middle of a guard-filled buffer: the guards must survive and the payload must equal want."""
    buf = rip.DeviceBuffer(out_bytes + 2 * pad)
    buf.upload(np.full(out_bytes + 2 * pad, 0xA5, np.uint8))
    launch(buf.ptr + pad)
    got = buf.download((out_bytes + 2 * pad,))
    buf.free()
    assert (got[:pad] == 0xA5).all() and (got[pad + out_bytes:] == 0xA5).all(), f"{name}: wrote outside its output"
    _eq(got[pad: pad + out_bytes].reshape(want.shape), want, name)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(2, 131, 248), (1, 75, 76)])
def test_heavy_replay_stays_inside_the_output_buffer(oracle, shape, opt):
    """The perturbed sets replay 3-8 % of the pixels: through the streaming kernels (blur_stream5_kernel for 5x5,
    blur_streamk_kernel -- whose deferred replays patch the output byte by byte -- for 9x9 and 17x17) into a canary-padded buffer."""
    n, h, wd = shape
    frames = blur_frames(shape, seed=21)
    d_in = rip.DeviceBuffer(frames.nbytes).upload(frames)
    opt("RIP_BLUR_STREAM", 1)
    for k, d in ((5, 1.5e-4), (9, 1.5e-4), (17, 1e-4), (17, 1.5e-4)):
        c = _pert(k, d)
        w = case_weights(c, rip.gauss_weights)
        want = np.stack([oracle.blur(f, k, weights=w, threads=0) for f in frames])
        _, cnt = _counted(lambda: _canary_run(f"{case_id(c)} {shape}", frames.nbytes,
                                              lambda p: rip.gauss_dev(d_in.ptr, p, wd, h, n, 4, k, w), want))
        assert cnt > 0, f"{case_id(c)}: no replays counted"


def _staircase_rgba(seed):
    """Blocks of 9 x 9 pixels of every level 0..255 (constant windows of every value: the constant-window tables), with noise
    in one channel so that the replay runs too."""
    lv = np.kron(np.arange(256, dtype=np.uint8).reshape(16, 16), np.ones((9, 9), np.uint8))
    img = np.repeat(lv[..., None], 4, axis=2)
    img[..., 2] = np.random.default_rng(seed).integers(0, 256, lv.shape, dtype=np.uint8)
    img[..., 3] = 255
    return np.ascontiguousarray(img)


@pytest.mark.gpu
@pytest.mark.parametrize("k,sigma_a,pert_b,force", [(5, 1.0, 1.5e-4, "RIP_BLUR_TILED"), (5, 1.5, 1.5e-4, "RIP_BLUR_STREAM"),
                                                    (9, 2.5, 1.5e-4, "RIP_BLUR_STREAM"), (17, 6.0, 1.5e-4, "RIP_BLUR_STREAM")])
def test_weight_caches_follow_the_weights(oracle, k, sigma_a, pert_b, force, opt):
    """The per-weight plans (launch_blur_sep's Plan, the fused kernel's flat_dec table) are keyed by the weights: A, B, A of
    the same K on one stream, no synchronisation in between, must each give their own result."""
    opt(force, 1)
    img = _staircase_rgba(31)
    h, wd = img.shape[:2]
    wa = rip.gauss_weights(k, sigma_a)
    wb = case_weights(_pert(k, pert_b), rip.gauss_weights)
    d_in = rip.DeviceBuffer(img.nbytes).upload(img)
    outs = [rip.DeviceBuffer(img.nbytes) for _ in range(3)]
    for o, w in zip(outs, (wa, wb, wa)):
        rip.gauss_dev(d_in.ptr, o.ptr, wd, h, 1, 4, k, w)
    want_a, want_b = oracle.blur(img, k, weights=wa, threads=0), oracle.blur(img, k, weights=wb, threads=0)
    assert not np.array_equal(want_a, want_b)
    for i, (o, want) in enumerate(zip(outs, (want_a, want_b, want_a))):
        _eq(o.download(img.shape), want, f"gauss {k}x{k} {force}, launch {i} of A, B, A")
    if k == 5:
        rgb = np.ascontiguousarray(img[:, : wd // 8 * 8, :3])
        rgb[: 2 * h // 3, :, 2] = rgb[: 2 * h // 3, :, 0]   # grey blocks (constant gray: the flat table decides) above noise
        fw = rgb.shape[1]
        d_rgb = rip.DeviceBuffer(rgb.nbytes).upload(rgb)
        for w_a, w_b in ((wa, wb), (rip.gauss_weights(5, 1.0), rip.gauss_weights(5, 1.5))):
            fouts = [rip.DeviceBuffer(h * fw) for _ in range(3)]
            for o, w in zip(fouts, (w_a, w_b, w_a)):
                rip.fused_dev(d_rgb.ptr, o.ptr, fw, h, 1, rip.FMT_RGB8, 5, w)
            fa, fb = oracle.fused(rgb, 5, weights=w_a, threads=0), oracle.fused(rgb, 5, weights=w_b, threads=0)
            assert not np.array_equal(fa, fb)
            for i, (o, want) in enumerate(zip(fouts, (fa, fb, fa))):
                _eq(o.download((h, fw)), want, f"fused 5x5, launch {i} of A, B, A")


@pytest.mark.gpu
@pytest.mark.parametrize("k", [5, 17])
def test_two_host_threads_with_different_weights_on_one_context(ctx, oracle, k):
    img = _staircase_rgba(32)
    ws = [rip.gauss_weights(k, 1.0 if k == 5 else 6.0), case_weights(_pert(k, 1.5e-4), rip.gauss_weights)]
    wants = [oracle.blur(img, k, weights=w, threads=0) for w in ws]
    errors = []

    def worker(i):
        try:
            for _ in range(20):
                _eq(ctx.process(img, rip.OP_GAUSSIAN, rip.FMT_RGBA8, ksize=k, weights=ws[i].copy()), wants[i], f"thread {i}")
        except Exception as e:   # (reported by the main thread)
            errors.append(e)

    threads = [threading.Thread(target=worker, args=(i,)) for i in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
