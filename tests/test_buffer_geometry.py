"""The device operations across the geometry of the buffers a caller hands in, bit for bit against the C oracle.

The library picks its kernels from that geometry as much as from the content:

* pointer alignment: rip_fused / rip_sobel run the streaming x2 kernel only when d_in is 4-byte aligned (16-byte for RGBA) and
  d_out 4-byte aligned (fused_supported), 8 or 4 pixels per lane by 8/16-byte alignment (x2_npx), else the tile kernel or
  launch_sobel; rip_gray has an aligned and a byte-granular kernel; sobel_kernel picks its store width per row; RGBA rip_gauss
  needs 4-byte aligned buffers and fails with RIP_EINVAL otherwise;
* row bands: rip_fused takes any input band that covers the rows its output band needs; the x2 kernel clamps rows to the band;
* grid slabs: kernels that carry frames in gridDim.z launch batches of more than 65535 frames in slabs;
* byte offsets past 2^31 and 2^32 in one call, and the 16-bit column field of the streaming KxK blur's replay list.

Every output goes into the middle of a canary-filled buffer (or a slot between canary gaps), and every input band sits between
poison rows, so that a kernel writing outside its output or reading outside its band fails the comparison.  Where the route is
observable it is checked: rip.slow_path_stats counts for the x2 fused kernel and the guard-band blur kernels and stays 0 for the
tile and exact kernels; rip.launch_count gives the number of slabs.
"""
import numpy as np
import pytest

import rip_b200 as rip
from test_blur_weight_space import PERTURBED, blur_frames, case_weights

PAD = 256 * 1024
CANARY = 0xA5


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


def _launches(fn):
    before = rip.launch_count()
    fn()
    return rip.launch_count() - before


# ---- frames and the oracle, cached per frame and K -------------------------------------------------------------------
CN = {rip.FMT_GRAY8: 1, rip.FMT_NV12: 1, rip.FMT_RGB8: 3, rip.FMT_BGR8: 3, rip.FMT_RGBA8: 4, rip.FMT_BGRA8: 4}
FMT_NAME = {rip.FMT_GRAY8: "GRAY8", rip.FMT_NV12: "NV12", rip.FMT_RGB8: "RGB8", rip.FMT_BGR8: "BGR8", rip.FMT_RGBA8: "RGBA8",
            rip.FMT_BGRA8: "BGRA8"}


def frames_of(fmt, n, h, w, seed=0):
    """A noise batch in the host layout of fmt: (n, h, w, cn), (n, h, w), or for NV12 (n, h*3/2, w) -- the luma plane, then a
    chroma plane of other noise that no operation here may read."""
    rng = np.random.default_rng([n, h, w, CN[fmt], seed])
    if fmt == rip.FMT_NV12:
        return rng.integers(0, 256, (n, h * 3 // 2, w), dtype=np.uint8)
    shape = (n, h, w) if CN[fmt] == 1 else (n, h, w, CN[fmt])
    return rng.integers(0, 256, shape, dtype=np.uint8)


def image_of(fmt, f, h):
    """The image an operation sees in frame f: the luma plane of NV12, colour channels in RGB order for the oracle."""
    if fmt == rip.FMT_NV12:
        return np.ascontiguousarray(f[:h])
    if fmt in (rip.FMT_BGR8, rip.FMT_BGRA8):
        return np.ascontiguousarray(f[..., [2, 1, 0] + ([3] if CN[fmt] == 4 else [])])
    return f


class Oracle:
    """The oracle's results for one frame and one K, computed once per module."""

    def __init__(self, oracle):
        self.o, self.cache = oracle, {}

    def _get(self, key, fn):
        if key not in self.cache:
            self.cache[key] = fn()
        return self.cache[key]

    def gray(self, img):
        return self._get(("gray", img.shape, img.tobytes()), lambda: self.o.gray(img, threads=0))

    def luma(self, img):
        return img if img.ndim == 2 else self.gray(img)

    def sobel(self, img):
        return self._get(("sobel", img.shape, img.tobytes()), lambda: self.o.sobel(self.luma(img), threads=0))

    def blur(self, img, k, w):
        return self._get(("blur", k, w.tobytes(), img.shape, img.tobytes()), lambda: self.o.blur(img, k, weights=w, threads=0))

    def fused(self, img, k, w):
        return self._get(("fused", k, w.tobytes(), img.shape, img.tobytes()),
                         lambda: self.o.sobel(self.blur(img, k, w), threads=0) if img.ndim == 2
                         else self.o.fused(img, k, weights=w, threads=0))


@pytest.fixture(scope="module")
def ref(oracle):
    return Oracle(oracle)


@pytest.fixture(scope="module")
def bufs():
    """One input and one canary-padded output buffer for the alignment sweep (largest frame: 251 x 67 x 4 x 3 frames)."""
    cap = 251 * 68 * 4 * 3 + 64
    d_in, d_out = rip.DeviceBuffer(cap), rip.DeviceBuffer(cap + 2 * PAD)
    yield d_in, d_out
    d_in.free()
    d_out.free()


def _canary(d_out, out_bytes, out_off, launch, want, name):
    """Launch into d_out + PAD + out_off, inside a canary-filled region: the canaries must survive and the payload must equal want
    (want None: the call must fail and leave the whole region untouched; returns the error)."""
    region = out_bytes + 2 * PAD
    d_out.upload(np.full(region, CANARY, np.uint8))
    err = None
    try:
        launch(d_out.ptr + PAD + out_off)
    except rip.RipError as e:
        if want is not None:
            raise
        err = e
    got = d_out.download((region,))
    if want is None:
        assert err is not None, f"{name}: accepted, expected RIP_EINVAL"
        assert (got == CANARY).all(), f"{name}: a rejected call wrote into the output buffer"
        return err
    assert (got[:PAD + out_off] == CANARY).all() and (got[PAD + out_off + out_bytes:] == CANARY).all(), \
        f"{name}: wrote outside its output"
    _eq(got[PAD + out_off: PAD + out_off + out_bytes].reshape(want.shape), want, name)
    return None


# ---- 1. alignment sweep ------------------------------------------------------------------------------------------------
IN_OFFSETS = (0, 1, 2, 3, 4, 8, 12)
OUT_OFFSETS = (0, 1, 4, 8)
OFFSET_PAIRS = [(i, o) for i in IN_OFFSETS for o in OUT_OFFSETS]
WIDTHS = (4, 8, 12, 36, 124, 248, 250, 251)
HEIGHTS = (1, 2, 3, 5, 67)


def sweep(fmt, in_offsets=IN_OFFSETS, out_offsets=OUT_OFFSETS):
    """(w, h, n, in_off, out_off) for every width x height, batches of 1 and 3 alternating, offset pairs spread so that every pair
    occurs and every width meets five different ones.  NV12 frames take an even height and an even width."""
    pairs = [(i, o) for i in in_offsets for o in out_offsets]
    cases = []
    for wi, w in enumerate(WIDTHS):
        for hi, h in enumerate(HEIGHTS):
            j = wi * len(HEIGHTS) + hi
            if fmt == rip.FMT_NV12:
                w, h = w + (w & 1), h + (h & 1)
            cases.append((w, h, (1, 3)[j % 2]) + pairs[(j * 11) % len(pairs)])
    assert {c[3:] for c in cases} == set(pairs)
    return cases


def test_sweep_meets_every_width_height_batch_and_offset_pair():
    for fmt in (rip.FMT_RGB8, rip.FMT_NV12):
        cases = sweep(fmt)
        assert len(cases) == len(WIDTHS) * len(HEIGHTS) and {c[2] for c in cases} == {1, 3}
        for w in WIDTHS:
            mine = [c for c in cases if c[0] == (w + (w & 1) if fmt == rip.FMT_NV12 else w)]
            assert len({c[3:] for c in mine}) == len(HEIGHTS) and len({c[2] for c in mine}) == 2, (fmt, w)
        if fmt == rip.FMT_NV12:
            assert all(c[0] % 2 == 0 and c[1] % 2 == 0 for c in cases) and any(c[0] % 4 == 2 for c in cases)


def _upload(d_in, frames, in_off):
    d_in.upload(frames, offset=in_off)
    return d_in.ptr + in_off


@pytest.mark.gpu
@pytest.mark.parametrize("out_mode", [rip.GRAY_OUT_U8, rip.GRAY_OUT_RGBA], ids=["u8", "rgba"])
@pytest.mark.parametrize("fmt", [rip.FMT_RGB8, rip.FMT_BGR8, rip.FMT_RGBA8, rip.FMT_BGRA8], ids=FMT_NAME.get)
def test_gray_any_alignment(bufs, ref, fmt, out_mode):
    d_in, d_out = bufs
    for w, h, n, io, oo in sweep(fmt):
        fr = frames_of(fmt, n, h, w)
        want = np.stack([ref.gray(image_of(fmt, f, h)) for f in fr])
        if out_mode == rip.GRAY_OUT_RGBA:
            want = np.concatenate([np.repeat(want[..., None], 3, axis=-1), np.full(want.shape + (1,), 255, np.uint8)], axis=-1)
        p = _upload(d_in, fr, io)
        _canary(d_out, want.nbytes, oo, lambda q: rip.gray_dev(p, q, w, h, n, fmt, out_mode), want,
                f"gray {FMT_NAME[fmt]} {n}x{h}x{w} in+{io} out+{oo}")


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", [rip.FMT_GRAY8, rip.FMT_RGB8, rip.FMT_RGBA8, rip.FMT_NV12], ids=FMT_NAME.get)
def test_sobel_any_alignment(bufs, ref, fmt):
    """The no-blur x2 kernel where the width and the alignment allow it, launch_sobel elsewhere (NV12 batches of widths 2 mod 4
    and unaligned NV12 batches included: launch_sobel steps over each frame's chroma plane)."""
    d_in, d_out = bufs
    for w, h, n, io, oo in sweep(fmt):
        fr = frames_of(fmt, n, h, w)
        want = np.stack([ref.sobel(image_of(fmt, f, h)) for f in fr])
        p = _upload(d_in, fr, io)
        _canary(d_out, want.nbytes, oo, lambda q: rip.sobel_dev(p, q, w, h, n, fmt), want,
                f"sobel {FMT_NAME[fmt]} {n}x{h}x{w} in+{io} out+{oo}")


# (pixels per lane concern the 5x5 x2 kernel only: 17x17 always runs the tile kernel)
FUSED_SWEEP = [(f, 5, npx) for f in (rip.FMT_RGB8, rip.FMT_RGBA8, rip.FMT_GRAY8, rip.FMT_NV12) for npx in (0, 4)] + \
              [(f, 17, 0) for f in (rip.FMT_RGB8, rip.FMT_RGBA8, rip.FMT_GRAY8, rip.FMT_NV12)]


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,k,npx", FUSED_SWEEP, ids=[f"{FMT_NAME[f]}-k{k}-npx{n or 'auto'}" for f, k, n in FUSED_SWEEP])
def test_fused_any_alignment(bufs, ref, fmt, k, npx, opt):
    if npx:
        opt("RIP_FUSED_NPX", npx)
    d_in, d_out = bufs
    wt = rip.gauss_weights(k, 1.0 if k == 5 else 6.0)
    for w, h, n, io, oo in sweep(fmt):
        fr = frames_of(fmt, n, h, w)
        want = np.stack([ref.fused(image_of(fmt, f, h), k, wt) for f in fr])
        p = _upload(d_in, fr, io)
        _canary(d_out, want.nbytes, oo, lambda q: rip.fused_dev(p, q, w, h, n, fmt, k, wt), want,
                f"fused {k}x{k} {FMT_NAME[fmt]} {n}x{h}x{w} in+{io} out+{oo} npx={npx}")


BLUR_FORCES = ("RIP_BLUR_STREAM", "RIP_BLUR_TILED", "RIP_BLUR_EXACT")


@pytest.mark.gpu
@pytest.mark.parametrize("k", [5, 17])
@pytest.mark.parametrize("force", BLUR_FORCES)
def test_gauss_gray8_any_alignment(bufs, ref, force, k, opt):
    opt(force, 1)
    d_in, d_out = bufs
    wt = rip.gauss_weights(k, 1.0 if k == 5 else 6.0)
    for w, h, n, io, oo in sweep(rip.FMT_GRAY8):
        fr = frames_of(rip.FMT_GRAY8, n, h, w)
        want = np.stack([ref.blur(f, k, wt) for f in fr])
        p = _upload(d_in, fr, io)
        _canary(d_out, want.nbytes, oo, lambda q: rip.gauss_dev(p, q, w, h, n, 1, k, wt), want,
                f"gauss GRAY8 {k}x{k} {force} {n}x{h}x{w} in+{io} out+{oo}")


@pytest.mark.gpu
@pytest.mark.parametrize("k", [5, 17])
@pytest.mark.parametrize("force", BLUR_FORCES)
def test_gauss_rgba_needs_4_byte_alignment(bufs, ref, force, k, opt):
    """RGBA: offsets 0/4/8/12 run (streaming kernels forced: blur_stream5_kernel for 5x5, blur_streamk_kernel for 17x17); an input
    or output offset of 1 to 3 bytes fails with RIP_EINVAL and leaves the output untouched."""
    opt(force, 1)
    d_in, d_out = bufs
    wt = rip.gauss_weights(k, 1.0 if k == 5 else 6.0)
    for w, h, n, io, oo in sweep(rip.FMT_RGBA8, (0, 4, 8, 12), (0, 4, 8)):
        fr = frames_of(rip.FMT_RGBA8, n, h, w)
        want = np.stack([ref.blur(f, k, wt) for f in fr])
        p = _upload(d_in, fr, io)
        _canary(d_out, want.nbytes, oo, lambda q: rip.gauss_dev(p, q, w, h, n, 4, k, wt), want,
                f"gauss RGBA {k}x{k} {force} {n}x{h}x{w} in+{io} out+{oo}")
    fr = frames_of(rip.FMT_RGBA8, 2, 5, 36)
    for io, oo in [(1, 0), (2, 0), (3, 0), (0, 1), (0, 2), (0, 3), (1, 1), (3, 8)]:
        p = _upload(d_in, fr, io)
        err = _canary(d_out, fr.nbytes, oo, lambda q: rip.gauss_dev(p, q, 36, 5, 2, 4, k, wt), None,
                      f"gauss RGBA {force} in+{io} out+{oo}")
        assert "rc=-1" in str(err) and "4-byte aligned" in str(err), err


def x2_route(fmt, w, h, io, oo):
    """fused_supported(): the x2 kernel takes W % 4 == 0, H >= 2 (NV12: even), d_in 4-byte (RGBA: 16-byte) and d_out 4-byte aligned."""
    return w >= 4 and w % 4 == 0 and h >= 2 and io % (16 if CN[fmt] == 4 else 4) == 0 and oo % 4 == 0


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", [rip.FMT_RGB8, rip.FMT_RGBA8, rip.FMT_GRAY8, rip.FMT_NV12], ids=FMT_NAME.get)
def test_fused_route_follows_alignment(bufs, ref, fmt):
    """On a flat frame every blurred pixel of the x2 kernel lies in its guard band (value 100, not 0): the x2 kernel counts at least
    one per output pixel (more where segments overlap); the tile kernel, which runs for unaligned buffers, counts none -- and both
    give the oracle's bits."""
    d_in, d_out = bufs
    w, h, n = 128, 16, 2
    fr = np.full(frames_of(fmt, n, h, w).shape, 100, np.uint8)
    w5 = rip.gauss_weights(5, 1.0)
    want = np.stack([ref.fused(image_of(fmt, f, h), 5, w5) for f in fr])
    seen = set()
    for io, oo in OFFSET_PAIRS + [(16, 0), (16, 4)]:
        p = _upload(d_in, fr, io)
        _, cnt = _counted(lambda: _canary(d_out, want.nbytes, oo, lambda q: rip.fused_dev(p, q, w, h, n, fmt, 5, w5), want,
                                          f"fused flat {FMT_NAME[fmt]} in+{io} out+{oo}"))
        x2 = x2_route(fmt, w, h, io, oo)
        seen.add(x2)
        if x2:
            assert n * h * w <= cnt <= 3 * n * h * w, \
                f"in+{io} out+{oo}: the x2 kernel should have run and counted every pixel, counted {cnt}"
        else:
            assert cnt == 0, f"in+{io} out+{oo}: the tile kernel should have run, yet {cnt} replays were counted"
    assert seen == {True, False}


@pytest.mark.gpu
def test_gauss_route_follows_alignment(bufs, ref, opt):
    """Frames whose sums land in the guard band (test_blur_weight_space.blur_frames: noise, black sky with dim pixels, flat
    patches): the guard-band kernels count replays at every offset they accept, the exact kernel counts none."""
    d_in, d_out = bufs
    rgba = blur_frames()
    n, h, w = rgba.shape[:3]
    gray = np.ascontiguousarray(rgba[..., 1])
    wt = rip.gauss_weights(5, 1.0)
    for force in BLUR_FORCES:
        opt(force, 1)
        for img, cn, offsets in ((rgba, 4, [(0, 0), (4, 8), (12, 4), (8, 0)]), (gray, 1, OFFSET_PAIRS)):
            want = np.stack([ref.blur(f, 5, wt) for f in img])
            for io, oo in offsets:
                p = _upload(d_in, img, io)
                _, cnt = _counted(lambda: _canary(d_out, want.nbytes, oo, lambda q: rip.gauss_dev(p, q, w, h, n, cn, 5, wt), want,
                                                  f"gauss {cn}ch {force} in+{io} out+{oo}"))
                if force == "RIP_BLUR_EXACT":
                    assert cnt == 0, (force, cn, io, oo, cnt)
                else:
                    assert 0 < cnt <= want.size, (force, cn, io, oo, cnt)
        opt(force, 0)


# ---- NV12 EDGE on any even width ---------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n,h,w", [(3, 768, 1366), (5, 4, 6), (2, 6, 250)])
def test_nv12_edge_batches_of_any_even_width(ctx, ref, n, h, w):
    """1366 x 768 (a laptop panel; width 2 mod 4) and other widths the x2 kernel does not take: launch_sobel reads each frame's luma
    plane and steps over its chroma plane, through the device API and the host pipeline."""
    fr = frames_of(rip.FMT_NV12, n, h, w, seed=3)
    want = np.stack([ref.sobel(f[:h]) for f in fr])
    _eq(ctx.process(fr, rip.OP_EDGE, rip.FMT_NV12), want, f"EDGE NV12 {n}x{h}x{w} host pipeline")
    wt = rip.gauss_weights(5, 1.0)
    _eq(ctx.process(fr, rip.OP_FUSED, rip.FMT_NV12, ksize=5, weights=wt), np.stack([ref.fused(f[:h], 5, wt) for f in fr]),
        f"FUSED NV12 {n}x{h}x{w} host pipeline")
    d_in, d_out = rip.DeviceBuffer(fr.nbytes + 8), rip.DeviceBuffer(want.nbytes + 8)
    try:
        for io, oo in ((0, 0), (1, 3), (2, 4)):
            d_in.upload(fr, offset=io)
            rip.sobel_dev(d_in.ptr + io, d_out.ptr + oo, w, h, n, rip.FMT_NV12)
            _eq(d_out.download(want.shape, offset=oo), want, f"rip_sobel NV12 {n}x{h}x{w} in+{io} out+{oo}")
    finally:
        d_in.free()
        d_out.free()


@pytest.mark.gpu
def test_nv12_odd_height_is_rejected_by_the_device_ops():
    """An NV12 frame is W*H*3/2 bytes with H even; with an odd H the batch has no frame stride."""
    d = rip.DeviceBuffer(4096)
    try:
        with pytest.raises(rip.RipError, match="even height"):
            rip.sobel_dev(d.ptr, d.ptr + 2048, 8, 5, 2, rip.FMT_NV12)
        with pytest.raises(rip.RipError, match="even height"):
            rip.fused_dev(d.ptr, d.ptr + 2048, 8, 5, 2, rip.FMT_NV12, 5, rip.gauss_weights(5, 1.0))
    finally:
        d.free()


# ---- 2. row bands of every kernel size ----------------------------------------------------------------------------------
BAND_H, BAND_W = 36, 128
BAND_KS = (1, 3, 5, 7, 17, 31)
POISON_ROWS = 4


def band_image(fmt):
    """Noise with a flat bottom (value 100: the x2 kernel's guard band holds every pixel there, so its count shows it ran)."""
    img = frames_of(rip.FMT_GRAY8 if fmt == rip.FMT_NV12 else fmt, 1, BAND_H, BAND_W, seed=9)[0]
    img[-10:] = 100
    return np.ascontiguousarray(img)


def needed_rows(h, k, o0, o1):
    """Rows [g0, g1) of the input that output rows [o0, o1) need: one row for Sobel, then k // 2 for the blur, clipped."""
    b0, b1 = max(0, o0 - 1), min(h, o1 + 1)
    return max(0, b0 - k // 2), min(h, b1 + k // 2)


def run_bands(img, fmt, k, wt, bands, seed=0):
    """Run rip_fused once per (in_row0, in_row1, out_row0, out_row1): every input band sits between rows of poison in one device
    buffer, every output band in a slot between canary gaps of another.  Returns the output bands (the canaries are checked)."""
    rng = np.random.default_rng(seed)
    cn = 1 if img.ndim == 2 else img.shape[2]
    row = BAND_W * cn
    parts, in_offs, pos = [], [], 0
    for i0, i1, _, _ in bands:
        parts.append(rng.integers(0, 256, POISON_ROWS * row, dtype=np.uint8))
        pos += POISON_ROWS * row
        in_offs.append(pos)
        parts.append(img[i0:i1].reshape(-1))
        pos += (i1 - i0) * row
    parts.append(rng.integers(0, 256, POISON_ROWS * row, dtype=np.uint8))
    staged = np.concatenate(parts)
    gap = 4 * BAND_W
    out_offs, pos = [], gap
    for _, _, o0, o1 in bands:
        out_offs.append(pos)
        pos += (o1 - o0) * BAND_W + gap
    d_in, d_out = rip.DeviceBuffer(staged.nbytes), rip.DeviceBuffer(pos)
    try:
        d_in.upload(staged)
        d_out.upload(np.full(pos, CANARY, np.uint8))
        for (i0, i1, o0, o1), pi, po in zip(bands, in_offs, out_offs):
            rip.fused_dev(d_in.ptr + pi, d_out.ptr + po, BAND_W, BAND_H, 1, fmt, k, wt, in_row0=i0, in_rows=i1 - i0,
                          out_row0=o0, out_rows=o1 - o0)
        got = d_out.download((pos,))
    finally:
        d_in.free()
        d_out.free()
    outs, prev = [], 0
    for (_, _, o0, o1), po in zip(bands, out_offs):
        assert (got[prev:po] == CANARY).all(), f"band {o0}..{o1} or its predecessor wrote outside its output"
        outs.append(got[po: po + (o1 - o0) * BAND_W].reshape(o1 - o0, BAND_W))
        prev = po + (o1 - o0) * BAND_W
    assert (got[prev:] == CANARY).all(), "the last band wrote outside its output"
    return outs


def test_band_rows_gives_the_minimal_cover():
    """rip_band_rows with halo k/2 + 1 hands out exactly the rows rip_fused checks for (clipped at the image), so the partitions
    below run every band with the least input it accepts; the out bands tile the frame."""
    for k in BAND_KS:
        for nb in range(1, BAND_H + 1):
            parts = [rip.band_rows(BAND_H, nb, i, k // 2 + 1) for i in range(nb)]
            assert [p[2] for p in parts] == [sum(p[3] for p in parts[:i]) for i in range(nb)] and sum(p[3] for p in parts) == BAND_H
            for i0, ni, o0, no in parts:
                assert (i0, i0 + ni) == needed_rows(BAND_H, k, o0, o0 + no), (k, nb, o0, no)


def band_cases(k):
    """Input bands that cover more than the halo, output bands of one row, and row counts around the x2 segment."""
    h, half = BAND_H, k // 2 + 1
    mid0, mid1 = h // 3, 2 * h // 3
    minimal = lambda o0, o1: needed_rows(h, k, o0, o1) + (o0, o1)
    cases = [(0, h, mid0, mid1),                                                        # the whole frame for a middle band
             (max(0, mid0 - half - 5), min(h, mid1 + half), mid0, mid1),                # extra rows above only
             (max(0, mid0 - half), min(h, mid1 + half + 5), mid0, mid1),                # extra rows below only
             (0, min(h, 2 + half + 3), 0, 2),
             minimal(0, 1), minimal(h - 1, h), minimal(h // 2, h // 2 + 1),             # one output row: top, bottom, middle
             minimal(1, 2), minimal(h - 2, h - 1), minimal(3, h - 3)]
    return cases


BAND_PARAMS = [(f, k, "tile") for f in (rip.FMT_RGB8, rip.FMT_RGBA8, rip.FMT_GRAY8, rip.FMT_NV12) for k in BAND_KS] + \
              [(f, 5, "x2") for f in (rip.FMT_RGB8, rip.FMT_RGBA8, rip.FMT_GRAY8, rip.FMT_NV12)]


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,k,route", BAND_PARAMS, ids=[f"{FMT_NAME[f]}-k{k}-{r}" for f, k, r in BAND_PARAMS])
def test_fused_row_bands_every_kernel_size(ref, fmt, k, route, opt):
    """Every partition rip_band_rows makes (minimal halos k/2 + 1, clipped at the image) from one band up to one band per row,
    oversized input bands and one-row output bands, on the x2 kernel (5x5; rows per segment automatic and forced to 3, so that
    output bands are shorter than one segment and longer than several) and on the tile kernel (every K; forced for 5x5).
    NV12 bands are passed as plain luma rows."""
    img = band_image(fmt)
    wt = rip.gauss_weights(k, 1.0 if k <= 7 else k / 3.0)
    whole = ref.fused(img, k, wt)
    if route == "tile" and k == 5:
        opt("RIP_FUSED_GENERIC", 1)
    for seg in ((0, 3) if route == "x2" else (0,)):
        opt("RIP_FUSED_SEG", seg)
        for nb in range(1, BAND_H + 1):
            parts = [rip.band_rows(BAND_H, nb, i, k // 2 + 1) for i in range(nb)]
            bands = [(i0, i0 + ni, o0, o0 + no) for i0, ni, o0, no in parts]
            for (_, _, o0, o1), got in zip(bands, run_bands(img, fmt, k, wt, bands, seed=nb)):
                _eq(got, whole[o0:o1], f"{FMT_NAME[fmt]} {k}x{k} {route} seg={seg}: {nb} bands, rows {o0}..{o1}")
        cases = band_cases(k)
        for (i0, i1, o0, o1), got in zip(cases, run_bands(img, fmt, k, wt, cases)):
            _eq(got, whole[o0:o1], f"{FMT_NAME[fmt]} {k}x{k} {route} seg={seg}: input rows {i0}..{i1}, output rows {o0}..{o1}")
    opt("RIP_FUSED_SEG", 0)
    # the route: the x2 kernel counts the flat rows' pixels, the tile kernel nothing
    parts = [rip.band_rows(BAND_H, 3, i, k // 2 + 1) for i in range(3)]
    _, cnt = _counted(lambda: run_bands(img, fmt, k, wt, [(i0, i0 + ni, o0, o0 + no) for i0, ni, o0, no in parts]))
    if route == "x2":
        assert cnt > 0, "the x2 kernel should have run on the bands"
    else:
        assert cnt == 0, f"{cnt} replays counted: the x2 kernel ran where the tile kernel should have"


@pytest.mark.gpu
@pytest.mark.parametrize("h,seg", [(33, 0), (37, 4), (65, 0), (66, 5)])
@pytest.mark.parametrize("fmt", [rip.FMT_RGB8, rip.FMT_GRAY8])
@pytest.mark.parametrize("npx", [0, 4], ids=["npx-auto", "npx4"])
def test_fused_whole_frames_whose_last_segment_has_one_row(ctx, ref, h, seg, fmt, npx, opt):
    """Whole frames whose height is 1 more than a multiple of the x2 kernel's rows per segment (32 by default on small batches,
    or forced): the last segment stores one row, the image's last, whose Sobel reflects at the border; the rows its blur reads are
    flat (value 100) above noise, so they go through the guard band.  (A one-row segment that ends above the image's last row --
    a row band -- is covered by test_fused_row_bands_every_kernel_size.)"""
    if npx:
        opt("RIP_FUSED_NPX", npx)
    opt("RIP_FUSED_SEG", seg)
    fr = frames_of(fmt, 3, h, 128, seed=h)
    for i, flat in enumerate((3, 4, 6)):
        fr[i, h - flat:] = 100
    wt = rip.gauss_weights(5, 1.0)
    want = np.stack([ref.fused(f, 5, wt) for f in fr])
    got, cnt = _counted(lambda: ctx.process(fr, rip.OP_FUSED, fmt, ksize=5, weights=wt))
    _eq(got, want, f"fused {FMT_NAME[fmt]} 3x{h}x128 seg={seg} (statistics build)")
    assert cnt > 0, "the x2 kernel should have run"
    _eq(ctx.process(fr, rip.OP_FUSED, fmt, ksize=5, weights=wt), want, f"fused {FMT_NAME[fmt]} 3x{h}x128 seg={seg}")


@pytest.mark.gpu
@pytest.mark.parametrize("k", BAND_KS)
def test_fused_band_that_misses_a_needed_row_is_rejected(k):
    """An input band one row short above or below the rows an output band needs, an input band past the last row, and output rows
    outside the image all fail with RIP_EINVAL; the minimal band is accepted."""
    h, wd = BAND_H, BAND_W
    wt = rip.gauss_weights(k, 1.0 if k <= 7 else k / 3.0)
    d_in, d_out = rip.DeviceBuffer(h * wd * 3), rip.DeviceBuffer(h * wd)
    try:
        def call(i0, i1, o0, o1):
            rip.fused_dev(d_in.ptr, d_out.ptr, wd, h, 1, rip.FMT_RGB8, k, wt, in_row0=i0, in_rows=i1 - i0, out_row0=o0, out_rows=o1 - o0)

        for o0, o1 in ((0, 1), (h // 2, h // 2 + 3), (h - 1, h), (1, h - 1), (k // 2 + 2, k // 2 + 3)):
            if o1 > h:
                continue
            g0, g1 = needed_rows(h, k, o0, o1)
            call(g0, g1, o0, o1)
            with pytest.raises(rip.RipError, match="does not cover"):
                call(g0 + 1, g1, o0, o1)
            with pytest.raises(rip.RipError, match="does not cover"):
                call(g0, g1 - 1, o0, o1)
        with pytest.raises(rip.RipError, match="does not cover"):
            call(1, h + 1, 4, 8)
        for o0, o1 in ((h - 2, h + 1), (-1, 2), (3, 3)):
            with pytest.raises(rip.RipError, match="outside the image"):
                call(0, h, o0, o1)
    finally:
        d_in.free()
        d_out.free()


# ---- 3. the host banded pipeline ------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def big_frames():
    """4099 rows (ragged sub-bands of 1024 and 1025 rows) of RGB, at a width that is a multiple of 4 and one that is not."""
    rng = np.random.default_rng(4099)
    return {wd: rng.integers(0, 256, (4099, wd, 3), dtype=np.uint8) for wd in (4096, 4094)}


@pytest.mark.gpu
@pytest.mark.parametrize("wd,op,k", [(4096, rip.OP_FUSED, 17), (4096, rip.OP_FUSED, 5), (4096, rip.OP_EDGE, 0),
                                     (4094, rip.OP_FUSED, 5), (4094, rip.OP_EDGE, 0)])
def test_host_banded_pipeline_in_four_sub_bands(ctx, oracle, big_frames, wd, op, k):
    """One 4099 x wd RGB frame on a one-device context: rip_submit cuts it into 4 sub-bands with their own halos (one launch each),
    from pageable and from pinned memory.  Width 4094 is not a multiple of 4: EDGE runs launch_sobel and FUSED the tile kernel."""
    img = big_frames[wd]
    wt = rip.gauss_weights(k, 6.0 if k == 17 else 1.0) if k else None
    if op == rip.OP_EDGE:
        want = oracle.sobel(oracle.gray(img, threads=0), threads=0)
    else:
        want = oracle.fused(img, k, weights=wt, threads=0)
    pin = rip.PinnedBuffer(img.nbytes)
    try:
        pinned = pin.array.reshape(img.shape)
        pinned[...] = img
        for name, src in (("pageable", img), ("pinned", pinned)):
            got = {}
            n = _launches(lambda: got.setdefault("out", ctx.process(src, op, rip.FMT_RGB8, ksize=k, weights=wt, banded=True)))
            assert n == 4, f"{name}: {n} launches, expected one per sub-band (4)"
            _eq(got["out"], want, f"banded {wd} op={op} k={k} {name}")
    finally:
        pin.free()


# ---- 4. more than 65535 frames -----------------------------------------------------------------------------------------------
N_MANY = 65540
CHECK_FRAMES = (0, 65534, 65535, 65536, N_MANY - 1)


def _many(fmt, h, w, seed):
    return frames_of(fmt, N_MANY, h, w, seed)


def _check_frames(d_out, per_frame_shape, want_of, what):
    per = int(np.prod(per_frame_shape))
    for i in CHECK_FRAMES:
        _eq(d_out.download(per_frame_shape, offset=i * per), want_of(i), f"{what}, frame {i}")


@pytest.mark.gpu
@pytest.mark.parametrize("cn,k,slabs", [(1, 5, 2), (4, 3, 2), (4, 5, 1)], ids=["gray-k5-exact", "rgba-k3-exact", "rgba-k5-stream"])
def test_gauss_more_than_65535_frames(ref, cn, k, slabs):
    """GRAY8 5x5 and RGBA 3x3: the tiled kernel (frames in gridDim.z) refuses, the exact kernel runs in two slabs.  RGBA 5x5: the
    input is large enough for blur_stream5_kernel, whose grid is 1-D (one launch)."""
    h, w = 3, 5
    fr = _many(rip.FMT_GRAY8 if cn == 1 else rip.FMT_RGBA8, h, w, 65 + k)
    wt = rip.gauss_weights(k, 1.0)
    d_in, d_out = rip.DeviceBuffer(fr.nbytes), rip.DeviceBuffer(fr.nbytes)
    try:
        d_in.upload(fr)
        assert _launches(lambda: rip.gauss_dev(d_in.ptr, d_out.ptr, w, h, N_MANY, cn, k, wt)) == slabs
        _check_frames(d_out, fr.shape[1:], lambda i: ref.blur(fr[i], k, wt), f"gauss {cn}ch {k}x{k}")
    finally:
        d_in.free()
        d_out.free()


@pytest.mark.gpu
@pytest.mark.parametrize("h,w,slabs", [(4, 4, 1), (3, 5, 2)], ids=["4x4-x2", "3x5-tile"])
def test_fused_more_than_65535_frames(ref, h, w, slabs):
    """4 x 4 frames take the x2 kernel (1-D grid), 3 x 5 frames the tile kernel in two slabs."""
    fr = _many(rip.FMT_RGB8, h, w, 7)
    wt = rip.gauss_weights(5, 1.0)
    d_in, d_out = rip.DeviceBuffer(fr.nbytes), rip.DeviceBuffer(N_MANY * h * w)
    try:
        d_in.upload(fr)
        assert _launches(lambda: rip.fused_dev(d_in.ptr, d_out.ptr, w, h, N_MANY, rip.FMT_RGB8, 5, wt)) == slabs
        _check_frames(d_out, (h, w), lambda i: ref.fused(fr[i], 5, wt), f"fused {h}x{w}")
    finally:
        d_in.free()
        d_out.free()


@pytest.mark.gpu
def test_gray_and_nv12_sobel_more_than_65535_frames(ref):
    """rip_gray (1-D grid), and rip_sobel on NV12 frames of width 6 (launch_sobel in two slabs, each slab starting at its first
    frame's luma plane)."""
    fr = _many(rip.FMT_RGB8, 3, 5, 8)
    d_in, d_out = rip.DeviceBuffer(fr.nbytes), rip.DeviceBuffer(N_MANY * 15)
    try:
        d_in.upload(fr)
        assert _launches(lambda: rip.gray_dev(d_in.ptr, d_out.ptr, 5, 3, N_MANY, rip.FMT_RGB8)) == 1
        _check_frames(d_out, (3, 5), lambda i: ref.gray(fr[i]), "gray 3x5")
    finally:
        d_in.free()
        d_out.free()
    nv = _many(rip.FMT_NV12, 4, 6, 9)
    d_in, d_out = rip.DeviceBuffer(nv.nbytes), rip.DeviceBuffer(N_MANY * 24)
    try:
        d_in.upload(nv)
        assert _launches(lambda: rip.sobel_dev(d_in.ptr, d_out.ptr, 6, 4, N_MANY, rip.FMT_NV12)) == 2
        _check_frames(d_out, (4, 6), lambda i: ref.sobel(nv[i][:4]), "sobel NV12 4x6")
    finally:
        d_in.free()
        d_out.free()


# ---- 5. byte offsets past 2^31 and 2^32 ---------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_byte_offsets_past_2_31_and_2_32(ref):
    """520 RGBA 1080p frames (4.31 GB) in one call: frames 258/259 hold input byte 2^31 and frames 517/518 byte 2^32.  Frame i is
    the base frame rolled by i columns, so a frame read from the wrong place gives a different result."""
    n, h, w = 520, 1080, 1920
    fb = h * w * 4
    assert 258 * fb < 2 ** 31 < 259 * fb and 517 * fb < 2 ** 32 < 518 * fb
    base = frames_of(rip.FMT_RGBA8, 1, h, w, seed=520)[0]
    base[: h // 4, :, :3] = 0   # black sky and alpha 255, as a camera frame has them
    base[..., 3] = 255
    check = (258, 259, 517, 518, 519)
    frame = {i: np.ascontiguousarray(np.roll(base, i, axis=1)) for i in check}
    wt = rip.gauss_weights(5, 1.0)
    held = []
    try:
        d_in = rip.DeviceBuffer(n * fb)
        held.append(d_in)
        for i in range(n):
            d_in.upload(frame[i] if i in frame else np.roll(base, i, axis=1), offset=i * fb)
        d_u8 = rip.DeviceBuffer(n * h * w)
        held.append(d_u8)
        runs = [("gray", lambda: rip.gray_dev(d_in.ptr, d_u8.ptr, w, h, n, rip.FMT_RGBA8), lambda f: ref.gray(f)),
                ("sobel", lambda: rip.sobel_dev(d_in.ptr, d_u8.ptr, w, h, n, rip.FMT_RGBA8), lambda f: ref.sobel(f)),
                ("fused", lambda: rip.fused_dev(d_in.ptr, d_u8.ptr, w, h, n, rip.FMT_RGBA8, 5, wt), lambda f: ref.fused(f, 5, wt))]
        for name, launch, want in runs:
            launch()
            for i in check:
                _eq(d_u8.download((h, w), offset=i * h * w), want(frame[i]), f"{name}, frame {i}")
        d_u8.free()
        d_rgba = rip.DeviceBuffer(n * fb)
        held.append(d_rgba)
        rip.gauss_dev(d_in.ptr, d_rgba.ptr, w, h, n, 4, 5, wt)   # (blur_stream5_kernel: 1.08 Gpx is far past its 0.3 Mpx threshold)
        for i in check:
            _eq(d_rgba.download((h, w, 4), offset=i * fb), ref.blur(frame[i], 5, wt), f"gauss 5x5, frame {i}")
    finally:
        for b in held:
            b.free()


# ---- 6. the packed column field of the streaming KxK blur ---------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("k", [9, 17])
@pytest.mark.parametrize("w", [65536, 65537])
def test_streamk_replays_in_columns_above_32768(ref, opt, k, w):
    """blur_streamk_kernel packs the replay column into 16 bits and takes W <= 65536; at 65537 the tiled kernel runs.  The left
    half is black (its sums are exactly 0: nothing to replay) and the right half is noise under weights whose guard band is wide
    (3-8 % of the pixels replay), so the replays sit in columns 32768 .. W - 1."""
    opt("RIP_BLUR_STREAM", 1)
    h, x0 = 40, 32768
    wt = case_weights(next(("perturbed",) + c for c in PERTURBED if c[0] == k and c[3] == 1.5e-4), rip.gauss_weights)
    img = np.zeros((h, w, 4), np.uint8)
    img[:, x0:] = np.random.default_rng(w + k).integers(0, 256, (h, w - x0, 4), dtype=np.uint8)
    # the oracle on the right part only: left of it every window is black (blur 0), and the clamp at the crop's edge repeats black
    s = x0 - 2 * k
    want = np.zeros_like(img)
    want[:, s:] = ref.blur(np.ascontiguousarray(img[:, s:]), k, wt)
    d_in = rip.DeviceBuffer(img.nbytes)
    try:
        d_in.upload(img)
        d_out = rip.DeviceBuffer(img.nbytes + 2 * PAD)
        try:
            _, cnt = _counted(lambda: _canary(d_out, img.nbytes, 0, lambda q: rip.gauss_dev(d_in.ptr, q, w, h, 1, 4, k, wt), want,
                                              f"gauss {k}x{k} {h}x{w}"))
        finally:
            d_out.free()
    finally:
        d_in.free()
    assert cnt > 0, "no replays counted"
