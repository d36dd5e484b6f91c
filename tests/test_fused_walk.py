"""The streaming fused kernel (gray -> 5x5 blur -> Sobel, and gray -> Sobel) along its walk, bit for bit against the C oracle.

Its correctness depends on the walk as much as on the arithmetic: head, main-loop trips and tail of every segment of rows
(tests/fused_walk_ref.py restates them), and the bands, halo lanes and border lanes across the row.  The cold paths -- the gray
fix, the flat-lane shortcut with its run history, the 25-tap replay -- run in every one of these positions, with different code
in each.  So the frames here are noise with cold-path pixels planted at rows and columns computed from the walk:

* replay pixels: 5x5 constant patches of a gray value v whose constant window sums to just below an integer (the reference
  truncates to rint - 1, the fast path lands on rint), on noise, so that the lane neighbourhood is not constant;
* flat lanes: 5 x (NPX + 4) patches of v aligned to a lane, taller ones whose run history crosses trips and reaches the tail, and
  near misses with one outermost-column pixel of another value;
* gray-fix pixels (RGB / BGR / RGBA): (r, g, b) triples whose reference gray is t / 1000 - 1.

On the CPU the restated walk is pinned to facts read from the source, the GPU grid below is shown to reach every walk class of a
stated universe, and every planted feature is shown to be one whose skipped fix changes the oracle's blurred or gray byte.  On
the GPU both instances run that grid with forced segment lengths, forced 8 and 4 pixels per lane, batches of two and three
frames, every lane_last, row bands through rip_fused and rip_process_host_banded, and one warp walking a whole frame.
"""
import functools

import numpy as np
import pytest

import fused_walk_ref as R
import rip_b200 as rip

W_ROWS = 256                      # row sweep width: 2 bands at 8 pixels per lane, 3 at 4
SEGS = list(range(1, 14)) + [16, 31, 32, 33, 64, 127, 128, 129, 256]
WHOLE = 1 << 20                   # a forced segment length >= H: one segment for the whole frame
WHOLE_HEIGHTS = list(range(2, 25)) + [31, 32, 33]
FMTS = {"RGB8": rip.FMT_RGB8, "BGR8": rip.FMT_BGR8, "RGBA8": rip.FMT_RGBA8, "GRAY8": rip.FMT_GRAY8, "NV12": rip.FMT_NV12}
CN = {"RGB8": 3, "BGR8": 3, "RGBA8": 4, "GRAY8": 1, "NV12": 1}
SIGMA = 1.5
CANARY = 0xA5


# ---- the grid ----------------------------------------------------------------------------------------------------------
def universe(seg):
    """Every walk class (both instances) of whole frames with RIP_FUSED_SEG = seg, over all heights up to six segments and 24
    rows more (one segment: up to 80 rows): first, middle, second-to-last and last segments of every length, and every distance of
    a segment's end from the frame's end that the main loop's stop NB rows before the end can see."""
    hs = range(2, 80) if seg == WHOLE else range(2, 6 * seg + 24)
    return {(b,) + c for b in (True, False) for h in hs for c in R.frame_classes(h, seg, b)}


@functools.lru_cache(None)
def heights_for(seg):
    """Heights below 3 * seg + 8 (one segment: WHOLE_HEIGHTS), picked in increasing order while they add a class.  They are drawn
    from a smaller range than universe(seg), so the coverage test below can fail: it shows that frames of about three segments
    reach every class of frames twice as tall."""
    hs = WHOLE_HEIGHTS if seg == WHOLE else range(2, 3 * seg + 8)
    want, seen, out = universe(seg), set(), []
    cls = lambda h: {(b,) + c for b in (True, False) for c in R.frame_classes(h, seg, b)}
    for h in hs:
        new = cls(h) - seen
        if new:
            out.append(h)
            seen |= new
        if seen == want:
            break
    return tuple(out)


def row_cases():
    return [(seg, h) for seg in SEGS + [WHOLE] for h in heights_for(seg)]


def column_widths(npx):
    """Widths that give every lane_last 1 .. 31 (31 only on a band followed by one whose lane_last is 1), the exact multiple of
    the band width, and 4 .. 7 bands (n_bands % 4 = 0 .. 3: the idle warps of the last block)."""
    band = 30 * npx
    ws = [npx * m for m in range(1, 32)]
    ws += [band * n + npx * m for n, m in ((3, 1), (4, 0), (4, 5), (5, 17), (6, 29), (7, 0))]
    return sorted(set(ws))


# ---- frames --------------------------------------------------------------------------------------------------------------
@functools.lru_cache(None)
def weights():
    return np.ascontiguousarray(rip.gauss_weights(5, SIGMA), np.float32)


def grey_ramp(oracle):
    """gray(c, c, c) for every c: the gray value a grey colour pixel becomes."""
    return oracle.gray(np.repeat(np.arange(256, dtype=np.uint8)[None, :, None], 3, axis=2))[0]


_FIX = {}


def fix_values(oracle):
    """Grey colour values c whose gray v = gray(c, c, c) has a constant window that sums to just below an integer (flat_dec
    bit set): {c: v}; and the gray-fix triples.  (Computed once: the weights and the oracle's gray are fixed.)"""
    if not _FIX:
        gv = grey_ramp(oracle)
        _FIX["good"] = {c: int(gv[c]) for c in range(256) if R.near_integer_below(R.ref_sum(np.full(25, gv[c]), weights()))}
        _FIX["triples"] = R.gray_fix_triples(oracle)
    return _FIX["good"], _FIX["triples"]


def features(h, w, npx, kind_seed):
    """Where the features go: replay centres, flat-lane patches (y0, x0, rows, near-miss column or None)."""
    cols = R.interest_columns(w, npx)
    rng = np.random.default_rng(kind_seed)
    replay = [(y, x) for i, x in enumerate(cols) for y in range(h) if (y - i) % 6 == 0]
    flats = []
    cw = R.column_walk(w, npx)
    x0s = [ln.x for bd in cw["bands"] for ln in bd["lanes"] if ln.lane in (9, 20) and ln.in_img and ln.x + npx + 2 <= w]
    for j, y0 in enumerate(range(1, h - 4, 13)):
        x0 = x0s[j % len(x0s)] if x0s else None
        if x0 is None:
            break
        rows = 5 if j % 3 == 0 else min(14 + int(rng.integers(0, 6)), h - y0)
        miss = None if j % 3 != 2 else (x0 - 2 if j % 2 == 0 else x0 + npx + 1)
        flats.append((y0, x0, rows, miss))
    return replay, flats


def masks(h, w, npx, seed):
    """(pixels of the replay and flat-lane patches, pixels that get gray-fix triples in colour frames): the triples go on every
    row of the interest columns and their neighbours, and around the flat-lane patches, outside the patches."""
    replay, flats = features(h, w, npx, seed)
    patch = np.zeros((h, w), bool)
    for y, x in replay:
        patch[max(0, y - 2):y + 3, max(0, x - 2):x + 3] = True
    for y0, x0, rows, miss in flats:
        patch[y0:y0 + rows, x0 - 2:x0 + npx + 2] = True
    gf = np.zeros((h, w), bool)
    for x in R.interest_columns(w, npx):
        gf[:, max(0, x - 3):x + 4] = True
    for y0, x0, rows, miss in flats:
        gf[max(0, y0 - 3):y0 + rows + 3, x0 - 5:x0 + npx + 5] = True
    return patch, gf & ~patch


def planted_batch(fmt_name, n, h, w, npx, seed, oracle):
    """(host frames, the images the oracle sees (RGB order / luma), replay centres, flat-lane centres)."""
    good, triples = fix_values(oracle)
    cn = CN[fmt_name]
    rng = np.random.default_rng([n, h, w, npx, cn, seed])
    replay, flats = features(h, w, npx, seed)
    imgs, hosts = [], []
    for f in range(n):
        c = list(good)[int(rng.integers(0, len(good)))] if cn > 1 else None
        v = int(rng.choice([good[k] for k in good])) if cn == 1 else good[c]
        val = c if cn > 1 else v
        img = rng.integers(0, 256, (h, w, 3) if cn > 1 else (h, w), dtype=np.uint8)
        patch, gf = masks(h, w, npx, seed)
        if cn > 1:
            img[gf] = triples[rng.integers(0, len(triples), int(gf.sum()))]
        img[patch] = val
        for y0, x0, rows, miss in flats:
            if miss is not None:
                img[y0 + 2, miss] = (val + 2) % 256
        imgs.append(img)
        if fmt_name == "BGR8":
            hosts.append(img[..., ::-1])
        elif fmt_name == "RGBA8":
            hosts.append(np.concatenate([img, rng.integers(0, 256, (h, w, 1), dtype=np.uint8)], axis=2))
        elif fmt_name == "NV12":
            hosts.append(np.concatenate([img, rng.integers(0, 256, (h // 2, w), dtype=np.uint8)], axis=0))
        else:
            hosts.append(img)
    flat_centres = [(y0 + 2 + k, x0 + j) for y0, x0, rows, miss in flats if miss is None
                    for k in range(rows - 4) for j in range(npx)]
    return np.ascontiguousarray(np.stack(hosts)), imgs, replay, flat_centres


def gray_of(img, oracle):
    return img if img.ndim == 2 else oracle.gray(img, threads=0)


def want_fused(img, oracle):
    g = gray_of(img, oracle)
    return oracle.sobel(oracle.blur(g, 5, weights=weights(), threads=0), threads=0)


def want_sobel(img, oracle):
    return oracle.sobel(gray_of(img, oracle), threads=0)


# ---- 1. the walk, restated -------------------------------------------------------------------------------------------------
def test_walk_matches_the_source():
    """Head 7 rows (blur) / 3 (Sobel) when the segment has two output rows or more, 6 / 2 for one row; a one-row segment has no
    main trip; tails of 1 .. 8 and 1 .. 12 rows (the last segment's main loop stops NB rows before the frame's end); every
    step between the first and last storing row stores; the Sobel stage reflects exactly at yb = 1 and yb = H."""
    for blur, full, short, tails in ((True, 7, 6, set(range(1, 9))), (False, 3, 2, set(range(1, 13)))):
        seen_tails = set()
        for seg in SEGS:
            for h in range(2, 3 * seg + 20):
                for ys, ye, w in R.frame_walks(h, seg, blur):
                    assert w.head == (short if ye - ys == 1 else full), (blur, seg, h, ys)
                    if ye - ys == 1:
                        assert w.trips == 0
                    seen_tails.add(w.tail)
                    stored = [s.r - R.halo(blur) for s in w.steps if s.stores]
                    assert stored == list(range(ys, ye)), (blur, seg, h, ys)
                    top = [s for s in w.steps if s.reflect_top and s.stores]
                    assert len(top) == (ys == 0) and all(s.r - R.halo(blur) == 0 for s in top)
                    bottom = [s for s in w.steps if s.reflect_bottom]
                    assert len(bottom) == (ye == h) and all(s is w.steps[-1] and s.part == "tail" for s in bottom)
                    assert all(s.part != "main" for s in w.steps if s.reflect_top or s.reflect_bottom)
                    assert len(w.steps) == ye - ys + 2 * R.halo(blur)
        assert seen_tails == tails, (blur, sorted(seen_tails))
    # the in_rows cut: a band whose input ends right below its output rows
    w = R.row_walk(10, 40, 7, 36, 100, True)
    assert w.cut and w.tail > 3
    assert not R.row_walk(10, 40, 0, 100, 100, True).cut


def test_columns_and_sub_bands_match_the_source():
    cw = R.column_walk(256, 8)
    assert (cw["n_bands"], cw["n_band_groups"], cw["idle_warps"]) == (2, 1, 2)
    assert [b["lane_last"] for b in cw["bands"]] == [32, 2]
    lanes = cw["bands"][1]["lanes"]
    assert lanes[0].need == 1 << 7 and lanes[31].need == 0 and lanes[2].e_right and not lanes[3].in_img
    assert cw["bands"][0]["lanes"][31].need == 1 and cw["bands"][0]["lanes"][1].e_left
    single = R.column_walk(120, 4)
    assert single["n_bands"] == 1 and single["bands"][0]["lane_last"] == 30 and single["bands"][0]["edge_warp"]
    assert R.sub_bands(2048, 4100, 3) == 2 and R.sub_bands(4096, 4100, 3) == 4 and R.sub_bands(2048, 100, 3) == 1


def test_grid_reaches_every_walk_class():
    """The row sweep's heights reach every (head, trips capped at 2, tail, holds row 0, holds row H - 1) class of both instances
    for every forced segment length and for one segment per frame; every trip phase and head / tail row holds a planted replay
    pixel; the column sweep gives every lane_last 1 .. 31, the exact multiple, n_bands % 4 = 0 .. 3 and a single band that holds
    both borders."""
    total = {True: set(), False: set()}
    for seg in SEGS + [WHOLE]:
        got = {(b,) + c for h in heights_for(seg) for b in (True, False) for c in R.frame_classes(h, seg, b)}
        assert got == universe(seg), seg
        for b in (True, False):
            total[b] |= {(seg,) + c[1:] for c in got if c[0] == b}
    print(f"walk classes reached: blur {len(total[True])}, Sobel {len(total[False])} over {len(SEGS) + 1} segment lengths, "
          f"{len(row_cases())} (segment, height) cases")
    # trip phases and head / tail rows hold replay pixels (blurred row yb is replayed in the step that completes it), and with
    # colour input gray-fix pixels (gray row r is fixed in the step that consumes it; rows outside the frame are clamped)
    for i, (seg, h) in enumerate(row_cases()):
        for npx in (8, 4):
            replay, _ = features(h, W_ROWS, npx, i)
            rows = {y for y, _ in replay}
            walk = [s for _, _, w in R.frame_walks(h, seg, True) for s in w.steps if s.blur_runs and s.stores and 0 <= s.yb < h]
            assert {(s.part, s.phase) for s in walk if s.yb in rows} == {(s.part, s.phase) for s in walk}, (seg, h, npx)
            gf_rows = set(np.nonzero(masks(h, W_ROWS, npx, i)[1].any(axis=1))[0])
            for blur in (True, False):
                walk = [s for _, _, w in R.frame_walks(h, seg, blur) for s in w.steps if s.stores]
                held = {(s.part, s.phase) for s in walk if min(max(s.r, 0), h - 1) in gf_rows}
                assert held == {(s.part, s.phase) for s in walk}, (seg, h, npx, blur)
    for npx in (8, 4):
        last = set()
        groups = set()
        for w in column_widths(npx):
            cw = R.column_walk(w, npx)
            last |= {b["lane_last"] for b in cw["bands"] if b["lane_last"] <= 31}
            groups.add(cw["n_bands"] % 4)
        assert last == set(range(1, 32)) and groups == {0, 1, 2, 3}
        assert 30 * npx in column_widths(npx)


@pytest.mark.parametrize("fmt_name", list(FMTS))
@pytest.mark.parametrize("npx", [8, 4])
def test_planted_features_are_sensitive(oracle, fmt_name, npx):
    """Every replay centre and every flat-lane pixel has a window that the reference truncates to rint - 1 right next to rint:
    skipping its fix makes the oracle's blurred byte one larger, and that changes the oracle's Sobel output.  Every gray-fix
    pixel's reference gray is t / 1000 - 1 (skipping the fix makes the gray byte one larger)."""
    w = weights()
    for seg, h in [(3, 29), (1, 12), (WHOLE, 33)]:
        if fmt_name == "NV12" and h % 2:
            h += 1
        _, imgs, replay, flat_centres = planted_batch(fmt_name, 2, h, W_ROWS, npx, seg, oracle)
        for img in imgs:
            g = gray_of(img, oracle)
            b = oracle.blur(g, 5, weights=w, threads=0)
            pad = np.pad(g, 2, mode="edge")
            out = oracle.sobel(b, threads=0)
            for y, x in replay + flat_centres:
                s = R.ref_sum(pad[y:y + 5, x:x + 5], w)
                assert R.near_integer_below(s), (fmt_name, y, x, s)
                assert int(b[y, x]) == int(np.rint(s)) - 1, (y, x)
                skipped = b.copy()
                skipped[y, x] += 1   # the fast path's value: the fix skipped
                assert not np.array_equal(oracle.sobel(skipped, threads=1), out), f"{fmt_name}: a skipped fix at {(y, x)} is masked"
            if img.ndim == 3:
                c = img.astype(int)
                t = 299 * c[..., 0] + 587 * c[..., 1] + 114 * c[..., 2]
                fixed = (t % 1000 == 0) & (t > 0) & (g.astype(int) == t // 1000 - 1)
                assert fixed.sum() > len(R.interest_columns(W_ROWS, npx)) * h, fmt_name
    assert len(replay) >= len(R.interest_columns(W_ROWS, npx)) * (h // 6) and flat_centres


# ---- the flat-lane run history -------------------------------------------------------------------------------------------
HIST_SIGMA = 1e4                  # box-like weights: windows whose rows differ by multiples of 5 sum to within 2^-16 of an integer
HIST_CASES = [(seg, h) for seg in list(range(1, 14)) + [16, 32, WHOLE] for h in (40, 47)]


@functools.lru_cache(None)
def hist_weights():
    return np.ascontiguousarray(rip.gauss_weights(5, HIST_SIGMA), np.float32)


_PROBES = {}


def hist_probe_values(oracle):
    """[(gray (w, u, v), grey colours giving them)] from R.run_history_probes, three distinct values, the closest first."""
    if not _PROBES:
        gv = grey_ramp(oracle)
        inv = {}
        for c in range(256):
            inv.setdefault(int(gv[c]), c)
        p = R.run_history_probes(hist_weights()).astype(int)
        p = p[np.argsort(np.abs(p[:, 1] - p[:, 2]) + np.abs(p[:, 0] - p[:, 2]), kind="stable")]
        _PROBES["v"] = [(tuple(t), tuple(inv[x] for x in t)) for t in p.tolist() if len(set(t)) == 3 and all(x in inv for x in t)][:16]
    return _PROBES["v"]


def hist_rows(h, seed):
    """First rows y0 of the probes (rows w, u, v, v, v, v at y0 .. y0 + 5, noise between), and of the tall one, whose v rows go on
    to the frame's last row: its run of constant rows crosses trips and reaches the tail."""
    tall = h - 16
    return list(range(1 + seed % 9, tall - 8, 9)), tall


def hist_batch(fmt_name, n, h, w, seed, oracle):
    """Noise frames with probe rows constant across the whole width: every lane of every band holds them, border lanes included.
    Returns (host frames, oracle images, [(y0, (w, u, v))])."""
    vals = hist_probe_values(oracle)
    rng = np.random.default_rng([n, h, w, seed, CN[fmt_name]])
    starts, tall = hist_rows(h, seed)
    probes = [(y0, int(rng.integers(0, len(vals)))) for y0 in starts + [tall]]
    imgs, hosts = [], []
    for _ in range(n):
        img = rng.integers(0, 256, (h, w, 3) if CN[fmt_name] > 1 else (h, w), dtype=np.uint8)
        for y0, k in probes:
            gray3, col3 = vals[k]
            seq = col3 if CN[fmt_name] > 1 else gray3
            rows = [seq[0], seq[1]] + [seq[2]] * ((h - y0 - 2) if y0 == tall else 4)
            for i, val in enumerate(rows):
                img[y0 + i] = val
        imgs.append(img)
        hosts.append(img if fmt_name != "RGBA8" else np.concatenate([img, np.full((h, w, 1), 255, np.uint8)], axis=2))
    return np.ascontiguousarray(np.stack(hosts)), imgs, [(y0, vals[k][0]) for y0, k in probes]


def hist_steps(h, seg, seed):
    """(part, phase) of the steps where a probe's history decides: newest row y0 + 5, with the step before it (newest row y0 + 4)
    past the warm-up in the same walk, so that it recorded the run of 3."""
    starts, tall = hist_rows(h, seed)
    out = set()
    for _, _, w in R.frame_walks(h, seg, True):
        by_r = {s.r: s for s in w.steps}
        for y0 in starts + [tall]:
            s0, s1 = by_r.get(y0 + 4), by_r.get(y0 + 5)
            if s0 and s1 and s0.blur_runs and s1.blur_runs:
                out.add((s1.part, s1.phase))
    return out


def test_run_history_probes_reach_every_part_and_are_sensitive(oracle):
    """The probes decide in head steps, in every main-loop phase and in tail steps over the GPU cases; for each of them the
    reference's blurred row is trunc(S) of the window (u, v, v, v, v), a history one row too long would answer with flat_dec[v]
    instead, and that answer changes the oracle's Sobel output."""
    parts = set()
    for i, (seg, h) in enumerate(HIST_CASES):
        parts |= hist_steps(h, seg, i)
    assert parts == {("head", -1), ("main", 0), ("main", 1), ("main", 2), ("tail", -1)}, parts
    wt = hist_weights()
    fd = R.flat_dec(wt)
    assert len(hist_probe_values(oracle)) == 16
    for fmt_name in ("GRAY8", "RGB8"):
        for i, (seg, h) in enumerate(HIST_CASES):
            _, imgs, probes = hist_batch(fmt_name, 1, h, W_ROWS, i, oracle)
            g = gray_of(imgs[0], oracle)
            b = oracle.blur(g, 5, weights=wt, threads=0)
            out = oracle.sobel(b, threads=0)
            for y0, (gw, gu, gv) in probes:
                assert (g[y0] == gw).all() and (g[y0 + 1] == gu).all() and (g[y0 + 2:y0 + 6] == gv).all()
                s = R.ref_sum_rows([gu, gv, gv, gv, gv], wt)
                truth, flat = int(np.trunc(s)), int(np.rint(s)) - int(fd[gv])
                assert (b[y0 + 3] == truth).all() and flat != truth, (y0, gw, gu, gv)
                wrong = b.copy()
                wrong[y0 + 3] = flat
                assert not np.array_equal(oracle.sobel(wrong, threads=1), out), (fmt_name, y0)


# ---- 2. GPU --------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    if rip.device_count() < 1:
        pytest.fail("GPU tests need a CUDA device: librip_cuda has no CPU fallback")
    return 0


def _eq(got, want, what):
    if not np.array_equal(got, want):
        idx = np.argwhere(got != want)
        raise AssertionError(f"{what}: {len(idx)} of {want.size} bytes differ, first at {idx[0].tolist()}")


def run_dev(frames, fmt, h, w, blur, wt=None):
    """One call of rip_fused (K = 5) or rip_sobel on the batch, the output between canaries."""
    n = frames.shape[0]
    pad = 4096
    out_bytes = n * h * w
    d_in, d_out = rip.DeviceBuffer(frames.nbytes), rip.DeviceBuffer(out_bytes + 2 * pad)
    try:
        d_in.upload(frames)
        d_out.upload(np.full(out_bytes + 2 * pad, CANARY, np.uint8))
        if blur:
            rip.fused_dev(d_in.ptr, d_out.ptr + pad, w, h, n, fmt, 5, weights() if wt is None else wt)
        else:
            rip.sobel_dev(d_in.ptr, d_out.ptr + pad, w, h, n, fmt)
        got = d_out.download((out_bytes + 2 * pad,))
    finally:
        d_in.free()
        d_out.free()
    assert (got[:pad] == CANARY).all() and (got[pad + out_bytes:] == CANARY).all(), "wrote outside its output"
    return got[pad:pad + out_bytes].reshape(n, h, w)


def counted(fn):
    rip.slow_path_stats(True)
    try:
        out = fn()
    finally:
        cnt = rip.slow_path_stats(False)
    return out, cnt


def check_batch(oracle, fmt_name, seg, h, w, npx, seed, blur, opt):
    opt("RIP_FUSED_SEG", seg)
    opt("RIP_FUSED_NPX", 4 if npx == 4 else 0)
    n = 2 + seed % 2
    frames, imgs, replay, _ = planted_batch(fmt_name, n, h, w, npx, seed, oracle)
    got, cnt = counted(lambda: run_dev(frames, FMTS[fmt_name], h, w, blur))
    for i, img in enumerate(imgs):
        want = want_fused(img, oracle) if blur else want_sobel(img, oracle)
        _eq(got[i], want, f"{fmt_name} {'fused' if blur else 'sobel'} npx={npx} seg={seg} {h}x{w} frame {i}")
    if blur:
        assert cnt >= len(replay), f"{cnt} replays counted for {len(replay)} planted replay pixels: did the x2 kernel run?"


ROW_CASES = row_cases()


@pytest.mark.gpu
@pytest.mark.parametrize("blur", [True, False], ids=["fused", "sobel"])
@pytest.mark.parametrize("npx", [8, 4])
@pytest.mark.parametrize("fmt_name", list(FMTS))
def test_row_sweep(oracle, dev, fmt_name, npx, blur, opt):
    """Every forced segment length with heights k * seg + t that reach every walk class, batches of 2 and 3 frames."""
    for i, (seg, h) in enumerate(ROW_CASES):
        if fmt_name == "NV12" and h % 2:
            continue
        check_batch(oracle, fmt_name, seg, h, W_ROWS, npx, i, blur, opt)
    if fmt_name == "NV12":   # the odd heights, as the even height above them
        for i, (seg, h) in enumerate(ROW_CASES):
            if h % 2:
                check_batch(oracle, fmt_name, seg, h + 1, W_ROWS, npx, i, blur, opt)


@pytest.mark.gpu
@pytest.mark.parametrize("blur", [True, False], ids=["fused", "sobel"])
@pytest.mark.parametrize("npx", [8, 4])
@pytest.mark.parametrize("fmt_name", ["RGB8", "GRAY8"])
def test_column_sweep(oracle, dev, fmt_name, npx, blur, opt):
    """Every lane_last, partial blocks, a single band holding both borders, at segment lengths 1, 4 and 7."""
    for i, w in enumerate(column_widths(npx)):
        for seg, h in ((1, 6), (4, 17), (7, 23)):
            check_batch(oracle, fmt_name, seg, h, w, npx, i, blur, opt)


@pytest.mark.gpu
@pytest.mark.parametrize("npx", [8, 4])
def test_constant_frame_counts_every_needed_pixel_of_every_step(dev, npx, opt):
    """On a constant frame every pixel is inside the guard band, so the statistics count exactly the needed pixels (lanes 1 .. 30
    whole, one pixel of each halo lane) of every step that gets past the warm-up: n + 2 rows per segment of n rows."""
    v = 3
    for seg, h, w in ((1, 7, 256), (3, 11, 248), (5, 40, 968), (WHOLE, 70, 120)):
        opt("RIP_FUSED_SEG", seg)
        opt("RIP_FUSED_NPX", 4 if npx == 4 else 0)
        frames = np.full((2, h, w), v, np.uint8)
        got, cnt = counted(lambda: run_dev(frames, rip.FMT_GRAY8, h, w, True))
        assert (got == 0).all()
        want = 2 * R.blur_steps_of_frame(h, seg) * R.need_pixels_per_row(w, npx)
        assert cnt == want, f"seg={seg} {h}x{w} npx={npx}: {cnt} pixels counted, the walk needs {want}"


def run_band(oracle_img, host, fmt, h, w, band, blur):
    i0, i1, o0, o1 = band
    cn = 1 if host.ndim == 2 else host.shape[2]
    rows = np.ascontiguousarray(host[i0:i1])
    pad = 4 * w
    d_in, d_out = rip.DeviceBuffer(rows.nbytes), rip.DeviceBuffer((o1 - o0) * w + 2 * pad)
    try:
        d_in.upload(rows)
        d_out.upload(np.full((o1 - o0) * w + 2 * pad, CANARY, np.uint8))
        rip.fused_dev(d_in.ptr, d_out.ptr + pad, w, h, 1, fmt, 5, weights(), in_row0=i0, in_rows=i1 - i0, out_row0=o0,
                      out_rows=o1 - o0)
        got = d_out.download(((o1 - o0) * w + 2 * pad,))
    finally:
        d_in.free()
        d_out.free()
    assert (got[:pad] == CANARY).all() and (got[pad + (o1 - o0) * w:] == CANARY).all(), f"band {band} wrote outside its output"
    return got[pad:pad + (o1 - o0) * w].reshape(o1 - o0, w)


@pytest.mark.gpu
@pytest.mark.parametrize("npx", [8, 4])
@pytest.mark.parametrize("fmt_name", ["RGB8", "GRAY8"])
def test_fused_row_bands_with_forced_segments(oracle, dev, fmt_name, npx, opt):
    """rip_band_rows partitions into 1 .. 7 and one-row bands, plus oversized input bands, at forced segment lengths: the main
    loop cut by in_rows, one-row segments inside a band."""
    h, w = 61, 256
    frames, imgs, _, _ = planted_batch(fmt_name, 1, h, w, npx, 7, oracle)
    want = want_fused(imgs[0], oracle)
    opt("RIP_FUSED_NPX", 4 if npx == 4 else 0)
    for seg in (1, 2, 3, 5, 8, 32):
        opt("RIP_FUSED_SEG", seg)
        for nb in (1, 2, 3, 7, h):
            for i in range(nb):
                i0, ni, o0, no = rip.band_rows(h, nb, i, 3)
                _eq(run_band(imgs[0], frames[0], FMTS[fmt_name], h, w, (i0, i0 + ni, o0, o0 + no), True), want[o0:o0 + no],
                    f"{fmt_name} npx={npx} seg={seg}: band {i} of {nb}")
        for band in ((0, h, 20, 41), (10, 50, 20, 41), (0, 9, 0, 4), (h - 9, h, h - 4, h)):
            _eq(run_band(imgs[0], frames[0], FMTS[fmt_name], h, w, band, True), want[band[2]:band[3]],
                f"{fmt_name} npx={npx} seg={seg}: oversized band {band}")


@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(2048, 4100), (4096, 4100)], ids=["2-sub-bands", "4-sub-bands"])
def test_banded_sobel_cuts_the_main_loop(oracle, dev, w, h, opt):
    """EDGE through rip_process_host_banded on frames big enough for 2 and 4 sub-bands, whose in_rows cut the NB = 6 main loop,
    at forced segment lengths 5, 7 and 64."""
    assert R.sub_bands(w, h, 3) == (2 if w == 2048 else 4)
    rng = np.random.default_rng(w)
    img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    _, triples = fix_values(oracle)
    img[::3, ::5] = triples[rng.integers(0, len(triples), img[::3, ::5].shape[:2])]
    want = want_sobel(img, oracle)
    ctx = rip.Context([0])
    try:
        for seg in (5, 7, 64):
            opt("RIP_FUSED_SEG", seg)
            _eq(ctx.process(img, rip.OP_EDGE, rip.FMT_RGB8, banded=True), want, f"banded EDGE {w}x{h} seg={seg}")
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("blur", [True, False], ids=["fused", "sobel"])
def test_one_warp_walks_the_whole_frame(oracle, dev, blur, opt):
    """A forced segment length >= H: hundreds of main trips per warp, at 1100 rows and on one 4K frame."""
    opt("RIP_FUSED_SEG", WHOLE)
    for fmt_name, h, w, n in (("RGB8", 1100, 256, 2), ("GRAY8", 1100, 120, 3), ("RGB8", 2160, 3840, 1)):
        check_batch(oracle, fmt_name, WHOLE, h, w, 8, n, blur, opt)


@pytest.mark.gpu
@pytest.mark.parametrize("npx", [8, 4])
@pytest.mark.parametrize("fmt_name", ["GRAY8", "RGB8"])
def test_flat_run_history(oracle, dev, fmt_name, npx, opt):
    """Row-constant probes whose flat test stops one row short of the oldest row of the next window: a run history that claims
    one row too many answers with flat_dec[v] there, and the output is wrong.  Box-like weights (sigma 1e4)."""
    opt("RIP_FUSED_NPX", 4 if npx == 4 else 0)
    wt = hist_weights()
    for i, (seg, h) in enumerate(HIST_CASES):
        opt("RIP_FUSED_SEG", seg)
        frames, imgs, probes = hist_batch(fmt_name, 2, h, W_ROWS, i, oracle)
        got, cnt = counted(lambda: run_dev(frames, FMTS[fmt_name], h, W_ROWS, True, wt))
        for k, img in enumerate(imgs):
            g = gray_of(img, oracle)
            _eq(got[k], oracle.sobel(oracle.blur(g, 5, weights=wt, threads=0), threads=0),
                f"{fmt_name} npx={npx} seg={seg} h={h} frame {k}, probes at rows {[y0 for y0, _ in probes]}")
        assert cnt > 0, "no guard-band pixel counted: did the x2 kernel run?"
