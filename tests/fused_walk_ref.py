"""Plain restatement of how the streaming fused kernel (fused_x2_kernel, csrc/rip_fused_x3.cuh) walks a frame, and frames whose
cold-path pixels sit at positions computed from that walk.

Rows: every warp walks one segment of output rows [ys, ye) in three parts (run_rows_x2): a head of SPECIAL steps with run-time
ring slots, a main loop of trips of NB steps with compile-time slots (NB = 3 with the blur stage, step KS = 0/1/2 of a trip;
NB = 6 for gray -> Sobel), and a tail of SPECIAL steps, which applies BORDER_REFLECT_101 in y.  Step r consumes input row r and
stores output row r - HALO (HALO = 3 with the blur stage, 1 without); with the blur stage it completes blurred row yb = r - 2.

Columns: warps hold bands of 30 * NPX columns, four to a block; lane L of band b holds pixels x = 30 NPX b - NPX + NPX L ..
+ NPX - 1.  Lanes 1..30 store; halo lanes 0 and 31 only feed the pixel next to the band (`need`); the lanes that hold
column 0 / W - 1 take the border rules in x.
"""
from dataclasses import dataclass, field

import numpy as np

WARPS_PER_BLOCK = 4


def halo(blur):
    return 3 if blur else 1


def nb(blur):
    return 3 if blur else 6


# ---- rows ------------------------------------------------------------------------------------------------------------------
def forced_seg_rows(seg, out_rows):
    """pick_seg_rows with RIP_FUSED_SEG = seg > 0: the forced length, at most the band's output rows."""
    return seg if seg < out_rows else out_rows


def segments(out_row0, out_rows, seg_rows):
    """The (ys, ye) of every segment of an output band (fused_x2_kernel: ys = out_row0 + seg * seg_rows)."""
    n_segs = (out_rows + seg_rows - 1) // seg_rows
    return [(out_row0 + s * seg_rows, min(out_row0 + (s + 1) * seg_rows, out_row0 + out_rows)) for s in range(n_segs)]


def sub_bands(width, height, cn, n_devices=1):
    """rip_submit's number of sub-bands per device in row-band mode (one frame, `n_devices` devices in the context)."""
    used = min(height, n_devices)
    band_bytes = width * cn * (height // used + 1)
    sub = min(max(band_bytes // (12 << 20), 1), 4)
    return 1 if height // (used * sub) < 64 else sub


@dataclass
class Step:
    r: int            # input row the step consumes (before the clamp to the band)
    part: str         # "head", "main" or "tail"
    trip: int         # main loop: trip index, else -1
    phase: int        # main loop: step of the trip (KS for the blur instance, 0 .. 5 without it), else -1
    stores: bool      # stores output row r - HALO
    yb: int           # row of the image the Sobel stage consumes (blurred row with the blur stage, gray row without)
    blur_runs: bool   # the blur stage gets past the warm-up return (its cold paths can run)
    reflect_top: bool     # yb == 1: row -1 of the Sobel stage is reflected to row 1
    reflect_bottom: bool  # yb == H: row H is reflected to row H - 2


@dataclass
class Walk:
    head: int
    trips: int
    tail: int
    cut: bool         # in_rows stopped the main loop short of r_last - 1
    steps: list = field(default_factory=list)


def row_walk(ys, ye, in_row0, in_rows, H, blur, with_steps=True):
    """run_rows_x2 and the setup of fused_x2_kernel for one segment (with_steps=False: the lengths only)."""
    hl, n_b = halo(blur), nb(blur)
    r = ys - hl
    r_store, r_last = ys + hl, ye - 1 + hl
    steps, n_steps = [], [0]

    def step(r, part, trip=-1, phase=-1):
        n_steps[0] += 1
        if not with_steps:
            return
        yb = r - 2 if blur else r
        special = part != "main"
        blur_runs = (not blur) or (not special) or r >= r_store - 2
        stores = (r_store <= r <= r_last) if special else True
        steps.append(Step(r, part, trip, phase, stores, yb, blur_runs,
                          special and blur_runs and yb == 1, special and blur_runs and yb == H))

    slot = 1   # newest gray row's ring slot (blur instance)
    while (r <= r_store or (blur and slot not in (2, 5))) and r < r_last:
        if blur:
            slot = 0 if slot == 5 else slot + 1
        step(r, "head")
        r += 1
    head = n_steps[0]
    uncut = r_last - 1
    r_main_last = min(uncut, in_row0 + in_rows - 1 - n_b)
    trips = 0
    while r + n_b - 1 <= r_main_last:
        for k in range(n_b):
            step(r + k, "main", trips, k)
        r += n_b
        trips += 1
    trips_uncut = max(0, (uncut - (r - n_b * trips) + 1) // n_b)
    tail0 = n_steps[0]
    while r <= r_last:
        step(r, "tail")
        r += 1
    return Walk(head, trips, n_steps[0] - tail0, trips < trips_uncut, steps)


def walk_class(w, ys, ye, H, cap=2):
    """(head length, main trips capped at `cap`, tail length, holds row 0, holds row H - 1) of one segment's walk."""
    return (w.head, min(w.trips, cap), w.tail, ys == 0, ye == H)


def frame_walks(H, seg, blur, in_row0=0, in_rows=None, out_row0=0, out_rows=None, with_steps=True):
    """[(ys, ye, Walk)] of every segment of one frame or row band with RIP_FUSED_SEG = seg."""
    in_rows = H - in_row0 if in_rows is None else in_rows
    out_rows = H - out_row0 if out_rows is None else out_rows
    sr = forced_seg_rows(seg, out_rows)
    return [(ys, ye, row_walk(ys, ye, in_row0, in_rows, H, blur, with_steps)) for ys, ye in segments(out_row0, out_rows, sr)]


def frame_classes(H, seg, blur, **band):
    return {walk_class(w, ys, ye, H) for ys, ye, w in frame_walks(H, seg, blur, with_steps=False, **band)}


def blur_steps_of_frame(H, seg, **band):
    """Steps of the blur instance that get past the warm-up return, summed over the segments of one frame or band."""
    return sum(sum(s.blur_runs for s in w.steps) for _, _, w in frame_walks(H, seg, True, **band))


# ---- columns ---------------------------------------------------------------------------------------------------------------
@dataclass
class Lane:
    band: int
    lane: int
    x: int            # first pixel
    in_img: bool
    stores: bool
    need: int         # bit j: pixel j's blurred value feeds an output
    e_left: bool
    e_right: bool


def column_walk(W, npx):
    """n_bands, n_band_groups, the warps of the last block that return at once, and every lane of every band."""
    band_w = 30 * npx
    n_bands = (W + band_w - 1) // band_w
    n_groups = (n_bands + WARPS_PER_BLOCK - 1) // WARPS_PER_BLOCK
    idle = n_groups * WARPS_PER_BLOCK - n_bands
    bands = []
    for b in range(n_bands):
        xw0 = b * band_w
        lane_last = (W - xw0) // npx
        lanes = []
        for L in range(32):
            x = xw0 - npx + npx * L
            in_img = 0 <= x < W
            need = 0 if not in_img else (1 << (npx - 1)) if L == 0 else 1 if L == 31 else (1 << npx) - 1
            lanes.append(Lane(b, L, x, in_img, in_img and 1 <= L <= 30, need, b == 0 and L == 1, L == lane_last))
        bands.append(dict(lane_last=lane_last, edge_warp=b == 0 or lane_last <= 31, lanes=lanes))
    return dict(n_bands=n_bands, n_band_groups=n_groups, idle_warps=idle, bands=bands)


def need_pixels_per_row(W, npx):
    return sum(bin(ln.need).count("1") for bd in column_walk(W, npx)["bands"] for ln in bd["lanes"])


def interest_columns(W, npx):
    """Columns where the x walk changes: lane 1's first pixel and lane 30's last of every band, the two columns on either side of
    every band boundary (the halo lanes' `need` pixels and their neighbours), the first and last pixel of the e_right lane, and
    columns 0, 1, W - 2, W - 1."""
    cw, cols = column_walk(W, npx), {0, 1, W - 2, W - 1}
    for b, bd in enumerate(cw["bands"]):
        for ln in bd["lanes"]:
            if ln.in_img and ln.lane == 1:
                cols.add(ln.x)
            if ln.in_img and ln.lane == 30:
                cols.add(ln.x + npx - 1)
            if ln.e_right:
                cols |= {ln.x, ln.x + npx - 1}
        if b:
            cols |= {b * 30 * npx + d for d in (-2, -1, 0, 1)}
    return sorted(c for c in cols if 0 <= c < W)


# ---- the reference's arithmetic on one window --------------------------------------------------------------------------
def ref_sum(window, w25):
    """GaussianBlur.cpp's sum for one 5x5 window: float accumulator from 0, ky-major / kx-minor, every product and add rounded."""
    acc = np.float32(0.0)
    for p, w in zip(np.asarray(window, np.float32).reshape(-1), np.asarray(w25, np.float32).reshape(-1)):
        acc = np.float32(acc + np.float32(p * w))
    return acc


def flat_dec(w25):
    """Bit v of the kernel's flat_dec table (plan_flat_table): a constant window of gray v sums to just below an integer."""
    out = []
    for v in range(256):
        s = ref_sum(np.full(25, v, np.float32), w25)
        out.append(bool(s < np.rint(s)))
    return out


def ref_sum_rows(rows, w25):
    """ref_sum of windows whose five rows are each constant: rows[ky] is an array of the values of row ky (oldest first)."""
    w25 = np.asarray(w25, np.float32).reshape(5, 5)
    rows = [np.asarray(r, np.float32) for r in rows]
    acc = np.zeros(np.broadcast(*rows).shape, np.float32)
    for ky in range(5):
        for kx in range(5):
            acc = (acc + (rows[ky] * w25[ky, kx]).astype(np.float32)).astype(np.float32)
    return acc


def run_history_probes(w25, tol=2.0 ** -16):
    """Gray values (w, u, v) for rows w, u, v, v, v, v, each constant across a lane's NPX + 4 columns, that check the flat-lane
    run history of blur_flat_lane.  Every pixel of such a lane has the same window, so the fast path's values are bit-identical
    and the flat test runs.  Newest row r = the fourth v: the window (w, u, v, v, v) lies inside the guard band, its flat test
    finds rows r .. r-2 constant and stops at u, and records a run of 3.  Row r + 1 = the last v: the window (u, v, v, v, v) lies
    inside the band too, and the history lets the test start at row r + 1 - 4 = u, which breaks the run: the lane replays.  A
    history that claimed one row more would skip u and answer with flat_dec[v], which differs from the reference's result here."""
    fd = np.array(flat_dec(w25))
    u, v, w = (a.ravel() for a in np.meshgrid(np.arange(256), np.arange(256), np.arange(256), indexing="ij"))
    keep = (u != v) & (w != v)
    u, v, w = u[keep], v[keep], w[keep]
    s1, s2 = ref_sum_rows([w, u, v, v, v], w25), ref_sum_rows([u, v, v, v, v], w25)
    n1, n2 = np.rint(s1), np.rint(s2)
    inside = (np.abs(s1 - n1) < tol) & (n1 > 0) & (np.abs(s2 - n2) < tol) & (n2 > 0)
    flat_wrong = np.where(fd[v], s2 >= n2, s2 < n2)
    ok = inside & flat_wrong
    return np.stack([w[ok], u[ok], v[ok]], axis=1)


def near_integer_below(s, tol=2.0 ** -16):
    """The reference truncates s to rint(s) - 1 while s is so close to rint(s) that the kernel's fast path lands on rint(s):
    a blurred byte that is one too large if the cold path that fixes it is skipped."""
    n = np.rint(s)
    return bool(s < n and n - s < tol and n > 0)


def gray_fix_triples(oracle):
    """Every (r, g, b) whose t = 299 r + 587 g + 114 b is a positive multiple of 1000 and whose reference gray is t / 1000 - 1."""
    r, g = np.meshgrid(np.arange(256), np.arange(256), indexing="ij")
    r, g = r.reshape(-1, 1), g.reshape(-1, 1)
    b = np.arange(256).reshape(1, -1)
    t = 299 * r + 587 * g + 114 * b
    ii, bb = np.nonzero((t % 1000 == 0) & (t > 0))
    cand = np.stack([r[ii, 0], g[ii, 0], bb], axis=1).astype(np.uint8)
    c = cand.astype(int)
    q = (299 * c[:, 0] + 587 * c[:, 1] + 114 * c[:, 2]) // 1000
    got = oracle.gray(cand.reshape(1, -1, 3))[0].astype(int)
    return cand[got == q - 1]
