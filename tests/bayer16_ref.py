"""10- to 16-bit Bayer raw frames -> 8-bit colour, restated in numpy -- test infrastructure only (the checker, never the thing
under test).

The decode is OpenCV's composition, bit for bit:
    cv2.cvtColor(raw16, COLOR_Bayer**2RGB)                    (CV_16U in, CV_16U out)
    rgb16.convertTo(rgb8, CV_8U, 1.0 / (1 << (bits - 8)))
The demosaic is bayer_ref's: the same formulas, border rule and pattern names, evaluated on the full 16-bit samples (sums of
four samples need 18 bits).  The reduction divides each channel by 2^s, s = bits - 8, rounds half to even and saturates:
    q = min(255, (v + 2^(s-1) - 1 + ((v >> s) & 1)) >> s)
A full-scale sample saturates (10-bit 1023 / 4 = 255.75 -> 256 -> 255), and sample bits above bit `bits - 1` are used as they
are.  tests/test_bayer16_color.py pins this to cv2 and to the cv2 outputs recorded in tests/golden/cv2_bayer16.npz.

Host arrays as the library's Python API takes them: one frame is (H, W) uint16, a batch (N, H, W).
"""
from __future__ import annotations

import numpy as np

from bayer_ref import CV2_CODE, ORDERS, PATTERNS, RED_AT  # noqa: F401  (the pattern names are shared with 8 bits)

BITS = (10, 12, 14, 16)


def demosaic(frame: np.ndarray, pattern: str) -> np.ndarray:
    """One (H, W) frame of integer samples -> (H, W, 3) int64 R, G, B before any reduction (what cvtColor gives on CV_16U)."""
    h, w = frame.shape
    assert h >= 3 and w >= 3, frame.shape
    p = frame.astype(np.int64)
    c = p[1:-1, 1:-1]
    hs = p[1:-1, :-2] + p[1:-1, 2:]
    vs = p[:-2, 1:-1] + p[2:, 1:-1]
    ds = p[:-2, :-2] + p[:-2, 2:] + p[2:, :-2] + p[2:, 2:]
    ry, rx = RED_AT[pattern]
    yy, xx = np.mgrid[1:h - 1, 1:w - 1]
    red_row, red_col = (yy & 1) == ry, (xx & 1) == rx
    red, blue = red_row & red_col, ~red_row & ~red_col
    g_red_row = red_row & ~red_col
    cross, diag, hh, vv = (hs + vs + 2) >> 2, (ds + 2) >> 2, (hs + 1) >> 1, (vs + 1) >> 1
    r = np.select([red, blue, g_red_row], [c, diag, hh], vv)
    g = np.where(red | blue, cross, c)
    b = np.select([red, blue, g_red_row], [diag, c, vv], hh)
    ys, xs = np.clip(np.arange(h), 1, h - 2) - 1, np.clip(np.arange(w), 1, w - 2) - 1
    return np.stack([r, g, b], -1)[ys][:, xs]


def reduce(v: np.ndarray, bits: int) -> np.ndarray:
    """convertTo(CV_8U, 1.0 / 2^(bits - 8)) of non-negative integers: divide, round half to even, saturate."""
    s = bits - 8
    v = np.asarray(v, np.int64)
    return np.minimum(255, (v + (1 << (s - 1)) - 1 + ((v >> s) & 1)) >> s).astype(np.uint8)


def decode(frames: np.ndarray, pattern: str, bits: int, order: str = "rgb") -> np.ndarray:
    """frames of `pattern` at `bits` (one (H, W) uint16, or a batch (N, H, W)) -> (.., H, W, 3|4) u8 in `order`."""
    a = np.asarray(frames)
    if a.ndim == 3:
        return np.stack([decode(f, pattern, bits, order) for f in a])
    q = reduce(demosaic(a, pattern), bits)
    if order.startswith("bgr"):
        q = q[..., ::-1]
    if len(order) == 4:
        q = np.concatenate([q, np.full(q.shape[:-1] + (1,), 255, np.uint8)], -1)
    return np.ascontiguousarray(q)


def hash_noise(h: int, w: int, bits: int, seed: int) -> np.ndarray:
    """(h, w) uint16 noise of `bits` bits from integer arithmetic alone (splitmix64 of the pixel index), so that a large
    recorded case needs neither its stored bytes nor a particular numpy random stream."""
    z = np.arange(h * w, dtype=np.uint64) + np.uint64(seed * 0x9E3779B97F4A7C15 % (1 << 64))
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    z ^= z >> np.uint64(31)
    return (z >> np.uint64(64 - bits)).astype(np.uint16).reshape(h, w)


def cv2_decode(frame: np.ndarray, pattern: str, bits: int, order: str) -> np.ndarray:
    """OpenCV's composition: the CV_16U demosaic, then the scale to CV_8U.  Python's cv2 has no Mat.convertTo;
    convertScaleAbs is the same saturate_cast(v * alpha) on these non-negative values.  The 16-bit RGBA alpha is 65535,
    which the scale saturates to 255."""
    import cv2
    code = getattr(cv2, f"COLOR_Bayer{CV2_CODE[pattern]}2{order.upper()}")
    rgb16 = cv2.cvtColor(np.ascontiguousarray(frame, np.uint16), code)
    assert rgb16.dtype == np.uint16
    return cv2.convertScaleAbs(rgb16, alpha=1.0 / (1 << (bits - 8)))
