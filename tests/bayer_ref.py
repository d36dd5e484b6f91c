"""8-bit Bayer raw frames -> colour (bilinear demosaic), restated in numpy -- test infrastructure only (the checker, never the
thing under test).

Patterns are named by the sensor's top-left 2x2, as V4L2 (V4L2_PIX_FMT_SRGGB8, ...) and GenICam (BayerRG8, ...) name them.
OpenCV names a pattern by the 2x2 that starts at (1, 1), so its codes read the other way round (CV2_CODE below).

The decode is OpenCV's default cvtColor(COLOR_Bayer**2RGB), bit for bit.  For an interior pixel (1 <= y <= H-2,
1 <= x <= W-2) with raw byte c, h the sum of its left and right neighbours, v the sum of the pixels above and below, n = h + v
and d the sum of the four diagonals:
    red site:              R = c, G = (n + 2) >> 2, B = (d + 2) >> 2
    blue site:             B = c, G = (n + 2) >> 2, R = (d + 2) >> 2
    green site, red row:   G = c, R = (h + 1) >> 1, B = (v + 1) >> 1
    green site, blue row:  G = c, B = (h + 1) >> 1, R = (v + 1) >> 1
Border pixels copy their interior neighbour: out(y, x) = out(clamp(y, 1, H-2), clamp(x, 1, W-2)).  W and H are at least 3.
tests/test_bayer_color.py pins this to cv2 and to the cv2 outputs recorded in tests/golden/cv2_bayer.npz.

Host arrays as the library's Python API takes them: one frame is (H, W) u8, a batch (N, H, W).
"""
from __future__ import annotations

import numpy as np

PATTERNS = ("rggb", "bggr", "grbg", "gbrg")
ORDERS = ("rgb", "bgr", "rgba", "bgra")
# the OpenCV conversion with the same result: cv2.COLOR_Bayer<CV2_CODE[p]>2RGB (and 2BGR / 2RGBA / 2BGRA)
CV2_CODE = {"rggb": "BG", "bggr": "RG", "grbg": "GB", "gbrg": "GR"}
# (row, column) of the red site in the top-left 2x2
RED_AT = {"rggb": (0, 0), "bggr": (1, 1), "grbg": (0, 1), "gbrg": (1, 0)}


def decode(frames: np.ndarray, pattern: str, order: str = "rgb") -> np.ndarray:
    """frames of `pattern` (one (H, W), or a batch (N, H, W)) -> (.., H, W, 3|4) u8 in `order`."""
    a = np.asarray(frames)
    if a.ndim == 3:
        return np.stack([decode(f, pattern, order) for f in a])
    h, w = a.shape
    assert h >= 3 and w >= 3, a.shape
    p = a.astype(np.int32)
    c = p[1:-1, 1:-1]
    hs = p[1:-1, :-2] + p[1:-1, 2:]
    vs = p[:-2, 1:-1] + p[2:, 1:-1]
    ds = p[:-2, :-2] + p[:-2, 2:] + p[2:, :-2] + p[2:, 2:]
    ry, rx = RED_AT[pattern]
    yy, xx = np.mgrid[1:h - 1, 1:w - 1]
    red_row, red_col = (yy & 1) == ry, (xx & 1) == rx
    red, blue = red_row & red_col, ~red_row & ~red_col
    g_red_row, g_blue_row = red_row & ~red_col, ~red_row & red_col
    cross, diag, hh, vv = (hs + vs + 2) >> 2, (ds + 2) >> 2, (hs + 1) >> 1, (vs + 1) >> 1
    r = np.select([red, blue, g_red_row], [c, diag, hh], vv)
    g = np.where(red | blue, cross, c)
    b = np.select([red, blue, g_red_row], [diag, c, vv], hh)
    ys, xs = np.clip(np.arange(h), 1, h - 2) - 1, np.clip(np.arange(w), 1, w - 2) - 1
    chans = {"rgb": (r, g, b), "bgr": (b, g, r)}[order[:3]]
    if len(order) == 4:
        chans = chans + (np.full_like(r, 255),)
    return np.stack(chans, -1).astype(np.uint8)[ys][:, xs]


def cv2_decode(frame: np.ndarray, pattern: str, order: str) -> np.ndarray:
    import cv2
    return cv2.cvtColor(np.ascontiguousarray(frame), getattr(cv2, f"COLOR_Bayer{CV2_CODE[pattern]}2{order.upper()}"))
