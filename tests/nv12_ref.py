"""NV12 -> colour, restated in numpy -- test infrastructure only (the checker, never the thing under test).

OpenCV's cvtColor(COLOR_YUV2RGB_NV12) and its BGR / RGBA / BGRA siblings (BT.601 limited range, 20-bit fixed point, one
U,V pair per 2x2 block).  tests/test_nv12_color.py pins this restatement to cv2 on all 2^24 (Y, U, V) triples and to the
cv2 outputs recorded in tests/golden/cv2_nv12.npz; everything downstream (gray, blur, Sobel) is the C oracle's.
"""
from __future__ import annotations

import numpy as np

ORDERS = ("rgb", "bgr", "rgba", "bgra")


def decode(nv12: np.ndarray, order: str = "rgb") -> np.ndarray:
    """nv12: (H*3/2, W) or (N, H*3/2, W) u8, W and H even -> (.., H, W, 3|4) u8 in `order`."""
    a = np.asarray(nv12)
    if a.ndim == 3:
        return np.stack([decode(f, order) for f in a])
    h3, w = a.shape
    h = h3 * 2 // 3
    assert h3 == h * 3 // 2 and h % 2 == 0 and w % 2 == 0, a.shape
    Y = a[:h].astype(np.int64)
    uv = a[h:].reshape(h // 2, w // 2, 2).astype(np.int64)
    u = np.repeat(np.repeat(uv[..., 0] - 128, 2, 0), 2, 1)
    v = np.repeat(np.repeat(uv[..., 1] - 128, 2, 0), 2, 1)
    y = np.maximum(Y - 16, 0) * 1220542
    half = 1 << 19
    r = np.clip((y + 1673527 * v + half) >> 20, 0, 255)
    g = np.clip((y - 852492 * v - 409993 * u + half) >> 20, 0, 255)
    b = np.clip((y + 2116026 * u + half) >> 20, 0, 255)
    chans = {"rgb": (r, g, b), "bgr": (b, g, r)}[order[:3]]
    if len(order) == 4:
        chans = chans + (np.full_like(r, 255),)
    return np.stack(chans, -1).astype(np.uint8)


def to_rgba(rgb: np.ndarray) -> np.ndarray:
    """(.., H, W, 3) -> (.., H, W, 4) with alpha 255: the reference's container after cvtColor(BGR2RGBA)."""
    return np.concatenate([rgb, np.full(rgb.shape[:-1] + (1,), 255, np.uint8)], -1)


def exhaustive_frame() -> np.ndarray:
    """A 4096 x 4096 NV12 frame holding every (Y, U, V) triple once: 2x2 block b has U = (b // 64) & 255,
    V = b // 16384 and the four luma values 4 (b % 64) .. 4 (b % 64) + 3 (top left, top right, bottom left, bottom right)."""
    nb = 2048
    b = np.arange(nb * nb, dtype=np.int64).reshape(nb, nb)
    y0 = 4 * (b % 64)
    Y = np.empty((4096, 4096), np.uint8)
    Y[0::2, 0::2], Y[0::2, 1::2], Y[1::2, 0::2], Y[1::2, 1::2] = y0, y0 + 1, y0 + 2, y0 + 3
    uv = np.empty((2048, 2048, 2), np.uint8)
    uv[..., 0] = (b // 64) & 255
    uv[..., 1] = b // 16384
    return np.concatenate([Y, uv.reshape(2048, 4096)], 0)


def from_bgr(bgr: np.ndarray) -> np.ndarray:
    """An NV12 frame of an even-sized BGR image by cv2 (BGR2YUV_I420, then U and V interleaved).  Needs cv2."""
    import cv2
    h, w = bgr.shape[:2]
    i420 = cv2.cvtColor(np.ascontiguousarray(bgr), cv2.COLOR_BGR2YUV_I420)
    planes, n = i420[h:].reshape(-1), (h // 2) * (w // 2)
    u, v = planes[:n].reshape(h // 2, w // 2), planes[n:].reshape(h // 2, w // 2)
    return np.concatenate([i420[:h], np.stack([u, v], -1).reshape(h // 2, w)], 0)


def cv2_decode(nv12: np.ndarray, order: str) -> np.ndarray:
    import cv2
    code = {"rgb": cv2.COLOR_YUV2RGB_NV12, "bgr": cv2.COLOR_YUV2BGR_NV12, "rgba": cv2.COLOR_YUV2RGBA_NV12,
            "bgra": cv2.COLOR_YUV2BGRA_NV12}[order]
    return cv2.cvtColor(np.ascontiguousarray(nv12), code)
