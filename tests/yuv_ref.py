"""YUYV / UYVY / I420 (and NV12) -> colour, restated in numpy -- test infrastructure only (the checker, never the thing under
test).

Each layout is unpacked to per-pixel Y, U and V; the colour is then the integer formula of tests/nv12_ref.py (OpenCV's
cvtColor, BT.601 limited range, 20-bit fixed point).  tests/test_yuv_color.py pins this restatement to cv2 on all 2^24
(Y, U, V) triples per layout and to the cv2 outputs recorded in tests/golden/cv2_yuv.npz.

Host arrays as the library's Python API takes them: YUYV and UYVY frames are (H, W, 2) (the CV_8UC2 Mat of a V4L2 capture),
I420 and NV12 frames are (H*3/2, W); a leading batch axis is allowed everywhere.
"""
from __future__ import annotations

import numpy as np

LAYOUTS = ("yuyv", "uyvy", "i420")
ORDERS = ("rgb", "bgr", "rgba", "bgra")


def unpack(frame: np.ndarray, layout: str):
    """One frame -> (Y, U, V), each (H, W) int64: the luma and the chroma that serves each pixel."""
    a = np.asarray(frame)
    if layout in ("yuyv", "uyvy"):
        h, w, two = a.shape
        assert two == 2 and w % 2 == 0, a.shape
        flat = a.reshape(h, w // 2, 4).astype(np.int64)   # one pixel pair per 4 bytes
        iy, iu, iv = (0, 1, 3) if layout == "yuyv" else (1, 0, 2)
        Y = np.stack([flat[..., iy], flat[..., iy + 2]], -1).reshape(h, w)
        return Y, np.repeat(flat[..., iu], 2, 1), np.repeat(flat[..., iv], 2, 1)
    h3, w = a.shape
    h = h3 * 2 // 3
    assert h3 == h * 3 // 2 and h % 2 == 0 and w % 2 == 0, a.shape
    chroma = a[h:].reshape(-1).astype(np.int64)
    if layout == "i420":
        n = (h // 2) * (w // 2)
        u, v = chroma[:n].reshape(h // 2, w // 2), chroma[n:].reshape(h // 2, w // 2)
    else:
        assert layout == "nv12", layout
        uv = chroma.reshape(h // 2, w // 2, 2)
        u, v = uv[..., 0], uv[..., 1]
    up = lambda c: np.repeat(np.repeat(c, 2, 0), 2, 1)   # noqa: E731
    return a[:h].astype(np.int64), up(u), up(v)


def decode(frames: np.ndarray, layout: str, order: str = "rgb") -> np.ndarray:
    """frames of `layout` (one, or a batch) -> (.., H, W, 3|4) u8 in `order`."""
    a = np.asarray(frames)
    if a.ndim == (4 if layout in ("yuyv", "uyvy") else 3):
        return np.stack([decode(f, layout, order) for f in a])
    Y, U, V = unpack(a, layout)
    u, v = U - 128, V - 128
    y = np.maximum(Y - 16, 0) * 1220542
    half = 1 << 19
    r = np.clip((y + 1673527 * v + half) >> 20, 0, 255)
    g = np.clip((y - 852492 * v - 409993 * u + half) >> 20, 0, 255)
    b = np.clip((y + 2116026 * u + half) >> 20, 0, 255)
    chans = {"rgb": (r, g, b), "bgr": (b, g, r)}[order[:3]]
    if len(order) == 4:
        chans = chans + (np.full_like(r, 255),)
    return np.stack(chans, -1).astype(np.uint8)


def i420_from_nv12(nv12: np.ndarray) -> np.ndarray:
    """The same image as I420: NV12's interleaved chroma split into a U plane and a V plane."""
    h3, w = nv12.shape
    h = h3 * 2 // 3
    uv = nv12[h:].reshape(h // 2, w // 2, 2)
    planes = np.concatenate([uv[..., 0].reshape(-1), uv[..., 1].reshape(-1)])
    return np.concatenate([nv12[:h], planes.reshape(h // 2, w)], 0)


def packed_from_planes(Y: np.ndarray, U: np.ndarray, V: np.ndarray, layout: str) -> np.ndarray:
    """A YUYV or UYVY frame, (H, W, 2), from luma (H, W) and one U, V per pixel pair, (H, W/2) each."""
    h, w = Y.shape
    q = np.empty((h, w // 2, 4), np.uint8)
    iy, iu, iv = (0, 1, 3) if layout == "yuyv" else (1, 0, 2)
    q[..., iy], q[..., iy + 2], q[..., iu], q[..., iv] = Y[:, 0::2], Y[:, 1::2], U, V
    return q.reshape(h, w, 2)


def exhaustive_frame(layout: str) -> np.ndarray:
    """A 4096 x 4096 frame holding every (Y, U, V) triple once.
    YUYV / UYVY: pixel pair p has U = (p // 128) & 255, V = p // 32768 and the luma values 2 (p % 128), 2 (p % 128) + 1.
    I420: tests/nv12_ref.exhaustive_frame() with its chroma split into planes."""
    if layout == "i420":
        import nv12_ref
        return i420_from_nv12(nv12_ref.exhaustive_frame())
    p = np.arange(4096 * 2048, dtype=np.int64).reshape(4096, 2048)
    Y = np.empty((4096, 4096), np.uint8)
    Y[:, 0::2], Y[:, 1::2] = 2 * (p % 128), 2 * (p % 128) + 1
    return packed_from_planes(Y, ((p // 128) & 255).astype(np.uint8), (p // 32768).astype(np.uint8), layout)


def cv2_decode(frame: np.ndarray, layout: str, order: str) -> np.ndarray:
    import cv2
    name = f"COLOR_YUV2{order.upper()}_{layout.upper()}"
    return cv2.cvtColor(np.ascontiguousarray(frame), getattr(cv2, name))
