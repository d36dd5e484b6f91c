"""Packed 10- and 12-bit Bayer raw frames, restated in numpy -- test infrastructure only (the checker, never the thing under
test).

Four layouts, rows of W*b/8 bytes with no padding:
    mipi10     MIPI CSI-2 RAW10: 4 pixels in 5 bytes.  Bytes 0-3 hold bits 9..2 of pixels 0-3; byte 4 holds bits 1..0 of
               pixel i at bit positions 2i+1..2i.
    mipi12     MIPI CSI-2 RAW12: 2 pixels in 3 bytes.  Bytes 0-1 hold bits 11..4 of pixels 0 and 1; byte 2 holds pixel 0's
               bits 3..0 in its low nibble and pixel 1's in its high nibble.
    genicam10  GenICam PFNC BayerRG10p ...: an LSB-first bit stream, pixel i at stream bits 10i .. 10i+9, stream bit k at
               bit k % 8 of byte k // 8.
    genicam12  the same with 12 bits per pixel.
The MIPI layouts are written as byte arithmetic and the GenICam ones as a bit stream (np.unpackbits / np.packbits, little
bit order), so the two share no code.  The decode is unpack, then bayer16_ref.decode at the same depth: the decode of
RIP_FMT_BAYER_<pattern>10 / 12 on the unpacked frame, which tests/test_bayer16_color.py pins to cv2.

Host arrays as the library's Python API takes them: one frame is (H, row_bytes) uint8, a batch (N, H, row_bytes).
"""
from __future__ import annotations

import numpy as np

import bayer16_ref as R16

LAYOUTS = ("mipi10", "mipi12", "genicam10", "genicam12")


def bits_of(layout: str) -> int:
    return int(layout[-2:])


def row_bytes(layout: str, w: int) -> int:
    b = bits_of(layout)
    assert w * b % 8 == 0, (layout, w)
    return w * b // 8


def pack(samples: np.ndarray, layout: str) -> np.ndarray:
    """(.., H, W) integer samples of bits_of(layout) bits -> (.., H, row_bytes) uint8."""
    s = np.asarray(samples).astype(np.uint16)
    b = bits_of(layout)
    assert (s >> b == 0).all(), "samples wider than the layout"
    *lead, w = s.shape
    if layout == "mipi10":
        g = s.reshape(*lead, w // 4, 4)
        lo = (g[..., 0] & 3) | (g[..., 1] & 3) << 2 | (g[..., 2] & 3) << 4 | (g[..., 3] & 3) << 6
        out = np.concatenate([g >> 2, lo[..., None]], -1)
    elif layout == "mipi12":
        g = s.reshape(*lead, w // 2, 2)
        lo = (g[..., 0] & 15) | (g[..., 1] & 15) << 4
        out = np.concatenate([g >> 4, lo[..., None]], -1)
    else:
        bitplanes = (s[..., None] >> np.arange(b, dtype=np.uint16)) & 1   # (.., W, b), bit 0 first
        return np.packbits(bitplanes.reshape(*lead, w * b).astype(np.uint8), axis=-1, bitorder="little")
    return out.reshape(*lead, -1).astype(np.uint8)


def unpack(packed: np.ndarray, layout: str) -> np.ndarray:
    """(.., H, row_bytes) uint8 -> (.., H, W) uint16 samples."""
    p = np.asarray(packed, np.uint8)
    b = bits_of(layout)
    *lead, nb = p.shape
    if layout == "mipi10":
        g = p.reshape(*lead, nb // 5, 5).astype(np.uint16)
        s = np.stack([g[..., i] << 2 | (g[..., 4] >> (2 * i)) & 3 for i in range(4)], -1)
    elif layout == "mipi12":
        g = p.reshape(*lead, nb // 3, 3).astype(np.uint16)
        s = np.stack([g[..., 0] << 4 | g[..., 2] & 15, g[..., 1] << 4 | g[..., 2] >> 4], -1)
    else:
        stream = np.unpackbits(p, axis=-1, bitorder="little").reshape(*lead, nb * 8 // b, b).astype(np.uint16)
        return (stream << np.arange(b, dtype=np.uint16)).sum(-1, dtype=np.uint16)
    return s.reshape(*lead, -1)


def decode(packed: np.ndarray, pattern: str, layout: str, order: str = "rgb") -> np.ndarray:
    """packed frames of `pattern` in `layout` -> (.., H, W, 3|4) u8 in `order`."""
    return R16.decode(unpack(packed, layout), pattern, bits_of(layout), order)
