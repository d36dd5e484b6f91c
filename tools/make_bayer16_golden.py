"""Write tests/golden/cv2_bayer16.npz: OpenCV's 10- to 16-bit Bayer -> 8-bit colour composition (cvtColor(COLOR_Bayer**2RGB)
on the CV_16U frame, then the scale to CV_8U), recorded so that the tests pin the decode to cv2 on machines without it.

    python tools/make_bayer16_golden.py      (needs cv2)

Every case holds uint16 frames for one depth and is read as each of the four patterns at that depth.  Keys:
  "<bits>.<case>.in"                     the raw frames, (N, H, W) uint16
  "<pattern><bits>.<case>.<order>"       cv2's result for each frame, for order in rgb, bgra
  "<pattern><bits>.artemis.<order>.sha256"
                                         the SHA-256 of cv2's output for all four orders on bayer16_ref.hash_noise(1023, 683,
                                         bits, bits): a 683 x 1023 (W x H: the reference's Artemis image) noise frame that
                                         is computed, not stored (the frame and the outputs would be megabytes)
Cases, at every depth: in-range noise of 3x3, 3x4, 4x3, odd x odd, even x odd, odd x even and W % 8 == 0 with odd H; noise
with the padding bits above the depth set (10, 12 and 14 bits); flat frames of 0, full scale and 65535; flat frames of every
tie value v = (2q + 1) 2^(s-1), s = bits - 8 (q = 0 .. 255, even and odd quotients), and noise drawn from tie values; one
full-scale pixel at every position of a 5x5 frame; horizontal and vertical ramps over the full range.
"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import bayer16_ref as R  # noqa: E402

ORDERS = ("rgb", "bgra")   # both channel orders and the alpha channel; the other two are the same bytes rearranged


def cases(bits):
    rng = np.random.default_rng(0x42313600 + bits)
    top, s = (1 << bits) - 1, bits - 8
    out = {}
    for h, w in ((3, 3), (3, 4), (4, 3), (7, 9), (6, 9), (9, 6), (5, 16)):
        out[f"noise{h}x{w}"] = rng.integers(0, top + 1, (2, h, w), dtype=np.uint16)
    if bits < 16:
        out["padded"] = rng.integers(0, 1 << 16, (2, 9, 16), dtype=np.uint16)
    out["flat"] = np.stack([np.full((4, 5), v, np.uint16) for v in (0, top, 0xffff)])
    ties = ((2 * np.arange(256) + 1) << (s - 1)).astype(np.uint16)   # v / 2^s = q + 1/2, q = 0 .. 255
    out["ties"] = np.broadcast_to(ties[:, None, None], (256, 3, 4)).copy()
    out["tienoise"] = rng.choice(ties, (2, 9, 16)).astype(np.uint16)
    impulses = np.zeros((25, 5, 5), np.uint16)
    impulses.reshape(25, 25)[np.arange(25), np.arange(25)] = top
    out["impulse5x5"] = impulses
    ramp = np.linspace(0, top, 512).round().astype(np.uint16)
    out["hramp"] = np.broadcast_to(ramp, (1, 5, 512)).copy()
    out["vramp"] = np.broadcast_to(ramp[:, None], (1, 512, 5)).copy()
    return out


def main():
    import cv2
    out = {}
    for bits in R.BITS:
        for name, frames in cases(bits).items():
            out[f"{bits}.{name}.in"] = frames
            for pattern in R.PATTERNS:
                for order in ORDERS:
                    out[f"{pattern}{bits}.{name}.{order}"] = np.stack([R.cv2_decode(f, pattern, bits, order) for f in frames])
        artemis = R.hash_noise(1023, 683, bits, bits)
        for pattern in R.PATTERNS:
            for order in R.ORDERS:
                digest = hashlib.sha256(np.ascontiguousarray(R.cv2_decode(artemis, pattern, bits, order)).tobytes()).digest()
                out[f"{pattern}{bits}.artemis.{order}.sha256"] = np.frombuffer(digest, np.uint8)
    path = os.path.join(ROOT, "tests", "golden", "cv2_bayer16.npz")
    np.savez_compressed(path, **out)
    print(f"wrote {path}: {len(out)} arrays, {os.path.getsize(path)} bytes, cv2 {cv2.__version__}")


if __name__ == "__main__":
    main()
