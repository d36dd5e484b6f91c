"""Write tests/golden/cv2_bayer.npz: OpenCV's Bayer -> colour conversions (the default bilinear demosaic), recorded so that
the tests pin the decode to cv2 on machines without it.

    python tools/make_bayer_golden.py      (needs cv2)

Every case is read as each of the four patterns.  Keys:
  "<case>.in"                        the raw frames, (N, H, W) u8
  "<pattern>.<case>.<order>"         cv2.cvtColor(COLOR_Bayer<CV2 code>2<ORDER>) of each frame, for order in rgb, bgra
  "artemis.in", "<pattern>.artemis.<order>.sha256"
                                     one seeded noise frame of 683 x 1023 (W x H: the reference's Artemis image) and the
                                     SHA-256 of cv2's output for all four orders (the outputs themselves would be megabytes)
Cases: seeded noise of 3x3, 3x4, 4x3, odd x odd, even x odd, odd x even, W % 8 == 0 with odd H; all 0 and all 255; the 0/255
checkerboard at both phases and 255 on one site of every 2x2 (each of the four); one bright pixel at every position of a
5x5 frame; horizontal and vertical ramps.
"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import bayer_ref as R  # noqa: E402

ORDERS = ("rgb", "bgra")   # both channel orders and the alpha channel; the other two are the same bytes rearranged


def cases():
    rng = np.random.default_rng(0x42415945)
    out = {}
    for h, w in ((3, 3), (3, 4), (4, 3), (7, 9), (6, 9), (9, 6), (5, 16), (33, 40)):
        out[f"noise{h}x{w}"] = rng.integers(0, 256, (3, h, w), dtype=np.uint8)
    out["flat"] = np.stack([np.zeros((6, 7), np.uint8), np.full((6, 7), 255, np.uint8)])
    yy, xx = np.mgrid[0:7, 0:8]
    lattices = [((yy + xx) & 1) == p for p in (0, 1)] + [((yy & 1) == a) & ((xx & 1) == b) for a in (0, 1) for b in (0, 1)]
    out["lattice"] = np.stack([255 * m.astype(np.uint8) for m in lattices])
    impulses = np.zeros((25, 5, 5), np.uint8)
    impulses.reshape(25, 25)[np.arange(25), np.arange(25)] = 255
    out["impulse5x5"] = impulses
    ramp = (np.arange(300) % 256).astype(np.uint8)
    out["hramp"] = np.broadcast_to(ramp, (1, 7, 300)).copy()
    out["vramp"] = np.broadcast_to(ramp[:, None], (1, 300, 7)).copy()
    return out


def main():
    import cv2
    out = {}
    for name, frames in cases().items():
        out[f"{name}.in"] = frames
        for pattern in R.PATTERNS:
            for order in ORDERS:
                out[f"{pattern}.{name}.{order}"] = np.stack([R.cv2_decode(f, pattern, order) for f in frames])
    artemis = np.random.default_rng(683).integers(0, 256, (1023, 683), dtype=np.uint8)
    out["artemis.in"] = artemis
    for pattern in R.PATTERNS:
        for order in R.ORDERS:
            digest = hashlib.sha256(np.ascontiguousarray(R.cv2_decode(artemis, pattern, order)).tobytes()).digest()
            out[f"{pattern}.artemis.{order}.sha256"] = np.frombuffer(digest, np.uint8)
    path = os.path.join(ROOT, "tests", "golden", "cv2_bayer.npz")
    np.savez_compressed(path, **out)
    print(f"wrote {path}: {len(out)} arrays, cv2 {cv2.__version__}")


if __name__ == "__main__":
    main()
