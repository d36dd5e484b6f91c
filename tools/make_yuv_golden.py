"""Write tests/golden/cv2_yuv.npz: OpenCV's YUYV / UYVY / I420 -> colour conversions, recorded so that the tests pin the
decode to cv2 on machines without it.

    python tools/make_yuv_golden.py      (needs cv2)

Keys: "<layout>.<case>.in" input frames (YUYV / UYVY (H, W, 2), I420 (H*3/2, W)) and "<layout>.<case>.<order>"
cv2.cvtColor(COLOR_YUV2<ORDER>_<LAYOUT>) of it, for order in rgb, bgra.  Cases are seeded noise frames (every byte uniform
over 0..255) of awkward shapes: I420 with W/2 odd (W = 6, 10, 1022), YUYV / UYVY with odd heights (1, 3, 5) and widths
that are not multiples of 8, and a few ordinary shapes of each.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import yuv_ref as R  # noqa: E402

SHAPES = {   # (H, W)
    "i420": [(2, 6), (4, 10), (6, 1022), (2, 2), (16, 24), (74, 76)],
    "yuyv": [(1, 6), (3, 10), (5, 2), (1, 1022), (16, 24), (75, 76)],
    "uyvy": [(1, 6), (3, 10), (5, 2), (1, 1022), (16, 24), (75, 76)],
}
ORDERS = ("rgb", "bgra")   # both channel orders and the alpha channel; the other two are the same bytes rearranged


def main():
    out = {}
    rng = np.random.default_rng(0x595556)
    for layout, shapes in SHAPES.items():
        for h, w in shapes:
            shape = (h * 3 // 2, w) if layout == "i420" else (h, w, 2)
            frame = rng.integers(0, 256, shape, dtype=np.uint8)
            out[f"{layout}.{h}x{w}.in"] = frame
            for order in ORDERS:
                out[f"{layout}.{h}x{w}.{order}"] = R.cv2_decode(frame, layout, order)
    path = os.path.join(ROOT, "tests", "golden", "cv2_yuv.npz")
    np.savez_compressed(path, **out)
    import cv2
    print(f"wrote {path}: {len(out)} arrays, cv2 {cv2.__version__}")


if __name__ == "__main__":
    main()
