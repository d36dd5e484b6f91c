"""Write tests/golden/cv2_nv12.npz: OpenCV's NV12 -> colour conversions, recorded so that the NV12 tests pin the
decode to cv2 on machines without it.

    python tools/make_nv12_golden.py      (needs cv2)

Keys: "<case>.nv12" (H*3/2, W) input frames and "<case>.<order>" cv2.cvtColor(COLOR_YUV2<ORDER>_NV12) of it, for
order in rgb, bgra.  Cases: seeded noise frames ("syn.HxW"; luma and chroma uniform over 0..255) and the
reference's own images (tests/golden/images.npz), cropped to even sizes and converted to NV12 by cv2 (BGR2YUV_I420 with
U and V interleaved).
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import nv12_ref as R  # noqa: E402

SYN_SHAPES = [(2, 2), (2, 6), (6, 10), (16, 24), (74, 76), (120, 162)]
REF_IMAGES = ["Tulips_square75", "Artemis_square75", "Artemis_small240", "Tulips_small240"]
ORDERS = ("rgb", "bgra")   # both channel orders and the alpha channel; the other two are the same bytes rearranged


def main():
    out = {}
    rng = np.random.default_rng(0x4E5612)
    for h, w in SYN_SHAPES:
        out[f"syn.{h}x{w}.nv12"] = rng.integers(0, 256, (h * 3 // 2, w), dtype=np.uint8)
    imgs = np.load(os.path.join(ROOT, "tests", "golden", "images.npz"))
    for name in REF_IMAGES:
        bgr = imgs[name + ".bgr"]
        h, w = bgr.shape[0] & ~1, bgr.shape[1] & ~1
        out[f"ref.{name}.nv12"] = R.from_bgr(bgr[:h, :w])
    for key in [k for k in out if k.endswith(".nv12")]:
        for order in ORDERS:
            out[key[:-5] + "." + order] = R.cv2_decode(out[key], order)
    path = os.path.join(ROOT, "tests", "golden", "cv2_nv12.npz")
    np.savez_compressed(path, **out)
    import cv2
    print(f"wrote {path}: {len(out)} arrays, cv2 {cv2.__version__}")


if __name__ == "__main__":
    main()
