"""The format table (csrc/rip_formats.h) against include/rip_cuda.h: every RIP_FMT_* code has exactly one row, named after
its enumerator; the Bayer pattern, depth and packing match the name; and the accepted shapes and bytes per frame match a
restatement of the header's documentation of each format.  The library and the C++ Controller take every format fact from
the table, so a wrong row fails here, without a GPU."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "opencl-development-real-time-image-processing_b200")

# FormatLayout and BayerPacking, in their order in rip_formats.h
INTERLEAVED, NV12_LUMA, YUV420, YUV422, BAYER = range(5)
UNPACKED, MIPI, GENICAM = range(3)
PATTERNS = ["RGGB", "BGGR", "GRBG", "GBRG"]   # the order of codes 12-15
WIDTHS = [1, 2, 3, 4, 5, 6, 7, 8, 9, 16, 17, 684, 4096]
HEIGHTS = [1, 2, 3, 4, 5, 1023]


def _enumerators():
    with open(os.path.join(ROOT, "include", "rip_cuda.h")) as f:
        text = f.read()
    return {int(code): name for name, code in re.findall(r"\bRIP_FMT_(\w+)\s*=\s*(\d+)", text)}


@pytest.fixture(scope="module")
def table(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("formats") / "formats_probe")
    subprocess.run(["/usr/bin/g++", "-std=c++17", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                    "-I", os.path.join(PKG, "csrc"), os.path.join(ROOT, "tests", "cpp", "formats_probe.cpp"), "-o", exe], check=True)
    out = subprocess.run([exe], check=True, capture_output=True, text=True).stdout
    rows, shapes, absent = {}, {}, []
    for line in out.splitlines():
        kind, *f = line.split()
        if kind == "none":
            absent.append(int(f[0]))
        elif kind == "row":
            rows[int(f[0])] = dict(zip(["name", "layout", "channels", "bgr", "pattern", "bits", "packing", "decodes", "num", "den",
                                        "w_mul", "h_mul", "w_min", "h_min"], [f[1]] + [int(v) for v in f[2:]]))
        else:
            code, w, h, ok, nbytes = map(int, f)
            shapes[code, w, h] = (bool(ok), nbytes)
    return rows, shapes, absent


def _bayer(name):
    """(pattern index, bits, packing) parsed from a Bayer enumerator's name, or None."""
    m = re.fullmatch(r"BAYER_(RGGB|BGGR|GRBG|GBRG)(8|10|12|14|16)(P_MIPI|P_GENICAM)?", name)
    if not m:
        return None
    return PATTERNS.index(m[1]), int(m[2]), {None: UNPACKED, "P_MIPI": MIPI, "P_GENICAM": GENICAM}[m[3]]


def _expected(name, w, h):
    """(accepted, bytes per frame) of a W x H frame, as include/rip_cuda.h documents each format."""
    px = w * h
    interleaved = {"GRAY8": 1, "RGB8": 3, "BGR8": 3, "RGBA8": 4, "BGRA8": 4}
    if name in interleaved:
        return True, px * interleaved[name]
    if name == "NV12":   # the luma plane, then W*H/2 bytes of chroma; H even
        return h % 2 == 0, px * 3 // 2
    if name in ("NV12_COLOR", "I420"):   # the same sizes; W and H even
        return w % 2 == 0 and h % 2 == 0, px * 3 // 2
    if name in ("YUYV", "UYVY"):   # 2*W bytes per row; W even, any H
        return w % 2 == 0, px * 2
    _, bits, packing = _bayer(name)
    if packing == UNPACKED:   # one byte (8 bits) or one 16-bit word per sample; W >= 3 and H >= 3 of any parity
        return w >= 3 and h >= 3, px * (1 if bits == 8 else 2)
    per = 4 if bits == 10 else 2   # rows of W*5/4 or W*3/2 bytes: W a multiple of 4 (10-bit) or 2 (12-bit), at least 4; H >= 3
    return w % per == 0 and w >= 4 and h >= 3, px * bits // 8


def test_one_row_per_enumerator(table):
    rows, _, absent = table
    enums = _enumerators()
    assert set(rows) == set(enums)
    assert sorted(absent) == sorted(set(range(-1, 65)) - set(enums))
    assert {0, 2, *range(32, 40), 56, 64, -1} <= set(absent)
    for code, name in enums.items():
        assert rows[code]["name"] == name, code


def test_rows_restate_names(table):
    rows, _, _ = table
    for code, r in rows.items():
        name = r["name"]
        bayer = _bayer(name)
        if bayer:
            layout, channels = BAYER, 3
        elif name in ("GRAY8", "RGB8", "BGR8", "RGBA8", "BGRA8"):
            layout, channels = INTERLEAVED, {"GRAY8": 1, "RGB8": 3, "BGR8": 3}.get(name, 4)
        else:
            layout, channels = {"NV12": (NV12_LUMA, 1), "NV12_COLOR": (YUV420, 3), "I420": (YUV420, 3),
                                "YUYV": (YUV422, 3), "UYVY": (YUV422, 3)}[name]
        assert (r["layout"], r["channels"]) == (layout, channels), name
        assert r["bgr"] == name.startswith("BGR"), name
        assert r["decodes"] == (layout not in (INTERLEAVED, NV12_LUMA)), name
        assert (r["pattern"], r["bits"], r["packing"]) == (bayer or (-1, 0, UNPACKED)), name


def test_shapes_and_bytes(table):
    rows, shapes, _ = table
    bad = []
    for code, r in rows.items():
        for w in WIDTHS:
            for h in HEIGHTS:
                ok, nbytes = shapes[code, w, h]
                want_ok, want_bytes = _expected(r["name"], w, h)
                if ok != want_ok or (ok and nbytes != want_bytes):
                    bad.append((r["name"], w, h, ok, nbytes, want_ok, want_bytes))
    assert not bad, bad[:10]
