"""B200-native gray / Gaussian / Sobel / fused image path -- Python binding of the C ABI.

The product is `librip_cuda.so` (hand-written sm_100a kernels behind `include/rip_cuda.h`) plus the
C++ host classes in `host/` that mirror the reference's Controller / ProgramHandler / Comparator /
FileHandler.  This module is the ctypes view of that C ABI used by tests, `bench.py` and
`__graft_entry__.py`; it contains no compute of its own and NO CPU fallback: if the CUDA library is
missing or no GPU is present, the compute calls raise.

The package directory name has hyphens, so import it through the `rip_b200` shim at the repo root.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
# RIP_LIB_PATH lets A/B experiments load an alternative build of the same library (tools/ab/*.so)
LIB_PATH = os.environ.get("RIP_LIB_PATH") or os.path.join(_PKG, "librip_cuda.so")

# ---- constants (include/rip_cuda.h) ----
FMT_GRAY8, FMT_RGB8, FMT_RGBA8, FMT_BGR8, FMT_BGRA8, FMT_NV12, FMT_NV12_COLOR = 1, 3, 4, 5, 6, 7, 8
FMT_YUYV, FMT_UYVY, FMT_I420 = 9, 10, 11
# 8-bit Bayer raw frames, named by the sensor's top-left 2x2 (V4L2 SRGGB8 / SBGGR8 / SGRBG8 / SGBRG8, GenICam BayerRG8 / ...)
FMT_BAYER_RGGB8, FMT_BAYER_BGGR8, FMT_BAYER_GRBG8, FMT_BAYER_GBRG8 = 12, 13, 14, 15
# 10- to 16-bit Bayer raw frames, one little-endian uint16 per sample, LSB-aligned (V4L2 SRGGB10 ... SGBRG16, GenICam
# BayerRG10 ... BayerGB16, unpacked); MSB-aligned samples are a 16-bit stream
FMT_BAYER_RGGB10, FMT_BAYER_BGGR10, FMT_BAYER_GRBG10, FMT_BAYER_GBRG10 = 16, 17, 18, 19
FMT_BAYER_RGGB12, FMT_BAYER_BGGR12, FMT_BAYER_GRBG12, FMT_BAYER_GBRG12 = 20, 21, 22, 23
FMT_BAYER_RGGB14, FMT_BAYER_BGGR14, FMT_BAYER_GRBG14, FMT_BAYER_GBRG14 = 24, 25, 26, 27
FMT_BAYER_RGGB16, FMT_BAYER_BGGR16, FMT_BAYER_GRBG16, FMT_BAYER_GBRG16 = 28, 29, 30, 31
# the formats whose host arrays are uint16 (every other format takes uint8)
FMTS_U16 = frozenset(range(FMT_BAYER_RGGB10, FMT_BAYER_GBRG16 + 1))
# packed 10- and 12-bit Bayer raw frames, rows of W*5/4 or W*3/2 bytes with no padding: MIPI CSI-2 RAW10 / RAW12 (V4L2
# SRGGB10P / SRGGB12P ..., libcamera *10_CSI2P / *12_CSI2P) and GenICam's LSB-first bit streams (BayerRG10p / BayerRG12p ...)
FMT_BAYER_RGGB10P_MIPI, FMT_BAYER_BGGR10P_MIPI, FMT_BAYER_GRBG10P_MIPI, FMT_BAYER_GBRG10P_MIPI = 40, 41, 42, 43
FMT_BAYER_RGGB12P_MIPI, FMT_BAYER_BGGR12P_MIPI, FMT_BAYER_GRBG12P_MIPI, FMT_BAYER_GBRG12P_MIPI = 44, 45, 46, 47
FMT_BAYER_RGGB10P_GENICAM, FMT_BAYER_BGGR10P_GENICAM, FMT_BAYER_GRBG10P_GENICAM, FMT_BAYER_GBRG10P_GENICAM = 48, 49, 50, 51
FMT_BAYER_RGGB12P_GENICAM, FMT_BAYER_BGGR12P_GENICAM, FMT_BAYER_GRBG12P_GENICAM, FMT_BAYER_GBRG12P_GENICAM = 52, 53, 54, 55
# the packed formats: their host arrays are uint8 (N, H, row_bytes), and W is derived from row_bytes
FMTS_PACKED = frozenset(range(FMT_BAYER_RGGB10P_MIPI, FMT_BAYER_GBRG12P_GENICAM + 1))


def packed_bits(fmt: int) -> int:
    """Bits per sample of a packed Bayer format: 10 or 12."""
    assert fmt in FMTS_PACKED, f"format {fmt} is not a packed Bayer format"
    return 10 if (fmt - FMT_BAYER_RGGB10P_MIPI) % 8 < 4 else 12


OP_GRAY, OP_EDGE, OP_GAUSSIAN, OP_FUSED = 0, 1, 2, 3
GRAY_OUT_U8, GRAY_OUT_RGBA = 0, 1
MAX_KSIZE = 31
# elements per pixel of the host array's last axis; 1 for the planar formats, whose frames are (H*3/2, W) arrays, and for Bayer
# frames, (H, W) arrays (uint16 for 10 to 16 bits; packed: (H, row_bytes) uint8).  YUYV and UYVY are (H, W, 2): the CV_8UC2
# Mat that V4L2 capture returns with CAP_PROP_CONVERT_RGB off.
CHANNELS = {FMT_GRAY8: 1, FMT_RGB8: 3, FMT_BGR8: 3, FMT_RGBA8: 4, FMT_BGRA8: 4, FMT_NV12: 1, FMT_NV12_COLOR: 1,
            FMT_YUYV: 2, FMT_UYVY: 2, FMT_I420: 1,
            FMT_BAYER_RGGB8: 1, FMT_BAYER_BGGR8: 1, FMT_BAYER_GRBG8: 1, FMT_BAYER_GBRG8: 1,
            **{f: 1 for f in FMTS_U16}, **{f: 1 for f in FMTS_PACKED}}

# every symbol include/rip_cuda.h declares (checked by tests/test_abi.py)
ABI_SYMBOLS = [
    "rip_abi_version", "rip_last_error_string", "rip_device_count", "rip_device_name", "rip_device_get_info",
    "rip_device_pci_bus_id",
    "rip_ctx_create", "rip_ctx_destroy", "rip_ctx_device_count", "rip_ctx_device",
    "rip_module_load", "rip_module_release", "rip_kernel_get", "rip_kernel_release", "rip_kernel_op",
    "rip_stream_create", "rip_stream_destroy", "rip_stream_sync", "rip_device_sync",
    "rip_event_create", "rip_event_destroy", "rip_event_record", "rip_event_sync", "rip_event_elapsed_ns",
    "rip_malloc_device", "rip_free_device", "rip_malloc_pinned", "rip_free_pinned",
    "rip_memcpy_h2d_async", "rip_memcpy_d2h_async", "rip_memset_device_async",
    "rip_gauss_weights", "rip_gray", "rip_convert", "rip_gauss", "rip_sobel", "rip_fused", "rip_fused_workspace_bytes",
    "rip_launch_count", "rip_debug_slow_path_stats", "rip_debug_selftest", "rip_debug_set_option",
    "rip_out_bytes_per_frame", "rip_process_host", "rip_process_host_banded", "rip_shard_frames", "rip_band_rows",
    "rip_submit", "rip_ticket_done", "rip_collect", "rip_host_register", "rip_host_unregister",
]


class RipError(RuntimeError):
    pass


class OpDesc(C.Structure):
    _fields_ = [("op", C.c_int), ("in_format", C.c_int), ("gray_out", C.c_int), ("ksize", C.c_int),
                ("weights", C.POINTER(C.c_float))]


class DeviceInfo(C.Structure):
    _fields_ = [("name", C.c_char * 128), ("sm_count", C.c_int), ("cc_major", C.c_int), ("cc_minor", C.c_int),
                ("clock_khz", C.c_int), ("l2_bytes", C.c_int), ("global_mem_bytes", C.c_size_t),
                ("smem_per_sm_bytes", C.c_size_t)]


_lib = None


def lib() -> C.CDLL:
    """Load librip_cuda.so; raises if it has not been built (there is no fallback path)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RipError(f"{LIB_PATH} is missing: build it with `python {os.path.join(_PKG, 'build.py')}` "
                       "(nvcc, sm_100a).  There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, u8p, f32p, i32p = C.c_void_p, C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_int)
    u64p, szp = C.POINTER(C.c_uint64), C.POINTER(C.c_size_t)
    sig = {
        "rip_abi_version": ([], C.c_int),
        "rip_last_error_string": ([], C.c_char_p),
        "rip_device_count": ([i32p], C.c_int),
        "rip_device_name": ([C.c_int, C.c_char_p, C.c_size_t], C.c_int),
        "rip_device_pci_bus_id": ([C.c_int, C.c_char_p, C.c_size_t], C.c_int),
        "rip_device_get_info": ([C.c_int, C.POINTER(DeviceInfo)], C.c_int),
        "rip_ctx_create": ([i32p, C.c_int, C.POINTER(vp)], C.c_int),
        "rip_ctx_destroy": ([vp], C.c_int),
        "rip_ctx_device_count": ([vp, i32p], C.c_int),
        "rip_ctx_device": ([vp, C.c_int, i32p], C.c_int),
        "rip_module_load": ([vp, C.c_char_p, C.POINTER(vp)], C.c_int),
        "rip_module_release": ([vp], C.c_int),
        "rip_kernel_get": ([vp, C.c_char_p, C.POINTER(vp)], C.c_int),
        "rip_kernel_release": ([vp], C.c_int),
        "rip_kernel_op": ([vp, i32p], C.c_int),
        "rip_stream_create": ([C.c_int, C.POINTER(vp)], C.c_int),
        "rip_stream_destroy": ([C.c_int, vp], C.c_int),
        "rip_stream_sync": ([C.c_int, vp], C.c_int),
        "rip_device_sync": ([C.c_int], C.c_int),
        "rip_event_create": ([C.c_int, C.POINTER(vp)], C.c_int),
        "rip_event_destroy": ([vp], C.c_int),
        "rip_event_record": ([vp, vp], C.c_int),
        "rip_event_sync": ([vp], C.c_int),
        "rip_event_elapsed_ns": ([vp, vp, u64p], C.c_int),
        "rip_malloc_device": ([C.c_int, C.c_size_t, C.POINTER(vp)], C.c_int),
        "rip_free_device": ([C.c_int, vp], C.c_int),
        "rip_malloc_pinned": ([C.c_size_t, C.POINTER(vp)], C.c_int),
        "rip_free_pinned": ([vp], C.c_int),
        "rip_memcpy_h2d_async": ([C.c_int, vp, vp, C.c_size_t, vp], C.c_int),
        "rip_memcpy_d2h_async": ([C.c_int, vp, vp, C.c_size_t, vp], C.c_int),
        "rip_memset_device_async": ([C.c_int, vp, C.c_int, C.c_size_t, vp], C.c_int),
        "rip_gauss_weights": ([C.c_int, C.c_float, f32p], C.c_int),
        "rip_gray": ([C.c_int, vp, u8p, u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int], C.c_int),
        "rip_convert": ([C.c_int, vp, u8p, u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int], C.c_int),
        "rip_gauss": ([C.c_int, vp, u8p, u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, f32p], C.c_int),
        "rip_sobel": ([C.c_int, vp, u8p, u8p, C.c_int, C.c_int, C.c_int, C.c_int], C.c_int),
        "rip_fused": ([C.c_int, vp, u8p, u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, f32p,
                       C.c_int, C.c_int, C.c_int, C.c_int, vp, C.c_size_t], C.c_int),
        "rip_fused_workspace_bytes": ([C.c_int, C.c_int, C.c_int, C.c_int, szp], C.c_int),
        "rip_launch_count": ([u64p], C.c_int),
        "rip_debug_slow_path_stats": ([C.c_int, C.c_int, u64p], C.c_int),
        "rip_debug_selftest": ([C.c_int, u64p, u64p], C.c_int),
        "rip_debug_set_option": ([C.c_char_p, C.c_int], C.c_int),
        "rip_out_bytes_per_frame": ([C.POINTER(OpDesc), C.c_int, C.c_int, szp], C.c_int),
        "rip_process_host": ([vp, C.POINTER(OpDesc), vp, vp, C.c_int, C.c_int, C.c_int, u64p], C.c_int),
        "rip_process_host_banded": ([vp, C.POINTER(OpDesc), vp, vp, C.c_int, C.c_int, u64p], C.c_int),
        "rip_submit": ([vp, C.POINTER(OpDesc), vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(vp)], C.c_int),
        "rip_ticket_done": ([vp, i32p], C.c_int),
        "rip_collect": ([vp, u64p], C.c_int),
        "rip_host_register": ([vp, C.c_size_t], C.c_int),
        "rip_host_unregister": ([vp], C.c_int),
        "rip_shard_frames": ([C.c_int, C.c_int, C.c_int, i32p, i32p], C.c_int),
        "rip_band_rows": ([C.c_int, C.c_int, C.c_int, C.c_int, i32p, i32p, i32p, i32p], C.c_int),
    }
    for name, (args, res) in sig.items():
        fn = getattr(L, name)
        fn.argtypes, fn.restype = args, res
    _lib = L
    return L


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().rip_last_error_string().decode(errors="replace")
        raise RipError(f"{what or 'librip_cuda'} failed (rc={rc}): {msg}")


# ---------------------------------------------------------------------------------------------
# thin helpers
# ---------------------------------------------------------------------------------------------
def device_count() -> int:
    n = C.c_int(0)
    rc = lib().rip_device_count(C.byref(n))
    return n.value if rc == 0 else 0


def device_info(device: int = 0) -> DeviceInfo:
    info = DeviceInfo()
    check(lib().rip_device_get_info(device, C.byref(info)), "rip_device_get_info")
    return info


def bind_host_to_device_numa(device: int = 0) -> dict:
    """Pin the calling process to the CPUs of the NUMA node the GPU hangs off, so that buffers pinned afterwards
    (first touch) and the copy-issuing thread are local to it.  For one-process-per-GPU launchers; returns what it
    did ({} when the topology cannot be read: containers without /sys, single-node hosts)."""
    try:
        buf = C.create_string_buffer(32)
        check(lib().rip_device_pci_bus_id(device, buf, 32), "rip_device_pci_bus_id")
        bdf = buf.value.decode().lower()
        base = f"/sys/bus/pci/devices/{bdf}"
        with open(base + "/numa_node") as f:
            node = int(f.read().strip())
        with open(base + "/local_cpulist") as f:
            spec = f.read().strip()
        cpus = set()
        for part in spec.split(","):
            if not part:
                continue
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if node < 0 or not cpus:
            return {}
        os.sched_setaffinity(0, cpus)
        return {"pci": bdf, "numa_node": node, "cpus": len(cpus)}
    except Exception:
        return {}


def launch_count() -> int:
    v = C.c_uint64(0)
    check(lib().rip_launch_count(C.byref(v)))
    return v.value


def slow_path_stats(enable: bool, device: int = 0) -> int:
    v = C.c_uint64(0)
    check(lib().rip_debug_slow_path_stats(device, int(enable), C.byref(v)), "rip_debug_slow_path_stats")
    return v.value


def set_option(name: str, value: int) -> None:
    """Experiment switch (rip_debug_set_option): e.g. set_option("FUSED_NPX", 4)."""
    check(lib().rip_debug_set_option(name.encode(), int(value)), "rip_debug_set_option")


def selftest(device: int = 0) -> tuple[int, int]:
    c, m = C.c_uint64(0), C.c_uint64(0)
    check(lib().rip_debug_selftest(device, C.byref(c), C.byref(m)), "rip_debug_selftest")
    return c.value, m.value


def shard_frames(n_frames: int, n_parts: int, index: int) -> tuple[int, int]:
    """(first, count) of the contiguous block of frames part `index` of `n_parts` owns (rip_shard_frames)."""
    first, count = C.c_int(), C.c_int()
    check(lib().rip_shard_frames(n_frames, n_parts, index, C.byref(first), C.byref(count)), "rip_shard_frames")
    return first.value, count.value


def band_rows(height: int, n_parts: int, index: int, halo: int) -> tuple[int, int, int, int]:
    """(in_row0, in_rows, out_row0, out_rows) of row band `index` of `n_parts` (rip_band_rows)."""
    v = [C.c_int() for _ in range(4)]
    check(lib().rip_band_rows(height, n_parts, index, halo, *[C.byref(x) for x in v]), "rip_band_rows")
    return tuple(x.value for x in v)


def gauss_weights(ksize: int, sigma: float) -> np.ndarray:
    """The product's own weight generator (host C++; reference Controller.cpp:352-372)."""
    w = np.empty((ksize, ksize), np.float32)
    check(lib().rip_gauss_weights(ksize, C.c_float(sigma), w.ctypes.data_as(C.POINTER(C.c_float))), "rip_gauss_weights")
    return w


def _f32p(a: np.ndarray | None):
    if a is None:
        return C.POINTER(C.c_float)()
    assert a.dtype == np.float32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.POINTER(C.c_float))


class DeviceBuffer:
    """cudaMalloc'ed bytes on one device (rip_malloc_device)."""

    def __init__(self, nbytes: int, device: int = 0):
        self.device, self.nbytes = device, int(nbytes)
        p = C.c_void_p()
        check(lib().rip_malloc_device(device, self.nbytes, C.byref(p)), "rip_malloc_device")
        self.ptr = p.value

    def upload(self, host: np.ndarray, stream=None, offset: int = 0) -> "DeviceBuffer":
        host = np.ascontiguousarray(host)
        assert offset + host.nbytes <= self.nbytes
        check(lib().rip_memcpy_h2d_async(self.device, self.ptr + offset, host.ctypes.data, host.nbytes, stream))
        check(lib().rip_stream_sync(self.device, stream))
        return self

    def download(self, shape, dtype=np.uint8, stream=None, offset: int = 0) -> np.ndarray:
        out = np.empty(shape, dtype)
        assert offset + out.nbytes <= self.nbytes
        check(lib().rip_memcpy_d2h_async(self.device, out.ctypes.data, self.ptr + offset, out.nbytes, stream))
        check(lib().rip_stream_sync(self.device, stream))
        return out

    def free(self):
        if self.ptr:
            lib().rip_free_device(self.device, self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class PinnedBuffer:
    """cudaHostAlloc'ed host memory exposed as a numpy u8 array."""

    def __init__(self, nbytes: int):
        self.nbytes = int(nbytes)
        p = C.c_void_p()
        check(lib().rip_malloc_pinned(self.nbytes, C.byref(p)), "rip_malloc_pinned")
        self.ptr = p.value
        self.array = np.ctypeslib.as_array((C.c_uint8 * self.nbytes).from_address(self.ptr))

    def free(self):
        if self.ptr:
            self.array = None
            lib().rip_free_pinned(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Event:
    def __init__(self, device: int = 0):
        p = C.c_void_p()
        check(lib().rip_event_create(device, C.byref(p)), "rip_event_create")
        self.ptr = p.value

    def record(self, stream=None):
        check(lib().rip_event_record(self.ptr, stream))

    def sync(self):
        check(lib().rip_event_sync(self.ptr))

    def elapsed_ns(self, stop: "Event") -> int:
        ns = C.c_uint64(0)
        check(lib().rip_event_elapsed_ns(self.ptr, stop.ptr, C.byref(ns)))
        return ns.value

    def __del__(self):
        try:
            if self.ptr:
                lib().rip_event_destroy(self.ptr)
        except Exception:
            pass


# ---- device-resident ops on raw device pointers (ints) ----
def gray_dev(d_in: int, d_out: int, w: int, h: int, n: int, fmt: int, out_mode: int = GRAY_OUT_U8, device=0, stream=None):
    """rip_gray: the reference's gray of RGB8 / BGR8 / RGBA8 / BGRA8 frames, or of NV12_COLOR, YUYV, UYVY, I420 or Bayer
    frames (8 to 16 bits, or packed at 10 and 12) decoded in the same kernel."""
    check(lib().rip_gray(device, stream, d_in, d_out, w, h, n, fmt, out_mode), "rip_gray")


def convert_dev(d_in: int, d_out: int, w: int, h: int, n: int, in_fmt: int, out_fmt: int, device=0, stream=None):
    """rip_convert: NV12_COLOR, YUYV, UYVY, I420 or Bayer frames -> RGB8 / BGR8 / RGBA8 / BGRA8 (OpenCV's cvtColor
    arithmetic; Bayer: its default bilinear demosaic, then for 10 to 16 bits convertTo(CV_8U, 1 / 2^(bits - 8)); packed
    samples are unpacked first)."""
    check(lib().rip_convert(device, stream, d_in, d_out, w, h, n, in_fmt, out_fmt), "rip_convert")


def gauss_dev(d_in: int, d_out: int, w: int, h: int, n: int, channels: int, ksize: int, weights: np.ndarray,
              device=0, stream=None):
    weights = np.ascontiguousarray(weights, np.float32)
    check(lib().rip_gauss(device, stream, d_in, d_out, w, h, n, channels, ksize, _f32p(weights)), "rip_gauss")


def sobel_dev(d_in: int, d_out: int, w: int, h: int, n: int, fmt: int, device=0, stream=None):
    check(lib().rip_sobel(device, stream, d_in, d_out, w, h, n, fmt), "rip_sobel")


def fused_workspace_bytes(w: int, in_rows: int, n: int, ksize: int) -> int:
    b = C.c_size_t(0)
    check(lib().rip_fused_workspace_bytes(w, in_rows, n, ksize, C.byref(b)))
    return b.value


def fused_dev(d_in: int, d_out: int, w: int, h: int, n: int, fmt: int, ksize: int, weights: np.ndarray,
              in_row0: int = 0, in_rows: int | None = None, out_row0: int = 0, out_rows: int | None = None,
              d_ws: int | None = None, ws_bytes: int = 0, device=0, stream=None):
    weights = np.ascontiguousarray(weights, np.float32)
    in_rows = h if in_rows is None else in_rows
    out_rows = h if out_rows is None else out_rows
    check(lib().rip_fused(device, stream, d_in, d_out, w, h, n, fmt, ksize, _f32p(weights), in_row0, in_rows,
                          out_row0, out_rows, d_ws, ws_bytes), "rip_fused")


# ---------------------------------------------------------------------------------------------
# host-buffer pipeline (the call the C++ Controller makes): numpy in, numpy out
# ---------------------------------------------------------------------------------------------
class Context:
    """rip_ctx: a set of devices with cached buffers and streams (replaces cl_context + queue)."""

    def __init__(self, devices=None):
        devs = list(devices) if devices is not None else [0]
        arr = (C.c_int * len(devs))(*devs)
        p = C.c_void_p()
        check(lib().rip_ctx_create(arr, len(devs), C.byref(p)), "rip_ctx_create")
        self.ptr, self.devices = p.value, devs

    def close(self):
        if self.ptr:
            lib().rip_ctx_destroy(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _desc(self, op, fmt, gray_out=GRAY_OUT_U8, ksize=0, weights=None):
        d = OpDesc()
        d.op, d.in_format, d.gray_out, d.ksize = op, fmt, gray_out, ksize
        # the descriptor keeps its weights alive: two threads calling process() on one Context must not free each other's
        # weights while the C call reads them
        d.keep_weights = None if weights is None else np.ascontiguousarray(weights, np.float32)
        d.weights = _f32p(d.keep_weights)
        return d

    def _shapes(self, frames: np.ndarray, op, fmt, gray_out, ksize, weights, out):
        a = frames
        if fmt in FMTS_U16:
            assert a.dtype == np.dtype("<u2"), \
                f"format {fmt} (10- to 16-bit Bayer) takes native little-endian uint16 arrays, got {a.dtype.str}"
        else:
            assert a.dtype == np.uint8, f"format {fmt} takes uint8 arrays, got {a.dtype}"
        assert a.flags["C_CONTIGUOUS"]
        cn = CHANNELS[fmt]
        if cn == 1:
            if a.ndim == 2:
                a = a[None]
            n, h, w = a.shape
            if fmt in (FMT_NV12, FMT_NV12_COLOR, FMT_I420):
                assert h % 3 == 0
                h = h * 2 // 3
            elif fmt in FMTS_PACKED:   # the last axis is the row's bytes: 4 pixels in 5 (10-bit) or 2 in 3 (12-bit)
                bits = packed_bits(fmt)
                group = 5 if bits == 10 else 3
                assert w % group == 0, \
                    f"format {fmt} ({bits}-bit packed Bayer) takes rows of a multiple of {group} bytes, got {w}"
                w = w * 8 // bits
        else:
            if a.ndim == 3:
                a = a[None]
            n, h, w, c = a.shape
            assert c == cn, f"format needs {cn} channels, array has {c}"
        d = self._desc(op, fmt, gray_out, ksize, weights)
        ob = C.c_size_t(0)
        check(lib().rip_out_bytes_per_frame(C.byref(d), w, h, C.byref(ob)))
        per = ob.value // (w * h)
        shape = (n, h, w) if per == 1 else (n, h, w, per)
        if out is None:
            out = np.empty(shape, np.uint8)
        assert out.nbytes == ob.value * n and out.flags["C_CONTIGUOUS"]
        squeeze = frames.ndim == (2 if cn == 1 else 3)
        return a, d, n, h, w, shape, out, squeeze

    def process(self, frames: np.ndarray, op: int, fmt: int, *, gray_out=GRAY_OUT_U8, ksize=0, weights=None,
                out: np.ndarray | None = None, banded: bool = False, prof: bool = False):
        """frames: (N, H, W, C) or (H, W, C) / (H, W) u8 host array (pageable or pinned); NV12 / NV12_COLOR / I420:
        (N, H*3/2, W) or (H*3/2, W), the luma plane followed by the chroma planes; YUYV / UYVY: (N, H, W, 2) or (H, W, 2);
        Bayer: (N, H, W) or (H, W), one raw byte per pixel (uint8) for the 8-bit formats, one little-endian uint16 per pixel
        for 10 to 16 bits; packed Bayer: (N, H, row_bytes) or (H, row_bytes) uint8, the row's packed bytes (W*5/4 at 10 bits,
        W*3/2 at 12), W derived from row_bytes.  Every other format takes uint8."""
        a, d, n, h, w, shape, out, squeeze = self._shapes(frames, op, fmt, gray_out, ksize, weights, out)
        pr = (C.c_uint64 * 6)() if prof else None
        if banded:
            assert n == 1
            check(lib().rip_process_host_banded(self.ptr, C.byref(d), a.ctypes.data, out.ctypes.data, w, h, pr),
                  "rip_process_host_banded")
        else:
            check(lib().rip_process_host(self.ptr, C.byref(d), a.ctypes.data, out.ctypes.data, w, h, n, pr),
                  "rip_process_host")
        res = out.reshape(shape)
        if squeeze:
            res = res[0]
        return (res, list(pr)) if prof else res

    def submit(self, frames: np.ndarray, op: int, fmt: int, *, gray_out=GRAY_OUT_U8, ksize=0, weights=None,
               out: np.ndarray | None = None, banded: bool = False, prof: bool = False) -> "Ticket":
        """Asynchronous form of process() (rip_submit): returns at once; Ticket.collect() waits and returns the output.
        `frames` must stay untouched until then."""
        a, d, n, h, w, shape, out, squeeze = self._shapes(frames, op, fmt, gray_out, ksize, weights, out)
        t = C.c_void_p()
        flags = (1 if banded else 0) | (2 if prof else 0)
        check(lib().rip_submit(self.ptr, C.byref(d), a.ctypes.data, out.ctypes.data, w, h, n, flags, C.byref(t)), "rip_submit")
        return Ticket(t.value, a, out, shape, squeeze, prof)


class Ticket:
    """One job in flight (rip_ticket).  Keeps the input and output arrays alive until collect()."""

    def __init__(self, ptr, a, out, shape, squeeze, prof):
        self.ptr, self._in, self._out, self._shape, self._squeeze, self._prof = ptr, a, out, shape, squeeze, prof

    def done(self) -> bool:
        v = C.c_int(0)
        check(lib().rip_ticket_done(self.ptr, C.byref(v)), "rip_ticket_done")
        return bool(v.value)

    def collect(self):
        assert self.ptr, "ticket already collected"
        pr = (C.c_uint64 * 6)() if self._prof else None
        ptr, self.ptr = self.ptr, None
        check(lib().rip_collect(ptr, pr), "rip_collect")
        res = self._out.reshape(self._shape)
        if self._squeeze:
            res = res[0]
        return (res, list(pr)) if self._prof else res

    def __del__(self):
        try:
            if self.ptr:
                lib().rip_collect(self.ptr, None)
        except Exception:
            pass
