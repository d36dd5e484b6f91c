"""CPU-side checks of the drop-in boundary: the C-ABI library builds, loads and exports every
symbol include/rip_cuda.h declares; host-only entry points behave; compute entry points fail loudly
(no CPU fallback) when there is no GPU."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import rip_b200 as rip

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_is_built_in_tree():
    import __graft_entry__ as g
    g.build()
    assert os.path.exists(rip.LIB_PATH)
    assert os.path.dirname(rip.LIB_PATH).startswith(ROOT)


def test_every_declared_symbol_is_exported():
    hdr = open(os.path.join(ROOT, "include", "rip_cuda.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(rip_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    L = rip.lib()
    for name in sorted(declared):
        assert hasattr(L, name), f"{name} declared in rip_cuda.h but not exported"
    assert declared == set(rip.ABI_SYMBOLS), declared ^ set(rip.ABI_SYMBOLS)
    assert L.rip_abi_version() == 1


def test_sass_is_sm_100a():
    import shutil
    import subprocess
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([cuobjdump, "-lelf", rip.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out, out


def test_weights_generator_matches_oracle(oracle):
    # product generator (host C++ in librip_cuda) vs the oracle's restatement of Controller.cpp:352-372
    for k, s in ((5, 1.0), (5, 1.5), (3, 0.8), (7, 2.0), (17, 6.0), (31, 9.5)):
        assert np.array_equal(rip.gauss_weights(k, s), oracle.gauss_weights(k, s)), (k, s)


def test_weights_generator_rejects_bad_arguments():
    for k, s in ((4, 1.0), (0, 1.0), (33, 1.0), (5, 0.0), (5, -1.0)):
        with pytest.raises(rip.RipError):
            rip.gauss_weights(k, s)


def test_fused_needs_no_workspace():
    """rip_fused runs every shape and kernel size as one kernel: the workspace query answers 0 and still validates."""
    for w, in_rows, n, k in ((3840, 2160, 32, 5), (683, 1023, 1, 17), (75, 75, 4, 3), (1, 1, 1, 31), (1922, 7, 2, 9)):
        assert rip.fused_workspace_bytes(w, in_rows, n, k) == 0, (w, in_rows, n, k)
    for w, in_rows, n in ((0, 16, 1), (16, 0, 1), (16, 16, 0), (-4, 16, 1)):
        with pytest.raises(rip.RipError):
            rip.fused_workspace_bytes(w, in_rows, n, 5)


@pytest.mark.skipif(rip.device_count() > 0, reason="only meaningful on a box without a GPU")
def test_compute_fails_loudly_without_gpu():
    with pytest.raises(rip.RipError, match="no CUDA device|no CPU fallback"):
        rip.Context([0])
    with pytest.raises(rip.RipError):
        rip.DeviceBuffer(16)
    with pytest.raises(rip.RipError):
        rip.gray_dev(16, 32, 4, 4, 1, rip.FMT_RGB8)


def test_product_never_links_the_oracle():
    # the product library and package sources must not reference the oracle
    import subprocess
    out = subprocess.run(["ldd", rip.LIB_PATH], capture_output=True, text=True).stdout
    assert "oracle" not in out
    pkg = rip.PKG_DIR
    for dirpath, _, files in os.walk(pkg):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh", ".h", ".hpp", ".cpp")):
                txt = open(os.path.join(dirpath, fn), errors="replace").read()
                assert "rip_oracle" not in txt and "import oracle" not in txt, os.path.join(dirpath, fn)


def test_numa_binding_helper_is_harmless_without_a_gpu():
    """bind_host_to_device_numa() must never raise: it returns {} when the device or the topology cannot be read."""
    import os
    import rip_b200 as rip
    before = os.sched_getaffinity(0)
    info = rip.bind_host_to_device_numa(0)
    assert isinstance(info, dict)
    if not info:
        assert os.sched_getaffinity(0) == before
    else:
        os.sched_setaffinity(0, before)
