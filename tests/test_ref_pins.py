"""Pins that tie the oracle (and the product's host-side generator) to the REFERENCE itself rather than to values
the oracle wrote:

* Gaussian weights: tests/golden/ref_weights.json holds the float32 bit patterns produced by the reference's own
  Controller::_GenerateGausianKernel (src/GaussianBlur/src/Controller.cpp:342-362 of the reference), compiled from
  the reference's sources as oracle/_ref and recorded by tools/make_ref_weights.py.
* Blur: a second, independently written float32 restatement of PerformCPU's accumulation
  (/root/reference/src/GaussianBlur/GaussianBlur.cpp:236-258) in numpy -- separate code, separate language -- must agree
  with the C oracle, and the same loop with the taps visited in a different order must NOT (so the check is sensitive
  to tap order, fused multiply-adds and double accumulation).
"""
import ctypes as C
import json
import os

import numpy as np
import pytest

import rip_b200 as rip

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def ref_weights():
    with open(os.path.join(GOLDEN, "ref_weights.json")) as f:
        return json.load(f)["cases"]


def test_weights_equal_the_reference_generator_bit_for_bit(oracle, ref_weights):
    assert {"k5_s1.0", "k5_s1.5", "k17_s6.0"} <= set(ref_weights)
    for case in ref_weights.values():
        k, s = case["ksize"], case["sigma"]
        want = np.array(case["bits"], np.uint32).reshape(k, k)
        assert np.array_equal(oracle.gauss_weights(k, s).view(np.uint32), want), ("oracle", k, s)
        assert np.array_equal(rip.gauss_weights(k, s).view(np.uint32), want), ("rip_gauss_weights", k, s)


def _blur_numpy(img, w, order="ky-major"):
    """GaussianBlur.cpp:236-258 restated with numpy float32 scalars: acc starts at 0.0f, one rounded product and one
    rounded add per tap, clamp-to-edge coordinates, (uchar) of the clamped sum.  Vectorised over pixels only -- the tap
    sequence is the Python loop."""
    k = w.shape[0]
    r = k // 2
    h, wd = img.shape[:2]
    pad = np.pad(img, ((r, r), (r, r)) + ((0, 0),) * (img.ndim - 2), mode="edge").astype(np.float32)
    acc = np.zeros(img.shape, np.float32)
    taps = [(ky, kx) for ky in range(k) for kx in range(k)]
    if order == "kx-major":
        taps = [(ky, kx) for kx in range(k) for ky in range(k)]
    elif order == "reversed":
        taps = taps[::-1]
    for ky, kx in taps:
        prod = (pad[ky:ky + h, kx:kx + wd] * np.float32(w[ky, kx])).astype(np.float32)
        acc = (acc + prod).astype(np.float32)
    return np.clip(acc, 0.0, 255.0).astype(np.uint8)  # (truncation: values are >= 0)


@pytest.mark.parametrize("k,sigma", [(5, 1.0), (5, 1.5), (17, 6.0)])
def test_blur_oracle_equals_an_independent_float32_loop(oracle, k, sigma):
    rng = np.random.default_rng(77 + k)
    img = rng.integers(0, 256, (96, 128, 4), dtype=np.uint8)
    w = oracle.gauss_weights(k, sigma)
    assert np.array_equal(oracle.blur(img, k, weights=w), _blur_numpy(img, w))


def _staircase(block=12):
    """16 x 16 blocks of constant level 0..255: the interior of every block has a constant 5x5 window, whose sum
    v * (w0 + w1 + ...) sits within a few ulps of the integer v -- so the truncated result depends on every rounding."""
    lv = np.arange(256, dtype=np.uint8).reshape(16, 16)
    return np.kron(lv, np.ones((block, block), np.uint8))


def test_blur_kat_is_sensitive_to_tap_order_and_precision(oracle):
    """A KAT that can fail: on near-integer sums the reference's ky-major / kx-minor float32 sequence, the same taps
    kx-major, reversed, and a double accumulation all truncate differently somewhere; the oracle must reproduce the
    first one exactly (weights: an asymmetric normalised 5x5 kernel and the reference's sigma 1.0 / 1.5 kernels)."""
    img = _staircase()
    rng = np.random.default_rng(5)
    wa = rng.uniform(0.2, 1.0, (5, 5)).astype(np.float32)
    wa = (wa / wa.sum(dtype=np.float32)).astype(np.float32)
    differs = 0
    for w in (wa, oracle.gauss_weights(5, 1.0), oracle.gauss_weights(5, 1.5)):
        want = _blur_numpy(img, w)
        assert np.array_equal(oracle.blur(img, 5, weights=w), want)
        pad = np.pad(img, 2, mode="edge").astype(np.float64)
        acc = np.zeros(img.shape, np.float64)
        for ky in range(5):
            for kx in range(5):
                acc += pad[ky:ky + img.shape[0], kx:kx + img.shape[1]] * float(w[ky, kx])
        variants = [_blur_numpy(img, w, "kx-major"), _blur_numpy(img, w, "reversed"), np.clip(acc, 0, 255).astype(np.uint8)]
        differs += sum(int(not np.array_equal(v, want)) for v in variants)
    assert differs >= 3, "the staircase image no longer separates tap orders: the KAT has lost its teeth"


def test_blur_flat_255_sigma15_is_254_sigma10_is_255(oracle):
    """The reference's own weights do not sum to 1 in float32: with sigma 1.5 (GaussianBlur.cpp:16) a flat 255 image
    comes out 254, with sigma 1.0 it stays 255 -- both through the oracle and through the independent loop."""
    flat = np.full((12, 12), 255, np.uint8)
    for sigma, v in ((1.5, 254), (1.0, 255)):
        w = oracle.gauss_weights(5, sigma)
        assert int(oracle.blur(flat, 5, weights=w).max()) == v == int(_blur_numpy(flat, w).max())
        assert int(oracle.blur(flat, 5, weights=w).min()) == v


def test_oracle_ref_library_is_test_infrastructure_only():
    """Nothing in the product links or loads oracle/_ref."""
    pkg = os.path.join(os.path.dirname(GOLDEN), "..", "opencl-development-real-time-image-processing_b200")
    for root, _, files in os.walk(pkg):
        for fn in files:
            if fn.endswith((".cu", ".cuh", ".cpp", ".hpp", ".h", ".py")):
                with open(os.path.join(root, fn), errors="replace") as f:
                    txt = f.read()
                assert "librip_ref_weights" not in txt and "oracle/_ref" not in txt, fn
