"""The Canny oracle (oracle/canny_oracle.py) against OpenCV: the stored cv2.Canny fixture everywhere, a live cv2.Canny where
OpenCV is installed.  The device kernels are checked against this oracle in tests/test_gpu_canny.py."""
import math
import os

import numpy as np
import pytest
import torch

import canny_oracle as CO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "canny_cv2.pt")


def golden_cases():
    """(input image, low, high, cv2 edge map [H, W] uint8) of every case in tests/golden/canny_cv2.pt."""
    g = torch.load(GOLDEN)
    out = []
    for c in g["cases"]:
        H, W = c["H"], c["W"]
        img = CO.serpentine_image() if c["kind"] == "serpentine" else CO.blurred_noise(c["seed"], H, W)
        edges = np.unpackbits(c["bits"].numpy(), count=H * W).reshape(H, W) * np.uint8(255)
        out.append((img, c["low"], c["high"], edges))
    return out


def test_oracle_matches_stored_cv2_output():
    cases = golden_cases()
    assert len(cases) == 13 and os.path.getsize(GOLDEN) < 200_000
    for img, lo, hi, edges in cases:
        got = CO.canny_u8(img, lo, hi)
        assert got.shape == img.shape and got.dtype == np.uint8
        assert (got == edges[..., None]).all(), (img.shape, lo, hi, int((got[..., 0] != edges).sum()))


def test_serpentine_is_one_long_component():
    cls = CO.canny_classes(CO.serpentine_image(), 100, 200)
    edges = CO.canny_u8(CO.serpentine_image(), 100, 200)[..., 0]
    assert int((cls == 2).sum()) == 22
    assert int((edges > 0).sum()) == int((cls > 0).sum()) == 62762


def test_thresholds_are_floored_and_ordered():
    assert CO.canny_thresholds(100.7, 200.2) == (100, 200)
    assert CO.canny_thresholds(200, 100) == (100, 200)
    assert CO.canny_thresholds(-0.5, 1e9) == (-1, 2041)
    for bad in (math.nan, math.inf, -math.inf):
        with pytest.raises(ValueError):
            CO.canny_thresholds(bad, 200)


def _live_inputs():
    rng = np.random.default_rng(7)
    out = []
    for i in range(24):
        H, W = (int(v) for v in rng.integers(1, 160, 2))
        img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8) if i % 3 == 0 else CO.blurred_noise(100 + i, H, W)
        lo, hi = [(100, 200), (200, 100), (100.7, 200.2), (0, 0), (255, 255), (10.5, 250.9)][i % 6]
        out.append((img, lo, hi))
    flat = np.zeros((9, 11, 3), np.uint8)
    out += [(flat, 100, 200), (flat, -5, -1), (CO.serpentine_image(), 100, 200), (CO.serpentine_image(), 30, 31)]
    return out


def test_oracle_matches_live_cv2():
    cv2 = pytest.importorskip("cv2")
    for img, lo, hi in _live_inputs():
        ref = cv2.Canny(np.ascontiguousarray(img), lo, hi)
        got = CO.canny_u8(img, lo, hi)
        assert (got == ref[..., None]).all(), (img.shape, lo, hi, int((got[..., 0] != ref).sum()))
