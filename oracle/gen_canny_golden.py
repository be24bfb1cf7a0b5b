"""Generates tests/golden/canny_cv2.pt: cv2.Canny edge maps of seeded synthetic images, so machines without OpenCV can still
check the Canny oracle and the device kernels against OpenCV itself.

Each case stores how to rebuild its input (canny_oracle.blurred_noise(seed, H, W) or the serpentine image), the thresholds,
and cv2.Canny's [H, W] output bit-packed with np.packbits (row-major, 255 -> 1).  Needs cv2.   Run:
    python oracle/gen_canny_golden.py
"""
import os
import sys

import cv2
import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import canny_oracle as CO  # noqa: E402

SIZES = [(37, 53), (64, 96), (256, 256)]
THRESHOLDS = [(100.0, 200.0), (50.0, 120.0), (10.0, 250.0), (100.7, 200.2)]


def cases():
    """(kind, seed, H, W, low, high) of every fixture case; tests rebuild the inputs from these."""
    out = [("noise", 11 + i, H, W, lo, hi) for i, (H, W) in enumerate(SIZES) for lo, hi in THRESHOLDS]
    out.append(("serpentine", 0, 512, 512, 100.0, 200.0))
    return out


def make_input(kind, seed, H, W):
    return CO.serpentine_image() if kind == "serpentine" else CO.blurred_noise(seed, H, W)


def main():
    rec = []
    for kind, seed, H, W, lo, hi in cases():
        edges = cv2.Canny(make_input(kind, seed, H, W), lo, hi)
        rec.append({"kind": kind, "seed": seed, "H": H, "W": W, "low": lo, "high": hi,
                    "bits": torch.from_numpy(np.packbits(edges.reshape(-1) > 0))})
    path = os.path.join(ROOT, "tests", "golden", "canny_cv2.pt")
    torch.save({"cv2_version": cv2.__version__, "cases": rec}, path)
    print(f"wrote {path}: {len(rec)} cases, {os.path.getsize(path)} bytes, cv2 {cv2.__version__}")


if __name__ == "__main__":
    main()
