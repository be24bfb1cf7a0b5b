"""ORACLE — TEST INFRASTRUCTURE ONLY.  Never imported by the product path.

NumPy restatement of OpenCV's `cv2.Canny(img, low, high)` with the arguments the reference uses
(apertureSize=3, L2gradient=False) on an 8-bit 3-channel HWC image, i.e. the edge map of
the reference's src/image_prep.py:6-12 before it is replicated to three channels.  Integer arithmetic throughout, so
the result is exact, and it depends on neither cv2 nor scipy (tests compare it against cv2 where cv2 is installed,
and against tests/golden/canny_cv2.pt everywhere).

  1. thresholds: floor() each, swap if low > high (gradient magnitudes lie in [0, 2040])
  2. per channel 3x3 Sobel dx (right - left, weights 1,2,1) and dy (bottom - top), replicated border
  3. per pixel the channel with the largest |dx| + |dy| (first channel on a tie) supplies mag, dx, dy
  4. non-maximum suppression in fixed point (tan 22.5 deg ~ 13573 / 2^15) with mag = 0 outside the image
  5. candidate: kept and mag > low; strong: candidate and mag > high
  6. hysteresis: 255 for every candidate 8-connected (through candidates) to a strong one, else 0
"""
from __future__ import annotations

import math
from collections import deque
from typing import Tuple

import numpy as np


def canny_thresholds(low: float, high: float) -> Tuple[int, int]:
    """The integer thresholds cv2.Canny compares against (floored, ordered)."""
    if not (math.isfinite(low) and math.isfinite(high)):
        raise ValueError("Canny thresholds must be finite")
    lo, hi = math.floor(low), math.floor(high)
    if lo > hi:
        lo, hi = hi, lo
    return max(-1, min(lo, 2041)), max(-1, min(hi, 2041))


def canny_classes(img_hwc_u8: np.ndarray, low: float, high: float) -> np.ndarray:
    """Steps 1-5: [H, W] uint8, 0 = not a candidate, 1 = weak candidate, 2 = strong candidate."""
    img = np.asarray(img_hwc_u8)
    if img.dtype != np.uint8 or img.ndim != 3 or img.shape[2] != 3:
        raise ValueError("expected an [H, W, 3] uint8 image")
    lo, hi = canny_thresholds(low, high)
    H, W, _ = img.shape
    p = np.pad(img.astype(np.int32), ((1, 1), (1, 1), (0, 0)), mode="edge")
    col = lambda c: p[0:H, c:c + W] + 2 * p[1:H + 1, c:c + W] + p[2:H + 2, c:c + W]     # vertical 1,2,1 sums
    row = lambda r: p[r:r + H, 0:W] + 2 * p[r:r + H, 1:W + 1] + p[r:r + H, 2:W + 2]     # horizontal 1,2,1 sums
    dx3, dy3 = col(2) - col(0), row(2) - row(0)
    mag3 = np.abs(dx3) + np.abs(dy3)
    ch = np.argmax(mag3, axis=2)[..., None]                       # first maximum wins ties
    dx = np.take_along_axis(dx3, ch, 2)[..., 0].astype(np.int64)
    dy = np.take_along_axis(dy3, ch, 2)[..., 0].astype(np.int64)
    m = np.take_along_axis(mag3, ch, 2)[..., 0].astype(np.int64)
    mp = np.pad(m, 1)                                             # zero magnitude outside the image
    nb = lambda oy, ox: mp[1 + oy:1 + oy + H, 1 + ox:1 + ox + W]
    ax, ay = np.abs(dx), np.abs(dy) << 15
    tg22 = ax * 13573
    tg67 = tg22 + (ax << 16)
    pos = (dx ^ dy) >= 0                                          # s = +1
    keep_h = (m > nb(0, -1)) & (m >= nb(0, 1))
    keep_v = (m > nb(-1, 0)) & (m >= nb(1, 0))
    keep_d = np.where(pos, (m > nb(-1, -1)) & (m > nb(1, 1)), (m > nb(-1, 1)) & (m > nb(1, -1)))
    keep = np.where(ay < tg22, keep_h, np.where(ay > tg67, keep_v, keep_d))
    cand = keep & (m > lo)
    return (cand.astype(np.uint8) + (cand & (m > hi)).astype(np.uint8))


def canny_u8(img_hwc_u8: np.ndarray, low: float, high: float) -> np.ndarray:
    """cv2.Canny(img, low, high) replicated to three channels: [H, W, 3] uint8 in {0, 255}."""
    cls = canny_classes(img_hwc_u8, low, high)
    H, W = cls.shape
    Wp = W + 2                                                    # flat indices into the zero-padded class map
    todo = bytearray(np.pad(cls, 1).tobytes())                    # non-zero: candidate not reached yet
    done = bytearray(len(todo))
    offs = (-Wp - 1, -Wp, -Wp + 1, -1, 1, Wp - 1, Wp, Wp + 1)
    q = deque(int(p) for p in np.flatnonzero(np.pad(cls, 1) == 2))   # flood fill from the strong pixels, as cv2 does
    for p in q:
        todo[p], done[p] = 0, 255
    while q:
        p = q.popleft()
        for o in offs:
            n = p + o
            if todo[n]:
                todo[n], done[n] = 0, 255
                q.append(n)
    out = np.frombuffer(bytes(done), np.uint8).reshape(H + 2, Wp)[1:-1, 1:-1]
    return np.repeat(out[..., None], 3, axis=2)


def serpentine_image() -> np.ndarray:
    """512x512 stress image: one 4-px band snaking over the whole image, a single high-contrast spot at its start.  At
    thresholds (100, 200) its edge map is one 8-connected component of 62,762 pixels of which 22 are strong."""
    img = np.full((512, 512, 3), 100, np.uint8)
    for k, y in enumerate(range(4, 504, 8)):
        img[y:y + 4, 8:504] = 130                                 # 4-px band
        x0 = 500 if k % 2 == 0 else 8
        img[y:y + 12, x0:x0 + 4] = 130                            # connector to the next band, alternating right / left
    img[4:8, 8:16] = 200                                          # the only high-contrast spot
    return img


def blurred_noise(seed: int, H: int, W: int) -> np.ndarray:
    """Seeded photo-like test input: uniform noise, box-blurred (integer arithmetic, platform independent)."""
    rng = np.random.default_rng(seed)
    x = rng.integers(0, 256, size=(H + 4, W + 4, 3), dtype=np.int64)
    s = sum(x[dy:dy + H, dx:dx + W] for dy in range(5) for dx in range(5))
    return ((s + 12) // 25).astype(np.uint8)
