"""Measures the device Canny (Engine.canny_u8) and the photo -> edges -> image path; prints the GPU's name and power limit
beside the numbers and one JSON line at the end.

1. canny_u8 device time: CUDA events around >= 200 back-to-back calls after a warm-up, at batch 8 x 512^2 and 1 x 720x1280.
   The inputs (6 MB at batch 8) stay resident in the 126 MB L2 across calls, so this is the warm-cache time.  Achieved
   bytes per second count the algorithmic minimum of 6 bytes per pixel (3 in, 3 out).
2. Photo to image at SD-Turbo width, bf16, batch 8, 512^2, on seeded uniform noise blurred with a Gaussian of sigma 1.5
   (photo-like edge densities; union-find work grows with the density, so it is reported):
   GPU arm   host photo -> H2D -> canny_u8 -> forward_u8 -> D2H
   host arm  cv2.Canny per image on the host -> H2D -> forward_u8 -> D2H   (only when cv2 imports)

Usage: python tests/gpu_canny_bench.py [--reps 200] [--steps 20] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "oracle"), os.path.join(ROOT, "img2img-turbo_b200")]


def blurred_photos(B, H, W, sigma=1.5, seed=0):
    """uint8 [B,H,W,3]: uniform noise through a separable Gaussian (radius 5, reflected border), rounded."""
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(B * 3, 1, H, W, generator=g) * 255
    r = 5
    k = torch.exp(-torch.arange(-r, r + 1, dtype=torch.float64) ** 2 / (2 * sigma * sigma))
    k = (k / k.sum()).float()
    x = F.conv2d(F.pad(x, (r, r, 0, 0), mode="reflect"), k.view(1, 1, 1, -1))
    x = F.conv2d(F.pad(x, (0, 0, r, r), mode="reflect"), k.view(1, 1, -1, 1))
    return x.round().clamp(0, 255).to(torch.uint8).view(B, 3, H, W).permute(0, 2, 3, 1).contiguous()


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def canny_device_ms(eng, x, reps):
    out = torch.empty_like(x)
    for _ in range(10):
        eng.canny_u8(x, 100, 200, out=out)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        eng.canny_u8(x, 100, 200, out=out)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gpu_canny_bench needs a CUDA device")
    from pix2pix_turbo import Pix2Pix_Turbo
    info = gpu_info()
    print("gpu (name, power limit):", info, flush=True)
    m = Pix2Pix_Turbo()
    m.set_eval()
    m.to(torch.bfloat16)
    eng = m._get_engine()
    res = {"gpu": info, "canny": []}
    for B, H, W in ((8, 512, 512), (1, 720, 1280)):
        x = blurred_photos(B, H, W, seed=1).cuda()
        ms, edges = canny_device_ms(eng, x, max(a.reps, 200))
        n = B * H * W
        row = {"batch": B, "H": H, "W": W, "ms": ms, "edge_density": (edges[..., 0] > 0).float().mean().item(),
               "GBps_at_6B_per_px": 6 * n / (ms * 1e-3) / 1e9, "reps": max(a.reps, 200)}
        res["canny"].append(row)
        print("canny_u8", row, flush=True)

    # photo -> image, batch 8 x 512^2, bf16
    B, S, prompt = 8, 512, "a photo"
    photos = blurred_photos(B, S, S, seed=2).pin_memory()
    host_out = torch.empty(B, S, S, 3, dtype=torch.uint8).pin_memory()
    eps = torch.randn(B, 4, S // 8, S // 8, generator=torch.Generator().manual_seed(3)).to(torch.bfloat16).cuda()

    def loop(step):
        with torch.no_grad():
            for _ in range(3):
                host_out.copy_(step(), non_blocking=True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(a.steps):
                host_out.copy_(step(), non_blocking=True)
                torch.cuda.synchronize()
            return B * a.steps / (time.perf_counter() - t0)

    gpu_step = lambda: m.forward_u8(m.canny_u8(photos.cuda(non_blocking=True)), prompt, eps=eps)
    res["photo_to_image"] = {"batch": B, "size": S, "dtype": "bf16", "steps": a.steps, "canny_thresholds": [100, 200],
                             "edge_density": (m.canny_u8(photos)[..., 0] > 0).float().mean().item(),
                             "gpu_arm_img_per_s": loop(gpu_step)}
    try:
        import cv2
    except ImportError:
        cv2 = None
    if cv2 is None:
        print("host arm: not measured (cv2 does not import here)")
        res["photo_to_image"]["host_arm_img_per_s"] = None
    else:
        pin = torch.empty(B, S, S, 3, dtype=torch.uint8).pin_memory()
        np_photos = photos.numpy()

        def host_step():
            e = np.stack([cv2.Canny(p, 100, 200) for p in np_photos])
            pin.copy_(torch.from_numpy(np.repeat(e[..., None], 3, axis=3)))
            return m.forward_u8(pin.cuda(non_blocking=True), prompt, eps=eps)
        res["photo_to_image"]["host_arm_img_per_s"] = loop(host_step)
        res["photo_to_image"]["cv2"] = cv2.__version__
        res["photo_to_image"]["host_cpu_threads"] = cv2.getNumThreads()
    print("photo_to_image", res["photo_to_image"], flush=True)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
