"""Small Canny workload for compute-sanitizer (memcheck / racecheck / synccheck): a batch of two 512x512 photo-like images
and the serpentine stress image, each checked against the oracle.  Usage:
    compute-sanitizer --tool memcheck python tests/sanitize_canny.py
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "oracle"), os.path.join(ROOT, "img2img-turbo_b200")]
import canny_oracle as CO  # noqa: E402
import i2it  # noqa: E402
import weights as W  # noqa: E402


def main():
    eng = i2it.Engine(torch.bfloat16, i2it.PIX2PIX, cfg=W.TINY)
    for imgs in ([CO.blurred_noise(1, 512, 512), CO.blurred_noise(2, 512, 512)], [CO.serpentine_image()]):
        out = eng.canny_u8(torch.from_numpy(np.stack(imgs)).cuda(), 100, 200).cpu().numpy()
        for i, img in enumerate(imgs):
            assert (out[i] == CO.canny_u8(img, 100, 200)).all(), i
    torch.cuda.synchronize()
    print("SANITIZE_CANNY_OK")


if __name__ == "__main__":
    main()
