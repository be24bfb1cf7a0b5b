"""-m gpu: Canny edge maps on the device (i2it_canny_u8, Engine.canny_u8, Pix2Pix_Turbo.canny_u8) against the integer oracle
(oracle/canny_oracle.py), OpenCV's stored outputs (tests/golden/canny_cv2.pt) and a live cv2.Canny when OpenCV is installed,
bit for bit; then the photo -> edges -> image path against the reference CLI's host flow."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import canny_oracle as CO
from test_canny import golden_cases

pytestmark = pytest.mark.gpu

SIZES = [(1, 1), (7, 13), (37, 53), (64, 128), (389, 517), (512, 512), (720, 1280)]
THRESHOLDS = [(100, 200), (200, 100), (100.7, 200.2), (0, 0), (255, 255)]


@pytest.fixture(scope="module")
def eng():
    import i2it
    import weights as W
    return i2it.Engine(torch.bfloat16, i2it.PIX2PIX, cfg=W.TINY)


def _cv2():
    try:
        import cv2
        return cv2
    except ImportError:
        return None


def _device_edges(eng, imgs, lo, hi):
    x = torch.from_numpy(np.stack(imgs)).cuda()
    out = eng.canny_u8(x, lo, hi)
    torch.cuda.synchronize()
    assert out.shape == x.shape and out.dtype == torch.uint8
    return out.cpu().numpy()


@pytest.mark.parametrize("H,W", SIZES)
def test_canny_matches_oracle_and_cv2(eng, H, W):
    cv2 = _cv2()
    imgs = [CO.blurred_noise(1000 + H + W, H, W), np.random.default_rng(H * W).integers(0, 256, (H, W, 3), dtype=np.uint8)]
    for lo, hi in THRESHOLDS:
        got = _device_edges(eng, imgs, lo, hi)
        for i, img in enumerate(imgs):
            ref = CO.canny_u8(img, lo, hi)
            bad = int((got[i] != ref).sum())
            assert bad == 0, (H, W, lo, hi, i, bad)
            if cv2 is not None:
                assert (got[i] == cv2.Canny(img, lo, hi)[..., None]).all(), (H, W, lo, hi, i)


def test_canny_serpentine_component(eng):
    """62,762 edge pixels in one 8-connected chain that only 22 strong pixels at its start can reach."""
    img = CO.serpentine_image()
    got = _device_edges(eng, [img], 100, 200)[0]
    assert int((got[..., 0] == 255).sum()) == 62762
    assert (got == CO.canny_u8(img, 100, 200)).all()


def test_canny_matches_stored_cv2_output(eng):
    for img, lo, hi, edges in golden_cases():
        got = _device_edges(eng, [img], lo, hi)[0]
        assert (got == edges[..., None]).all(), (img.shape, lo, hi, int((got[..., 0] != edges).sum()))


def test_canny_deterministic_and_batch_independent(eng):
    imgs = [CO.blurred_noise(s, 512, 512) for s in (21, 22, 23)]
    imgs[2] = CO.serpentine_image()
    a = _device_edges(eng, imgs, 100, 200)
    b = _device_edges(eng, imgs, 100, 200)
    assert np.array_equal(a, b)
    for i, img in enumerate(imgs):
        assert np.array_equal(a[i], _device_edges(eng, [img], 100, 200)[0]), i


def test_canny_rejects_invalid_arguments(eng):
    """Bad arguments come back as errors with a message, never as a device fault; the handle keeps working."""
    x = torch.from_numpy(CO.blurred_noise(5, 40, 60)[None]).cuda()
    out = torch.empty_like(x)
    lib, st = eng.lib, C.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: C.c_void_p(t.data_ptr())

    def err(rc):
        assert rc != 0
        return eng.lib.i2it_last_error(eng._h).decode()

    assert "null" in err(lib.i2it_canny_u8(eng._h, None, 1, 40, 60, 100.0, 200.0, p(out), st))
    assert "null" in err(lib.i2it_canny_u8(eng._h, p(x), 1, 40, 60, 100.0, 200.0, None, st))
    assert "positive" in err(lib.i2it_canny_u8(eng._h, p(x), 0, 40, 60, 100.0, 200.0, p(out), st))
    assert "positive" in err(lib.i2it_canny_u8(eng._h, p(x), 1, 40, -1, 100.0, 200.0, p(out), st))
    assert "2^31" in err(lib.i2it_canny_u8(eng._h, p(x), 1 << 20, 2048, 2048, 100.0, 200.0, p(out), st))
    assert lib.i2it_canny_u8(None, p(x), 1, 40, 60, 100.0, 200.0, p(out), st) != 0
    for bad in (math.nan, math.inf):
        with pytest.raises(RuntimeError, match="finite"):
            eng.canny_u8(x, bad, 200)
    with pytest.raises(ValueError):
        eng.canny_u8(x.float(), 100, 200)
    with pytest.raises(ValueError):
        eng.canny_u8(x[..., :2].contiguous(), 100, 200)
    got = eng.canny_u8(x, 100, 200)
    assert (got.cpu().numpy()[0] == CO.canny_u8(x.cpu().numpy()[0], 100, 200)).all()


@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
def test_photo_to_image_matches_reference_flow(dt):
    """forward_u8(canny_u8(photo)) == the reference CLI's host flow, bit for bit: canny_from_pil (cv2.Canny, replicated to three
    channels) -> F.to_tensor -> model -> ToPILImage()(out * 0.5 + 0.5)   (src/inference_paired.py:47-50,72)."""
    import weights as W
    from pix2pix_turbo import Pix2Pix_Turbo
    m = Pix2Pix_Turbo(cfg=W.TINY, perturb_norm=True)
    m.set_eval()
    m.to(dt)
    H, Wd = 64, 128
    photos = np.stack([CO.blurred_noise(s, H, Wd) for s in (31, 32)])
    eps = torch.randn(2, 4, H // 8, Wd // 8, generator=torch.Generator().manual_seed(4))
    edges = m.canny_u8(photos)                                      # host input
    assert torch.equal(m.canny_u8(torch.from_numpy(photos).cuda()), edges)   # device input
    assert torch.equal(m.canny_u8(photos[0]), edges[:1])            # single HWC image
    got = m.forward_u8(edges, "a photo", eps=eps)
    c_t = torch.stack([torch.from_numpy(CO.canny_u8(p, 100, 200)).permute(2, 0, 1).float().div(255) for p in photos])
    y = m(c_t.to(dt).cuda(), "a photo", eps=eps)
    ref = (y.cpu() * 0.5 + 0.5).mul(255).byte().permute(0, 2, 3, 1)
    torch.cuda.synchronize()
    assert torch.equal(got.cpu(), ref)
