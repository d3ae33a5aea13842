"""CPU tests of the image side of the augmentation: every 8-bit step of oracle/pil_oracle.py against the installed Pillow,
the whole oracle chain against css_b200.aug._augment_image, and css_b200.aug.draw_image_params against the RNG consumption
of that chain.  Exact equality throughout: the GPU kernels (css_aug_image.cu) are written from these restatements."""
import random

import numpy as np
import pytest
import torch
from PIL import Image, ImageEnhance, ImageFilter

from oracle import pil_oracle as O
from tests.test_aug_host import seed_all


def rgb_image(h, w, seed):
    return np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)


def smooth_image(h, w, seed):
    """Natural-looking content (gradients + noise) so that the colour ops see structure, not only noise."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    base = np.stack([np.sin(yy / (5 + c) + xx / (7 + 2 * c) + c) for c in range(3)], -1) * 100 + 128
    return np.clip(base + rng.normal(0, 20, (h, w, 3)), 0, 255).astype(np.uint8)


def all_colours():
    v = np.arange(1 << 24, dtype=np.uint32)
    return np.stack([(v >> 16) & 255, (v >> 8) & 255, v & 255], -1).astype(np.uint8).reshape(4096, 4096, 3)


RESAMPLE_PAIRS = [(321, 160), (321, 642), (321, 321), (769, 384), (769, 1538), (500, 375), (375, 500), (333, 266),
                  (266, 333), (100, 99), (99, 100), (1, 5), (5, 1), (7, 3), (3, 7), (2, 4), (4, 2), (321, 240), (321, 481),
                  (769, 576), (769, 1153), (1024, 512), (513, 1024), (40, 17), (17, 40), (64, 64), (10, 31), (31, 10),
                  (200, 201), (201, 200), (321, 203), (321, 587)]


@pytest.mark.parametrize("n_in,n_out", RESAMPLE_PAIRS)
def test_resample_bilinear_vs_pillow(n_in, n_out):
    """Up, down and same size along each axis alone, and along both."""
    for h_in, w_in, h_out, w_out in ((7, n_in, 7, n_out), (n_in, 9, n_out, 9), (n_in, n_in, n_out, n_out),
                                     (n_in, 11, n_out, 13)):
        img = rgb_image(h_in, w_in, n_in * 7 + n_out)
        ref = np.asarray(Image.fromarray(img).resize((w_out, h_out), Image.BILINEAR))
        np.testing.assert_array_equal(O.pil_resize_bilinear(img, h_out, w_out), ref)


def test_reflect_index_vs_numpy_pad():
    for n in (1, 2, 3, 5, 160, 321):
        for pad in (0, 1, n - 1, n, n + 1, 3 * n + 2):
            pad = max(pad, 0)
            a = np.arange(n)
            ref = np.pad(a, (0, pad), mode="reflect")
            np.testing.assert_array_equal(O.reflect_index(np.arange(n + pad), n), ref)


def test_l24_vs_pillow_all_colours():
    img = all_colours()
    np.testing.assert_array_equal(O.pil_l24(img), np.asarray(Image.fromarray(img).convert("L")))


BLEND_FACTORS = [0.0, 0.5, 0.75, 0.7500001, 0.81234, 0.9999999, 1.0, 1.0000001, 1.1, 1.2345678, 1.25, 1.75, 2.0, -0.3]


@pytest.mark.parametrize("alpha", BLEND_FACTORS)
def test_blend_all_byte_pairs_vs_pillow(alpha):
    a = np.repeat(np.arange(256, dtype=np.uint8), 256).reshape(256, 256)
    b = np.tile(np.arange(256, dtype=np.uint8), 256).reshape(256, 256)
    a3, b3 = np.stack([a, b, a], -1), np.stack([b, a, b], -1)
    ref = np.asarray(Image.blend(Image.fromarray(a3), Image.fromarray(b3), alpha))
    np.testing.assert_array_equal(O.pil_blend(a3, b3, alpha), ref)


@pytest.mark.parametrize("f", [0.75, 0.9123, 1.0, 1.1, 1.25])
def test_enhancers_vs_pillow(f):
    f = float(np.float32(f))
    for seed, make in ((1, rgb_image), (2, smooth_image)):
        img = make(61, 47, seed)
        pil = Image.fromarray(img)
        np.testing.assert_array_equal(O.pil_brightness(img, f), np.asarray(ImageEnhance.Brightness(pil).enhance(f)))
        np.testing.assert_array_equal(O.pil_contrast(img, f), np.asarray(ImageEnhance.Contrast(pil).enhance(f)))
        np.testing.assert_array_equal(O.pil_saturation(img, f), np.asarray(ImageEnhance.Color(pil).enhance(f)))


def test_rgb_to_hsv_vs_pillow_all_colours():
    img = all_colours()
    np.testing.assert_array_equal(O.pil_rgb_to_hsv(img), np.asarray(Image.fromarray(img).convert("HSV")))


def test_hsv_to_rgb_vs_pillow_all_triples():
    hsv = all_colours()
    ref = np.asarray(Image.fromarray(hsv, "HSV").convert("RGB"))
    np.testing.assert_array_equal(O.pil_hsv_to_rgb(hsv), ref)


@pytest.mark.parametrize("hue", [-0.25, -0.1234, -1 / 255, 0.0, 0.05, 0.25])
def test_hue_vs_torchvision_all_colours(hue):
    import torchvision.transforms.functional as TF
    img = all_colours()
    hue_byte = np.int32(hue * 255).astype(np.uint8)
    ref = np.asarray(TF.adjust_hue(Image.fromarray(img), hue))
    np.testing.assert_array_equal(O.pil_hue(img, hue_byte), ref)


BLUR_RADII = list(np.linspace(0.15, 1.15, 101)) + [0.01, 0.1, 1.5, 2.0, 2.7, 3.3, 4.0]


def test_box_blur_vs_pillow_radius_sweep():
    img = smooth_image(37, 53, 3)
    pil = Image.fromarray(img)
    for radius in BLUR_RADII:
        ref = np.asarray(pil.filter(ImageFilter.GaussianBlur(radius=float(radius))))
        np.testing.assert_array_equal(O.pil_gaussian_blur(img, radius), ref, err_msg=f"radius {radius}")


@pytest.mark.parametrize("h,w", [(1, 1), (2, 3), (5, 4), (9, 1), (1, 9)])
def test_box_blur_vs_pillow_tiny_images(h, w):
    img = rgb_image(h, w, h * 10 + w)
    for radius in (0.15, 0.7, 1.15, 3.0):
        ref = np.asarray(Image.fromarray(img).filter(ImageFilter.GaussianBlur(radius=radius)))
        np.testing.assert_array_equal(O.pil_gaussian_blur(img, radius), ref)


def test_image_lut_is_to_tensor_normalize():
    import torchvision.transforms.functional as TF
    from css_b200 import aug
    img = np.stack([np.arange(256, dtype=np.uint8).reshape(16, 16)[:, ::d] for d in (1, -1, 1)], -1)
    img[..., 2] = img[..., 2].T
    ref = TF.normalize(TF.to_tensor(Image.fromarray(img)), mean=list(aug._MEAN), std=list(aug._STD)).numpy()
    lut = aug.image_lut().numpy()
    np.testing.assert_array_equal(np.stack([lut[c][img[..., c]] for c in range(3)]), ref)


def _chain_vs_oracle(B, H, W, crop, scale, augmentation, seed):
    """_augment_image on each image and the oracle chain on the drawn parameters: same image, same geometry, same
    generator states afterwards."""
    import torchvision.transforms.functional as TF
    from css_b200 import aug
    x = torch.from_numpy(np.stack([smooth_image(H, W, seed + k).transpose(2, 0, 1) for k in range(B)]).astype(np.float32) / 255)
    x = x.clamp(0, 1)
    seed_all(seed)
    ref, ref_geo = zip(*[aug._augment_image(TF.to_pil_image(x[k]), crop, scale, augmentation) for k in range(B)])
    states = (random.getstate(), np.random.get_state()[1].copy(), torch.get_rng_state())
    seed_all(seed)
    geo, params = aug.draw_image_params(B, H, W, crop, scale, augmentation)
    assert random.getstate() == states[0]
    assert np.array_equal(np.random.get_state()[1], states[1])
    assert torch.equal(torch.get_rng_state(), states[2])
    np.testing.assert_array_equal(geo, np.asarray(ref_geo, np.int32))
    lut = aug.image_lut().numpy()
    ch, cw = ref[0].shape[1:]
    for k in range(B):
        np.testing.assert_array_equal(O.aug_image(x[k].numpy(), geo[k], params[k], (ch, cw), lut), ref[k].numpy())
    return params


@pytest.mark.parametrize("seed", range(4))
def test_oracle_chain_vs_augment_image_voc(seed):
    """VOC's two trips at a reduced size: scale 0.5..1.5 without jitter, then scale 1 with jitter / blur / flip."""
    _chain_vs_oracle(3, 81, 81, (81, 81), (0.5, 1.5), False, 100 + seed)
    p = _chain_vs_oracle(6, 81, 81, (81, 81), (1.0, 1.0), True, 200 + seed)
    assert p[:, 0].any()


def test_oracle_chain_vs_augment_image_cityscapes_quirk():
    """crop_size = -1 is (raw_w, raw_h); a non-square image makes the swap visible."""
    _chain_vs_oracle(2, 48, 64, -1, (0.5, 2.0), True, 7)
    _chain_vs_oracle(3, 60, 60, (40, 52), (0.5, 2.0), True, 8)


@pytest.mark.parametrize("trip", ["scale", "fixed"])
def test_draw_image_params_rng_streams(trip):
    """Over many seeds: draw_image_params leaves `random`, numpy and torch's CPU generator exactly where the PIL chain
    leaves them, and draws the same geometry (the pixels are not needed for that)."""
    import torchvision.transforms.functional as TF
    from css_b200 import aug
    scale, augmentation = ((0.5, 1.5), True) if trip == "scale" else ((1.0, 1.0), True)
    pil = TF.to_pil_image(torch.rand(3, 33, 33))
    for seed in range(40):
        seed_all(seed)
        ref_geo = [aug._augment_image(pil, (33, 33), scale, augmentation)[1] for _ in range(4)]
        states = (random.getstate(), np.random.get_state()[1].copy(), torch.get_rng_state())
        seed_all(seed)
        geo, params = aug.draw_image_params(4, 33, 33, (33, 33), scale, augmentation)
        assert random.getstate() == states[0]
        assert np.array_equal(np.random.get_state()[1], states[1])
        assert torch.equal(torch.get_rng_state(), states[2])
        np.testing.assert_array_equal(geo, np.asarray(ref_geo, np.int32))
        assert set(np.unique(params[params[:, 0] == 1][:, 1:5])) <= {0, 1, 2, 3}

