"""GPU parity of the image side of the augmentation (css_aug_image): batch_transform_* against the PIL chain
(`_augment_image`, the reference's own code) at the training sizes, each op against the oracle with forced parameters,
the exhaustive colour table through the hue op, and CUDA-graph replay.  Everything is 8-bit work: the bar is exact equality."""
import numpy as np
import pytest
import torch

from oracle import pil_oracle as O
from tests.test_aug_host import seed_all
from tests.test_aug_image_host import all_colours, smooth_image

pytestmark = pytest.mark.gpu

P = {n: i for i, n in enumerate(("jitter", "order0", "order1", "order2", "order3", "brightness", "contrast", "saturation",
                                 "hue_byte", "blur", "radius"))}


def images_batch(B, H, W, seed):
    """Normalised images (what the model shells pass to batch_transform_*) of natural-looking content."""
    from css_b200 import aug
    x = np.stack([smooth_image(H, W, seed + k).transpose(2, 0, 1) for k in range(B)]).astype(np.float32) / 255
    mean, std = np.asarray(aug._MEAN, np.float32)[:, None, None], np.asarray(aug._STD, np.float32)[:, None, None]
    return torch.from_numpy((x - mean) / std).cuda()


def pil_batch(images, crop_size, scale_size, augmentation):
    """The image side of batch_transform_* as the PIL chain computes it: one device->host copy, _augment_image per image."""
    import torchvision.transforms.functional as TF
    from css_b200 import aug
    host = aug._unnormalise(images).cpu()
    out, geo = zip(*[aug._augment_image(TF.to_pil_image(host[k]), crop_size, scale_size, augmentation)
                     for k in range(host.shape[0])])
    return torch.stack(out), np.asarray(geo, np.int32)


@pytest.mark.parametrize("H,W,B,crop,seeds", [(321, 321, 8, (321, 321), (0, 1, 2)), (769, 769, 4, (769, 769), (3, 4)),
                                              (200, 300, 3, -1, (5,))])
def test_batch_transform_2_vs_pil_chain(H, W, B, crop, seeds):
    """Both trips of a training step: scale 0.5..1.5 without jitter, then scale 1 with jitter / blur / flip."""
    from css_b200 import aug
    rng = np.random.default_rng(H)
    label = torch.from_numpy(rng.integers(0, 21, (B, H, W)).astype(np.float32)).cuda()
    c1, c2 = (torch.from_numpy(rng.random((B, H, W), np.float32)).cuda() for _ in range(2))
    for seed in seeds:
        for scale, augmentation in (((0.5, 1.5), False), ((1.0, 1.0), True)):
            images = images_batch(B, H, W, 10 * seed)
            seed_all(seed)
            ref, ref_geo = pil_batch(images, crop, scale, augmentation)
            state = torch.get_rng_state()
            seed_all(seed)
            r = aug.batch_transform_2(images, label, c1, c2, crop_size=crop, scale_size=scale, augmentation=augmentation)
            assert torch.equal(torch.get_rng_state(), state)
            assert r[0].is_cuda and r[0].shape == ref.shape
            np.testing.assert_array_equal(r[0].cpu().numpy(), ref.numpy(), err_msg=f"seed {seed} scale {scale}")
            ol, oc = aug.transform_maps([label], [c1, c2], ref_geo, tuple(ref.shape[2:]))
            assert torch.equal(r[1], ol[0]) and torch.equal(r[2], oc[0]) and torch.equal(r[3], oc[1])


def _run(x01, geo, params, crop):
    """transform_images on an unnormalised batch vs the oracle chain, image by image."""
    from css_b200 import aug
    got = aug.transform_images(torch.from_numpy(x01).cuda(), geo, params, crop).cpu().numpy()
    lut = aug.image_lut().numpy()
    for k in range(x01.shape[0]):
        np.testing.assert_array_equal(got[k], O.aug_image(x01[k], geo[k], params[k], crop, lut), err_msg=f"image {k}")


def _x01(B, H, W, seed):
    return np.stack([smooth_image(H, W, seed + k).transpose(2, 0, 1) for k in range(B)]).astype(np.float32) / 255


def _params(B, **kw):
    p = np.zeros((B, len(P)), np.float32)
    for k, v in kw.items():
        p[:, P[k]] = v
    return p


def test_each_jitter_op_alone_and_contrast_at_every_position():
    import itertools
    H = W = 96
    orders = list(itertools.permutations(range(4)))                # contrast at every position, every order
    B = len(orders)
    x = _x01(B, H, W, 1)
    geo = np.tile(np.asarray([H, W, 0, 0, 0], np.int32), (B, 1))
    for fb, fc, fs, hue in ((1.0, 1.0, 1.0, 0), (0.75, 1.0, 1.0, 0), (1.0, 0.75, 1.0, 0), (1.0, 1.25, 1.0, 0),
                            (1.0, 1.0, 1.25, 0), (1.0, 1.0, 0.75, 0), (1.0, 1.0, 1.0, 200), (1.2345, 0.8123, 1.1111, 37)):
        p = _params(B, jitter=1, brightness=fb, contrast=fc, saturation=fs, hue_byte=hue)
        p[:, 1:5] = np.asarray(orders, np.float32)
        _run(x, geo, p, (H, W))


def test_blur_flip_and_radius_sweep():
    H, W = 70, 90                                                  # several tiles, partial ones at the edges
    radii = np.concatenate([np.linspace(0.15, 1.15, 21), [0.01, 2.0, 3.3, 4.0]]).astype(np.float32)
    B = len(radii)
    x = _x01(B, H, W, 2)
    geo = np.tile(np.asarray([H, W, 0, 0, 0], np.int32), (B, 1))
    geo[::2, 4] = 1
    _run(x, geo, _params(B, blur=1, radius=radii), (H, W))
    _run(x, geo, _params(B), (H, W))


@pytest.mark.parametrize("H,W", [(321, 321), (769, 769), (120, 77)])
def test_resize_pad_crop(H, W):
    """Up, down, one axis only, pads longer than the resized image (reflected more than once), random crops."""
    rng = np.random.default_rng(W)
    ch, cw = min(H, 321), min(W, 321)
    rows = []
    for ratio_h, ratio_w in ((1.0, 1.0), (0.5, 0.5), (2.0, 2.0), (1.0, 0.6), (1.7, 1.0), (0.3, 0.25), (1.3, 0.9)):
        rh, rw = max(int(H * ratio_h), 1), max(int(W * ratio_w), 1)
        ph, pw = max(rh, ch), max(rw, cw)
        rows.append((rh, rw, rng.integers(0, ph - ch + 1), rng.integers(0, pw - cw + 1), rng.integers(0, 2)))
    geo = np.asarray(rows, np.int32)
    B = len(rows)
    p = _params(B, jitter=1, brightness=1.1, contrast=0.9, saturation=1.2, hue_byte=5, blur=1, radius=0.7)
    p[:, 1:5] = (3, 1, 0, 2)
    _run(_x01(B, H, W, 3), geo, p, (ch, cw))


@pytest.mark.parametrize("hue", [-0.25, -0.1, 0.0, 0.05, 0.25])
def test_hue_all_colours(hue):
    """Every one of the 2^24 colours through the GPU hue op (the other three factors 1.0: exact identities)."""
    from css_b200 import aug
    import torchvision.transforms.functional as TF
    from PIL import Image
    img = all_colours()
    x = torch.from_numpy(((img.astype(np.float32) + 0.5) / 255).transpose(2, 0, 1)[None].copy()).cuda()
    geo = np.asarray([[4096, 4096, 0, 0, 0]], np.int32)
    p = _params(1, jitter=1, brightness=1.0, contrast=1.0, saturation=1.0, hue_byte=np.int32(hue * 255).astype(np.uint8))
    p[:, 1:5] = (3, 0, 2, 1)
    got = aug.transform_images(x, geo, p, (4096, 4096))[0]
    ref = np.asarray(TF.adjust_hue(Image.fromarray(img), hue))
    lut = aug.image_lut().cuda()
    want = torch.stack([lut[c][torch.from_numpy(ref[..., c].astype(np.int64)).cuda()] for c in range(3)])
    assert torch.equal(got, want)


def test_cuda_graph_replay_equals_eager():
    from css_b200 import aug
    B, H, W, crop = 4, 160, 160, (160, 160)
    seed_all(9)
    geo, params = aug.draw_image_params(B, H, W, crop, (0.5, 1.5), True)
    x = torch.from_numpy(_x01(B, H, W, 4)).cuda()
    g_dev, p_dev = torch.from_numpy(geo).cuda(), torch.from_numpy(params).cuda()
    eager = aug.transform_images(x, g_dev, p_dev, crop)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        aug.transform_images(x, g_dev, p_dev, crop)                # warm-up off the capture
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = aug.transform_images(x, g_dev, p_dev, crop)
    x.copy_(torch.from_numpy(_x01(B, H, W, 5)))
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, aug.transform_images(x, g_dev, p_dev, crop))
    assert not torch.equal(out, eager)


def test_transform_images_rejects_bad_input():
    from css_b200 import aug
    geo, p = np.asarray([[8, 8, 0, 0, 0]], np.int32), _params(1)
    with pytest.raises(RuntimeError, match="CUDA"):
        aug.transform_images(torch.rand(1, 3, 8, 8), geo, p, (8, 8))
    with pytest.raises(RuntimeError, match="B,3,H,W"):
        aug.transform_images(torch.rand(1, 1, 8, 8).cuda(), geo, p, (8, 8))
    with pytest.raises(RuntimeError, match="geometry"):
        aug.transform_images(torch.rand(2, 3, 8, 8).cuda(), geo, _params(2), (8, 8))
    with pytest.raises(RuntimeError, match="radius"):
        aug.transform_images(torch.rand(1, 3, 8, 8).cuda(), geo, _params(1, blur=1, radius=5.0), (8, 8))
