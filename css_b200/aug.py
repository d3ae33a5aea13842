"""GPU-resident augmentation of the image and of the pseudo-label / confidence maps (SURVEY.md 8(f)-2).

The reference sends every image and map of every image GPU -> PIL -> GPU twice per step (dataset_helpers/VOC.py:284-302
into transform_* :64-274 and back, driven by batch_transform_* :312-352) and mixes images with a Python loop of small
kernels behind four all_gathers (generate_cut_gather_* :354-477).  Here

  * the host only DRAWS: `draw_image_params` consumes the Python and torch RNG streams exactly as the reference's PIL
    chain does (`_augment_image`, kept as the in-tree reference) and returns the geometry and the per-image jitter / blur
    parameters, without touching pixels;
  * the IMAGE never leaves the GPU: `css_aug_image` replays Pillow's 8-bit arithmetic (bilinear resize, reflect pad,
    crop, ColorJitter, GaussianBlur, flip, to_tensor + normalize) bit-identically (`transform_images`);
  * the MAPS never leave the GPU: `css_aug_index` + `css_aug_maps` replay the drawn geometry (Pillow NEAREST resize
    table, bottom/right padding with 255 / 0, crop, flip) and the 8-bit round trip (label -1 <-> 255, conf ->
    floor(conf * 255) / 255) bit-exactly;
  * CutMix / CutOut / ClassMix is one fused launch (`css_cut_mix`); with several ranks only rank 0's batch is
    broadcast, because the reference's partner index `(i + 1) % batch_size` always lands in rank 0's slice of the
    gathered batch (VOC.py:386,428,469).

`batch_transform`, `batch_transform_2`, `batch_transform_3`, `generate_cut_gather`, `generate_cut_gather_2`,
`generate_cut_gather_3` keep the reference's names, arguments and return values; `css_b200.install.install(...,
gpu_aug=True)` routes the model shells through them.
"""
import random

import numpy as np
import torch
import torch.distributed as dist

from . import _lib
from ._lib import check, ptr, stream_ptr

_MEAN = (0.485, 0.456, 0.406)
_STD = (0.229, 0.224, 0.225)


# ---------------------------------------------------------------------------------------------------------------
# image side: the PIL chain (the reference), the host-side draws, the GPU replay
# ---------------------------------------------------------------------------------------------------------------
def _tv():
    import torchvision.transforms as T
    import torchvision.transforms.functional as TF
    return T, TF


def _unnormalise(images):
    """ImageNet de-normalisation with the reference's two-step arithmetic (VOC.py:304-308), batched."""
    _, TF = _tv()
    x = TF.normalize(images, mean=[0., 0., 0.], std=[1 / s for s in _STD])
    return TF.normalize(x, mean=[-m for m in _MEAN], std=[1., 1., 1.])


def _augment_image(pil, crop_size, scale_size, augmentation):
    """One image through the reference's resize / pad / crop / jitter / blur / flip chain (the image lines of
    VOC.py:126-196).  Returns (normalised tensor [3,ch,cw], (resized_h, resized_w, top, left, flip)): the geometry is
    what the maps have to replay."""
    from PIL import ImageFilter
    T, TF = _tv()
    raw_w, raw_h = pil.size
    ratio = random.uniform(scale_size[0], scale_size[1])
    rh, rw = int(raw_h * ratio), int(raw_w * ratio)
    pil = TF.resize(pil, (rh, rw), T.InterpolationMode.BILINEAR)
    if crop_size == -1:
        crop_size = (raw_w, raw_h)
    ch, cw = int(crop_size[0]), int(crop_size[1])
    if ch > rh or cw > rw:
        pil = TF.pad(pil, padding=(0, 0, max(cw - rw, 0), max(ch - rh, 0)), padding_mode='reflect')
    top, left, _, _ = T.RandomCrop.get_params(pil, output_size=(ch, cw))
    pil = TF.crop(pil, top, left, ch, cw)
    flip = False
    if augmentation:
        if torch.rand(1) > 0.2:
            pil = T.ColorJitter((0.75, 1.25), (0.75, 1.25), (0.75, 1.25), (-0.25, 0.25))(pil)
        if torch.rand(1) > 0.5:
            pil = pil.filter(ImageFilter.GaussianBlur(radius=random.uniform(0.15, 1.15)))
        if torch.rand(1) > 0.5:
            pil = TF.hflip(pil)
            flip = True
    img = TF.normalize(TF.to_tensor(pil), mean=list(_MEAN), std=list(_STD))
    return img, (rh, rw, int(top), int(left), int(flip))


# Columns of the per-image parameter table (float32 [B, 11]; every value is exactly representable): jitter on/off, the
# ColorJitter order (0 brightness, 1 contrast, 2 saturation, 3 hue), the three blend factors, the hue shift as the byte
# torchvision adds to H, blur on/off and the GaussianBlur radius (Pillow takes it as a C float).
IMAGE_PARAMS = ("jitter", "order0", "order1", "order2", "order3", "brightness", "contrast", "saturation", "hue_byte", "blur",
                "radius")


def draw_image_params(B, H, W, crop_size, scale_size, augmentation):
    """Draws what `_augment_image` draws for B images of H x W, in the same order from the same generators (`random`,
    torch's CPU generator; numpy is not used), without touching pixels.  Returns (geometry int32 [B,5] = resized_h,
    resized_w, top, left, flip -- what `transform_maps` replays -- and the float32 [B, len(IMAGE_PARAMS)] table)."""
    T, _ = _tv()
    jitter = T.ColorJitter((0.75, 1.25), (0.75, 1.25), (0.75, 1.25), (-0.25, 0.25))
    geometry = np.zeros((B, 5), np.int32)
    params = np.zeros((B, len(IMAGE_PARAMS)), np.float32)
    for k in range(B):
        ratio = random.uniform(scale_size[0], scale_size[1])
        rh, rw = int(H * ratio), int(W * ratio)
        crop = (W, H) if crop_size == -1 else crop_size
        ch, cw = int(crop[0]), int(crop[1])
        # a stand-in of the padded image's shape: RandomCrop draws nothing when it equals the crop
        top, left, _, _ = T.RandomCrop.get_params(torch.zeros(()).expand(3, max(rh, ch), max(rw, cw)), output_size=(ch, cw))
        flip = 0
        if augmentation:
            if torch.rand(1) > 0.2:
                order, fb, fc, fs, fh = jitter.get_params(jitter.brightness, jitter.contrast, jitter.saturation, jitter.hue)
                params[k, 0] = 1
                params[k, 1:5] = order.numpy()
                params[k, 5:8] = fb, fc, fs
                params[k, 8] = np.int32(fh * 255).astype(np.uint8)           # torchvision's adjust_hue byte
            if torch.rand(1) > 0.5:
                params[k, 9], params[k, 10] = 1, random.uniform(0.15, 1.15)
            if torch.rand(1) > 0.5:
                flip = 1
        geometry[k] = rh, rw, top, left, flip
    return geometry, params


def image_lut():
    """float32 [3,256]: byte -> to_tensor + normalize, computed with the very torch CPU ops torchvision applies."""
    _, TF = _tv()
    x = torch.arange(256, dtype=torch.uint8).view(1, 1, 256).expand(3, 1, 256).to(torch.float32).div(255)
    return TF.normalize(x, mean=list(_MEAN), std=list(_STD)).reshape(3, 256).contiguous()


# ---------------------------------------------------------------------------------------------------------------
# map side (GPU)
# ---------------------------------------------------------------------------------------------------------------
def _label_arg(t, name):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f"css_b200: `{name}` must be a CUDA tensor (no CPU fallback)")
    if t.dtype == torch.float32:
        return t.contiguous(), _lib.LABEL_F32
    if t.dtype == torch.int64:
        return t.contiguous(), _lib.LABEL_I64
    raise RuntimeError(f"css_b200: `{name}` must be float32 or int64, got {t.dtype}")


def _conf_arg(t, name):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f"css_b200: `{name}` must be a CUDA tensor (no CPU fallback)")
    if t.dtype != torch.float32:
        raise RuntimeError(f"css_b200: `{name}` must be float32, got {t.dtype}")
    return t.contiguous()


def transform_maps(labels, confs, geometry, crop_hw, max_resized=None):
    """Replays `geometry` (int tensor/array [B,5]: resized_h, resized_w, top, left, flip) on up to two label maps and up to
    two confidence maps [B,H,W] that stay on the GPU.  Returns (labels int64 [B,ch,cw] with -1 = ignore, confs float32).
    A CUDA `geometry` together with `max_resized` (an upper bound of every resized_h / resized_w) keeps the call free of
    host synchronisation, e.g. for CUDA-graph capture."""
    labels, confs = list(labels), list(confs)
    if not labels and not confs:
        raise RuntimeError("css_b200: transform_maps needs at least one map")
    if len(labels) > 2 or len(confs) > 2:
        raise RuntimeError("css_b200: transform_maps takes at most two label maps and two confidence maps")
    first = (labels + confs)[0]
    dev = first.device
    B, H, W = first.shape
    ch, cw = int(crop_hw[0]), int(crop_hw[1])
    la = [_label_arg(t, "label") for t in labels]
    if len(la) == 2 and la[0][1] != la[1][1]:
        raise RuntimeError("css_b200: the two label maps must have the same dtype")
    cf = [_conf_arg(t, "logits") for t in confs]
    for t in [x[0] for x in la] + cf:
        if tuple(t.shape) != (B, H, W):
            raise RuntimeError("css_b200: every map must be [B,H,W] with the same shape")
    if isinstance(geometry, torch.Tensor) and geometry.is_cuda:
        geo = geometry.to(torch.int32).contiguous()
        max_r = int(max_resized) if max_resized is not None else int(geo[:, :2].max().item())
    else:
        geo_host = np.ascontiguousarray(np.asarray(geometry, dtype=np.int32).reshape(B, 5))
        geo = torch.from_numpy(geo_host).pin_memory().to(dev, non_blocking=True)
        max_r = int(max(geo_host[:, 0].max(), geo_host[:, 1].max()))
    ymap = torch.empty((B, max_r), device=dev, dtype=torch.int32)
    xmap = torch.empty((B, max_r), device=dev, dtype=torch.int32)
    out_l = [torch.empty((B, ch, cw), device=dev, dtype=torch.int64) for _ in la]
    out_c = [torch.empty((B, ch, cw), device=dev, dtype=torch.float32) for _ in cf]
    lib = _lib.load()

    def at(seq, i):
        return ptr(seq[i]) if i < len(seq) else None

    with torch.cuda.device(dev):
        check(lib.css_aug_index(ptr(geo), B, H, W, max_r, ptr(ymap), ptr(xmap), stream_ptr()), "css_aug_index")
        check(lib.css_aug_maps(at([x[0] for x in la], 0), at([x[0] for x in la], 1), la[0][1] if la else _lib.LABEL_F32,
                               at(cf, 0), at(cf, 1), ptr(geo), ptr(ymap), ptr(xmap), B, H, W, max_r, ch, cw,
                               at(out_l, 0), at(out_l, 1), at(out_c, 0), at(out_c, 1), stream_ptr()), "css_aug_maps")
    return out_l, out_c


_LUTS = {}


def _lut(dev):
    """image_lut() on `dev`, made once per device (so that a captured CUDA graph finds it in place)."""
    key = str(dev)
    if key not in _LUTS:
        _LUTS[key] = image_lut().to(dev)
    return _LUTS[key]


def _table_arg(t, shape, dtype, dev, name):
    if isinstance(t, torch.Tensor) and t.is_cuda:
        if tuple(t.shape) != shape:
            raise RuntimeError(f"css_b200: `{name}` must be {list(shape)}, got {list(t.shape)}")
        return t.to(dtype).contiguous(), None
    a = np.asarray(t.cpu() if isinstance(t, torch.Tensor) else t, dtype={torch.int32: np.int32, torch.float32: np.float32}[dtype])
    if a.shape != shape:
        raise RuntimeError(f"css_b200: `{name}` must be {list(shape)}, got {list(a.shape)}")
    a = np.ascontiguousarray(a)
    return torch.from_numpy(a).pin_memory().to(dev, non_blocking=True), a


def transform_images(images, geometry, params, crop_hw):
    """The image side of `_augment_image` for a whole batch on the GPU, bit-identical to the Pillow chain.
    images: unnormalised CUDA float32 [B,3,H,W] in [0, 1] (what `_unnormalise` returns); geometry: int [B,5] and params:
    float [B, len(IMAGE_PARAMS)] as drawn by `draw_image_params`.  Returns the normalised float32 [B,3,ch,cw].  With
    CUDA `geometry` and `params` the call does no host synchronisation (CUDA-graph capturable)."""
    if not isinstance(images, torch.Tensor) or not images.is_cuda:
        raise RuntimeError("css_b200: `images` must be a CUDA tensor (no CPU fallback)")
    if images.dtype != torch.float32 or images.dim() != 4 or images.shape[1] != 3:
        raise RuntimeError(f"css_b200: `images` must be float32 [B,3,H,W], got {images.dtype} {list(images.shape)}")
    images = images.contiguous()
    B, _, H, W = images.shape
    ch, cw = int(crop_hw[0]), int(crop_hw[1])
    if ch <= 0 or cw <= 0:
        raise RuntimeError(f"css_b200: bad crop size {(ch, cw)}")
    dev = images.device
    geo, _ = _table_arg(geometry, (B, 5), torch.int32, dev, "geometry")
    par, par_host = _table_arg(params, (B, len(IMAGE_PARAMS)), torch.float32, dev, "params")
    if par_host is not None:
        r = par_host[par_host[:, IMAGE_PARAMS.index("blur")] != 0, IMAGE_PARAMS.index("radius")]
        if ((r < 0) | (r > 4)).any():
            raise RuntimeError("css_b200: GaussianBlur radius must be in [0, 4]")
    lib = _lib.load()
    out = torch.empty((B, 3, ch, cw), device=dev, dtype=torch.float32)
    ws_bytes = lib.css_aug_image_workspace_bytes(B, ch, cw)
    ws = torch.empty(ws_bytes, device=dev, dtype=torch.uint8)
    with torch.cuda.device(dev):
        check(lib.css_aug_image(ptr(images), B, H, W, ptr(geo), ptr(par), ptr(_lut(dev)), ch, cw, ptr(ws), ws_bytes, ptr(out),
                                stream_ptr()), "css_aug_image")
    return out


def _batch_transform(images, labels, confs, crop_size, scale_size, augmentation):
    if not images.is_cuda:
        raise RuntimeError("css_b200: `images` must be a CUDA tensor (no CPU fallback)")
    B, _, H, W = images.shape
    geometry, params = draw_image_params(B, H, W, crop_size, scale_size, augmentation)
    crop = (W, H) if crop_size == -1 else crop_size
    crop_hw = (int(crop[0]), int(crop[1]))
    geo = torch.from_numpy(geometry).pin_memory().to(images.device, non_blocking=True)
    image_trans = transform_images(_unnormalise(images), geo, params, crop_hw)
    out_l, out_c = transform_maps(labels, confs, geo, crop_hw, max_resized=int(geometry[:, :2].max()))
    return image_trans, out_l, out_c


def batch_transform(images, labels, logits=None, crop_size=(512, 512), scale_size=(0.8, 1.0), augmentation=True):
    """Drop-in for dataset_helpers/VOC.py:312-323."""
    img, l, c = _batch_transform(images, [labels], [logits], crop_size, scale_size, augmentation)
    return img, l[0], c[0]


def batch_transform_2(images, labels, logits_1=None, logits_2=None, crop_size=(512, 512), scale_size=(0.8, 1.0),
                      augmentation=True):
    """Drop-in for dataset_helpers/VOC.py:325-337."""
    img, l, c = _batch_transform(images, [labels], [logits_1, logits_2], crop_size, scale_size, augmentation)
    return img, l[0], c[0], c[1]


def batch_transform_3(images, labels1, labels2, logits_1=None, logits_2=None, crop_size=(512, 512), scale_size=(0.8, 1.0),
                      augmentation=True):
    """Drop-in for dataset_helpers/VOC.py:339-352."""
    img, l, c = _batch_transform(images, [labels1, labels2], [logits_1, logits_2], crop_size, scale_size, augmentation)
    return img, l[0], l[1], c[0], c[1]


# ---------------------------------------------------------------------------------------------------------------
# CutOut / CutMix / ClassMix
# ---------------------------------------------------------------------------------------------------------------
CUT_MODES = {"cutout": 0, "cutmix": 1, "classmix": 2}


def draw_cut_box(image_h, image_w, ratio=2):
    """The region generate_cutout_mask zeroes (VOC.py:518-535), as (y0, y1, x0, x1) clipped to the image; consumes
    np.random exactly like the reference (three randint draws)."""
    area = image_h * image_w / ratio
    bw = np.random.randint(image_w / ratio + 1, image_w)
    bh = np.round(area / bw)
    x0 = np.random.randint(0, image_w - bw + 1)
    y0 = np.random.randint(0, image_h - bh + 1)
    x1, y1 = int(x0 + bw), int(y0 + bh)
    return int(y0), min(y1, image_h), int(x0), min(x1, image_w)


def draw_class_set(label_map):
    """ClassMix: half of the label values present in `label_map`, picked with torch.randperm (VOC.py:511-516)."""
    present = torch.unique(label_map)
    chosen = present[torch.randperm(len(present))][:len(present) // 2]
    return [int(v) for v in chosen.tolist()]


def _class_bits(values):
    """Label value v in [-1, 62] -> bit v + 1 of a 64-bit set."""
    bits = 0
    for v in values:
        if not -1 <= v <= 62:
            raise RuntimeError(f"css_b200: classmix label value {v} outside [-1, 62]")
        bits |= 1 << (v + 1)
    return bits - (1 << 64) if bits >= (1 << 63) else bits


def cut_mix(image, labels, confs, mode, boxes=None, class_sets=None, partner=None):
    """One fused launch: out[i] = keep ? own[i] : partner[(i+1) % B]  (cutout: 0 / -1 instead of the partner).
    boxes: int [B,4] (y0, y1, x0, x1) of the replaced region; class_sets: per image the label values that keep the own
    pixels; partner: (image, labels, confs) the partners come from (default: the same batch)."""
    if mode not in CUT_MODES:
        raise ValueError('mode must be in cutout, cutmix, or classmix')
    if not image.is_cuda:
        raise RuntimeError("css_b200: `image` must be a CUDA tensor (no CPU fallback)")
    dev = image.device
    image = _conf_arg(image, "image")
    B, CH, H, W = image.shape
    labels = [_label_arg(t, "label")[0] for t in labels]
    for t in labels:
        if t.dtype != torch.int64:
            raise RuntimeError("css_b200: cut_mix labels must be int64")
    confs = [_conf_arg(t, "logits") for t in confs]
    if len(labels) not in (1, 2) or len(confs) not in (1, 2):
        raise RuntimeError("css_b200: cut_mix takes one or two label maps and one or two confidence maps")
    p_image, p_labels, p_confs = (image, labels, confs) if partner is None else partner
    p_image = _conf_arg(p_image, "partner image")
    p_labels = [_label_arg(t, "partner label")[0] for t in p_labels]
    p_confs = [_conf_arg(t, "partner logits") for t in p_confs]
    if mode == "classmix":
        spec = torch.tensor([_class_bits(s) for s in class_sets], dtype=torch.int64).pin_memory().to(dev, non_blocking=True)
        box_t = None
    else:
        box_t = torch.from_numpy(np.ascontiguousarray(np.asarray(boxes, np.int32).reshape(B, 4))).pin_memory().to(dev, non_blocking=True)
        spec = None
    o_img = torch.empty_like(image)
    o_lab = [torch.empty_like(t) for t in labels]
    o_conf = [torch.empty_like(t) for t in confs]
    lib = _lib.load()

    def at(seq, i):
        return ptr(seq[i]) if i < len(seq) else None

    with torch.cuda.device(dev):
        check(lib.css_cut_mix(ptr(image), at(labels, 0), at(labels, 1), at(confs, 0), at(confs, 1),
                              ptr(p_image), at(p_labels, 0), at(p_labels, 1), at(p_confs, 0), at(p_confs, 1),
                              ptr(box_t), ptr(spec), CUT_MODES[mode], B, CH, H, W,
                              ptr(o_img), at(o_lab, 0), at(o_lab, 1), at(o_conf, 0), at(o_conf, 1), stream_ptr()),
              "css_cut_mix")
    return o_img, o_lab, o_conf


def _generate_cut_gather(image, labels, confs, mode):
    batch_size, _, H, W = image.shape
    world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    rank = dist.get_rank() if world > 1 else 0
    labels = [t.long() for t in labels]
    if mode == 'none':
        return image, labels, confs
    if mode not in CUT_MODES:
        raise ValueError('mode must be in cutout, cutmix, or classmix')
    if mode == 'cutout' and len(labels) == 2:
        # generate_cut_gather_3 never fills its second label list in this mode and dies in torch.cat (VOC.py:453-461)
        raise RuntimeError("css_b200: mode 'cutout' with two label maps is broken in the reference (VOC.py:453-461)")
    partner = None
    if world > 1 and mode != 'cutout':
        # partner (i + 1) % batch_size indexes the GATHERED batch, i.e. always rank 0's images (VOC.py:428)
        partner = tuple(_broadcast0(x) for x in (image, labels, confs))
    total = batch_size * world
    boxes = class_sets = None
    if mode == 'classmix':
        # every rank draws torch.randperm(number of label values present) for EVERY gathered image, in gathered order
        # (VOC.py:381,423,465 -> :511-516).  What the draws for other ranks' images need from those ranks is only that number (it
        # fixes how much of the CPU generator's stream a permutation consumes), so one all_gather of `batch_size` counts replaces
        # the gather of the label maps; this rank's own images get their real draws at their place in the sequence.
        own = range(rank * batch_size, (rank + 1) * batch_size)
        if world > 1:
            n_all = [None] * world                                # a few ints per rank: backend-agnostic object gather
            dist.all_gather_object(n_all, [int(torch.unique(labels[0][i]).numel()) for i in range(batch_size)])
            counts = [n for per_rank in n_all for n in per_rank]
        class_sets = []
        for i in range(total):
            if i in own:
                class_sets.append(draw_class_set(labels[0][i - rank * batch_size]))
            else:
                torch.randperm(int(counts[i]))                    # advance the generator exactly as the reference does
    else:
        ratio = 2
        drawn = [draw_cut_box(H, W, ratio) for _ in range(total)]      # every rank draws for the whole gathered batch
        boxes = drawn[rank * batch_size:(rank + 1) * batch_size]
    return cut_mix(image, labels, confs, mode, boxes=boxes, class_sets=class_sets, partner=partner)


def _broadcast0(x):
    if isinstance(x, (list, tuple)):
        return [_broadcast0(t) for t in x]
    buf = x.contiguous().clone()
    dist.broadcast(buf, src=0)
    return buf


def generate_cut_gather(image, label, logits, mode='cutout'):
    """Drop-in for dataset_helpers/VOC.py:354-391."""
    img, l, c = _generate_cut_gather(image, [label], [logits], mode)
    return img, l[0], c[0]


def generate_cut_gather_2(image, label, logits1, logits2, mode='cutout'):
    """Drop-in for dataset_helpers/VOC.py:393-434."""
    img, l, c = _generate_cut_gather(image, [label], [logits1, logits2], mode)
    return img, l[0], c[0], c[1]


def generate_cut_gather_3(image, label1, label2, logits1, logits2, mode='cutout'):
    """Drop-in for dataset_helpers/VOC.py:436-477."""
    img, l, c = _generate_cut_gather(image, [label1, label2], [logits1, logits2], mode)
    return img, l[0], l[1], c[0], c[1]
