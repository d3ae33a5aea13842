"""Numpy restatement of the IMAGE's trip through the augmentation (css_b200/aug.py::_augment_image), step by step in
Pillow's 8-bit arithmetic: Resample.c (bilinear), numpy's reflect pad, Blend.c + ImageEnhance (brightness, contrast,
saturation), Convert.c (L24, RGB <-> HSV), BoxBlur.c (GaussianBlur), torchvision's to_tensor / normalize.
Images are uint8 [h, w, 3].  Every function is checked against the installed Pillow in tests/test_aug_image_host.py;
these are what css_b200/csrc/css_aug_image.cu is written from, operation for operation (the C float / double
promotions are spelled out with explicit casts).

Test infrastructure, like oracle/css_oracle.py: nothing under css_b200/ imports it."""
import numpy as np

F32, F64 = np.float32, np.float64
PIL_PRECISION_BITS = 22           # Resample.c: 32 - 8 - 2


def pil_resample_coeffs(n_in, n_out):
    """Resample.c precompute_coeffs + normalize_coeffs_8bpc for the bilinear filter (support 1) along one axis.
    Returns (xmin [n_out], count [n_out], fixed-point coefficients int64 [n_out, ksize])."""
    scale = F64(n_in) / F64(n_out)
    filterscale = max(scale, F64(1.0))
    support = F64(1.0) * filterscale
    ksize = int(np.ceil(support)) * 2 + 1
    ss = F64(1.0) / filterscale
    xx = np.arange(n_out, dtype=np.float64)
    center = F64(0.0) + (xx + 0.5) * scale
    xmin = np.maximum(np.trunc(center - support + 0.5).astype(np.int64), 0)
    xmax = np.minimum(np.trunc(center + support + 0.5).astype(np.int64), n_in) - xmin
    w = np.zeros((n_out, ksize), np.float64)
    ww = np.zeros(n_out, np.float64)
    for x in range(ksize):
        t = np.abs(((x + xmin).astype(np.float64) - center + 0.5) * ss)
        wx = np.where(t < 1.0, 1.0 - t, 0.0)
        wx = np.where(x < xmax, wx, 0.0)
        w[:, x] = wx
        ww = ww + wx                                              # sequential, as the C loop
    w = np.where(ww[:, None] != 0.0, w / np.where(ww == 0.0, 1.0, ww)[:, None], w)
    scaled = w * F64(1 << PIL_PRECISION_BITS)
    k = np.where(w < 0, np.trunc(-0.5 + scaled), np.trunc(0.5 + scaled)).astype(np.int64)
    return xmin, xmax, k


def _pil_resample_axis(img, n_out, axis):
    xmin, count, k = pil_resample_coeffs(img.shape[axis], n_out)
    src = np.moveaxis(img.astype(np.int64), axis, 0)
    acc = np.full((n_out,) + src.shape[1:], 1 << (PIL_PRECISION_BITS - 1), np.int64)
    extra = (slice(None),) + (None,) * (src.ndim - 1)
    for x in range(k.shape[1]):
        idx = np.minimum(xmin + x, src.shape[0] - 1)
        acc += src[idx] * np.where(x < count, k[:, x], 0)[extra]
    out = np.clip(acc >> PIL_PRECISION_BITS, 0, 255).astype(np.uint8)
    return np.moveaxis(out, 0, axis)


def pil_resize_bilinear(img, out_h, out_w):
    """Image.resize((out_w, out_h), BILINEAR): horizontal pass first (clipped to uint8), then vertical; a pass runs only
    when its axis changes size."""
    if out_w != img.shape[1]:
        img = _pil_resample_axis(img, out_w, 1)
    if out_h != img.shape[0]:
        img = _pil_resample_axis(img, out_h, 0)
    return img


def reflect_index(i, n):
    """np.pad(..., mode='reflect') source index of position i >= 0 of an axis of length n, also for pads longer than n."""
    i = np.asarray(i, np.int64)
    if n == 1:
        return np.zeros_like(i)
    m = i % (2 * (n - 1))
    return np.where(m < n, m, 2 * (n - 1) - m)


def pil_l24(img):
    """Convert.c rgb2l: L = (19595 R + 38470 G + 7471 B + 0x8000) >> 16."""
    c = img.astype(np.int64)
    return ((c[..., 0] * 19595 + c[..., 1] * 38470 + c[..., 2] * 7471 + 0x8000) >> 16).astype(np.uint8)


def pil_blend(im1, im2, alpha):
    """Image.blend(im1, im2, alpha) (Blend.c): float alpha; in1 + alpha * (in2 - in1) in float, truncated, clipped when
    extrapolating (alpha outside [0, 1])."""
    a = F32(alpha)
    i1 = np.asarray(im1).astype(np.int64)
    t = i1.astype(np.float32) + a * (np.asarray(im2).astype(np.int64) - i1).astype(np.float32)
    return np.clip(t, F32(0), F32(255)).astype(np.uint8)


def pil_brightness(img, f):
    return pil_blend(np.zeros_like(img), img, f)


def pil_saturation(img, f):
    return pil_blend(np.repeat(pil_l24(img)[..., None], 3, axis=-1), img, f)


def pil_contrast_mean(img):
    """ImageEnhance.Contrast's grey level: int(ImageStat mean of the L image + 0.5)."""
    return int(F64(int(pil_l24(img).astype(np.int64).sum())) / F64(img.shape[0] * img.shape[1]) + 0.5)


def pil_contrast(img, f):
    return pil_blend(np.full_like(img, pil_contrast_mean(img)), img, f)


def pil_rgb_to_hsv(img):
    """Convert.c rgb2hsv_row, with its float / double promotions."""
    c = img.astype(np.int64)
    r, g, b = c[..., 0], c[..., 1], c[..., 2]
    maxc, minc = c.max(-1), c.min(-1)
    grey = maxc == minc
    cr = np.where(grey, 1, maxc - minc).astype(np.float32)
    s = cr / np.where(grey, 1, maxc).astype(np.float32)
    rc, gc, bc = ((maxc - v).astype(np.float32) / cr for v in (r, g, b))
    h = np.where(r == maxc, bc - gc,
                 np.where(g == maxc, (F64(2.0) + rc.astype(np.float64) - bc.astype(np.float64)).astype(np.float32),
                          (F64(4.0) + gc.astype(np.float64) - rc.astype(np.float64)).astype(np.float32)))
    h = np.fmod(h.astype(np.float64) / 6.0 + 1.0, 1.0).astype(np.float32)
    uh = np.clip(np.trunc(h.astype(np.float64) * 255.0), 0, 255)
    us = np.clip(np.trunc(s.astype(np.float64) * 255.0), 0, 255)
    out = np.stack([np.where(grey, 0, uh), np.where(grey, 0, us), maxc], -1)
    return out.astype(np.uint8)


def pil_hsv_to_rgb(hsv):
    """Convert.c hsv2rgb, with its float / double promotions."""
    c = hsv.astype(np.int64)
    h, s, v = c[..., 0], c[..., 1], c[..., 2]
    hd = h.astype(np.float32).astype(np.float64) * 6.0 / 255.0
    i = np.floor(hd).astype(np.int64)
    f = (hd - i.astype(np.float32).astype(np.float64)).astype(np.float32)
    fs = (s.astype(np.float32).astype(np.float64) / 255.0).astype(np.float32)
    vd = v.astype(np.float32).astype(np.float64)
    rnd = lambda x: np.clip(np.where(x < 0, -np.floor(-x + 0.5), np.floor(x + 0.5)), 0, 255).astype(np.int64)   # noqa: E731
    p = rnd(vd * (1.0 - fs.astype(np.float64)))
    q = rnd(vd * (1.0 - (fs * f).astype(np.float64)))
    t = rnd(vd * (1.0 - fs.astype(np.float64) * (1.0 - f.astype(np.float64))))
    sel = i % 6
    cases = [(v, t, p), (q, v, p), (p, v, t), (p, q, v), (t, p, v), (v, p, q)]
    out = np.zeros(c.shape, np.int64)
    for k, (a, b2, c2) in enumerate(cases):
        m = sel == k
        out[m] = np.stack([a, b2, c2], -1)[m]
    out[s == 0] = np.stack([v, v, v], -1)[s == 0]
    return out.astype(np.uint8)


def pil_hue(img, hue_byte):
    """torchvision adjust_hue on a PIL image: RGB -> HSV, H += hue_byte (mod 256), HSV -> RGB."""
    hsv = pil_rgb_to_hsv(img)
    hsv[..., 0] = (hsv[..., 0].astype(np.int64) + int(hue_byte)) & 255
    return pil_hsv_to_rgb(hsv)


def pil_box_blur_radius(radius, passes=3):
    """BoxBlur.c _gaussian_blur_radius: the extended box radius of `passes` box blurs approximating a Gaussian."""
    r = F32(radius)
    sigma2 = F32(r * r / F32(passes))
    L = F32(np.sqrt(F64(12.0) * F64(sigma2) + F64(1.0)))
    l = F32(np.floor((F64(L) - 1.0) / 2.0))                     # noqa: E741
    a = F32(F32(2) * l + F32(1)) * F32(l * F32(l + F32(1)) - F32(3) * sigma2)
    a = F32(a / F32(F32(6) * F32(sigma2 - F32(l + F32(1)) * F32(l + F32(1)))))
    return F32(l + a)


def pil_box_blur_pass(img, box_radius, axis):
    """One ImagingLineBoxBlur pass along `axis` (edges clamped): ww, fw in 8.24 fixed point, uint8 result."""
    fr = F32(box_radius)
    r = int(fr)
    ww = int(F32(F32(1 << 24) / F32(F32(fr * F32(2)) + F32(1))))
    fw = ((1 << 24) - (2 * r + 1) * ww) // 2
    src = np.moveaxis(img.astype(np.int64), axis, 0)
    n = src.shape[0]
    x = np.arange(n)
    acc = np.zeros_like(src)
    for d in range(-r, r + 1):
        acc += src[np.clip(x + d, 0, n - 1)]
    far = src[np.clip(x - r - 1, 0, n - 1)] + src[np.clip(x + r + 1, 0, n - 1)]
    out = ((acc * ww + far * fw + (1 << 23)) >> 24).astype(np.uint8)
    return np.moveaxis(out, 0, axis)


def pil_gaussian_blur(img, radius, passes=3):
    """img.filter(ImageFilter.GaussianBlur(radius)): `passes` horizontal box passes, then `passes` vertical ones."""
    br = pil_box_blur_radius(radius, passes)
    if br == 0:
        return img.copy()
    for axis in (1, 0):
        for _ in range(passes):
            img = pil_box_blur_pass(img, br, axis)
    return img


def image_to_byte(x):
    """to_pil_image of a float [3,H,W] image in [0, 1]: mul(255).byte() -> uint8 [H,W,3]."""
    return (np.asarray(x, np.float32) * F32(255.0)).astype(np.float32).astype(np.int64).astype(np.uint8).transpose(1, 2, 0)


def aug_image(x, geo, params, crop_hw, lut):
    """One image through _augment_image's chain with the drawn parameters.  x: unnormalised float [3,H,W];
    geo = (resized_h, resized_w, top, left, flip); params: one row of css_b200.aug.draw_image_params' table
    (IMAGE_PARAMS order); lut: float [3,256] byte -> normalised value.  Returns float [3,ch,cw]."""
    rh, rw, top, left, flip = (int(v) for v in geo)
    ch, cw = int(crop_hw[0]), int(crop_hw[1])
    img = pil_resize_bilinear(image_to_byte(x), rh, rw)
    ys = reflect_index(np.arange(top, top + ch), rh)
    xs = reflect_index(np.arange(left, left + cw), rw)
    img = img[ys][:, xs]
    jitter, order, (fb, fc, fs), hue, blur, radius = (params[0], params[1:5], params[5:8], params[8], params[9], params[10])
    if jitter:
        for op in order.astype(np.int64):
            if op == 0:
                img = pil_brightness(img, fb)
            elif op == 1:
                img = pil_contrast(img, fc)
            elif op == 2:
                img = pil_saturation(img, fs)
            else:
                img = pil_hue(img, int(hue))
    if blur:
        img = pil_gaussian_blur(img, radius)
    if flip:
        img = img[:, ::-1]
    lut = np.asarray(lut, np.float32)
    return np.stack([lut[c][img[..., c]] for c in range(3)])
