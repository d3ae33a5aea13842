// The IMAGE's trip through the augmentation, on the GPU and bit-identical to the Pillow chain it replaces
// (css_b200/aug.py::_augment_image: to_pil_image -> bilinear resize -> reflect pad -> crop -> ColorJitter -> GaussianBlur ->
// hflip -> to_tensor + normalize).  The host draws every random parameter (aug.draw_image_params); these kernels replay
// Pillow's 8-bit arithmetic on them.  The specification is oracle/pil_oracle.py (pil_* functions, each checked against the
// installed Pillow): every step below is the same operation sequence.  nvcc contracts a*b+c into FMA by default, which
// would change roundings, so every float / double operation of that arithmetic is an explicit __f*_rn / __d*_rn intrinsic.
//
// Two launches per batch:
//   front: per output pixel -- byte conversion, resize (only the pixels the crop needs: each resized pixel is a pointwise
//          function of the input), reflect pad, crop, the jitter ops that precede contrast; per-image sum of L for
//          contrast's grey level, which needs the whole crop at that point of the chain;
//   back : per 32x32 tile with a halo in shared memory -- contrast and the jitter ops after it, the 3+3 box passes of
//          GaussianBlur, flip, byte -> normalised float through the host-built lookup table.
#include "css_common.cuh"

#define AUG_GEO 5                            // resized_h, resized_w, top, left, flip
#define IMG_FRONT_Y 8                        // front: 32 x 8 threads, one output pixel each
#define IMG_TILE 32                          // back: 32 x 32 output pixels per block
#define BLUR_RMAX 3                          // largest integer box radius (GaussianBlur radius <= 4)
#define BLUR_HALO (3 * (BLUR_RMAX + 1))      // each box pass spoils r + 1 pixels at a tile's inner edge
#define BLUR_SPAN (IMG_TILE + 2 * BLUR_HALO)
#define PIL_PREC 22                          // Resample.c PRECISION_BITS

struct ImgParams {
    int jitter, order[4], hue, blur;
    float fb, fc, fs, radius;
};

__device__ __forceinline__ ImgParams load_params(const float* __restrict__ p) {
    ImgParams q;
    q.jitter = p[CSS_AUG_P_JITTER] != 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) q.order[k] = (int)p[CSS_AUG_P_ORDER + k];
    q.fb = p[CSS_AUG_P_BRIGHTNESS];
    q.fc = p[CSS_AUG_P_CONTRAST];
    q.fs = p[CSS_AUG_P_SATURATION];
    q.hue = (int)p[CSS_AUG_P_HUE_BYTE] & 255;
    q.blur = p[CSS_AUG_P_BLUR] != 0.f;
    q.radius = p[CSS_AUG_P_RADIUS];
    return q;
}

__device__ __forceinline__ uint32_t pack3(const int c[3]) { return (uint32_t)c[0] | ((uint32_t)c[1] << 8) | ((uint32_t)c[2] << 16); }
__device__ __forceinline__ void unpack3(uint32_t v, int c[3]) {
    c[0] = v & 255;
    c[1] = (v >> 8) & 255;
    c[2] = (v >> 16) & 255;
}
__device__ __forceinline__ int clamp8(int v) { return min(max(v, 0), 255); }

// ---- resize (Resample.c, bilinear, box = the whole input) ------------------------------------------------------------------
struct Taps {
    int xmin, n;
    double center, ss, ww;
};

__device__ __forceinline__ double tap_weight(const Taps& t, int x) {
    const double v = fabs(__dmul_rn(__dadd_rn(__dsub_rn((double)(x + t.xmin), t.center), 0.5), t.ss));
    return v < 1.0 ? __dsub_rn(1.0, v) : 0.0;
}

// precompute_coeffs for output index xx: source window and the sum of its weights
__device__ Taps taps_of(int n_in, int n_out, int xx) {
    Taps t;
    const double scale = __ddiv_rn((double)n_in, (double)n_out);
    const double filterscale = scale < 1.0 ? 1.0 : scale;      // support = 1.0 * filterscale
    t.center = __dmul_rn(__dadd_rn((double)xx, 0.5), scale);
    t.ss = __ddiv_rn(1.0, filterscale);
    t.xmin = max((int)__dadd_rn(__dsub_rn(t.center, filterscale), 0.5), 0);
    const int xmax = min((int)__dadd_rn(__dadd_rn(t.center, filterscale), 0.5), n_in);
    t.n = xmax - t.xmin;
    t.ww = 0.0;
    for (int x = 0; x < t.n; ++x) t.ww = __dadd_rn(t.ww, tap_weight(t, x));
    return t;
}

// normalize_coeffs_8bpc: weight / sum -> 22-bit fixed point with +-0.5 rounding
__device__ __forceinline__ int tap_fixed(const Taps& t, int x) {
    double k = tap_weight(t, x);
    if (t.ww != 0.0) k = __ddiv_rn(k, t.ww);
    const double s = __dmul_rn(k, (double)(1 << PIL_PREC));
    return k < 0.0 ? (int)__dadd_rn(-0.5, s) : (int)__dadd_rn(0.5, s);
}

// to_pil_image: mul(255).byte()
__device__ __forceinline__ int to_byte(const float* p) { return ((int)__fmul_rn(__ldg(p), 255.f)) & 255; }

// resized pixel (ry, rx) of one image: the horizontal pass first (clipped to uint8), then the vertical one; an axis that
// keeps its size is copied
__device__ void resample_px(const float* __restrict__ img, int H, int W, int rh, int rw, int ry, int rx, int out[3]) {
    const size_t plane = (size_t)H * W;
    const bool nh = rw != W, nv = rh != H;
    Taps th, tv;
    if (nh) th = taps_of(W, rw, rx);
    if (nv) tv = taps_of(H, rh, ry);
    const int y0 = nv ? tv.xmin : ry, ny = nv ? tv.n : 1;
    int accv[3] = {1 << (PIL_PREC - 1), 1 << (PIL_PREC - 1), 1 << (PIL_PREC - 1)};
    for (int j = 0; j < ny; ++j) {
        const float* row = img + (size_t)(y0 + j) * W;
        int hv[3];
        if (nh) {
            int acc[3] = {1 << (PIL_PREC - 1), 1 << (PIL_PREC - 1), 1 << (PIL_PREC - 1)};
            for (int i = 0; i < th.n; ++i) {
                const int k = tap_fixed(th, i);
#pragma unroll
                for (int c = 0; c < 3; ++c) acc[c] += to_byte(row + c * plane + th.xmin + i) * k;
            }
#pragma unroll
            for (int c = 0; c < 3; ++c) hv[c] = clamp8(acc[c] >> PIL_PREC);
        } else {
#pragma unroll
            for (int c = 0; c < 3; ++c) hv[c] = to_byte(row + c * plane + rx);
        }
        if (!nv) {
#pragma unroll
            for (int c = 0; c < 3; ++c) out[c] = hv[c];
            return;
        }
        const int k = tap_fixed(tv, j);
#pragma unroll
        for (int c = 0; c < 3; ++c) accv[c] += hv[c] * k;
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) out[c] = clamp8(accv[c] >> PIL_PREC);
}

// np.pad(mode='reflect') index, also when the pad is longer than the axis
__device__ __forceinline__ int reflect_index(int i, int n) {
    if (n == 1) return 0;
    const int p = 2 * (n - 1), m = i % p;
    return m < n ? m : p - m;
}

// ---- ColorJitter (ImageEnhance = Blend.c with a float alpha; Convert.c L24 and RGB <-> HSV) -----------------------------
__device__ __forceinline__ int blend(int in1, int in2, float a) {
    const float t = __fadd_rn((float)in1, __fmul_rn(a, (float)(in2 - in1)));
    return (int)fminf(fmaxf(t, 0.f), 255.f);                  // interpolation stays in range; extrapolation clips
}

__device__ __forceinline__ int l24(const int c[3]) { return (c[0] * 19595 + c[1] * 38470 + c[2] * 7471 + 0x8000) >> 16; }

__device__ __forceinline__ void rgb_to_hsv(const int c[3], int hsv[3]) {
    const int r = c[0], g = c[1], b = c[2];
    const int maxc = max(r, max(g, b)), minc = min(r, min(g, b));
    hsv[2] = maxc;
    if (maxc == minc) {
        hsv[0] = hsv[1] = 0;
        return;
    }
    const float cr = (float)(maxc - minc);
    const float s = __fdiv_rn(cr, (float)maxc);
    const float rc = __fdiv_rn((float)(maxc - r), cr), gc = __fdiv_rn((float)(maxc - g), cr), bc = __fdiv_rn((float)(maxc - b), cr);
    float h;
    if (r == maxc) h = __fsub_rn(bc, gc);
    else if (g == maxc) h = __double2float_rn(__dsub_rn(__dadd_rn(2.0, (double)rc), (double)bc));
    else h = __double2float_rn(__dsub_rn(__dadd_rn(4.0, (double)gc), (double)rc));
    h = __double2float_rn(fmod(__dadd_rn(__ddiv_rn((double)h, 6.0), 1.0), 1.0));
    hsv[0] = clamp8((int)__dmul_rn((double)h, 255.0));
    hsv[1] = clamp8((int)__dmul_rn((double)s, 255.0));
}

__device__ __forceinline__ void hsv_to_rgb(const int hsv[3], int c[3]) {
    const int h = hsv[0], s = hsv[1], v = hsv[2];
    if (s == 0) {
        c[0] = c[1] = c[2] = v;
        return;
    }
    const double hd = __ddiv_rn(__dmul_rn((double)h, 6.0), 255.0);
    const int i = (int)floor(hd);
    const float f = __double2float_rn(__dsub_rn(hd, (double)(float)i));
    const float fs = __double2float_rn(__ddiv_rn((double)s, 255.0));
    const double vd = (double)v;
    const int p = clamp8((int)round(__dmul_rn(vd, __dsub_rn(1.0, (double)fs))));
    const int q = clamp8((int)round(__dmul_rn(vd, __dsub_rn(1.0, (double)__fmul_rn(fs, f)))));
    const int t = clamp8((int)round(__dmul_rn(vd, __dsub_rn(1.0, __dmul_rn((double)fs, __dsub_rn(1.0, (double)f))))));
    switch (i % 6) {
        case 0: c[0] = v; c[1] = t; c[2] = p; break;
        case 1: c[0] = q; c[1] = v; c[2] = p; break;
        case 2: c[0] = p; c[1] = v; c[2] = t; break;
        case 3: c[0] = p; c[1] = q; c[2] = v; break;
        case 4: c[0] = t; c[1] = p; c[2] = v; break;
        default: c[0] = v; c[1] = p; c[2] = q; break;
    }
}

// one ColorJitter op (0 brightness, 1 contrast with grey level `mean`, 2 saturation, 3 hue) on one pixel
__device__ __forceinline__ void jitter_op(const ImgParams& P, int op, int mean, int c[3]) {
    if (op == 0) {
#pragma unroll
        for (int k = 0; k < 3; ++k) c[k] = blend(0, c[k], P.fb);
    } else if (op == 1) {
#pragma unroll
        for (int k = 0; k < 3; ++k) c[k] = blend(mean, c[k], P.fc);
    } else if (op == 2) {
        const int l = l24(c);
#pragma unroll
        for (int k = 0; k < 3; ++k) c[k] = blend(l, c[k], P.fs);
    } else {
        int hsv[3];
        rgb_to_hsv(c, hsv);
        hsv[0] = (hsv[0] + P.hue) & 255;
        hsv_to_rgb(hsv, c);
    }
}

// ---- GaussianBlur (BoxBlur.c) --------------------------------------------------------------------------------------------
__device__ float box_blur_radius(float radius) {                // _gaussian_blur_radius(radius, passes = 3)
    const float sigma2 = __fdiv_rn(__fmul_rn(radius, radius), 3.f);
    const float L = __double2float_rn(__dsqrt_rn(__dadd_rn(__dmul_rn(12.0, (double)sigma2), 1.0)));
    const float l = __double2float_rn(floor(__ddiv_rn(__dsub_rn((double)L, 1.0), 2.0)));
    const float l1 = __fadd_rn(l, 1.f);
    float a = __fmul_rn(__fadd_rn(__fmul_rn(2.f, l), 1.f), __fsub_rn(__fmul_rn(l, l1), __fmul_rn(3.f, sigma2)));
    a = __fdiv_rn(a, __fmul_rn(6.f, __fsub_rn(sigma2, __fmul_rn(l1, l1))));
    return __fadd_rn(l, a);
}

// ---- kernels ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32 * IMG_FRONT_Y) aug_image_front_kernel(const float* __restrict__ images, int H, int W,
                                                                           const int* __restrict__ geo,
                                                                           const float* __restrict__ params, int ch, int cw,
                                                                           uint32_t* __restrict__ pix,
                                                                           unsigned long long* __restrict__ lsum) {
    css_pdl_enter();
    __shared__ unsigned warp_l[IMG_FRONT_Y];
    const int b = blockIdx.z, x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * IMG_FRONT_Y + threadIdx.y;
    const int* g = geo + b * AUG_GEO;
    const int rh = g[0], rw = g[1], top = g[2], left = g[3];
    const ImgParams P = load_params(params + (size_t)b * CSS_AUG_IMAGE_PARAMS);
    unsigned l = 0;
    if (x < cw && y < ch) {
        int c[3];
        resample_px(images + (size_t)b * 3 * H * W, H, W, rh, rw, reflect_index(top + y, rh), reflect_index(left + x, rw), c);
        if (P.jitter) {
            bool before = true;                                 // the ops ahead of contrast
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                before = before && P.order[k] != 1;
                if (before) jitter_op(P, P.order[k], 0, c);
            }
            l = l24(c);
        }
        pix[((size_t)b * ch + y) * cw + x] = pack3(c);
    }
    if (!P.jitter) return;                                      // uniform per block
    l = __reduce_add_sync(0xffffffffu, l);
    if (threadIdx.x == 0) warp_l[threadIdx.y] = l;
    __syncthreads();
    if (threadIdx.x == 0 && threadIdx.y == 0) {
        unsigned long long s = 0;
#pragma unroll
        for (int w = 0; w < IMG_FRONT_Y; ++w) s += warp_l[w];
        atomicAdd(lsum + b, s);
    }
}

__global__ void __launch_bounds__(256) aug_image_back_kernel(const uint32_t* __restrict__ pix,
                                                             const unsigned long long* __restrict__ lsum,
                                                             const int* __restrict__ geo, const float* __restrict__ params,
                                                             const float* __restrict__ lut, int ch, int cw,
                                                             float* __restrict__ out) {
    css_pdl_enter();
    __shared__ uint32_t buf[2][BLUR_SPAN * BLUR_SPAN];
    __shared__ float slut[3 * 256];
    const int b = blockIdx.z, x0 = blockIdx.x * IMG_TILE, y0 = blockIdx.y * IMG_TILE, tid = threadIdx.x;
    for (int i = tid; i < 3 * 256; i += 256) slut[i] = lut[i];
    const ImgParams P = load_params(params + (size_t)b * CSS_AUG_IMAGE_PARAMS);
    const int flip = geo[b * AUG_GEO + 4];
    int mean = 0;
    if (P.jitter)                                               // ImageEnhance.Contrast: int(mean(L) + 0.5)
        mean = (int)__dadd_rn(__ddiv_rn((double)lsum[b], (double)((long long)ch * cw)), 0.5);
    // region = tile + halo, cut at the image's edges (there the clamped reads of the box passes are Pillow's)
    const int halo = P.blur ? BLUR_HALO : 0;
    const int gx0 = max(x0 - halo, 0), gx1 = min(x0 + IMG_TILE + halo, cw);
    const int gy0 = max(y0 - halo, 0), gy1 = min(y0 + IMG_TILE + halo, ch);
    const int sw = gx1 - gx0, sh = gy1 - gy0;
    for (int i = tid; i < sw * sh; i += 256) {
        const int yy = gy0 + i / sw, xx = gx0 + i % sw;
        uint32_t v = pix[((size_t)b * ch + yy) * cw + xx];
        if (P.jitter) {
            int c[3];
            unpack3(v, c);
            bool after = false;                                 // contrast and the ops after it
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                after = after || P.order[k] == 1;
                if (after) jitter_op(P, P.order[k], mean, c);
            }
            v = pack3(c);
        }
        buf[0][i] = v;
    }
    __syncthreads();
    int cur = 0;
    if (P.blur) {
        const float br = box_blur_radius(P.radius);
        if (br != 0.f) {
            const int r = (int)br;
            const unsigned ww = (unsigned)__fdiv_rn(16777216.f, __fadd_rn(__fmul_rn(br, 2.f), 1.f));
            const unsigned fw = ((1u << 24) - (unsigned)(2 * r + 1) * ww) / 2;
            for (int pass = 0; pass < 6; ++pass) {              // 3 horizontal passes, then 3 vertical ones
                const bool vert = pass >= 3;
                const int n = vert ? sh : sw;
                const uint32_t* src = buf[cur];
                uint32_t* dst = buf[cur ^ 1];
                for (int i = tid; i < sw * sh; i += 256) {
                    const int row = i / sw, col = i % sw, pos = vert ? row : col;
                    auto at = [&](int p) {
                        p = min(max(p, 0), n - 1);
                        return src[vert ? p * sw + col : row * sw + p];
                    };
                    unsigned acc[3] = {0, 0, 0}, far[3];
                    for (int d = -r; d <= r; ++d) {
                        const uint32_t v = at(pos + d);
                        acc[0] += v & 255;
                        acc[1] += (v >> 8) & 255;
                        acc[2] += (v >> 16) & 255;
                    }
                    const uint32_t a = at(pos - r - 1), z = at(pos + r + 1);
                    far[0] = (a & 255) + (z & 255);
                    far[1] = ((a >> 8) & 255) + ((z >> 8) & 255);
                    far[2] = ((a >> 16) & 255) + ((z >> 16) & 255);
                    int c[3];
#pragma unroll
                    for (int k = 0; k < 3; ++k) c[k] = (int)((acc[k] * ww + far[k] * fw + (1u << 23)) >> 24);
                    dst[i] = pack3(c);
                }
                __syncthreads();
                cur ^= 1;
            }
        }
    }
    const size_t plane = (size_t)ch * cw;
    for (int i = tid; i < IMG_TILE * IMG_TILE; i += 256) {
        const int yy = y0 + i / IMG_TILE, xx = x0 + i % IMG_TILE;
        if (yy >= ch || xx >= cw) continue;
        int c[3];
        unpack3(buf[cur][(yy - gy0) * sw + (xx - gx0)], c);
        const size_t o = (size_t)b * 3 * plane + (size_t)yy * cw + (flip ? cw - 1 - xx : xx);
#pragma unroll
        for (int k = 0; k < 3; ++k) out[o + k * plane] = slut[k * 256 + c[k]];
    }
}

static size_t lsum_bytes(int B) { return ((size_t)B * sizeof(unsigned long long) + 255) & ~(size_t)255; }

extern "C" size_t css_aug_image_workspace_bytes(int B, int ch, int cw) {
    if (B <= 0 || ch <= 0 || cw <= 0) return 0;
    return lsum_bytes(B) + (size_t)B * ch * cw * sizeof(uint32_t);
}

extern "C" int css_aug_image(const float* images, int B, int H, int W, const int32_t* geometry, const float* params,
                             const float* lut, int ch, int cw, void* workspace, size_t workspace_bytes, float* out, void* stream) {
    CSS_CHECK_ARG(images && geometry && params && lut && workspace && out, CSS_E_ARG, "css_aug_image: null pointer");
    CSS_CHECK_ARG(B > 0 && B <= 65535 && H > 0 && W > 0 && ch > 0 && cw > 0 && ch <= 65535 * IMG_FRONT_Y, CSS_E_ARG,
                  "css_aug_image: bad size");
    CSS_CHECK_ARG((size_t)B * 3 * H * W < (1ull << 62) && (size_t)B * ch * cw < (1ull << 62), CSS_E_SIZE, "css_aug_image: too large");
    CSS_CHECK_ARG(workspace_bytes >= css_aug_image_workspace_bytes(B, ch, cw), CSS_E_ARG,
                  "css_aug_image: workspace of %zu bytes, %zu needed", workspace_bytes, css_aug_image_workspace_bytes(B, ch, cw));
    cudaStream_t st = (cudaStream_t)stream;
    unsigned long long* lsum = (unsigned long long*)workspace;
    uint32_t* pix = (uint32_t*)((char*)workspace + lsum_bytes(B));
    cudaError_t e = cudaMemsetAsync(lsum, 0, (size_t)B * sizeof(unsigned long long), st);
    if (e != cudaSuccess) {
        css_set_error("css_aug_image: %s", cudaGetErrorString(e));
        return (int)e;
    }
    css_launch(aug_image_front_kernel, dim3((cw + 31) / 32, (ch + IMG_FRONT_Y - 1) / IMG_FRONT_Y, B), dim3(32, IMG_FRONT_Y),
               (size_t)0, st, images, H, W, geometry, params, ch, cw, pix, lsum);
    css_launch(aug_image_back_kernel, dim3((cw + IMG_TILE - 1) / IMG_TILE, (ch + IMG_TILE - 1) / IMG_TILE, B), dim3(256),
               (size_t)0, st, (const uint32_t*)pix, (const unsigned long long*)lsum, geometry, params, lut, ch, cw, out);
    CSS_CHECK_LAUNCH("css_aug_image", 2);
    return 0;
}
