// Stage 3 selection: valid / hard class sets per pixel and their ORDER-PRESERVING per-class compaction, plus the fused
// threshold glue that produces label_all / mask_all at representation resolution.
// Reference: generalframeworks/loss/loss.py:80,94-99,111-113; mix_label.py:175-183; cross_label.py:178-185;
// ori_pseudo.py:171-178; generalframeworks/utils.py:116-136.
//
// Compaction is a three-kernel stable counting sort (classify+count per 256-pixel tile -> exclusive scan over tiles ->
// scatter with ballot ranks), because the reference's sampled indices are ranks in row-major order inside each class
// list (SURVEY.md 7.3-3); an atomic-counter compaction would scramble them.  The scatter is a separate entry point
// (css_select_lists): a valid-list entry carries its pixel's inverse norm, which is final only once the rows are.
#include "css_common.cuh"

extern "C" int css_select_tiles(int N) { return (N + CSS_SEL_TILE - 1) / CSS_SEL_TILE; }

// tile_counts layout: row r = kind*C + c (kind 0 = valid, 1 = hard), T entries per row.
__global__ void __launch_bounds__(CSS_SEL_TILE) select_classify_kernel(const float* __restrict__ label, const float* __restrict__ mask,
                                                                       const float* __restrict__ prob, float strong, int C, int hw,
                                                                       int N, int T, uint32_t* __restrict__ valid_bits,
                                                                       uint32_t* __restrict__ hard_bits, int32_t* __restrict__ tile_counts,
                                                                       int32_t* __restrict__ meta) {
    css_pdl_enter();
    __shared__ int cnt[2 * CSS_CMAX];
    if (threadIdx.x < 2 * CSS_CMAX) cnt[threadIdx.x] = 0;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        meta[CSS_META_TICKET] = 0;           // ticket of the scan kernel's last-CTA election
        meta[CSS_META_ROWS_STALE] = 0;       // raised by css_rows_refresh's comparison later in the same step
    }
    __syncthreads();
    const int p = blockIdx.x * CSS_SEL_TILE + threadIdx.x;
    uint32_t vb = 0, hb = 0;
    if (p < N) {
        const int b = p / hw, s = p - b * hw;
        const float m = __ldg(mask + p);
        const float* lp = label + (size_t)b * C * hw + s;
        const float* pp = prob + (size_t)b * C * hw + s;
        // all C label planes of the pixel in flight at once, then the probabilities of its (normally single) valid class:
        // two round trips per pixel instead of a label -> prob chain per group of four classes
        float l[CSS_CMAX];
#pragma unroll
        for (int c = 0; c < CSS_CMAX; ++c) l[c] = (c < C) ? ldg_stream(lp + (size_t)c * hw) : 0.f;
#pragma unroll
        for (int c = 0; c < CSS_CMAX; ++c)
            if (__fmul_rn(l[c], m) != 0.f) vb |= 1u << c;       // valid_pixel = label * mask (loss.py:80), .bool() (:99,:111)
        for (uint32_t bits = vb; bits; bits &= bits - 1) {
            const int c = __ffs(bits) - 1;
            if (__ldg(pp + (size_t)c * hw) < strong) hb |= 1u << c;       // prob < strong_threshold (loss.py:99)
        }
        valid_bits[p] = vb;
        hard_bits[p] = hb;
    }
    uint32_t uni = __reduce_or_sync(0xffffffffu, vb);
    const int lane = threadIdx.x & 31;
    while (uni) {
        const int c = __ffs(uni) - 1;
        uni &= uni - 1;
        const int nv = __popc(__ballot_sync(0xffffffffu, (vb >> c) & 1u));
        const int nh = __popc(__ballot_sync(0xffffffffu, (hb >> c) & 1u));
        if (lane == 0) {
            atomicAdd(&cnt[c], nv);
            if (nh) atomicAdd(&cnt[CSS_CMAX + c], nh);
        }
    }
    __syncthreads();
    if (threadIdx.x < 2 * C) {
        const int kind = threadIdx.x / C, c = threadIdx.x - kind * C;
        tile_counts[(size_t)threadIdx.x * T + blockIdx.x] = cnt[kind * CSS_CMAX + c];
    }
}

// One CTA per tile_counts row (2C rows): exclusive scan over the T tiles in place.  Thread t owns a contiguous segment
// (independent loads), the 256 segment totals are scanned with shuffles.  The CTA that finishes last (ticket in
// meta[CSS_META_TICKET], zeroed by the classify kernel) assembles class totals and the present-class table into meta.
#define SCAN_THREADS 256
#define SCAN_MAXSEG 16
__global__ void __launch_bounds__(SCAN_THREADS) select_scan_kernel(int32_t* __restrict__ tile_counts, int C, int T, int32_t* __restrict__ meta) {
    css_pdl_enter();
    __shared__ int wsum[SCAN_THREADS / 32];
    __shared__ int is_last;
    const int r = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    int32_t* row = tile_counts + (size_t)r * T;
    const int len = (T + SCAN_THREADS - 1) / SCAN_THREADS;
    const int b0 = min(tid * len, T), b1 = min(b0 + len, T);
    int vals[SCAN_MAXSEG];
    int tot = 0;
    if (len <= SCAN_MAXSEG) {
#pragma unroll
        for (int i = 0; i < SCAN_MAXSEG; ++i) vals[i] = (b0 + i < b1) ? row[b0 + i] : 0;
#pragma unroll
        for (int i = 0; i < SCAN_MAXSEG; ++i) tot += vals[i];
    } else {
        for (int i = b0; i < b1; ++i) tot += row[i];
    }
    int inc = tot;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int n = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += n;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    int woff = 0, total = 0;
#pragma unroll
    for (int w2 = 0; w2 < SCAN_THREADS / 32; ++w2) {
        if (w2 < warp) woff += wsum[w2];
        total += wsum[w2];
    }
    int run = woff + inc - tot;
    if (len <= SCAN_MAXSEG) {
#pragma unroll
        for (int i = 0; i < SCAN_MAXSEG; ++i) {
            if (b0 + i < b1) row[b0 + i] = run;
            run += vals[i];
        }
    } else {
        for (int i = b0; i < b1; ++i) {
            const int v = row[i];
            row[i] = run;
            run += v;
        }
    }
    if (tid == 0) {
        const int kind = r / C, c = r - kind * C;
        meta[(kind ? CSS_META_N_HARD : CSS_META_N_VALID) + c] = total;
        __threadfence();
        is_last = (atomicAdd(meta + CSS_META_TICKET, 1) == 2 * C - 1);
    }
    __syncthreads();
    if (is_last && tid < 32) {
        // the last CTA's first warp builds the slot tables: lane c owns class c, so the per-class counts are fetched in ONE
        // round trip (a single thread walking 32 volatile words paid ~32 dependent L2 latencies)
        __threadfence();
        const int c = tid;
        int nv = 0;
        if (c < C) {
            nv = *((volatile int32_t*)meta + CSS_META_N_VALID + c);
        } else {
            meta[CSS_META_N_VALID + c] = 0;
            meta[CSS_META_N_HARD + c] = 0;
        }
        const unsigned present = __ballot_sync(0xffffffffu, c < C && nv > 0);    // classes with no local valid pixel are skipped (loss.py:96-97)
        const int V = __popc(present);
        if ((present >> c) & 1u) {
            const int slot = __popc(present & ((1u << c) - 1u));
            meta[CSS_META_CLS_OF_SLOT + slot] = c;
            meta[CSS_META_SLOT_OF_CLS + c] = slot;
        } else {
            meta[CSS_META_SLOT_OF_CLS + c] = -1;
        }
        if (c >= V) meta[CSS_META_CLS_OF_SLOT + c] = -1;
        if (c == 0) meta[CSS_META_V] = V;
    }
}

// valid_list entry = {pixel id, bits of 1 / max(||r||, 1e-8)}: the scorer's one load per candidate, and the same IEEE division
// it would do (the library builds without fast math), so the bits are those of the division in the scorer
__global__ void __launch_bounds__(CSS_SEL_TILE) select_scatter_kernel(const uint32_t* __restrict__ valid_bits, const uint32_t* __restrict__ hard_bits,
                                                                      const int32_t* __restrict__ tile_off, const float* __restrict__ norms,
                                                                      int C, int N, int T, int2* __restrict__ valid_list,
                                                                      int32_t* __restrict__ hard_list) {
    css_pdl_enter();
    __shared__ int wcnt[2][CSS_CMAX][CSS_SEL_TILE / 32];
    __shared__ int toff[2 * CSS_CMAX];             // this tile's offsets of all 2C lists: one round trip, not one per class
    for (int i = threadIdx.x; i < 2 * CSS_CMAX * (CSS_SEL_TILE / 32); i += CSS_SEL_TILE) (&wcnt[0][0][0])[i] = 0;
    if (threadIdx.x < 2 * C) toff[threadIdx.x] = tile_off[(size_t)threadIdx.x * T + blockIdx.x];
    __syncthreads();
    const int p = blockIdx.x * CSS_SEL_TILE + threadIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t vb = (p < N) ? valid_bits[p] : 0u;
    const uint32_t hb = (p < N) ? hard_bits[p] : 0u;
    const int inv_bits = vb ? __float_as_int(1.f / fmaxf(norms[p], 1e-8f)) : 0;
    const uint32_t uni = __reduce_or_sync(0xffffffffu, vb);
    for (uint32_t u = uni; u;) {
        const int c = __ffs(u) - 1;
        u &= u - 1;
        const int nv = __popc(__ballot_sync(0xffffffffu, (vb >> c) & 1u));
        const int nh = __popc(__ballot_sync(0xffffffffu, (hb >> c) & 1u));
        if (lane == 0) {
            wcnt[0][c][warp] = nv;
            wcnt[1][c][warp] = nh;
        }
    }
    __syncthreads();
    const uint32_t lt = (1u << lane) - 1u;
    for (uint32_t u = uni; u;) {
        const int c = __ffs(u) - 1;
        u &= u - 1;
        const uint32_t bv = __ballot_sync(0xffffffffu, (vb >> c) & 1u);
        const uint32_t bh = __ballot_sync(0xffffffffu, (hb >> c) & 1u);
        int ov = 0, oh = 0;
        for (int w2 = 0; w2 < warp; ++w2) {
            ov += wcnt[0][c][w2];
            oh += wcnt[1][c][w2];
        }
        if ((vb >> c) & 1u)
            valid_list[(size_t)c * N + toff[c] + ov + __popc(bv & lt)] = make_int2(p, inv_bits);
        if ((hb >> c) & 1u)
            hard_list[(size_t)c * N + toff[C + c] + oh + __popc(bh & lt)] = p;
    }
}

extern "C" int css_select(const float* label, const float* mask, const float* prob, float strong_threshold, int B2, int C,
                          int h, int w, uint32_t* valid_bits, uint32_t* hard_bits, int32_t* tile_counts, int32_t* meta, void* stream) {
    CSS_CHECK_ARG(label && mask && prob && valid_bits && hard_bits && tile_counts && meta, CSS_E_ARG, "css_select: null pointer");
    CSS_CHECK_ARG(B2 > 0 && h > 0 && w > 0, CSS_E_ARG, "css_select: non-positive size");
    CSS_CHECK_ARG(C >= 1 && C <= CSS_CMAX, CSS_E_DIM, "css_select: C must be in [1,%d]", CSS_CMAX);
    CSS_CHECK_ARG((long long)B2 * h * w * CSS_CMAX < (1ll << 31), CSS_E_SIZE, "css_select: too many pixels");
    cudaStream_t st = (cudaStream_t)stream;
    const int hw = h * w, N = B2 * hw, T = css_select_tiles(N);
    css_launch(select_classify_kernel, dim3(T), dim3(CSS_SEL_TILE), (size_t)(0), (cudaStream_t)(st), label, mask, prob, strong_threshold, C, hw, N, T, valid_bits, hard_bits,
                                                      tile_counts, meta);
    css_launch(select_scan_kernel, dim3(2 * C), dim3(SCAN_THREADS), (size_t)(0), (cudaStream_t)(st), tile_counts, C, T, meta);
    CSS_CHECK_LAUNCH("css_select", 2);
    return 0;
}

extern "C" int css_select_lists(const uint32_t* valid_bits, const uint32_t* hard_bits, const int32_t* tile_counts, const float* norms,
                                int C, int N, int32_t* valid_list, int32_t* hard_list, void* stream) {
    CSS_CHECK_ARG(valid_bits && hard_bits && tile_counts && norms && valid_list && hard_list, CSS_E_ARG, "css_select_lists: null pointer");
    CSS_CHECK_ARG(N > 0, CSS_E_ARG, "css_select_lists: non-positive size");
    CSS_CHECK_ARG(C >= 1 && C <= CSS_CMAX, CSS_E_DIM, "css_select_lists: C must be in [1,%d]", CSS_CMAX);
    CSS_CHECK_ARG((long long)N * CSS_CMAX < (1ll << 31), CSS_E_SIZE, "css_select_lists: too many pixels");
    const int T = css_select_tiles(N);
    css_launch(select_scatter_kernel, dim3(T), dim3(CSS_SEL_TILE), (size_t)(0), (cudaStream_t)stream, valid_bits, hard_bits, tile_counts, norms, C, N, T,
               reinterpret_cast<int2*>(valid_list), hard_list);
    CSS_CHECK_LAUNCH("css_select_lists", 1);
    return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// K0 (SURVEY.md 8(f)-1): weak-threshold mask + one-hot + nearest down-sampling in one pass.
//   mask_all  = nearest(cat(label_l >= 0, conf_u >= weak))                         mix_label.py:176-178
//   label_all = nearest(cat(onehot(relu(label_l)), onehot_u))                      mix_label.py:180-183
//   mode 0: onehot_u = label_onehot(label_u) (relu, utils.py:116-125); mode 1: label_onehot_2(label_u)[:,1:] (utils.py:127-136)
// Nearest source index as ATen: min(int(floorf(dst * (in/out))), in-1), scale in fp32.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) threshold_glue_kernel(const int64_t* __restrict__ label_l, const int64_t* __restrict__ label_u,
                                                             const float* __restrict__ conf_u, float weak, int mode, int B, int C,
                                                             int H, int W, int h, int w, float sy, float sx,
                                                             float* __restrict__ label_all, float* __restrict__ mask_all) {
    css_pdl_enter();
    const int hw = h * w;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= 2 * B * hw) return;
    const int bb = p / hw, s = p - bb * hw;
    const int y = s / w, x = s - y * w;
    const int Y = min((int)floorf(__fmul_rn((float)y, sy)), H - 1);
    const int X = min((int)floorf(__fmul_rn((float)x, sx)), W - 1);
    int cls;
    float m;
    if (bb < B) {
        const long long l = label_l[((size_t)bb * H + Y) * W + X];
        m = (l >= 0) ? 1.f : 0.f;
        cls = (int)max(l, 0ll);
    } else {
        const size_t o = ((size_t)(bb - B) * H + Y) * W + X;
        const long long l = label_u[o];
        m = (conf_u[o] >= weak) ? 1.f : 0.f;
        cls = (mode == 1) ? (int)l : (int)max(l, 0ll);
    }
    mask_all[p] = m;
    float* o = label_all + (size_t)bb * C * hw + s;
    for (int c = 0; c < C; ++c) o[(size_t)c * hw] = (c == cls) ? 1.f : 0.f;
}

extern "C" int css_threshold_glue(const int64_t* label_l, const int64_t* label_u, const float* conf_u, float weak_threshold,
                                  int mode, int B, int C, int H, int W, int h, int w, float* label_all, float* mask_all,
                                  void* stream) {
    CSS_CHECK_ARG(label_l && label_u && conf_u && label_all && mask_all, CSS_E_ARG, "css_threshold_glue: null pointer");
    CSS_CHECK_ARG(B > 0 && H > 0 && W > 0 && h > 0 && w > 0, CSS_E_ARG, "css_threshold_glue: non-positive size");
    CSS_CHECK_ARG(mode == 0 || mode == 1, CSS_E_ARG, "css_threshold_glue: bad mode %d", mode);
    CSS_CHECK_ARG(C >= 1 && C <= CSS_CMAX, CSS_E_DIM, "css_threshold_glue: C must be in [1,%d]", CSS_CMAX);
    CSS_CHECK_ARG(2ll * B * h * w * CSS_CMAX < (1ll << 31), CSS_E_SIZE, "css_threshold_glue: too many pixels");
    const int n = 2 * B * h * w;
    css_launch(threshold_glue_kernel, dim3((n + 255) / 256), dim3(256), (size_t)(0), (cudaStream_t)((cudaStream_t)stream), label_l, label_u, conf_u, weak_threshold, mode, B, C,
                                                                            H, W, h, w, (float)H / (float)h, (float)W / (float)w,
                                                                            label_all, mask_all);
    CSS_CHECK_LAUNCH("css_threshold_glue", 1);
    return 0;
}
