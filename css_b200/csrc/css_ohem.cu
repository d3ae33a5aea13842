// DESIGN.md f-5: ProbOhemCrossEntropy2d -- the supervised OHEM cross-entropy of the CityScapes scripts (reference:
// generalframeworks/loss/loss.py:8-46, called at mix_label.py:168-171), without a host synchronisation.
//   valid  = label != ignore_index (labels outside [0,C) count as ignored)
//   p_t    = softmax(pred[:, p])[label_p]
//   OHEM applies when min_kept > 0 and #valid >= min_kept; then kept = valid & p_t <= T, T = max(float32(thresh), kth),
//          kth = the min_kept-th smallest p_t of the valid pixels; otherwise kept = valid
//   loss   = sum_kept w[y] * (lse - x_y) / sum_kept w[y]          (w = 1 without class weights; 0/0 = nan when nothing is kept)
// The forward pass reads pred once (the C logits of a pixel stay in registers), writes lse / p_t / nll (12 B per pixel) and
// counts #valid and #(valid & p_t <= T0).  When that count is below min_kept, kth > T0 and an exact radix select finds it on
// the device: three digit passes (11 / 11 / 10 bits) over the bit patterns of p_t (non-negative floats: uint32 order is
// float order), each a shared-memory histogram pass plus a one-CTA scan, then one pass sums the kept set.  Every one of these
// launches reads the counts first and returns at once when the select is not needed, so there is no host round trip and the
// whole loss is CUDA-graph capturable.  Counts are integers and float sums are taken per CTA and added in a fixed order:
// results are deterministic.  The backward pass reads pred (kept pixels only) and lse once and writes grad_pred once.
#include "css_common.cuh"

#define OHEM_THREADS 256
#define OHEM_GRID 512          // CTAs of the grid-stride passes (histograms, kept-set sums)
#define OHEM_BINS 2048         // radix digits: bits 31..21, 20..10, 9..0

struct OhemState {
    int32_t num_valid;         // forward pass
    int32_t num_le_t0;         // forward pass: #(valid & p_t <= T0)
    int32_t num_sel;           // kept-set pass: #(valid & p_t <= kth)
    int32_t k;                 // rank still to find inside the digits fixed so far
    uint32_t prefix;           // bits of kth fixed so far
    float threshold;           // finalize: T used (+inf when OHEM does not apply)
    float scale;               // finalize: 1 / sum_kept w[y]
    int32_t pad;
    uint32_t hist[3][OHEM_BINS];
};

static inline size_t ohem_align(size_t x) { return (x + 255) & ~(size_t)255; }

struct OhemLayout {
    size_t state, fwd_partials, sel_partials, lse, pt, nll, total;
};

static OhemLayout ohem_layout(int B, int H, int W) {
    const size_t N = (size_t)B * H * W, nblk = (size_t)((H * W + OHEM_THREADS - 1) / OHEM_THREADS) * B;
    OhemLayout L;
    L.pt = 0;                                                 // documented in the header: p_t first
    L.lse = L.pt + ohem_align(N * sizeof(float));
    L.nll = L.lse + ohem_align(N * sizeof(float));
    L.state = L.nll + ohem_align(N * sizeof(float));
    L.fwd_partials = L.state + ohem_align(sizeof(OhemState));
    L.sel_partials = L.fwd_partials + ohem_align(nblk * 4 * sizeof(float));
    L.total = L.sel_partials + ohem_align(OHEM_GRID * 2 * sizeof(float));
    return L;
}

// the radix select (and the kept-set pass) runs only when OHEM applies and fewer than min_kept valid pixels have p_t <= T0
__device__ __forceinline__ bool ohem_needs_select(const OhemState* st, int min_kept) {
    return min_kept > 0 && st->num_valid >= min_kept && st->num_le_t0 < min_kept;
}

// fixed-order block sum of two floats (shuffle tree, then the warp sums in warp order); result valid in thread 0
__device__ __forceinline__ void ohem_block_sum2(float& a, float& b) {
    __shared__ float sa[OHEM_THREADS / 32], sb[OHEM_THREADS / 32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    a = warp_sum(a);
    b = warp_sum(b);
    if (lane == 0) {
        sa[warp] = a;
        sb[warp] = b;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        a = 0.f;
        b = 0.f;
#pragma unroll
        for (int i = 0; i < OHEM_THREADS / 32; ++i) {
            a += sa[i];
            b += sb[i];
        }
    }
}

// CT > 0: compile-time class count (the C logits of a pixel stay in registers: pred is read exactly once); CT == 0: any C.
// partials per CTA: [0] sum w*nll over valid & p_t <= T0, [1] sum w over the same, [2] / [3] the same over all valid pixels.
template <int CT>
__global__ void __launch_bounds__(OHEM_THREADS) ohem_forward_kernel(const float* __restrict__ pred, const int64_t* __restrict__ label,
                                                                    const float* __restrict__ weight, long long ignore_index, float t0,
                                                                    int C, int HW, float* __restrict__ lse_out, float* __restrict__ pt_out,
                                                                    float* __restrict__ nll_out, float* __restrict__ partials,
                                                                    OhemState* __restrict__ st) {
    css_pdl_enter();
    const int b = blockIdx.y, p = blockIdx.x * OHEM_THREADS + threadIdx.x;
    float a_wl = 0.f, a_w = 0.f, v_wl = 0.f, v_w = 0.f;
    int valid = 0, le = 0;
    if (p < HW) {
        const size_t n = (size_t)b * HW + p;
        const float* x = pred + (size_t)b * C * HW + p;
        const long long lab = label[n];
        valid = lab != ignore_index && lab >= 0 && lab < C;
        float m, s = 0.f, et = 0.f, xt = 0.f;
        if (CT > 0) {
            float v[CT > 0 ? CT : 1];
#pragma unroll
            for (int c = 0; c < CT; ++c) v[c] = ldg_stream(x + (size_t)c * HW);
            m = v[0];
#pragma unroll
            for (int c = 1; c < CT; ++c) m = fmaxf(m, v[c]);
#pragma unroll
            for (int c = 0; c < CT; ++c) {                  // serial class-order sum, as torch's spatial softmax
                const float e = expf(v[c] - m);
                s += e;
                if (c == lab) {
                    et = e;
                    xt = v[c];
                }
            }
        } else {
            m = -INFINITY;
            for (int c = 0; c < C; ++c) m = fmaxf(m, __ldg(x + (size_t)c * HW));
            for (int c = 0; c < C; ++c) s += expf(__ldg(x + (size_t)c * HW) - m);
            if (valid) {
                xt = __ldg(x + (size_t)lab * HW);
                et = expf(xt - m);
            }
        }
        const float lse = m + logf(s);
        lse_out[n] = lse;
        if (valid) {
            const float pt = et / s;                          // torch's softmax epilogue: exp(x - max) / sum
            const float nll = lse - xt;
            const float w = weight ? __ldg(weight + lab) : 1.f;
            pt_out[n] = pt;
            nll_out[n] = nll;
            le = pt <= t0;
            v_wl = w * nll;
            v_w = w;
            if (le) {
                a_wl = v_wl;
                a_w = w;
            }
        } else {
            pt_out[n] = __int_as_float(0x7fffffff);           // NaN: never <= any threshold, skipped by the histograms
            nll_out[n] = 0.f;
        }
    }
    const int nvalid = __popc(__ballot_sync(0xffffffffu, valid)), nle = __popc(__ballot_sync(0xffffffffu, le));
    __shared__ int wcnt[2][OHEM_THREADS / 32];
    if ((threadIdx.x & 31) == 0) {
        wcnt[0][threadIdx.x >> 5] = nvalid;
        wcnt[1][threadIdx.x >> 5] = nle;
    }
    ohem_block_sum2(a_wl, a_w);
    __syncthreads();
    ohem_block_sum2(v_wl, v_w);
    if (threadIdx.x == 0) {
        int c0 = 0, c1 = 0;
#pragma unroll
        for (int i = 0; i < OHEM_THREADS / 32; ++i) {
            c0 += wcnt[0][i];
            c1 += wcnt[1][i];
        }
        float* q = partials + ((size_t)b * gridDim.x + blockIdx.x) * 4;
        q[0] = a_wl;
        q[1] = a_w;
        q[2] = v_wl;
        q[3] = v_w;
        if (c0) atomicAdd(&st->num_valid, c0);
        if (c1) atomicAdd(&st->num_le_t0, c1);
    }
}

// one radix digit: histogram of the valid p_t whose higher digits equal the prefix found so far
template <int PASS>
__global__ void __launch_bounds__(OHEM_THREADS) ohem_hist_kernel(const float* __restrict__ pt, long long N, int min_kept,
                                                                 OhemState* __restrict__ st) {
    css_pdl_enter();
    if (!ohem_needs_select(st, min_kept)) return;
    constexpr int SHIFT = PASS == 0 ? 21 : PASS == 1 ? 10 : 0;
    constexpr int HI = PASS == 0 ? 0 : PASS == 1 ? 21 : 10;      // the digits above this one (PASS > 0)
    constexpr uint32_t MASK = PASS == 2 ? 1023u : 2047u;
    __shared__ uint32_t h[OHEM_BINS];
    for (int i = threadIdx.x; i < OHEM_BINS; i += OHEM_THREADS) h[i] = 0;
    __syncthreads();
    const uint32_t prefix = st->prefix;
    const long long stride = (long long)gridDim.x * OHEM_THREADS;
    for (long long base = (long long)blockIdx.x * OHEM_THREADS; base < N; base += stride) {   // warp-uniform trip count
        const long long n = base + threadIdx.x;
        const uint32_t u = n < N ? __float_as_uint(pt[n]) : 0xffffffffu;
        bool in = u < 0x7f800000u;                            // finite p_t = valid pixel (ignored ones hold NaN)
        if (PASS > 0) in = in && (u >> HI) == (prefix >> HI);
        const uint32_t bin = in ? (u >> SHIFT) & MASK : 0xffffffffu;
        // warp-aggregated: p_t of confident pixels fall into a handful of bins
        const unsigned peers = __match_any_sync(0xffffffffu, bin);
        if (in && (threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&h[bin], (uint32_t)__popc(peers));
    }
    __syncthreads();
    for (int i = threadIdx.x; i <= (int)MASK; i += OHEM_THREADS)
        if (h[i]) atomicAdd(&st->hist[PASS][i], h[i]);
}

// one CTA: the bin holding the k-th smallest value of this digit; fixes the digit in `prefix` and the rank left inside it
template <int PASS>
__global__ void __launch_bounds__(1024) ohem_scan_kernel(int min_kept, OhemState* __restrict__ st) {
    css_pdl_enter();
    if (!ohem_needs_select(st, min_kept)) return;
    constexpr int SHIFT = PASS == 0 ? 21 : PASS == 1 ? 10 : 0;
    constexpr int PER = PASS == 2 ? 1 : 2;                    // bins per thread: 2048 / 2048 / 1024 bins
    __shared__ uint32_t wsum[32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t k = PASS == 0 ? (uint32_t)min_kept : (uint32_t)st->k;
    uint32_t c[PER], own = 0;
#pragma unroll
    for (int j = 0; j < PER; ++j) {
        c[j] = st->hist[PASS][threadIdx.x * PER + j];
        own += c[j];
    }
    uint32_t incl = own;                                      // inclusive scan: warp, then across warps
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        uint32_t t = wsum[lane], s = t;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t u = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += u;
        }
        wsum[lane] = s - t;                                   // exclusive prefix of the warp totals
    }
    __syncthreads();
    uint32_t before = wsum[warp] + incl - own;
    if (before < k && before + own >= k) {                    // exactly one thread: 1 <= k <= total
#pragma unroll
        for (int j = 0; j < PER; ++j) {
            if (before + c[j] >= k) {
                st->prefix |= (uint32_t)(threadIdx.x * PER + j) << SHIFT;
                st->k = (int32_t)(k - before);
                break;
            }
            before += c[j];
        }
    }
}

// kept set when the select ran: valid & p_t <= kth (ignored pixels hold NaN and never compare <=)
__global__ void __launch_bounds__(OHEM_THREADS) ohem_select_sum_kernel(const float* __restrict__ pt, const float* __restrict__ nll,
                                                                       const int64_t* __restrict__ label, const float* __restrict__ weight,
                                                                       long long N, int min_kept, float* __restrict__ partials,
                                                                       OhemState* __restrict__ st) {
    css_pdl_enter();
    if (!ohem_needs_select(st, min_kept)) return;
    const float T = __uint_as_float(st->prefix);
    float wl = 0.f, ws = 0.f;
    int cnt = 0;
    for (long long n = (long long)blockIdx.x * OHEM_THREADS + threadIdx.x; n < N; n += (long long)gridDim.x * OHEM_THREADS) {
        if (pt[n] <= T) {
            const float w = weight ? __ldg(weight + label[n]) : 1.f;
            wl += w * nll[n];
            ws += w;
            ++cnt;
        }
    }
    __shared__ int scnt[OHEM_THREADS / 32];
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if ((threadIdx.x & 31) == 0) scnt[threadIdx.x >> 5] = cnt;
    ohem_block_sum2(wl, ws);
    if (threadIdx.x == 0) {
        int c = 0;
#pragma unroll
        for (int i = 0; i < OHEM_THREADS / 32; ++i) c += scnt[i];
        partials[2 * blockIdx.x] = wl;
        partials[2 * blockIdx.x + 1] = ws;
        if (c) atomicAdd(&st->num_sel, c);
    }
}

// one CTA: picks the kept set's partials, adds them in fixed order, writes loss, T, 1/sum w and the counts
__global__ void __launch_bounds__(OHEM_THREADS) ohem_finalize_kernel(const float* __restrict__ fwd_partials, int nfwd,
                                                                     const float* __restrict__ sel_partials, int nsel, int min_kept,
                                                                     float t0, OhemState* __restrict__ st, float* __restrict__ loss,
                                                                     float* __restrict__ threshold, int32_t* __restrict__ counts) {
    css_pdl_enter();
    const int nv = st->num_valid, n0 = st->num_le_t0;
    const bool ohem = min_kept > 0 && nv >= min_kept, sel = ohem && n0 < min_kept;
    const float* src = sel ? sel_partials : fwd_partials + (ohem ? 0 : 2);
    const int n = sel ? nsel : nfwd, stride = sel ? 2 : 4;
    float a = 0.f, w = 0.f;
    for (int i = threadIdx.x; i < n; i += OHEM_THREADS) {
        a += src[(size_t)i * stride];
        w += src[(size_t)i * stride + 1];
    }
    ohem_block_sum2(a, w);
    if (threadIdx.x == 0) {
        const float T = sel ? __uint_as_float(st->prefix) : ohem ? t0 : INFINITY;
        *loss = a / w;                                        // nothing kept: 0 / 0 = nan, as torch's mean over no pixel
        st->threshold = T;
        st->scale = 1.f / w;
        threshold[0] = T;
        counts[0] = nv;
        counts[1] = sel ? st->num_sel : ohem ? n0 : nv;
    }
}

template <int CT>
__global__ void __launch_bounds__(OHEM_THREADS) ohem_backward_kernel(const float* __restrict__ grad_out, const float* __restrict__ pred,
                                                                     const int64_t* __restrict__ label, const float* __restrict__ weight,
                                                                     const float* __restrict__ lse, const float* __restrict__ pt,
                                                                     const OhemState* __restrict__ st, int C, int HW,
                                                                     float* __restrict__ grad_pred) {
    css_pdl_enter();
    const int b = blockIdx.y, p = blockIdx.x * OHEM_THREADS + threadIdx.x;
    if (p >= HW) return;
    const size_t n = (size_t)b * HW + p;
    const float* x = pred + (size_t)b * C * HW + p;
    float* g = grad_pred + (size_t)b * C * HW + p;
    const bool kept = pt[n] <= st->threshold;                 // NaN (ignored) compares false
    if (!kept) {
        for (int c = 0; c < C; ++c) g[(size_t)c * HW] = 0.f;
        return;
    }
    const long long lab = label[n];
    const float l = lse[n];
    const float k = __ldg(grad_out) * st->scale * (weight ? __ldg(weight + lab) : 1.f);
    if (CT > 0) {
        float v[CT > 0 ? CT : 1];
#pragma unroll
        for (int c = 0; c < CT; ++c) v[c] = ldg_stream(x + (size_t)c * HW);
#pragma unroll
        for (int c = 0; c < CT; ++c) g[(size_t)c * HW] = k * (expf(v[c] - l) - (c == lab ? 1.f : 0.f));
    } else {
        for (int c = 0; c < C; ++c) g[(size_t)c * HW] = k * (expf(ldg_stream(x + (size_t)c * HW) - l) - (c == lab ? 1.f : 0.f));
    }
}

extern "C" size_t css_ohem_workspace_bytes(int B, int H, int W) {
    if (B <= 0 || H <= 0 || W <= 0 || (long long)B * H * W >= (1ll << 31)) return 0;
    return ohem_layout(B, H, W).total;
}

extern "C" int css_ohem_forward(const float* pred, const int64_t* target, const float* weight, long long ignore_index, float thresh,
                                int min_kept, int B, int C, int H, int W, void* workspace, size_t workspace_bytes, float* loss,
                                float* threshold, int32_t* counts, void* stream) {
    CSS_CHECK_ARG(pred && target && workspace && loss && threshold && counts, CSS_E_ARG, "css_ohem_forward: null pointer");
    CSS_CHECK_ARG(B > 0 && B <= 65535 && C > 0 && H > 0 && W > 0, CSS_E_ARG, "css_ohem_forward: bad size (B must be in [1,65535])");
    CSS_CHECK_ARG((long long)B * C * H * W < (1ll << 40) && (long long)B * H * W < (1ll << 31), CSS_E_SIZE, "css_ohem_forward: too large");
    const OhemLayout L = ohem_layout(B, H, W);
    CSS_CHECK_ARG(workspace_bytes >= L.total, CSS_E_SIZE, "css_ohem_forward: workspace of %zu bytes, %zu needed", workspace_bytes, L.total);
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = (char*)workspace;
    OhemState* state = (OhemState*)(ws + L.state);
    float *fwd_partials = (float*)(ws + L.fwd_partials), *sel_partials = (float*)(ws + L.sel_partials);
    float *lse = (float*)(ws + L.lse), *pt = (float*)(ws + L.pt), *nll = (float*)(ws + L.nll);
    const int HW = H * W, nblk = (HW + OHEM_THREADS - 1) / OHEM_THREADS;
    const long long N = (long long)B * HW;
    const int gsel = (int)((N + OHEM_THREADS - 1) / OHEM_THREADS < OHEM_GRID ? (N + OHEM_THREADS - 1) / OHEM_THREADS : OHEM_GRID);
    cudaError_t e = cudaMemsetAsync(state, 0, sizeof(OhemState), st);
    if (e != cudaSuccess) { css_set_error("css_ohem_forward: memset: %s", cudaGetErrorString(e)); return (int)e; }
    const dim3 grid(nblk, B);
    if (C == 19) css_launch(ohem_forward_kernel<19>, grid, dim3(OHEM_THREADS), (size_t)0, st, pred, target, weight, ignore_index, thresh, C, HW, lse, pt, nll, fwd_partials, state);
    else if (C == 21) css_launch(ohem_forward_kernel<21>, grid, dim3(OHEM_THREADS), (size_t)0, st, pred, target, weight, ignore_index, thresh, C, HW, lse, pt, nll, fwd_partials, state);
    else css_launch(ohem_forward_kernel<0>, grid, dim3(OHEM_THREADS), (size_t)0, st, pred, target, weight, ignore_index, thresh, C, HW, lse, pt, nll, fwd_partials, state);
    css_launch(ohem_hist_kernel<0>, dim3(gsel), dim3(OHEM_THREADS), (size_t)0, st, (const float*)pt, N, min_kept, state);
    css_launch(ohem_scan_kernel<0>, dim3(1), dim3(1024), (size_t)0, st, min_kept, state);
    css_launch(ohem_hist_kernel<1>, dim3(gsel), dim3(OHEM_THREADS), (size_t)0, st, (const float*)pt, N, min_kept, state);
    css_launch(ohem_scan_kernel<1>, dim3(1), dim3(1024), (size_t)0, st, min_kept, state);
    css_launch(ohem_hist_kernel<2>, dim3(gsel), dim3(OHEM_THREADS), (size_t)0, st, (const float*)pt, N, min_kept, state);
    css_launch(ohem_scan_kernel<2>, dim3(1), dim3(1024), (size_t)0, st, min_kept, state);
    css_launch(ohem_select_sum_kernel, dim3(gsel), dim3(OHEM_THREADS), (size_t)0, st, (const float*)pt, (const float*)nll, target, weight, N,
               min_kept, sel_partials, state);
    css_launch(ohem_finalize_kernel, dim3(1), dim3(OHEM_THREADS), (size_t)0, st, (const float*)fwd_partials, nblk * B,
               (const float*)sel_partials, gsel, min_kept, thresh, state, loss, threshold, counts);
    CSS_CHECK_LAUNCH("css_ohem_forward", 9);
    return 0;
}

extern "C" int css_ohem_backward(const float* grad_out, const float* pred, const int64_t* target, const float* weight, int B, int C,
                                 int H, int W, const void* workspace, size_t workspace_bytes, float* grad_pred, void* stream) {
    CSS_CHECK_ARG(grad_out && pred && target && workspace && grad_pred, CSS_E_ARG, "css_ohem_backward: null pointer");
    CSS_CHECK_ARG(B > 0 && B <= 65535 && C > 0 && H > 0 && W > 0, CSS_E_ARG, "css_ohem_backward: bad size (B must be in [1,65535])");
    CSS_CHECK_ARG((long long)B * C * H * W < (1ll << 40) && (long long)B * H * W < (1ll << 31), CSS_E_SIZE, "css_ohem_backward: too large");
    const OhemLayout L = ohem_layout(B, H, W);
    CSS_CHECK_ARG(workspace_bytes >= L.total, CSS_E_SIZE, "css_ohem_backward: workspace of %zu bytes, %zu needed", workspace_bytes, L.total);
    const char* ws = (const char*)workspace;
    const OhemState* state = (const OhemState*)(ws + L.state);
    const float *lse = (const float*)(ws + L.lse), *pt = (const float*)(ws + L.pt);
    const int HW = H * W;
    const dim3 grid((HW + OHEM_THREADS - 1) / OHEM_THREADS, B);
    cudaStream_t st = (cudaStream_t)stream;
    if (C == 19) css_launch(ohem_backward_kernel<19>, grid, dim3(OHEM_THREADS), (size_t)0, st, grad_out, pred, target, weight, lse, pt, state, C, HW, grad_pred);
    else if (C == 21) css_launch(ohem_backward_kernel<21>, grid, dim3(OHEM_THREADS), (size_t)0, st, grad_out, pred, target, weight, lse, pt, state, C, HW, grad_pred);
    else css_launch(ohem_backward_kernel<0>, grid, dim3(OHEM_THREADS), (size_t)0, st, grad_out, pred, target, weight, lse, pt, state, C, HW, grad_pred);
    CSS_CHECK_LAUNCH("css_ohem_backward", 1);
    return 0;
}
