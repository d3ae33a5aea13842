// Stage 3: anchor / negative sampling, query x {positive prototype, negatives} scoring at temperature, cross-entropy and
// d loss / d anchor in ONE pass over the gathered rows, then the dense-gradient scatter of the backward.
// Reference: generalframeworks/loss/loss.py:124-149 (+ negative_index_sampler :410-418) and its autograd backward.
//
// Every query draws its own Nn negatives (loss.py:137-142), so this is a per-query row gather (1 KB fp32 rows of the
// pixel-major copy written by css_rep_pass, scaled on the fly by the 1/max(||r||,1e-8) that each valid-list entry carries next to its
// pixel id), not a shared-operand GEMM: 2*D flops per 4*D gathered bytes.
// It is bound by the L2 -> SM gather path (the 107 MB copy is mostly L2 resident at VOC size), not by the tensor pipe.
//
// Work split: one CTA (4 warps) per (present-class slot k, query q); warp w owns candidates j = w, w+4, ...  A warp is
// four 8-lane groups; a group owns one candidate row at a time (8 lanes x 8 x 128-bit loads = the 1 KB row, every 128 B
// line read by exactly one group), reduces the dot with 3 shuffles and keeps an online-softmax state
// (m, l, sum_j 2^{z_j-m} r_hat_j) in registers, so the backward never re-gathers.  Packed fp32x2 FMAs (FFMA2, sm_100)
// halve the FMA issue slots of the dot and of the weighted row accumulation.  Candidate row ids for the next 32
// candidates are produced one per lane (Philox draw or fed index -> rotated segment -> one 8-byte class-list entry) and handed to
// the groups by shuffle.  The four warp states are merged through shared memory in a fixed order (deterministic).
#include "css_common.cuh"
#include <stdlib.h>
#include <string.h>

#define SC_WARPS 4
#define SC_THREADS (SC_WARPS * 32)

struct DrawKey {
    uint2 key;       // seed
    uint32_t off_lo, off_hi;
};

__device__ __forceinline__ DrawKey make_key(uint64_t seed, uint64_t offset) {
    DrawKey k;
    k.key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    k.off_lo = (uint32_t)offset;
    k.off_hi = (uint32_t)(offset >> 32);
    return k;
}

// anchor draw: uniform index into the class's hard list (loss.py:127)
__device__ __forceinline__ int draw_anchor(const DrawKey& dk, int k, int q, int n_hard) {
    const uint4 r = Philox::run(make_uint4(0xffffffffu, ((uint32_t)k << 24) | (uint32_t)q, dk.off_lo, dk.off_hi), dk.key);
    return (int)__umulhi(r.x, (uint32_t)n_hard);
}

// first i in [0, 31] with tab[i] > u  (tab is non-decreasing and tab[31] > u): 5-step binary search
template <typename T>
__device__ __forceinline__ int upper_bound32(const T* tab, T u) {
    int lo = 0;
#pragma unroll
    for (int step = 16; step > 0; step >>= 1)
        if (tab[lo + step - 1] <= u) lo += step;
    return lo;
}

// negative draw j in [0, Nn): class ~ Categorical(cdf row), index ~ Uniform inside that class's valid list (loss.py:136-142).
// Returns the index inside the class list and the rotated segment `seg`; rot_off[seg] + index is the reference's index
// into the rotated concatenation of the valid lists.
__device__ __forceinline__ int draw_negative(const DrawKey& dk, int k, int q, int j, const float* cdf_row, const int* rot_off,
                                             int& seg) {
    const uint4 r = Philox::run(make_uint4((uint32_t)j, ((uint32_t)k << 24) | (uint32_t)q, dk.off_lo, dk.off_hi), dk.key);
    const float u = (float)(r.x >> 8) * (1.0f / 16777216.0f);
    seg = upper_bound32(cdf_row, u);                       // cdf_row[i] == 1 for i >= V-2, u < 1
    const int n = rot_off[seg + 1] - rot_off[seg];
    return (int)__umulhi(r.y, (uint32_t)n);
}

// per-slot tables shared by the sampler and the scorer: rotated class order k+1..V-1,0..k-1, prefix offsets, CDF row
struct SlotTables {
    int rot_off[CSS_CMAX + 1];
    int rot_cls[CSS_CMAX];
    float cdf[CSS_CMAX];
};

__device__ __forceinline__ void build_slot_tables(SlotTables& t, const int32_t* __restrict__ meta,
                                                  const float* __restrict__ class_cdf, int k, int V) {
    // warp 0: one segment per lane, the prefix offsets by a shuffle scan (two dependent loads in all, not one per class)
    if (threadIdx.x < CSS_CMAX) {
        const int i = threadIdx.x;
        t.cdf[i] = class_cdf[k * CSS_CMAX + i];
        const int cls = (i < V - 1) ? meta[CSS_META_CLS_OF_SLOT + (k + 1 + i) % V] : -1;
        t.rot_cls[i] = cls;
        const int nv = (cls >= 0) ? meta[CSS_META_N_VALID + cls] : 0;
        int incl = nv;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int up = __shfl_up_sync(0xffffffffu, incl, o);
            if (i >= o) incl += up;
        }
        t.rot_off[i] = incl - nv;                      // segments past V-2 are empty: their offset is the total
        if (i == CSS_CMAX - 1) t.rot_off[CSS_CMAX] = incl;
    }
    __syncthreads();
}

// -------------------------------------------------------------------------------------------------------------------
// css_sample: materialise the draws (same device functions as the scorer uses on the fly)
// -------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) sample_kernel(const int32_t* __restrict__ meta, const float* __restrict__ class_cdf,
                                                     uint64_t seed, uint64_t offset, int Q, int Nn, int32_t* __restrict__ anchor_idx,
                                                     int32_t* __restrict__ neg_idx) {
    css_pdl_enter();
    __shared__ SlotTables tb;
    const int k = blockIdx.y;
    const int V = meta[CSS_META_V];
    if (k >= V || V <= 1) return;
    const int c = meta[CSS_META_CLS_OF_SLOT + k];
    const int n_hard = meta[CSS_META_N_HARD + c];
    if (n_hard == 0) return;
    build_slot_tables(tb, meta, class_cdf, k, V);
    const DrawKey dk = make_key(seed, offset);
    const long long total = (long long)Q * (Nn + 1);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int q = (int)(i / (Nn + 1)), j = (int)(i - (long long)q * (Nn + 1));
        if (j == 0) {
            anchor_idx[k * Q + q] = draw_anchor(dk, k, q, n_hard);
        } else {
            int seg;
            const int within = draw_negative(dk, k, q, j - 1, tb.cdf, tb.rot_off, seg);
            neg_idx[((size_t)k * Q + q) * Nn + (j - 1)] = tb.rot_off[seg] + within;
        }
    }
}

extern "C" int css_sample(const int32_t* meta, const float* class_cdf, uint64_t seed, uint64_t offset, int C, int Q, int Nn,
                          int32_t* anchor_idx, int32_t* neg_idx, void* stream) {
    CSS_CHECK_ARG(meta && class_cdf && anchor_idx && neg_idx, CSS_E_ARG, "css_sample: null pointer");
    CSS_CHECK_ARG(Q > 0 && Nn > 0 && Q < (1 << 24), CSS_E_ARG, "css_sample: bad Q/Nn");
    CSS_CHECK_ARG(C >= 1 && C <= CSS_CMAX, CSS_E_DIM, "css_sample: C must be in [1,%d]", CSS_CMAX);
    cudaStream_t st = (cudaStream_t)stream;
    cudaMemsetAsync(anchor_idx, 0xff, sizeof(int32_t) * (size_t)C * Q, st);
    cudaMemsetAsync(neg_idx, 0xff, sizeof(int32_t) * (size_t)C * Q * Nn, st);
    const long long total = (long long)Q * (Nn + 1);
    dim3 grid((unsigned)min((total + 255) / 256, 4096ll), C);
    css_launch(sample_kernel, dim3(grid), dim3(256), (size_t)(0), (cudaStream_t)(st), meta, class_cdf, seed, offset, Q, Nn, anchor_idx, neg_idx);
    CSS_CHECK_LAUNCH("css_sample", 1);
    return 0;
}

// -------------------------------------------------------------------------------------------------------------------
// css_score_ce
// -------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float group_sum8(float v) {     // reduce over the 8 lanes of a group
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    v += __shfl_xor_sync(0xffffffffu, v, 4);
    return v;
}

__device__ __forceinline__ float2 lo2(const float4& v) { return make_float2(v.x, v.y); }
__device__ __forceinline__ float2 hi2(const float4& v) { return make_float2(v.z, v.w); }

__device__ __forceinline__ float4 lds128(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}

// same dot with the anchor slice re-read from shared memory for every row (volatile asm: not hoisted), so that the 32
// anchor registers per lane are free and a fifth CTA fits on the SM
__device__ __forceinline__ float dot8_smem(uint32_t a_addr, const float4 (&r)[8]) {
    float2 s0 = make_float2(0.f, 0.f), s1 = s0, s2 = s0, s3 = s0;
#pragma unroll
    for (int i = 0; i < 8; i += 2) {
        const float4 a0 = lds128(a_addr + i * 128), a1 = lds128(a_addr + (i + 1) * 128);
        s0 = __ffma2_rn(make_float2(a0.x, a0.y), make_float2(r[i].x, r[i].y), s0);
        s1 = __ffma2_rn(make_float2(a0.z, a0.w), make_float2(r[i].z, r[i].w), s1);
        s2 = __ffma2_rn(make_float2(a1.x, a1.y), make_float2(r[i + 1].x, r[i + 1].y), s2);
        s3 = __ffma2_rn(make_float2(a1.z, a1.w), make_float2(r[i + 1].z, r[i + 1].w), s3);
    }
    return ((s0.x + s0.y) + (s1.x + s1.y)) + ((s2.x + s2.y) + (s3.x + s3.y));
}

// 32-element slice dot with packed fp32x2 FMAs, 4 independent chains
__device__ __forceinline__ float dot8(const float4 (&a)[8], const float4 (&r)[8]) {
    float2 s0 = make_float2(0.f, 0.f), s1 = s0, s2 = s0, s3 = s0;
#pragma unroll
    for (int i = 0; i < 8; i += 2) {
        s0 = __ffma2_rn(lo2(a[i]), lo2(r[i]), s0);
        s1 = __ffma2_rn(hi2(a[i]), hi2(r[i]), s1);
        s2 = __ffma2_rn(lo2(a[i + 1]), lo2(r[i + 1]), s2);
        s3 = __ffma2_rn(hi2(a[i + 1]), hi2(r[i + 1]), s3);
    }
    return ((s0.x + s0.y) + (s1.x + s1.y)) + ((s2.x + s2.y) + (s3.x + s3.y));
}

template <bool ASMEM, int NA>
__device__ __forceinline__ float score_dot(const float4 (&a)[NA], uint32_t a_addr, const float4 (&r)[8]) {
    if constexpr (ASMEM) return dot8_smem(a_addr, r);
    else return dot8(a, r);
}

struct Online {            // online softmax state (base 2) of one 8-lane group
    float m, l;
    float4 acc[8];
};

// `inv_nr` = 1 / max(||r||, 1e-8): the rows are stored raw, the state accumulates sum_j 2^{z_j-m} r_j / ||r_j||.
// FIX: cos <= 1, so m = scale2 = log2(e)/temp bounds every logit from above; with that fixed reference no running max, no
// rescaling and no data-dependent branch are needed (used whenever 2^(-2 scale2) is comfortably inside fp32, i.e. temp > 0.024;
// smaller temperatures take the online-max path).
template <bool WANT_GRAD, bool FIX>
__device__ __forceinline__ void online_update(Online& st, float z, bool valid, float inv_nr, const float4 (&r)[8]) {
    if (!FIX && valid && z > st.m) {               // group-uniform; rare after the first few rows
        const float sc = exp2f(st.m - z);          // m = -inf -> 0
        st.l *= sc;
        if (WANT_GRAD) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                st.acc[i].x *= sc;
                st.acc[i].y *= sc;
                st.acc[i].z *= sc;
                st.acc[i].w *= sc;
            }
        }
        st.m = z;
    }
    const float wgt = valid ? exp2f(z - st.m) : 0.f;
    st.l += wgt;
    if (WANT_GRAD) {
        const float wr = wgt * inv_nr;
        const float2 ww = make_float2(wr, wr);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float2 lo = __ffma2_rn(ww, lo2(r[i]), lo2(st.acc[i]));
            const float2 hi = __ffma2_rn(ww, hi2(r[i]), hi2(st.acc[i]));
            st.acc[i] = make_float4(lo.x, lo.y, hi.x, hi.y);
        }
    }
}

struct QueryShared {                     // per-CTA scratch for merging the SC_WARPS warp states
    float4 acc[SC_WARPS][CSS_D / 4];
    float m[SC_WARPS], l[SC_WARPS], pos[2];
};

// Publish a warp's state (m, l: lane 0; its slice of sum 2^{z-m} r_hat: already in sh.acc[warp]; the positive's logit and
// cosine: already in sh.pos), then merge the SC_WARPS warps in warp order and write the query's loss, anchor pixel and
// d loss / d anchor.
template <bool WANT_GRAD, typename RT>
__device__ __forceinline__ void finish_warps(float m, float l_w, QueryShared& sh, const RT* __restrict__ rows,
                                             const float4* __restrict__ proto_hat, float inv_na, int pa, int c, int k, int q, int Q,
                                             int V, float temp, float* __restrict__ loss_kq, int32_t* __restrict__ anchor_px,
                                             float4* __restrict__ grad_anchor) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float4 (&s_acc)[SC_WARPS][CSS_D / 4] = sh.acc;
    float (&s_m)[SC_WARPS] = sh.m;
    float (&s_l)[SC_WARPS] = sh.l;
    float (&s_pos)[2] = sh.pos;
    if (lane == 0) {
        s_m[warp] = m;
        s_l[warp] = l_w;
    }
    __syncthreads();
    if (warp != 0) return;

    // warp 0 merges the SC_WARPS warp states in warp order
    float M = s_m[0];
#pragma unroll
    for (int w2 = 1; w2 < SC_WARPS; ++w2) M = fmaxf(M, s_m[w2]);
    float sc[SC_WARPS], l = 0.f;
#pragma unroll
    for (int w2 = 0; w2 < SC_WARPS; ++w2) {
        sc[w2] = (s_m[w2] == -INFINITY) ? 0.f : exp2f(s_m[w2] - M);
        l += s_l[w2] * sc[w2];
    }
    // CE with target 0: logsumexp(z) - z_0 (loss.py:147), evaluated in base 2
    if (lane == 0) {
        loss_kq[k * Q + q] = 0.6931471805599453f * ((M + log2f(l)) - s_pos[0]);
        anchor_px[k * Q + q] = pa;
    }
    if (WANT_GRAD) {
        // dL/da = (sum_j g_j r_hat_j - (sum_j g_j cos_j) a_hat) / max(||a||, eps),  g_j = (pi_j - [j==0]) / (Q V temp)
        // with sum_j pi_j r_hat_j = acc / l and sum_j pi_j cos_j = a_hat . (acc / l)        (SURVEY.md Appendix A.4)
        const float inv_l = 1.f / l;
        const float4* php = proto_hat + (size_t)c * (CSS_D / 4);
        float4 S[2], av[2], ph[2];
        float sdot = 0.f;
#pragma unroll
        for (int h2 = 0; h2 < 2; ++h2) {
            const int col = lane + 32 * h2;
            float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int w2 = 0; w2 < SC_WARPS; ++w2) {
                const float4 v = s_acc[w2][col];
                t.x = fmaf(v.x, sc[w2], t.x);
                t.y = fmaf(v.y, sc[w2], t.y);
                t.z = fmaf(v.z, sc[w2], t.z);
                t.w = fmaf(v.w, sc[w2], t.w);
            }
            S[h2] = make_float4(t.x * inv_l, t.y * inv_l, t.z * inv_l, t.w * inv_l);
            av[h2] = row_f4(rows, (size_t)pa, col);         // raw anchor -> a_hat
            av[h2].x *= inv_na; av[h2].y *= inv_na; av[h2].z *= inv_na; av[h2].w *= inv_na;
            ph[h2] = __ldg(php + col);
            sdot += S[h2].x * av[h2].x + S[h2].y * av[h2].y + S[h2].z * av[h2].z + S[h2].w * av[h2].w;
        }
        sdot = warp_sum(sdot);
        const float scale = 1.f / ((float)Q * (float)V * temp);
        const float tt = (sdot - s_pos[1]) * scale;
        float4* g = grad_anchor + ((size_t)k * Q + q) * (CSS_D / 4);
#pragma unroll
        for (int h2 = 0; h2 < 2; ++h2) {
            float4 o;
            o.x = ((S[h2].x - ph[h2].x) * scale - tt * av[h2].x) * inv_na;
            o.y = ((S[h2].y - ph[h2].y) * scale - tt * av[h2].y) * inv_na;
            o.z = ((S[h2].z - ph[h2].z) * scale - tt * av[h2].z) * inv_na;
            o.w = ((S[h2].w - ph[h2].w) * scale - tt * av[h2].w) * inv_na;
            g[lane + 32 * h2] = o;
        }
    }
}

// Merge the four 8-lane groups of every warp, then the SC_WARPS warps (fixed order), and write the query's loss, anchor
// pixel and d loss / d anchor.
template <bool WANT_GRAD, typename RT>
__device__ __forceinline__ void finish_query(Online& st, float z0, float cos_pos, QueryShared& sh, const RT* __restrict__ rows,
                                             const float4* __restrict__ proto_hat, float inv_na, int pa, int c, int k, int q, int Q,
                                             int V, float temp, float* __restrict__ loss_kq, int32_t* __restrict__ anchor_px,
                                             float4* __restrict__ grad_anchor) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int grp = lane >> 3, l8 = lane & 7;
    // merge the four groups (xor 8, xor 16); afterwards every lane holds the warp's state for its column slice
#pragma unroll
    for (int o = 8; o <= 16; o <<= 1) {
        const float m_o = __shfl_xor_sync(0xffffffffu, st.m, o);
        const float l_o = __shfl_xor_sync(0xffffffffu, st.l, o);
        const float M = fmaxf(st.m, m_o);
        const float s_a = (st.m == -INFINITY) ? 0.f : exp2f(st.m - M);
        const float s_b = (m_o == -INFINITY) ? 0.f : exp2f(m_o - M);
        st.l = st.l * s_a + l_o * s_b;
        if (WANT_GRAD) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                st.acc[i].x = st.acc[i].x * s_a + __shfl_xor_sync(0xffffffffu, st.acc[i].x, o) * s_b;
                st.acc[i].y = st.acc[i].y * s_a + __shfl_xor_sync(0xffffffffu, st.acc[i].y, o) * s_b;
                st.acc[i].z = st.acc[i].z * s_a + __shfl_xor_sync(0xffffffffu, st.acc[i].z, o) * s_b;
                st.acc[i].w = st.acc[i].w * s_a + __shfl_xor_sync(0xffffffffu, st.acc[i].w, o) * s_b;
            }
        }
        st.m = M;
    }
    if (WANT_GRAD && grp == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) sh.acc[warp][i * 8 + l8] = st.acc[i];
    }
    if (threadIdx.x == 0) {
        sh.pos[0] = z0;
        sh.pos[1] = cos_pos;
    }
    finish_warps<WANT_GRAD, RT>(st.m, st.l, sh, rows, proto_hat, inv_na, pa, c, k, q, Q, V, temp, loss_kq, anchor_px,
                                grad_anchor);
}

// publishes the Philox offset of this call, offset + *step_counter, into meta and bumps the device-resident counter so the
// next call -- or the next replay of a captured CUDA graph -- draws fresh samples
__global__ void draw_offset_kernel(uint64_t offset, unsigned long long* __restrict__ step_counter, int32_t* __restrict__ meta) {
    css_pdl_enter();
    unsigned long long o = offset;
    if (step_counter) {
        o += *step_counter;
        *step_counter += 1ull;
    }
    meta[CSS_META_DRAW_OFFSET] = (int32_t)(uint32_t)o;
    meta[CSS_META_DRAW_OFFSET + 1] = (int32_t)(uint32_t)(o >> 32);
}

// candidate row `row` (>= 0: pixel-major row of the map, widened to fp32; < 0: the fp32 prototype row `pp`) -> r[0..7]
template <typename RT>
__device__ __forceinline__ void load_candidate(const RT* __restrict__ rows, const float4* __restrict__ pp, int row, int l8, float4 (&r)[8]) {
    if constexpr (sizeof(RT) == 4) {
        const float4* p = (row >= 0) ? reinterpret_cast<const float4*>(rows) + (size_t)row * (CSS_D / 4) + l8 : pp;
#pragma unroll
        for (int i = 0; i < 8; ++i) r[i] = __ldg(p + i * 8);
    } else {
        if (row >= 0) {                                    // group-uniform branch
            const uint2* p = reinterpret_cast<const uint2*>(rows) + (size_t)row * (CSS_D / 4) + l8;
            uint2 u[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) u[i] = __ldg(p + i * 8);
#pragma unroll
            for (int i = 0; i < 8; ++i) r[i] = bf16x4_to_f4(u[i]);
        } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) r[i] = __ldg(pp + i * 8);
        }
    }
}

// ids of the warp's candidates 32 b + lane: negative j - 1 = warp + SC_WARPS n  ->  its valid-list entry {pixel-major row, bits of
// 1 / max(||row||, 1e-8)}, or {-2, bits of 1} past the end (any finite inverse: those candidates carry weight 0)
template <bool FED>
__device__ __forceinline__ int2 ring_candidate_row(const SlotTables& tb, const DrawKey& dk, const int32_t* __restrict__ neg_idx,
                                                   const int2* __restrict__ valid_list, int k, int q, int Q, int Nn, int N, int n, int cnt) {
    if (n >= cnt) return make_int2(-2, __float_as_int(1.f));
    const int jm1 = (threadIdx.x >> 5) + SC_WARPS * n;
    int seg, within;
    if (FED) {
        const int idx = neg_idx[((size_t)k * Q + q) * Nn + jm1];
        seg = upper_bound32(tb.rot_off + 1, idx);
        within = idx - tb.rot_off[seg];
    } else {
        within = draw_negative(dk, k, q, jm1, tb.cdf, tb.rot_off, seg);
    }
    return valid_list[(size_t)tb.rot_cls[seg] * N + within];
}

// -------------------------------------------------------------------------------------------------------------------
// Whole-warp rows: every candidate row is spread over the 32 lanes (lane l holds float4 l and l + 32 of the 1 KB row), so the
// anchor slice and the gradient accumulator take 8 registers each, once per warp, instead of one full copy per 8-lane group.
// The registers this frees hold R rows per warp in flight: per batch, 2R back-to-back LDG.128 per lane.  The R partial dots
// are reduced by a transpose-reduce (xor 16 halves the values a lane holds, then xor 8, ..., until one is left; the last
// offsets finish the sum), which leaves the full dot of row lane / (32 / R) on every lane: about one shuffle per row
// instead of five, and one exp2 per lane covers the batch.  The batch's row ids and weights 2^{z-m} / ||r|| reach every lane
// through a few words of shared memory (one broadcast LDS.128 per four values: shuffles, one per value, cost the same MIO
// slots as these loads), and the rows are accumulated with 4 FFMA2 per row.  The online-max variant (!FIX) takes one warp max per batch.
// -------------------------------------------------------------------------------------------------------------------
template <int R>
__device__ __forceinline__ float transpose_sum(float (&d)[R], int lane) {
#pragma unroll
    for (int o = 16, n = R; n > 1; o >>= 1, n >>= 1) {
        const bool up = lane & o;
#pragma unroll
        for (int i = 0; i < n / 2; ++i) {
            const float send = up ? d[i] : d[i + n / 2];
            const float keep = up ? d[i + n / 2] : d[i];
            d[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
        }
    }
    float v = d[0];
#pragma unroll
    for (int o = 16 / R; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ float2 dot2x4(const float4& a0, const float4& a1, const float4& r0, const float4& r1) {
    float2 s = __fmul2_rn(lo2(a0), lo2(r0));
    s = __ffma2_rn(hi2(a0), hi2(r0), s);
    s = __ffma2_rn(lo2(a1), lo2(r1), s);
    return __ffma2_rn(hi2(a1), hi2(r1), s);
}

__device__ __forceinline__ void axpy4(float wr, const float4& r, float4& acc) {
    const float2 ww = make_float2(wr, wr);
    const float2 lo = __ffma2_rn(ww, lo2(r), lo2(acc));
    const float2 hi = __ffma2_rn(ww, hi2(r), hi2(acc));
    acc = make_float4(lo.x, lo.y, hi.x, hi.y);
}

// The fp32 gradient form of score_ce_kernel, after the slot tables and the anchor pixel `pa` are known (R rows per batch).
template <bool FIX, int R>
__device__ __forceinline__ void score_rows_wide(const float* __restrict__ rows, const float* __restrict__ norms, const float4* __restrict__ proto_hat,
                                                const int2* __restrict__ valid_list, const int32_t* __restrict__ neg_idx,
                                                const SlotTables& tb, QueryShared& sh, const DrawKey& dk, int pa, int c, int k, int q, int N,
                                                int Q, int Nn, int V, float temp, float* __restrict__ loss_kq, int32_t* __restrict__ anchor_px,
                                                float4* __restrict__ grad_anchor) {
    static_assert(R == 2 || R == 4 || R == 8 || R == 16, "R rows per batch, a power of two that divides the 32-id batch");
    constexpr int LPR = 32 / R;                                // lanes that end up holding one row's dot
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // warp w owns the negatives j - 1 = w + SC_WARPS n, n < cnt; their ids come 32 at a time, one per lane
    const int cnt = (Nn - warp + SC_WARPS - 1) / SC_WARPS;
    int2 cur = (neg_idx ? ring_candidate_row<true>(tb, dk, neg_idx, valid_list, k, q, Q, Nn, N, lane, cnt)
                        : ring_candidate_row<false>(tb, dk, neg_idx, valid_list, k, q, Q, Nn, N, lane, cnt));

    const float4* rows4 = reinterpret_cast<const float4*>(rows);
    const float4 a0 = __ldg(rows4 + (size_t)pa * (CSS_D / 4) + lane), a1 = __ldg(rows4 + (size_t)pa * (CSS_D / 4) + 32 + lane);
    const float inv_na = 1.f / fmaxf(norms[pa], 1e-8f);       // cosine_similarity eps (loss.py:146)
    const float scale2 = 1.4426950408889634f / temp;

    // candidate 0 = the (updated) prototype of class c (loss.py:143-144): scored by every warp, kept by warp 0
    float4 acc0, acc1;
    float m, l;                                                // l: this lane's share (one lane per row adds its weight)
    {
        const float4* pp = proto_hat + (size_t)c * (CSS_D / 4);
        const float4 p0 = __ldg(pp + lane), p1 = __ldg(pp + 32 + lane);
        const float2 s = dot2x4(a0, a1, p0, p1);
        const float cos_pos = warp_sum(s.x + s.y) * inv_na;
        const float z0 = cos_pos * scale2;
        m = FIX ? scale2 : (warp == 0 ? z0 : -INFINITY);
        const float w0 = (warp == 0) ? exp2f(z0 - m) : 0.f;
        l = (lane == 0) ? w0 : 0.f;
        acc0 = make_float4(w0 * p0.x, w0 * p0.y, w0 * p0.z, w0 * p0.w);
        acc1 = make_float4(w0 * p1.x, w0 * p1.y, w0 * p1.z, w0 * p1.w);
        if (threadIdx.x == 0) {                                // read by finish_warps after its barrier
            sh.pos[0] = z0;
            sh.pos[1] = cos_pos;
        }
    }

    // the id group's row ids and each batch's weights reach every lane through the warp's words of shared memory: one
    // broadcast LDS.128 per four values instead of one shuffle per value
    __shared__ __align__(16) int s_id[SC_WARPS][32];
    __shared__ __align__(16) float s_w[SC_WARPS][R];
#pragma unroll 1
    for (int base = 0; base < cnt; base += 32) {
        const int2 nxt = neg_idx ? ring_candidate_row<true>(tb, dk, neg_idx, valid_list, k, q, Q, Nn, N, base + 32 + lane, cnt)
                                 : ring_candidate_row<false>(tb, dk, neg_idx, valid_list, k, q, Q, Nn, N, base + 32 + lane, cnt);
        const int n_batches = min(32, cnt - base + R - 1) / R;
        __syncwarp();                                          // the previous group's ids have been read
        s_id[warp][lane] = cur.x;
        __syncwarp();
#pragma unroll 1
        for (int t = 0; t < n_batches; ++t) {
            float4 r[R][2];
            int ids[R];
#pragma unroll
            for (int i = 0; i < R; i += 4) {
                const int4 v = *reinterpret_cast<const int4*>(&s_id[warp][t * R + i]);
                ids[i] = v.x; ids[i + 1] = v.y; ids[i + 2] = v.z; ids[i + 3] = v.w;
            }
#pragma unroll
            for (int i = 0; i < R; ++i) {                      // past the end: row 0 (any finite row), weight 0
                const float4* p = rows4 + (size_t)max(ids[i], 0) * (CSS_D / 4) + lane;
                r[i][0] = __ldg(p);
                r[i][1] = __ldg(p + 32);
            }
            float d[R];
#pragma unroll
            for (int i = 0; i < R; ++i) {
                const float2 s = dot2x4(a0, a1, r[i][0], r[i][1]);
                d[i] = s.x + s.y;
            }
            const int mine = t * R + lane / LPR;               // the candidate whose dot this lane ends up with
            const float inv = __int_as_float(__shfl_sync(0xffffffffu, cur.y, mine));
            const float z = transpose_sum<R>(d, lane) * (inv_na * inv) * scale2;
            const bool valid = base + mine < cnt;
            if (!FIX) {
                float zm = valid ? z : -INFINITY;
#pragma unroll
                for (int o = LPR; o < 32; o <<= 1) zm = fmaxf(zm, __shfl_xor_sync(0xffffffffu, zm, o));
                if (zm > m) {                                  // warp-uniform
                    const float sc = exp2f(m - zm);            // m = -inf -> 0
                    l *= sc;
                    acc0 = make_float4(acc0.x * sc, acc0.y * sc, acc0.z * sc, acc0.w * sc);
                    acc1 = make_float4(acc1.x * sc, acc1.y * sc, acc1.z * sc, acc1.w * sc);
                    m = zm;
                }
            }
            const float wgt = valid ? exp2f(z - m) : 0.f;
            if (lane % LPR == 0) l += wgt;
            const float wr = wgt * inv;
            float w[R];
            if (lane % LPR == 0) s_w[warp][lane / LPR] = wr;
            __syncwarp();
#pragma unroll
            for (int i = 0; i < R; i += 4) {
                const float4 v = *reinterpret_cast<const float4*>(&s_w[warp][i]);
                w[i] = v.x; w[i + 1] = v.y; w[i + 2] = v.z; w[i + 3] = v.w;
            }
            __syncwarp();                                      // read before the next batch writes
#pragma unroll
            for (int i = 0; i < R; ++i) {
                axpy4(w[i], r[i][0], acc0);
                axpy4(w[i], r[i][1], acc1);
            }
        }
        cur = nxt;
    }
    sh.acc[warp][lane] = acc0;
    sh.acc[warp][lane + 32] = acc1;
    finish_warps<true, float>(m, warp_sum(l), sh, rows, proto_hat, inv_na, pa, c, k, q, Q, V, temp, loss_kq, anchor_px,
                              grad_anchor);
}


// fp32 rows with the gradient take the whole-warp layout above (8 rows per batch, 4 CTAs/SM; PREFETCH and ASMEM select among
// the forms of the 8-lane-group layout, which the bf16 and forward-only variants keep)
template <bool WANT_GRAD, bool PREFETCH, bool ASMEM, bool FIX, typename RT>
__global__ void __launch_bounds__(SC_THREADS, (WANT_GRAD && (!ASMEM || sizeof(RT) == 4)) ? 4 : 5) score_ce_kernel(
    const RT* __restrict__ rows, const float* __restrict__ norms, const float4* __restrict__ proto_hat,
    const float* __restrict__ class_cdf, const int2* __restrict__ valid_list, const int32_t* __restrict__ hard_list,
    const int32_t* __restrict__ meta, const int32_t* __restrict__ anchor_idx, const int32_t* __restrict__ neg_idx, uint64_t seed,
    int N, int Q, int Nn, float temp, float* __restrict__ loss_kq, int32_t* __restrict__ anchor_px, float4* __restrict__ grad_anchor) {
    css_pdl_enter();
    __shared__ SlotTables tb;
    __shared__ QueryShared sh;
    const int k = blockIdx.y, q = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int V = meta[CSS_META_V];
    const int c = (k < V) ? meta[CSS_META_CLS_OF_SLOT + k] : 0;
    const int n_hard = (k < V) ? meta[CSS_META_N_HARD + c] : 0;
    if (k >= V || V <= 1 || n_hard == 0) {         // absent slot / degenerate batch / no hard pixel (loss.py:116,125-130)
        if (threadIdx.x == 0) {
            loss_kq[k * Q + q] = 0.f;
            anchor_px[k * Q + q] = -1;
        }
        return;
    }
    build_slot_tables(tb, meta, class_cdf, k, V);

    const int grp = lane >> 3, l8 = lane & 7;
    const DrawKey dk = make_key(seed, ((uint64_t)(uint32_t)meta[CSS_META_DRAW_OFFSET + 1] << 32) | (uint32_t)meta[CSS_META_DRAW_OFFSET]);
    const int ai = anchor_idx ? anchor_idx[k * Q + q] : draw_anchor(dk, k, q, n_hard);
    const int pa = hard_list[(size_t)c * N + ai];
    if constexpr (WANT_GRAD && sizeof(RT) == 4) {
        score_rows_wide<FIX, 8>(rows, norms, proto_hat, valid_list, neg_idx, tb, sh, dk, pa, c, k, q, N, Q, Nn, V, temp, loss_kq, anchor_px,
                                grad_anchor);
        return;
    }
    __shared__ float4 s_a[ASMEM ? CSS_D / 4 : 1];
    float4 a[ASMEM ? 1 : 8];
    if (ASMEM) {
        if (threadIdx.x < CSS_D / 4) s_a[threadIdx.x] = row_f4(rows, (size_t)pa, threadIdx.x);
        __syncthreads();
    } else {
#pragma unroll
        for (int i = 0; i < (ASMEM ? 1 : 8); ++i) a[i] = row_f4(rows, (size_t)pa, i * 8 + l8);
    }
    const uint32_t a_addr = (uint32_t)__cvta_generic_to_shared(&s_a[ASMEM ? l8 : 0]);
    const float inv_na = 1.f / fmaxf(norms[pa], 1e-8f);       // cosine_similarity eps (loss.py:146)
    const float4* pp = proto_hat + (size_t)c * (CSS_D / 4) + l8;
    const float scale2 = 1.4426950408889634f / temp;          // logits in base 2: z2 = cos * log2(e) / temp

    Online st;
    st.m = FIX ? scale2 : -INFINITY;                  // FIX: cos <= 1 bounds every logit by scale2
    st.l = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) st.acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    float z0 = 0.f, cos_pos = 0.f;

    // warp w owns candidates j = w + 4 n; candidate 0 = the (updated) prototype of class c (loss.py:143-144)
    const int n_cand = Nn + 1;
    const int cnt = (n_cand - warp + SC_WARPS - 1) / SC_WARPS;
    for (int base = 0; base < cnt; base += 32) {
        // one candidate per lane: row id (-1 = prototype, -2 = past the end) and 1 / max(||row||, 1e-8)
        int my_row = -2;
        float my_inv = 1.f;
        {
            const int n = base + lane;
            const int j = warp + SC_WARPS * n;
            if (j == 0) {
                my_row = -1;                                   // proto_hat is already normalised
            } else if (n < cnt) {
                int seg, within;
                if (neg_idx) {
                    const int idx = neg_idx[((size_t)k * Q + q) * Nn + (j - 1)];
                    seg = upper_bound32(tb.rot_off + 1, idx);          // largest seg with rot_off[seg] <= idx
                    within = idx - tb.rot_off[seg];
                } else {
                    within = draw_negative(dk, k, q, j - 1, tb.cdf, tb.rot_off, seg);
                }
                const int2 e = valid_list[(size_t)tb.rot_cls[seg] * N + within];
                my_row = e.x;
                my_inv = __int_as_float(e.y);
            }
        }
        const int steps = min(8, (cnt - base + 3) >> 2);
        if (PREFETCH) {
            // software pipeline: the next candidate row is in flight while the current one is scored
            float4 rn[8];
            int row_n = __shfl_sync(0xffffffffu, my_row, grp);
            load_candidate(rows, pp, row_n, l8, rn);
#pragma unroll 1
            for (int t = 0; t < steps; ++t) {
                float4 r[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) r[i] = rn[i];
                const int row = row_n;
                const float inv = __shfl_sync(0xffffffffu, my_inv, t * 4 + grp);
                row_n = __shfl_sync(0xffffffffu, my_row, ((t + 1) & 7) * 4 + grp);
                if (t + 1 < steps) load_candidate(rows, pp, row_n, l8, rn);
                const float cosv = group_sum8(score_dot<ASMEM>(a, a_addr, r)) * (inv_na * inv);
                const float z = cosv * scale2;
                if (row == -1) {
                    z0 = z;
                    cos_pos = cosv;
                }
                online_update<WANT_GRAD, FIX>(st, z, row != -2, inv, r);
            }
        } else {
#pragma unroll 1
            for (int t = 0; t < steps; ++t) {
                const int row = __shfl_sync(0xffffffffu, my_row, t * 4 + grp);
                const float inv = __shfl_sync(0xffffffffu, my_inv, t * 4 + grp);
                float4 r[8];
                load_candidate(rows, pp, row, l8, r);
                const float cosv = group_sum8(score_dot<ASMEM>(a, a_addr, r)) * (inv_na * inv);
                const float z = cosv * scale2;
                if (row == -1) {
                    z0 = z;
                    cos_pos = cosv;
                }
                online_update<WANT_GRAD, FIX>(st, z, row != -2, inv, r);
            }
        }
    }

    finish_query<WANT_GRAD, RT>(st, z0, cos_pos, sh, rows, proto_hat, inv_na, pa, c, k, q, Q, V, temp, loss_kq, anchor_px, grad_anchor);
}

// -------------------------------------------------------------------------------------------------------------------
// The same scorer with the candidate rows staged through shared memory by 16-byte asynchronous copies (cp.async.cg, LDGSTS):
// the register kernel above can keep only ONE row per 8-lane group in flight (row + gradient state + anchor fill its 96
// registers), so a warp waits out a full L2 round trip for every four rows and the SM holds 20 warps x 4 KB = 80 KB in flight.
// Here every warp owns a ring of RING_STAGES x 4 rows in shared memory; the copies for step s + RING_STAGES - 1 are issued
// before step s is scored, so (RING_STAGES - 1) x 4 KB per warp stay in flight WHILE the warp computes, at no register cost.
// A lane copies exactly the 16-byte chunks it later reads (chunk i*8 + l8 of its group's row), so cp.async.wait_group alone
// orders a lane's reads after its own copies and no warp barrier is needed; a quarter-warp reads 128 contiguous bytes
// (conflict-free).  The anchor lives in registers (re-reading it from shared memory per row would put 3 KB of shared-memory
// traffic on every gathered KB).  fp32 rows with the gradient; everything else stays on the register kernel.
// -------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N_PENDING>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N_PENDING) : "memory"); }

#define RING_STAGE_BYTES (4 * CSS_D * 4)          // four fp32 rows, one per 8-lane group

template <bool FIX, bool FED, int STAGES, int MINB>
__global__ void __launch_bounds__(SC_THREADS, MINB) score_ce_ring_kernel(
    const float* __restrict__ rows, const float* __restrict__ norms, const float4* __restrict__ proto_hat,
    const float* __restrict__ class_cdf, const int2* __restrict__ valid_list, const int32_t* __restrict__ hard_list,
    const int32_t* __restrict__ meta, const int32_t* __restrict__ anchor_idx, const int32_t* __restrict__ neg_idx, uint64_t seed,
    int N, int Q, int Nn, float temp, float* __restrict__ loss_kq, int32_t* __restrict__ anchor_px, float4* __restrict__ grad_anchor) {
    css_pdl_enter();
    extern __shared__ __align__(128) unsigned char ring_smem[];
    __shared__ SlotTables tb;
    __shared__ QueryShared sh;
    const int k = blockIdx.y, q = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int V = meta[CSS_META_V];
    const int c = (k < V) ? meta[CSS_META_CLS_OF_SLOT + k] : 0;
    const int n_hard = (k < V) ? meta[CSS_META_N_HARD + c] : 0;
    if (k >= V || V <= 1 || n_hard == 0) {
        if (threadIdx.x == 0) {
            loss_kq[k * Q + q] = 0.f;
            anchor_px[k * Q + q] = -1;
        }
        return;
    }
    const int grp = lane >> 3, l8 = lane & 7;
    const DrawKey dk = make_key(seed, ((uint64_t)(uint32_t)meta[CSS_META_DRAW_OFFSET + 1] << 32) | (uint32_t)meta[CSS_META_DRAW_OFFSET]);
    const int ai = FED ? anchor_idx[k * Q + q] : draw_anchor(dk, k, q, n_hard);
    const int pa = hard_list[(size_t)c * N + ai];              // in flight while the slot tables are built
    build_slot_tables(tb, meta, class_cdf, k, V);

    // warp w owns the negatives j - 1 = w + SC_WARPS n, n < cnt, four per step (one per group)
    const int cnt = (Nn - warp + SC_WARPS - 1) / SC_WARPS;
    const int T = (cnt + 3) >> 2;
    int2 cur = ring_candidate_row<FED>(tb, dk, neg_idx, valid_list, k, q, Q, Nn, N, lane, cnt);
    int2 nxt = ring_candidate_row<FED>(tb, dk, neg_idx, valid_list, k, q, Q, Nn, N, 32 + lane, cnt);

    // this lane's 16-byte chunks of the ring: stage s, chunk i at lane_base + s * RING_STAGE_BYTES + i * 128
    const uint32_t ring0 = (uint32_t)__cvta_generic_to_shared(ring_smem) + warp * (STAGES * RING_STAGE_BYTES) + grp * (CSS_D * 4) + l8 * 16;
    const char* rows_b = reinterpret_cast<const char*>(rows) + l8 * 16;
    auto issue = [&](uint32_t stage_off, int row) {
        const char* src = rows_b + (size_t)max(row, 0) * (CSS_D * 4);      // past the end: any finite row, weight 0
#pragma unroll
        for (int i = 0; i < 8; ++i) cp_async16(ring0 + stage_off + i * 128, src + i * 128);
    };
    uint32_t wr_off = 0, rd_off = 0;
#pragma unroll
    for (int p = 0; p < STAGES - 1; ++p) {
        issue(wr_off, __shfl_sync(0xffffffffu, cur.x, p * 4 + grp));
        cp_async_commit();
        wr_off += RING_STAGE_BYTES;
    }

    float4 a[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = row_f4(rows, (size_t)pa, i * 8 + l8);
    const float inv_na = 1.f / fmaxf(norms[pa], 1e-8f);       // cosine_similarity eps (loss.py:146)
    const float scale2 = 1.4426950408889634f / temp;

    Online st;
    st.m = FIX ? scale2 : -INFINITY;
    st.l = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) st.acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);

    // candidate 0 = the (updated) prototype of class c (loss.py:143-144): scored by every warp, kept by warp 0 / group 0
    float z0, cos_pos;
    {
        const float4* pp = proto_hat + (size_t)c * (CSS_D / 4) + l8;
        float4 r[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) r[i] = __ldg(pp + i * 8);
        cos_pos = group_sum8(dot8(a, r)) * inv_na;
        z0 = cos_pos * scale2;
        online_update<true, FIX>(st, z0, warp == 0 && grp == 0, 1.f, r);
    }

    // Batches of 8 steps (the ids of 32 candidates live one per lane).  A partial last batch runs all 8 steps: candidates past the
    // end carry weight 0 and copy row 0 (the loop has a single exit, which keeps the accumulators out of local memory).
#pragma unroll 1
    for (int b = 0; b * 8 < T; ++b) {
#pragma unroll 1
        for (int t = 0; t < 8; ++t) {
            {   // copies of step s + STAGES - 1
                const int tp = t + (STAGES - 1);
                const int prow = __shfl_sync(0xffffffffu, (tp < 8) ? cur.x : nxt.x, (tp & 7) * 4 + grp);
                issue(wr_off, prow);
                cp_async_commit();
                wr_off = (wr_off + RING_STAGE_BYTES == STAGES * RING_STAGE_BYTES) ? 0u : wr_off + RING_STAGE_BYTES;
            }
            cp_async_wait<STAGES - 1>();
            const int row = __shfl_sync(0xffffffffu, cur.x, t * 4 + grp);
            const float inv = __int_as_float(__shfl_sync(0xffffffffu, cur.y, t * 4 + grp));
            float4 r[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) r[i] = lds128(ring0 + rd_off + i * 128);
            rd_off = (rd_off + RING_STAGE_BYTES == STAGES * RING_STAGE_BYTES) ? 0u : rd_off + RING_STAGE_BYTES;
            const float cosv = group_sum8(dot8(a, r)) * (inv_na * inv);
            online_update<true, FIX>(st, cosv * scale2, row >= 0, inv, r);
        }
        cur = nxt;
        nxt = ring_candidate_row<FED>(tb, dk, neg_idx, valid_list, k, q, Q, Nn, N, (b + 2) * 32 + lane, cnt);
    }
    cp_async_wait<0>();
    finish_query<true, float>(st, z0, cos_pos, sh, rows, proto_hat, inv_na, pa, c, k, q, Q, V, temp, loss_kq, anchor_px, grad_anchor);
}

// -------------------------------------------------------------------------------------------------------------------
// Hybrid with the bulk-copy engine: LDGSTS copies queue on the SM's L1 data pipe like the register loads do (global wavefronts +
// the shared-memory write), which is why the ring above loses.  Here every PERIOD-th step of a warp comes in through cp.async.bulk
// (the TMA unit writes shared memory on its own port, completion on an mbarrier) and the other steps are plain register loads, so
// the two paths fetch concurrently: 4 KB per warp in flight on each.  The bulk path alone tops out near 31 B/clk/SM (round 1).
// NBUF buffers of four rows per warp; buffered step j uses buffer j % NBUF, refilled NBUF buffered steps (NBUF * PERIOD steps) ahead.
// -------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void sc_mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void sc_mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "SC_WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra SC_DONE;\n\t"
        "bra SC_WAIT_LOOP;\n\t"
        "SC_DONE:\n\t"
        "}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void sc_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void sc_bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes),
                 "r"(bar) : "memory");
}

template <bool FIX, bool FED, int PERIOD, int NBUF, int MINB>
__global__ void __launch_bounds__(SC_THREADS, MINB) score_ce_bulk_kernel(
    const float* __restrict__ rows, const float* __restrict__ norms, const float4* __restrict__ proto_hat,
    const float* __restrict__ class_cdf, const int2* __restrict__ valid_list, const int32_t* __restrict__ hard_list,
    const int32_t* __restrict__ meta, const int32_t* __restrict__ anchor_idx, const int32_t* __restrict__ neg_idx, uint64_t seed,
    int N, int Q, int Nn, float temp, float* __restrict__ loss_kq, int32_t* __restrict__ anchor_px, float4* __restrict__ grad_anchor) {
    static_assert(NBUF * PERIOD <= 8 && 8 % PERIOD == 0 && (8 / PERIOD) % NBUF == 0, "refill distance must stay inside the next id batch");
    css_pdl_enter();
    __shared__ __align__(128) unsigned char stage_smem[SC_WARPS * NBUF * RING_STAGE_BYTES];
    __shared__ __align__(8) unsigned long long bars[SC_WARPS * NBUF];
    __shared__ SlotTables tb;
    __shared__ QueryShared sh;
    const int k = blockIdx.y, q = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int V = meta[CSS_META_V];
    const int c = (k < V) ? meta[CSS_META_CLS_OF_SLOT + k] : 0;
    const int n_hard = (k < V) ? meta[CSS_META_N_HARD + c] : 0;
    if (k >= V || V <= 1 || n_hard == 0) {
        if (threadIdx.x == 0) {
            loss_kq[k * Q + q] = 0.f;
            anchor_px[k * Q + q] = -1;
        }
        return;
    }
    const int grp = lane >> 3, l8 = lane & 7;
    const uint32_t bar0 = (uint32_t)__cvta_generic_to_shared(bars) + warp * NBUF * 8;
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < NBUF; ++i) sc_mbar_init(bar0 + i * 8, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    const DrawKey dk = make_key(seed, ((uint64_t)(uint32_t)meta[CSS_META_DRAW_OFFSET + 1] << 32) | (uint32_t)meta[CSS_META_DRAW_OFFSET]);
    const int ai = FED ? anchor_idx[k * Q + q] : draw_anchor(dk, k, q, n_hard);
    const int pa = hard_list[(size_t)c * N + ai];
    build_slot_tables(tb, meta, class_cdf, k, V);              // (its barrier also publishes the mbarrier inits)

    const int cnt = (Nn - warp + SC_WARPS - 1) / SC_WARPS;
    const int T = (cnt + 3) >> 2;
    int2 cur = ring_candidate_row<FED>(tb, dk, neg_idx, valid_list, k, q, Q, Nn, N, lane, cnt);
    int2 nxt = ring_candidate_row<FED>(tb, dk, neg_idx, valid_list, k, q, Q, Nn, N, 32 + lane, cnt);

    const uint32_t grp_buf = (uint32_t)__cvta_generic_to_shared(stage_smem) + warp * (NBUF * RING_STAGE_BYTES) + grp * (CSS_D * 4);
    const uint32_t buf = grp_buf + l8 * 16;
    auto refill = [&](int ib, int row) {       // the group's leader copies the group's row; lane 0 arms the warp's barrier
        if (lane == 0) sc_mbar_expect_tx(bar0 + ib * 8, RING_STAGE_BYTES);
        if (l8 == 0) sc_bulk_g2s(grp_buf + ib * RING_STAGE_BYTES, reinterpret_cast<const char*>(rows) + (size_t)max(row, 0) * (CSS_D * 4), CSS_D * 4, bar0 + ib * 8);
    };
#pragma unroll
    for (int i = 0; i < NBUF; ++i) refill(i, __shfl_sync(0xffffffffu, cur.x, i * PERIOD * 4 + grp));

    float4 a[8];                                               // the anchor stays in registers (128 registers, 4 CTAs/SM)
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = row_f4(rows, (size_t)pa, i * 8 + l8);
    const float inv_na = 1.f / fmaxf(norms[pa], 1e-8f);
    const float scale2 = 1.4426950408889634f / temp;

    Online st;
    st.m = FIX ? scale2 : -INFINITY;
    st.l = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) st.acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);

    float z0, cos_pos;
    {
        const float4* pp = proto_hat + (size_t)c * (CSS_D / 4) + l8;
        float4 r[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) r[i] = __ldg(pp + i * 8);
        cos_pos = group_sum8(dot8(a, r)) * inv_na;
        z0 = cos_pos * scale2;
        online_update<true, FIX>(st, z0, warp == 0 && grp == 0, 1.f, r);
    }

    uint32_t parity = 0;
#pragma unroll 1
    for (int b = 0; b * 8 < T; ++b) {
        const bool more = (b + 1) * 8 < T;               // a next batch exists: refills may reach into it
#pragma unroll 1
        for (int tb0 = 0; tb0 < 8; tb0 += NBUF * PERIOD) {
#pragma unroll
          for (int ib = 0; ib < NBUF; ++ib) {
            const int t0 = tb0 + ib * PERIOD;
            {   // buffered step
                const int row = __shfl_sync(0xffffffffu, cur.x, t0 * 4 + grp);
                const float inv = __int_as_float(__shfl_sync(0xffffffffu, cur.y, t0 * 4 + grp));
                sc_mbar_wait(bar0 + ib * 8, parity);
                float4 r[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) r[i] = lds128(buf + ib * RING_STAGE_BYTES + i * 128);
                const float cosv = group_sum8(dot8(a, r)) * (inv_na * inv);
                __syncwarp();                                   // every lane has read the buffer
                const int tp = t0 + NBUF * PERIOD;
                const int prow = __shfl_sync(0xffffffffu, (tp < 8) ? cur.x : nxt.x, (tp & 7) * 4 + grp);
                if (tp < 8 || more) refill(ib, prow);
                online_update<true, FIX>(st, cosv * scale2, row >= 0, inv, r);
            }
#pragma unroll
            for (int u = 1; u < PERIOD; ++u) {                  // register steps
                const int t = t0 + u;
                const int row = __shfl_sync(0xffffffffu, cur.x, t * 4 + grp);
                const float inv = __int_as_float(__shfl_sync(0xffffffffu, cur.y, t * 4 + grp));
                const float4* p = reinterpret_cast<const float4*>(rows) + (size_t)max(row, 0) * (CSS_D / 4) + l8;
                float4 r[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) r[i] = __ldg(p + i * 8);
                const float cosv = group_sum8(dot8(a, r)) * (inv_na * inv);
                online_update<true, FIX>(st, cosv * scale2, row >= 0, inv, r);
            }
          }
          parity ^= 1u;
        }
        cur = nxt;
        nxt = ring_candidate_row<FED>(tb, dk, neg_idx, valid_list, k, q, Q, Nn, N, (b + 2) * 32 + lane, cnt);
    }
    finish_query<true, float>(st, z0, cos_pos, sh, rows, proto_hat, inv_na, pa, c, k, q, Q, V, temp, loss_kq, anchor_px, grad_anchor);
}

// loss = (1/V) sum_k (1/Q) sum_q loss_kq ; exactly 0 when V <= 1 (loss.py:116-117,149).  One block, fixed-order tree.
__global__ void __launch_bounds__(256) loss_reduce_kernel(const float* __restrict__ loss_kq, const int32_t* __restrict__ meta, int Q,
                                                          float* __restrict__ loss) {
    css_pdl_enter();
    __shared__ float part[8];
    const int V = meta[CSS_META_V];
    float s = 0.f;
    if (V > 1) {
        for (int i0 = threadIdx.x; i0 < V * Q; i0 += 256 * 8) {            // 8 loads in flight, added in index order
            float v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = (i0 + u * 256 < V * Q) ? loss_kq[i0 + u * 256] : 0.f;
#pragma unroll
            for (int u = 0; u < 8; ++u) s += v[u];
        }
    }
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (int i = 0; i < 8; ++i) t += part[i];
        *loss = (V > 1) ? t / ((float)Q * (float)V) : 0.f;
    }
}

// which kernel scores fp32 rows with the gradient: 0 = register kernel (default: whole-warp rows, 8 rows per batch in flight per
// warp at 4 CTAs/SM, the most the 128-register budget holds without spills; the 5376 CTAs of the bench shape make 9.08 waves),
// 1 = shared-memory ring (2 stages, cp.async), 2 = register / bulk-copy hybrid on 8-lane groups; css_set_scorer_path() overrides
// CSS_B200_SCORER=reg|ring|bulk, which overrides the default
#ifndef CSS_SCORER_DEFAULT
#define CSS_SCORER_DEFAULT 0
#endif
static int g_scorer_path = -1;
extern "C" int css_set_scorer_path(int path) {
    g_scorer_path = (path < 0 || path > 2) ? -1 : path;
    return 0;
}
static int css_scorer_path() {
    if (g_scorer_path >= 0) return g_scorer_path;
    static int env = -1;
    if (env < 0) {
        const char* v = getenv("CSS_B200_SCORER");
        env = !v ? CSS_SCORER_DEFAULT : !strcmp(v, "reg") ? 0 : !strcmp(v, "ring") ? 1 : !strcmp(v, "bulk") ? 2 : CSS_SCORER_DEFAULT;
    }
    return env;
}

template <bool FIX, bool FED, int STAGES, int MINB, typename... Args>
static cudaError_t launch_ring(dim3 grid, cudaStream_t st, Args... args) {
    static bool configured = false;
    const size_t smem = (size_t)SC_WARPS * STAGES * RING_STAGE_BYTES;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(score_ce_ring_kernel<FIX, FED, STAGES, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        configured = true;
    }
    return css_launch(score_ce_ring_kernel<FIX, FED, STAGES, MINB>, grid, dim3(SC_THREADS), smem, st, args...);
}

template <bool FIX, bool FED, int PERIOD, int NBUF, int MINB, typename... Args>
static cudaError_t launch_bulk(dim3 grid, cudaStream_t st, Args... args) {
    return css_launch(score_ce_bulk_kernel<FIX, FED, PERIOD, NBUF, MINB>, grid, dim3(SC_THREADS), (size_t)0, st, args...);
}

extern "C" int css_score_ce(const void* rows, int rows_dtype, const float* norms, const float* proto_hat, const float* class_cdf,
                            const int32_t* valid_list, const int32_t* hard_list, int32_t* meta, const int32_t* anchor_idx,
                            const int32_t* neg_idx, uint64_t seed, uint64_t offset, uint64_t* step_counter, int N, int C, int D, int Q,
                            int Nn, float temp, float* loss_kq, int32_t* anchor_px, float* grad_anchor, float* loss, void* stream) {
    CSS_CHECK_ARG(rows && norms && proto_hat && class_cdf && valid_list && hard_list && meta && loss_kq && anchor_px && loss,
                  CSS_E_ARG, "css_score_ce: null pointer");
    CSS_CHECK_ARG((anchor_idx == nullptr) == (neg_idx == nullptr), CSS_E_ARG,
                  "css_score_ce: anchor_idx and neg_idx must be fed together");
    CSS_CHECK_ARG(N > 0 && Q > 0 && Nn > 0 && Q < (1 << 24), CSS_E_ARG, "css_score_ce: bad N/Q/Nn");
    CSS_CHECK_ARG(rows_dtype == CSS_DTYPE_F32 || rows_dtype == CSS_DTYPE_BF16, CSS_E_DTYPE, "css_score_ce: rows dtype %d", rows_dtype);
    CSS_CHECK_ARG(Q <= 65535 * 32768, CSS_E_SIZE, "css_score_ce: Q too large");
    if (int e = css_check_dims(C, D)) return e;
    cudaStream_t st = (cudaStream_t)stream;
    css_launch(draw_offset_kernel, dim3(1), dim3(1), (size_t)(0), (cudaStream_t)(st), offset, (unsigned long long*)step_counter, meta);
    dim3 grid(Q, C);
    // fixed-reference softmax whenever 2^(-2 log2(e)/temp) is far from fp32 underflow (temp > ~0.024); online max otherwise
    const bool fix = (2.f * 1.4426950408889634f / temp) < 120.f;
#define SC_ARGS(RT_) (const RT_*)rows, norms, (const float4*)proto_hat, class_cdf, (const int2*)valid_list, hard_list, (const int32_t*)meta, anchor_idx, neg_idx, seed, \
                     N, Q, Nn, temp, loss_kq, anchor_px, (float4*)grad_anchor
#define SC_RUN(RT_)                                                                                                 \
    do {                                                                                                            \
        if (grad_anchor) {                                                                                          \
            if (fix) css_launch(score_ce_kernel<true, false, true, true, RT_>, dim3(grid), dim3(SC_THREADS), (size_t)(0), (cudaStream_t)(st), SC_ARGS(RT_));         \
            else css_launch(score_ce_kernel<true, false, true, false, RT_>, dim3(grid), dim3(SC_THREADS), (size_t)(0), (cudaStream_t)(st), SC_ARGS(RT_));           \
        } else {                                                                                                    \
            if (fix) score_ce_kernel<false, sizeof(RT_) == 4, false, true, RT_><<<grid, SC_THREADS, 0, st>>>(SC_ARGS(RT_));       \
            else score_ce_kernel<false, sizeof(RT_) == 4, false, false, RT_><<<grid, SC_THREADS, 0, st>>>(SC_ARGS(RT_));         \
        }                                                                                                           \
    } while (0)
    const int path = (grad_anchor && rows_dtype == CSS_DTYPE_F32) ? css_scorer_path() : 0;
    if (path > 0) {
#define RING_ARGS (const float*)rows, norms, (const float4*)proto_hat, class_cdf, (const int2*)valid_list, hard_list, (const int32_t*)meta, anchor_idx, neg_idx, \
                  seed, N, Q, Nn, temp, loss_kq, anchor_px, (float4*)grad_anchor
#define RING_RUN(S_, B_) (neg_idx ? (fix ? launch_ring<true, true, S_, B_>(grid, st, RING_ARGS) : launch_ring<false, true, S_, B_>(grid, st, RING_ARGS)) \
                                  : (fix ? launch_ring<true, false, S_, B_>(grid, st, RING_ARGS) : launch_ring<false, false, S_, B_>(grid, st, RING_ARGS)))
#define BULK_RUN(P_, N_, B_) (neg_idx ? (fix ? launch_bulk<true, true, P_, N_, B_>(grid, st, RING_ARGS) : launch_bulk<false, true, P_, N_, B_>(grid, st, RING_ARGS)) \
                                     : (fix ? launch_bulk<true, false, P_, N_, B_>(grid, st, RING_ARGS) : launch_bulk<false, false, P_, N_, B_>(grid, st, RING_ARGS)))
        const cudaError_t e = path == 1 ? RING_RUN(2, 4) : BULK_RUN(2, 1, 4);
#undef BULK_RUN
#undef RING_RUN
#undef RING_ARGS
        if (e != cudaSuccess) { css_set_error("css_score_ce: ring launch: %s", cudaGetErrorString(e)); return (int)e; }
    } else if (rows_dtype == CSS_DTYPE_F32) SC_RUN(float);
    else SC_RUN(__nv_bfloat16);
#undef SC_RUN
#undef SC_ARGS
    css_launch(loss_reduce_kernel, dim3(1), dim3(256), (size_t)(0), (cudaStream_t)(st), loss_kq, meta, Q, loss);
    CSS_CHECK_LAUNCH("css_score_ce", 3);
    return 0;
}
