// Development microbenchmark: random 1 KB row gathers from a 104 976-row (107 MB, L2-resident) table, 5376 warps x 512 rows,
// in the two layouts the fp32 scorer can use (css_score.cu):
//   group: a warp is four 8-lane groups, one row per group at a time (score_ce_kernel / score_ce_bulk_kernel);
//   wide:  every row is spread over the whole warp (lane l holds float4 l and l + 32), R rows per batch, loaded in one batch
//          ("one") or as two alternating halves of R/2 rows, the next half in flight while the current one is scored ("halves").
// Each runs at 16, 20 and 24 warps/SM (launch bound + padding shared memory), with no math ("load": the rows are only summed)
// or with a stub of the scorer's per-row work ("stub"): the dot with a register anchor, its reduction (group: 3 shuffles; wide:
// the batched transpose-reduce), one exp2, the weight broadcast and the accumulation into a register gradient slice.
// `dev_gather_wide ids` runs only the candidate-id comparison (wide R = 8, one batch, 16 warps/SM, with the stub), in three
// ways of getting a batch's row ids and inverse norms:
//   (a) ids read contiguously, as above, inverse norm 1;
//   (b) per candidate a random 4-byte id from a class list, then a dependent 4-byte norm load and 1 / max(norm, 1e-8)
//       (IEEE division), the norm of the next 32 ids loaded after the batch's first rows, as score_rows_wide did;
//   (c) per candidate one random 8-byte {id, bits of the inverse norm} list entry.
// The list positions are random (they stand in for the scorer's Philox draws); the stub scales each dot and weight by the
// inverse norm, so no load is dead.  Five alternating rounds of the three.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -Xptxas -v -o dev_gather_wide dev_gather_wide.cu
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#define N_WARPS 5376
#define PER_WARP 512

__device__ __forceinline__ float2 lo2(const float4& v) { return make_float2(v.x, v.y); }
__device__ __forceinline__ float2 hi2(const float4& v) { return make_float2(v.z, v.w); }
__device__ __forceinline__ void axpy4(float w, const float4& r, float4& acc) {
    const float2 ww = make_float2(w, w);
    const float2 lo = __ffma2_rn(ww, lo2(r), lo2(acc)), hi = __ffma2_rn(ww, hi2(r), hi2(acc));
    acc = make_float4(lo.x, lo.y, hi.x, hi.y);
}
__device__ __forceinline__ float sum4(const float4& v) { return (v.x + v.y) + (v.z + v.w); }

// ---- layout (a): four 8-lane groups ------------------------------------------------------------------------------------
template <bool STUB, int MINB>
__global__ void __launch_bounds__(128, MINB) group_kernel(const float4* __restrict__ rows, const int* __restrict__ idx, float* __restrict__ out) {
    extern __shared__ float pad[];
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31, grp = lane >> 3, l8 = lane & 7;
    const int* my = idx + (size_t)warp * PER_WARP;
    float4 a[8], acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { a[i] = rows[(size_t)warp * 64 + i * 8 + l8]; acc[i] = make_float4(0.f, 0.f, 0.f, 0.f); }
    float l = 0.f;
    int ids = my[lane];
#pragma unroll 1
    for (int b = 0; b < PER_WARP; b += 32) {
        const int nxt = (b + 32 < PER_WARP) ? my[b + 32 + lane] : 0;
#pragma unroll 1
        for (int t = 0; t < 8; ++t) {
            const float4* p = rows + (size_t)__shfl_sync(0xffffffffu, ids, t * 4 + grp) * 64 + l8;
            float4 r[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) r[i] = __ldg(p + i * 8);
            if (STUB) {
                float2 s0 = make_float2(0.f, 0.f), s1 = s0, s2 = s0, s3 = s0;
#pragma unroll
                for (int i = 0; i < 8; i += 2) {
                    s0 = __ffma2_rn(lo2(a[i]), lo2(r[i]), s0);
                    s1 = __ffma2_rn(hi2(a[i]), hi2(r[i]), s1);
                    s2 = __ffma2_rn(lo2(a[i + 1]), lo2(r[i + 1]), s2);
                    s3 = __ffma2_rn(hi2(a[i + 1]), hi2(r[i + 1]), s3);
                }
                float d = ((s0.x + s0.y) + (s1.x + s1.y)) + ((s2.x + s2.y) + (s3.x + s3.y));
                d += __shfl_xor_sync(0xffffffffu, d, 1);
                d += __shfl_xor_sync(0xffffffffu, d, 2);
                d += __shfl_xor_sync(0xffffffffu, d, 4);
                const float w = exp2f(d * 1e-3f - 2.f);
                l += w;
#pragma unroll
                for (int i = 0; i < 8; ++i) axpy4(w, r[i], acc[i]);
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i) l += sum4(r[i]);
            }
        }
        ids = nxt;
    }
    float s = l;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += sum4(acc[i]);
    if (s == 123.456f) out[0] = s + pad[0];
}

// ---- layout (b): whole-warp rows ------------------------------------------------------------------------------------------
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

template <int H>
__device__ __forceinline__ void load_rows(const float4* __restrict__ rows, int ids, int t0, int lane, float4 (&r)[H][2]) {
#pragma unroll
    for (int i = 0; i < H; ++i) {
        const float4* p = rows + (size_t)__shfl_sync(0xffffffffu, ids, t0 + i) * 64 + lane;
        r[i][0] = __ldg(p);
        r[i][1] = __ldg(p + 32);
    }
}

template <bool STUB, int H>
__device__ __forceinline__ void work_rows(const float4 (&r)[H][2], const float4& a0, const float4& a1, float4& acc0, float4& acc1, float& l,
                                          int lane) {
    if (STUB) {
        float d[H];
#pragma unroll
        for (int i = 0; i < H; ++i) {
            float2 s = __fmul2_rn(lo2(a0), lo2(r[i][0]));
            s = __ffma2_rn(hi2(a0), hi2(r[i][0]), s);
            s = __ffma2_rn(lo2(a1), lo2(r[i][1]), s);
            s = __ffma2_rn(hi2(a1), hi2(r[i][1]), s);
            d[i] = s.x + s.y;
        }
        const float w = exp2f(transpose_sum<H>(d, lane) * 1e-3f - 2.f);
        if (lane % (32 / H) == 0) l += w;
#pragma unroll
        for (int i = 0; i < H; ++i) {
            const float wi = __shfl_sync(0xffffffffu, w, i * (32 / H));
            axpy4(wi, r[i][0], acc0);
            axpy4(wi, r[i][1], acc1);
        }
    } else {
#pragma unroll
        for (int i = 0; i < H; ++i) l += sum4(r[i][0]) + sum4(r[i][1]);
    }
}

template <bool STUB, int R, bool HALVES, int MINB>
__global__ void __launch_bounds__(128, MINB) wide_kernel(const float4* __restrict__ rows, const int* __restrict__ idx, float* __restrict__ out) {
    extern __shared__ float pad[];
    constexpr int H = HALVES ? R / 2 : R;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    const int* my = idx + (size_t)warp * PER_WARP;
    const float4 a0 = rows[(size_t)warp * 64 + lane], a1 = rows[(size_t)warp * 64 + 32 + lane];
    float4 acc0 = make_float4(0.f, 0.f, 0.f, 0.f), acc1 = acc0;
    float l = 0.f;
    int ids = my[lane];
#pragma unroll 1
    for (int b = 0; b < PER_WARP; b += 32) {
        const int nxt = (b + 32 < PER_WARP) ? my[b + 32 + lane] : 0;
        if (!HALVES) {
#pragma unroll 1
            for (int t = 0; t < 32; t += R) {
                float4 r[R][2];
                load_rows<R>(rows, ids, t, lane, r);
                work_rows<STUB, R>(r, a0, a1, acc0, acc1, l, lane);
            }
        } else {
            float4 ra[H][2], rb[H][2];
            load_rows<H>(rows, ids, 0, lane, ra);
#pragma unroll 1
            for (int t = 0; t < 32; t += R) {
                load_rows<H>(rows, ids, t + H, lane, rb);
                work_rows<STUB, H>(ra, a0, a1, acc0, acc1, l, lane);
                if (t + R < 32) load_rows<H>(rows, ids, t + R, lane, ra);
                work_rows<STUB, H>(rb, a0, a1, acc0, acc1, l, lane);
            }
        }
        ids = nxt;
    }
    const float s = l + sum4(acc0) + sum4(acc1);
    if (s == 123.456f) out[0] = s + pad[0];
}

// ---- candidate ids (whole-warp rows, R = 8, one batch, stub) -------------------------------------------------------------
template <int MODE>
__device__ __forceinline__ int batch_ids(const int* __restrict__ list, const float* __restrict__ norms, const int2* __restrict__ entries,
                                         int pos, float& inv) {
    if (MODE == 0) { inv = 1.f; return pos; }
    if (MODE == 1) { const int id = list[pos]; inv = 1.f / fmaxf(norms[id], 1e-8f); return id; }
    const int2 e = entries[pos];
    inv = __int_as_float(e.y);
    return e.x;
}

template <int MODE, int MINB>
__global__ void __launch_bounds__(128, MINB) ids_kernel(const float4* __restrict__ rows, const int* __restrict__ idx, const int* __restrict__ list,
                                                        const float* __restrict__ norms, const int2* __restrict__ entries, float* __restrict__ out) {
    extern __shared__ float pad[];
    constexpr int R = 8, LPR = 32 / R;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    const int* my = idx + (size_t)warp * PER_WARP;
    const float4 a0 = rows[(size_t)warp * 64 + lane], a1 = rows[(size_t)warp * 64 + 32 + lane];
    float4 acc0 = make_float4(0.f, 0.f, 0.f, 0.f), acc1 = acc0;
    float l = 0.f, cur_inv;
    int cur = batch_ids<MODE>(list, norms, entries, my[lane], cur_inv);
#pragma unroll 1
    for (int b = 0; b < PER_WARP; b += 32) {
        const int pos = (b + 32 < PER_WARP) ? my[b + 32 + lane] : 0;
        int nxt;
        float nxt_inv = 1.f, nxt_nrm = 1.f;
        if (MODE == 1) nxt = list[pos];                           // its norm is loaded after the batch's first rows
        else nxt = batch_ids<MODE>(list, norms, entries, pos, nxt_inv);
#pragma unroll 1
        for (int t = 0; t < 32; t += R) {
            float4 r[R][2];
            load_rows<R>(rows, cur, t, lane, r);
            float d[R];
#pragma unroll
            for (int i = 0; i < R; ++i) {
                float2 s = __fmul2_rn(lo2(a0), lo2(r[i][0]));
                s = __ffma2_rn(hi2(a0), hi2(r[i][0]), s);
                s = __ffma2_rn(lo2(a1), lo2(r[i][1]), s);
                s = __ffma2_rn(hi2(a1), hi2(r[i][1]), s);
                d[i] = s.x + s.y;
            }
            const float inv = __shfl_sync(0xffffffffu, cur_inv, t + lane / LPR);
            const float w = exp2f(transpose_sum<R>(d, lane) * inv * 1e-3f - 2.f);
            if (lane % LPR == 0) l += w;
            const float wr = w * inv;
#pragma unroll
            for (int i = 0; i < R; ++i) {
                const float wi = __shfl_sync(0xffffffffu, wr, i * LPR);
                axpy4(wi, r[i][0], acc0);
                axpy4(wi, r[i][1], acc1);
            }
            if (MODE == 1 && t == 0) nxt_nrm = norms[nxt];
        }
        cur = nxt;
        cur_inv = (MODE == 1) ? 1.f / fmaxf(nxt_nrm, 1e-8f) : nxt_inv;
    }
    const float s = l + sum4(acc0) + sum4(acc1);
    if (s == 123.456f) out[0] = s + pad[0];
}

// ---- driver --------------------------------------------------------------------------------------------------------------
typedef void (*Kern)(const float4*, const int*, float*);

// `launch(smem)` launches kernel `kf` once with that much padding shared memory
template <typename Launch>
static double run_kernel(const void* kf, Launch launch, int target_ctas, const char* name, double clk_ghz, int n_sm) {
    cudaFuncAttributes fa;
    cudaFuncGetAttributes(&fa, kf);
    int smem = 0, occ = 0;
    for (smem = 0; smem <= 200 * 1024; smem += 512) {         // the least padding that leaves target_ctas CTAs per SM
        cudaFuncSetAttribute(kf, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kf, 128, smem);
        if (occ <= target_ctas) break;
    }
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    float best = 1e30f;
    for (int rep = 0; rep < 5; ++rep) {
        cudaEventRecord(e0);
        launch(smem);
        cudaEventRecord(e1);
        cudaEventSynchronize(e1);
        float ms;
        cudaEventElapsedTime(&ms, e0, e1);
        if (rep >= 1 && ms < best) best = ms;
    }
    const double bytes = (double)N_WARPS * PER_WARP * 1024;
    const double tbs = bytes / (best * 1e-3) / 1e12;
    printf("%-28s warps/SM %2d (regs %3d, spill %3d B): %7.1f us  %6.2f TB/s  %6.1f B/clk/SM  (%s)\n", name, occ * 4, fa.numRegs,
           (int)fa.localSizeBytes, best * 1e3, tbs, bytes / (best * 1e-3) / (clk_ghz * 1e9) / n_sm, cudaGetErrorString(cudaGetLastError()));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return tbs;
}

static double run(Kern k, int target_ctas, const char* name, const float4* rows, const int* idx, float* out, double clk_ghz, int n_sm) {
    return run_kernel((const void*)k, [&](int smem) { k<<<N_WARPS / 4, 128, smem>>>(rows, idx, out); }, target_ctas, name, clk_ghz, n_sm);
}

typedef void (*IdsKern)(const float4*, const int*, const int*, const float*, const int2*, float*);
static double run_ids(IdsKern k, const char* name, const float4* rows, const int* idx, const int* list, const float* norms,
                      const int2* entries, float* out, double clk_ghz, int n_sm) {
    return run_kernel((const void*)k, [&](int smem) { k<<<N_WARPS / 4, 128, smem>>>(rows, idx, list, norms, entries, out); }, 4, name,
                      clk_ghz, n_sm);
}

int main(int argc, char** argv) {
    const bool ids_only = argc > 1 && !strcmp(argv[1], "ids");
    const int n_rows = 104976;
    float4* rows;
    int* idx;
    float* out;
    cudaMalloc(&rows, (size_t)n_rows * 1024);
    cudaMemset(rows, 0, (size_t)n_rows * 1024);
    cudaMalloc(&idx, (size_t)N_WARPS * PER_WARP * 4);
    cudaMalloc(&out, 4);
    int* h = (int*)malloc((size_t)N_WARPS * PER_WARP * 4);
    srand(1);
    for (size_t i = 0; i < (size_t)N_WARPS * PER_WARP; ++i) h[i] = (int)(((uint64_t)rand() * 2654435761u) % n_rows);
    cudaMemcpy(idx, h, (size_t)N_WARPS * PER_WARP * 4, cudaMemcpyHostToDevice);
    int clk_khz = 0, n_sm = 0;
    cudaDeviceGetAttribute(&clk_khz, cudaDevAttrClockRate, 0);
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, 0);
    const double ghz = clk_khz * 1e-6;
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, 0);
    printf("%s, %d SMs, max SM clock %.3f GHz (B/clk/SM at that clock); 104976 rows (107 MB), %d x %d gathers of 1 KB, best of 4\n",
           prop.name, n_sm, ghz, N_WARPS, PER_WARP);
#define ALL(STUB, TAG)                                                                                                         \
    run(group_kernel<STUB, 4>, 4, "group " TAG, rows, idx, out, ghz, n_sm);                                                   \
    run(group_kernel<STUB, 5>, 5, "group " TAG, rows, idx, out, ghz, n_sm);                                                   \
    run(group_kernel<STUB, 6>, 6, "group " TAG, rows, idx, out, ghz, n_sm);                                                   \
    run(wide_kernel<STUB, 4, false, 4>, 4, "wide R4 one " TAG, rows, idx, out, ghz, n_sm);                                     \
    run(wide_kernel<STUB, 4, false, 5>, 5, "wide R4 one " TAG, rows, idx, out, ghz, n_sm);                                     \
    run(wide_kernel<STUB, 4, false, 6>, 6, "wide R4 one " TAG, rows, idx, out, ghz, n_sm);                                     \
    run(wide_kernel<STUB, 4, true, 4>, 4, "wide R4 halves " TAG, rows, idx, out, ghz, n_sm);                                   \
    run(wide_kernel<STUB, 4, true, 5>, 5, "wide R4 halves " TAG, rows, idx, out, ghz, n_sm);                                   \
    run(wide_kernel<STUB, 4, true, 6>, 6, "wide R4 halves " TAG, rows, idx, out, ghz, n_sm);                                   \
    run(wide_kernel<STUB, 8, false, 4>, 4, "wide R8 one " TAG, rows, idx, out, ghz, n_sm);                                     \
    run(wide_kernel<STUB, 8, false, 5>, 5, "wide R8 one " TAG, rows, idx, out, ghz, n_sm);                                     \
    run(wide_kernel<STUB, 8, false, 6>, 6, "wide R8 one " TAG, rows, idx, out, ghz, n_sm);                                     \
    run(wide_kernel<STUB, 8, true, 4>, 4, "wide R8 halves " TAG, rows, idx, out, ghz, n_sm);                                   \
    run(wide_kernel<STUB, 8, true, 5>, 5, "wide R8 halves " TAG, rows, idx, out, ghz, n_sm);                                   \
    run(wide_kernel<STUB, 8, true, 6>, 6, "wide R8 halves " TAG, rows, idx, out, ghz, n_sm)
    if (ids_only) {
        // list[p]: a row id; norms in [0.5, 2); entries[p] = {list[p], bits of 1 / max(norms[list[p]], 1e-8)}
        int* hl = (int*)malloc((size_t)n_rows * 4);
        float* hn = (float*)malloc((size_t)n_rows * 4);
        int2* he = (int2*)malloc((size_t)n_rows * 8);
        for (int i = 0; i < n_rows; ++i) hn[i] = 0.5f + 1.5f * (float)rand() / (float)RAND_MAX;
        for (int i = 0; i < n_rows; ++i) {
            hl[i] = (int)(((uint64_t)rand() * 2654435761u) % n_rows);
            const float inv = 1.f / fmaxf(hn[hl[i]], 1e-8f);
            int bits;
            memcpy(&bits, &inv, 4);
            he[i] = make_int2(hl[i], bits);
        }
        int* dl;
        float* dn;
        int2* de;
        cudaMalloc(&dl, (size_t)n_rows * 4);
        cudaMalloc(&dn, (size_t)n_rows * 4);
        cudaMalloc(&de, (size_t)n_rows * 8);
        cudaMemcpy(dl, hl, (size_t)n_rows * 4, cudaMemcpyHostToDevice);
        cudaMemcpy(dn, hn, (size_t)n_rows * 4, cudaMemcpyHostToDevice);
        cudaMemcpy(de, he, (size_t)n_rows * 8, cudaMemcpyHostToDevice);
        for (int round = 0; round < 5; ++round) {
            printf("round %d\n", round);
            run_ids(ids_kernel<0, 4>, "ids (a) contiguous", rows, idx, dl, dn, de, out, ghz, n_sm);
            run_ids(ids_kernel<1, 4>, "ids (b) list + norm + div", rows, idx, dl, dn, de, out, ghz, n_sm);
            run_ids(ids_kernel<2, 4>, "ids (c) 8-byte entry", rows, idx, dl, dn, de, out, ghz, n_sm);
        }
        printf("last error: %s\n", cudaGetErrorString(cudaDeviceSynchronize()));
        return 0;
    }
    ALL(false, "load");
    ALL(true, "stub");
    printf("last error: %s\n", cudaGetErrorString(cudaDeviceSynchronize()));
    return 0;
}
