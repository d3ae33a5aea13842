/*
 * css_b200.h -- C ABI of libcss_b200.so: the B200 (sm_100a) representation-space hot path of CSS.
 *
 * Drop-in boundary.  The reference (WangChangqi98/CSS) is pure Python/PyTorch and has no FFI of its own;
 * every entry point below therefore replaces a block of eager PyTorch statements, cited as
 * <file>:<lines> relative to the reference root.  The Python bindings a maintainer adds on the
 * reference side are shown in INTEGRATION.md (ctypes, `css_b200/_lib.py`).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in `_host`; tensors are contiguous, NCHW;
 *   - the caller owns every buffer (inputs, outputs, scratch); no data-path entry point allocates or frees
 *     device memory or keeps global device state.  ONE documented exception, set-up only: css_comm_alloc /
 *     css_comm_free own the small (<= 0.6 MB) peer-memory exchange buffer, because memory that is exported with a
 *     CUDA IPC handle must be its own cudaMalloc allocation (a sub-block of a caching allocator's segment cannot be);
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*), performs no host
 *     synchronisation, and is CUDA-graph capturable;
 *   - return value: 0 = ok, <0 = argument error (see CSS_E_*), >0 = cudaError_t of the failed launch;
 *     `css_last_error()` returns a thread-local message for the last non-zero return;
 *   - D (feature width) must be 256: the reference hard-codes output_dim=256 (mix_label.py:75,93);
 *     C (classes) must be in [1, 32] (per-pixel class sets are 32-bit masks).
 *
 * Pixel ids: pixel (b, y, x) of a [B, *, h, w] map has id (b*h + y)*w + x, the row-major order in which the
 * reference's boolean-mask gathers enumerate pixels (loss.py:111-112).
 */
#ifndef CSS_B200_H
#define CSS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CSS_B200_VERSION 100

#define CSS_E_ARG      (-1)   /* null pointer / non-positive size                     */
#define CSS_E_DIM      (-2)   /* D != 256 or C outside [1,32]                          */
#define CSS_E_DTYPE    (-3)   /* unsupported rep dtype                                 */
#define CSS_E_SIZE     (-4)   /* problem exceeds an int32 index range                  */

#define CSS_DTYPE_F32  0
#define CSS_DTYPE_BF16 1

#define CSS_SIM_COS      0    /* cosine similarities                                   */
#define CSS_SIM_SOFTMAX  1    /* softmax_c(cos / temp)                                 */

#define CSS_FUSE_NONE    0    /* cross / ori strategies: no fused label                */
#define CSS_FUSE_MIX     1    /* mix strategy: agree ? label_cls : 255                 */

/* number of int32 words in the selection meta block (see css_select) */
#define CSS_META_WORDS   256
/* offsets (int32 words) into meta */
#define CSS_META_V            0      /* number of locally present classes                        */
#define CSS_META_N_VALID      32     /* [32] valid-pixel count per class                          */
#define CSS_META_N_HARD       64     /* [32] hard-pixel count per class                           */
#define CSS_META_CLS_OF_SLOT  96     /* [32] class id of the k-th present class (increasing)      */
#define CSS_META_SLOT_OF_CLS  128    /* [32] slot of a class, -1 when absent                      */
#define CSS_META_TICKET       160    /* internal: last-CTA election of the scan kernel            */
#define CSS_META_DRAW_OFFSET  162    /* [2] lo/hi words of the Philox offset used by the last css_score_ce */
#define CSS_META_ROWS_STALE   164    /* cleared by css_select, raised by css_rows_refresh when the carried rows differ */

int         css_version(void);
const char* css_last_error(void);
/* number of streaming multiprocessors of the current device (grid sizing); <0 on error */
int         css_sm_count(void);
/* cumulative number of CUDA kernels this library has launched in this process (bench.py's gpu_launches) */
unsigned long long css_launch_count(void);
/* Programmatic dependent launch: every kernel of the library is launched with the programmatic-stream-serialization attribute
 * and begins with griddepcontrol.wait (nothing is read before the previous grid of the stream has completed and flushed) followed
 * by griddepcontrol.launch_dependents, so consecutive launches of the path overlap their scheduling with the previous kernel's
 * tail, eagerly and inside captured CUDA graphs.  OFF by default (measured on B200: 0.478 ms/step with it, 0.475 without -- the
 * early-launched CTAs hold SM resources while they wait); css_set_pdl(1) or CSS_B200_PDL=1 turns it on. */
int css_set_pdl(int on);

/* ---- stage 1 / 1b (+ the loss's pixel-major copy): ONE streaming read of an NCHW representation map -----------------
 * css_rep_pass produces any combination of
 *  (a) sim_out [B,C,h,w] f32: cosine (mode CSS_SIM_COS) or softmax_c(cos/temp) (CSS_SIM_SOFTMAX) similarity of every
 *      pixel's D-vector against the class prototypes.  Replaces ddp_model.py:104-110 (teacher sim_mat) and
 *      :147-154 / :230-237 (student prob_all).  Needs prototypes [C,D] and proto_scratch f32[2*D*32] (normalised,
 *      transposed prototypes; F.normalize eps 1e-12).
 *  (b) rows [N*D] + norms f32[N]: the pixel-major copy (row p = pixel id p, raw values, SAME dtype as rep: a bf16 map gives
 *      lossless bf16 rows and halves the gather bytes) and ||x_p||, from which the loss gathers candidate rows and
 *      accumulates class sums (loss.py:85,102,111-112,142).
 * NULL sim_out skips (a); NULL rows/norms skips (b).  css_sim_map is (a) alone.
 * rep_dtype: CSS_DTYPE_F32 or CSS_DTYPE_BF16 (bf16 is widened exactly; all arithmetic and all outputs stay fp32).
 */
int css_rep_pass(const void* rep, int rep_dtype, const float* prototypes, float* proto_scratch,
                 int B, int C, int D, int h, int w, int mode, float temp,
                 float* sim_out, void* rows, float* norms, void* stream);
int css_sim_map(const void* rep, int rep_dtype, const float* prototypes, float* proto_scratch,
                int B, int C, int D, int h, int w, int mode, float temp, float* out, void* stream);
/* (a) has two implementations for fp32 maps: tcgen05.mma kind::tf32 with TMEM accumulators and an fp32-exact hi/lo operand split
 * (css_sim_tc.cu), and packed-FFMA2 CUDA-core dots (css_sim.cu; always used for bf16 maps and for (b) alone).
 * css_set_rep_pass_path(1 / 0) selects one for this process, -1 returns to the default / the CSS_B200_REP_PASS=tc|fma
 * environment variable.  Both meet the path's tolerances (similarities abs 2e-6, labels identical away from 1e-5 near-ties). */
int css_set_rep_pass_path(int use_tc);

/* ---- channels-last maps (extension; the reference's maps are NCHW) ---------------------------------------------------------------
 * A representation map produced by a channels_last network (torch.channels_last: strides (h*w*D, 1, w*D, D)) is, in memory,
 * [pixel][D]: it IS the pixel-major row table the loss gathers from.  css_rep_pass_nhwc computes the similarities (a) straight
 * from it -- 2-D TMA tiles into shared memory, tcgen05.mma kind::tf32 with an exact hi/lo split, TMEM accumulators -- and
 * ||x_p||; there is no pixel-major copy to write.  sim_out [B,C,h,w] f32 (NCHW, as the callers expect) and norms f32[N] may
 * each be NULL (norms alone: prototypes may be NULL).  float32 only; rep_rows must be 16-byte aligned.
 * css_grad_scatter_nhwc writes the dense gradient in the same memory format: zero fill + one row update per anchor.
 * css_rows_refresh_nhwc is the twin of css_rows_refresh: `src_rows` is the map the carried norms came from.
 */
int css_rep_pass_nhwc(const void* rep_rows, int rep_dtype, const float* prototypes, float* proto_scratch,
                      int B, int C, int D, int h, int w, int mode, float temp, float* sim_out, float* norms, void* stream);
int css_grad_scatter_nhwc(const float* grad_out, const int32_t* anchor_px, const float* grad_anchor,
                          int n_anchor, int B2, int D, int h, int w, float* grad_rows, void* stream);
int css_rows_refresh_nhwc(const void* rep_rows, const void* src_rows, float* norms, float* proto_scratch, int32_t* meta,
                          int B, int D, int h, int w, void* stream);

/* ---- carried rows: "are these still the rows of THIS map?" ---------------------------------------------------------------
 * The reference wraps the model in DistributedDataParallel(find_unused_parameters=True) (mix_label.py:76-77,
 * cross_label.py, ori_pseudo.py alike); DDP's output sink clones rep_all, so the loss (loss.py:75) receives equal content at
 * a different address than the map the student pass read.  css_rows_refresh keeps the one-read property without trusting
 * addresses: a sampled bit-for-bit comparison of `rep` with `rows` (4 channels of every pixel, 64 apart, rotating with the
 * pixel id) raises meta[CSS_META_ROWS_STALE] on any difference, and the rows-only pass that follows in the same call
 * rewrites rows / norms from `rep` only if that word is set (otherwise it returns at once).  Call after css_select of the same
 * step (which clears the word).  Two launches, no host synchronisation, graph-capturable.
 */
int css_rows_refresh(const void* rep, int rep_dtype, void* rows, float* norms, int32_t* meta,
                     int B, int D, int h, int w, void* stream);

/* ---- stage 1 / 1' / 2 ----------------------------------------------------------------------------------------
 * Fused bilinear (align_corners=True) up-sampling + softmax + max of the similarity map and of the class logits,
 * plus the mix-label fusion, at crop resolution; the [B,C,H,W] up-sampled tensors are never materialised.
 * Replaces ddp_model.py:111-118 (Model_mix), :196-199 (Model_cross), :36-37 (Model_ori_pseudo).
 *   sim     [B,C,h,w] f32 or NULL (then the *_rep outputs and `fused` must be NULL)
 *   logits  [B,C,h,w] f32 or NULL (then the *_cls outputs and `fused` must be NULL)
 *   conf_*  [B,H,W] f32, label_* [B,H,W] i64, fused [B,H,W] f32 in {0..C-1, 255}; any output may be NULL.
 */
int css_upsample_label_fuse(const float* sim, const float* logits, float temp, int fuse_mode,
                            int B, int C, int h, int w, int H, int W,
                            float* conf_rep, int64_t* label_rep, float* conf_cls, int64_t* label_cls,
                            float* fused, void* stream);

/* ---- stage 3: selection ----------------------------------------------------------------------------------------
 * valid[p,c] = label[p,c]*mask[p] != 0, hard[p,c] = valid && prob[p,c] < strong_threshold, and the ORDER-PRESERVING
 * (row-major) per-class compaction of both.  Replaces loss.py:80,94-99,111-113.
 * css_select classifies and counts; css_select_lists writes the lists, once the norms of the rows the scorer will read are
 * final (after css_rep_pass / css_rows_refresh of the same step), because every valid-list entry carries its pixel's inverse norm.
 *   label [B2,C,h,w] f32, mask [B2,1,h,w] f32, prob [B2,C,h,w] f32          N = B2*h*w
 *   valid_bits, hard_bits   u32[N]      per-pixel class sets
 *   tile_counts             i32[2*C*T]  scratch, T = css_select_tiles(N); css_select leaves the lists' tile offsets in it
 *   meta                    i32[CSS_META_WORDS]   counts / present classes, layout CSS_META_*
 *   norms                   f32[N]      ||r_p|| (from css_rep_pass / css_rep_pass_nhwc / css_rows_refresh)
 *   valid_list              i32[C*N*2]  entry (c*N + i) = {pixel id, bits of the f32 1 / max(norms[id], 1e-8)}: class c's
 *                                       entries start at c*N (fixed stride, no cross-class scan)
 *   hard_list               i32[C*N]    class c's pixel ids start at c*N
 */
int css_select_tiles(int N);
int css_select(const float* label, const float* mask, const float* prob, float strong_threshold,
               int B2, int C, int h, int w,
               uint32_t* valid_bits, uint32_t* hard_bits, int32_t* tile_counts, int32_t* meta, void* stream);
int css_select_lists(const uint32_t* valid_bits, const uint32_t* hard_bits, const int32_t* tile_counts, const float* norms,
                     int C, int N, int32_t* valid_list, int32_t* hard_list, void* stream);

/* ---- stage 4a: per-class statistics ----------------------------------------------------------------------------------
 * Per-class feature sums and counts of this rank from the pixel-major rows: the all-reduce payload that replaces the
 * reference's all_gather (loss.py:77,81,102).  Deterministic (no atomics).
 *   rows [N*D] of rows_dtype (from css_rep_pass), valid_bits u32[N], meta i32[CSS_META_WORDS] (from css_select: the local counts)
 *   partials  f32[css_class_blocks(N) * C * D] + touched u32[css_class_blocks(N)]   scratch
 *   class_stats f32[C*(D+1)]  row c = [sum_d ... , count]
 */
int css_class_blocks(int N);
int css_class_stats(const void* rows, int rows_dtype, const uint32_t* valid_bits, const int32_t* meta, int N, int C, int D,
                    float* partials, uint32_t* touched, float* class_stats, void* stream);

/* ---- stage 4b: prototype EMA --------------------------------------------------------------------------------------
 * For every class present on THIS rank: mean = global_sum / global_count; prototypes[c] = mean if sum(prototypes[c])==0
 * else alpha*prototypes[c] + one_minus_alpha*mean, in place.  Replaces loss.py:101-109.  (one_minus_alpha is passed
 * separately because the reference evaluates 1 - alpha in double before rounding to fp32.)  Also emits what scoring needs:
 *   proto_hat f32[C*D]   updated prototypes / max(norm, 1e-8)
 *   class_cdf f32[32*32] row k: inclusive CDF of softmax(cos(P_k, P_j)/temp) over the other present classes in the
 *                        rotated order k+1..V-1,0..k-1 (loss.py:133-135)
 *   class_stats is the (all-reduced) [C, D+1] block; meta supplies the LOCAL counts.
 *   update_rule: CSS_UPDATE_LOCAL  = the reference's rule: a rank touches prototypes[c] only if c is present in ITS batch
 *                                    (loss.py:96-97), so per-rank prototypes may drift apart exactly as in the reference;
 *                CSS_UPDATE_GLOBAL = extension: every class with a positive GLOBAL count is updated on every rank -- ranks that
 *                                    start from equal prototypes stay bit-identical, no broadcast needed.
 */
#define CSS_UPDATE_LOCAL  0
#define CSS_UPDATE_GLOBAL 1
int css_proto_ema(float* prototypes, const float* class_stats, const int32_t* meta, float alpha,
                  float one_minus_alpha, float temp, int update_rule, int C, int D, float* proto_hat, float* class_cdf,
                  void* stream);

/* ---- stage 3: sampling (materialised; the scoring kernel can also draw on the fly) ---------------------------------
 * Anchors: Q uniform indices into each present class's hard list (loss.py:127).  Negatives: Nn iid draws of
 * (class ~ Categorical(class_cdf[k]), index ~ Uniform within that class's valid list), expressed as indices into the
 * rotated concatenation of valid lists (loss.py:136-142).  Philox4x32-10 keyed by (seed, offset); no host sync.
 *   anchor_idx i32[C*Q], neg_idx i32[C*Q*Nn]  (slot-major; slots >= V and slots without hard pixels are left at -1)
 */
int css_sample(const int32_t* meta, const float* class_cdf, uint64_t seed, uint64_t offset, int C, int Q, int Nn,
               int32_t* anchor_idx, int32_t* neg_idx, void* stream);

/* ---- stage 3: scoring + cross-entropy + d loss / d anchor ------------------------------------------------------------
 * Replaces loss.py:124-149 and its autograd backward up to the anchor rows.  rows / norms come from css_rep_pass, valid_list /
 * hard_list from css_select_lists with the same norms (norms itself is read for the anchors only).
 *   anchor_idx / neg_idx: as produced by css_sample or recorded from the reference; NULL = draw on the fly with
 *   (seed, offset + *step_counter), bit-identical to css_sample with the same (seed, offset).
 *   step_counter: optional DEVICE u64, read as an offset increment and incremented by one by the call, so that replays of a
 *   captured CUDA graph keep drawing fresh samples; NULL = use `offset` alone.  The offset actually used is left in
 *   meta[CSS_META_DRAW_OFFSET..+1].
 *   loss_kq f32[C*Q], anchor_px i32[C*Q] (pixel id of each anchor, -1 if none), grad_anchor f32[C*Q*D] or NULL,
 *   loss f32[1] = (1/V) sum_k (1/Q) sum_q loss_kq, exactly 0 when V <= 1.
 */
int css_score_ce(const void* rows, int rows_dtype, const float* norms, const float* proto_hat, const float* class_cdf,
                 const int32_t* valid_list, const int32_t* hard_list, int32_t* meta,
                 const int32_t* anchor_idx, const int32_t* neg_idx, uint64_t seed, uint64_t offset, uint64_t* step_counter,
                 int N, int C, int D, int Q, int Nn, float temp,
                 float* loss_kq, int32_t* anchor_px, float* grad_anchor, float* loss, void* stream);

/* fp32 rows with the gradient have three implementations of the same arithmetic: the register kernel (one candidate row per 8-lane
 * group in flight), a shared-memory ring fed by 16-byte cp.async copies, and a hybrid in which every other step of a warp arrives
 * through cp.async.bulk + mbarrier while the rest are register loads (default).  Measured on B200 (V321 / C768 scorer alone):
 * 252 / 308 us, 280 / 302 us, 244 / 310 us; over the configs[4] sweep the hybrid shortens the whole step by 2 % on average
 * (DESIGN.md section 4).  css_set_scorer_path(0 | 1 | 2) selects one, -1 returns to the default / the
 * CSS_B200_SCORER=reg|ring|bulk environment variable.  The draws are identical on every path; the sums are taken in a different
 * order (the positive first), so results agree to rounding, not bit for bit. */
int css_set_scorer_path(int path);

/* ---- backward: dense grad_rep ------------------------------------------------------------------------------------------
 * grad_rep [B2,D,h,w] f32 = 0, then += (*grad_out) * grad_anchor[kq] at every anchor pixel (duplicates accumulate).
 * Replaces the autograd index_put / zeros_like chain of loss.py:111-112,128 (SURVEY.md 3.3).
 */
int css_grad_scatter(const float* grad_out, const int32_t* anchor_px, const float* grad_anchor,
                     int n_anchor, int B2, int D, int h, int w, float* grad_rep, void* stream);

/* ---- stage 2 glue fast path (SURVEY.md 8(f)-1) -----------------------------------------------------------------------------
 * Fused weak-threshold mask + one-hot + nearest down-sampling: emits label_all / mask_all at rep resolution directly
 * from the crop-resolution label maps.  Replaces mix_label.py:175-183 (mode 1: label_onehot_2 for the unlabelled half),
 * cross_label.py:178-185 and ori_pseudo.py:171-178 (mode 0).
 *   label_l [B,H,W] i64, label_u [B,H,W] i64, conf_u [B,H,W] f32 -> label_all [2B,C,h,w] f32, mask_all [2B,1,h,w] f32
 */
int css_threshold_glue(const int64_t* label_l, const int64_t* label_u, const float* conf_u, float weak_threshold,
                       int mode, int B, int C, int H, int W, int h, int w,
                       float* label_all, float* mask_all, void* stream);

/* ---- Attention_Threshold_Loss (SURVEY.md 8(f)-3) ------------------------------------------------------------------------------
 * out = mean over {p : CE_p > 0} of w_b * CE(pred[:,p], label_p), w_b = #(conf_b >= threshold) / #(label_b >= 0); label -1 is
 * ignored.  Replaces loss.py:48-64 (forward) and its autograd backward.
 *   pred [B,C,H,W] f32, label [B,H,W] i64, conf [B,H,W] f32
 *   lse f32[B*H*W] (saved for backward), partials f32[B * css_atl_blocks(H,W)], counts i32[3*B], scale f32[B] (saved), loss f32[1]
 */
int css_atl_blocks(int H, int W);
int css_atl_forward(const float* pred, const int64_t* label, const float* conf, float threshold, int B, int C, int H, int W,
                    float* lse, float* partials, int32_t* counts, float* scale, float* loss, void* stream);
int css_atl_backward(const float* grad_out, const float* pred, const int64_t* label, const float* lse, const float* scale,
                     int B, int C, int H, int W, float* grad_pred, void* stream);

/* ---- ProbOhemCrossEntropy2d, the supervised OHEM cross-entropy (DESIGN.md f-5) ---------------------------------------------------
 * valid = target != ignore_index (labels outside [0,C) are treated as ignored); p_t = softmax(pred[:,p])[target_p].
 * When min_kept > 0 and #valid >= min_kept: kept = valid & p_t <= T, T = max(thresh, kth), kth = the min_kept-th smallest p_t
 * of the valid pixels, found by an exact radix select on the device; otherwise kept = valid and T = +inf.  All comparisons are
 * float32.  loss = sum_kept w[y] (lse - x_y) / sum_kept w[y], nan when nothing is kept.  Replaces loss.py:8-46 (forward) and
 * its autograd backward; unlike the reference it makes no host synchronisation and is CUDA-graph capturable.
 *   pred [B,C,H,W] f32, target [B,H,W] i64, weight f32[C] or NULL (= all ones)
 *   workspace of css_ohem_workspace_bytes(B,H,W) bytes (0 for a bad size); the forward writes it and the backward reads it.
 *   After the forward its first B*H*W floats hold p_t per pixel id (NaN on ignored pixels): kept = p_t <= threshold.
 *   loss f32[1], threshold f32[1] = T, counts i32[2] = #valid, #kept
 *   backward: grad_pred [B,C,H,W] f32 = grad_out * w[y] / sum_kept w * (softmax - onehot) on kept pixels, 0 elsewhere
 */
size_t css_ohem_workspace_bytes(int B, int H, int W);
int css_ohem_forward(const float* pred, const int64_t* target, const float* weight, long long ignore_index, float thresh,
                     int min_kept, int B, int C, int H, int W, void* workspace, size_t workspace_bytes, float* loss,
                     float* threshold, int32_t* counts, void* stream);
int css_ohem_backward(const float* grad_out, const float* pred, const int64_t* target, const float* weight, int B, int C, int H,
                      int W, const void* workspace, size_t workspace_bytes, float* grad_pred, void* stream);

/* ---- augmentation hand-off of the label / confidence maps (SURVEY.md 8(f)-2) ------------------------------------------------
 * The maps' trip tensor -> PIL 'L' image -> NEAREST resize -> bottom/right pad (255 / 0) -> crop -> hflip -> tensor, kept on the
 * GPU.  Replaces, for the maps, tensor_to_pil_* + transform_* + the host->device copies of batch_transform_*
 * (dataset_helpers/VOC.py:64-352); the image keeps the PIL path, which is where the host draws `geometry`.
 *   geometry i32[B,5] (device) = resized_h, resized_w, top, left, flip per image
 *   css_aug_index: ymap / xmap i32[B,max_r] = Pillow's NEAREST source index tables for H -> resized_h, W -> resized_w
 *                  (running double sum, replayed sequentially), max_r >= every resized_h / resized_w
 *   css_aug_maps : label_a/label_b [B,H,W] f32 or i64 (label_dtype; values 0..254, 255 or -1 = ignore), conf_a/conf_b [B,H,W] f32,
 *                  any of them nullable -> out_label_* i64[B,ch,cw] (-1 = ignore), out_conf_* f32 = floor(conf * 255) / 255
 */
#define CSS_LABEL_F32 0
#define CSS_LABEL_I64 1
int css_aug_index(const int32_t* geometry, int B, int H, int W, int max_r, int32_t* ymap, int32_t* xmap, void* stream);
int css_aug_maps(const void* label_a, const void* label_b, int label_dtype, const float* conf_a, const float* conf_b,
                 const int32_t* geometry, const int32_t* ymap, const int32_t* xmap, int B, int H, int W, int max_r,
                 int ch, int cw, int64_t* out_label_a, int64_t* out_label_b, float* out_conf_a, float* out_conf_b,
                 void* stream);

/* CutOut / CutMix / ClassMix of one rank's batch in one launch.  Replaces the per-image loop of generate_cut_gather_*
 * (dataset_helpers/VOC.py:354-477): out[i] = keep ? own[i] : partner[(i + 1) % B]; CutOut writes 0 (image, conf) / -1 (label_a)
 * instead of the partner.  keep = pixel outside boxes[i] = (y0, y1, x0, x1)  (cutout, cutmix), or own label_a value v in
 * class_sets[i] (bit v + 1, v in [-1, 62])  (classmix).  The p_* maps are the batch the partners come from: the same
 * pointers on one rank, rank 0's batch otherwise (the reference's partner index always lands in rank 0's slice).
 *   image [B,CH,H,W] f32, label_a (label_b nullable) [B,H,W] i64, conf_a (conf_b nullable) [B,H,W] f32
 */
#define CSS_CUT_CUTOUT 0
#define CSS_CUT_CUTMIX 1
#define CSS_CUT_CLASSMIX 2
int css_cut_mix(const float* image, const int64_t* label_a, const int64_t* label_b, const float* conf_a, const float* conf_b,
                const float* p_image, const int64_t* p_label_a, const int64_t* p_label_b, const float* p_conf_a,
                const float* p_conf_b, const int32_t* boxes, const uint64_t* class_sets, int mode, int B, int CH, int H, int W,
                float* out_image, int64_t* out_label_a, int64_t* out_label_b, float* out_conf_a, float* out_conf_b,
                void* stream);

/* ---- the image's trip through the same augmentation, bit-identical to the Pillow chain ----------------------------------------
 * to_pil_image -> bilinear resize -> reflect pad (bottom / right) -> crop -> ColorJitter -> GaussianBlur -> hflip -> to_tensor +
 * normalize, in Pillow's 8-bit arithmetic (css_b200/aug.py::_augment_image is the reference; oracle/pil_oracle.py the
 * specification).  Replaces, for the image, the device->host copy, the per-image PIL loop and the host->device copy of
 * batch_transform_* (dataset_helpers/VOC.py:126-196, 312-352).
 *   images   f32[B,3,H,W] unnormalised, in [0, 1] (byte = trunc(x * 255))
 *   geometry i32[B,5]     resized_h, resized_w, top, left, flip (as for css_aug_maps)
 *   params   f32[B,CSS_AUG_IMAGE_PARAMS] per image, columns CSS_AUG_P_*: jitter on/off, the four-op order (0 brightness,
 *            1 contrast, 2 saturation, 3 hue), the three blend factors, the hue shift as a byte added to H, blur on/off and
 *            the GaussianBlur radius, which must be <= 4 (integer box radius <= 3)
 *   lut      f32[3,256]  byte -> normalised value per channel (to_tensor + normalize)
 *   workspace of css_aug_image_workspace_bytes(B, ch, cw) bytes -> out f32[B,3,ch,cw]
 */
#define CSS_AUG_IMAGE_PARAMS   11
#define CSS_AUG_P_JITTER       0
#define CSS_AUG_P_ORDER        1    /* [4] */
#define CSS_AUG_P_BRIGHTNESS   5
#define CSS_AUG_P_CONTRAST     6
#define CSS_AUG_P_SATURATION   7
#define CSS_AUG_P_HUE_BYTE     8
#define CSS_AUG_P_BLUR         9
#define CSS_AUG_P_RADIUS       10
size_t css_aug_image_workspace_bytes(int B, int ch, int cw);
int css_aug_image(const float* images, int B, int H, int W, const int32_t* geometry, const float* params, const float* lut,
                  int ch, int cw, void* workspace, size_t workspace_bytes, float* out, void* stream);

/* ---- the exchange step over NVLink peer memory (SURVEY.md 8(e)) -----------------------------------------------------------------
 * Sum of every rank's class_stats [C, D+1] block over the ranks of ONE node, in rank order (bit-identical on all ranks).
 * Replaces concat_all_gather of rep / label (loss.py:77,81; ddp_model.py:241-250) and, on one node, the NCCL all-reduce.
 *   css_comm_alloc  : cudaMalloc + zero a communication buffer for `world` ranks (css_comm_bytes(world) bytes)
 *   css_comm_export : 64-byte CUDA IPC handle of the own buffer (HOST pointer) -- exchanged by the caller (e.g. all_gather_object)
 *   css_comm_open   : map a peer's buffer from its handle; css_comm_close unmaps it; css_comm_free releases the own buffer
 *   css_stats_allreduce: class_stats (device, in place) <- sum over ranks.  peer_buffers: DEVICE array of `world` device
 *                     pointers, entry r = rank r's buffer as mapped in this process (entry `rank` = local_buffer).  One launch,
 *                     no host synchronisation, CUDA-graph capturable; every rank must make the same sequence of calls.
 *   A peer that does not arrive within the timeout (css_comm_set_timeout_ms, process-wide, default 600 000 ms like the NCCL
 *   watchdog) does not hang the GPU and does not poison anything: class_stats is left as this rank's LOCAL statistics and the
 *   event is counted; css_comm_timeouts(buffer) returns that count from pinned host memory without synchronising, so the
 *   caller can poll it every step and raise.
 */
int css_comm_set_timeout_ms(unsigned long long ms);
int css_comm_timeouts(void* buffer);
/* diagnostics (blocking device read, never inside a timed region): out5_host = {completed calls, timeouts, total nanoseconds
 * the calls spent waiting for the slowest peer's block, total ns from kernel entry until the pushed block was fenced, total ns
 * inside the kernel} */
int css_comm_stats(void* buffer, unsigned long long* out5_host);
size_t css_comm_bytes(int world);
int css_comm_alloc(int world, void** buffer);
int css_comm_free(void* buffer);
int css_comm_export(void* buffer, unsigned char* handle64);
int css_comm_open(const unsigned char* handle64, void** peer_buffer);
int css_comm_close(void* peer_buffer);
int css_stats_allreduce(float* class_stats, void* local_buffer, void* const* peer_buffers, int rank, int world, int C, int D,
                        void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CSS_B200_H */
