"""Contrast_Loss: drop-in for generalframeworks/loss/loss.py:66-149 running on the CUDA kernels of libcss_b200.

Same constructor, same forward signature, same side effect (prototypes are updated IN PLACE before scoring and the
updated prototype is the positive), same degenerate behaviour (exactly 0 with a dense zero gradient when fewer than
two classes are present).  Differences, all opt-in or invisible to callers:
  * no host synchronisation anywhere (counts, present classes, V live on the device);
  * the 116 MB/rank all_gather of loss.py:77,81 is replaced by one all-reduce of [C, D+1] per-class sums/counts;
  * sampling uses a device Philox stream; `forward(..., _indices=(anchor_idx, neg_idx))` feeds recorded draws
    (e.g. the reference's) for bit-exact verification.
"""
import os

import torch
import torch.distributed as dist
import torch.nn as nn

from . import _lib
from ._lib import check, ptr, stream_ptr
from .ops import _cuda_f32, _proto_scratch, is_channels_last, rep_norms_nhwc, rep_rows, rows_view


class _Workspace:
    """Scratch buffers of one problem shape, owned by the Python side (the library never allocates)."""

    def __init__(self, B2, C, D, h, w, Q, Nn, device):
        lib = _lib.load()
        N = B2 * h * w
        T = lib.css_select_tiles(N)
        with torch.cuda.device(device):
            G = lib.css_class_blocks(N)
        i32 = dict(device=device, dtype=torch.int32)
        f32 = dict(device=device, dtype=torch.float32)
        self.key = (B2, C, D, h, w, Q, Nn, str(device))
        self.N, self.T, self.G = N, T, G
        self.valid_bits = torch.empty(N, **i32)
        self.hard_bits = torch.empty(N, **i32)
        self.tile_counts = torch.empty(2 * C * T, **i32)
        self.valid_list = torch.empty(C * N * 2, **i32)          # {pixel id, bits of its inverse norm} per entry
        self.hard_list = torch.empty(C * N, **i32)
        self.meta = torch.zeros(_lib.META_WORDS, **i32)
        self.partials = torch.empty(G * C * D, **f32)
        self.touched = torch.empty(G, **i32)
        self.class_stats = torch.empty(C, D + 1, **f32)
        self.proto_hat = torch.empty(C * D, **f32)
        self.class_cdf = torch.empty(_lib.CMAX * _lib.CMAX, **f32)
        self.loss_kq = torch.empty(C * Q, **f32)


def allreduce_class_stats(class_stats, group=None):
    """Sum the [C, D+1] per-class (feature sums | counts) block over all ranks: the one exchange step of the path.
    mean_c = sum_ranks(sums_c) / sum_ranks(count_c) equals the reference's mean over all_gather'ed rows
    (loss.py:77-81,102).  No-op on a single process."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(class_stats, op=dist.ReduceOp.SUM, group=group)
    return class_stats


class _ContrastFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, rep, label, mask, prob, prototypes, mod, indices, want_grad, cache):
        lib = _lib.load()
        B2, D, h, w = rep.shape
        C = label.shape[1]
        Q, Nn = mod.num_queries, mod.num_negatives
        dev = rep.device
        ws = mod._workspace(B2, C, D, h, w, dev)
        N = ws.N
        st = stream_ptr()
        check(lib.css_select(ptr(label), ptr(mask), ptr(prob), float(mod.strong_threshold), B2, C, h, w, ptr(ws.valid_bits),
                             ptr(ws.hard_bits), ptr(ws.tile_counts), ptr(ws.meta), st), "css_select")
        how = cache.match(rep) if cache is not None else "miss"
        nhwc = is_channels_last(rep)
        if nhwc:                                # channels-last: the map is its own row table; only the norms are carried
            rows = rows_view(rep)
            if how == "miss":
                norms = rep_norms_nhwc(rep)
            else:
                norms = cache.norms
                if how == "verify":             # equal content at another address (DDP's output clone): checked on the device
                    check(lib.css_rows_refresh_nhwc(ptr(rep), ptr(cache.src), ptr(norms), ptr(_proto_scratch(dev)), ptr(ws.meta), B2, D, h, w, st),
                          "css_rows_refresh_nhwc")
                    cache.rebind(rep)
                    cache.rows = rows
        elif how == "miss":
            rows, norms = rep_rows(rep)
        else:                                   # rows written by the same read that produced `prob`
            rows, norms = cache.rows, cache.norms
        rows_dt = _lib.DTYPE_BF16 if rows.dtype == torch.bfloat16 else _lib.DTYPE_F32
        if how == "verify" and not nhwc:        # equal content at another address (DDP's output clone): checked on the device
            check(lib.css_rows_refresh(ptr(rep), rows_dt, ptr(rows), ptr(norms), ptr(ws.meta), B2, D, h, w, st), "css_rows_refresh")
            cache.rebind(rep)
        # the valid-list entries carry the inverse norms, final only now that the rows are resolved
        check(lib.css_select_lists(ptr(ws.valid_bits), ptr(ws.hard_bits), ptr(ws.tile_counts), ptr(norms), C, N, ptr(ws.valid_list),
                                   ptr(ws.hard_list), st), "css_select_lists")
        check(lib.css_class_stats(ptr(rows), rows_dt, ptr(ws.valid_bits), ptr(ws.meta), N, C, D, ptr(ws.partials), ptr(ws.touched),
                                  ptr(ws.class_stats), st), "css_class_stats")
        mod._exchange(ws.class_stats, C, D, dev)
        # sync_prototypes (extension): every rank applies the SAME update to every globally present class from the summed
        # statistics, so equal prototypes stay equal without a broadcast; default = the reference's rank-local rule
        rule = _lib.UPDATE_GLOBAL if mod.sync_prototypes else _lib.UPDATE_LOCAL
        check(lib.css_proto_ema(ptr(prototypes), ptr(ws.class_stats), ptr(ws.meta), float(mod.alpha), float(1 - mod.alpha),
                                float(mod.temp), rule, C, D, ptr(ws.proto_hat), ptr(ws.class_cdf), st), "css_proto_ema")
        torch.autograd.graph.increment_version(prototypes)     # updated in place through the raw pointer: tell autograd
        anchor_px = torch.empty(C * Q, device=dev, dtype=torch.int32)
        grad_anchor = torch.empty(C * Q * D, device=dev, dtype=torch.float32) if want_grad else None
        loss = torch.empty((), device=dev, dtype=torch.float32)
        a_idx, n_idx = (None, None) if indices is None else indices
        seed, offset = mod._next_draw_key()
        counter = mod._device_counter(dev)
        ev = mod.score_events
        if ev is not None:                       # bench.py times the dominant kernel live, on the launching stream
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        check(lib.css_score_ce(ptr(rows), rows_dt, ptr(norms), ptr(ws.proto_hat), ptr(ws.class_cdf), ptr(ws.valid_list),
                               ptr(ws.hard_list), ptr(ws.meta), ptr(a_idx), ptr(n_idx), seed, offset, ptr(counter), N, C, D, Q, Nn,
                               float(mod.temp), ptr(ws.loss_kq), ptr(anchor_px), ptr(grad_anchor), ptr(loss), st), "css_score_ce")
        if ev is not None:
            e1.record()
            ev.append((e0, e1))
        ctx.shape = (B2, D, h, w)
        ctx.nhwc_stride = tuple(rep.stride()) if nhwc else None
        ctx.rep_dtype = rep.dtype
        ctx.n_anchor = C * Q
        ctx.save_for_backward(anchor_px, grad_anchor)
        mod.last = dict(ws=ws, anchor_px=anchor_px, grad_anchor=grad_anchor, seed=seed, offset=offset, rows=rows, norms=norms,
                        rows_from_cache=how != "miss", rows_cache_mode=how)
        return loss

    @staticmethod
    def backward(ctx, grad_out):
        anchor_px, grad_anchor = ctx.saved_tensors
        if grad_anchor is None:
            raise RuntimeError("css_b200: Contrast_Loss backward without forward-time gradient state")
        B2, D, h, w = ctx.shape
        lib = _lib.load()
        go = grad_out.detach().to(torch.float32).contiguous()
        if ctx.nhwc_stride is not None:         # channels-last map: the gradient keeps the memory format (zero fill + row updates)
            grad_rep = torch.empty_strided(ctx.shape, ctx.nhwc_stride, device=anchor_px.device, dtype=torch.float32)
            with torch.cuda.device(anchor_px.device):
                check(lib.css_grad_scatter_nhwc(ptr(go), ptr(anchor_px), ptr(grad_anchor), ctx.n_anchor, B2, D, h, w, ptr(grad_rep),
                                                stream_ptr()), "css_grad_scatter_nhwc")
            return grad_rep, None, None, None, None, None, None, None, None
        grad_rep = torch.empty(ctx.shape, device=anchor_px.device, dtype=torch.float32)
        with torch.cuda.device(anchor_px.device):
            check(lib.css_grad_scatter(ptr(go), ptr(anchor_px), ptr(grad_anchor), ctx.n_anchor, B2, D, h, w, ptr(grad_rep),
                                       stream_ptr()), "css_grad_scatter")
        if ctx.rep_dtype != torch.float32:
            grad_rep = grad_rep.to(ctx.rep_dtype)
        return grad_rep, None, None, None, None, None, None, None, None


class Contrast_Loss(nn.Module):
    """Same constructor and forward as the reference's Contrast_Loss (loss.py:66-75)."""

    def __init__(self, num_queries, num_negatives, temp=0.5, mean=False, strong_threshold=0.97, alpha=0.99,
                 seed=None, process_group=None, sync_prototypes=False, exchange=None):
        super().__init__()
        self.temp = temp
        self.mean = mean                      # unused by the reference as well (loss.py:70)
        self.num_queries = num_queries
        self.num_negatives = num_negatives
        self.strong_threshold = strong_threshold
        self.alpha = alpha
        self.process_group = process_group
        # extension, default off (the reference lets per-rank prototypes drift): update every globally present class on every rank
        self.sync_prototypes = sync_prototypes
        # how the [C, D+1] class statistics are summed over ranks: "peer" = css_stats_allreduce over NVLink peer memory
        # (one node), "nccl" = dist.all_reduce, "auto" = peer when every rank can map every other rank's buffer, else nccl
        self.exchange = exchange or os.environ.get("CSS_B200_EXCHANGE", "auto")
        if self.exchange not in ("auto", "peer", "nccl"):
            raise ValueError("exchange must be 'auto', 'peer' or 'nccl'")
        self._reducer = None
        self._seed = seed
        self._step = 0
        self._counter = None
        self._ws = {}                         # one workspace per problem shape, never freed: a captured graph may still write to it
        self.last = None
        self.score_events = None              # set to a list to collect (start, end) CUDA events around css_score_ce

    # ---- sampler state: (seed, offset) of the device Philox stream; one offset per forward call -------------------
    def set_sampler(self, seed, step=0):
        self._seed, self._step = int(seed), int(step)
        self._counter = None

    def _device_counter(self, device):
        """Device-resident step counter of the Philox stream: the kernels read it as the draw offset and bump it, so the
        sampler advances without any host involvement (eager calls and CUDA-graph replays alike)."""
        if self._counter is None or self._counter.device != device:
            if torch.cuda.is_current_stream_capturing():
                raise RuntimeError("css_b200: the first Contrast_Loss.forward must run outside CUDA-graph capture (it creates the "
                                   "device-resident sampler counter a captured graph then advances on every replay)")
            self._counter = torch.full((1,), self._step, device=device, dtype=torch.int64)
        return self._counter

    def draw_offset(self):
        """Offset the NEXT forward will draw from (reads the device counter: synchronises; verification only)."""
        return self._step if self._counter is None else int(self._counter.item())

    def _next_draw_key(self):
        if self._seed is None:   # derived from torch's CPU generator so torch.manual_seed() makes runs reproducible
            self._seed = int(torch.randint(0, 2 ** 62, (1,)).item())
            if dist.is_available() and dist.is_initialized():
                self._seed ^= 0x9E3779B97F4A7C15 * (dist.get_rank() + 1) & (2 ** 63 - 1)
        return self._seed & (2 ** 64 - 1), 0

    def _exchange(self, class_stats, C, D, device):
        """The one exchange step of the path (loss.py:77-81,102 in the reference: two all_gathers of whole maps)."""
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(self.process_group) <= 1:
            return class_stats
        if self.exchange != "nccl" and self._reducer is None:
            from .comm import PeerStatsReducer
            self._reducer = PeerStatsReducer(device, self.process_group)       # collective: first forward of every rank
            if not self._reducer.ok and self.exchange == "peer":
                raise RuntimeError("css_b200: exchange='peer' but the ranks cannot map each other's memory (CUDA IPC)")
        if self._reducer is not None and self._reducer.ok:
            return self._reducer.allreduce(class_stats, C, D)
        return allreduce_class_stats(class_stats, self.process_group)

    def exchange_mode(self):
        """'peer', 'nccl' or 'none' (single process / not used yet): what the last forward used."""
        if self._reducer is not None and self._reducer.ok:
            return "peer"
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(self.process_group) > 1:
            return "nccl"
        return "none"

    def _workspace(self, B2, C, D, h, w, device):
        key = (B2, C, D, h, w, self.num_queries, self.num_negatives, str(device))
        ws = self._ws.get(key)
        if ws is None:
            if torch.cuda.is_current_stream_capturing():
                raise RuntimeError("css_b200: run one eager Contrast_Loss.forward of this shape before capturing it in a CUDA graph")
            ws = self._ws[key] = _Workspace(B2, C, D, h, w, self.num_queries, self.num_negatives, device)
        return ws

    def clear_workspaces(self):
        """Drops the per-shape scratch buffers (only when no captured CUDA graph refers to them any more)."""
        self._ws = {}

    def forward(self, rep, label, mask, prob, prototypes, _indices=None):
        """rep [B2,256,h,w], label [B2,C,h,w], mask [B2,1,h,w], prob [B2,C,h,w], prototypes [C,256] (updated in place).
        _indices: optional (anchor_idx int32 [C,Q], neg_idx int32 [C,Q,Nn]) slot-major device tensors of recorded draws."""
        if not rep.is_cuda:
            raise RuntimeError("css_b200: Contrast_Loss needs CUDA tensors (no CPU fallback)")
        if rep.dtype not in (torch.float32, torch.bfloat16):
            raise RuntimeError(f"css_b200: rep must be float32 or bfloat16, got {rep.dtype}")
        if not (prototypes.is_cuda and prototypes.dtype == torch.float32 and prototypes.is_contiguous()):
            raise RuntimeError("css_b200: prototypes must be a contiguous float32 CUDA tensor (it is updated in place)")
        if rep.shape[1] != _lib.D or prototypes.shape != (label.shape[1], _lib.D):
            raise RuntimeError("css_b200: rep must be [B2,256,h,w] and prototypes [C,256]")
        if mask.shape[1] != 1 or label.shape != prob.shape or label.shape[0] != rep.shape[0] or label.shape[2:] != rep.shape[2:]:
            raise RuntimeError("css_b200: label/prob must be [B2,C,h,w] and mask [B2,1,h,w] at rep resolution")
        want_grad = torch.is_grad_enabled() and rep.requires_grad
        rep_c = rep if (rep.is_contiguous() or is_channels_last(rep)) else rep.contiguous()
        label_c, mask_c, prob_c = _cuda_f32(label, "label"), _cuda_f32(mask, "mask"), _cuda_f32(prob, "prob")
        if _indices is not None:
            a, n = _indices
            if not (a.is_cuda and n.is_cuda and a.dtype == torch.int32 and n.dtype == torch.int32):
                raise RuntimeError("css_b200: _indices must be int32 CUDA tensors")
            _indices = (a.contiguous(), n.contiguous())
        cache = getattr(prob, "_css_rows", None)
        with torch.cuda.device(rep.device):
            return _ContrastFn.apply(rep_c, label_c, mask_c, prob_c, prototypes.detach(), self, _indices, want_grad, cache)

    # ---- verification helpers (read device state back: they synchronise, never used on the training path) --------------
    def selection(self):
        """Present classes, counts and the valid / hard pixel-id lists of the last forward, as Python objects."""
        ws = self.last["ws"]
        meta = ws.meta.cpu().numpy()
        V = int(meta[_lib.META_V])
        present = [int(c) for c in meta[_lib.META_CLS_OF_SLOT:_lib.META_CLS_OF_SLOT + V]]
        out = dict(V=V, present=present, num_list=[], n_hard=[], valid_ids=[], hard_ids=[])
        for c in present:
            nv, nh = int(meta[_lib.META_N_VALID + c]), int(meta[_lib.META_N_HARD + c])
            out["num_list"].append(nv)
            out["n_hard"].append(nh)
            out["valid_ids"].append(ws.valid_list[2 * c * ws.N:2 * (c * ws.N + nv):2].cpu().numpy())
            out["hard_ids"].append(ws.hard_list[c * ws.N:c * ws.N + nh].cpu().numpy())
        return out

    def sample_indices(self, seed, offset):
        """Materialise the draws the scorer would make on the fly for (seed, offset) on the last forward's selection."""
        ws = self.last["ws"]
        C = ws.key[1]
        dev = ws.meta.device
        a = torch.empty(C, self.num_queries, device=dev, dtype=torch.int32)
        n = torch.empty(C, self.num_queries, self.num_negatives, device=dev, dtype=torch.int32)
        lib = _lib.load()
        with torch.cuda.device(dev):
            check(lib.css_sample(ptr(ws.meta), ptr(ws.class_cdf), int(seed), int(offset), C, self.num_queries,
                                 self.num_negatives, ptr(a), ptr(n), stream_ptr()), "css_sample")
        return a, n


class _AttentionThresholdFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, label, conf, threshold):
        lib = _lib.load()
        B, C, H, W = pred.shape
        dev = pred.device
        nblk = lib.css_atl_blocks(H, W)
        lse = torch.empty(B * H * W, device=dev, dtype=torch.float32)
        partials = torch.empty(B * nblk, device=dev, dtype=torch.float32)
        counts = torch.empty(3 * B, device=dev, dtype=torch.int32)
        scale = torch.empty(B, device=dev, dtype=torch.float32)
        loss = torch.empty((), device=dev, dtype=torch.float32)
        check(lib.css_atl_forward(ptr(pred), ptr(label), ptr(conf), float(threshold), B, C, H, W, ptr(lse), ptr(partials), ptr(counts),
                                  ptr(scale), ptr(loss), stream_ptr()), "css_atl_forward")
        ctx.save_for_backward(pred, label, lse, scale)
        return loss

    @staticmethod
    def backward(ctx, grad_out):
        pred, label, lse, scale = ctx.saved_tensors
        lib = _lib.load()
        B, C, H, W = pred.shape
        grad_pred = torch.empty_like(pred)
        go = grad_out.detach().to(torch.float32).contiguous()
        with torch.cuda.device(pred.device):
            check(lib.css_atl_backward(ptr(go), ptr(pred), ptr(label), ptr(lse), ptr(scale), B, C, H, W, ptr(grad_pred), stream_ptr()),
                  "css_atl_backward")
        return grad_pred, None, None, None


class Attention_Threshold_Loss(nn.Module):
    """Drop-in for generalframeworks/loss/loss.py:48-64 (same constructor and forward), SURVEY.md 8(f)-3: one fused forward
    pass over the logits (+ one backward pass) instead of ~6 passes over [B,C,H,W] tensors and a masked_select."""

    def __init__(self, strong_threshold):
        super().__init__()
        self.strong_threshold = strong_threshold

    def forward(self, pred: torch.Tensor, pseudo_label: torch.Tensor, logits: torch.Tensor):
        if not (pred.is_cuda and pseudo_label.is_cuda and logits.is_cuda):
            raise RuntimeError("css_b200: Attention_Threshold_Loss needs CUDA tensors (no CPU fallback)")
        if pred.dtype != torch.float32:
            raise RuntimeError(f"css_b200: pred must be float32, got {pred.dtype}")
        if pred.dim() != 4 or pseudo_label.shape != (pred.shape[0],) + tuple(pred.shape[2:]) or logits.shape != pseudo_label.shape:
            raise RuntimeError("css_b200: pred must be [B,C,H,W], pseudo_label and logits [B,H,W]")
        pred_c = pred if pred.is_contiguous() else pred.contiguous()
        with torch.cuda.device(pred.device):
            return _AttentionThresholdFn.apply(pred_c, pseudo_label.long().contiguous(), logits.float().contiguous(),
                                               self.strong_threshold)


# the 19 CityScapes class weights of the reference (loss.py:8-46, use_weight=True)
CITYSCAPES_CLASS_WEIGHTS = (0.8373, 0.918, 0.866, 1.0345, 1.0166, 0.9969, 0.9754, 1.0489, 0.8786, 1.0023,
                            0.9539, 0.9843, 1.1116, 0.9037, 1.0865, 1.0955, 1.0865, 1.1529, 1.0507)
_INT32_MAX = 2 ** 31 - 1


class _OhemFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, target, weight, ignore_index, thresh, min_kept, ws, threshold, counts):
        lib = _lib.load()
        B, C, H, W = pred.shape
        loss = torch.empty((), device=pred.device, dtype=torch.float32)
        check(lib.css_ohem_forward(ptr(pred), ptr(target), ptr(weight), int(ignore_index), float(thresh), int(min_kept), B, C, H, W,
                                   ptr(ws), ws.numel(), ptr(loss), ptr(threshold), ptr(counts), stream_ptr()), "css_ohem_forward")
        ctx.save_for_backward(pred, target, weight, ws)
        return loss

    @staticmethod
    def backward(ctx, grad_out):
        pred, target, weight, ws = ctx.saved_tensors
        lib = _lib.load()
        B, C, H, W = pred.shape
        grad_pred = torch.empty_like(pred)
        go = grad_out.detach().to(torch.float32).contiguous()
        with torch.cuda.device(pred.device):
            check(lib.css_ohem_backward(ptr(go), ptr(pred), ptr(target), ptr(weight), B, C, H, W, ptr(ws), ws.numel(), ptr(grad_pred),
                                        stream_ptr()), "css_ohem_backward")
        return grad_pred, None, None, None, None, None, None, None, None


class ProbOhemCrossEntropy2d(nn.Module):
    """Drop-in for generalframeworks/loss/loss.py:8-46 (same constructor and forward): the supervised OHEM cross-entropy.

    Pixels whose label is not `ignore_index` are valid.  With p_t the softmax probability of a pixel's own label, the loss is
    the (class-weighted) mean cross-entropy over the valid pixels with p_t <= T, T = max(float32(thresh), the min_kept-th
    smallest p_t); over all valid pixels when min_kept <= 0 or fewer than min_kept pixels are valid; nan when none is valid.
    One fused pass over `pred` forward (plus, only when the threshold is not float32(thresh), an exact radix select over the
    per-pixel p_t) and one backward, all on the device with no host synchronisation: it can be captured in a CUDA graph.

    Differences from the reference:
      * the reference's `logger.info('Labels: ...')` when min_kept > #valid is dropped (it needs the count on the host);
      * labels outside [0, C) other than ignore_index are treated as ignored (torch would raise a device-side assert);
      * only reduction='mean' exists (what the scripts use); `down_ratio` is accepted and unused, as in the reference;
      * `pred` must be a float32 CUDA tensor (no CPU fallback); the caller's `target` is never modified.
    After each forward, `self.last` holds device tensors `num_valid`, `threshold` (the T used, +inf when OHEM did not apply),
    `num_kept` and `p_t` ([B,H,W], nan on ignored pixels; kept = p_t <= threshold), for verification; nothing reads them on
    the training path.
    """

    def __init__(self, ignore_index, reduction='mean', thresh=0.6, min_kept=256, down_ratio=1, use_weight=False):
        super().__init__()
        if reduction != 'mean':
            raise ValueError(f"css_b200: ProbOhemCrossEntropy2d supports reduction='mean' only, got {reduction!r}")
        self.ignore_index = ignore_index
        self.reduction = reduction
        self.thresh = float(thresh)
        self.min_kept = int(min_kept)
        self.down_ratio = down_ratio
        self.use_weight = use_weight
        self.register_buffer("weight", torch.tensor(CITYSCAPES_CLASS_WEIGHTS, dtype=torch.float32) if use_weight else None)
        self.last = None

    def forward(self, pred, target):
        if not (pred.is_cuda and target.is_cuda):
            raise RuntimeError("css_b200: ProbOhemCrossEntropy2d needs CUDA tensors (no CPU fallback)")
        if pred.dtype != torch.float32:
            raise RuntimeError(f"css_b200: pred must be float32, got {pred.dtype}")
        if pred.dim() != 4 or target.numel() != pred.shape[0] * pred.shape[2] * pred.shape[3]:
            raise RuntimeError("css_b200: pred must be [B,C,H,W] and target hold B*H*W labels")
        if target.dtype.is_floating_point or target.dtype == torch.bool:
            raise RuntimeError(f"css_b200: target must hold integer labels, got {target.dtype}")
        weight = None
        if self.weight is not None:
            if self.weight.numel() != pred.shape[1]:
                raise RuntimeError(f"css_b200: use_weight=True has {self.weight.numel()} class weights, pred has {pred.shape[1]} classes")
            weight = self.weight if self.weight.device == pred.device else self.weight.to(pred.device)
        pred_c = pred.contiguous()                           # channels-last or strided pred: one copy into NCHW
        target_c = target.reshape(-1).to(torch.int64).contiguous()
        B, _, H, W = pred.shape
        dev = pred.device
        # per-call scratch (the forward writes it, the backward reads lse / p_t / T from it); p_t per pixel comes first
        ws = torch.empty(_lib.load().css_ohem_workspace_bytes(B, H, W), device=dev, dtype=torch.uint8)
        threshold = torch.empty((), device=dev, dtype=torch.float32)
        counts = torch.empty(2, device=dev, dtype=torch.int32)
        min_kept = min(self.min_kept, _INT32_MAX)            # beyond any int32 pixel count: OHEM never applies either way
        with torch.cuda.device(dev):
            loss = _OhemFn.apply(pred_c, target_c, weight, int(self.ignore_index), self.thresh, min_kept, ws, threshold, counts)
        self.last = dict(num_valid=counts[0], threshold=threshold, num_kept=counts[1],
                         p_t=ws[:4 * B * H * W].view(torch.float32).view(B, H, W))
        return loss
