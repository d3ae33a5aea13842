"""Per-op device timings (CUDA events, inputs rotated through > L2-sized pools so every launch reads cold HBM).
Development aid for kernel tuning:  python tools/kbench.py [--workload voc321_mix] [--iters 50]"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import css_b200  # noqa: E402
from css_b200 import _lib  # noqa: E402
from bench import WORKLOADS, make_inputs  # noqa: E402


def timeit(fn, iters, warm=3):
    """Device time per call: `iters` calls are captured into ONE CUDA graph (no host launch overhead in the number)."""
    for i in range(warm):
        fn(i)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(iters):
            fn(i)
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e3     # us


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="voc321_mix")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--pool", type=int, default=4)
    ap.add_argument("--bf16", action="store_true", help="bf16 representation maps (bf16 pixel-major rows)")
    ap.add_argument("--tc", action="store_true", help="tcgen05 rep pass (css_sim_tc.cu) instead of the FFMA2 one")
    a = ap.parse_args()
    _lib.load().css_set_rep_pass_path(1 if a.tc else 0)
    cfg = WORKLOADS[a.workload]
    B, C, h, w, H, W, Q, Nn, temp = (cfg[k] for k in ("B", "C", "h", "w", "H", "W", "Q", "Nn", "temp"))
    host = make_inputs(cfg, 0)
    dev = torch.device("cuda")
    P = a.pool
    rdt = torch.bfloat16 if a.bf16 else torch.float32
    nhwc = cfg.get("layout") == "nhwc"
    fmt = torch.channels_last if nhwc else torch.contiguous_format
    rep_u = [(host["rep_u"].to(dev).to(rdt) + 0).contiguous(memory_format=fmt) for _ in range(P)]
    rep_all = [(host["rep_all"].to(dev).to(rdt) + 0).contiguous(memory_format=fmt) for _ in range(P)]
    pred_u = host["pred_u"].to(dev)
    label, mask = host["label"].to(dev), host["mask"].to(dev)
    protos = host["prototypes"].to(dev)
    res = {}
    res["sim_map teacher (cos)"] = timeit(lambda i: css_b200.ops.cos_sim_map(rep_u[i % P], protos), a.iters)
    res["sim_map student (softmax)"] = timeit(lambda i: css_b200.ops.proto_softmax_sim(rep_all[i % P], protos, temp), a.iters)
    sim = css_b200.ops.cos_sim_map(rep_u[0], protos)
    res["upsample_label_fuse (mix)"] = timeit(lambda i: css_b200.ops.upsample_label_fuse(sim, pred_u, temp, (H, W), "mix"), a.iters)
    prob = css_b200.ops.proto_softmax_sim(rep_all[0], protos, temp)
    crit = css_b200.Contrast_Loss(num_queries=Q, num_negatives=Nn, temp=temp, strong_threshold=cfg["strong"], seed=1).cuda()
    with torch.no_grad():
        crit(rep_all[0], label, mask, prob, protos.clone())
    ws = crit.last["ws"]
    lib = _lib.load()
    from css_b200._lib import ptr, stream_ptr, check
    N = ws.N
    D = 256
    B2 = 2 * B

    def select(i):
        check(lib.css_select(ptr(label), ptr(mask), ptr(prob), float(cfg["strong"]), B2, C, h, w, ptr(ws.valid_bits), ptr(ws.hard_bits),
                             ptr(ws.tile_counts), ptr(ws.valid_list), ptr(ws.hard_list), ptr(ws.meta), stream_ptr()), "select")

    rows, norms = crit.last["rows"], crit.last["norms"]
    rows_dt = 1 if rows.dtype == torch.bfloat16 else 0

    def stream(i):
        check(lib.css_class_stats(ptr(rows), rows_dt, ptr(ws.valid_bits), ptr(ws.meta), N, C, D, ptr(ws.partials), ptr(ws.touched),
                                  ptr(ws.class_stats), stream_ptr()), "class_stats")

    p2 = protos.clone()

    def ema(i):
        check(lib.css_proto_ema(ptr(p2), ptr(ws.class_stats), ptr(ws.meta), 0.99, 0.01, temp, 0, C, D, ptr(ws.proto_hat),
                                ptr(ws.class_cdf), stream_ptr()), "ema")

    anchor_px = torch.empty(C * Q, device=dev, dtype=torch.int32)
    grad_anchor = torch.empty(C * Q * D, device=dev, dtype=torch.float32)
    loss = torch.empty((), device=dev)

    def score(i, grad=True):
        check(lib.css_score_ce(ptr(rows), rows_dt, ptr(norms), ptr(ws.proto_hat), ptr(ws.class_cdf), ptr(ws.valid_list),
                               ptr(ws.hard_list), ptr(ws.meta), None, None, 7, i, None, N, C, D, Q, Nn, temp, ptr(ws.loss_kq),
                               ptr(anchor_px), ptr(grad_anchor) if grad else None, ptr(loss), stream_ptr()), "score")

    grads = [torch.empty(B2, D, h, w, device=dev) for _ in range(P)]
    one = torch.ones((), device=dev)

    def scatter(i):
        fn = lib.css_grad_scatter_nhwc if nhwc else lib.css_grad_scatter
        check(fn(ptr(one), ptr(anchor_px), ptr(grad_anchor), C * Q, B2, D, h, w, ptr(grads[i % P]), stream_ptr()), "scatter")

    g0 = torch.Generator().manual_seed(0)
    ll = torch.randint(-1, C, (B, H, W), generator=g0).to(dev)
    lu = torch.randint(-1, C, (B, H, W), generator=g0).to(dev)
    cu = torch.rand(B, H, W, generator=g0).to(dev)
    res["threshold_glue K0 (8(f)-1, not in path sum)"] = timeit(
        lambda i: css_b200.ops.threshold_glue(ll, lu, cu, 0.7, C, (h, w), "mix" if cfg["strategy"] == "mix" else "ori"), a.iters)
    atl = css_b200.Attention_Threshold_Loss(0.97).cuda()
    pl = torch.randn(B, C, H, W, generator=g0).to(dev)

    def atl_step(i):
        pp_ = pl.detach().requires_grad_(True)
        (gr,) = torch.autograd.grad(atl(pp_, lu, cu), pp_)

    res["attention_threshold_loss fwd+bwd (8(f)-3, not in path sum)"] = timeit(atl_step, a.iters)
    ohem = css_b200.ProbOhemCrossEntropy2d(ignore_index=-1, thresh=0.7, min_kept=50000 * B).cuda()

    def ohem_step(i):
        pp_ = pl.detach().requires_grad_(True)
        (gr,) = torch.autograd.grad(ohem(pp_, lu), pp_)

    res["prob_ohem_ce fwd+bwd (f-5, not in path sum)"] = timeit(ohem_step, a.iters)
    # 8(f)-2: both trips of the maps through the augmentation + CutMix, at the crop size
    from css_b200 import aug
    import numpy as np
    rng = np.random.default_rng(0)
    geo = np.zeros((B, 5), np.int32)
    for b in range(B):
        r = rng.uniform(0.5, 1.5)
        rh, rw = int(H * r), int(W * r)
        geo[b] = (rh, rw, rng.integers(0, max(rh, H) - H + 1), rng.integers(0, max(rw, W) - W + 1), b & 1)
    geo_d = torch.from_numpy(geo).to(dev)
    fused = torch.where(lu < 0, torch.full_like(lu, 255), lu).float()
    cu2 = torch.rand(B, H, W, generator=g0).to(dev)
    res["aug maps trip: index + 3 maps (8(f)-2, not in path sum)"] = timeit(
        lambda i: aug.transform_maps([fused], [cu, cu2], geo_d, (H, W), max_resized=int(1.5 * max(H, W)) + 1), a.iters)
    x01 = torch.rand(B, 3, H, W, generator=g0).to(dev)
    g_img = torch.from_numpy(np.concatenate([geo[:, :4], np.ones((B, 1), np.int32)], 1)).to(dev)
    p_img = torch.tensor([[1, 3, 1, 0, 2, 1.1, 0.9, 1.2, 17, 1, 1.0]] * B, device=dev)
    res["aug image trip: resize + jitter + blur + flip (not in path sum)"] = timeit(
        lambda i: aug.transform_images(x01, g_img, p_img, (H, W)), a.iters)
    img = torch.randn(B, 3, H, W, generator=g0).to(dev)
    boxes =torch.tensor([[H // 4, 3 * H // 4, W // 8, 7 * W // 8]] * B, dtype=torch.int32, device=dev)
    o_img, o_l, o_c, o_c2 = torch.empty_like(img), torch.empty_like(lu), torch.empty_like(cu), torch.empty_like(cu)

    def cutmix(i):
        check(lib.css_cut_mix(ptr(img), ptr(lu), None, ptr(cu), ptr(cu2), ptr(img), ptr(lu), None, ptr(cu), ptr(cu2), ptr(boxes), None,
                              _lib.CUT_CUTMIX, B, 3, H, W, ptr(o_img), ptr(o_l), None, ptr(o_c), ptr(o_c2), stream_ptr()), "cut_mix")

    res["cut_mix image + 3 maps (8(f)-2, not in path sum)"] = timeit(cutmix, a.iters)
    res["select (3 kernels)"] = timeit(select, a.iters)
    res["class_stats (+reduce)"] = timeit(stream, a.iters)
    res["rep_rows only (ori flow)"] = timeit(lambda i: (css_b200.ops.rep_norms_nhwc if nhwc else css_b200.ops.rep_rows)(rep_all[i % P]), a.iters)
    res["proto_ema (+cdf)"] = timeit(ema, a.iters)
    for path, name in ((0, "register kernel"), (1, "ring 2 stages"), (2, "register/bulk hybrid")):
        if rows_dt == 0:
            lib.css_set_scorer_path(path)
            res[f"score_ce fwd+grad, {name} (not in path sum)"] = timeit(score, a.iters)
    lib.css_set_scorer_path(-1)
    res["score_ce fwd+grad (+reduce)"] = timeit(score, a.iters)
    res["score_ce fwd only"] = timeit(lambda i: score(i, False), a.iters)
    res["grad_scatter (+memset)"] = timeit(scatter, a.iters)
    tot = sum(v for k, v in res.items() if "not in path sum" not in k and k not in ("score_ce fwd only", "rep_rows only (ori flow)"))
    for k, v in res.items():
        print(f"{k:60s} {v:9.1f} us")
    print(f"{'sum (path)':34s} {tot:9.1f} us")
    print(json.dumps({"workload": a.workload, "us": res}))


if __name__ == "__main__":
    main()
