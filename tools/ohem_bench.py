"""Time of the supervised OHEM loss: oracle/ohem_ref.py (the reference's eager statements) against the fused
css_b200.ProbOhemCrossEntropy2d, forward + backward.

    python tools/ohem_bench.py [--reps 20] [--iters 20] [--out profiles/<name>.json]

For CityScapes (crop 769 x 769, B = 4, C = 19) and VOC (crop 321 x 321, B = 8, C = 21), ignore_index 255, thresh 0.7 and
min_kept = 50000 * B (the CPS CityScapes setting), in both branches of the loss:
  * "t0":     untrained logits (synth.logits_for): most p_t <= 0.7, the threshold is float32(0.7) and no selection runs;
  * "select": confident logits: fewer than min_kept pixels have p_t <= 0.7, the threshold is the min_kept-th smallest p_t.
For each it measures
  * fused device time: `iters` forward + backward calls captured in ONE CUDA graph, `pred` rotated through a pool of
    tensors larger than the 126 MB L2, CUDA events around the replay;
  * device time of both from torch.profiler: the sum of the GPU activities (kernels, memsets, copies) of `reps` calls,
    per call (the reference cannot be captured: it synchronises with the host three times per call);
  * wall time per call, each call ending in a device synchronise, the two implementations alternating in one run.
The results of the two are compared once per case (kept count, threshold, loss).  Algorithmic bytes are the bytes the fused
kernels have to move (pred read forward, pred read on kept pixels and grad written backward, per-pixel maps); the HBM
rate they are set against is a device-to-device copy measured in the same run.  The card's name and power limit are read
in the same run and written beside the numbers."""
import argparse
import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

import css_b200  # noqa: E402
from css_b200 import synth  # noqa: E402
from oracle import ohem_ref  # noqa: E402

CONFIGS = {"C769": dict(B=4, C=19, H=769, W=769), "V321": dict(B=8, C=21, H=321, W=321)}
L2_BYTES = 126 * 2 ** 20


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                           capture_output=True, text=True, timeout=60)
        vals = [v.strip() for v in r.stdout.strip().split(",")]
    except (OSError, subprocess.SubprocessError):
        vals = []
    out = {"torch_device_name": torch.cuda.get_device_name()}
    if len(vals) == 3:
        out.update(name=vals[0], power_limit=vals[1], max_sm_clock=vals[2])
    return out


def hbm_copy_gbps(nbytes=2 ** 30, reps=10):
    src = torch.empty(nbytes, dtype=torch.uint8, device="cuda").fill_(1)
    dst = torch.empty_like(src)
    for _ in range(2):
        dst.copy_(src)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        dst.copy_(src)
    e1.record()
    torch.cuda.synchronize()
    return 2 * nbytes * reps / (e0.elapsed_time(e1) * 1e-3) / 1e9


def inputs(cfg, branch, seed):
    B, C, H, W = (cfg[k] for k in "BCHW")
    g = synth._gen(seed)
    cls = synth.class_map(B, C, H, W, g, ignore_frac=0.05)
    if branch == "t0":
        pred = synth.logits_for(cls, C, g)
    else:
        pred = 6.0 * F.one_hot(cls.clamp_min(0), C).permute(0, 3, 1, 2).float() + torch.randn(B, C, H, W, generator=g)
    return pred.contiguous().cuda(), torch.where(cls < 0, torch.full_like(cls, 255), cls).cuda()


def fwd_bwd(crit, pred, target):
    leaf = pred.detach().requires_grad_(True)
    (g,) = torch.autograd.grad(crit(leaf, target), leaf)
    return g


def graph_us(crit, pool, target, iters):
    for i in range(3):
        fwd_bwd(crit, pool[i % len(pool)], target)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for i in range(iters):
            fwd_bwd(crit, pool[i % len(pool)], target)
    graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    graph.replay()
    e1.record()
    torch.cuda.synchronize()
    del graph
    return e0.elapsed_time(e1) / iters * 1e3


def profiler_us(crit, pool, target, reps):
    """Sum of the GPU activities of `reps` eager calls, per call (us)."""
    from torch.profiler import ProfilerActivity, profile
    fwd_bwd(crit, pool[0], target)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(reps):
            fwd_bwd(crit, pool[i % len(pool)], target)
        torch.cuda.synchronize()
    total = 0.0
    for e in prof.key_averages():
        t = getattr(e, "self_device_time_total", None)
        if t is None:
            t = getattr(e, "self_cuda_time_total", 0.0)
        total += t
    return total / reps


def wall_ms(crit, pred, target):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fwd_bwd(crit, pred, target)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ohem_bench: needs a CUDA device")
    res = {"card": card(), "hbm_copy_GBps": hbm_copy_gbps(), "reps": a.reps, "iters": a.iters, "cases": {}}
    for name, cfg in CONFIGS.items():
        B, C, H, W = (cfg[k] for k in "BCHW")
        kw = dict(ignore_index=255, thresh=0.7, min_kept=50000 * B)
        fused = css_b200.ProbOhemCrossEntropy2d(**kw).cuda()
        ref = ohem_ref.ProbOhemCrossEntropy2d(**kw).cuda()
        for branch in ("t0", "select"):
            pred, target = inputs(cfg, branch, 100 + len(res["cases"]))
            pool_n = max(2, math.ceil(2.5 * L2_BYTES / (pred.numel() * 4)))
            pool = [pred] + [pred + 0 for _ in range(pool_n - 1)]
            # same results, and the branch each one took
            l_f = fused(pred, target)
            l_r = ref(pred, target)
            kept = int(fused.last["num_kept"])
            T = float(fused.last["threshold"])
            assert kept == int(ref.last["valid_mask"].sum()), (name, branch)
            assert (branch == "select") == isinstance(ref.last["threshold"], torch.Tensor), (name, branch)
            assert abs(l_f.item() - l_r.item()) <= 1e-4 * abs(l_r.item()), (name, branch, l_f.item(), l_r.item())
            N, P = B * H * W, B * C * H * W * 4
            sel = 5 * 4 * N if branch == "select" else 0           # three histogram reads of p_t + p_t / nll of the kept-set sum
            alg = P + 8 * N + 12 * N + sel + (kept * C * 4 + P + 8 * N + 8 * N)
            row = {"B": B, "C": C, "crop": [H, W], "min_kept": kw["min_kept"], "threshold": T, "num_kept": kept,
                   "num_valid": int(fused.last["num_valid"]), "loss_fused": l_f.item(), "loss_reference": l_r.item(),
                   "pool": pool_n, "algorithmic_bytes": alg}
            row["fused_graph_device_us"] = graph_us(fused, pool, target, a.iters)
            row["fused_profiler_device_us"] = profiler_us(fused, pool, target, a.reps)
            row["reference_profiler_device_us"] = profiler_us(ref, pool, target, a.reps)
            t_f, t_r = [], []
            for rep in range(a.reps + 1):                          # rep 0 warms both up
                tf = wall_ms(fused, pool[rep % pool_n], target)
                tr = wall_ms(ref, pool[rep % pool_n], target)
                if rep:
                    t_f.append(tf)
                    t_r.append(tr)
            row.update(fused_wall_ms_median=float(np.median(t_f)), reference_wall_ms_median=float(np.median(t_r)),
                       fused_wall_ms=t_f, reference_wall_ms=t_r)
            gbps = alg / (row["fused_graph_device_us"] * 1e-6) / 1e9
            row["fused_GBps"] = gbps
            row["fused_share_of_measured_hbm"] = gbps / res["hbm_copy_GBps"]
            res["cases"][f"{name} {branch}"] = row
            print(f"{name} {branch}: T={T:.6g} kept={kept}  fused {row['fused_graph_device_us']:.1f} us graph / "
                  f"{row['fused_profiler_device_us']:.1f} us profiler / {row['fused_wall_ms_median']:.3f} ms wall;  reference "
                  f"{row['reference_profiler_device_us']:.1f} us profiler / {row['reference_wall_ms_median']:.3f} ms wall;  "
                  f"{gbps:.0f} GB/s = {100 * row['fused_share_of_measured_hbm']:.0f} % of the measured copy rate")
            del pool, pred
            torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
