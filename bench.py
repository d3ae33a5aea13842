#!/usr/bin/env python
"""bench.py -- contrastive-path pixels/sec of the CSS representation-space hot path on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload voc321_mix|...] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

One "step" = one pass of the four-stage path over one synthetic batch per GPU (SURVEY.md 8(d) `t_path`):
    teacher  : cosine map of rep_u vs prototypes -> fused bilinear-up + softmax + max (rep & logit space) + mix fusion
    student  : prob_all = softmax(cos(rep_all, prototypes)/temp)
    loss fwd : selection/compaction, one streaming read of rep_all (class sums + pixel-major normalised copy),
               [all-reduce of per-class sums|counts when N > 1], prototype EMA, sampling + scoring + CE
    loss bwd : dense grad_rep (zero fill + anchor scatter)
The DeepLabv3+ backbone, data loading and augmentation are outside the path (BASELINE.json north_star).
`pixels` = rep-resolution pixels of rep_all per step = 2B*h*w per GPU.  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[1]/[2] shape: VOC, 321x321 crops, B=8 per GPU, rep 81x81, 21 classes
    "voc321_mix": dict(B=8, C=21, h=81, w=81, H=321, W=321, Q=256, Nn=512, temp=0.5, strong=0.8, weak=0.7, strategy="mix"),
    "voc321_ori": dict(B=8, C=21, h=81, w=81, H=321, W=321, Q=256, Nn=512, temp=0.5, strong=0.97, weak=0.7, strategy="ori"),
    # BASELINE.json configs[3]: CityScapes, 768x768 crops, deep-stem rep 193x193, 19 classes, B=4 per GPU (YAML)
    "city768_cross": dict(B=4, C=19, h=193, w=193, H=769, W=769, Q=256, Nn=512, temp=0.5, strong=0.8, weak=0.7, strategy="cross"),
    # extension (VERDICT r1 item 9): the same VOC step on CHANNELS-LAST representation maps (model.to(memory_format=torch.channels_last)):
    # the map is its own pixel-major row table, TMA + tcgen05 similarity pass, no transposing copy.  Not a BASELINE configuration.
    "voc321_mix_nhwc": dict(B=8, C=21, h=81, w=81, H=321, W=321, Q=256, Nn=512, temp=0.5, strong=0.8, weak=0.7, strategy="mix", layout="nhwc"),
    "city768_cross_nhwc": dict(B=4, C=19, h=193, w=193, H=769, W=769, Q=256, Nn=512, temp=0.5, strong=0.8, weak=0.7, strategy="cross", layout="nhwc"),
    # BASELINE.json configs[0]: the reference's own CPU-runnable case (loss only)
    "voc81_b1_loss": dict(B=1, C=21, h=81, w=81, H=321, W=321, Q=256, Nn=512, temp=0.5, strong=0.97, weak=0.7, strategy="ori"),
}
D = 256
METRIC = "contrastive_path_pixels_per_sec"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="voc321_mix", choices=sorted(WORKLOADS))
    ap.add_argument("--e2e-steps", type=int, default=30)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--cpu-budget-s", type=float, default=float(os.environ.get("CSS_CPU_BUDGET_S", 240)))
    ap.add_argument("--no-gpu-eager-reference", action="store_true", help="skip the reference-on-this-GPU context line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (rank 0) as DIR/<name>.npy in float32; "
                         f"an array of more than {DUMP_MAX_ELEMS} elements is reduced to a fixed seeded sample of its flat indices")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


DUMP_MAX_ELEMS = 1 << 21      # 8 MB per array: at most 4 maps + grad_rep + prob + loss + prototypes stay under 64 MB
DUMP_SEED = 20240607


def dump_outputs(outputs, out_dir):
    """Copies the named device tensors to DIR/<name>.npy as float32.  A larger array becomes the elements at
    DUMP_MAX_ELEMS flat (logical, row-major) indices drawn without replacement from a generator seeded with DUMP_SEED and
    sorted, so the sample depends only on the array's size and two builds write comparable files."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        t = t.detach()
        if t.numel() > DUMP_MAX_ELEMS:
            idx = np.sort(np.random.default_rng(DUMP_SEED).choice(t.numel(), DUMP_MAX_ELEMS, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def make_inputs(cfg, rank):
    """Synthetic tensors of the workload (CPU); seed 3407 (+rank), SURVEY.md 8(d)."""
    import torch
    from css_b200 import synth
    B, C, h, w = cfg["B"], cfg["C"], cfg["h"], cfg["w"]
    seed = 3407 + 1000 * rank
    t = synth.teacher_batch(B, C, h, w, seed=seed)
    s = synth.student_batch(2 * B, C, h, w, seed=seed + 1, strategy=cfg["strategy"])
    protos = 0.5 * s["centers"] + 0.3 * synth.warm_prototypes(C, seed=3407, zero_rows=(C - 1,))
    return dict(rep_u=t["rep_u"], pred_u=t["pred_u"], rep_all=s["rep"], label=s["label"], mask=s["mask"],
                prob_ori=torch.softmax(s["logits"], dim=1), prototypes=protos)


def path_bytes(cfg, v_eff):
    """Algorithmic bytes per step per GPU (SURVEY.md 8(d)); fp32 everywhere (s = 4)."""
    B, C, h, w, H, W, Q, Nn = (cfg[k] for k in ("B", "C", "h", "w", "H", "W", "Q", "Nn"))
    Nu, N, NU = B * h * w, 2 * B * h * w, B * H * W
    out_b = {"mix": 28, "cross": 24, "ori": 12}[cfg["strategy"]]
    if cfg["strategy"] == "ori":
        stream = Nu * 4 * C + NU * out_b + N * (2 * D * 4 + 2 * 4 * C + 4)
    else:
        stream = Nu * (D * 4 + 4 * C) + NU * out_b + N * (2 * D * 4 + 2 * 4 * C + 4)
    gather = v_eff * Q * (Nn + 1) * D * 4
    return stream, gather


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index, period=0.01):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.sm, self.reasons, self.sm_max = [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            hnd = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.sm_max = nv.nvmlDeviceGetMaxClockInfo(hnd, nv.NVML_CLOCK_SM)
            names = {getattr(nv, n): n[len("nvmlClocksEventReason"):] for n in dir(nv) if n.startswith("nvmlClocksEventReason")
                     and isinstance(getattr(nv, n), int)}
            if not names:
                names = {getattr(nv, n): n[len("nvmlClocksThrottleReason"):] for n in dir(nv)
                         if n.startswith("nvmlClocksThrottleReason") and isinstance(getattr(nv, n), int)}
            self.ok = True
            while not self._stop_evt.is_set():
                self.sm.append(nv.nvmlDeviceGetClockInfo(hnd, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(hnd)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(hnd)
                for bit, name in names.items():
                    if bit and (r & bit) and name not in ("None", "GpuIdle", "All"):
                        self.reasons.add(name)
                time.sleep(self.period)
        except Exception as e:  # NVML missing: report that no clocks were sampled
            self.err = repr(e)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": ["unsampled"]}
        s = sorted(self.sm)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons), "samples": len(s)}


def physical_gpu_index(local_rank):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


def pin_to_gpu_numa_node(index):
    """Moves this process onto the CPUs NVML reports as local to GPU `index` (so that the pinned staging buffers allocated next
    are first-touched on that NUMA node) and returns what it did; the previous affinity is restored by unpin_cpu()."""
    info = {"gpu": index, "cpus_before": len(os.sched_getaffinity(0)), "pinned": False}
    try:
        import pynvml as nv
        nv.nvmlInit()
        hnd = nv.nvmlDeviceGetHandleByIndex(index)
        words = nv.nvmlDeviceGetCpuAffinity(hnd, (os.cpu_count() + 63) // 64)
        cpus = {64 * i + b for i, wd in enumerate(words) for b in range(64) if (int(wd) >> b) & 1}
        try:
            info["numa_node"] = int(nv.nvmlDeviceGetNumaNodeId(hnd))
        except Exception:
            info["numa_node"] = None
        usable = cpus & os.sched_getaffinity(0)
        info["gpu_local_cpus"] = len(cpus)
        if usable and usable != os.sched_getaffinity(0):
            _AFFINITY_STACK.append(os.sched_getaffinity(0))
            os.sched_setaffinity(0, usable)
            info["pinned"] = True
    except Exception as e:
        info["error"] = repr(e)
    return info


_AFFINITY_STACK = []


def unpin_cpu():
    if _AFFINITY_STACK:
        os.sched_setaffinity(0, _AFFINITY_STACK.pop())


_PROBE = None


def run_probe(rows, n_warps, n_per_warp):
    """Ceilings of the access patterns, measured live (tools/dev/css_probe.cu): {'l2_gather_gbs', 'copy_gbs'} or None."""
    global _PROBE
    import ctypes
    import torch
    path = os.path.join(ROOT, "tools", "dev", "libcss_probe.so")
    if not os.path.exists(path) or rows.dtype != torch.float32:
        return None
    try:
        if _PROBE is None:
            _PROBE = ctypes.CDLL(path)
            _PROBE.css_probe_gather_gbs.restype = ctypes.c_double
            _PROBE.css_probe_gather_gbs.argtypes = [ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
            _PROBE.css_probe_copy_gbs.restype = ctypes.c_double
            _PROBE.css_probe_copy_gbs.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int]
        torch.cuda.synchronize()
        scratch = torch.zeros(4, device=rows.device)
        n_per_warp = max(16, (n_per_warp // 16) * 16)
        g = _PROBE.css_probe_gather_gbs(rows.data_ptr(), rows.shape[0], int(n_warps), int(n_per_warp), 3, scratch.data_ptr())
        a = torch.empty(256 << 20, device=rows.device, dtype=torch.uint8)
        b = torch.empty_like(a)
        c = _PROBE.css_probe_copy_gbs(b.data_ptr(), a.data_ptr(), a.numel(), 5)
        torch.cuda.synchronize()
        return {"l2_gather_gbs": g if g > 0 else None, "copy_gbs": c if c > 0 else None}
    except Exception as e:
        sys.stderr.write(f"bench: probe failed ({e!r})\n")
        return None


# ------------------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline on the host cores: the UNMODIFIED reference (oracle/ref_bench.py, `kind: "reference"`) when its
# tree is on this box (baseline/_ref, CSS_REFERENCE_ROOT or /root/reference), otherwise the oracle port (numpy restatement,
# `kind: "port"`).  The only place bench.py executes anything under oracle/.
# ------------------------------------------------------------------------------------------------------------------
_PROB_CACHE = {}


def run_cpu(cfg, steps, warmup, budget_s, rank_inputs):
    if os.environ.get("CSS_BENCH_CPU_KIND", "auto") != "port":
        try:
            from oracle import ref_bench
            if ref_bench.available():
                return ref_bench.run_cpu(cfg, rank_inputs, steps, warmup, budget_s)
        except Exception as e:      # a broken copy of the reference must not take the bench down: say so and use the port
            sys.stderr.write(f"bench: reference CPU arm unavailable ({e!r}); timing the oracle port instead\n")
    return run_cpu_port(cfg, steps, warmup, budget_s, rank_inputs)


def _cached_prob(inp, protos, temp, n_sub):
    """prob of the images beyond the timed sub-batch (needed as an input of the loss, computed once, outside the timing;
    prototypes drift slowly under the EMA, which does not change the cost of anything that is timed)."""
    from oracle import css_oracle as O
    key = (id(inp["rep_all"]), n_sub)
    if key not in _PROB_CACHE:
        _PROB_CACHE[key] = O.proto_softmax_sim(inp["rep_all"][n_sub:], protos, temp)
    return _PROB_CACHE[key]


def cpu_path_step(cfg, inp, protos, b_sub, q_sub):
    """One pass of the path on CPU with the oracle port, on a bounded sample: stage 1/2 on `b_sub` of B teacher images,
    loss fwd+bwd with `q_sub` of Q queries per class.  Returns (t_stage12, t_loss)."""
    import numpy as np
    from oracle import css_oracle as O
    C, H, W, temp = cfg["C"], cfg["H"], cfg["W"], cfg["temp"]
    t0 = time.perf_counter()
    if cfg["strategy"] == "ori":
        O.cls_pseudo_label(inp["pred_u"][:b_sub], (H, W))
        prob = inp["prob_ori"]
    else:
        _, label_rep, _ = O.rep_pseudo_label(inp["rep_u"][:b_sub], protos, temp, (H, W))
        _, label_cls = O.cls_pseudo_label(inp["pred_u"][:b_sub], (H, W))
        if cfg["strategy"] == "mix":
            O.mix_fuse(label_cls, label_rep, C)
        t_half = time.perf_counter()
        n_sub = 2 * b_sub                                              # student prob_all is linear in pixels: time it on a
        prob_sub = O.proto_softmax_sim(inp["rep_all"][:n_sub], protos, temp)   # sub-batch and scale, compute the rest untimed
        t_prob = (time.perf_counter() - t_half) * (inp["rep_all"].shape[0] / n_sub)
        prob = prob_sub if n_sub == inp["rep_all"].shape[0] else np.concatenate(
            [prob_sub, _cached_prob(inp, protos, temp, n_sub)])
    t1 = time.perf_counter()
    O.contrast_loss(inp["rep_all"], inp["label"], inp["mask"], prob, protos, num_queries=q_sub, num_negatives=cfg["Nn"],
                    temp=temp, strong_threshold=cfg["strong"], alpha=0.99, want_grad=True)
    t2 = time.perf_counter()
    if cfg["strategy"] == "ori":
        return (t1 - t0), 0.0, (t2 - t1)
    return t_half - t0, t_prob, (t2 - t1)


def run_cpu_port(cfg, steps, warmup, budget_s, rank_inputs):
    """Times the oracle port for `steps` steps after `warmup`, inside `budget_s` seconds by shrinking the per-step
    sample (teacher images, queries per class) and scaling the time back to the full step."""
    import numpy as np
    import torch
    inp = {k: v.numpy() for k, v in rank_inputs.items()}
    protos = inp["prototypes"].copy()
    cores = len(os.sched_getaffinity(0))
    torch.set_num_threads(cores)
    B, Q = cfg["B"], cfg["Q"]
    N = 2 * B * cfg["h"] * cfg["w"]
    # calibrate: the loss time is affine in the queries per class, t(q) = F + q*c (per-class fixed work + per-query work), so two
    # small runs give F and c and a step timed with q_sub queries is scaled as F + (t - F) * Q / q_sub (not t * Q / q_sub,
    # which would bill the reference Q/q_sub times for its fixed work); stage 1/2 and the student prob are linear in images
    np.random.seed(0)
    torch.manual_seed(0)
    b_sub = 1
    cpu_path_step(cfg, inp, protos.copy(), b_sub, 2)                       # warm numpy / BLAS threads, page in the inputs
    a, p, l8 = cpu_path_step(cfg, inp, protos.copy(), b_sub, 8)
    _, _, l32 = cpu_path_step(cfg, inp, protos.copy(), b_sub, 32)
    c_q = max((l32 - l8) / 24.0, 1e-6)
    fixed = max(l8 - 8 * c_q, 0.0)
    total_steps = steps + warmup
    per_step_budget = max(budget_s / max(total_steps, 1), 0.05)
    q_sub = 8
    while b_sub < B and (a + p) * 2 + fixed + q_sub * c_q <= 0.6 * per_step_budget:
        a, p, b_sub = a * 2, p, b_sub * 2            # p is already reported scaled to the full batch; its cost grows with b_sub
    while q_sub < Q and a + fixed + (2 * q_sub) * c_q <= per_step_budget:
        q_sub *= 2
    b_sub, q_sub = min(b_sub, B), min(q_sub, Q)
    ts = []
    for i in range(total_steps):
        a, p, l = cpu_path_step(cfg, inp, protos, b_sub, q_sub)
        if i >= warmup:
            l_full = l if q_sub == Q else fixed + max(l - fixed, 0.0) * (Q / q_sub)
            ts.append(a * (B / b_sub) + p + l_full)       # p is already scaled to the full batch
    t_step = sum(ts) / max(len(ts), 1)
    sample = (f"oracle port (numpy); each step = stage 1/2 on {b_sub} of {B} teacher images + student prob on {2 * b_sub} of "
              f"{2 * B} images + loss fwd+bwd on the full batch with {q_sub} of {Q} queries/class (Nn={cfg['Nn']}); stage 1/2 and prob "
              f"times are scaled by B/{b_sub}; the loss time t is scaled as F + (t - F)*Q/{q_sub} with the calibrated per-step fixed "
              f"cost F = {fixed:.2f} s")
    return dict(value=N / t_step, t_step=t_step, cores=cores, sample=sample, kind="port")


def reference_arm(args, cfg):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return 0
    inp = make_inputs(cfg, 0)
    r = run_cpu(cfg, args.steps, args.warmup, args.cpu_budget_s, inp)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": "pixels/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["t_step"] * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, cfg),
        "cpu_baseline": {"value": r["value"], "unit": "pixels/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
        "e2e": {"value": r["value"], "unit": "pixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


def workload_config(args, cfg):
    return {"workload": f"{args.workload}: {cfg['strategy']} strategy, B={cfg['B']}/GPU, C={cfg['C']}, rep {cfg['h']}x{cfg['w']}x{D} "
                        f"-> crop {cfg['H']}x{cfg['W']}, Q={cfg['Q']}, Nn={cfg['Nn']}, temp={cfg['temp']}, strong={cfg['strong']} "
                        + ("(channels-last representation maps: extension, not a BASELINE configuration)" if cfg.get("layout") == "nhwc" else
                           "(BASELINE configs[1] shape; four-stage path incl. rep-space label + fusion of configs[2])"),
            "pixels_per_step_per_gpu": 2 * cfg["B"] * cfg["h"] * cfg["w"],
            "parallelism": f"batch-sharded x{args.gpus}, one sum of the [C,D+1] class sums|counts block per step",
            "l2": "no explicit flush: per-step working set (rep_u + rep_all + pixel-major copy + grad_rep ~ 400 MB) exceeds the 126 MB L2"}


# ------------------------------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def quiet_stdout():
    """Everything written to fd 1 from here on (NCCL's version banner, library chatter) goes to stderr; the JSON line is
    written to the saved descriptor by emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def time_in_graph(fn, iters=20, warm=3):
    """Average device time (ms) of one call of `fn`: `iters` calls captured into ONE CUDA graph and replayed between two CUDA
    events on the launching stream (no host launch gaps inside the number)."""
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(iters):
            fn()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    args = parse()
    cfg = WORKLOADS[args.workload]
    quiet_stdout()
    if args.impl == "reference":
        return reference_arm(args, cfg)

    import torch
    import torch.distributed as dist
    import css_b200
    from css_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", 1))
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (there is no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()

    B, C, h, w, H, W, Q, Nn = (cfg[k] for k in ("B", "C", "h", "w", "H", "W", "Q", "Nn"))
    temp, strategy = cfg["temp"], cfg["strategy"]
    N = 2 * B * h * w
    host = make_inputs(cfg, rank)
    if cfg.get("layout") == "nhwc":              # what a channels_last network hands over: same values, [pixel][channel] memory
        for k in ("rep_u", "rep_all"):
            host[k] = host[k].contiguous(memory_format=torch.channels_last)
    gpu = {k: v.to(dev) for k, v in host.items()}
    protos = gpu["prototypes"].clone()
    crit = css_b200.Contrast_Loss(num_queries=Q, num_negatives=Nn, temp=temp, strong_threshold=cfg["strong"], alpha=0.99,
                                  seed=3407 + rank).to(dev)

    def step(t, rep_for_loss=None):
        """one pass of the path on device-resident tensors `t`; returns (loss, grad_rep, {name: map the augmentation receives},
        prob_all or None where prob is an input).
        rep_for_loss: what DistributedDataParallel(find_unused_parameters=True) hands the loss instead of rep_all (a clone)."""
        if strategy == "ori":
            conf, lab = css_b200.ops.cls_pseudo_label(t["pred_u"], (H, W))
            prob, prob_out = t["prob_ori"], None
            maps = {"label_cls": lab, "conf_cls": conf}
        else:
            o = css_b200.ops.pseudo_labels(t["rep_u"], t["pred_u"], protos, temp, (H, W), fuse="mix" if strategy == "mix" else "none")
            prob = prob_out = css_b200.ops.proto_softmax_sim(t["rep_all"], protos, temp)
            names = ("fused", "conf_cls", "conf_rep") if strategy == "mix" else ("label_cls", "label_rep", "conf_cls", "conf_rep")
            maps = {k: o[k] for k in names}
        rep = (t["rep_all"] if rep_for_loss is None else rep_for_loss).detach().requires_grad_(True)
        loss = crit(rep, t["label"], t["mask"], prob, protos)
        (grad,) = torch.autograd.grad(loss, rep)
        return loss, grad, maps, prob_out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up ------------------------------------------------------------------------------------------------
    for _ in range(max(args.warmup, 3)):
        loss, grad, _, _ = step(gpu)
    barrier()
    meta = crit.last["ws"].meta.cpu().numpy()
    V = int(meta[_lib.META_V])
    v_eff = sum(1 for k in range(V) if meta[_lib.META_N_HARD + meta[_lib.META_CLS_OF_SLOT + k]] > 0) if V > 1 else 0
    loss_value = float(loss.item())

    # ---- the one exchange step, checked on the real GPUs (outside every timed region): peer-memory kernel == dist.all_reduce ----
    exchange_check = None
    if world > 1:
        torch.manual_seed(1000 + rank)
        blk = torch.randn(C, D + 1, device=dev)
        ref_sum = blk.clone()
        dist.all_reduce(ref_sum)                                     # NCCL
        mine = blk.clone()
        crit._exchange(mine, C, D, dev)                              # what Contrast_Loss.forward calls
        gathered = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(gathered, mine)
        exact = torch.zeros(C, D + 1, device=dev, dtype=torch.float64)
        blocks = [torch.empty_like(blk) for _ in range(world)]
        dist.all_gather(blocks, blk)
        for b_ in blocks:
            exact += b_.double()
        exchange_check = {"mode": crit.exchange_mode(),
                          "max_abs_diff_vs_nccl_all_reduce": float((mine - ref_sum).abs().max().item()),
                          "max_abs_diff_vs_fp64_sum": float((mine.double() - exact).abs().max().item()),
                          "bit_identical_on_all_ranks": bool(all(torch.equal(g_, gathered[0]) for g_ in gathered)),
                          "block": [C, D + 1], "ranks": world}
        barrier()

    # ---- one step captured as a CUDA graph (the library is capturable: no host sync, caller-owned buffers) -------------
    def capture(tensors, rep_for_loss=None):
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                step(tensors, rep_for_loss)
        torch.cuda.current_stream().wait_stream(side)
        with torch.cuda.graph(g):
            out = step(tensors, rep_for_loss)
        return g, out

    use_graph = not args.no_graph
    graph = None
    if use_graph:
        try:
            graph, graph_out = capture(gpu)
            graph.replay()
            barrier()
        except Exception as e:   # e.g. a collective that cannot be captured on this stack: fall back to eager launches
            sys.stderr.write(f"bench: CUDA graph capture failed ({e!r}); timing eager launches\n")
            graph, use_graph = None, False

    def run_step():
        if graph is not None:
            graph.replay()
            return graph_out
        return step(gpu)

    # ---- timed region: device-resident inputs ------------------------------------------------------------------------
    sampler = ClockSampler(physical_gpu_index(local_rank))
    sampler.start()
    launches_per_step = None
    if graph is not None:      # launches inside a replayed graph are not re-counted by the library: count one eager step
        l0 = lib.css_launch_count()
        step(gpu)
        launches_per_step = lib.css_launch_count() - l0
        barrier()
    launches0 = lib.css_launch_count()
    reducer = getattr(crit, "_reducer", None)
    comm0 = reducer.stats() if (reducer is not None and reducer.ok) else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps - 1):
        run_step()
    out = run_step()                         # only the last step's results are kept (what --dump-outputs writes)
    e1.record()
    barrier()
    elapsed_ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:      # before anything below runs the path again (prototypes are updated in place)
        loss_t, grad_t, maps_t, prob_t = out
        dump_outputs({"loss": loss_t, "grad_rep": grad_t, **maps_t, **({"prob_all": prob_t} if prob_t is not None else {}),
                      "prototypes": protos}, args.dump_outputs)
    comm1 = reducer.stats() if comm0 is not None else None
    launches = lib.css_launch_count() - launches0 if graph is None else launches_per_step * args.steps
    clocks = sampler.stop()
    # live CUDA-event timing of the kernels the rooflines report: each op alone, 20 launches captured in one CUDA graph and
    # replayed between two events on the launching stream (eager launches would add host launch gaps to a 70 us kernel)
    last = crit.last
    ws_, rows_, norms_ = last["ws"], last["rows"], last["norms"]
    rows_dt_ = _lib.DTYPE_BF16 if rows_.dtype == torch.bfloat16 else _lib.DTYPE_F32
    ga_ = torch.empty(C * Q * D, device=dev, dtype=torch.float32)
    apx_ = torch.empty(C * Q, device=dev, dtype=torch.int32)
    loss_ = torch.empty((), device=dev, dtype=torch.float32)
    cnt_ = torch.zeros(1, device=dev, dtype=torch.int64)

    def score_once():
        _lib.check(lib.css_score_ce(_lib.ptr(rows_), rows_dt_, _lib.ptr(norms_), _lib.ptr(ws_.proto_hat), _lib.ptr(ws_.class_cdf),
                                    _lib.ptr(ws_.valid_list), _lib.ptr(ws_.hard_list), _lib.ptr(ws_.meta), None, None, 3407, 0,
                                    _lib.ptr(cnt_), N, C, D, Q, Nn, float(temp), _lib.ptr(ws_.loss_kq), _lib.ptr(apx_), _lib.ptr(ga_),
                                    _lib.ptr(loss_), _lib.stream_ptr()), "css_score_ce")

    score_avg_ms = time_in_graph(score_once)
    rep_ms = {}
    if strategy != "ori":
        rep_ms["student"] = time_in_graph(lambda: css_b200.ops.proto_softmax_sim(gpu["rep_all"], protos, temp))
        rep_ms["teacher"] = time_in_graph(lambda: css_b200.ops.cos_sim_map(gpu["rep_u"], protos))
    else:
        rep_ms["rows_only"] = time_in_graph(lambda: css_b200.ops.rep_rows(gpu["rep_all"]))
    barrier()
    t_all = [torch.zeros(1, device=dev, dtype=torch.float64) for _ in range(world)]
    t_mine = torch.tensor([elapsed_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_gather(t_all, t_mine)
    else:
        t_all = [t_mine]
    per_rank_ms = [float(t.item()) / args.steps for t in t_all]
    ms_per_step = max(per_rank_ms)
    value = world * N / (ms_per_step * 1e-3)
    multi = None
    if world > 1:
        wait_us = None
        if comm0 is not None:
            calls = max(comm1["calls"] - comm0["calls"], 1)
            w_mine = torch.tensor([(comm1[k] - comm0[k]) / calls / 1e3 for k in ("wait_ns_total", "push_ns_total", "kernel_ns_total")],
                                  device=dev, dtype=torch.float64)
            w_all = [torch.zeros_like(w_mine) for _ in range(world)]
            dist.all_gather(w_all, w_mine)
            wait_us = [round(float(x[0].item()), 2) for x in w_all]
            push_us = [round(float(x[1].item()), 2) for x in w_all]
            kern_us = [round(float(x[2].item()), 2) for x in w_all]
        s_ = sorted(per_rank_ms)
        multi = {"per_rank_ms_per_step": {"min": s_[0], "median": s_[len(s_) // 2], "max": s_[-1]},
                 "exchange_wait_us_per_step_by_rank": wait_us,
                 "exchange_push_us_per_step_by_rank": push_us if wait_us is not None else None,
                 "exchange_kernel_us_per_step_by_rank": kern_us if wait_us is not None else None,
                 "note": "every rank times the same K steps with its own events; the step time reported is the max; "
                         "exchange_wait = time the peer-memory kernel spent waiting for the slowest rank's block (rank skew), "
                         "exchange_push = kernel entry until its own block is stored on every peer and fenced, exchange_kernel = whole "
                         "kernel (globaltimer inside css_stats_allreduce)"}

    # ---- the step as the UNMODIFIED scripts drive it: DistributedDataParallel(find_unused_parameters=True) clones rep_all, the
    # loss verifies the carried rows on the device (css_rows_refresh) instead of re-reading the map ---------------------------
    ddp_line = None
    if strategy != "ori":
        rep_clone = gpu["rep_all"].clone()
        try:
            if use_graph:
                g2, _ = capture(gpu, rep_clone)
                run2 = g2.replay
            else:
                run2 = lambda: step(gpu, rep_clone)
            for _ in range(3):
                run2()
            barrier()
            e0.record()
            for _ in range(args.steps):
                run2()
            e1.record()
            barrier()
            t2 = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(t2, op=dist.ReduceOp.MAX)
            ddp_line = {"ms_per_step": float(t2.item()) / args.steps, "rows_cache_mode": crit.last["rows_cache_mode"],
                        "rows_stale_flag": int(crit.last["ws"].meta[_lib.META_ROWS_STALE].item()),
                        "note": "same step with the loss fed a CLONE of rep_all (what DDP's output sink does, mix_label.py:77): the rows "
                                "carried by prob are verified on the device, no second read of the map"}
            g2 = None
        except Exception as e:
            ddp_line = {"error": repr(e)}

    # ---- e2e: host buffers, H2D of every input + D2H of the loss and of the maps the augmentation receives -----------------
    keys = ["rep_u", "pred_u", "rep_all", "label", "mask"] if strategy != "ori" else ["pred_u", "rep_all", "label", "mask", "prob_ori"]
    numa = pin_to_gpu_numa_node(physical_gpu_index(local_rank))          # before the pinned buffers are allocated (first touch)
    pinned = {k: host[k].clone(memory_format=torch.preserve_format).pin_memory() for k in keys}
    unpin_cpu()
    # two staging sets: the H2D copy of step i+1 (copy stream) overlaps the kernels of step i; every step still uploads all
    # of its inputs from pinned host memory and reads its loss and label / confidence maps back
    staged = [{k: torch.empty_like(gpu[k]) for k in keys} for _ in range(2)]
    for st_set in staged:
        for k in gpu:
            if k not in keys:
                st_set[k] = gpu[k]
    h2d = sum(v.numel() * v.element_size() for v in pinned.values())
    copy_stream = torch.cuda.Stream()
    ready = [torch.cuda.Event(), torch.cuda.Event()]      # inputs of the set have landed
    done = [torch.cuda.Event(), torch.cuda.Event()]       # the step that read the set has finished

    e2e_graphs = [None, None]
    if use_graph:
        try:
            e2e_graphs = [capture(staged[0]), capture(staged[1])]
        except Exception as e:
            sys.stderr.write(f"bench: e2e graph capture failed ({e!r}); eager\n")
            e2e_graphs = [None, None]
    _, _, maps0, _ = step(staged[0])
    host_maps = [torch.empty(m.shape, dtype=m.dtype).pin_memory() for m in maps0.values()]
    d2h = 4 + sum(m.numel() * m.element_size() for m in host_maps)

    def upload(i):
        s_ = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(done[s_])
            for k in keys:
                staged[s_][k].copy_(pinned[k], non_blocking=True)
            ready[s_].record(copy_stream)

    def e2e_run(n):
        for ev in done:
            ev.record()
        upload(0)
        for i in range(n):
            s_ = i % 2
            if i + 1 < n:
                upload(i + 1)
            torch.cuda.current_stream().wait_event(ready[s_])
            if e2e_graphs[s_] is not None:
                e2e_graphs[s_][0].replay()
                loss, _, maps, _ = e2e_graphs[s_][1]
            else:
                loss, grad, maps, _ = step(staged[s_])
            for hm, m in zip(host_maps, maps.values()):      # what the reference flow ships to the host for the PIL augmentation
                hm.copy_(m, non_blocking=True)
            done[s_].record()
            float(loss.item())                # D2H read of the step's result (synchronises; the map copies precede it in stream order)

    e2e_run(4)
    barrier()
    e0.record()
    e2e_run(args.e2e_steps)
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    t_e2e = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    e2e_value = world * N / (float(t_e2e.item()) / args.e2e_steps * 1e-3)
    # the H2D leg alone (same pinned buffers, same copy stream, nothing else running): what the host side can deliver per rank
    barrier()
    e0.record()
    for _ in range(5):
        with torch.cuda.stream(copy_stream):
            for k in keys:
                staged[0][k].copy_(pinned[k], non_blocking=True)
    copy_stream.synchronize()
    e1.record()
    barrier()
    t_h2d = torch.tensor([e0.elapsed_time(e1) / 5], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_h2d, op=dist.ReduceOp.MAX)
    h2d_only_ms = float(t_h2d.item())

    # ---- rooflines ------------------------------------------------------------------------------------------------------
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"
    stream_b, gather_b = path_bytes(cfg, v_eff)
    achieved = gather_b / (score_avg_ms * 1e-3) / 1e9 if score_avg_ms > 0 else 0.0
    prof = {}
    prof_path = os.path.join(ROOT, "profiles", "kernel_traffic.json")
    if os.path.exists(prof_path):
        try:
            prof = json.load(open(prof_path)).get(args.workload, {})
        except Exception:
            prof = {}
    scorer_env = os.environ.get("CSS_B200_SCORER", "bulk")          # the library's default path is the register / bulk-copy hybrid
    scorer_kernel = {"reg": "score_ce_kernel", "ring": "score_ce_ring_kernel"}.get(scorer_env, "score_ce_bulk_kernel") \
        if crit.last["rows"].dtype == torch.float32 else "score_ce_kernel"
    traffic = prof.get(scorer_kernel)
    # ceiling of the access pattern, measured live on this device with the step's own pixel-major copy as the table
    probe = run_probe(crit.last["rows"], v_eff * Q if v_eff else Q, Nn)
    gather_peak = probe.get("l2_gather_gbs") if probe else None
    roofline = {"bound": "l2_gather", "kernel": f"{scorer_kernel} (css_score_ce)", "achieved": achieved,
                "peak": gather_peak, "unit": "GB/s", "frac": (achieved / gather_peak) if gather_peak else None,
                "peak_source": "measured live by tools/dev/css_probe.cu: random 1 KB-row gathers from this step's own pixel-major copy "
                               f"({crit.last['rows'].numel() * crit.last['rows'].element_size() / 1e6:.0f} MB table), no math, best of 3 "
                               "variants" if gather_peak else "probe library absent (tools/dev/libcss_probe.so)",
                "traffic": traffic, "algorithmic_bytes_per_launch": gather_b, "avg_launch_ms": score_avg_ms,
                "share_of_step": score_avg_ms / ms_per_step,
                "hbm": {"peak": peak, "peak_source": peak_src,
                        "dram_gbs": (traffic / (score_avg_ms * 1e-3) / 1e9) if (traffic and score_avg_ms > 0) else None,
                        "dram_frac_of_hbm": (traffic / (score_avg_ms * 1e-3) / 1e9 / peak) if (traffic and score_avg_ms > 0) else None,
                        "logical_over_hbm": achieved / peak,
                        "l2_served_frac": (1.0 - traffic / gather_b) if (traffic and gather_b) else None},
                "note": "the dominant kernel gathers one 1 KB row per (query, candidate) pair (SURVEY.md 8(d): V*Q*(Nn+1)*D*4 logical bytes); "
                        "the table is mostly L2 resident, so the bound is the L2->SM gather path, not HBM: `achieved`/`peak` are logical "
                        "gather GB/s against the live-measured ceiling of that pattern; `hbm` says what reached DRAM (ncu dram bytes "
                        "per launch from profiles/kernel_traffic.json) and how the logical figure compares with measured HBM bandwidth",
                "path": {"bytes_stream": stream_b, "bytes_gather": gather_b,
                         "achieved_gbs": (stream_b + gather_b) / (ms_per_step * 1e-3) / 1e9,
                         "frac_of_hbm": (stream_b + gather_b) / (ms_per_step * 1e-3) / 1e9 / peak,
                         "compulsory_gbs": stream_b / (ms_per_step * 1e-3) / 1e9,
                         "compulsory_frac_of_hbm": stream_b / (ms_per_step * 1e-3) / 1e9 / peak}}
    # the HBM-bound streaming kernel: the student rep pass (one read of rep_all -> prob_all + pixel-major rows + norms)
    roofline_hbm = None
    if rep_ms.get("student"):
        t_st = rep_ms["student"]
        s_el = 4
        nhwc = cfg.get("layout") == "nhwc"
        alg = N * (D * s_el + 4 * C + 4) if nhwc else N * (D * s_el + 4 * C + D * s_el + 4)
        tr = prof.get("rep_pass_student")
        roofline_hbm = {"bound": "hbm", "kernel": ("rep_pass_nhwc_kernel (css_rep_pass_nhwc, student: one TMA read of the channels-last rep_all -> prob_all + "
                                   "norms, tcgen05 / TMEM; timed with the prototype-preparation launch of the same call)") if nhwc else
                        ("rep_pass_kernel<SOFTMAX, rows> (css_rep_pass, student: one read of rep_all -> prob_all + pixel-major "
                         "rows + norms; timed with the prototype-preparation launch of the same call)"), "achieved": alg / (t_st * 1e-3) / 1e9, "peak": peak,
                        "unit": "GB/s", "frac": alg / (t_st * 1e-3) / 1e9 / peak, "peak_source": peak_src, "traffic": tr,
                        "algorithmic_bytes_per_launch": alg, "avg_launch_ms": t_st, "share_of_step": t_st / ms_per_step,
                        "dram_frac_of_hbm": (tr / (t_st * 1e-3) / 1e9 / peak) if tr else None,
                        "copy_gbs_live": probe.get("copy_gbs") if probe else None,
                        "teacher_avg_launch_ms": rep_ms.get("teacher")}

    cpu = None
    gpu_eager = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # one bounded sample of the same workload on the host cores (the unmodified reference when it is on this box), ~10-30 s
        r = run_cpu(cfg, 1, 0, 25.0, host)
        cpu = {"value": r["value"], "unit": "pixels/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]}
        if not args.no_gpu_eager_reference:
            try:      # context line (BASELINE.md 3.6): the same unmodified reference code, eager, on this GPU
                from oracle import ref_bench
                if ref_bench.available():
                    gpu_eager = ref_bench.run_gpu_eager(cfg, host, steps=2, warmup=1, device=str(dev))
            except Exception as e:
                gpu_eager = {"error": repr(e)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "pixels/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(args, cfg), "roofline": roofline, "roofline_hbm_kernel": roofline_hbm,
            "cpu_baseline": cpu, "reference_gpu_eager": gpu_eager,
            "e2e": {"value": e2e_value, "unit": "pixels/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": float(t_e2e.item()) / args.e2e_steps, "steps": args.e2e_steps,
                    "h2d_only_ms_per_step": h2d_only_ms, "h2d_only_gbs_per_rank": h2d / (h2d_only_ms * 1e-3) / 1e9, "host_numa": numa,
                    "d2h": "loss scalar + the label / confidence maps the reference flow hands to the host-side augmentation"},
            "gpu_launches": int(launches) * world, "launch_mode": "cuda_graph" if graph is not None else "eager",
            "exchange": {"peer": "css_stats_allreduce over NVLink peer memory (one launch, rank-ordered sum)",
                         "nccl": "torch.distributed all_reduce", "none": "single process"}[crit.exchange_mode()],
            "exchange_check": exchange_check, "multi_gpu": multi, "ddp_clone_step": ddp_line,
            "clocks": clocks, "loss": loss_value, "present_classes": V, "scored_classes": v_eff,
        }
        emit(line)
    if world == 1 and dist.is_initialized():
        dist.destroy_process_group()
    if world > 1:
        # graphs that captured NCCL work must be released before the communicator goes away; then leave without the
        # interpreter's atexit teardown, which can deadlock on a communicator that was used inside a captured graph
        graph = None
        e2e_graphs = [None, None]
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)
    return 0


if __name__ == "__main__":
    sys.exit(main())
