"""Time of the image side of the augmentation: the PIL chain against css_aug_image.

    python tools/aug_image_bench.py [--reps 10] [--iters 50] [--out profiles/<name>.json]

For each size a training step uses -- V321 (VOC crop 321 x 321, B = 8) and C768 (CityScapes crop 769 x 769, B = 4) --
it measures
  * the device time of the image trip alone (`transform_images` with device-resident parameters; `iters` calls in one CUDA
    graph, CUDA events around the replay; same input every call, so it is read from L2 after the first);
  * the wall time of a whole `batch_transform_2` call (image + one label map + two confidence maps), both trips of a
    step, with the PIL chain (host copy, `_augment_image` per image, copy back) and with the GPU path, alternating in one
    run; every call ends in a device synchronise.  The two outputs are compared for equality on every call.
The card's name and power limit are read in the same run and written beside the numbers."""
import argparse
import json
import os
import random
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from css_b200 import aug  # noqa: E402

SIZES = {"V321": dict(B=8, H=321, W=321), "C768": dict(B=4, H=769, W=769)}
TRIPS = {"trip1 scale 0.5-1.5": ((0.5, 1.5), False), "trip2 scale 1 + jitter/blur/flip": ((1.0, 1.0), True)}


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


def pil_batch_transform_2(images, label, c1, c2, crop_size, scale_size, augmentation):
    """batch_transform_2 with the image on the PIL chain (what the GPU path replaces)."""
    import torchvision.transforms.functional as TF
    host = aug._unnormalise(images).cpu()
    out, geo = zip(*[aug._augment_image(TF.to_pil_image(host[k]), crop_size, scale_size, augmentation)
                     for k in range(host.shape[0])])
    ol, oc = aug.transform_maps([label], [c1, c2], np.asarray(geo, np.int32), out[0].shape[1:])
    return torch.stack(out).pin_memory().to(images.device, non_blocking=True), ol[0], oc[0], oc[1]


def device_time_us(B, H, W, iters):
    torch.manual_seed(0)
    geo, params = aug.draw_image_params(B, H, W, (H, W), (1.0, 1.0), True)
    params[:, 0] = params[:, 9] = 1                                  # every image: jitter and blur
    params[:, 1:5] = (3, 1, 0, 2)
    params[:, 5:9] = (1.1, 0.9, 1.2, 17)
    params[:, 10] = 1.0
    x = torch.rand(B, 3, H, W, device="cuda")
    g, p = torch.from_numpy(geo).cuda(), torch.from_numpy(params).cuda()
    for _ in range(3):
        aug.transform_images(x, g, p, (H, W))
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(iters):
            aug.transform_images(x, g, p, (H, W))
    graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    graph.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e3


def wall_ms(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("aug_image_bench: needs a CUDA device")
    res = {"card": card(), "torch_threads": torch.get_num_threads(), "reps": a.reps, "sizes": {}}
    for name, s in SIZES.items():
        B, H, W = s["B"], s["H"], s["W"]
        row = {"B": B, "crop": [H, W], "device_us_image_trip": device_time_us(B, H, W, a.iters)}
        rng = np.random.default_rng(0)
        mean, std = (torch.tensor(v).view(1, 3, 1, 1) for v in (aug._MEAN, aug._STD))
        images = ((torch.from_numpy(rng.random((B, 3, H, W), np.float32)) - mean) / std).cuda()     # normalised [0, 1] content
        label = torch.from_numpy(rng.integers(0, 21, (B, H, W)).astype(np.float32)).cuda()
        c1, c2 = (torch.from_numpy(rng.random((B, H, W), np.float32)).cuda() for _ in range(2))
        for trip, (scale, augm) in TRIPS.items():
            kw = dict(crop_size=(H, W), scale_size=scale, augmentation=augm)
            t_pil, t_gpu = [], []
            for rep in range(a.reps + 1):                               # rep 0 warms both paths up
                torch.manual_seed(rep)
                random.seed(rep)
                dt_p, rp = wall_ms(lambda: pil_batch_transform_2(images, label, c1, c2, **kw))
                torch.manual_seed(rep)
                random.seed(rep)
                dt_g, rg = wall_ms(lambda: aug.batch_transform_2(images, label, c1, c2, **kw))
                if not all(torch.equal(u, v) for u, v in zip(rp, rg)):
                    raise SystemExit(f"aug_image_bench: outputs differ at {name} {trip} rep {rep}")
                if rep:
                    t_pil.append(dt_p)
                    t_gpu.append(dt_g)
            row[trip] = {"pil_ms_median": float(np.median(t_pil)), "gpu_ms_median": float(np.median(t_gpu)),
                         "pil_ms": t_pil, "gpu_ms": t_gpu}
        res["sizes"][name] = row
        print(f"{name}: image trip {row['device_us_image_trip']:.1f} us device; " + "; ".join(
            f"{t}: PIL {row[t]['pil_ms_median']:.2f} ms, GPU {row[t]['gpu_ms_median']:.2f} ms" for t in TRIPS))
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
