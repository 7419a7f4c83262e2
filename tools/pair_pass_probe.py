"""Pair-pass probe: what the broad phase costs per step on three scenes, and what its hierarchy looks like.

Scenes: the headline pyramid (447 rows, 100 128 boxes), the config-3 tumbler (100 x 100 boxes in a turning container) and
the config-5 field (256 pyramids of 45 rows in one world). After --warmup steps, --steps steps are stepped one at a time
and for each the probe reads the pair-stage time (stage_ms()[0]: the commit of this step plus the search that ran behind
the previous one), the moved proxies, the hierarchy's level count and the large-leaf list size; it reports the median and
maximum of the time and the number of re-sorts in the window. One JSON line per scene, after the GPU's name and power
limit.

--profile DIR adds, per scene, a separate run of one step under torch.profiler (CUDA activities) and writes the kernel
times of that step to DIR/<scene>_kernels.json.

    python tools/pair_pass_probe.py [--steps 60] [--warmup 20] [--profile DIR] [--scenes pyramid,tumbler,field]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from solver2d_b200 import capi, device, scenes  # noqa: E402

DT = 1.0 / 60.0
SCENES = {
    "pyramid": lambda P: scenes.pyramid(P, "TGS_Soft", base_count=447),
    "tumbler": lambda P: scenes.tumbler(P, "TGS_Soft"),
    "field": lambda P: scenes.pyramid_field(P, "TGS_Soft", count=256, base_count=45),
}


def gpu_info() -> str:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True)
    return out.stdout.strip().splitlines()[0]


def measure(dev, P, name, warmup, steps):
    sc = SCENES[name](P)
    dw = device.DeviceWorld.attach(dev, sc.world)
    for _ in range(warmup):
        sc.step(DT, 4, 2, True)
    rebuilds0 = dw.counters().pairRebuildCount
    pair_ms, moved, levels, large = [], [], [], []
    for _ in range(steps):
        sc.step(DT, 4, 2, True)
        dw.sync()  # the search behind this step has to be finished for its time to count
        pair_ms.append(dw.stage_ms()[0])
        c = dw.counters()
        moved.append(c.movedCount)
        levels.append(c.treeHeight)
        large.append(c.largeLeafCount)
    c = dw.counters()
    sc.destroy()
    return {
        "scene": name, "steps": steps, "warmup": warmup,
        "pair_ms_median": float(np.median(pair_ms)), "pair_ms_max": float(np.max(pair_ms)),
        "moved_median": int(np.median(moved)), "moved_max": int(np.max(moved)),
        "levels": sorted(set(levels)), "large_leaves": sorted(set(large)),
        "rebuilds_in_window": c.pairRebuildCount - rebuilds0, "shapes": c.shapeCapacity,
    }


def profile(dev, P, name, warmup, out_dir):
    import torch
    from torch.profiler import ProfilerActivity, profile as tprofile

    sc = SCENES[name](P)
    dw = device.DeviceWorld.attach(dev, sc.world)
    for _ in range(warmup):
        sc.step(DT, 4, 2, True)
    dw.sync()
    with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
        sc.step(DT, 4, 2, True)
        dw.sync()
        torch.cuda.synchronize()
    kernels = {}
    for ev in prof.key_averages():
        us = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        if us > 0:
            kernels[ev.key] = {"us": float(us), "calls": int(ev.count)}
    sc.destroy()
    kernels = dict(sorted(kernels.items(), key=lambda kv: -kv[1]["us"]))
    with open(os.path.join(out_dir, f"{name}_kernels.json"), "w") as fh:
        json.dump(kernels, fh, indent=1)
    return kernels


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--profile", default=None, help="directory for the per-kernel split of one step per scene")
    ap.add_argument("--scenes", default="pyramid,tumbler,field")
    args = ap.parse_args()
    if args.steps < 60:
        ap.error("--steps: at least 60")
    names = args.scenes.split(",")
    for n in names:
        if n not in SCENES:
            ap.error(f"unknown scene {n}")

    P = capi.Solver2D(device.LIB_PATH)
    dev = device.Device()
    print(json.dumps({"gpu": gpu_info()}), flush=True)
    for name in names:
        print(json.dumps(measure(dev, P, name, args.warmup, args.steps)), flush=True)
    if args.profile:
        os.makedirs(args.profile, exist_ok=True)
        for name in names:
            kernels = profile(dev, P, name, args.warmup, args.profile)
            pair = {k: v for k, v in kernels.items() if k.startswith(("s2b", "void cub", "Memset", "Memcpy"))}
            print(json.dumps({"scene": name, "profiled_step_kernels_us": {k: round(v["us"], 1) for k, v in pair.items()}}),
                  flush=True)


if __name__ == "__main__":
    main()
