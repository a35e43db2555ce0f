"""Omni3D AP evaluation on the GPU: 2D + 3D evaluate + accumulate + summarize from device-resident detections.

    python tools/bench_eval.py [--images 20000] [--cats 50] [--oracle-images 1000] [--out PATH]

Prints one JSON line: the synchronised wall time of Omni3DEval (median of --reps runs after a warm-up), the per-kernel
CUDA times of a separate torch.profiler run (sorts included), the CPU numpy oracle's time on a smaller seeded set
(--oracle-images, stated in the output), and the GPU name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import evalgen  # noqa: E402
from omni3d_b200.evaluation import Omni3DEval  # noqa: E402


def run(gt, res):
    e2 = Omni3DEval(gt, "2D")
    e2.add_results(res)
    torch.cuda.synchronize()
    t = time.perf_counter()
    e3 = e2.for_mode("3D")
    logs = []
    for e in (e2, e3):
        e.evaluate()
        e.accumulate()
        logs.append(e.summarize())
    torch.cuda.synchronize()
    return time.perf_counter() - t, logs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=20000)
    ap.add_argument("--cats", type=int, default=50)
    ap.add_argument("--oracle-images", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_eval needs a CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    t0 = time.perf_counter()
    gt, res = evalgen.make_set(a.images, a.cats, seed=0, gt_per_img=5, fp_per_img=20)
    gen_s = time.perf_counter() - t0
    run(gt, res)                                                     # warm-up: module load, allocator
    times = [run(gt, res)[0] for _ in range(a.reps)]
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        run(gt, res)
    kern = {}
    for ev in prof.key_averages():
        if ev.device_type == torch.autograd.DeviceType.CUDA and ev.self_device_time_total > 0:
            kern[ev.key[:80]] = round(ev.self_device_time_total / 1e3, 3)
    kern = dict(sorted(kern.items(), key=lambda kv: -kv[1])[:15])
    from oracle import omni3d_eval_oracle as oracle
    ogt, ores = evalgen.make_set(a.oracle_images, a.cats, seed=0, gt_per_img=5, fp_per_img=20)
    t0 = time.perf_counter()
    for mode in ("2D", "3D"):
        p, ev = oracle.evaluate(ogt, oracle.load_res(ogt, ores), mode)
        prec, rec, _ = oracle.accumulate(p, oracle.per_cat_area(p, ev))
        oracle.summarize(p, prec, rec)
    oracle_s = time.perf_counter() - t0
    out = {"workload": {"images": a.images, "categories": a.cats, "gt": len(gt["annotations"]), "detections": len(res),
                        "seed": 0, "generation_s": round(gen_s, 2)},
           "gpu": q, "eval_2d_3d_s": {"median": float(np.median(times)), "all": [round(x, 4) for x in times]},
           "profile_cuda_ms_top": kern,
           "oracle_cpu": {"images": a.oracle_images, "detections": len(ores), "s": round(oracle_s, 2)}}
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
