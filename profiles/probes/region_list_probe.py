"""Probe: the cost of returning neighbour lists from region_growing.knn_pca (gsl_region_knn_pca).

200 000 blob points (BASELINE config C1's cloud size); for k in {10, 64, 65, 500, 2000} one call with
and one without want_knn, alternated, each timed with CUDA events after a warm-up of every shape.  A
separate torch.profiler pass gives the two kernels' own times (knn_pca_kernel: selection, moments and,
for k > 64, the unordered list; knn_order_kernel: the (distance, index) sort of the rows).  The card's
name and power limit are read in the same run.

    python profiles/probes/region_list_probe.py [--reps 15] [--out profiles/region_lists_b200.json]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import numpy as np
import torch

rg = importlib.import_module("3d_gaussian_splatting_project_b200.region_growing")

KS = [10, 64, 65, 500, 2000]


def blobs(rng, n, spread=0.3):
    centres = rng.uniform(-2, 2, size=(10, 3))
    return (centres[rng.integers(0, 10, n)] + rng.normal(0, spread, size=(n, 3))).astype(np.float32)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = (s.strip() for s in q.split(","))
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def call(d, k, lists):
    return rg.knn_pca(d, k, want_residuals=False, want_knn=lists)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=200_000)
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("region_list_probe needs a CUDA device")
    d = torch.from_numpy(blobs(np.random.default_rng(1), a.n)).cuda()
    for k in KS:                                         # warm-up: modules, workspace, every shape
        for lists in (False, True):
            call(d, k, lists)
    torch.cuda.synchronize()
    rows = []
    for k in KS:
        ms = {False: [], True: []}
        for _ in range(a.reps):
            for lists in (False, True):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                out = call(d, k, lists)
                e1.record()
                torch.cuda.synchronize()
                ms[lists].append(e0.elapsed_time(e1))
                del out
        row = dict(k=k, path="in-kernel rank sort" if k <= 64 else "emit + knn_order_kernel")
        for lists, tag in ((False, "without_lists"), (True, "with_lists")):
            v = np.array(ms[lists])
            row[tag + "_ms"] = dict(median=float(np.median(v)), min=float(v.min()), max=float(v.max()))
        row["list_cost_ms"] = row["with_lists_ms"]["median"] - row["without_lists_ms"]["median"]
        rows.append(row)
        print(json.dumps(row))
    # kernel times from one profiled call per shape with lists
    from torch.profiler import ProfilerActivity, profile
    kernels = {}
    for k in KS:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            call(d, k, True)
            torch.cuda.synchronize()
        for ev in prof.key_averages():
            for tag in ("knn_pca_kernel", "knn_order_kernel"):
                if tag in ev.key:
                    kernels.setdefault(str(k), {})[tag + "_ms"] = ev.device_time_total / 1e3 / max(ev.count, 1)
    print(json.dumps(kernels))
    res = dict(probe="region_list_probe", points=a.n, cloud="ten Gaussian blobs, sigma 0.3, centres in [-2, 2]^3, seed 1",
               reps=a.reps, timing="CUDA events around region_growing.knn_pca (want_residuals=False), median/min/max over reps",
               device=card(), rows=rows, kernel_ms_with_lists=kernels)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res["device"]))


if __name__ == "__main__":
    main()
