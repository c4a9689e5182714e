#!/usr/bin/env python
"""Benchmark of the hot path: Gaussian x view votes/s (label lifting) and K-means iters/s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

Workload (BASELINE.json configs[3] + configs[4], the shape the metric is quoted on; it fits
one GPU): 6M Gaussians x 300 views of 1920x1080 label maps with 151 label values, and K-means
K=64 on 6M x 59 float32 features.  Total work is fixed; Gaussians (rows) are split across the
ranks, every view is replicated ("scaling": "strong").  Data is synthetic (scene.py).

One "step" = one lifting pass over this rank's Gaussians and all views (gsl_lift_prepare +
gsl_lift_gather + gsl_lift_majority: ordering and per-tile verdicts, the projection + gather sweep,
the majority vote) with positions and packed maps resident in HBM.  K-means iterations
(gsl_kmeans_step_exchange: assignment + sums, then reduction fused with the cross-rank exchange
and the update) are timed the same way and reported under "kmeans".  `e2e` is the same lifting
through the public Python entry point (deep_learning_segmentation.lift_labels) with pinned HOST
inputs: int32 maps and positions go to the device and labels are copied back, all inside the
timed region; `h2d_bytes_per_step` is counted from the tensors actually copied.

Parity is checked inside this run, at every rank count, against the CPU oracle (the checker, never
the thing timed): lifting labels of a 2M-Gaussian sample, the near-boundary count of that sample,
K-means labels after one step on 1M rows, centroids bit-equal across ranks, and the distance of the
sharded float64 update from the reference's float32 mean and from the exact mean ("parity").

`--impl reference` times the reference's CPU algorithm instead: the reference is pure Python
and cannot be compiled, so this runs the oracle's C port of it (oracle/gsl_oracle.c, OpenMP,
every core the process may use) on a bounded sample of the same workload.

`--dump-outputs DIR` writes, after the run, what the last timed step returned, as float32 .npy
files: lift_labels (one label per Gaussian), and kmeans_labels, kmeans_centroids, kmeans_shift
of the last timed K-means iteration.  The inputs are seeded, so two builds run with the same
arguments can be compared file by file.  The files stay under 64 MB: for larger workloads the
label arrays keep the same fraction of their rows, picked by np.random.default_rng(0), in order.

Nothing is written into the repository tree, which may be read-only: no bytecode, and the
libraries are the ones `__graft_entry__.build()` compiled.
"""
from __future__ import annotations

import argparse
import atexit
import importlib
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
PKG = "3d_gaussian_splatting_project_b200"

METRIC = "gaussian_view_votes_per_s"
UNIT = "votes/s"


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError(f"{s} is not a positive integer")
    return v


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=20,
                    help="timed lifting passes, K-means iterations and end-to-end calls")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["native", "reference"], default="native")
    ap.add_argument("--gaussians", type=int, default=6_000_000)
    ap.add_argument("--views", type=int, default=300)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--kmeans-rows", type=int, default=6_000_000)
    ap.add_argument("--kmeans-dim", type=int, default=59)
    ap.add_argument("--kmeans-k", type=int, default=64)
    ap.add_argument("--parity-gaussians", type=int, default=2_000_000)
    ap.add_argument("--parity-rows", type=int, default=1_000_000)
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true", help="no CPU oracle legs (parity and cpu_baseline become null)")
    ap.add_argument("--skip-kmeans", action="store_true")
    ap.add_argument("--skip-next", action="store_true", help="no section-8f rows (viewer depth sort / hit test, region-growing normals)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy")
    return ap.parse_args()


def workload_config(a):
    return {
        "workload": f"C4+C5: lift {a.gaussians} Gaussians x {a.views} views {a.width}x{a.height} (151 labels, 32px blocks); "
                    f"k-means K={a.kmeans_k} on {a.kmeans_rows}x{a.kmeans_dim} f32",
        "gaussians": a.gaussians, "views": a.views, "map": [a.height, a.width],
        "kmeans": {"rows": a.kmeans_rows, "dim": a.kmeans_dim, "k": a.kmeans_k},
        "partition": f"gaussian-slices x{a.gpus}, views replicated",
        "l2": "inputs (packed label maps 642 MB; K-means rows 1.4 GB) exceed the 126 MB L2; no explicit flush",
    }


def peak_hbm():
    return 6521.1, "HBM copy bandwidth measured on a B200 (DESIGN.md section 4)"


def ncu_traffic(name, world):
    """DRAM bytes per launch from the committed ncu capture of this workload on ONE GPU
    (profiles/traffic.json); not known for other rank counts."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if world != 1 or not os.path.exists(path):
        return None
    try:
        return json.load(open(path)).get(name)
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20", "-i", str(self.index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
            atexit.register(self.stop)             # also when the run fails: no nvidia-smi left behind
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self):
        if self.proc is not None and self.proc.poll() is None:
            self.proc.terminate()
            self.proc.wait()

    def summary(self, t0, t1):
        sm, mx, reasons, power = [], [], set(), []
        for ts, line in self.rows:
            if ts < t0 - 0.02 or ts > t1 + 0.05:
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); power.append(float(f[6]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": float(max(power))}


# ----------------------------------------------------------------------------------------
# synthetic scene
# ----------------------------------------------------------------------------------------
def build_scene(a, gs, pinned):
    import torch
    cams = gs.scene.lookat_cameras(a.views, width=a.width, height=a.height, seed=4)
    pos = gs.scene.gaussian_cloud(a.gaussians, 1.5, seed=4)
    shape = (a.views, a.height, a.width)
    if pinned:
        maps_t = torch.empty(shape, dtype=torch.int32, pin_memory=True)
        maps = maps_t.numpy()
    else:
        maps_t, maps = None, np.empty(shape, np.int32)
    gs.scene.block_label_maps(a.views, a.height, a.width, block=32, lo=-1, hi=149, seed=1000, out=maps)
    return cams, pos, maps, maps_t


def kmeans_init(a, feats):
    np.random.seed(0)
    return feats[np.random.choice(a.kmeans_rows, a.kmeans_k, replace=False)]


DUMP_BYTES = 60_000_000          # array data; with the .npy headers the files stay under 64 MB


def dump_outputs(path, arrays):
    """Write each array as path/<name>.npy in float32 (labels are small integers: exact).  Over
    DUMP_BYTES in all, every array above 1 MB keeps the same fraction of its rows, a seeded
    sorted sample; the small ones (centroids, shift) are written whole."""
    arrays = {name: np.asarray(x, np.float32) for name, x in arrays.items()}
    small = sum(x.nbytes for x in arrays.values() if x.nbytes <= 1 << 20)
    big = sum(x.nbytes for x in arrays.values() if x.nbytes > 1 << 20)
    keep = min(1.0, (DUMP_BYTES - small) / big) if big else 1.0
    os.makedirs(path, exist_ok=True)
    for name, x in arrays.items():
        if keep < 1.0 and x.nbytes > 1 << 20:
            rows = np.random.default_rng(0).choice(len(x), int(len(x) * keep), replace=False)
            x = x[np.sort(rows)]
        np.save(os.path.join(path, name + ".npy"), x)


# ----------------------------------------------------------------------------------------
# CPU legs: the oracle's C port of the reference algorithm on the host cores
# ----------------------------------------------------------------------------------------
def cpu_lift_sample(a, orc, cams, pos, maps, n_s, want_near=False):
    views = orc.make_views(cams, [(a.height, a.width)] * a.views)
    t0 = time.perf_counter()
    labels, near, vis = orc.lift_votes(pos[:n_s], views, maps, eps=1e-4, want_near=want_near)
    dt = time.perf_counter() - t0
    return n_s * a.views / dt, dt, vis, labels, near


def cpu_kmeans_sample(a, orc, data, cen):
    t0 = time.perf_counter()
    lab = orc.kmeans_assign(data, cen)
    orc.kmeans_update(data, lab, cen)
    dt = time.perf_counter() - t0
    return 1.0 / (dt * a.kmeans_rows / len(data)), dt, lab


def next_rows(a, gs, orc, pos, labels_host, dev):
    """SURVEY section 8f rows N3 / N4 on one GPU: the viewer worker's depth sort and click hit test over the
    bench cloud, and region_growing.py's normals (k = 2000) over its first 200 000 points; each checked
    against the oracle (when available) and timed with CUDA events, the oracle timed beside it."""
    import torch
    viewer, rgrow = gs.viewer, importlib.import_module(gs.__name__ + ".region_growing")
    out = {}
    dpos = torch.from_numpy(pos).to(dev)
    dlab = torch.from_numpy(np.ascontiguousarray(labels_host, np.int32)).to(dev)
    n = int(dpos.shape[0])

    def timed(fn, reps):
        fn()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            r = fn()
        e1.record()
        torch.cuda.synchronize(dev)
        return r, e0.elapsed_time(e1) / reps

    view = [1.0, 0, 0, 0, 0, 1.0, 0, 0, 0, 0, 1.0, 0, 0, 0, 6.0, 1.0]              # cloud pushed to z = 6 (column-major)
    proj = [1.2, 0, 0, 0, 0, 1.2 * 16 / 9, 0, 0, 0, 0, 1.01, 1.0, 0, 0, -0.2, 0]
    vp = viewer.multiply4(proj, view)
    order, ms = timed(lambda: viewer.run_sort(dpos, vp), 10)
    row = {"gaussians": n, "ms": ms, "gaussians_per_s": n / (ms * 1e-3), "kernels": "depth + bucket + 2 x (histogram, scan, scatter)"}
    if orc is not None:
        t0 = time.perf_counter()
        want = orc.viewer_depth_sort(pos, vp)
        row["cpu_ms"] = (time.perf_counter() - t0) * 1e3
        row["equals_oracle"] = bool(np.array_equal(order.cpu().numpy(), want))
    out["viewer_depth_sort (gaussians_selection.js:417-462)"] = row

    clicks = [(960.0, 540.0), (700.5, 400.25), (1200.0, 650.0), (10.0, 10.0)]
    def hits():
        return [viewer.perform_hit_testing(x, y, view, proj, (1920, 1080), dpos, dlab, return_index=True) for x, y in clicks]
    got, ms = timed(hits, 3)
    row = {"gaussians": n, "clicks": len(clicks), "ms_per_click": ms / len(clicks), "selected": [g[1] for g in got],
           "note": "per click: project all Gaussians, reduce, read the label back (one host sync)"}
    if orc is not None:
        t0 = time.perf_counter()
        want = [orc.viewer_hit_test(pos, labels_host, vp, x, y, (1920, 1080)) for x, y in clicks]
        row["cpu_ms_per_click"] = (time.perf_counter() - t0) * 1e3 / len(clicks)
        row["equals_oracle"] = bool(got == want)
    out["viewer_hit_test (gaussians_selection.js:361-395)"] = row

    m, k = min(200_000, n), 2000
    if m >= k:
        sub = dpos[:m].contiguous()
        res, ms = timed(lambda: rgrow.knn_pca(sub, k), 2)
        st = rgrow.knn_pca(sub, k, want_stats=True)["stats"].cpu().numpy()
        row = {"points": m, "k": k, "ms": ms, "points_per_s": m / (ms * 1e-3),
               "walks_per_query": float(st[0]) / m, "points_visited_per_neighbour_found": float(st[1]) / (m * k),
               "note": "normals + residuals of region_growing.py compute_normals / compute_residuals (k = 2000 as in its __main__)"}
        if orc is not None:
            q0, q1 = m // 2, m // 2 + 200
            t0 = time.perf_counter()
            ref = orc.region_knn_pca(pos[:m], k, queries=(q0, q1))
            cpu_s = time.perf_counter() - t0
            ok = ref["gap"][q0:q1] > 1e-2
            dots = (res["normals"][q0:q1].cpu().numpy() * ref["normals"][q0:q1]).sum(1)
            row["cpu_ms_scaled_to_all_points"] = cpu_s * 1e3 * m / (q1 - q0)
            row["cpu_sample"] = f"{q1 - q0} queries, brute-force C/OpenMP oracle on {orc.max_threads()} threads"
            row["max_1_minus_abs_cos_vs_oracle"] = float((1 - np.abs(dots[ok])).max()) if ok.any() else None
            row["max_abs_residual_diff_vs_oracle"] = float(np.abs(res["residuals"][q0:q1].cpu().numpy() - ref["residuals"][q0:q1])[ok].max()) if ok.any() else None
        out["region_knn_pca (region_growing.py:78-163)"] = row
    return out


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as orc
    gs = importlib.import_module(PKG)
    orc.build()
    cores = orc.set_threads()                      # every core of the box, whatever OMP_NUM_THREADS torchrun exported
    cams, pos, maps, _ = build_scene(a, gs, pinned=False)
    n_s = int(min(len(pos), max(1000, 6.0e8 // a.views)))
    cpu_lift_sample(a, orc, cams, pos, maps, max(1000, n_s // 12))          # warm-up
    times = []
    for _ in range(a.steps):
        _, dt, _, _, _ = cpu_lift_sample(a, orc, cams, pos, maps, n_s)
        times.append(dt)
    value = float(n_s * a.views * len(times) / np.sum(times))
    rows = min(3_000_000, a.kmeans_rows)
    feats = gs.scene.blob_features(a.kmeans_rows, a.kmeans_dim, n_blobs=64, seed=5)
    k_rate, k_dt, _ = cpu_kmeans_sample(a, orc, feats[:rows], kmeans_init(a, feats))
    sample = (f"lifting: first {n_s} of {a.gaussians} Gaussians x all {a.views} views per step; "
              f"k-means: {rows} of {a.kmeans_rows} rows, 1 iteration, time scaled to full size")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": float(np.mean(times) * 1e3 * a.gaussians / n_s),
        "ms_per_step_note": f"measured on {n_s} Gaussians per step and scaled by {a.gaussians / n_s:.2f} to the full scene (the timed steps themselves take {np.mean(times):.2f} s each)",
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(a),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "kmeans": {"metric": "kmeans_iters_per_s", "value": k_rate, "unit": "iters/s", "cores": cores},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "reference is pure Python (12 us per pair measured, BASELINE.md); this arm is the oracle's C/OpenMP port of the same algorithm",
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------
# native arm
# ----------------------------------------------------------------------------------------
def run_native(a):
    import torch
    import torch.distributed as dist
    gs = importlib.import_module(PKG)
    ops, sharding, dls, km = gs.ops, gs.sharding, gs.deep_learning_segmentation, gs.k_means
    native = importlib.import_module(PKG + "._native")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the native arm has no CPU path")
    rank, world, local = sharding.init_from_env("nccl")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world != a.gpus:
        raise SystemExit(f"--gpus {a.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {a.gpus}")
    launches = native.lib().gsl_launch_count
    orc = None
    if rank == 0 and not a.skip_cpu:
        from oracle import oracle as orc
        orc.build()
        orc.set_threads()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    cams, pos, maps, maps_pinned = build_scene(a, gs, pinned=True)
    lo, hi = sharding.slice_bounds(a.gaussians, rank, world)
    n_r = hi - lo
    H, W, V = a.height, a.width, a.views
    views = ops.make_views(cams, [(H, W)] * V)

    # ---- resident inputs: positions slice + packed maps (staged 8 views at a time)
    d_pos = torch.from_numpy(pos[lo:hi]).to(dev)
    PB = ops.packed_map_bytes(H, W)                # strip layout: 16-pixel strips + a ring of zero codes
    packed = torch.empty(V * PB, dtype=torch.uint8, device=dev)
    for v0 in range(0, V, 8):
        v1 = min(v0 + 8, V)
        chunk = maps_pinned[v0:v1].to(dev, non_blocking=True)
        ops.pack_labels(chunk, label_min=-1, n_classes=151, out=packed[v0 * PB:v1 * PB], check_range=False)
    # staging cost of the pack pre-pass (5 bytes per pixel), timed on a resident 8-view chunk
    pack_ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    n_chunk = min(8, V)
    scratch = torch.empty(n_chunk * PB, dtype=torch.uint8, device=dev)
    for i in range(6):
        if i == 1:
            pack_ev[0].record()
        ops.pack_labels(chunk[:n_chunk], label_min=-1, n_classes=151, out=scratch, check_range=False)
    pack_ev[1].record()
    torch.cuda.synchronize()
    pack_ms = pack_ev[0].elapsed_time(pack_ev[1]) / 5 * (V / n_chunk)
    del chunk, scratch
    run_prepare, run_gather, run_majority, run_sweep, labels = ops.lift_phases(d_pos, views, packed, -1, 151)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()

    # ---- lifting, device resident
    for _ in range(a.warmup):
        run_prepare(); run_sweep()
    barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(a.steps + 1)]
    t_wall0 = time.time()
    n_launch0 = launches()
    for i in range(a.steps):                       # the timed steps: ordering + verdicts, then sweep || majority
        ev[i].record(); run_prepare(); run_sweep()
    ev[a.steps].record()
    n_lift_launches = launches() - n_launch0
    dump = {}
    if a.dump_outputs:
        lift_out = labels.clone()                  # the per-phase runs below write `labels` again
    barrier()
    t_wall1 = time.time()
    total_ms = sharding.barrier_max_ms(ev[0].elapsed_time(ev[-1]), dev)
    # the phases one by one (not overlapped), for the per-kernel numbers
    pe = [torch.cuda.Event(enable_timing=True) for _ in range(4 * a.steps)]
    for i in range(a.steps):
        pe[4 * i].record(); run_prepare()
        pe[4 * i + 1].record(); run_gather()
        pe[4 * i + 2].record(); run_majority()
        pe[4 * i + 3].record()
    barrier()
    prepare_ms = float(np.mean([pe[4 * i].elapsed_time(pe[4 * i + 1]) for i in range(a.steps)]))
    sweep_ms = float(np.mean([pe[4 * i + 1].elapsed_time(pe[4 * i + 2]) for i in range(a.steps)]))
    major_ms = float(np.mean([pe[4 * i + 2].elapsed_time(pe[4 * i + 3]) for i in range(a.steps)]))
    sweep_ms_max = sharding.barrier_max_ms(sweep_ms, dev)
    ms_per_step = total_ms / a.steps
    value = a.gaussians * V / (ms_per_step * 1e-3)
    label_hist = torch.bincount((labels + 1).clamp(min=0).long(), minlength=152)[:3].tolist()

    # ---- lifting parity, every rank count: a sample of the job's first Gaussians against the oracle
    parity = {"lifting": None, "kmeans": None}
    cpu = None
    all_labels = sharding.gather_labels(labels, a.gaussians, rank, world)
    if a.dump_outputs:
        dump["lift_labels"] = sharding.gather_labels(lift_out, a.gaussians, rank, world)
        del lift_out
    if orc is not None:
        n_s = min(a.parity_gaussians, a.gaussians)
        r, dt, vis, want, near = cpu_lift_sample(a, orc, cams, pos, maps, n_s, want_near=True)
        got = all_labels[:n_s].cpu().numpy()
        diff = got != want
        parity["lifting"] = {
            "sample": f"first {n_s} Gaussians of the job x all {V} views, gathered from {world} rank(s)",
            "labels_match": bool(not diff.any()), "mismatches": int(diff.sum()),
            "mismatches_outside_near_boundary_set": int((diff & (near == 0)).sum()),
            "near_boundary_count": int(near.sum()), "near_eps_px": 1e-4, "visible_pairs": int(vis),
        }
        cpu = {"value": r, "unit": UNIT, "cores": orc.max_threads(), "kind": "port",
               "sample": f"first {n_s} Gaussians x all {V} views ({dt:.1f} s of C/OpenMP oracle, near-boundary diagnostic included)",
               "labels_match_gpu": bool(not diff.any())}
    del all_labels

    # ---- K-means, device resident
    kres, t_k1 = None, t_wall1
    if not a.skip_kmeans:
        klo, khi = sharding.slice_bounds(a.kmeans_rows, rank, world)
        feats = gs.scene.blob_features(a.kmeans_rows, a.kmeans_dim, n_blobs=64, seed=5)
        init = kmeans_init(a, feats)
        feats_pinned = torch.from_numpy(feats[klo:khi]).pin_memory()
        d_feats = feats_pinned.to(dev)
        d_cen = torch.from_numpy(init).to(dev)
        k_labels = torch.empty(khi - klo, dtype=torch.int32, device=dev)
        sums = torch.empty((a.kmeans_k, a.kmeans_dim + 1), dtype=torch.float64, device=dev)
        new_c, shift = torch.empty_like(d_cen), torch.empty(1, dtype=torch.float32, device=dev)

        # exchange of the K x (D+1) float64 sums: fused into the reduction kernel over peer memory
        # (default), or reduce kernel + NCCL all-reduce + finalize kernel (GSLIFT_KMEANS_EXCHANGE=nccl)
        use_peer = os.environ.get("GSLIFT_KMEANS_EXCHANGE", "peer") != "nccl"
        xch = ops.KMeansExchange(a.kmeans_k, a.kmeans_dim, dev) if use_peer else None

        def k_iter(cen):
            if xch is not None:
                xch.step(d_feats, cen, k_labels, new_c, shift)
                return
            ops.kmeans_step(d_feats, cen, k_labels, sums)
            if world > 1:
                dist.all_reduce(sums)
            ops.kmeans_finalize(sums, cen, new_c, shift)

        # parity of one step from the seeded initialisation, at this rank count
        k_iter(d_cen)
        torch.cuda.synchronize()
        kpar = {"mode": "fast: float64 per-cluster sums, exchanged over peer memory, one rounding to float32 (shardable); "
                        "the reference's own update is a float32 sequential sum (km:126), reproduced bit for bit by update='ordered' on one GPU"}
        if world > 1:
            gathered = [torch.empty_like(new_c) for _ in range(world)]
            dist.all_gather(gathered, new_c)
            kpar["centroids_bit_equal_across_ranks"] = bool(all(torch.equal(g, gathered[0]) for g in gathered))
        step_labels = sharding.gather_labels(k_labels, a.kmeans_rows, rank, world)
        if orc is not None:
            n_k = min(a.parity_rows, a.kmeans_rows)
            full_lab = step_labels.cpu().numpy()
            want_lab = orc.kmeans_assign(feats[:n_k], init)
            kpar["labels_sample"] = f"first {n_k} rows after one step from the seeded initialisation"
            kpar["labels_match"] = bool(np.array_equal(full_lab[:n_k], want_lab))
            # centroids: given the same labels, the reference's float32 sequential mean (km:126) and the exact mean
            ref32, _ = orc.kmeans_update(feats, full_lab, init)
            ref64 = orc.kmeans_update_f64(feats, full_lab, init)
            got_c = new_c.cpu().numpy().astype(np.float64)

            def rel(x, y):           # SURVEY 8c: max over centroids of |delta|_inf / |c_ref|_inf
                return float(np.max(np.abs(x - y).max(axis=1) / np.maximum(np.abs(y).max(axis=1), 1e-30)))
            kpar["rel_err_vs_reference_f32_mean"] = rel(got_c, ref32.astype(np.float64))
            kpar["rel_err_vs_exact_mean"] = rel(got_c, ref64.astype(np.float64))
            kpar["reference_f32_mean_vs_exact_mean"] = rel(ref32.astype(np.float64), ref64.astype(np.float64))
            kpar["tolerance"] = ("north_star: 1e-5 relative.  The sharded update is the exact mean rounded once; its distance from the "
                                 "reference's float32 mean is the reference's own accumulation error (SURVEY H6), which is what "
                                 "reference_f32_mean_vs_exact_mean shows")
            if world == 1:
                ordered_c, _ = ops.kmeans_update_ordered(d_feats, k_labels, d_cen)
                kpar["ordered_bit_exact"] = bool(np.array_equal(ordered_c.cpu().numpy().view(np.uint32), ref32.view(np.uint32)))
        del step_labels
        parity["kmeans"] = kpar

        for _ in range(a.warmup):
            k_iter(d_cen)
        barrier()
        kev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        cur = d_cen.clone()
        k_launch0 = launches()
        kev[0].record()
        for _ in range(a.steps):
            k_iter(cur)
            cur.copy_(new_c)                       # real Lloyd iterations: centroids move
        kev[1].record()
        k_launches = launches() - k_launch0
        if a.dump_outputs:                         # the ordered-update timing below writes k_labels again
            dump["kmeans_centroids"], dump["kmeans_shift"] = new_c.clone(), shift.clone()
            dump["kmeans_labels"] = sharding.gather_labels(k_labels.clone(), a.kmeans_rows, rank, world)
        barrier()
        t_k1 = time.time()
        k_ms = sharding.barrier_max_ms(kev[0].elapsed_time(kev[1]), dev) / a.steps
        peak, peak_src = peak_hbm()
        rows_r = khi - klo
        k_bytes = rows_r * (4 * a.kmeans_dim + 4) + 2 * a.kmeans_k * a.kmeans_dim * 4
        kres = {"metric": "kmeans_iters_per_s", "value": 1e3 / k_ms, "unit": "iters/s", "ms_per_iter": k_ms,
                "update": "fast (float64 segmented sums" + ((", exchange of K x (D+1) f64 fused into the reduction kernel over peer memory)" if use_peer else ", NCCL all-reduce of K x (D+1) f64)") if world > 1 else ")"),
                "roofline": {"bound": "hbm", "achieved": k_bytes / (k_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                             "frac": k_bytes / (k_ms * 1e-3) / 1e9 / peak, "traffic": ncu_traffic("kmeans_step_kernel", world),
                             "algorithmic_bytes": k_bytes, "peak_source": peak_src},
                "gpu_launches_per_iter": k_launches / a.steps}
        if world == 1:
            # reference-order (bit-exact) update, single device
            oev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            ops.kmeans_assign(d_feats, d_cen, k_labels); ops.kmeans_update_ordered(d_feats, k_labels, d_cen)
            torch.cuda.synchronize()
            oev[0].record()
            for _ in range(3):
                ops.kmeans_assign(d_feats, d_cen, k_labels)
                ops.kmeans_update_ordered(d_feats, k_labels, d_cen)
            oev[1].record(); torch.cuda.synchronize()
            kres["ordered_ms_per_iter"] = oev[0].elapsed_time(oev[1]) / 3
        if not a.skip_e2e:
            call_s = []
            for rep in range(3 + a.steps):             # three warm-up calls (allocator, pinned buffers, NCCL), then the timed ones
                barrier()
                t0 = time.perf_counter()
                dd = feats_pinned.to(dev, non_blocking=True)
                cen_e, lab_e, it_e = km.lloyd(dd, d_cen, max_iter=5, tol=0.0, update="fast", verbose=False)
                lab_host = dls._to_host(lab_e)
                barrier()
                if rep >= 3:
                    call_s.append(time.perf_counter() - t0)
                del dd
            dt = sharding.barrier_max_ms(float(np.mean(call_s)) * 1e3, dev) * 1e-3
            kres["e2e"] = {"value": 5 / dt, "unit": "iters/s", "calls": a.steps,
                           "call": "k_means.lloyd(max_iter=5) incl. H2D rows + final assignment + D2H labels",
                           "h2d_bytes_per_call": int(feats_pinned.numel() * 4 * 1), "d2h_bytes_per_call": int(lab_host.size * 4)}
        if orc is not None:
            rows = min(3_000_000, a.kmeans_rows)
            kr, kdt, _ = cpu_kmeans_sample(a, orc, feats[:rows], init)
            kres["cpu_baseline"] = {"value": kr, "unit": "iters/s", "cores": orc.max_threads(), "kind": "port",
                                    "sample": f"{rows} rows, 1 iteration ({kdt:.2f} s), time scaled to {a.kmeans_rows} rows"}
        del d_feats, feats_pinned, feats

    if rank == 0:
        sampler.stop()
    clocks = sampler.summary(t_wall0, time.time() if a.skip_kmeans else t_k1) if rank == 0 else None

    # ---- e2e lifting: public entry point, pinned host inputs, copies inside the timed region
    e2e = None
    if not a.skip_e2e:
        pos_pinned = torch.from_numpy(pos[lo:hi]).pin_memory()
        seg_list = [maps_pinned[v] for v in range(V)]
        steps_e = a.steps
        warm_e = 3                                     # W >= 3: allocator blocks and both pinned result buffers exist
        got = None
        per_call = []
        for i in range(warm_e + steps_e):
            if i == warm_e:
                barrier()
                t0 = time.perf_counter()
            tc = time.perf_counter()
            got = dls.lift_labels(pos_pinned, cams, seg_list, None, device=dev)      # returns host labels: synchronous
            if i >= warm_e:
                per_call.append((time.perf_counter() - tc) * 1e3)
        barrier()
        dt = (time.perf_counter() - t0) / steps_e
        dt = sharding.barrier_max_ms(dt * 1e3, dev) * 1e-3
        same = bool(np.array_equal(got, labels.cpu().numpy()))
        # bytes that crossed PCIe in the last call, counted by lift_labels from the tensors it copied
        # (job-wide: every rank uploads its share of the views and its own positions)
        st = dict(dls.last_call_stats)
        h2d = st["h2d_bytes"] * world if world > 1 else st["h2d_bytes"]
        if world > 1:
            staging = (f"every rank uploads and packs {V // world}-{-(-V // world)} of the {V} views in chunks of 16 and pushes each packed chunk "
                       f"into all ranks' buffers over peer memory while the next chunk crosses PCIe")
        else:
            staging = (f"{st['views_as_int32']} views cross as int32 and are packed on the device, {st['views_narrowed_on_host']} are narrowed "
                       f"to uint8 codes on the host cores meanwhile")
        e2e = {"value": a.gaussians * V / dt, "unit": UNIT, "ms_per_step": dt * 1e3, "calls": steps_e,
               "ms_per_call_rank0": [round(x, 2) for x in per_call],
               "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": a.gaussians * 4,
               "labels_equal_resident_run": same, "staging": staging,
               "call": "deep_learning_segmentation.lift_labels(positions, cameras, seg_maps) with pinned host int32 maps"}

    nxt = None
    if world == 1 and not a.skip_next:
        nxt = next_rows(a, gs, orc, pos, labels.cpu().numpy(), dev)

    if rank == 0:
        peak, peak_src = peak_hbm()
        alg_bytes = 16 * n_r + V * H * W
        ach = alg_bytes / (sweep_ms_max * 1e-3) / 1e9
        ach_step = alg_bytes / (ms_per_step * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_config(a),
            "dtype_note": "labels equal the reference's float64 evaluation bit for bit; every pair is screened in float32 with a proven error bound and re-evaluated in float64 when the bound cannot decide it (about 1 % of pairs)",
            "value_incl_pack": a.gaussians * V / ((ms_per_step + pack_ms) * 1e-3),
            "kernels_ms": {"prepare (ordering + per-tile verdicts)": prepare_ms, "lift_gather_kernel": sweep_ms,
                           "lift_majority_kernel": major_ms,
                           "note": "each phase timed alone with CUDA events; the timed step runs the same three phases back to back on one stream",
                           "pack_labels_all_views_staging (once per scene, not in value)": pack_ms},
            "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                         "traffic": ncu_traffic("lift_gather_kernel", world), "kernel": "lift_gather_kernel",
                         "algorithmic_bytes": alg_bytes, "peak_source": peak_src,
                         "note": "algorithmic bytes = 16 N_r + 1 V H W (SURVEY 8d, uint8 maps), one launch sweeps all views; the kernel is instruction-issue bound (float32 screening + float64 re-evaluation of undecided pairs), not HBM bound, see DESIGN.md; traffic is the ncu capture of this workload on one GPU"},
            "roofline_step": {"bound": "hbm", "achieved": ach_step, "peak": peak, "unit": "GB/s", "frac": ach_step / peak,
                              "note": "same algorithmic bytes over the whole step (prepare + gather + majority)"},
            "parity": parity,
            "cpu_baseline": cpu, "e2e": e2e, "kmeans": kres, "next_rows": nxt,
            "gpu_launches": int(n_lift_launches),
            "gpu_launches_note": "counted by the library (gsl_launch_count) around the timed lifting region; the radix sort's CUB kernels (5 per step) are not in the count",
            "clocks": clocks, "clocks_window": "lifting + k-means timed regions, nvidia-smi -lms 20", "label_histogram_head": label_hist,
        }
        print(json.dumps(line))
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, {name: t.cpu().numpy() for name, t in dump.items()})
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    a = parse_args()
    if a.impl == "reference":
        if a.dump_outputs:
            raise SystemExit("bench.py: --dump-outputs writes what the native arm computed; it has no meaning with --impl reference")
        run_reference(a)
    else:
        run_native(a)


if __name__ == "__main__":
    main()
