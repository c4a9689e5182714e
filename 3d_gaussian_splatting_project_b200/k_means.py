"""Drop-in for the reference's `3D_clustering/k_means.py`: same functions, prints and CLI, with
the per-point KDTree loop and the per-cluster boolean-mask means replaced by GPU kernels.

    get_vertex_info, k_means_kd_tree, k_means_with_color, add_label_proberty, COLORS

Semantics kept from the reference (line numbers are the reference's):
  * init draws `np.random.choice(N, k, replace=False)` from the GLOBAL NumPy stream (:63, :111),
    so `np.random.seed(s)` before the call gives the reference's start;
  * every iteration prints its index and the centroid shift (:66/:83, :114/:131);
  * on convergence it prints "Converged after i iterations." and breaks BEFORE adopting the new
    centroids (:84-88, :132-136), so the final assignment uses the pre-update centroids;
  * an empty cluster keeps its old centroid (:78, :126);
  * labels come back as int64, centroids float32, `colors` recoloured in place with
    COLORS[c % 8] (divided by 255.0 only in k_means_with_color, :100 vs :148).

`update=` selects how the mean is formed:
  "ordered" (default on one GPU)  NumPy's arithmetic: a float32 sum from +0.0, sequential in index
            order for D >= 2 and NumPy's pairwise sum for D = 1; bit-identical centroids, hence
            identical trajectories;
  "fast"    float64 segmented sums, shardable; centroids agree with the reference to its own
            float32 rounding (about 1e-5 relative on clusters of 1e5 members).
Under torch.distributed (world size > 1) `lloyd` is the sharded entry point: each rank passes ITS
rows and the SAME centroids, and `update` is forced to "fast" (the reference entry points broadcast
rank 0's initial draw before they call it); the partial sums and counts are exchanged inside the reduction kernel over peer memory
(ops.KMeansExchange -> gsl_kmeans_step_exchange).  GSLIFT_KMEANS_EXCHANGE=nccl selects the
three-step form instead (reduce kernel, NCCL all-reduce of K x (D+1) float64, finalize kernel),
which is also what is used when torch cannot set up symmetric memory on the machine.
"""
from __future__ import annotations

import argparse
import os

import numpy as np
import torch

from . import ops, plyio

COLORS = [[252, 199, 55], [242, 107, 15], [231, 56, 121], [126, 24, 145],
          [247, 44, 91], [255, 116, 139], [167, 212, 119], [228, 241, 172]]


def get_vertex_info(plydata):
    """(points [N,3], colors [N,3]) from x/y/z and f_dc_0..2, printing both (reference :10-31)."""
    vertex = plydata["vertex"]
    points = np.column_stack((vertex["x"], vertex["y"], vertex["z"]))
    colors = np.column_stack((vertex["f_dc_0"], vertex["f_dc_1"], vertex["f_dc_2"]))
    print(points)
    print(colors)
    return points, colors


def _dist_world():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        return dist
    return None


_exchanges = {}


def _make_exchange(centroids, dist):
    """The fused exchange for this (K, D, device), or None when the three-step NCCL form is asked
    for (GSLIFT_KMEANS_EXCHANGE=nccl) or symmetric memory cannot be set up.  Cached: the buffers are
    a collective allocation."""
    if os.environ.get("GSLIFT_KMEANS_EXCHANGE", "peer") == "nccl":
        return None
    key = (centroids.shape[0], centroids.shape[1], str(centroids.device), dist is not None)
    if key not in _exchanges:
        try:
            _exchanges[key] = ops.KMeansExchange(centroids.shape[0], centroids.shape[1], centroids.device)
        except Exception as exc:       # symmetric memory unavailable (no peer access, old torch): NCCL
            import sys
            if dist is None:
                raise
            print(f"gslift: peer-memory exchange unavailable ({exc}); using NCCL all-reduce", file=sys.stderr)
            _exchanges[key] = None
    return _exchanges[key]


_LOOKAHEAD = 2      # iterations enqueued before the shift of an earlier one is read back (lloyd)


def lloyd(data, centroids, max_iter=100, tol=1e-4, update=None, verbose=True, device=None):
    """The iteration shared by both reference entry points, on device tensors.

    data float32 [N,D] (this rank's rows), centroids float32 [K,D] (replicated).
    Returns (centroids, labels int32 device tensor, iterations run).

    The device never waits for the host: every iteration's shift (km:131) travels to a pinned
    host word asynchronously and is read -- and printed, in order -- `GSLIFT_LLOYD_LOOKAHEAD`
    (default 2) iterations later, while the next iterations are already enqueued.  When an
    earlier iteration turns out to have converged, the iterations enqueued past it are simply
    discarded: the reference breaks BEFORE adopting the new centroids (km:132-136), so the result
    is the centroid set that iteration was given.  Under torch.distributed every rank sees the same
    shifts and makes the same decisions, so all ranks issue the same exchanges."""
    dist = _dist_world()
    if update is None:
        update = os.environ.get("GSLIFT_KMEANS_UPDATE", "ordered")
    if dist is not None:
        update = "fast"
    if update not in ("ordered", "fast"):
        raise ValueError(f"update must be 'ordered' or 'fast', not {update!r}")
    labels = torch.empty(data.shape[0], dtype=torch.int32, device=data.device)
    sums = torch.empty((centroids.shape[0], centroids.shape[1] + 1), dtype=torch.float64, device=data.device)
    exchange = _make_exchange(centroids, dist) if update == "fast" else None
    if exchange is not None and exchange.world > 1:
        # ranks may arrive seconds apart (I/O, garbage collection); the in-kernel exchange waits for
        # peers with a bounded spin, so line the ranks up before the first one
        dist.barrier()
    depth = max(int(os.environ.get("GSLIFT_LLOYD_LOOKAHEAD", _LOOKAHEAD)), 0)
    pinned = torch.empty(depth + 1, dtype=torch.float32, pin_memory=True)
    stream = torch.cuda.current_stream(data.device)
    pending = []                     # (iteration, centroids it was given, centroids it produced, pinned slot, event)
    done, final = 0, None

    def settle(entry):
        """Read one iteration's shift; True when it converged (km:131-136)."""
        nonlocal done, final
        iteration, given, produced, slot, ev = entry
        ev.synchronize()
        shift_value = np.float32(pinned[slot].item())
        if exchange is not None and exchange.world > 1 and np.isnan(shift_value):
            raise RuntimeError("K-means exchange returned a NaN shift: a rank did not reach the exchange within the time-out "
                               "(GSLIFT_EXCHANGE_TIMEOUT_MS; every rank must call lloyd with the same max_iter/tol), or the data is not finite")
        done = iteration + 1
        if verbose:
            print(iteration)
            print(shift_value)
        if shift_value < tol:
            if verbose:
                print(f"Converged after {iteration + 1} iterations.")
            final = given
            return True
        final = produced
        return False

    converged = False
    for iteration in range(max_iter):
        if exchange is not None:
            new_centroids, shift = exchange.step(data, centroids, labels)
        elif update == "fast":
            ops.kmeans_step(data, centroids, labels, sums)
            if dist is not None:
                dist.all_reduce(sums)                       # K x (D+1) float64 over NCCL
            new_centroids, shift = ops.kmeans_finalize(sums, centroids)
        else:
            ops.kmeans_assign(data, centroids, labels)
            new_centroids, shift = ops.kmeans_update_ordered(data, labels, centroids)
        slot = iteration % (depth + 1)
        pinned[slot:slot + 1].copy_(shift, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(stream)
        pending.append((iteration, centroids, new_centroids, slot, ev))
        centroids = new_centroids
        while len(pending) > depth and not converged:
            converged = settle(pending.pop(0))
        if converged:
            break
    while pending and not converged:
        converged = settle(pending.pop(0))
    if final is None:                                       # max_iter == 0
        final = centroids
    ops.kmeans_assign(data, final, labels)
    return final, labels, done


def _run(data_np, k, colors, max_iter, tol, palette_scale, update):
    data_np = np.ascontiguousarray(data_np, dtype=np.float32)
    N, _ = data_np.shape
    start = data_np[np.random.choice(N, k, replace=False)]
    device = torch.device("cuda")
    data = torch.from_numpy(data_np).to(device)
    start_dev = torch.from_numpy(start).to(device)
    dist = _dist_world()
    if dist is not None:
        # lloyd() needs the SAME centroids on every rank; each rank drew from its own rows and its
        # own NumPy stream, so rank 0's draw is the one everybody uses
        dist.broadcast(start_dev, src=0)
    centroids, labels, _ = lloyd(data, start_dev, max_iter, tol, update)
    palette = (np.array(COLORS) / 255.0 if palette_scale else np.array(COLORS)).astype(np.float32)
    if colors.dtype == np.float32:
        colors_dev = torch.from_numpy(np.ascontiguousarray(colors)).to(device)
        ops.recolor(labels, torch.from_numpy(palette).to(device), colors_dev)
    else:   # the reference assigns the float64 palette into whatever dtype `colors` has
        wide = np.array(COLORS) / 255.0 if palette_scale else np.array(COLORS)
        pal = torch.from_numpy(wide.astype(colors.dtype)).to(device)
        colors_dev = pal[labels.long() % len(COLORS)]
    colors[...] = colors_dev.cpu().numpy()
    return centroids.cpu().numpy(), labels.cpu().numpy().astype(np.int64), colors


def k_means_kd_tree(data, k, colors, max_iter=100, tol=1e-4, update=None):
    """K-means on an arbitrary feature block [N,D] (reference :46-103)."""
    return _run(data, k, colors, max_iter, tol, False, update)


def k_means_with_color(points, k, colors, max_iter=100, tol=1e-4, update=None):
    """K-means on concat(points, colors) (reference :107-151)."""
    data = np.concatenate((points, colors), axis=1)
    return _run(data, k, colors, max_iter, tol, True, update)


def add_label_proberty(ply_data, output_ply, label):
    """Append an int32 `label` property and write an ASCII PLY (reference :169-194)."""
    vertex = plyio.describe_with_label(ply_data["vertex"].data, label)
    plyio.write_ply(output_ply, [("vertex", vertex)], text=True)
    print(f"New PLY file with label added saved to {output_ply}")


def main(argv=None):
    parser = argparse.ArgumentParser(description="K-means clustering on a point cloud.")
    parser.add_argument("--file_path", type=str, required=True, help="Path to the input PLY file.")
    parser.add_argument("--save_path", type=str, required=True, help="Path to save the modified PLY file.")
    parser.add_argument("--k", type=int, default=10, help="Number of clusters for k-means.")
    args = parser.parse_args(argv)

    with open(args.file_path, "rb") as fh:
        plydata = plyio.read_ply(fh)
    points, colors = get_vertex_info(plydata)
    _, labels, colors = k_means_with_color(points, args.k, colors, max_iter=10)
    print(labels)
    add_label_proberty(plydata, args.save_path, labels)


if __name__ == "__main__":
    main()
