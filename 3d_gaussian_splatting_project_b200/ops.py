"""Host-side operators over libgslift.so.  PyTorch is used for device memory and streams only;
every computation below is a call through the C ABI of include/gslift.h.

Citations: dls = deep_learning_segmentation.py, km = 3D_clustering/k_means.py (reference).
"""
from __future__ import annotations

import numpy as np
import torch

from ._native import VIEW_DTYPE, check, lib

DEFAULT_LABEL_MIN = -1      # YOLO background / Mask2Former "no segment" (dls:101)
DEFAULT_N_CLASSES = 254     # codes 1..254 (GSL_MAX_CODES); covers ADE20K (150) and COCO (80) ids plus -1


def _require_cuda(t: torch.Tensor, name: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(f"{name} must live on a CUDA device (there is no CPU path)")
    if not t.is_contiguous():
        raise RuntimeError(f"{name} must be contiguous")


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


class _Workspace:
    """Per-device scratch tensor, grown on demand and reused across calls."""

    def __init__(self):
        self._buf = {}

    def get(self, device: torch.device, nbytes: int) -> torch.Tensor:
        key = (device.type, device.index)
        buf = self._buf.get(key)
        if buf is None or buf.numel() < nbytes:
            buf = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=device)
            self._buf[key] = buf
        return buf


_ws = _Workspace()


# --------------------------------------------------------------------------------------
# lifting
# --------------------------------------------------------------------------------------
def packed_map_bytes(seg_h: int, seg_w: int) -> int:
    """Bytes of one packed label map of seg_h x seg_w pixels (include/gslift.h: 16-pixel strips
    plus a ring of zero codes, followed by the coarse table of 8 x 8-pixel cells)."""
    strips_x = (int(seg_w) + 15) // 16 + 2
    rows_pad = ((int(seg_h) + 7) // 8 + 2) * 8
    coarse = (2 * strips_x * (rows_pad // 8) + 15) // 16 * 16        # one byte per 8 x 8-pixel cell
    return strips_x * rows_pad * 16 + coarse


def packed_offsets(map_shapes) -> np.ndarray:
    """Byte offset of every view's packed map when the maps are laid out back to back, plus
    the total as the last entry (int64 [V + 1])."""
    sizes = [packed_map_bytes(h, w) for h, w in map_shapes]
    return np.concatenate(([0], np.cumsum(sizes, dtype=np.int64))).astype(np.int64)


def make_views(cameras, map_shapes, image_sizes=None) -> np.ndarray:
    """Camera dicts (cameras.json schema, dls:54-63) -> GslView table.

    map_shapes[v] = (seg_h, seg_w) of view v's segmentation map (dls:267);
    image_sizes[v] = (orig_w, orig_h) of the opened image (dls:263), default the map size.
    `t` is evaluated with the reference's own expression `-R @ p` (dls:66) so it carries the
    same rounding the reference would see on this host.  Packed maps are laid out back to back
    (packed_offsets).
    """
    n = len(cameras)
    views = np.zeros(n, VIEW_DTYPE)
    if n == 0:
        return views
    shapes = np.array([[int(s) for s in sh] for sh in map_shapes], dtype=np.int64).reshape(n, 2)      # (seg_h, seg_w)
    images = shapes[:, ::-1] if image_sizes is None else np.array([[int(s) for s in sz] for sz in image_sizes], dtype=np.int64)
    R = np.array([cam["rotation"] for cam in cameras])
    p = np.array([cam["position"] for cam in cameras])
    if R.dtype != np.float64 or R.shape != (n, 3, 3) or p.dtype != np.float64 or p.shape != (n, 3):
        R = np.array([np.array(cam["rotation"], dtype=np.float64) for cam in cameras]).reshape(n, 3, 3)
        p = np.array([np.array(cam["position"], dtype=np.float64) for cam in cameras]).reshape(n, 3)
    views["R"] = R.reshape(n, 9)
    t = views["t"]
    for v in range(n):                       # one 3x3 matrix-vector product per camera, as the reference does it
        t[v] = -R[v] @ p[v]
    width = np.array([cam["width"] for cam in cameras])
    height = np.array([cam["height"] for cam in cameras])
    views["fx"] = [cam["fx"] for cam in cameras]
    views["fy"] = [cam["fy"] for cam in cameras]
    views["half_w"], views["half_h"] = width / 2, height / 2
    views["width"], views["height"] = width, height
    views["scale_x"] = shapes[:, 1] / images[:, 0]
    views["scale_y"] = shapes[:, 0] / images[:, 1]
    views["seg_w"], views["seg_h"] = shapes[:, 1], shapes[:, 0]
    views["map_offset"] = packed_offsets([(int(h), int(w)) for h, w in shapes])[:-1]
    return views


def _runs(shapes, v0, v1):
    """(first view, count) of the runs of equal map shapes among views [v0, v1): one pack launch each."""
    v = v0
    while v < v1:
        n = 1
        while v + n < v1 and shapes[v + n] == shapes[v]:
            n += 1
        yield v, n
        v += n


def pack_labels(maps: torch.Tensor, shapes=None, label_min: int = DEFAULT_LABEL_MIN,
                n_classes: int = DEFAULT_N_CLASSES, out: torch.Tensor | None = None,
                check_range: bool = True) -> torch.Tensor:
    """int32 label maps (device) -> uint8 codes `label - label_min + 1` in the library's tiled
    layout, maps back to back (packed_offsets).

    maps    [n, h, w] or [h, w] tensor, or a flat tensor together with `shapes` = [(h, w), ...]
            listing the row-major maps it holds back to back.
    """
    _require_cuda(maps, "maps")
    if maps.dtype != torch.int32:
        raise TypeError("maps must be int32 (what segment_image returns, dls:158)")
    if shapes is None:
        if maps.dim() == 2:
            shapes = [tuple(maps.shape)]
        elif maps.dim() == 3:
            shapes = [tuple(maps.shape[1:])] * maps.shape[0]
        else:
            raise ValueError("flat maps need shapes=[(h, w), ...]")
    shapes = [(int(h), int(w)) for h, w in shapes]
    if sum(h * w for h, w in shapes) != maps.numel():
        raise ValueError("shapes do not add up to maps.numel()")
    offs = packed_offsets(shapes)
    if out is None:
        out = torch.empty(int(offs[-1]), dtype=torch.uint8, device=maps.device)
    elif out.numel() < int(offs[-1]) or out.dtype != torch.uint8:
        raise ValueError(f"out must be uint8 with at least {int(offs[-1])} elements")
    err = torch.zeros(1, dtype=torch.int32, device=maps.device)
    flat = maps.reshape(-1)
    L = lib()
    with torch.cuda.device(maps.device):
        src = 0
        for v, n in _runs(shapes, 0, len(shapes)):
            h, w = shapes[v]
            check(L.gsl_pack_labels(flat.data_ptr() + 4 * src, n, w, h, out.data_ptr() + int(offs[v]),
                                    int(label_min), int(n_classes), err.data_ptr(), _stream()))
            src += n * h * w
    if check_range and int(err.item()) != 0:
        raise ValueError(f"label map value outside [{label_min}, {label_min + n_classes})")
    return out


def label_range(maps: torch.Tensor):
    """(min, max) of an int32 device tensor, computed on the device."""
    _require_cuda(maps, "maps")
    mm = torch.tensor([2**31 - 1, -2**31], dtype=torch.int32, device=maps.device)
    with torch.cuda.device(maps.device):
        check(lib().gsl_label_range(maps.data_ptr(), maps.numel(), mm.data_ptr(), _stream()))
    lo, hi = (int(v) for v in mm.tolist())
    return lo, hi


def _check_lift(pos: torch.Tensor, views: np.ndarray, packed: torch.Tensor | None):
    _require_cuda(pos, "pos")
    if pos.dtype != torch.float32 or pos.dim() != 2 or pos.shape[1] != 3:
        raise TypeError("pos must be float32 [N, 3]")
    views = np.ascontiguousarray(views)
    if views.dtype != VIEW_DTYPE:
        raise TypeError("views must come from make_views")
    if len(views) and packed is not None:
        _require_cuda(packed, "packed")
        need = max(int(r["map_offset"]) + packed_map_bytes(int(r["seg_h"]), int(r["seg_w"])) for r in views)
        if packed.numel() < need:
            raise ValueError(f"packed holds {packed.numel()} bytes, views address {need}")
    return views


def lift_near(pos: torch.Tensor, views: np.ndarray, near_eps: float = 1e-4) -> torch.Tensor:
    """uint8 [N]: 1 where some (Gaussian, view) lies within near_eps of a decision edge -- the set
    the parity criterion exempts from bit-exactness (float64, every pair)."""
    views = _check_lift(pos, views, None)
    N, V = pos.shape[0], len(views)
    near = torch.empty(N, dtype=torch.uint8, device=pos.device)
    L = lib()
    ws = _ws.get(pos.device, L.gsl_lift_workspace_bytes(N, V))
    with torch.cuda.device(pos.device):
        check(L.gsl_lift_near(pos.data_ptr(), N, views.ctypes.data, V, near.data_ptr(), float(near_eps),
                              ws.data_ptr(), ws.numel(), _stream()))
    return near


def lift_votes(pos: torch.Tensor, views: np.ndarray, packed: torch.Tensor,
               label_min: int = DEFAULT_LABEL_MIN, n_classes: int = DEFAULT_N_CLASSES,
               want_near: bool = False, near_eps: float = 1e-4,
               out: torch.Tensor | None = None):
    """Vote loop + majority of assign_labels (dls:255-306) on precomputed, packed maps.

    pos float32 [N,3] (device), views from make_views, packed uint8 (device).
    Returns labels int32 [N] (device); with want_near also a uint8 [N] near-boundary mask.
    """
    views = _check_lift(pos, views, packed)
    N, V = pos.shape[0], len(views)
    labels = out if out is not None else torch.empty(N, dtype=torch.int32, device=pos.device)
    near = torch.empty(N, dtype=torch.uint8, device=pos.device) if want_near else None
    L = lib()
    ws = _ws.get(pos.device, L.gsl_lift_workspace_bytes(N, V))
    with torch.cuda.device(pos.device):
        check(L.gsl_lift_votes(pos.data_ptr(), N, views.ctypes.data, V,
                               packed.data_ptr() if V else None, int(label_min), int(n_classes),
                               labels.data_ptr(), near.data_ptr() if want_near else None,
                               float(near_eps), ws.data_ptr(), ws.numel(), _stream()))
    return (labels, near) if want_near else labels


def lift_phases(pos: torch.Tensor, views: np.ndarray, packed: torch.Tensor,
                label_min: int = DEFAULT_LABEL_MIN, n_classes: int = DEFAULT_N_CLASSES,
                out: torch.Tensor | None = None, best: torch.Tensor | None = None):
    """lift_votes as its ABI steps.  Returns (run_prepare, run_gather, run_majority, run_sweep, labels):
    zero-argument callables that enqueue gsl_lift_prepare (ordering + per-tile verdicts; reads no
    maps), gsl_lift_gather (projection + visibility + gather into the vote sheet) and
    gsl_lift_majority on the current stream (benchmarks put events between them); run_sweep is
    gsl_lift_sweep = the gather over all Gaussians, then the majority over all of them, back to back
    on the same stream (the two steps lift_votes runs after the prepare step)."""
    views = _check_lift(pos, views, packed)
    N, V = pos.shape[0], len(views)
    labels = out if out is not None else torch.empty(N, dtype=torch.int32, device=pos.device)
    L = lib()
    ws = _ws.get(pos.device, L.gsl_lift_workspace_bytes(N, V))

    def run_prepare():
        check(L.gsl_lift_prepare(pos.data_ptr(), N, views.ctypes.data, V, ws.data_ptr(), ws.numel(), _stream()))

    def run_gather():
        check(L.gsl_lift_gather(pos.data_ptr(), N, views.ctypes.data, V, packed.data_ptr() if V else None,
                                ws.data_ptr(), ws.numel(), _stream()))

    def run_majority():
        check(L.gsl_lift_majority(N, V, int(label_min), int(n_classes), labels.data_ptr(),
                                  best.data_ptr() if best is not None else None, ws.data_ptr(), ws.numel(), _stream()))

    def run_sweep():
        check(L.gsl_lift_sweep(pos.data_ptr(), N, views.ctypes.data, V, packed.data_ptr() if V else None,
                               int(label_min), int(n_classes), labels.data_ptr(),
                               best.data_ptr() if best is not None else None, ws.data_ptr(), ws.numel(), _stream()))

    return run_prepare, run_gather, run_majority, run_sweep, labels


def lift_merge(labels: torch.Tensor, best: torch.Tensor, labels_b: torch.Tensor, best_b: torch.Tensor):
    """In place: (labels, best) <- whichever of the two candidates has the larger vote key (more
    votes, earlier first sighting on a tie: the reference's rule across label ranges)."""
    for name, x in (("labels", labels), ("best", best), ("labels_b", labels_b), ("best_b", best_b)):
        _require_cuda(x, name)
    with torch.cuda.device(labels.device):
        check(lib().gsl_lift_merge(labels.data_ptr(), best.data_ptr(), labels_b.data_ptr(), best_b.data_ptr(),
                                   labels.numel(), _stream()))
    return labels, best


# --------------------------------------------------------------------------------------
# K-means
# --------------------------------------------------------------------------------------
def _check_kmeans(data: torch.Tensor, centroids: torch.Tensor):
    _require_cuda(data, "data")
    _require_cuda(centroids, "centroids")
    if data.dtype != torch.float32 or centroids.dtype != torch.float32:
        raise TypeError("data and centroids must be float32 (km:109)")
    if data.dim() != 2 or centroids.dim() != 2 or data.shape[1] != centroids.shape[1]:
        raise ValueError("data [N,D] and centroids [K,D] must agree on D")
    return data.shape[0], data.shape[1], centroids.shape[0]


def kmeans_assign(data: torch.Tensor, centroids: torch.Tensor, out: torch.Tensor | None = None):
    """labels int32 [N]: nearest centroid, scipy-order float64 distance (km:116-122)."""
    N, D, K = _check_kmeans(data, centroids)
    labels = out if out is not None else torch.empty(N, dtype=torch.int32, device=data.device)
    L = lib()
    ws = _ws.get(data.device, L.gsl_kmeans_workspace_bytes(N, D, K))
    with torch.cuda.device(data.device):
        check(L.gsl_kmeans_assign(data.data_ptr(), N, D, centroids.data_ptr(), K, labels.data_ptr(),
                                  ws.data_ptr(), ws.numel(), _stream()))
    return labels


def kmeans_step(data: torch.Tensor, centroids: torch.Tensor, labels: torch.Tensor | None = None,
                sums: torch.Tensor | None = None):
    """Assignment fused with per-cluster float64 sums/counts.  Returns (labels, sums[K,D+1])."""
    N, D, K = _check_kmeans(data, centroids)
    if labels is None:
        labels = torch.empty(N, dtype=torch.int32, device=data.device)
    if sums is None:
        sums = torch.empty((K, D + 1), dtype=torch.float64, device=data.device)
    L = lib()
    ws = _ws.get(data.device, L.gsl_kmeans_workspace_bytes(N, D, K))
    with torch.cuda.device(data.device):
        check(L.gsl_kmeans_step(data.data_ptr(), N, D, centroids.data_ptr(), K, labels.data_ptr(),
                                sums.data_ptr(), ws.data_ptr(), ws.numel(), _stream()))
    return labels, sums


def kmeans_finalize(sums: torch.Tensor, old: torch.Tensor, new: torch.Tensor | None = None,
                    shift: torch.Tensor | None = None):
    """(new centroids f32 [K,D], shift f32 [1]) from reduced sums (km:125-131)."""
    _require_cuda(sums, "sums")
    _require_cuda(old, "old")
    K, D = old.shape
    if sums.dtype != torch.float64 or tuple(sums.shape) != (K, D + 1):
        raise ValueError("sums must be float64 [K, D+1]")
    if new is None:
        new = torch.empty_like(old)
    if shift is None:
        shift = torch.empty(1, dtype=torch.float32, device=old.device)
    with torch.cuda.device(old.device):
        check(lib().gsl_kmeans_finalize(sums.data_ptr(), old.data_ptr(), K, D, new.data_ptr(),
                                        shift.data_ptr(), _stream()))
    return new, shift


class KMeansExchange:
    """Per-job state of the fused K-means exchange (gsl_kmeans_step_exchange): this rank's exchange
    buffer, everybody's peer-mapped pointers to it, and the call counter.

    world == 1: an ordinary device buffer.  world > 1: a torch symmetric-memory allocation
    (CUDA peer mapping over NVLink) rendezvoused over the process group, so that every rank's
    kernel can store its partial sums straight into every other rank's buffer."""

    def __init__(self, K: int, D: int, device: torch.device, group=None):
        import ctypes
        import torch.distributed as dist
        self.K, self.D, self.device = int(K), int(D), torch.device(device)
        self.world = dist.get_world_size(group) if (dist.is_available() and dist.is_initialized()) else 1
        self.rank = dist.get_rank(group) if self.world > 1 else 0
        nbytes = lib().gsl_kmeans_exchange_bytes(self.world, self.D, self.K)
        if nbytes == 0:
            raise ValueError(f"unsupported exchange shape: world={self.world}, K={K}, D={D}")
        if self.world > 1:
            import torch.distributed._symmetric_memory as symm_mem
            grp = group if group is not None else dist.group.WORLD
            self.buf = symm_mem.empty(nbytes, dtype=torch.uint8, device=self.device)
            self.buf.zero_()
            self._handle = symm_mem.rendezvous(self.buf, grp.group_name)
            ptrs = [int(p) for p in self._handle.buffer_ptrs]
            torch.cuda.synchronize(self.device)
            dist.barrier(group=grp)                # every buffer is zeroed before anyone pushes into it
        else:
            self.buf = torch.zeros(nbytes, dtype=torch.uint8, device=self.device)
            ptrs = [self.buf.data_ptr()]
        self._ptrs = (ctypes.c_void_p * self.world)(*ptrs)
        self.seq = 0
        self.sums = torch.empty((self.K, self.D + 1), dtype=torch.float64, device=self.device)

    def step(self, data: torch.Tensor, centroids: torch.Tensor, labels: torch.Tensor,
             new: torch.Tensor | None = None, shift: torch.Tensor | None = None):
        """One sharded Lloyd pass; returns (new centroids, shift); self.sums holds the totals.
        A collective: every rank of the group must call it."""
        N, D, K = _check_kmeans(data, centroids)
        if (K, D) != (self.K, self.D):
            raise ValueError("exchange was built for a different K, D")
        if new is None:
            new = torch.empty_like(centroids)
        if shift is None:
            shift = torch.empty(1, dtype=torch.float32, device=data.device)
        L = lib()
        ws = _ws.get(data.device, L.gsl_kmeans_workspace_bytes(N, D, K))
        self.seq += 1
        with torch.cuda.device(data.device):
            check(L.gsl_kmeans_step_exchange(data.data_ptr(), N, D, centroids.data_ptr(), K, labels.data_ptr(),
                                             self.rank, self.world, self._ptrs, self.seq, new.data_ptr(),
                                             shift.data_ptr(), self.sums.data_ptr(), ws.data_ptr(), ws.numel(), _stream()))
        return new, shift


def kmeans_update_ordered(data: torch.Tensor, labels: torch.Tensor, old: torch.Tensor, validate: bool = False):
    """Reference-order float32 sequential mean (km:125-128 bit for bit).  Single device.
    Labels outside [0, K) are skipped by the kernels and turn the shift into NaN; validate=True
    waits for the result and raises GslError(GSL_ERANGE) in that case."""
    N, D, K = _check_kmeans(data, old)
    _require_cuda(labels, "labels")
    if labels.dtype != torch.int32 or labels.numel() != N:
        raise TypeError("labels must be int32 [N]")
    new = torch.empty_like(old)
    shift = torch.empty(1, dtype=torch.float32, device=old.device)
    L = lib()
    ws = _ws.get(data.device, L.gsl_kmeans_workspace_bytes(N, D, K))
    with torch.cuda.device(data.device):
        check(L.gsl_kmeans_update_ordered(data.data_ptr(), labels.data_ptr(), N, D, K, old.data_ptr(),
                                          new.data_ptr(), shift.data_ptr(), ws.data_ptr(), ws.numel(), _stream()))
    if validate and bool(torch.isnan(shift).item()) and bool(((labels < 0) | (labels >= K)).any().item()):
        from ._native import GslError
        raise GslError(-4, f"gsl_kmeans_update_ordered: a label lies outside [0, {K})")
    return new, shift


def recolor(labels: torch.Tensor, palette: torch.Tensor, colors: torch.Tensor):
    """colors[i] = palette[labels[i] % 8] in place (km:99-101, :147-149)."""
    _require_cuda(labels, "labels")
    _require_cuda(colors, "colors")
    _require_cuda(palette, "palette")
    if palette.dtype != torch.float32 or palette.numel() != 24 or colors.dtype != torch.float32:
        raise TypeError("palette must be float32 [8,3], colors float32 [N,3]")
    with torch.cuda.device(labels.device):
        check(lib().gsl_recolor(labels.data_ptr(), labels.numel(), palette.data_ptr(), colors.data_ptr(), _stream()))
    return colors
