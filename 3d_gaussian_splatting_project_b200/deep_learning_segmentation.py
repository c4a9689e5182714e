"""Drop-in for the reference's `deep_learning_segmentation.py` with the N x V vote loop moved to
the GPU library.  Same public names, signatures, prints, CLI flags and output file:

    load_cameras, load_gaussians, project_gaussian, assign_labels, save_labeled_ply, main

What changed: `assign_labels` no longer walks Gaussians in Python (reference :274-306).  It
still visits the cameras in order, still skips a camera whose `<input_dir>/<img_name>.png` is
missing with the same warning (:257-259), still asks the 2-D segmenter for one map per view
(:266) -- but each map is uploaded and packed as it arrives and one `lift_votes` call
(include/gslift.h) produces the labels.

The 2-D segmentation stage itself (SegFormer / Mask2Former / YOLO inference, reference
:85-238) is upstream of this path and is not re-implemented.  `assign_labels` finds a
segmenter in this order:
  1. the `segmenter=` argument: callable(image_path, output_dir, model_type) -> int array [H, W]
  2. with GSLIFT_REUSE_SEGMAPS=1 only: a precomputed `<output_dir>/<img_name>_segmap.npy`, the
     file the reference's `segment_image` writes for every view (:165); the reference itself
     always recomputes, so reuse is opt-in and announced per view
  3. the reference's own `initialize_model` / `segment_image`, imported from the checkout
     named by $GSLIFT_REFERENCE_DIR
"""
from __future__ import annotations

import argparse
import importlib.util
import json
import os

import numpy as np
import torch
from PIL import Image

from . import ops, plyio

GAUSSIAN_DTYPE = np.dtype([("position", np.float32, 3), ("scale", np.float32, 3), ("rotation", np.float32, 4)])


def load_cameras(camera_file):
    """cameras.json -> list of dicts (reference :17-22)."""
    with open(camera_file, "r") as fh:
        return json.load(fh)


def load_gaussians(ply_file):
    """PLY -> (structured array with `position` filled from x/y/z, parsed PLY) (reference :25-40).
    `scale` and `rotation` stay zero, as in the reference."""
    ply = plyio.read_ply(ply_file)
    vertex = ply["vertex"]
    gaussians = np.zeros(len(vertex), dtype=GAUSSIAN_DTYPE)
    for axis, name in enumerate(("x", "y", "z")):
        gaussians["position"][:, axis] = vertex[name]
    return gaussians, ply


def project_gaussian(position, camera):
    """Scalar projection of one Gaussian mean (reference :43-82): (int x, int y) or None.
    Kept for API parity; the fast path evaluates the same float64 expressions on the GPU."""
    R = np.array(camera["rotation"])
    cam = R @ position + (-R @ np.array(camera["position"]))
    if cam[2] <= 0:
        return None
    w, h = camera["width"], camera["height"]
    u = (camera["fx"] * cam[0] / cam[2]) + w / 2
    v = (camera["fy"] * cam[1] / cam[2]) + h / 2
    if 0 <= u < w and 0 <= v < h:
        return (int(u), int(v))
    return None


# ----------------------------------------------------------------------------------------
# segmenter plumbing (upstream stage, not part of the hot path)
# ----------------------------------------------------------------------------------------
_ref_module = None


def _reference_module():
    """Import the reference's deep_learning_segmentation.py by path (for its segmenter)."""
    global _ref_module
    if _ref_module is None:
        root = os.environ.get("GSLIFT_REFERENCE_DIR")
        path = os.path.join(root, "deep_learning_segmentation.py") if root else None
        if not path or not os.path.exists(path):
            raise RuntimeError(
                "no segmenter: pass segmenter=..., provide <output_dir>/<img_name>_segmap.npy, or set "
                "GSLIFT_REFERENCE_DIR to a checkout of the reference (its segment_image is used unchanged)")
        spec = importlib.util.spec_from_file_location("_gslift_reference_dls", path)
        _ref_module = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(_ref_module)
    return _ref_module


class _UpstreamSegmenter:
    """Lazily builds the reference's model once and calls its segment_image per view."""

    def __init__(self, model_type):
        self.model_type = model_type
        self._state = None

    def __call__(self, image_path, output_dir, model_type):
        ref = _reference_module()
        if self._state is None:
            device = torch.device("cuda" if torch.cuda.is_available() else "cpu")
            processor, model = ref.initialize_model(self.model_type, device)
            model.to(device)
            self._state = (processor, model, device)
        processor, model, device = self._state
        return ref.segment_image(image_path, output_dir, processor, model, device, model_type)


def _precomputed_map(output_dir, img_name):
    """<output_dir>/<img_name>_segmap.npy, the file the reference's segment_image writes (:165).
    The reference recomputes (and overwrites) it on every run; reusing it is therefore opt-in:
    GSLIFT_REUSE_SEGMAPS=1, announced per view."""
    if os.environ.get("GSLIFT_REUSE_SEGMAPS") != "1":
        return None
    path = os.path.join(output_dir, f"{img_name}_segmap.npy") if output_dir else None
    if path and os.path.exists(path):
        print(f"Using precomputed segmentation map {path}")
        return np.load(path)
    return None


# ----------------------------------------------------------------------------------------
# the hot path
# ----------------------------------------------------------------------------------------
_side_streams = {}                 # per (device, role): the copy stream of the uploads, the push stream of the peer pushes
last_call_stats = {}               # bytes lift_labels moved over PCIe in its last call (this process)
_pinned_codes = {}                 # pinned uint8 staging for host-narrowed views (grown to the largest scene seen)
_host_stage = {"px_per_s": None, "fixed_s": 0.008}   # calibrated by use: host narrowing rate (pixels per second, all
                                                      # threads, with the DMA engine running) and the other host time of a call
_PCIE_BYTES_PER_S = 54e9           # pinned host -> device copy rate of a PCIe 5 x16 link (profiles/probes/h2d_probe.py)
_symm_packed = {}                  # per (device, bytes): symmetric-memory packed buffer of the multi-rank staging
CH = 16                            # views per staging chunk


def _dist():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        return dist, dist.get_world_size(), dist.get_rank()
    return None, 1, 0


def _side_stream(device, role):
    key = (device.type, device.index, role)
    if key not in _side_streams:
        _side_streams[key] = torch.cuda.Stream(device)
    return _side_streams[key]


def _host_cores():
    """Host cores this process may run on (affinity / cgroup aware where the platform tells)."""
    try:
        return len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        return os.cpu_count() or 1


def _host_fraction(seg_maps, n_px):
    """Share of the views whose maps are narrowed to 1-byte codes on the host before they cross
    the bus.  The DMA engine moves 4 bytes per pixel for the others meanwhile; with P pixels in all,
    tp = bus time per byte, th = host time per pixel and c = the other host work of the call
    (enqueueing, the view table), both sides finish together when
        c + f P th = P tp (4 - 3 f)   =>   f = (4 P tp - c) / (P (th + 3 tp)).
    GSLIFT_HOST_STAGE=<fraction> fixes it (0 = all maps cross as int32)."""
    if any(isinstance(m, torch.Tensor) and m.is_cuda for m in seg_maps):
        return 0.0
    env = os.environ.get("GSLIFT_HOST_STAGE")
    if env is not None:
        return min(max(float(env), 0.0), 1.0)
    cores = _host_cores()
    if cores < 8:
        return 0.0
    rate = _host_stage["px_per_s"] or 0.9e9 * cores
    tp, th, c = 1.0 / _PCIE_BYTES_PER_S, 1.0 / rate, _host_stage["fixed_s"]
    if n_px <= 0:
        return 0.0
    return min(max((4 * n_px * tp - c) / (n_px * (th + 3 * tp)), 0.0), 0.85)


def _host_ptr(m):
    """(address, keep-alive) of a host int32 map, converting only if it is not int32 / contiguous."""
    if isinstance(m, torch.Tensor):
        t = m if (m.dtype == torch.int32 and m.is_contiguous()) else m.to(torch.int32).contiguous()
        return t.data_ptr(), t
    arr = m if (isinstance(m, np.ndarray) and m.dtype == np.int32 and m.flags.c_contiguous) else np.ascontiguousarray(m, np.int32)
    return arr.ctypes.data, arr


def _as_int32_tensor(m):
    return m if isinstance(m, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(m, np.int32))


def _copy_views(seg_maps, sizes, v0, v1, dst):
    """Enqueue (current stream) the copies of maps [v0, v1) into the flat int32 device tensor `dst`;
    maps that lie back to back in one host allocation (slices of one big pinned tensor) cross in a
    single copy.  Returns the number of pixels."""
    off, v = 0, v0
    while v < v1:
        src = _as_int32_tensor(seg_maps[v])
        n, last = sizes[v], v
        if src.dtype == torch.int32 and src.is_contiguous() and not src.is_cuda:
            while last + 1 < v1:
                nxt = seg_maps[last + 1]
                if not (isinstance(nxt, torch.Tensor) and nxt.dtype == torch.int32 and nxt.is_contiguous() and not nxt.is_cuda
                        and nxt.untyped_storage().data_ptr() == src.untyped_storage().data_ptr()
                        and nxt.storage_offset() == src.storage_offset() + n):
                    break
                last += 1
                n += sizes[last]
            flat = torch.as_strided(src, (n,), (1,), src.storage_offset())
        else:
            flat = src.reshape(-1)
        dst[off:off + n].copy_(flat, non_blocking=True)
        off += n
        v = last + 1
    return off


def _upload_all(seg_maps, shapes, device):
    """Every map, uploaded (current stream) as one flat int32 device tensor."""
    sizes = [h * w for h, w in shapes]
    staged = torch.empty(int(sum(sizes)), dtype=torch.int32, device=device)
    _copy_views(seg_maps, sizes, 0, len(seg_maps), staged)
    return staged


def _chunk_plan(shapes, host_fraction):
    """How one process stages its views.  Views [0, v_int32) cross the bus as int32 in chunks of CH;
    the remaining chunks (round(host_fraction * chunks) of them) are narrowed to 1-byte codes on the
    host in `batches` of view ranges, two chunks at a time while more than three remain and then one
    at a time, so that little is left to upload once the host is done.  Returns (v_int32, batches,
    bytes the maps put on the bus)."""
    V = len(shapes)
    n_chunks = -(-V // CH)
    n_dev = n_chunks - int(round(host_fraction * n_chunks))
    batches, b0 = [], n_dev
    while b0 < n_chunks:
        b1 = b0 + (2 if n_chunks - b0 > 3 else 1)
        batches.append((b0 * CH, min(b1 * CH, V)))
        b0 = b1
    v_int32 = min(n_dev * CH, V)
    px = [h * w for h, w in shapes]
    return v_int32, batches, 4 * sum(px[:v_int32]) + sum(px[v_int32:])


def _stage_int32(seg_maps, shapes, sizes, starts, pstarts, device, v_lo, v_hi, packed, before_wait, on_chunk):
    """Views [v_lo, v_hi) cross the bus as int32 in chunks of CH views, two staging buffers in flight
    on the copy stream, and are packed on the current stream with the default code window
    (gsl_pack_labels).  `starts` / `pstarts` are the pixel / packed-byte offsets of every view.

    The first two uploads are enqueued before anything else happens on the host; `before_wait`
    (the Gaussian ordering, which reads no maps) is called right after them, and `packed` is
    allocated after it when None.  `on_chunk(v0, v1, packed)`, when given, is called once chunk
    [v0, v1) has been packed (enqueued on the current stream) and the upload that refills its buffer
    has been enqueued.  Returns (packed, int32 device tensor [min, max] of the values uploaded)."""
    from ._native import check, lib
    L = lib()
    main = torch.cuda.current_stream(device)
    copy = _side_stream(device, "copy")
    copy.wait_stream(main)          # device-resident maps may still be being written; freed blocks may still be in use
    chunks = list(range(v_lo, v_hi, CH))
    chunk_px = max([int(starts[min(v0 + CH, v_hi)] - starts[v0]) for v0 in chunks] + [1])
    with torch.cuda.stream(copy):
        slots = [torch.empty(chunk_px, dtype=torch.int32, device=device) for _ in range(2)]
    for sl in slots:
        sl.record_stream(main)
    slot_free, ready, n_px = [None, None], [None] * len(chunks), [0] * len(chunks)

    def upload(ci):
        v0 = chunks[ci]
        with torch.cuda.stream(copy):
            if slot_free[ci % 2] is not None:
                copy.wait_event(slot_free[ci % 2])
            n_px[ci] = _copy_views(seg_maps, sizes, v0, min(v0 + CH, v_hi), slots[ci % 2])
            ready[ci] = torch.cuda.Event()
            ready[ci].record(copy)

    for ci in range(min(2, len(chunks))):                        # the transfer starts now
        upload(ci)
    before_wait()
    if packed is None:
        packed = torch.empty(int(pstarts[-1]), dtype=torch.uint8, device=device)
    minmax = torch.tensor([2**31 - 1, -2**31], dtype=torch.int32, device=device)
    err = torch.zeros(1, dtype=torch.int32, device=device)
    # everything below is enqueued without waiting
    for ci, v0 in enumerate(chunks):
        v1 = min(v0 + CH, v_hi)
        buf = slots[ci % 2]
        main.wait_event(ready[ci])
        check(L.gsl_label_range(buf.data_ptr(), n_px[ci], minmax.data_ptr(), main.cuda_stream))
        for v, n in ops._runs(shapes, v0, v1):
            check(L.gsl_pack_labels(buf.data_ptr() + 4 * int(starts[v] - starts[v0]), n, shapes[v][1], shapes[v][0],
                                    packed.data_ptr() + int(pstarts[v]), ops.DEFAULT_LABEL_MIN, ops.DEFAULT_N_CLASSES,
                                    err.data_ptr(), main.cuda_stream))
        slot_free[ci % 2] = torch.cuda.Event()
        slot_free[ci % 2].record(main)
        if ci + 2 < len(chunks):
            upload(ci + 2)                                       # refills the slot just packed
        if on_chunk is not None:
            on_chunk(v0, v1, packed)
    return packed, minmax


def _stage_single(seg_maps, shapes, device, before_wait, on_packed):
    """One-process staging of HOST (or device) maps, organised around the PCIe transfer, which is
    what such a call waits for (N2 of SURVEY 8f):

      * the first chunks of 16 views cross the bus as int32 and are packed on the device
        (_stage_int32);
      * the remaining chunks are narrowed to 1-byte codes by the host cores meanwhile
        (gsl_host_pack_labels), cross as uint8 behind the int32 chunks, and are laid out on the
        device (gsl_tile_codes).

    _chunk_plan makes the split.  `on_packed(v0, v1, packed)` is called every time the packed maps
    of views [0, v1) have been enqueued on the main stream, so that the caller can sweep them while
    later maps are still crossing the bus.  Codes are label + 2 (label_min = -1, 254 codes).
    Returns (packed, lo, hi), the value range seen, which the caller checks, re-staging when the
    labels do not fit that window."""
    import ctypes
    import time
    from ._native import check, lib
    L = lib()
    V = len(seg_maps)
    sizes = [h * w for h, w in shapes]
    starts = np.concatenate(([0], np.cumsum(sizes))).astype(np.int64)     # pixels, row-major staging
    pstarts = ops.packed_offsets(shapes)                                   # bytes, packed layout
    hv0, batches, h2d_bytes = _chunk_plan(shapes, _host_fraction(seg_maps, int(starts[-1])))
    main = torch.cuda.current_stream(device)
    copy = _side_stream(device, "copy")
    t_call0 = time.perf_counter()
    with torch.cuda.device(device):
        packed, minmax = _stage_int32(seg_maps, shapes, sizes, starts, pstarts, device, 0, hv0, None, before_wait, on_packed)
        # ---- views [hv0, V) narrowed on the host, a batch at a time, while the DMA engine is busy with the above
        host_mm = (ctypes.c_int * 2)(2**31 - 1, -2**31)
        if batches:
            host_px = int(starts[V] - starts[hv0])
            if _pinned_codes.get("n", 0) < host_px:
                # sized for every view of the scene, so that a later call whose calibrated split moves
                # more views to the host does not pay a pinned allocation inside its timed region
                t_alloc = time.perf_counter()
                _pinned_codes["buf"] = torch.empty(int(starts[V]), dtype=torch.uint8, pin_memory=True)
                _pinned_codes["n"] = int(starts[V])
                t_call0 += time.perf_counter() - t_alloc         # a one-time cost, not part of the calibration
            pinned = _pinned_codes["buf"]
            with torch.cuda.stream(copy):
                codes = torch.empty(host_px, dtype=torch.uint8, device=device)
            codes.record_stream(main)
            bad = ctypes.c_int(0)
            t_narrow, px_narrow = 0.0, 0
            for vb0, vb1 in batches:
                keep = [_host_ptr(seg_maps[v]) for v in range(vb0, vb1)]
                ptrs = (ctypes.c_void_p * len(keep))(*[k[0] for k in keep])
                npx = (ctypes.c_int64 * len(keep))(*[sizes[v] for v in range(vb0, vb1)])
                off0, off1 = int(starts[vb0] - starts[hv0]), int(starts[vb1] - starts[hv0])
                t0 = time.perf_counter()
                check(L.gsl_host_pack_labels(ptrs, npx, len(keep), ops.DEFAULT_LABEL_MIN, ops.DEFAULT_N_CLASSES,
                                             pinned.data_ptr() + off0, _host_cores(), host_mm, ctypes.byref(bad)))
                t_narrow += time.perf_counter() - t0
                px_narrow += off1 - off0
                with torch.cuda.stream(copy):
                    codes[off0:off1].copy_(pinned[off0:off1], non_blocking=True)
                    landed = torch.cuda.Event()
                    landed.record(copy)
                main.wait_event(landed)
                for v, n in ops._runs(shapes, vb0, vb1):
                    check(L.gsl_tile_codes(codes.data_ptr() + int(starts[v] - starts[hv0]), n, shapes[v][1], shapes[v][0],
                                           packed.data_ptr() + int(pstarts[v]), main.cuda_stream))
                on_packed(vb0, vb1, packed)
            if t_narrow > 0:
                _host_stage["px_per_s"] = px_narrow / t_narrow
                # the other host work of this call; first calls also pay allocations, hence the cap
                _host_stage["fixed_s"] = min(max(time.perf_counter() - t_call0 - t_narrow, 0.0), 0.015)
        lo, hi = (int(x) for x in minmax.tolist())           # synchronises: every copy has been consumed
    last_call_stats.update(h2d_bytes=h2d_bytes, views_as_int32=hv0, views_narrowed_on_host=V - hv0)
    return packed, min(lo, int(host_mm[0])), max(hi, int(host_mm[1]))


def _stage_sharded(seg_maps, shapes, device, dist, world, rank, before_wait):
    """Multi-rank staging: every rank holds the same host maps but uploads and packs only its
    contiguous block of views (_stage_int32), and PUSHES every packed chunk straight into all ranks'
    packed buffers over peer memory (torch symmetric memory = CUDA peer mapping over NVLink) while
    the next chunk crosses PCIe.  The PCIe cost per rank drops by the world size and no collective
    library call sits on the data path; one barrier at the end publishes the buffers.
    Returns (packed, lo, hi) as _stage_single does."""
    V = len(seg_maps)
    sizes = [h * w for h, w in shapes]
    starts = np.concatenate(([0], np.cumsum(sizes))).astype(np.int64)
    pstarts = ops.packed_offsets(shapes)
    total = int(pstarts[-1])
    per, extra = divmod(V, world)
    cuts = [r * per + min(r, extra) for r in range(world + 1)]
    v_lo, v_hi = cuts[rank], cuts[rank + 1]
    main = torch.cuda.current_stream(device)
    peers = None
    use_symm = os.environ.get("GSLIFT_STAGE_EXCHANGE", "symm") != "nccl"
    if use_symm:
        try:
            import torch.distributed._symmetric_memory as symm_mem
            key = (device.index, total)
            if key not in _symm_packed:
                _symm_packed.clear()                 # one scene at a time: drop the previous mapping
                buf = symm_mem.empty(max(total, 16), dtype=torch.uint8, device=device)
                hdl = symm_mem.rendezvous(buf, dist.group.WORLD.group_name)
                _symm_packed[key] = (buf, hdl, [hdl.get_buffer(r, (max(total, 16),), torch.uint8) for r in range(world)])
            packed, hdl, peers = _symm_packed[key]
        except Exception:                            # no peer access on this machine: NCCL broadcast below
            peers = None
    if peers is None:
        packed = torch.empty(total, dtype=torch.uint8, device=device)
    else:
        # nobody may still be sweeping the previous call's maps when the pushes of this one arrive
        dist.barrier()
    push = _side_stream(device, "push")

    def push_chunk(v0, v1, packed):
        """Push packed views [v0, v1) to every peer while the next chunk uploads."""
        done = torch.cuda.Event()
        done.record(main)
        a, b = int(pstarts[v0]), int(pstarts[v1])
        with torch.cuda.stream(push):
            push.wait_event(done)
            for k in range(1, world):
                r = (rank + k) % world
                peers[r][a:b].copy_(packed[a:b], non_blocking=True)

    with torch.cuda.device(device):
        packed, minmax = _stage_int32(seg_maps, shapes, sizes, starts, pstarts, device, v_lo, v_hi, packed, before_wait,
                                      push_chunk if peers is not None else None)
        mm = torch.stack([minmax[0].to(torch.int64), -minmax[1].to(torch.int64)])
        dist.all_reduce(mm, op=dist.ReduceOp.MIN)
        if peers is not None:
            main.wait_stream(push)
            torch.cuda.current_stream(device).synchronize()
            dist.barrier()                           # every rank's pushes have landed everywhere
        else:
            for r in range(world):
                a, b = int(pstarts[cuts[r]]), int(pstarts[cuts[r + 1]])
                if b > a:
                    dist.broadcast(packed[a:b], src=r)
        lo, hi = int(mm[0].item()), -int(mm[1].item())
    last_call_stats.update(h2d_bytes=4 * int(starts[v_hi] - starts[v_lo]), views_as_int32=V, views_narrowed_on_host=0)
    return packed, lo, hi


def lift_labels(positions, cameras, seg_maps, image_sizes=None, device=None, want_near=False,
                near_eps=1e-4, label_min=None, n_classes=None):
    """Majority-vote labels for `positions` given one segmentation map per camera.

    positions   float32 [N,3] array or tensor (under torch.distributed: THIS rank's Gaussians)
    cameras     camera dicts, in voting order
    seg_maps    list of int arrays [seg_h, seg_w] (NumPy or tensors), one per camera; any int32
                label values (more than 254 distinct values are lifted in several passes)
    image_sizes per camera (orig_w, orig_h); default = the map's own size (scale 1.0)
    label_min, n_classes  optional explicit code window, both or neither (values outside it raise)
    Returns int32 NumPy labels (and the near-boundary mask when want_near).
    """
    from ._native import check, lib
    device = torch.device(device if device is not None else "cuda")
    trace = os.environ.get("GSLIFT_TRACE") == "1"
    if trace:
        import sys, time
        t_enter = time.perf_counter()
    shapes = [tuple(int(x) for x in m.shape) for m in seg_maps]
    if any(len(sh) != 2 for sh in shapes):
        raise ValueError("every segmentation map must be 2-D [seg_h, seg_w]")
    if (label_min is None) != (n_classes is None):
        raise ValueError("give both label_min and n_classes, or neither")
    dist, world, rank = _dist()
    V = len(cameras)
    if len(seg_maps) != V:
        raise ValueError("one segmentation map per camera")
    L = lib()
    main = torch.cuda.current_stream(device)
    state = {}

    def prepare():
        """Positions to the device, view table, ordering + verdicts: needs no maps, so it is
        enqueued right behind the first uploads."""
        pos = positions if isinstance(positions, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(positions, np.float32))
        pos = pos.to(device=device, dtype=torch.float32, non_blocking=True).contiguous()
        views = ops.make_views(cameras, shapes, image_sizes)
        N = pos.shape[0]
        ws = ops._ws.get(device, L.gsl_lift_workspace_bytes(N, V))
        with torch.cuda.device(device):
            check(L.gsl_lift_prepare(pos.data_ptr(), N, views.ctypes.data, V, ws.data_ptr(), ws.numel(), main.cuda_stream))
        state.update(pos=pos, views=views, N=N, ws=ws)

    def gather(packed, v0, v1):
        with torch.cuda.device(device):
            check(L.gsl_lift_gather_range(state["pos"].data_ptr(), state["N"], state["views"].ctypes.data, V, v0, v1,
                                          packed.data_ptr(), state["ws"].data_ptr(), state["ws"].numel(), main.cuda_stream))

    def sweep(packed, lmin, ncls, best=None, v_from=0):
        """Gather views [v_from, V) (earlier ones were swept while the maps were uploading), then the majority."""
        labels = torch.empty(state["N"], dtype=torch.int32, device=device)
        gather(packed, v_from, V)
        with torch.cuda.device(device):
            check(L.gsl_lift_majority(state["N"], V, int(lmin), int(ncls), labels.data_ptr(),
                                      best.data_ptr() if best is not None else None,
                                      state["ws"].data_ptr(), state["ws"].numel(), main.cuda_stream))
        return labels

    swept = [0]

    def sweep_resident(v0, v1, packed):
        """Staging callback: views [0, v1) are packed (enqueued on the main stream); gather the
        complete groups of 32 among them -- a sweep CTA takes two 16-view windows."""
        target = v1 if v1 == V else v1 // 32 * 32
        if target > swept[0]:
            gather(packed, swept[0], target)
            swept[0] = target

    if V == 0 or positions.shape[0] == 0:
        labels = np.full(positions.shape[0], -1, dtype=np.int32)
        return (labels, np.zeros(positions.shape[0], np.uint8)) if want_near else labels

    lmin, ncls = ops.DEFAULT_LABEL_MIN, ops.DEFAULT_N_CLASSES
    wide = False
    if label_min is not None:
        lmin, ncls = int(label_min), int(n_classes)
        prepare()
        staged = _upload_all(seg_maps, shapes, device)
        packed = ops.pack_labels(staged, shapes, lmin, ncls)              # raises on a value outside the window
        last_call_stats.update(h2d_bytes=4 * staged.numel(), views_as_int32=V, views_narrowed_on_host=0)
    else:
        if world > 1:
            packed, lo, hi = _stage_sharded(seg_maps, shapes, device, dist, world, rank, prepare)
        else:
            packed, lo, hi = _stage_single(seg_maps, shapes, device, prepare, sweep_resident)
        wide = lo < lmin or hi > lmin + ncls - 1
        ncls = min(max(hi - lmin + 1, 1), ncls) if hi >= lo else 1      # fewer histogram rows per Gaussian
    if not wide:
        labels = sweep(packed, lmin, ncls, v_from=swept[0])
        n_passes = 1
    else:
        staged = _upload_all(seg_maps, shapes, device)
        last_call_stats["h2d_bytes"] += 4 * staged.numel()
        uniq = torch.unique(staged)                                     # sorted
        dense = torch.searchsorted(uniq, staged).to(torch.int32)        # every value -> its rank among the distinct values
        n_ids = int(uniq.numel())
        labels = best = None
        packed = torch.empty(int(ops.packed_offsets(shapes)[-1]), dtype=torch.uint8, device=device)
        P = ops.DEFAULT_N_CLASSES
        for first in range(0, n_ids, P):
            n_here = min(P, n_ids - first)
            ops.pack_labels(dense, shapes, first, n_here, out=packed, check_range=False)
            b = torch.empty(state["N"], dtype=torch.int32, device=device)       # uint32 keys, carried as int32 storage
            lab = sweep(packed, first, n_here, best=b)
            if labels is None:
                labels, best = lab, b
            else:
                ops.lift_merge(labels, best, lab, b)
        seen = labels >= 0
        labels = torch.where(seen, uniq[labels.clamp(min=0).long()], labels)           # dense id -> the map's own value
        n_passes = -(-n_ids // P)
    last_call_stats.update(h2d_bytes=last_call_stats["h2d_bytes"] + int(state["pos"].numel()) * 4,
                           d2h_bytes=int(state["N"]) * 4, label_passes=n_passes)
    if trace:
        torch.cuda.synchronize(device)
        print(f"[gslift trace] lift_labels: staging + sweep {1e3 * (time.perf_counter() - t_enter):.2f} ms, "
              f"{last_call_stats['views_as_int32']} views as int32, {last_call_stats['views_narrowed_on_host']} narrowed on the host",
              file=sys.stderr)
    if want_near:
        near = ops.lift_near(state["pos"], state["views"], near_eps)
        return _to_host(labels), _to_host(near)
    return _to_host(labels)


def _to_host(t: torch.Tensor) -> np.ndarray:
    """Device tensor -> NumPy through a pinned staging tensor (a pageable `.cpu()` of 24 MB costs
    ~10 ms; pinned, it is PCIe speed).  The array owns its pinned storage."""
    trace = os.environ.get("GSLIFT_TRACE") == "1"
    if trace:
        import sys, time
        t0 = time.perf_counter()
    host = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    if trace:
        t1 = time.perf_counter()
    host.copy_(t, non_blocking=True)
    torch.cuda.current_stream(t.device).synchronize()
    if trace:
        print(f"[gslift trace] result to host: pinned alloc {1e3 * (t1 - t0):.2f} ms, copy {1e3 * (time.perf_counter() - t1):.2f} ms", file=sys.stderr)
    return host.numpy()


def assign_labels(gaussians, cameras, input_dir, output_dir, model_type="mask2former", segmenter=None):
    """Label every Gaussian by majority vote over its projections (reference :241-308).

    Returns np.int32 [N]; -1 for Gaussians no view sees."""
    upstream = None
    used, maps, sizes = [], [], []
    for camera in cameras:
        img_path = os.path.join(input_dir, camera["img_name"] + ".png")
        if not os.path.exists(img_path):
            print(f"Warning: Image {camera['img_name']} not found")
            continue
        print(f"Processing image {os.path.basename(img_path)}...")
        with Image.open(img_path) as image:
            size = (image.size[0], image.size[1])
        if segmenter is not None:
            seg_map = segmenter(img_path, output_dir, model_type)
        else:
            seg_map = _precomputed_map(output_dir, camera["img_name"])
            if seg_map is None:
                if upstream is None:
                    upstream = _UpstreamSegmenter(model_type)
                seg_map = upstream(img_path, output_dir, model_type)
        used.append(camera)
        maps.append(np.asarray(seg_map))
        sizes.append(size)
    positions = np.ascontiguousarray(gaussians["position"], np.float32)
    if not used:
        return np.full(len(positions), -1, dtype=np.int32)
    return lift_labels(positions, used, maps, sizes)


def save_labeled_ply(output_file, plydata, labels):
    """Write the input vertices plus an int32 `label` column as binary PLY (reference :311-332)."""
    vertex = plyio.describe_with_label(plydata["vertex"].data, labels)
    plyio.write_ply(output_file, [("vertex", vertex)], text=False)


def main():
    parser = argparse.ArgumentParser(description="Add labels to gaussians PLY file")
    parser.add_argument("--ply_file", help="Input PLY file with gaussians data")
    parser.add_argument("--camera_file", help="JSON file with camera data")
    parser.add_argument("--input_dir", help="Directory containing input images")
    parser.add_argument("--output_dir", help="Output directory to saved segmented input images")
    parser.add_argument("--output_file", help="Output PLY file with labels")
    parser.add_argument("--model", choices=["segformer", "mask2former", "yolo"], default="mask2former",
                        help="Choose segmentation model: mask2former or yolo")
    args = parser.parse_args()

    print("Loading cameras...")
    cameras = load_cameras(args.camera_file)
    print("Loading gaussians...")
    gaussians, plydata = load_gaussians(args.ply_file)
    print("Assigning labels...")
    labels = assign_labels(gaussians, cameras, args.input_dir, args.output_dir, model_type=args.model)
    print("Saving labeled PLY file...")
    save_labeled_ply(args.output_file, plydata, labels)
    print(f"Done! Labeled PLY file saved as {args.output_file}")

    values, counts = np.unique(labels, return_counts=True)
    print("\nLabel statistics:")
    print(f"Total gaussians: {len(labels)}")
    print(f"Number of unique labels: {len(values)}")
    print("Label counts:")
    for value, count in zip(values, counts):
        print(f"Label {value}: {count} gaussians ({100 * count / len(labels):.2f}%)")


if __name__ == "__main__":
    main()
