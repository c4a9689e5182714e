"""Host-side logic that needs no GPU: view tables, PLY I/O, drop-in surfaces, sharding (gloo)."""
import inspect
import io
import os
import subprocess
import sys
import contextlib

import numpy as np
import pytest

from util import load_lift_case, pkg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_make_views_matches_oracle_table(oracle):
    c = load_lift_case("lift_bundled_halfres")
    mine = pkg("ops").make_views(c["cameras"], c["shapes"], c["sizes"])
    ref = oracle.make_views(c["cameras"], c["shapes"], c["sizes"])
    assert mine.dtype.itemsize == ref.dtype.itemsize == 176
    for name in mine.dtype.names:
        if name != "map_offset":                               # the library packs maps in its own tiled layout
            assert np.array_equal(mine[name], ref[name]), name     # incl. t = -R @ p, bit for bit
    ops = pkg("ops")
    offs = ops.packed_offsets(c["shapes"])
    L = pkg("_native").lib()
    for (h, w) in [(1080, 1920), (1038, 1557), (1, 1), (77, 51), (2075, 3114)]:       # host formula == the library's
        assert ops.packed_map_bytes(h, w) == L.gsl_packed_map_bytes(w, h)
    assert np.array_equal(mine["map_offset"], offs[:-1]) and ops.packed_map_bytes(1080, 1920) == 122 * 137 * 128 + 33440
    assert mine["scale_x"][0] == 1.0 and mine["width"][0] == 3114


def test_ply_roundtrip_binary_and_ascii(tmp_path):
    plyio, scene = pkg("plyio"), pkg("scene")
    v = scene.standin_3dgs_vertices(257, seed=3)
    labels = np.arange(257, dtype=np.int64) % 11 - 1
    out = plyio.describe_with_label(v, labels)
    assert out.dtype.names[-1] == "label" and out.dtype["label"] == np.dtype("<i4")
    b, a = tmp_path / "b.ply", tmp_path / "a.ply"
    plyio.write_ply(b, [("vertex", out)], text=False)
    plyio.write_ply(a, [("vertex", out)], text=True)
    head = open(b, "rb").read(4096).split(b"end_header\n")[0].decode().splitlines()
    assert head[:3] == ["ply", "format binary_little_endian 1.0", "element vertex 257"]
    assert head[3] == "property float x" and head[-1] == "property int label" and len(head) == 3 + 63
    assert os.path.getsize(b) == len("\n".join(head)) + 1 + len("end_header\n") + 257 * 63 * 4
    for path, text in ((b, False), (a, True)):
        back = plyio.read_ply(path)
        assert back.text == text
        got = back["vertex"].data
        assert got.dtype.names == out.dtype.names
        for n in out.dtype.names:
            assert np.array_equal(got[n], out[n]), n         # %.18g round-trips float32 exactly
    first = open(a).read().split("end_header\n")[1].splitlines()[0].split()
    assert len(first) == 63 and first[-1] == "-1"
    assert first[0] == "%.18g" % float(v["x"][0])


def test_dropin_surfaces_match_reference_signatures():
    dls, km = pkg("deep_learning_segmentation"), pkg("k_means")
    assert list(inspect.signature(dls.assign_labels).parameters)[:5] == ["gaussians", "cameras", "input_dir", "output_dir", "model_type"]
    assert inspect.signature(dls.assign_labels).parameters["model_type"].default == "mask2former"
    assert list(inspect.signature(dls.project_gaussian).parameters) == ["position", "camera"]
    assert list(inspect.signature(dls.save_labeled_ply).parameters) == ["output_file", "plydata", "labels"]
    p = inspect.signature(km.k_means_with_color).parameters
    assert list(p)[:5] == ["points", "k", "colors", "max_iter", "tol"] and p["max_iter"].default == 100 and p["tol"].default == 1e-4
    assert list(inspect.signature(km.k_means_kd_tree).parameters)[:5] == ["data", "k", "colors", "max_iter", "tol"]
    assert len(km.COLORS) == 8 and km.COLORS[3] == [126, 24, 145]


def test_region_growing_and_viewer_surfaces_match_reference():
    """Names and parameters of 3D_clustering/region_growing.py (rg:11-261) and of the viewer worker's
    functions (gaussians_selection.js:110, :361, :417), snake case for the latter."""
    rg, viewer = pkg("region_growing"), pkg("viewer")
    want = {"get_vertex_info": ["plydata"], "generate_sphere_ply": ["radius", "subdivisions", "filename"],
            "compute_normals": ["V1", "k"], "compute_residuals": ["V1", "normals", "k"],
            "segmentation_3D": ["points", "normals", "residuals", "residual_threshold", "angle_threshold", "k"],
            "set_clusters": ["plydata", "R", "modified_path"]}
    for name, params in want.items():
        assert list(inspect.signature(getattr(rg, name)).parameters) == params, name
    sp = inspect.signature(rg.generate_sphere_ply).parameters
    assert (sp["radius"].default, sp["subdivisions"].default, sp["filename"].default) == (1.0, 50, "sphere.ply")
    assert list(inspect.signature(viewer.perform_hit_testing).parameters)[:5] == ["x", "y", "view_matrix", "projection_matrix", "viewport"]
    assert list(inspect.signature(viewer.run_sort).parameters)[:2] == ["positions", "view_proj"]
    assert viewer.NO_SELECTION == -999999
    # multiply4 is plain host arithmetic: column-major product in the worker's association order
    a = [float(i) for i in range(1, 17)]
    ident = [1.0 if i % 5 == 0 else 0.0 for i in range(16)]
    assert viewer.multiply4(a, ident) == a and viewer.multiply4(ident, a) == a


def test_generate_sphere_ply_text(tmp_path, capsys):
    """rg:42-76: header and the '%.6f %.6f %.6f 255 0 0' rows, (subdivisions + 1) * subdivisions vertices."""
    rg = pkg("region_growing")
    path = tmp_path / "s.ply"
    rg.generate_sphere_ply(radius=2.0, subdivisions=4, filename=str(path))
    assert capsys.readouterr().out == f"Sphere saved to {path}\n"
    lines = path.read_text().split("\n")
    assert lines[:10] == ["ply", "format ascii 1.0", "element vertex 20", "property float x", "property float y", "property float z",
                          "property uchar red", "property uchar green", "property uchar blue", "end_header"]
    assert lines[10] == "0.000000 0.000000 2.000000 255 0 0"                 # theta = 0: the pole
    assert lines[10 + 8] == "2.000000 0.000000 0.000000 255 0 0"             # theta = pi/2, phi = 0
    assert len(lines) == 10 + 20 + 1 and lines[-1] == ""


def test_project_gaussian_scalar_matches_oracle(oracle):
    dls = pkg("deep_learning_segmentation")
    c = load_lift_case("lift_lookat_fullres")
    for i in range(0, 400, 7):
        cam = c["cameras"][i % len(c["cameras"])]
        assert dls.project_gaussian(c["pos"][i], cam) == oracle.project_py(c["pos"][i], cam)


def test_assign_labels_skips_missing_images_like_the_reference(tmp_path):
    dls = pkg("deep_learning_segmentation")
    g = np.zeros(5, dls.GAUSSIAN_DTYPE)
    cams = load_lift_case("lift_degenerate")["cameras"]
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        labels = dls.assign_labels(g, cams, str(tmp_path), str(tmp_path))
    assert labels.dtype == np.int32 and np.array_equal(labels, np.full(5, -1))
    assert buf.getvalue().splitlines() == [f"Warning: Image {c['img_name']} not found" for c in cams]


def test_cli_flags_unchanged():
    for script, flags in (("deep_learning_segmentation.py", ["--ply_file", "--camera_file", "--input_dir", "--output_dir", "--output_file", "--model"]),
                          (os.path.join("3D_clustering", "k_means.py"), ["--file_path", "--save_path", "--k"])):
        out = subprocess.run([sys.executable, os.path.join(ROOT, script), "--help"], capture_output=True, text=True, cwd=ROOT)
        assert out.returncode == 0, out.stderr
        for f in flags:
            assert f in out.stdout


def test_slice_bounds_partition():
    sb = pkg("sharding").slice_bounds
    for n in (0, 1, 7, 1000, 6_000_000):
        for w in (1, 2, 3, 8):
            cuts = [sb(n, r, w) for r in range(w)]
            assert cuts[0][0] == 0 and cuts[-1][1] == n
            assert all(cuts[i][1] == cuts[i + 1][0] for i in range(w - 1))
            sizes = [hi - lo for lo, hi in cuts]
            assert max(sizes) - min(sizes) <= 1


def test_lift_labels_staging_plan():
    """The one-process staging plan of lift_labels: views [0, v_int32) cross as int32, the host
    narrows the rest in batches of two 16-view chunks while more than three chunks remain, then one
    chunk at a time; every view is staged once, in order, and the bytes on the bus follow the split."""
    plan, CH = pkg("deep_learning_segmentation")._chunk_plan, 16
    px = 1080 * 1920                                     # the benchmark: 300 views of 1920 x 1080
    assert plan([(1080, 1920)] * 300, 0.4) == (176, [(176, 208), (208, 240), (240, 272), (272, 288), (288, 300)],
                                                4 * 176 * px + 124 * px)
    assert plan([(1080, 1920)] * 300, 0.0) == (300, [], 4 * 300 * px)
    assert plan([(200, 320)] * 48, 0.5) == (16, [(16, 32), (32, 48)], (4 * 16 + 32) * 200 * 320)
    for V in (1, 15, 16, 17, 33, 48, 63, 64, 65, 300, 401):
        shapes = [(7 + v % 5, 11 + v % 3) for v in range(V)]
        sizes = [h * w for h, w in shapes]
        n_chunks = -(-V // CH)
        for f in (0.0, 0.1, 0.25, 0.4, 0.5, 0.85, 1.0):
            v_int32, batches, nbytes = plan(shapes, f)
            assert v_int32 == min((n_chunks - round(f * n_chunks)) * CH, V)
            ranges = [(0, v_int32)] + batches
            assert [a for a, _ in ranges[1:]] == [b for _, b in ranges[:-1]] and ranges[-1][1] == V   # once, in order
            assert all(a % CH == 0 and a < b for a, b in batches)
            per_batch = [-(-(b - a) // CH) for a, b in batches]                                     # chunks per batch
            m = n_chunks - v_int32 // CH if batches else 0
            k = max(0, (m - 2) // 2)
            assert per_batch == [2] * k + [1] * (m - 2 * k)
            assert nbytes == 4 * sum(sizes[:v_int32]) + sum(sizes[v_int32:])


_WORKER = r'''
import os, sys, importlib
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from oracle import oracle as orc
gs = importlib.import_module("3d_gaussian_splatting_project_b200")
rank, world, _ = gs.sharding.init_from_env("gloo")
# K-means exchange step on CPU tensors: per-rank float64 sums/counts from the oracle,
# all-reduced, must equal the single-process sums; slices preserve index order.
data = gs.scene.blob_features(5003, 7, n_blobs=5, seed=9)
cen = data[:6].copy()
lo, hi = gs.sharding.slice_bounds(len(data), rank, world)
lab = orc.kmeans_assign(data[lo:hi], cen)
sums = np.zeros((6, 8))
for k in range(6):
    m = lab == k
    sums[k, :7] = data[lo:hi][m].astype(np.float64).sum(0); sums[k, 7] = m.sum()
t = torch.from_numpy(sums); dist.all_reduce(t)
full = orc.kmeans_assign(data, cen)
assert np.array_equal(full[lo:hi], lab)
want = np.zeros((6, 8))
for k in range(6):
    m = full == k
    want[k, :7] = data[m].astype(np.float64).sum(0); want[k, 7] = m.sum()
assert np.allclose(t.numpy(), want, rtol=1e-13, atol=0), np.abs(t.numpy() - want).max()
got = gs.sharding.gather_labels(torch.from_numpy(lab.astype(np.int32)), len(data), rank, world)
if rank == 0:
    assert np.array_equal(got.numpy(), full.astype(np.int32))
ms = gs.sharding.barrier_max_ms(float(rank + 1), "cpu")
assert ms == world
dist.barrier(); dist.destroy_process_group()
print("ok", rank)
'''


def test_sharding_world_size_2_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", OMP_NUM_THREADS="2")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29731", str(script), ROOT],
                         capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert out.stdout.count("ok") == 2


def test_host_label_narrowing_matches_numpy():
    """gsl_host_pack_labels (host-side staging helper, no device): codes, value range and the
    out-of-range flag against NumPy, over sizes around the 32-pixel vector width, several maps per
    call and thread ranges that cross map boundaries."""
    import ctypes
    L = pkg("_native").lib()
    rng = np.random.default_rng(0)

    def run(maps, label_min, n_classes, n_threads):
        tot = sum(m.size for m in maps)
        out = np.full(tot + 64, 0xAB, np.uint8)                   # guard bytes behind the output
        ptrs = (ctypes.c_void_p * len(maps))(*[m.ctypes.data for m in maps])
        npx = (ctypes.c_int64 * len(maps))(*[m.size for m in maps])
        mm = (ctypes.c_int * 2)(2**31 - 1, -2**31)
        bad = ctypes.c_int(0)
        assert L.gsl_host_pack_labels(ptrs, npx, len(maps), label_min, n_classes, out.ctypes.data, n_threads, mm, ctypes.byref(bad)) == 0
        assert (out[tot:] == 0xAB).all(), "wrote past the end"
        return out[:tot], (mm[0], mm[1]), bad.value

    for n in (0, 1, 31, 32, 33, 1000, 123457):
        a = rng.integers(-5, 300, n).astype(np.int32)
        got, mm, bad = run([a], -1, 254, 0)
        c = a.astype(np.int64) + 1
        want = np.where((c >= 0) & (c < 254), c + 1, 0).astype(np.uint8)
        assert np.array_equal(got, want), n
        if n:
            assert mm == (int(a.min()), int(a.max())) and bad == int(((c < 0) | (c >= 254)).any())
    maps = [rng.integers(-1, 150, s).astype(np.int32) for s in (70001, 5, 300000, 64, 0, 131072)]
    for nt in (1, 3, 5, 8):
        got, mm, bad = run(maps, -1, 151, nt)
        assert np.array_equal(got, (np.concatenate(maps) + 2).astype(np.uint8)) and bad == 0 and mm == (-1, 149)
    ext = np.array([-2**31, 2**31 - 1, 0, 7], np.int32)           # wrap-around of v - label_min must not alias a valid code
    got, mm, bad = run([ext], 5, 10, 1)
    assert got.tolist() == [0, 0, 0, 3] and bad == 1 and mm == (-2**31, 2**31 - 1)
    assert L.gsl_host_pack_labels(None, None, 1, -1, 254, None, 0, None, None) == -1
