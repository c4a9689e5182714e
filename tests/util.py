"""Shared helpers for the tests (fixture loading, package import)."""
import importlib
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
PKG = "3d_gaussian_splatting_project_b200"


def pkg(sub=None):
    return importlib.import_module(PKG if sub is None else f"{PKG}.{sub}")


def load_lift_case(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    cams = json.loads(str(z["cameras"]))
    shapes = z["map_shapes"]
    flat = z["maps_flat"].astype(np.int32)
    maps, off = [], 0
    for h, w in shapes:
        maps.append(flat[off:off + h * w].reshape(h, w))
        off += h * w
    sizes = [tuple(int(s) for s in row) for row in z["image_sizes"]]
    return dict(pos=z["pos"], cameras=cams, maps=maps, sizes=sizes, labels=z["labels"],
                flat=flat, shapes=shapes)


LIFT_CASES = ["lift_bundled_halfres", "lift_lookat_fullres", "lift_lookat_rescaled",
              "lift_lookat_regions", "lift_degenerate"]
KMEANS_CASES = ["kmeans_color_k10", "kmeans_kdtree_k64_d59", "kmeans_converged_k4", "kmeans_empty_k8"]


def blobs(rng, n, spread=0.3):
    """float32 [n, 3]: ten Gaussian blobs of the given spread with centres in [-2, 2]^3."""
    centres = rng.uniform(-2, 2, size=(10, 3))
    return (centres[rng.integers(0, 10, n)] + rng.normal(0, spread, size=(n, 3))).astype(np.float32)


def assert_bits_equal(got, want, what="centroids"):
    """float32 arrays equal bit for bit, so -0.0 != +0.0.  Any two NaNs count as equal: the GPU writes a
    canonical NaN where x86 keeps the payload and sign of an operand."""
    got, want = np.asarray(got, np.float32), np.asarray(want, np.float32)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    bad = (got.view(np.uint32) != want.view(np.uint32)) & ~(np.isnan(got) & np.isnan(want))
    if bad.any():
        first = [(tuple(int(j) for j in i), got[tuple(i)], want[tuple(i)]) for i in np.argwhere(bad)[:4]]
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.size} values differ in their bits; (index, got, want): {first}")


def load_kmeans_case(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    d = {k: z[k] for k in z.files}
    if "data" not in d:
        d["data"] = np.concatenate((d["points"], d["colors"]), axis=1)
    d["k"] = int(d["k"]); d["seed"] = int(d["seed"]); d["max_iter"] = int(d["max_iter"])
    d["stdout"] = str(d["stdout"])
    return d
