"""GPU parity of the region-growing numerics (csrc/region_growing.cu through the C ABI and the
region_growing.py mirror) with the golden vectors of the reference and with the oracle.

Bars (floating point, stated here):
  * neighbour lists (k <= 64): identical to KDTree.query's, exact distance ties aside
  * normals: 1 - |cos| < 1e-8 against the oracle / the reference where the normal is well defined
    (eigenvalue gap > 1e-2 of the largest), same orientation unless the point lies on its own plane
  * residuals: absolute 1e-5 of a cloud ~4 units wide (the reference's centroid is a float32
    sequential mean, the GPU's a float64 sum: ~1e-7); 1e-6 with the reference's normals handed in
  * segmentation_3D: the same partition into regions as the reference.
The exact neighbour sets for k > 64 are checked against a float64 reference in test_region_exact_sets.py."""
import contextlib
import io
import os

import numpy as np
import pytest
import torch

from util import GOLDEN, blobs, pkg

pytestmark = pytest.mark.gpu

REGION_CASES = ["region_planes_k40", "region_planes_k400", "region_planes_k2000"]
GAP_MIN = 1e-2


def load_region(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    return {k: z[k] for k in z.files}


def quiet(fn, *a, **kw):
    with contextlib.redirect_stdout(io.StringIO()) as out:
        r = fn(*a, **kw)
    return r, out.getvalue()


def check_against(oracle, pos, k, got_normals, got_residuals, ref, tol_cos=1e-8, tol_res=1e-5, rows=None):
    sel = slice(None) if rows is None else slice(*rows)
    ok = ref["gap"][sel] > GAP_MIN
    dots = (got_normals[sel] * ref["normals"][sel]).sum(1)
    assert (1 - np.abs(dots[ok])).max() < tol_cos
    flipped = ok & (dots < 0)
    assert (ref["residuals"][sel][flipped] < tol_res).all()
    assert np.abs(got_residuals[sel] - ref["residuals"][sel])[ok].max() < tol_res
    return int(ok.sum())


@pytest.mark.parametrize("name", REGION_CASES)
def test_golden_cases_through_the_mirror(oracle, name):
    rg = pkg("region_growing")
    g = load_region(name)
    pos, k = g["pos"], int(g["k"])
    normals, out = quiet(rg.compute_normals, pos, k)
    assert out.startswith("Calculating normals...\nProcessing point 0/") and out.endswith("Normal calculation complete.\n")
    assert normals.dtype == np.float64 and normals.shape == (len(pos), 3)
    residuals, out = quiet(rg.compute_residuals, pos, g["normals"], k)
    assert out.startswith("Calculating residuals...\n")
    assert np.abs(residuals - g["residuals"]).max() < 1e-6              # the reference's normals, our centroids
    ref = oracle.region_knn_pca(pos, k)
    own = rg.knn_pca(pos, k)
    check_against(oracle, pos, k, own["normals"].cpu().numpy(), own["residuals"].cpu().numpy(), ref)
    gold = dict(normals=g["normals"], residuals=g["residuals"], gap=ref["gap"])
    check_against(oracle, pos, k, normals, own["residuals"].cpu().numpy(), gold)
    # neighbour lists and the growth loop
    knn = rg.knn_pca(pos, int(g["kseg"]), want_normals=False, want_residuals=False, want_knn=True)["knn"].cpu().numpy()
    assert np.array_equal(knn, g["knn_seg"])
    regions = rg.segmentation_3D(pos, g["normals"], g["residuals"], residual_threshold=0.1, angle_threshold=0.05, k=int(g["kseg"]))
    assert len(regions) == int(g["n_regions"]) and sorted(len(r) for r in regions) == sorted(np.bincount(g["region_of"]).tolist())
    assert [len(r) for r in regions] == sorted((len(r) for r in regions), reverse=True)
    mine = np.empty(len(pos), np.int64)
    for r, members in enumerate(regions):
        mine[members] = r
    assert len(set(zip(mine.tolist(), g["region_of"].tolist()))) == len(regions)


@pytest.mark.parametrize("n, k", [(5000, 1), (5000, 10), (20_000, 64), (20_000, 2000), (3000, 3000), (40, 7), (33, 33)])
def test_random_clouds_equal_oracle(oracle, n, k):
    rg = pkg("region_growing")
    rng = np.random.default_rng(n + k)
    pos = blobs(rng, n)
    ref = oracle.region_knn_pca(pos, k, want_knn=k <= 64)
    got = rg.knn_pca(pos, k, want_centroids=True, want_knn=k <= 64)
    if k <= 64:
        assert np.array_equal(got["knn"].cpu().numpy(), ref["knn"])
    # the reference's centroid is a float32 SEQUENTIAL mean (rg:105): its own rounding grows with k
    # (~ sqrt(k) ulps of the running sum), the GPU's float64 sum does not drift
    assert np.abs(got["centroids"].cpu().numpy() - ref["centroids"]).max() < (2e-6 if k <= 64 else 2e-5)
    if k >= 7:
        check_against(oracle, pos, k, got["normals"].cpu().numpy(), got["residuals"].cpu().numpy(), ref)


def test_outliers_duplicates_and_degenerate_sets(oracle):
    rg = pkg("region_growing")
    rng = np.random.default_rng(77)
    # a dense blob plus far outliers: the outliers' searches climb to the coarsest levels / the whole array
    pos = np.concatenate((rng.normal(0, 0.05, size=(6000, 3)), rng.uniform(-500, 500, size=(40, 3)))).astype(np.float32)
    pos = pos[rng.permutation(len(pos))]
    for k in (16, 300):
        ref = oracle.region_knn_pca(pos, k, want_knn=k <= 64)
        got = rg.knn_pca(pos, k, want_centroids=True, want_knn=k <= 64)
        if k <= 64:
            assert np.array_equal(got["knn"].cpu().numpy(), ref["knn"])
        scale = np.abs(ref["centroids"]).max(1) + 1
        assert (np.abs(got["centroids"].cpu().numpy() - ref["centroids"]).max(1) / scale).max() < 1e-5
    # duplicated points: exact distance ties at the k-th neighbour go to the lower index on both sides
    base = blobs(rng, 500)
    dup = np.concatenate((base, base, base[:100]))[rng.permutation(1100)]
    for k in (2, 5, 24):
        ref = oracle.region_knn_pca(dup, k, want_knn=True)
        got = rg.knn_pca(dup, k, want_centroids=True, want_knn=True)
        assert np.array_equal(got["knn"].cpu().numpy(), ref["knn"]), k
        assert np.abs(got["centroids"].cpu().numpy() - ref["centroids"]).max() < 2e-6
    # a lattice: many exact ties at every distance
    ax = np.arange(12, dtype=np.float32)
    lat = np.stack(np.meshgrid(ax, ax, ax, indexing="ij"), -1).reshape(-1, 3)
    ref = oracle.region_knn_pca(lat, 20, want_knn=True)
    got = rg.knn_pca(lat, 20, want_knn=True, want_centroids=True)
    assert np.array_equal(got["knn"].cpu().numpy(), ref["knn"])
    # all points coincide; points on a line (normal ill defined: only the neighbour sets are compared)
    same = np.ones((300, 3), np.float32)
    got = rg.knn_pca(same, 10, want_knn=True)
    assert np.array_equal(got["knn"].cpu().numpy(), np.tile(np.arange(10, dtype=np.int32), (300, 1)))
    assert float(got["residuals"].abs().max()) == 0.0
    line = np.zeros((400, 3), np.float32); line[:, 0] = rng.permutation(400)
    ref = oracle.region_knn_pca(line, 9, want_knn=True)
    assert np.array_equal(rg.knn_pca(line, 9, want_knn=True)["knn"].cpu().numpy(), ref["knn"])
    # argument errors mirror scipy: non-finite data, k larger than the cloud
    bad = base.copy(); bad[3, 1] = np.nan
    with pytest.raises(ValueError):
        rg.knn_pca(bad, 5)
    with pytest.raises(Exception):
        rg.knn_pca(base[:10], 11)


def test_c1_size_cloud_k2000_sample_against_oracle(oracle):
    """BASELINE config C1's cloud size (200 000 points) with the reference's k = 2000 (rg:272): all normals
    on the GPU, a slice of 600 queries checked against the brute-force oracle."""
    rg = pkg("region_growing")
    rng = np.random.default_rng(1)
    pos = blobs(rng, 200_000)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dpos = torch.from_numpy(pos).cuda()
    rg.knn_pca(dpos, 2000)                       # warm-up (workspace allocation)
    ev0.record()
    got = rg.knn_pca(dpos, 2000)
    ev1.record()
    torch.cuda.synchronize()
    st = rg.knn_pca(dpos, 2000, want_stats=True)["stats"].cpu().numpy()
    print(f"\n200 000 points, k = 2000: {ev0.elapsed_time(ev1):.1f} ms on the GPU, {st[0] / 2e5:.2f} walks per query, "
          f"{st[1] / 4e8:.2f} points visited per neighbour found, {st[2] / 2e5:.2f} cubes too small, "
          f"{st[3] / 2e5:.2f} further select walks per query")
    assert st[0] / 2e5 < 8
    q0, q1 = 100_000, 100_600
    ref = oracle.region_knn_pca(pos, 2000, queries=(q0, q1))
    check_against(oracle, pos, 2000, got["normals"].cpu().numpy(), got["residuals"].cpu().numpy(), ref, rows=(q0, q1))


def test_floaters_do_not_degrade_the_grid(oracle):
    """Far outliers (floaters) stretch the bounding box a thousandfold; the grid is laid over the 0.5 - 99.5 %
    quantile range instead, so the search stays local -- and exact, outliers included."""
    rg = pkg("region_growing")
    rng = np.random.default_rng(8)
    pos = blobs(rng, 100_000)
    far = rng.uniform(-3000, 3000, size=(150, 3)).astype(np.float32)
    pos = np.concatenate((pos, far))[rng.permutation(100_150)]
    dpos = torch.from_numpy(pos).cuda()
    rg.knn_pca(dpos, 64, want_knn=True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    got = rg.knn_pca(dpos, 64, want_knn=True, want_stats=True)
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    visited = float(got["stats"][1]) / (len(pos) * 64)
    print(f"\n100 150 points with 150 floaters, k = 64: {ms:.1f} ms, {visited:.1f} points visited per neighbour found")
    assert visited < 200                                  # the whole cloud in one cell would be ~3000
    far_rows = np.flatnonzero(np.abs(pos).max(1) > 100)[:40]
    knn = got["knn"].cpu().numpy()
    for q0 in (0, 50_000):                                # two slices of ordinary points ...
        ref = oracle.region_knn_pca(pos, 64, want_knn=True, queries=(q0, q0 + 300))
        assert np.array_equal(knn[q0:q0 + 300], ref["knn"][q0:q0 + 300])
    for r in far_rows:                                    # ... and the floaters themselves
        ref = oracle.region_knn_pca(pos, 64, want_knn=True, queries=(int(r), int(r) + 1))
        assert np.array_equal(knn[r], ref["knn"][r])
