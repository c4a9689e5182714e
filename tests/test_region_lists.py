"""Neighbour lists of gsl_region_knn_pca (csrc/region_growing.cu) for 64 < k <= GSL_REGION_MAX_LIST.

Above k = 64 the selector writes every chosen index straight out in walk order and knn_order_kernel
sorts each row by (squared distance, index), KDTree.query's order.  The lists are checked
  * against the brute-force C oracle, bit for bit, on the clouds of test_region_exact_sets.py that
    reach each branch of the selection (and on 600 coincident points);
  * against scipy's cKDTree: sqrt of the recomputed squared distance along the list equals scipy's
    distance row bit for bit, and the index rows are equal wherever no two of the first k + 1 squared
    distances tie (on an exact tie scipy's order follows its tree layout: the documented exemption);
  * for structure (k distinct indices in [0, N), the query itself unless more than k points coincide
    with it, k = 64 and k = 65 agreeing on their first 64 entries), for leaving the normals,
    residuals, centroids and work counters bit-identical, for row offsets past 2^31, through
    segmentation_3D, and at the limit."""
import functools
import math
import os
import re

import numpy as np
import pytest
import torch

from test_region_exact_sets import centroid_tol, cloud
from util import GOLDEN, blobs, pkg

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
with open(os.path.join(ROOT, "include", "gslift.h")) as _f:
    MAX_LIST = int(re.search(r"#define\s+GSL_REGION_MAX_LIST\s+(\d+)", _f.read()).group(1))
ROWS = 200                                                  # queries compared per large cloud


def _coincident(rng):
    # 600 copies of one point among 5000 others: k = 300 takes the 300 lowest indices of the copies,
    # k = 600 takes exactly all of them
    back = rng.uniform(-1, 1, (5000, 3))
    back = back[np.linalg.norm(back, axis=1) > 0.2]
    pos = np.concatenate((np.tile([0.0, 0.0, 0.0], (600, 1)), back)).astype(np.float32)
    perm = rng.permutation(len(pos))
    pos = np.ascontiguousarray(pos[perm])
    copies = np.flatnonzero((pos == 0).all(1))
    return pos, np.sort(np.concatenate((copies[:150], rng.choice(np.setdiff1d(np.arange(len(pos)), copies), 50, replace=False))))


@functools.lru_cache(maxsize=None)
def points(name):
    """(float32 points, sorted query rows) of one cloud."""
    if name == "coincident":
        return _coincident(np.random.default_rng(31))
    pos, q = cloud(name)
    if len(q) > ROWS:
        q = np.sort(np.random.default_rng(len(pos)).choice(q, ROWS, replace=False))
    return pos, q


def oracle_rows(oracle, pos, k, rows):
    """The oracle's lists of `rows` (sorted), one call per contiguous run."""
    out = np.empty((len(rows), k), np.int32)
    start = 0
    while start < len(rows):
        end = start + 1
        while end < len(rows) and rows[end] == rows[end - 1] + 1:
            end += 1
        q0, q1 = int(rows[start]), int(rows[end - 1]) + 1
        out[start:end] = oracle.region_knn_pca(pos, k, want_knn=True, queries=(q0, q1))["knn"][q0:q1]
        start = end
    return out


def run(pos, k, knn=True, fill=-1, stats=False):
    """gsl_region_knn_pca through the C ABI with a list buffer pre-filled with `fill`: returns the device
    outputs (normals, residuals, centroids, optional knn and stats)."""
    native = pkg("_native")
    ops = pkg("ops")
    d = pos if isinstance(pos, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(pos, np.float32)).cuda()
    n = d.shape[0]
    out = dict(normals=torch.empty((n, 3), dtype=torch.float64, device=d.device),
               residuals=torch.empty(n, dtype=torch.float64, device=d.device),
               centroids=torch.empty((n, 3), dtype=torch.float64, device=d.device))
    if knn:
        out["knn"] = torch.full((n, k), fill, dtype=torch.int32, device=d.device)
    if stats:
        out["stats"] = torch.zeros(4, dtype=torch.int64, device=d.device)
    L = native.lib()
    ws = ops._ws.get(d.device, L.gsl_region_workspace_bytes(n))
    native.check(L.gsl_region_knn_pca(d.data_ptr(), n, int(k), None, out["normals"].data_ptr(), out["residuals"].data_ptr(),
                                      out["centroids"].data_ptr(), out["knn"].data_ptr() if knn else None,
                                      out["stats"].data_ptr() if stats else None, ws.data_ptr(), ws.numel(), ops._stream()))
    torch.cuda.synchronize()
    return out


def sq_dist(pos, q, idx):
    """float64 squared distances of points idx from point q in scipy's order ((dx*dx + dy*dy) + dz*dz)."""
    p = np.asarray(pos, np.float64)
    d = p[idx] - p[q][..., None, :] if np.ndim(q) else p[idx] - p[q]
    return (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]


ORACLE_CASES = [("blobs", 65), ("blobs", 100), ("blobs", 257), ("blobs", 2000),
                ("lattice", 65), ("lattice", 100), ("lattice", 257), ("lattice", 2000), ("lattice", MAX_LIST),
                ("quantized", 100), ("quantized", 2000), ("quantized", MAX_LIST),
                ("copies", 257), ("copies", 1800), ("copies", 2100), ("copies", MAX_LIST),
                ("coincident", 300), ("coincident", 600),
                ("clumps", 100), ("clumps", 2000),
                ("floaters", 65), ("floaters", 2000),
                ("near65", 65), ("near66", 66), ("near300", 300), ("near300", 257), ("near3000", 3000), ("near3000", 2000),
                ("plane", 65), ("plane", 2000), ("line", 257), ("line", 2000), ("line", MAX_LIST),
                ("sheets", 100), ("sheets", 2000)]


@pytest.mark.parametrize("name, k", ORACLE_CASES)
def test_lists_equal_the_oracle(oracle, name, k):
    """Every sampled row (every row when N <= 3000) equals the brute-force oracle's list bit for bit, and the
    whole output is k distinct indices in [0, N) per row, with no pre-filled -1 left."""
    pos, q = points(name)
    n = len(pos)
    if n <= 3000:
        q = np.arange(n)
    got = run(pos, k)["knn"]
    want = oracle_rows(oracle, pos, k, q)
    mine = got[torch.from_numpy(q).cuda()].cpu().numpy()
    bad = np.flatnonzero((mine != want).any(1))
    assert len(bad) == 0, [(int(q[i]), int(np.argmax(mine[i] != want[i]))) for i in bad[:5]]
    # structure of every row, checked on the device
    assert int(got.min()) >= 0 and int(got.max()) < n
    s = torch.sort(got, dim=1).values
    assert bool((s[:, 1:] != s[:, :-1]).all())


SCIPY_CASES = [("blobs", 2000), ("lattice", 100), ("quantized", 2000), ("copies", 1800), ("clumps", 2000),
               ("floaters", 257), ("plane", 257), ("sheets", 2000), ("near3000", 3000), ("coincident", 300)]


@pytest.mark.parametrize("name, k", SCIPY_CASES)
def test_lists_equal_scipy_ckdtree(name, k):
    """sqrt of our squared distances equals cKDTree.query's distances bit for bit; index rows are equal wherever
    the first k + 1 squared distances have no exact tie."""
    from scipy.spatial import cKDTree
    pos, q = points(name)
    n = len(pos)
    mine = run(pos, k)["knn"][torch.from_numpy(q).cuda()].cpu().numpy()
    kk = min(k + 1, n)
    dist, idx = cKDTree(pos).query(pos[q], kk)
    dist, idx = dist.reshape(len(q), kk), idx.reshape(len(q), kk)
    d2 = sq_dist(pos, q, mine)
    assert np.array_equal(np.sqrt(d2), dist[:, :k])
    assert (np.diff(d2, axis=1) >= 0).all()
    d2s = sq_dist(pos, q, idx)
    untied = (np.diff(d2s, axis=1) > 0).all(1)
    assert np.array_equal(mine[untied], idx[untied, :k])
    print(f"\n{name} k={k}: {len(q)} rows, {int(untied.sum())} without a tie")
    if name == "blobs":
        assert untied.mean() > 0.9                        # the index comparison is not vacuous


@pytest.mark.parametrize("name, k", [("blobs", 65), ("blobs", 2000), ("lattice", 257), ("copies", 1800),
                                     ("coincident", 300), ("coincident", 600), ("clumps", 2000), ("near300", 300)])
def test_list_structure_and_unchanged_outputs(name, k):
    """Each row holds its own query unless more than k points coincide with it (then the k lowest indices of
    those points); normals, residuals, centroids and work counters are the same bits with and without lists;
    the float64 centroid of every sampled list matches the kernel's."""
    pos, q = points(name)
    n = len(pos)
    with_list = run(pos, k, stats=True)
    without = run(pos, k, knn=False, stats=True)
    for key in ("normals", "residuals", "centroids", "stats"):
        assert torch.equal(with_list[key], without[key]), key
    knn = with_list["knn"]
    rows = torch.arange(n, device=knn.device)
    has_self = (knn == rows[:, None]).any(1).cpu().numpy()
    _, inverse, counts = torch.unique(torch.from_numpy(pos).cuda(), dim=0, return_inverse=True, return_counts=True)
    same = counts[inverse].cpu().numpy()                  # points at the query's coordinates, itself included
    crowded = same > k
    assert has_self[~crowded].all()
    for r in np.flatnonzero(crowded)[:50]:
        group = np.flatnonzero((pos == pos[r]).all(1))
        assert np.array_equal(np.sort(knn[r].cpu().numpy()), group[:k])
    if name == "coincident":
        assert crowded.sum() == (600 if k < 600 else 0)
    # the kernel's centroid against q + fsum(p - q) / k over the emitted list
    lists = knn[torch.from_numpy(q).cuda()].cpu().numpy()
    p64 = pos.astype(np.float64)
    cen = np.array([p64[r] + np.array([math.fsum(c) for c in (p64[lists[i]] - p64[r]).T]) / k for i, r in enumerate(q)])
    t = sq_dist(pos, q, lists).max(1)
    assert (np.abs(with_list["centroids"].cpu().numpy()[q] - cen).max(1) <= centroid_tol(pos, q, t)).all()


def test_k64_and_k65_agree_on_64_entries():
    """(d2, index) is a total order: the k = 64 list (ordered inside the selector) is the first 64 entries of
    the k = 65 list (ordered by knn_order_kernel)."""
    for name in ("blobs", "lattice", "quantized", "copies"):
        pos, _ = points(name)
        a = run(pos, 64)["knn"]
        b = run(pos, 65)["knn"]
        assert torch.equal(a, b[:, :64]), name


def test_row_offsets_past_2_31(oracle):
    """1.1 M points with k = 2000: N * k > 2^31 list entries.  The rows around entry 2^31 and the last rows equal
    the oracle's."""
    rng = np.random.default_rng(11)
    n, k = 1_100_000, 2000
    assert n * k > 2 ** 31
    pos = blobs(rng, n)
    knn = run(pos, k)["knn"]
    edge = 2 ** 31 // k
    for q0, q1 in ((edge - 2, edge + 3), (n - 40, n)):
        rows = np.arange(q0, q1)
        mine = knn[q0:q1].cpu().numpy()
        assert np.array_equal(mine, oracle_rows(oracle, pos, k, rows)), (q0, q1)
    del knn
    torch.cuda.empty_cache()


def _load(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    return {key: z[key] for key in z.files}


@pytest.mark.parametrize("name, k", [("region_planes_k40", 100), ("region_planes_k40", 1000),
                                     ("region_planes_k400", 100), ("region_planes_k400", 1000),
                                     ("region_planes_k2000", 100), ("region_planes_k2000", 1000),
                                     ("region_planes_k2000", 2000)])
def test_segmentation_3d_with_long_lists(oracle, name, k):
    """segmentation_3D with k > 64 returns the oracle's regions over the oracle's lists, largest first (rg:219)."""
    rg = pkg("region_growing")
    g = _load(name)
    pos = g["pos"]
    regions = rg.segmentation_3D(pos, g["normals"], g["residuals"], residual_threshold=0.1, angle_threshold=0.05, k=k)
    ref_knn = oracle.region_knn_pca(pos, k, want_knn=True)["knn"]
    region_of, r = oracle.region_grow(ref_knn, g["normals"], g["residuals"], 0.1, 0.05)
    want = [np.flatnonzero(region_of == i).tolist() for i in range(r)]
    want.sort(key=len, reverse=True)
    assert regions == want
    print(f"\n{name} k={k}: {len(regions)} regions, largest {len(regions[0])}")


def test_limit():
    """k = GSL_REGION_MAX_LIST + 1 with lists requested raises GslError naming the limit; without lists the
    normals are still computed."""
    rg = pkg("region_growing")
    native = pkg("_native")
    pos = blobs(np.random.default_rng(12), MAX_LIST + 5000)
    with pytest.raises(native.GslError, match=str(MAX_LIST)):
        rg.knn_pca(pos, MAX_LIST + 1, want_knn=True)
    nrm = rg.knn_pca(pos, MAX_LIST + 1, want_residuals=False)["normals"]
    assert bool(torch.isfinite(nrm).all())
    assert float((nrm.norm(dim=1) - 1).abs().max()) < 1e-12
