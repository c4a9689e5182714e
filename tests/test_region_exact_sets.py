"""Exact neighbour SETS of gsl_region_knn_pca (csrc/region_growing.cu) for k > 64, against a plain
float64 NumPy reference.  For k <= 64 the kernel returns neighbour lists and tests/test_gpu_region.py
compares them; above that only the set's moments leave the kernel, so the float64 centroid serves as
a fingerprint of the set.

Reference (`exact_knn`, `moments`):
  * d2 = ((dx*dx) + (dy*dy)) + (dz*dz), dx = float64(p) - float64(q), no FMA; the set is every point
    with d2 < t plus the lowest indices with d2 == t, t = the k-th smallest d2 (DESIGN.md 4.9);
  * centroid q + fsum(p - q) / k; covariance of the centred neighbours; numpy.linalg.eigh's smallest
    eigenvector, oriented by rg:120-121 (flip when dot(normal, q - centroid) > 0); residual |n . (q - c)|.

Bars (u = 2^-53, r = sqrt(t) bounds every |p - q| of the set):
  * centroid, per coordinate: 1e-12 * max(1, r) + 2^-50 * |q|_inf.  The kernel's lane-strided float64
    sums of k terms of size <= r are off by about (k/32 + 6) u r (7.4e-15 r at k = 2000); adding q
    costs half an ulp of the result on either side.  `test_one_point_error_is_visible` proves the bar
    sees a wrong set: trading the k-th neighbour for the next point (same order, other coordinates)
    moves the centroid by at least 100 times the bar on every sampled query.
  * normal, where (lambda_1 - lambda_0) / lambda_2 >= 1e-2: angle atan2(|n x n_ref|, |n . n_ref|) <= 1e-9
    (the angle, not 1 - |cos|, which cannot resolve below 1e-16).  Covariance rounding over a gap of
    1e-2 lambda_2 gives angles near 1e-12; one wrong neighbour turns the normal by ~1e-4.  The orientation
    must agree where |n_ref . (q - c)| clears both the angle and the centroid errors.
  * residual with the reference normals handed in: within the centroid bar.

Each GPU case is built to reach one branch of the selection; where the library's work counters can
show that it did, the test asserts it."""
import functools
import math

import numpy as np
import pytest

from util import blobs, pkg

GAP_MIN = 1e-2
ANGLE_TOL = 1e-9


# ---- reference -----------------------------------------------------------------------------------
def exact_knn(pos, k, queries):
    """Neighbour sets of `queries`: int32 [len(queries), k] ordered by (d2, index), whether the query has
    an exact tie at the k-th distance, that distance t, and the first point after the set in the same
    order whose coordinates differ from the k-th neighbour's (-1 if there is none)."""
    p = np.asarray(pos, np.float64)
    n = len(p)
    sets = np.empty((len(queries), k), np.int32)
    tie = np.zeros(len(queries), bool)
    t = np.empty(len(queries))
    nxt = np.full(len(queries), -1, np.int64)
    for r, q in enumerate(queries):
        d = p - p[q]
        d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
        t[r] = d2[np.argpartition(d2, k - 1)[k - 1]]
        below = np.flatnonzero(d2 < t[r])
        at = np.flatnonzero(d2 == t[r])
        s = np.concatenate((below, at[:k - len(below)]))
        sets[r] = s[np.lexsort((s, d2[s]))]
        tie[r] = len(at) > k - len(below)
        if k < n:
            rest = d2.copy()
            rest[s] = np.inf
            rest[(p == p[sets[r, -1]]).all(1)] = np.inf
            j = int(np.argmin(rest))                       # the first minimum: lowest index on a tie
            nxt[r] = j if np.isfinite(rest[j]) else -1
    return sets, tie, t, nxt


def moments(pos, q, sel):
    """Float64 centroid, oriented normal, relative eigen-gap and residual of the neighbour set `sel` of
    query q."""
    p = np.asarray(pos, np.float64)
    d = p[sel] - p[q]
    m = np.array([math.fsum(d[:, a]) for a in range(3)]) / len(sel)
    e = d - m
    w, v = np.linalg.eigh(e.T @ e)
    nrm = v[:, 0]
    if nrm @ -m > 0:                                       # rg:120-121, q - centroid = -m
        nrm = -nrm
    gap = (w[1] - w[0]) / w[2] if w[2] > 0 else 0.0
    return p[q] + m, nrm, gap, abs(nrm @ m)


def centroid_tol(pos, queries, t):
    return 1e-12 * np.maximum(1.0, np.sqrt(t)) + 2.0 ** -50 * np.abs(np.asarray(pos, np.float64)[queries]).max(1)


# ---- clouds: each returns (float32 points in shuffled order, query indices) ---------------------------
def _shuffle(rng, pos, queries):
    perm = rng.permutation(len(pos))
    where = np.empty_like(perm)
    where[perm] = np.arange(len(pos))
    return np.ascontiguousarray(pos[perm], np.float32), np.sort(where[queries])


def _sample(rng, n, m):
    return np.arange(n) if n <= m else rng.choice(n, m, replace=False)


def _blobs_c1(rng):
    pos = blobs(rng, 200_000)                              # BASELINE config C1's cloud size
    return pos, _sample(rng, len(pos), 300)


def _lattice(rng):
    ax = np.arange(30, dtype=np.float32)
    pos = np.stack(np.meshgrid(ax, ax, ax, indexing="ij"), -1).reshape(-1, 3)
    return _shuffle(rng, pos, _sample(rng, len(pos), 400))


def _quantized(rng):
    # float32 spacing at 1000 is 6.1e-5: many points share coordinates, and some distances tie
    pos = (rng.normal(0, 0.02, (60_000, 3)) + 1000.0).astype(np.float32)
    return pos, _sample(rng, len(pos), 400)


def _copies(rng):
    # queries: 1500 points within 0.05 of the origin.  600 copies of (1, 0, 0) come next, the background
    # lies beyond 1.5.  k = 1800 takes 300 of the 600 tied copies: a bucket of 600 tied through every
    # digit, resolved by serial lowest-index picks; k = 2100 takes all of them (need == bucket, `exact`).
    near = rng.normal(size=(1500, 3))
    near *= (0.05 * rng.uniform(0, 1, 1500) ** (1 / 3) / np.linalg.norm(near, axis=1))[:, None]
    far = rng.normal(size=(20_000, 3))
    far *= (rng.uniform(1.6, 3.0, 20_000) / np.linalg.norm(far, axis=1))[:, None]
    pos = np.concatenate((near, np.tile([1.0, 0.0, 0.0], (600, 1)), far))
    return _shuffle(rng, pos, np.arange(1500))


def _clumps(rng):
    # 40 clumps of 2500 points (sigma 1e-5) on a unit grid: the 2000-th distance (~2e-5) lies far below
    # R / 32 of any cube that holds a clump, so the leading digit is 0 and the select restarts on raw keys
    grid = np.stack(np.meshgrid(np.arange(4), np.arange(4), np.arange(3), indexing="ij"), -1).reshape(-1, 3)
    centres = grid[rng.choice(len(grid), 40, replace=False)]
    clumps = (centres[:, None, :] + rng.normal(0, 1e-5, (40, 2500, 3))).reshape(-1, 3)
    back = rng.uniform([-0.5, -0.5, -0.5], [3.5, 3.5, 2.5], (50_000, 3))
    pos = np.concatenate((clumps, back))
    queries = np.concatenate((rng.choice(100_000, 300, replace=False), 100_000 + rng.choice(50_000, 100, replace=False)))
    return _shuffle(rng, pos, queries)


def _floaters(_rng):
    # the cloud of test_gpu_region.test_floaters_do_not_degrade_the_grid, with its seed
    rng = np.random.default_rng(8)
    pos = blobs(rng, 100_000)
    far = rng.uniform(-3000, 3000, size=(150, 3)).astype(np.float32)
    pos = np.concatenate((pos, far))[rng.permutation(100_150)]
    floaters = np.flatnonzero(np.abs(pos).max(1) > 100)
    others = np.setdiff1d(np.arange(len(pos)), floaters)
    return pos, np.sort(np.concatenate((floaters, np.random.default_rng(9).choice(others, 300, replace=False))))


def _near_n(n):
    def build(rng):
        # 3 outliers 50 - 100 units out: k close to N needs the whole array (level 0, R^2 = inf)
        out = rng.uniform(50, 100, (3, 3)) * rng.choice([-1.0, 1.0], (3, 3))
        pos = np.concatenate((blobs(rng, n - 3), out))
        q = np.union1d(_sample(rng, n - 3, 397), np.arange(n - 3, n))
        return _shuffle(rng, pos, q)
    return build


def _plane(rng):
    pos = np.zeros((100_000, 3))
    pos[:, :2] = rng.uniform(-2, 2, (100_000, 2))
    return _shuffle(rng, pos, _sample(rng, len(pos), 400))


def _line(rng):
    pos = np.zeros((20_000, 3))
    pos[:, 0] = rng.uniform(-2, 2, 20_000)
    return _shuffle(rng, pos, _sample(rng, len(pos), 400))


def _sheets(rng):
    pos = np.zeros((100_000, 3))
    pos[:, :2] = rng.uniform(-1, 1, (100_000, 2))
    pos[50_000:, 2] = 1e-3
    return _shuffle(rng, pos, _sample(rng, len(pos), 400))


CLOUDS = {
    "blobs": _blobs_c1, "lattice": _lattice, "quantized": _quantized, "copies": _copies, "clumps": _clumps,
    "floaters": _floaters, "near65": _near_n(65), "near66": _near_n(66), "near300": _near_n(300),
    "near3000": _near_n(3000), "plane": _plane, "line": _line, "sheets": _sheets,
}
SET_CASES = [("blobs", 65), ("blobs", 256), ("blobs", 1000), ("blobs", 2000),
             ("lattice", 100), ("lattice", 500), ("lattice", 2000),
             ("quantized", 100), ("quantized", 2000),
             ("copies", 1800), ("copies", 2100),
             ("clumps", 2000),
             ("floaters", 2000),
             ("near65", 65), ("near65", 64), ("near66", 66), ("near66", 65),
             ("near300", 300), ("near300", 299), ("near300", 65),
             ("near3000", 3000), ("near3000", 2999), ("near3000", 65),
             ("plane", 2000), ("line", 500), ("sheets", 2000)]
LIST_CLOUDS = ["lattice", "quantized", "copies", "clumps", "floaters", "near300", "plane", "line", "sheets"]
LIST_QUERIES = 200


@functools.lru_cache(maxsize=None)
def cloud(name):
    return CLOUDS[name](np.random.default_rng(sorted(CLOUDS).index(name) + 100))


@functools.lru_cache(maxsize=None)
def reference(name, k):
    pos, queries = cloud(name)
    if k <= 64:
        queries = queries[:LIST_QUERIES]
    sets, tie, t, nxt = exact_knn(pos, k, queries)
    rows = [moments(pos, q, s) for q, s in zip(queries, sets)]
    return dict(queries=queries, sets=sets, tie=tie, t=t, nxt=nxt, tol=centroid_tol(pos, queries, t),
                centroid=np.array([r[0] for r in rows]), normal=np.array([r[1] for r in rows]),
                gap=np.array([r[2] for r in rows]), residual=np.array([r[3] for r in rows]))


# ---- CPU: the reference and the bar ---------------------------------------------------------------------
def _small_clouds():
    rng = np.random.default_rng(5)
    ax = np.arange(17, dtype=np.float32)
    lat = np.stack(np.meshgrid(ax, ax, ax, indexing="ij"), -1).reshape(-1, 3)
    base = blobs(rng, 1600)
    dup = np.concatenate((base, base, base))
    quant = (rng.normal(0, 0.005, (5000, 3)) + 1000.0).astype(np.float32)
    return {name: c[rng.permutation(len(c))] for name, c in (("lattice", lat), ("duplicates", dup), ("quantized", quant))}


@pytest.mark.parametrize("k", [65, 200, 1000])
@pytest.mark.parametrize("name", ["lattice", "duplicates", "quantized"])
def test_reference_equals_the_oracle(oracle, name, k):
    """exact_knn orders its sets like the brute-force C oracle's neighbour lists, ties included."""
    pos = _small_clouds()[name]
    q0, q1 = 1000, 1300
    want = oracle.region_knn_pca(pos, k, want_knn=True, queries=(q0, q1))["knn"][q0:q1]
    sets, tie, _, _ = exact_knn(pos, k, np.arange(q0, q1))
    assert np.array_equal(sets, want)
    assert tie.any()                                       # the tie rule is exercised


@pytest.mark.parametrize("name, k", SET_CASES)
def test_one_point_error_is_visible(name, k):
    """Trading the k-th neighbour for the next distinct point moves the centroid by >= 100x its bar."""
    pos, _ = cloud(name)
    ref = reference(name, k)
    ok = ref["nxt"] >= 0
    if k < len(pos):
        assert ok.all()
    p = pos.astype(np.float64)
    move = np.abs(p[ref["nxt"][ok]] - p[ref["sets"][ok, -1]]).max(1) / k
    assert (move >= 100 * ref["tol"][ok]).all(), (move / ref["tol"][ok]).min()


# ---- GPU --------------------------------------------------------------------------------------------------
def _angle(a, b):
    return np.arctan2(np.linalg.norm(np.cross(a, b), axis=1), np.abs((a * b).sum(1)))


@pytest.mark.gpu
@pytest.mark.parametrize("name, k", SET_CASES)
def test_sets_equal_the_exact_reference(name, k):
    """Centroids, normals and residuals of one call over the whole cloud, checked on the sampled queries."""
    rg = pkg("region_growing")
    pos, _ = cloud(name)
    n = len(pos)
    ref = reference(name, k)
    q = ref["queries"]
    got = rg.knn_pca(pos, k, want_centroids=True, want_stats=True)
    nin = np.zeros((n, 3))
    nin[:, 2] = 1.0
    nin[q] = ref["normal"]
    res = rg.knn_pca(pos, k, normals_in=nin, want_normals=False)["residuals"].cpu().numpy()[q]
    cen_all = got["centroids"].cpu().numpy()
    nrm_all = got["normals"].cpu().numpy()
    st = got["stats"].cpu().numpy()
    cen, nrm = cen_all[q], nrm_all[q]

    err = np.abs(cen - ref["centroid"]).max(1) / ref["tol"]
    ok = ref["gap"] >= GAP_MIN
    ang = _angle(nrm, ref["normal"])
    print(f"\n{name:9s} N={n:6d} k={k:4d}: {len(q)} queries, {int(ref['tie'].sum())} with a tie at the k-th distance, "
          f"centroid error <= {err.max():.2g} of the bar, normal angle <= {ang[ok].max() if ok.any() else 0:.2g} "
          f"({int(ok.sum())} well defined); per query: {st[0] / n:.2f} walks, {st[1] / (n * k):.2f} points visited "
          f"per neighbour, {st[2] / n:.2f} cubes too small, {st[3] / n:.2f} select walks")
    bad = np.flatnonzero(err > 1)
    assert len(bad) == 0, [(int(q[i]), cen[i].tolist(), ref["centroid"][i].tolist(), float(ref["t"][i]), bool(ref["tie"][i]))
                           for i in bad[:5]]
    assert (ang[ok] <= ANGLE_TOL).all(), [(int(q[i]), float(ang[i])) for i in np.flatnonzero(ok & (ang > ANGLE_TOL))[:5]]
    # orientation: the same side wherever the point's offset from its plane exceeds both errors
    margin = 2 * (ANGLE_TOL * np.linalg.norm(ref["centroid"] - pos[q].astype(np.float64), axis=1) + np.sqrt(3) * ref["tol"])
    sided = ok & (ref["residual"] > margin)
    assert ((nrm * ref["normal"]).sum(1)[sided] > 0).all()
    assert (np.abs(res - ref["residual"]) <= ref["tol"]).all()

    # evidence that the case reaches the branch it was built for
    if name == "lattice":
        assert ref["tie"].mean() > 0.9
    if name == "quantized":
        assert ref["tie"].any()
    if name == "copies" and k == 1800:
        assert ref["tie"].all()
        assert st[0] >= 1500 * 300                         # serial lowest-index picks: one walk per tied copy taken
    if name == "copies" and k == 2100:
        # need == bucket for the queries.  The counters cannot show it: they sum over every point, and
        # background points whose set takes only some of the copies do walk the serial path.
        assert not ref["tie"].any()
    if name.startswith("near") and k == n:
        # level 0 for every query: no validating walk (select walks + one moments walk each), and every
        # walk visits the whole array
        assert st[0] == st[3] + n and st[1] == st[0] * n
    if name == "clumps":
        assert st[3] >= 100_000                            # every clump point restarts its select on raw keys
    if name == "plane":
        assert (nrm_all[:, :2] == 0).all() and (np.abs(nrm_all[:, 2]) == 1).all()
        assert (got["residuals"].cpu().numpy() == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [33, 64])
@pytest.mark.parametrize("name", LIST_CLOUDS)
def test_lists_equal_the_exact_reference(name, k):
    """The k <= 64 variants of the same clouds: the list is the reference's (d2, index) order."""
    rg = pkg("region_growing")
    pos, _ = cloud(name)
    ref = reference(name, k)
    q = ref["queries"]
    got = rg.knn_pca(pos, k, want_knn=True, want_centroids=True)
    knn = got["knn"].cpu().numpy()[q]
    bad = np.flatnonzero((knn != ref["sets"]).any(1))
    assert len(bad) == 0, [(int(q[i]), knn[i].tolist(), ref["sets"][i].tolist()) for i in bad[:3]]
    assert (np.abs(got["centroids"].cpu().numpy()[q] - ref["centroid"]).max(1) <= ref["tol"]).all()
