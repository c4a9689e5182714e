"""The reference-order K-means update (update="ordered") against NumPy itself.

The reference forms every centroid as `data[labels == c].mean(axis=0)` (km:125-128), and the
ordered update promises those float32 values bit for bit.  Here NumPy's own expression is the
reference, not the C oracle, so a wrong model of NumPy's arithmetic shared by the kernel and the
oracle cannot hide.  NumPy's add.reduce starts from +0.0; for D >= 2 it sums the rows of the
gathered block in order, for D = 1 the column goes through its pairwise summation.

Centroids are compared by their bits (assert_bits_equal), so -0.0 against +0.0 fails.
The GPU tests call ops.kmeans_update_ordered with synthetic, shuffled labels so that the cluster
sizes are chosen exactly (block, batch and stage-ring edges of the kernels, edges of the pairwise
tree) and K = 1024 and D = 256 are reached.
"""
import contextlib
import io

import numpy as np
import pytest
import torch

from util import assert_bits_equal, pkg

F32 = np.float32
DEV = "cuda"
HELPER_MIN_N = 1 << 18          # from this N on, clusters with >= 1/16 of the members run on a helper stream
BAD_LABELS = (-1, None, 2**31 - 1, -2**31)    # None stands for K


# ---- the reference ---------------------------------------------------------------------------------------
def ref_update(data, labels, old):
    """km:126 literally, over the rows whose label lies in [0, K)."""
    K = len(old)
    keep = (labels >= 0) & (labels < K)
    data, labels = data[keep], labels[keep]
    return np.array([data[labels == c].mean(axis=0) if np.sum(labels == c) > 0 else old[c] for c in range(K)],
                    dtype=F32).reshape(old.shape)


def ref_update_sorted(data, labels, old):
    """The same means over contiguous slices of the rows sorted stably by label.  A slice of a C-contiguous
    array along axis 0 is C-contiguous, as data[mask] is, so NumPy sums it the same way (asserted below)."""
    K = len(old)
    idx = np.flatnonzero((labels >= 0) & (labels < K))
    order = idx[np.argsort(labels[idx], kind="stable")]
    rows = data[order]
    bounds = np.searchsorted(labels[order], np.arange(K + 1))
    new = old.copy()
    for c in range(K):
        if bounds[c + 1] > bounds[c]:
            new[c] = rows[bounds[c]:bounds[c + 1]].mean(axis=0)
    return new


def pairwise_sum(a):
    """NumPy's pairwise_sum (numpy/_core/src/umath/loops_utils.h.src) restated, float32 throughout."""
    n = len(a)
    if n < 8:
        res = F32(0.0)
        for v in a:
            res = F32(res + v)
        return res
    if n <= 128:
        m = n - n % 8
        r = a[:8].copy()
        for i in range(8, m, 8):
            r = r + a[i:i + 8]                      # eight float32 accumulators, elementwise
        res = F32(F32(F32(r[0] + r[1]) + F32(r[2] + r[3])) + F32(F32(r[4] + r[5]) + F32(r[6] + r[7])))
        for v in a[m:]:
            res = F32(res + v)
        return res
    n2 = n // 2
    n2 -= n2 % 8
    return F32(pairwise_sum(a[:n2]) + pairwise_sum(a[n2:]))


def pairwise_mean(a):
    """mean of a float32 (n, 1) column: the reduction's identity plus the pairwise sum, divided in float64."""
    return F32(np.float64(F32(F32(0.0) + pairwise_sum(a))) / len(a))


# ---- case construction -----------------------------------------------------------------------------------
def make_labels(sizes, rng, n_bad=0):
    """int32 labels with exactly sizes[c] rows of cluster c (and n_bad rows of out-of-range labels), shuffled
    so that a cluster's members are spread over the scatter's tiles and warps."""
    K = len(sizes)
    lab = np.repeat(np.arange(K, dtype=np.int64), sizes)
    if n_bad:
        bad = np.array([K if b is None else b for b in BAD_LABELS], np.int64)
        lab = np.concatenate([lab, bad[rng.integers(0, len(bad), n_bad)]])
    return rng.permutation(lab).astype(np.int32)


def normal_data(rng, n, d):
    """N(3, 1): the summation order changes the rounding."""
    return (rng.standard_normal((n, d), dtype=F32) + F32(3.0)).astype(F32)


BASE_SIZES = [0, 1, 3, 4, 5, 31, 32, 33, 63, 64, 65, 511, 512, 513, 1535, 1536, 1537, 3077]
D1_SIZES = [7, 8, 9, 127, 128, 129, 136, 137, 255, 256, 257]       # edges of the pairwise rule
SMALL_SIZES = [0, 1, 3, 4, 5, 31, 32, 33, 63, 64, 65]


def cycle(sizes, K, big=None):
    out = [sizes[c % len(sizes)] for c in range(K)]
    if big:
        out[0] = big
    return out


def value_cases():
    """(name, data, labels, old) with special values; shared by the oracle test and the GPU test."""
    rng = np.random.default_rng(77)
    cases = []
    for d in (1, 3):
        sizes = [1, 5, 9, 33, 130, 700, 0]
        lab = make_labels(sizes, rng)
        n = len(lab)
        old = normal_data(rng, len(sizes), d)

        x = normal_data(rng, n, d)
        x[:, 0] = -0.0                                                   # a column of -0.0 sums to +0.0
        cases.append((f"negative zero column d{d}", x, lab, old))

        x = normal_data(rng, n, d)
        x[:, -1] = (rng.standard_normal(n) * 1e-42).astype(F32)          # subnormal sums
        if d > 1:
            x[:, 1] = (rng.uniform(0.5, 1.0, n) * 1e-38).astype(F32)     # subnormal rows, sums that become normal
        cases.append((f"subnormal d{d}", x, lab, old))
        x = (rng.uniform(0.5, 1.0, (n, d)) * 1e-38).astype(F32)
        cases.append((f"subnormal to normal d{d}", x, lab, old))

        x = normal_data(rng, n, d)
        x[:, 0] = (rng.uniform(2.0, 3.4, n) * 1e38).astype(F32)         # the sum overflows part-way
        x[:, -1] = F32(3e38) * rng.choice([F32(1), F32(-1)], n)         # whether it overflows depends on the order
        cases.append((f"near max d{d}", x, lab, old))
        alt = np.tile(np.array([3e38, -3e38], F32), (n + 1) // 2)[:n]   # +,-,+,-: never overflows in order
        x = normal_data(rng, n, d)
        x[:, 0] = alt[np.argsort(np.argsort(lab, kind="stable"), kind="stable")]
        cases.append((f"alternating max d{d}", x, lab, old))

        x = normal_data(rng, n, d)
        members = [np.flatnonzero(lab == c) for c in range(len(sizes))]
        x[members[1][2], 0] = np.inf                                     # +inf
        x[members[3][0], 0], x[members[3][7], 0] = np.inf, -np.inf       # inf - inf = NaN
        x[members[4][100], -1] = np.nan
        x[members[5][3], -1] = -np.inf
        cases.append((f"inf and nan d{d}", x, lab, old))
    return cases


# ---- CPU ---------------------------------------------------------------------------------------------------
def test_pairwise_restatement_equals_numpy_for_one_feature():
    """Pins the D = 1 rule the kernel and the oracle implement: NumPy's mean of an (n, 1) block."""
    rng = np.random.default_rng(1)
    for n in list(range(1, 301)) + [8191, 8192, 8193, 1_000_003]:
        x = normal_data(rng, n, 1)
        assert_bits_equal(pairwise_mean(x[:, 0]), x.mean(axis=0)[0], f"n={n}")
        z = np.full((n, 1), -0.0, F32)
        assert_bits_equal(pairwise_mean(z[:, 0]), z.mean(axis=0)[0], f"-0.0, n={n}")
        assert_bits_equal(z.mean(axis=0), np.zeros(1, F32), f"-0.0 column mean is +0.0, n={n}")


def test_literal_and_sliced_reference_agree():
    rng = np.random.default_rng(2)
    for d, sizes in ((1, cycle(BASE_SIZES + D1_SIZES, 40)), (3, cycle(BASE_SIZES, 20)), (59, cycle(SMALL_SIZES, 30))):
        lab = make_labels(sizes, rng, n_bad=50)
        x = normal_data(rng, len(lab), d)
        old = normal_data(rng, len(sizes), d)
        assert_bits_equal(ref_update_sorted(x, lab, old), ref_update(x, lab, old), f"d={d}")


@pytest.mark.parametrize("name", [c[0] for c in value_cases()])
def test_oracle_update_equals_numpy_on_special_values(oracle, name):
    _, x, lab, old = next(c for c in value_cases() if c[0] == name)
    with np.errstate(all="ignore"):
        want = ref_update(x, lab, old)
    assert_bits_equal(oracle.kmeans_update(x, lab, old)[0], want, name)


def test_oracle_update_equals_numpy_for_one_feature(oracle):
    rng = np.random.default_rng(3)
    sizes = BASE_SIZES + D1_SIZES + [100_003]
    lab = make_labels(sizes, rng)
    x = normal_data(rng, len(lab), 1)
    old = normal_data(rng, len(sizes), 1)
    assert_bits_equal(oracle.kmeans_update(x, lab, old)[0], ref_update_sorted(x, lab, old), "D = 1")


# ---- GPU ---------------------------------------------------------------------------------------------------
def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def check_shift(shift, want_new, old, what):
    """|shift - ||ref - old||| <= 2e-6 max(1, ||ref - old||): float64 accumulation against NumPy's float32 norm.
    Where NumPy's float32 sum of squares overflows and the float64 one does not, against the float64 norm."""
    got = float(shift.item()) if torch.is_tensor(shift) else float(shift)
    with np.errstate(all="ignore"):
        diff = want_new - old
        want = float(np.linalg.norm(diff))
        if np.isinf(want) and np.isfinite(diff).all():
            want = float(np.sqrt(np.sum(np.square(diff.astype(np.float64)))))
    if not np.isfinite(want):
        assert got == want or (np.isnan(got) and np.isnan(want)), (what, got, want)
    else:
        assert abs(got - want) <= 2e-6 * max(1.0, want), (what, got, want)


def helper_stream_clusters():
    """Second word of the ordered update's workspace header: the clusters its last call counted as big
    (>= 1/16 of the valid members), which run on the helper stream when N >= 2^18."""
    buf = pkg("ops")._ws.get(torch.device(DEV, torch.cuda.current_device()), 0)
    off = (-buf.data_ptr()) % 256
    return int(buf[off:off + 8].view(torch.int32)[1].item())


def run_update(x, lab, old, **kw):
    ops = pkg("ops")
    new, shift = ops.kmeans_update_ordered(dev(x), dev(lab), dev(old), **kw)
    return new.cpu().numpy(), shift


SHAPES = [  # (D, K, cluster sizes)
    (1, 64, cycle(BASE_SIZES + D1_SIZES, 64, big=100_003)),
    (1, 1024, cycle(SMALL_SIZES + D1_SIZES[:8], 1024)),
    (1, 5, [0, 8, 257, 100_003, 1]),
    (2, 65, cycle(BASE_SIZES, 65)),
    (3, 5, [0, 3077, 1, 513, 100_003]),
    (31, 1024, cycle(SMALL_SIZES, 1024)),
    (32, 64, cycle(BASE_SIZES, 64)),
    (33, 65, cycle(BASE_SIZES, 65)),
    (59, 64, cycle(BASE_SIZES, 64, big=100_003)),
    (64, 5, [1537, 0, 63, 4, 512]),
    (65, 1, [100_003]),
    (100, 65, cycle(BASE_SIZES, 65)),
    (256, 64, cycle(BASE_SIZES, 64)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("d,k,sizes", SHAPES, ids=[f"d{d}-k{k}-n{sum(s)}" for d, k, s in SHAPES])
def test_shapes_single_stream(d, k, sizes):
    assert len(sizes) == k and sum(sizes) < HELPER_MIN_N
    rng = np.random.default_rng(d * 10_000 + k)
    lab = make_labels(sizes, rng)
    x = normal_data(rng, len(lab), d)
    old = normal_data(rng, k, d)
    want = ref_update_sorted(x, lab, old)
    got, shift = run_update(x, lab, old)
    assert_bits_equal(got, want, f"D={d} K={k}")
    check_shift(shift, want, old, f"D={d} K={k}")


def helper_cases():
    n = 1 << 20
    third = [1 << 16, (1 << 16) - 1]
    rest = n - sum(third)
    return [  # (name, sizes, out-of-range labels, clusters that must count as big)
        ("k16-all-exactly-1/16", [n // 16] * 16, 0, 16),
        ("k40-one-at-1/16-one-below", third + [rest // 38 + (i < rest % 38) for i in range(38)], 0, 1),
        ("k1024-uniform", [n // 1024] * 1024, 0, 0),
        ("k1", [HELPER_MIN_N], 0, 1),
        ("k40-with-bad-labels", third + [rest // 38 + (i < rest % 38) for i in range(38)], 40_000, 1),
    ]


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 59, 65])
@pytest.mark.parametrize("name", [c[0] for c in helper_cases()])
def test_helper_stream_split(d, name):
    """N >= 2^18: big clusters (16 n >= valid members) are chained on the helper stream, the rest on the
    caller's.  The big count is over VALID members: out-of-range labels must not move the threshold."""
    _, sizes, n_bad, n_big = next(c for c in helper_cases() if c[0] == name)
    assert sum(sizes) + n_bad >= HELPER_MIN_N
    assert sum(16 * s >= sum(sizes) and s > 0 for s in sizes) == n_big
    rng = np.random.default_rng(len(sizes) + d)
    lab = make_labels(sizes, rng, n_bad)
    x = normal_data(rng, len(lab), d)
    old = normal_data(rng, len(sizes), d)
    want = ref_update_sorted(x, lab, old)
    got, shift = run_update(x, lab, old)
    assert helper_stream_clusters() == n_big
    assert_bits_equal(got, want, name)
    if n_bad:
        assert np.isnan(float(shift.item()))
    else:
        check_shift(shift, want, old, name)


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 59])
def test_busy_caller_stream_back_to_back(d):
    """On a non-default stream that is still busy: inputs produced on it just before the call, results cloned
    on it just after, two calls without a synchronisation in between (fork, join, shared workspace)."""
    ops = pkg("ops")
    rng = np.random.default_rng(40 + d)
    n = 1 << 19
    inputs = []
    for sizes in ([n // 4, n // 4, n // 8, n // 8] + [n // 32] * 8, [n // 2] + [n // 64] * 32):
        lab = make_labels(sizes, rng)
        x = normal_data(rng, n, d)
        old = normal_data(rng, len(sizes), d)
        inputs.append((x, lab, old, ref_update_sorted(x, lab, old)))
    base = [(dev(x), dev(lab), dev(old)) for x, lab, old, _ in inputs]
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    outs = []
    with torch.cuda.stream(s):
        junk = torch.ones(1 << 26, device=DEV)
        for _ in range(30):
            junk.mul_(1.0001)                             # keeps s busy while the host enqueues the rest
        for bx, bl, bo in base:
            x, lab, old = bx * 1.0, bl.clone(), bo.clone()          # written on s right before the call
            new, shift = ops.kmeans_update_ordered(x, lab, old)
            outs.append((new.clone(), shift.clone()))
    s.synchronize()
    for (got, shift), (_, _, old, want) in zip(outs, inputs):
        assert_bits_equal(got.cpu().numpy(), want, f"D={d}")
        check_shift(shift, want, old, f"D={d}")


@pytest.mark.gpu
def test_out_of_range_labels():
    ops, native = pkg("ops"), pkg("_native")
    rng = np.random.default_rng(9)
    for d in (1, 5):
        sizes = [40, 0, 513, 3, 1537, 64, 0]
        lab = make_labels(sizes, rng, n_bad=300)
        assert {-1, 7, 2**31 - 1, -2**31} <= set(lab.tolist())
        x = normal_data(rng, len(lab), d)
        old = normal_data(rng, len(sizes), d)
        want = ref_update(x, lab, old)                    # over the valid rows; clusters 1 and 6 keep old
        assert_bits_equal(want[[1, 6]], old[[1, 6]], "reference keeps empty clusters")
        got, shift = run_update(x, lab, old)
        assert_bits_equal(got, want, f"D={d} with out-of-range labels")
        assert np.isnan(float(shift.item()))
        with pytest.raises(native.GslError):
            ops.kmeans_update_ordered(dev(x), dev(lab), dev(old), validate=True)
        ok = np.where((lab >= 0) & (lab < len(sizes)), lab, 0).astype(np.int32)
        got, shift = run_update(x, ok, old)               # the flag is per call, on the same workspace
        assert np.isfinite(float(shift.item()))
        assert_bits_equal(got, ref_update(x, ok, old), f"D={d} after a call with bad labels")


@pytest.mark.gpu
@pytest.mark.parametrize("name", [c[0] for c in value_cases()])
def test_special_values(name):
    _, x, lab, old = next(c for c in value_cases() if c[0] == name)
    with np.errstate(all="ignore"):
        want = ref_update(x, lab, old)
    got, shift = run_update(x, lab, old)
    assert_bits_equal(got, want, name)
    check_shift(shift, want, old, name)


@pytest.mark.gpu
@pytest.mark.parametrize("d,want", [(2, 0.8388608), (1, 1.0)])
def test_float32_stagnation_of_the_reference(d, want):
    """20 M rows of 1.0 in one cluster: NumPy's sequential float32 sum stalls at 2^24 for D >= 2 (the mean
    comes out 2^24 / 2e7 = 0.8388608 and must be reproduced, not improved); its pairwise sum for D = 1 is exact."""
    n = 20_000_000
    x = np.ones((n, d), F32)
    lab = np.zeros(n, np.int32)
    old = np.zeros((2, d), F32)
    ref = np.stack([x.mean(axis=0), old[1]])
    assert_bits_equal(ref[0], np.full(d, want, F32), "NumPy itself")
    got, shift = run_update(x, lab, old)
    assert_bits_equal(got, ref, f"D={d}")
    check_shift(shift, ref, old, f"D={d}")


@pytest.mark.gpu
def test_no_rows_and_empty_clusters_copy_old_bits():
    ops = pkg("ops")
    for d in (1, 3, 40):
        old = normal_data(np.random.default_rng(d), 6, d)
        old[0] = -0.0
        old[3, 0] = np.float32(np.nan)
        old[4, -1] = -0.0
        clean = old.copy()
        clean[3, 0] = 1.0
        for o in (clean, old):
            new, shift = ops.kmeans_update_ordered(torch.empty((0, d), device=DEV), torch.empty(0, dtype=torch.int32, device=DEV), dev(o))
            assert np.array_equal(new.cpu().numpy().view(np.uint32), o.view(np.uint32)), f"N=0 D={d}: old copied bit for bit"
            check_shift(shift, o, o, f"N=0 D={d}")       # 0, or NaN when old holds a NaN, as in NumPy
        assert float(shift.item()) != float(shift.item())
        rng = np.random.default_rng(100 + d)
        lab = make_labels([5, 0, 130, 0, 0, 9], rng)
        x = normal_data(rng, len(lab), d)
        got, shift = run_update(x, lab, old)
        want = ref_update(x, lab, old)
        assert_bits_equal(got, want, f"empty clusters D={d}")
        assert np.array_equal(got[[1, 3, 4]].view(np.uint32), old[[1, 3, 4]].view(np.uint32))
        check_shift(shift, want, old, f"empty clusters D={d}")


# ---- whole trajectories: the drop-in against the reference loop --------------------------------------------
COLORS = [[252, 199, 55], [242, 107, 15], [231, 56, 121], [126, 24, 145],
          [247, 44, 91], [255, 116, 139], [167, 212, 119], [228, 241, 172]]


def reference_k_means(data, k, colors, max_iter=100, tol=1e-4, given=None):
    """The reference's K-means loop (km:107-151) on a feature block.  `given` collects the centroids of every
    assignment, for the tie check (not part of the reference)."""
    from scipy.spatial import KDTree
    centroids = data[np.random.choice(data.shape[0], k, replace=False)]
    for i in range(max_iter):
        print(i)
        tree = KDTree(centroids)
        _, labels = tree.query(data)
        given.append(centroids)
        new_centroids = np.array([data[labels == c].mean(axis=0) if np.sum(labels == c) > 0 else centroids[c]
                                  for c in range(k)])
        shift = np.linalg.norm(new_centroids - centroids)
        print(shift)
        if shift < tol:
            print(f"Converged after {i + 1} iterations.")
            break
        centroids = new_centroids
    tree = KDTree(centroids)
    _, labels = tree.query(data)
    given.append(centroids)
    for i in range(len(labels)):
        colors[i] = COLORS[labels[i] % len(COLORS)]
    return centroids, labels, colors


TRAJECTORIES = [(1, 3, 20_000, 11), (1, 10, 50_000, 12), (2, 3, 30_000, 13), (2, 10, 40_000, 14),
                (3, 3, 25_000, 15), (3, 10, 50_000, 16), (6, 10, 30_000, 17)]


def trajectory_data(d, n, seed):
    rng = np.random.default_rng(seed)
    centres = rng.uniform(-4, 4, (6, d))
    x = (centres[rng.integers(0, 6, n)] + rng.normal(0, 0.8, (n, d))).astype(F32)
    if d == 6:
        x[:, 4] = -0.0                                    # one feature that is -0.0 everywhere
    return x


@pytest.mark.gpu
@pytest.mark.parametrize("d,k,n,seed", TRAJECTORIES, ids=[f"d{d}-k{k}-n{n}" for d, k, n, _ in TRAJECTORIES])
def test_dropin_trajectory_equals_reference_loop(oracle, d, k, n, seed):
    km = pkg("k_means")
    x = trajectory_data(d, n, seed)
    given, out_ref, out_gpu = [], io.StringIO(), io.StringIO()
    np.random.seed(seed)
    with contextlib.redirect_stdout(out_ref):
        cen_r, lab_r, col_r = reference_k_means(x, k, np.zeros((n, 3), F32), max_iter=10, given=given)
    for c in given:                                       # exact ties are the documented tree-layout exemption
        want, gap = oracle.kmeans_assign(x, c, want_gap=True)
        assert (gap > 0).all(), f"seed {seed} has exact distance ties"
    assert np.array_equal(want, lab_r)
    np.random.seed(seed)
    with contextlib.redirect_stdout(out_gpu):
        cen, lab, col = km.k_means_kd_tree(x, k, np.zeros((n, 3), F32), max_iter=10)
    assert np.array_equal(lab, lab_r)
    assert_bits_equal(cen, cen_r, f"final centroids D={d} K={k}")
    assert np.array_equal(col, col_r)
    mine, ref = out_gpu.getvalue().splitlines(), out_ref.getvalue().splitlines()
    assert len(mine) == len(ref), (mine, ref)
    for a, b in zip(mine, ref):                           # indices and "Converged" verbatim, shifts to 2e-6
        if a != b:
            assert abs(float(a) - float(b)) <= 2e-6 * max(1.0, abs(float(b))), (a, b)
