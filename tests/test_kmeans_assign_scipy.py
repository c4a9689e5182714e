"""The K-means assignment against scipy's own KDTree, at the shape and range edges of its screening.

The reference labels every row with `KDTree(centroids).query(row)` (km:116-122): the float64
nearest centroid, and on an exact tie whichever one the tree reaches first.  The kernels screen
with float32 or TF32 estimates and an error bound, and recompute only near ties in float64; they
promise the float64 scan's labels with exact ties going to the lowest index (DESIGN §2).

References (CPU):
  scan64   NumPy float64 distances in scipy's summation order (four running lanes over blocks of
           four dimensions, added ((a0 + a1) + a2) + a3, then a sequential tail; ckdtree's
           sqeuclidean_distance_double), first minimum, and the gap to the second smallest.
  KDTree   scipy's own query.  It must agree with scan64 on every finite row with gap > 0; exact
           ties and non-finite rows are compared with scan64 only.

Input sets: a shape grid around the tensor-core kernel's limits (8 <= D <= 64, 16 <= K <= 64),
ragged and multi-tile row counts, an unaligned row slice; values whose float32 ranking or distance
overflows, tiny values, mixed scales and offsets, NaN/Inf centroids; and data that drives every
refinement branch (pooled pairs, the refine_row fallback, s1 = 0).  The CPU tests check that the
references agree and that every adversarial set reaches the branch it targets (by emulating the
kernel's float32 arithmetic); the GPU tests check both kernels under every dispatch setting.
"""
import functools
from fractions import Fraction

import numpy as np
import pytest
import torch
from scipy.spatial import KDTree

from util import pkg

F32, F64 = np.float32, np.float64
DEV = "cuda"
FLT_MAX = float(np.finfo(F32).max)
TILE = 256                                   # rows per tile of both step kernels


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count if torch.cuda.is_available() else 148


# ---- references ------------------------------------------------------------------------------------------
def sqdist64(data, cen):
    """float64 [n, K] squared distances in scipy's order: (double)c - (double)x, four lanes, tail."""
    diff = cen.astype(F64)[None, :, :] - data.astype(F64)[:, None, :]
    sq = diff * diff
    D = data.shape[1]
    lanes = [np.zeros(sq.shape[:2]) for _ in range(4)]
    for i in range(0, D - D % 4, 4):
        for j in range(4):
            lanes[j] = lanes[j] + sq[:, :, i + j]
    s = ((lanes[0] + lanes[1]) + lanes[2]) + lanes[3]
    for i in range(D - D % 4, D):
        s = s + sq[:, :, i]
    return s


def scan64(data, cen, chunk=2048):
    """(labels int64, gap float64): the float64 scan from (inf, 0) with `d < best`, as the oracle."""
    labels = np.empty(len(data), np.int64)
    gap = np.empty(len(data), F64)
    with np.errstate(all="ignore"):
        for r0 in range(0, len(data), chunk):
            d = sqdist64(data[r0:r0 + chunk], cen)
            best = np.full(len(d), np.inf)
            second = np.full(len(d), np.inf)
            lab = np.zeros(len(d), np.int64)
            for k in range(d.shape[1]):
                dk = d[:, k]
                lt = dk < best
                second = np.where(lt, best, np.where(dk < second, dk, second))
                best = np.where(lt, dk, best)
                lab = np.where(lt, k, lab)
            labels[r0:r0 + chunk] = lab
            gap[r0:r0 + chunk] = second - best
    return labels, gap


# ---- float32 emulation of the kernels' screening arithmetic (to show each set reaches its branch) --------
def tf32(a):
    b = np.asarray(a, F32).view(np.uint32).astype(np.uint64)
    return ((b + 0x1000) & 0xFFFFE000).astype(np.uint32).view(F32)      # cvt.rna: nearest, ties away


def stage_a(data, cen, factor=2.0):
    """Stage A of kmeans_step_tc_kernel as it stood before its range guard: (g [n, K], candidate mask [n, K]),
    candidates within `factor` row bounds of the smallest g.  The dot products are summed in NumPy's order,
    not the MMA's; the sets below do not depend on it."""
    K = len(cen)
    with np.errstate(all="ignore"):
        mean = (cen.sum(0, dtype=F32) / F32(K)).astype(F32)
        cp = (cen - mean).astype(F32)
        cn2 = (cp * cp).sum(1, dtype=F32)
        ncu = np.sqrt(cn2) * F32(1.0001)
        ea, eb = F32(2.9296875e-3) * ncu, F32(4.76837158203125e-7) * ncu * ncu * F32(1.0001)
        xp = (data - mean).astype(F32)
        nx = np.sqrt((xp * xp).sum(1, dtype=F32)) * F32(1.0001)
        dot = (tf32(xp)[:, None, :] * tf32(cp)[None, :, :]).sum(2, dtype=F32)
        g = (cn2[None, :] - F32(2) * dot).astype(F32)
        gmin = np.fmin.reduce(g, axis=1)
        bound = nx * ea.max() + eb.max() + F32(4.76837158203125e-7) * nx * nx * F32(1.0001)
        thr = gmin + F32(factor) * bound * F32(1.000001)
        mask = g <= thr[:, None]
        mask[~mask.any(1) | ~(nx < np.inf)] = True
    return g, mask


_OVF = Fraction(2**128) - Fraction(2**103)       # exact values from here up round to +inf (ties to even)


def round_f32(v):
    """One correct rounding of an exact rational to float32 (nearest, ties to even, overflow to inf)."""
    if v == 0:
        return F32(0.0)
    sign, a = (-1 if v < 0 else 1), abs(v)
    if a >= _OVF:
        return F32(sign * np.inf)
    e = a.numerator.bit_length() - a.denominator.bit_length()
    while a >= Fraction(2) ** (e + 1):
        e += 1
    while a < Fraction(2) ** e:
        e -= 1
    q = Fraction(2) ** (max(e, -126) - 23)
    return F32(sign * float(round(a / q) * q))       # Fraction.__round__ is half-to-even; the product is exact in float64


def fma32(a, b, c):
    if not np.isfinite(c):
        return F32(c)
    return round_f32(Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c)))


def add32(a, b):
    if not (np.isfinite(a) and np.isfinite(b)):
        return F32(F32(a) + F32(b))
    return round_f32(Fraction(float(a)) + Fraction(float(b)))


def chain_one(x, c):
    """sqdist_f32 / refine_row: s = fmaf(d, d, s) over d = 0 .. D-1."""
    s = F32(0.0)
    for xi, ci in zip(x, c):
        df = F32(F32(xi) - F32(ci))
        s = fma32(df, df, s)
    return s


def chain_two(x, c):
    """sqdist_screen (CUDA-core kernel, D a multiple of 4): dims 0, 2 of every block of four into s0,
    dims 1, 3 into s1, then s0 + s1."""
    d = [F32(F32(xi) - F32(ci)) for xi, ci in zip(x, c)]
    s0 = s1 = F32(0.0)
    for i in range(0, len(d), 4):
        s0 = fma32(d[i], d[i], s0); s1 = fma32(d[i + 1], d[i + 1], s1)
        s0 = fma32(d[i + 2], d[i + 2], s0); s1 = fma32(d[i + 3], d[i + 3], s1)
    return add32(s0, s1)


@functools.lru_cache(None)
def flt_max_pair(chain):
    """(a, b), D = 8, for the row x = 0: b = (2^64, 0, ...) is nearer in float64 (d_b = 2^128), but the
    float32 chain rounds |a|^2 to FLT_MAX and overflows |b|^2.  Searched from a fixed seed near
    a_i = sqrt(FLT_MAX / 8)."""
    fn = {"one": chain_one, "two": chain_two}[chain]
    zero = np.zeros(8, F32)
    b = zero.copy()
    b[0] = F32(2.0**64)
    base = F32(np.sqrt(FLT_MAX / 8))
    rng = np.random.default_rng(1)
    for _ in range(20000):
        a = (base * (1 + rng.integers(-40, 40, 8) * 2.0**-24)).astype(F32)
        if sqdist64(zero[None], a[None])[0, 0] > sqdist64(zero[None], b[None])[0, 0] and np.isfinite(fn(zero, a)):
            return a, b
    raise AssertionError(f"no FLT_MAX pair found for the {chain}-chain sum")


# ---- input sets ------------------------------------------------------------------------------------------
SHAPE_D = [8, 9, 15, 16, 17, 31, 32, 33, 57, 63, 64]
SHAPE_K = [16, 17, 31, 32, 33, 63, 64]
SHAPE_N = [1, 31, 255, 256, 257, 4097]
GRID = [(d, SHAPE_K[i % 7], SHAPE_N[i % 6]) for i, d in enumerate(SHAPE_D)] + \
       [(d, SHAPE_K[(i + 3) % 7], SHAPE_N[(i + 3) % 6]) for i, d in enumerate(SHAPE_D)]


def near_ties(rng, n, cen, scale=1.0):
    """n rows: a quarter on bisecting planes of centroid pairs, an eighth next to them, an eighth equal
    to a centroid (s1 = 0, as in a first iteration), the rest N(0, scale)."""
    K, D = cen.shape
    pts = (rng.standard_normal((n, D)) * scale).astype(F32)
    n_mid, n_wob, n_eq = n // 4, n // 8, max(n // 8, 1)
    rows = rng.permutation(n)
    i, j = rng.integers(0, K, n_mid + n_wob), rng.integers(0, K, n_mid + n_wob)
    mid = ((cen[i].astype(F64) + cen[j]) / 2)
    mid[n_mid:] += rng.standard_normal((n_wob, D)) * scale * 1e-6
    pts[rows[:n_mid + n_wob]] = mid.astype(F32)
    pts[rows[n_mid + n_wob:n_mid + n_wob + n_eq]] = cen[rng.integers(0, K, len(rows[n_mid + n_wob:n_mid + n_wob + n_eq]))]
    return pts


def random_directions(rng, n, d, lo, hi):
    v = rng.standard_normal((n, d))
    return (v / np.linalg.norm(v, axis=1, keepdims=True) * rng.uniform(lo, hi, (n, 1))).astype(F32)


def pool_case(rng, tie_rows):
    """K = 16 at twelve positions 100 apart, the first four duplicated (k and k + 12).  Every warp's 32
    rows hold `tie_rows` rows next to a duplicated position (two exact-tie candidates each) and the
    rest next to a single one (one candidate): 2 * tie_rows pairs per warp."""
    D = 16
    pos = (rng.standard_normal((12, D)) * 100).astype(F32)
    cen = np.concatenate([pos, pos[:4]])
    rows = []
    for _ in range(8 * 8):                                   # 8 tiles of 8 warps
        which = np.concatenate([rng.integers(0, 4, tie_rows), rng.integers(4, 12, 32 - tie_rows)])
        rows.append(pos[rng.permutation(which)] + rng.standard_normal((32, D)).astype(F32) * F32(0.01))
    return np.concatenate(rows).astype(F32), cen


# name -> (group, builder(rng) -> (data, cen)); group picks the claim checked on the CPU
CASES = {}


def case(name, group):
    def reg(fn):
        CASES[name] = (group, fn)
        return fn
    return reg


for _d, _k, _n in GRID:
    def _grid(rng, d=_d, k=_k, n=_n):
        cen = rng.standard_normal((k, d)).astype(F32)
        return near_ties(rng, n, cen), cen
    case(f"grid_d{_d}_k{_k}_n{_n}", "grid")(_grid)


@case("multi_tile_ragged", "grid")
def _multi_tile(rng):
    # every CTA of the 2 * SMs grid walks three bulk-copied tiles; the last tile holds 5 rows
    cen = rng.standard_normal((33, 33)).astype(F32)
    return near_ties(rng, 2 * sm_count() * TILE * 3 + 5, cen), cen


@case("unaligned_slice", "unaligned")
def _unaligned(rng):
    # the GPU sees rows [1:] of this array: odd D, so the data pointer is 4 mod 16 and no tile is a TMA copy
    cen = rng.standard_normal((31, 17)).astype(F32)
    return near_ties(rng, 4098, cen), cen


@case("a_stage_a_overflow_issue", "a")
def _a_issue(rng):
    cen = np.zeros((16, 8), F32)
    cen[:8, 0], cen[8:, 0] = 2e19, -2e19
    cen[:, 1] = np.arange(16) * 1e17                          # distinct float64 distances from row 0 = (1e19, 0, ...)
    data = np.zeros((300, 8), F32)
    data[:, 0] = 1e19
    data[1:, 0] = rng.uniform(-1.5e19, 1.5e19, 299)
    data[1:, 1:] = rng.uniform(-3e18, 3e18, (299, 7))
    return data, cen


@case("a_stage_a_overflow_random", "a")
def _a_random(rng):
    half = random_directions(rng, 16, 16, 2e19, 1e20)
    cen = np.concatenate([half, -half[rng.permutation(16)]])  # mean ~ 0, so |x'| ~ |x|
    data = random_directions(rng, 2000, 16, 1e18, 1.7e19)
    data[:500] = (cen[rng.integers(0, 32, 500)] * rng.uniform(0.05, 0.17, (500, 1))).astype(F32)
    return data, cen


@case("b_dot_overflow", "b")
def _b(rng):
    cen = random_directions(rng, 32, 16, 1.3e19, 1.8e19)
    cen -= cen.mean(0)                                        # centred: |c'| = |c| up to rounding
    data = random_directions(rng, 2000, 16, 1.3e19, 1.8e19)
    near = cen[rng.integers(0, 32, 1000)].astype(F64)
    near += rng.standard_normal(near.shape) * 1e18
    near *= (rng.uniform(1.3e19, 1.8e19, (1000, 1)) / np.linalg.norm(near, axis=1, keepdims=True))
    data[:1000] = near.astype(F32)
    return data, cen


def _flt_max_set(chain, k, n):
    a, b = flt_max_pair(chain)
    pads = np.zeros((max(k - 2, 0), 8), F32)
    pads[:, 1] = (2.0**64 * (1 + np.arange(1, k - 1) / 8)).astype(F32)     # farther still, in both precisions
    return np.zeros((n, 8), F32), np.concatenate([a[None], b[None], pads])


for _chain in ("one", "two"):
    for _k, _n in ((16, 1), (16, 300), (2, 300)):
        case(f"c_flt_max_{_chain}_chain_k{_k}_n{_n}", "c")(lambda rng, c=_chain, k=_k, n=_n: _flt_max_set(c, k, n))


for _scale, (_d, _k) in zip((1e-17, 1e-19, 1e-20, 1e-22), ((16, 32), (33, 17), (8, 64), (64, 16))):
    def _tiny(rng, s=_scale, d=_d, k=_k):
        cen = (rng.standard_normal((k, d)) * s).astype(F32)
        return near_ties(rng, 3000, cen, scale=s), cen
    case(f"d_tiny_{_scale:g}", "d")(_tiny)


@case("e_mixed_scales", "e")
def _e_mixed(rng):
    scales = np.logspace(-3, 3, 24)
    cen = (rng.standard_normal((40, 24)) * scales).astype(F32)
    data = near_ties(rng, 5000, cen)
    data = (data * np.where(np.arange(5000)[:, None] % 2 == 0, scales, 1.0)).astype(F32)
    return data, cen


for _off, (_d, _k) in ((1e4, (32, 48)), (1e6, (57, 20))):
    def _offset(rng, off=_off, d=_d, k=_k):
        cen = (rng.standard_normal((k, d)) * 1e-2 + off).astype(F32)
        pts = (rng.standard_normal((5000, d)) * 1e-2 + off).astype(F32)
        pts[:1500] = near_ties(rng, 1500, cen.astype(F64) - off, scale=1e-2) + off
        return pts.astype(F32), cen
    case(f"e_offset_{_off:g}", "e")(_offset)


@case("f_nan_inf_centroids", "f")
def _f(rng):
    cen = rng.standard_normal((24, 16)).astype(F32)
    cen[5, 3] = np.nan
    cen[9, 0] = np.inf
    data = near_ties(rng, 2000, cen[[k for k in range(24) if k not in (5, 9)]])
    data[::50] = np.nan
    data[7::50, 2] = -np.inf
    return data, cen


@case("a_tf32_rounding_near_tie", "tf32")
def _tf32(rng):
    # Every value is exact, and the centroids sum to zero exactly, so x' = x and c' = c.  x_i = 1 + 2^-11 and
    # B_i = 4 + 2^-9 are TF32 ties and round up (cvt.rna), so g_B comes out 2^-4 low; A (x.A = 0, TF32-exact)
    # is nearer by 0.0099.  A's ranking value lands above g_B by more than half the row bound: the
    # factor 2 of the candidate threshold is what keeps A (and its tie -A) in the set.
    D = 8
    x = np.full(D, 1 + 2.0**-11, F32)
    a = np.array([2.828125, -2.828125] + [2.830078125, -2.830078125] * 3, F32)
    b = np.full(D, 4 + 2.0**-9, F32)
    h = np.array([[1 if bin(i & j).count("1") % 2 == 0 else -1 for j in range(D)] for i in range(D)], F32)
    pads = [v for i in range(2, 8) for v in (3 * h[i], -3 * h[i])]        # Hadamard rows: x.h = 0, g = 72
    return np.tile(x, (300, 1)), np.stack([a, -a, b, -b] + pads).astype(F32)


def _subnormal_set(n):
    # x = 0.  a = (t, ..., t), t^2 = 0.6 * 2^-149: the float32 sum rounds every partial sum up to the next
    # subnormal, to 16 * 2^-149, while b's single term is exactly 12 * 2^-149.  Float32 ranks b first by a
    # margin far beyond eps; float64 ranks a first (9.6 < 12).  Rows with s1 <= 1e-30 must go to float64.
    D = 16
    a = np.full(D, np.sqrt(0.6) * 2.0**-74.5, F32)
    b = np.zeros(D, F32)
    b[0] = np.sqrt(12.0) * 2.0**-74.5
    pads = np.zeros((14, D), F32)
    pads[:, 1] = 2.0**-70 * np.arange(1, 15)
    return np.zeros((n, D), F32), np.concatenate([a[None], b[None], pads]).astype(F32)


for _n in (1, 2, 300):
    case(f"d_subnormal_sums_n{_n}", "sub")(lambda rng, n=_n: _subnormal_set(n))


@case("refine_dup32_k64", "dup")
def _dup(rng):
    base = rng.standard_normal((32, 32)).astype(F32)
    return (rng.standard_normal((4097, 32)) * 0.5).astype(F32), np.concatenate([base, base])


@case("refine_pool_32_pairs", "pool32")
def _pool32(rng):
    return pool_case(rng, 16)


@case("refine_pool_34_pairs", "pool34")
def _pool34(rng):
    return pool_case(rng, 17)


@case("refine_rows_equal_centroids", "eq")
def _eq(rng):
    data = rng.standard_normal((3000, 20)).astype(F32)
    return data, data[rng.choice(3000, 40, replace=False)].copy()


@functools.lru_cache(None)
def get(name):
    """dict(data = rows the kernel sees, full = the array allocated (unaligned set: one more row), cen,
    labels, gap) -- deterministic per name."""
    group, build = CASES[name]
    rng = np.random.default_rng(sum(map(ord, name)) * 7919)
    full, cen = build(rng)
    full, cen = np.ascontiguousarray(full, F32), np.ascontiguousarray(cen, F32)
    data = full[1:] if group == "unaligned" else full
    labels, gap = scan64(data, cen)
    return dict(group=group, full=full, data=data, cen=cen, labels=labels, gap=gap)


NAMES = list(CASES)
SUM_SETS = [n for n in NAMES if CASES[n][0] in ("grid", "unaligned", "e")]


# ---- CPU: the references agree, and every set reaches its branch -----------------------------------------
@pytest.mark.parametrize("name", NAMES)
def test_scan64_equals_the_c_oracle(oracle, name):
    c = get(name)
    with np.errstate(all="ignore"):
        want, gap = oracle.kmeans_assign(c["data"], c["cen"], want_gap=True)
    assert np.array_equal(c["labels"], want)
    assert np.array_equal(c["gap"].view(np.uint64), gap.view(np.uint64)) or \
        np.array_equal(c["gap"], gap, equal_nan=True)


@pytest.mark.parametrize("name", [n for n in NAMES if CASES[n][0] != "f"])
def test_scan64_equals_scipy_kdtree(name):
    c = get(name)
    data, cen = c["data"].astype(F64), c["cen"].astype(F64)
    ok = np.isfinite(data).all(1) & (c["gap"] > 0)
    _, idx = KDTree(cen).query(data[ok], workers=-1)
    bad = np.flatnonzero(idx != c["labels"][ok])
    assert len(bad) == 0, f"{len(bad)} of {ok.sum()} rows: KDTree {idx[bad[:5]]} vs scan64 {c['labels'][ok][bad[:5]]}"
    assert ok.sum() > 0 or c["group"] in ("dup", "pool32", "pool34", "c", "tf32")


def test_sets_reach_their_branches():
    by = {}
    for n in NAMES:
        by.setdefault(CASES[n][0], []).append(n)
    # shape grid: every D and every K at least twice, every N, the multi-tile and unaligned edges
    shapes = [get(n)["cen"].shape for n in by["grid"] + by["unaligned"]]
    for d in SHAPE_D:
        assert sum(s[1] == d for s in shapes) >= 2, d
    for k in SHAPE_K:
        assert sum(s[0] == k for s in shapes) >= 2, k
    assert {len(get(n)["data"]) for n in by["grid"]} >= set(SHAPE_N)
    big = get("multi_tile_ragged")["data"]
    tiles, grid = -(-len(big) // TILE), 2 * sm_count()
    assert tiles // grid >= 3 and len(big) % TILE != 0
    u = get("unaligned_slice")
    assert u["data"].shape[1] % 2 == 1 and u["data"].ctypes.data - u["full"].ctypes.data == 4 * u["data"].shape[1]

    # (a) the nearest centroid's float32 ranking value is NaN, so stage A dropped it
    for n in by["a"]:
        c = get(n)
        g, mask = stage_a(c["data"], c["cen"])
        lab = c["labels"]
        hit = np.isnan(g[np.arange(len(lab)), lab]) & ~mask[np.arange(len(lab)), lab]
        xp = c["data"] - c["cen"].mean(0)
        assert hit.any(), n
        assert (np.linalg.norm(xp.astype(F64), axis=1) < 1.8e19).all(), n
    # (b) 2 x'.c' overflows float32 while |x'|, |c'| stay below 1.8e19
    c = get("b_dot_overflow")
    g, _ = stage_a(c["data"], c["cen"])
    assert np.isinf(g).any(1).mean() > 0.3
    # (c) float32 orders a ahead of b, float64 (and scipy) the other way round
    for chain, fn in (("one", chain_one), ("two", chain_two)):
        a, b = flt_max_pair(chain)
        zero = np.zeros(8, F32)
        assert fn(zero, a) == F32(FLT_MAX) and np.isinf(fn(zero, b))
        for n in by["c"]:
            if f"_{chain}_" in n:
                assert (get(n)["labels"] == 1).all(), n
                assert (get(n)["gap"] > 0).all(), n
    # (d) every row's nearest distance is below the float32 gate (1e-30): float64 decides; the smaller
    # scales put the products of the dot below FLT_MIN
    for n in by["d"]:
        c = get(n)
        best = sqdist64(c["data"], c["cen"]).min(1)
        assert (best < 1e-30).all(), n
        assert ((c["gap"] > 0) & (c["gap"] < 1e-6 * best)).any(), f"{n}: no near ties"
    assert (np.abs(get("d_tiny_1e-22")["cen"]).max() ** 2) < np.finfo(F32).tiny
    # (e) near ties (on the offsets, whose rows are quantized to float32 ulps, within 1e-3 or exact); the
    # offsets are 1e6 and 1e8 times the spread, and the scales of the mixed set span 1e6
    for n in by["e"]:
        c = get(n)
        best = sqdist64(c["data"], c["cen"]).min(1)
        assert (c["gap"] < 1e-3 * best).sum() > 10, n
        if "offset" in n:
            assert np.abs(c["cen"]).min() / c["cen"].std(0).max() > 1e5, n
    col = np.abs(get("e_mixed_scales")["cen"]).max(0)
    assert col.max() / col.min() > 1e5
    # TF32 rounding: A (and its tie -A) stays a candidate with the threshold's factor 2 and would not with 1/2
    c = get("a_tf32_rounding_near_tie")
    assert (c["labels"] == 0).all() and (c["gap"] == 0).all()               # A and -A tie exactly; A has index 0
    assert (sqdist64(c["data"], c["cen"])[:, 2] - sqdist64(c["data"], c["cen"])[:, 0] > 0).all()
    assert stage_a(c["data"], c["cen"])[1][:, 0].all() and not stage_a(c["data"], c["cen"], 0.5)[1][:, 0].any()
    # subnormal sums: float32 (either chain shape) puts b far ahead of a, float64 picks a
    a, b = get("d_subnormal_sums_n1")["cen"][:2]
    zero = np.zeros(16, F32)
    for fn in (chain_one, chain_two):
        sa, sb = fn(zero, a), fn(zero, b)
        assert sa == F32(16 * 2.0**-149) and sb == F32(12 * 2.0**-149), (sa, sb)
    assert (get("d_subnormal_sums_n1")["labels"] == 0).all()
    # (f) the NaN and the Inf centroid never win a finite row; NaN/Inf rows go to label 0
    c = get("f_nan_inf_centroids")
    fin = np.isfinite(c["data"]).all(1)
    assert not np.isin(c["labels"][fin], [5, 9]).any() and (c["labels"][~fin] == 0).all() and (~fin).any()
    # refinement: every row ties exactly; the pooled pairs of each warp are exactly 32 / 34
    c = get("refine_dup32_k64")
    assert (c["gap"] == 0).all() and (c["labels"] < 32).all()
    for n, pairs in (("refine_pool_32_pairs", 32), ("refine_pool_34_pairs", 34)):
        c = get(n)
        _, mask = stage_a(c["data"], c["cen"])
        per_row = mask.sum(1)
        assert set(per_row.tolist()) == {1, 2}, n
        per_warp = np.where(per_row > 1, per_row, 0).reshape(-1, 32).sum(1)
        assert (per_warp == pairs).all(), (n, set(per_warp.tolist()))
        assert (c["labels"] < 12).all()
    c = get("refine_rows_equal_centroids")
    assert (sqdist64(c["data"], c["cen"]).min(1) == 0).sum() >= 40


def test_exact_rounding_helpers():
    # round_f32 rounds once: the midpoint between FLT_MAX and 2^128 overflows (ties to even), just below it does not
    m = Fraction(2**128) - Fraction(2**103)
    assert np.isinf(round_f32(m)) and round_f32(m - 1) == F32(FLT_MAX)
    assert round_f32(Fraction(1, 3)) == F32(1 / 3) and round_f32(Fraction(2**-149)) == F32(2.0**-149)
    assert round_f32(Fraction(3, 2**150)) == F32(2.0**-148)            # subnormal tie to even
    rng = np.random.default_rng(4)
    for a, b, c in rng.standard_normal((200, 3)).astype(F32):
        assert fma32(a, b, c) == F32(Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c)))


# ---- GPU -------------------------------------------------------------------------------------------------
DISPATCH = {"default": {}, "cuda_cores": {"GSLIFT_KMEANS_TC": "0"}, "exact": {"GSLIFT_KMEANS_EXACT": "1"}}


def dev_rows(c):
    full = torch.from_numpy(c["full"]).to(DEV)
    return full[1:] if c["group"] == "unaligned" else full


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_labels_equal_scan64_every_kernel_and_dispatch(monkeypatch, name):
    ops = pkg("ops")
    c = get(name)
    data, cen = dev_rows(c), torch.from_numpy(c["cen"]).to(DEV)
    want = c["labels"]
    for setting, env in DISPATCH.items():
        monkeypatch.delenv("GSLIFT_KMEANS_TC", raising=False)
        monkeypatch.delenv("GSLIFT_KMEANS_EXACT", raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        for entry in ("kmeans_assign", "kmeans_step"):
            out = getattr(ops, entry)(data, cen)
            got = (out[0] if entry == "kmeans_step" else out).cpu().numpy().astype(np.int64)
            bad = np.flatnonzero(got != want)
            assert len(bad) == 0, (f"{name}, {entry}, {setting}: {len(bad)} of {len(want)} labels differ, first rows "
                                   f"{bad[:5].tolist()}: got {got[bad[:5]].tolist()}, want {want[bad[:5]].tolist()}, "
                                   f"gap {c['gap'][bad[:5]].tolist()}")


@pytest.mark.gpu
@pytest.mark.parametrize("name", SUM_SETS)
def test_fused_sums_within_the_summation_bound(name):
    """kmeans_step's float64 sums, read directly: counts exact; each (cluster, dim) within the recursive
    summation bound m 2^-53 sum|x|, m = members + grid + 32 (tile walk, per-CTA partials, 32-warp reduce)."""
    ops = pkg("ops")
    c = get(name)
    data, lab = c["data"], c["labels"]
    K, D = c["cen"].shape
    got_lab, sums = ops.kmeans_step(dev_rows(c), torch.from_numpy(c["cen"]).to(DEV))
    s = sums.cpu().numpy()
    assert np.array_equal(got_lab.cpu().numpy(), lab)
    counts = np.bincount(lab, minlength=K)
    assert np.array_equal(s[:, D], counts.astype(F64))
    order = np.argsort(lab, kind="stable")
    rows = data[order].astype(np.longdouble)
    starts = np.searchsorted(lab[order], np.arange(K))
    nz = counts > 0
    exact = np.zeros((K, D), np.longdouble)
    mag = np.zeros((K, D), np.longdouble)
    exact[nz] = np.add.reduceat(rows, starts[nz], axis=0)
    mag[nz] = np.add.reduceat(np.abs(rows), starts[nz], axis=0)
    grid = min(-(-len(data) // TILE), 2 * sm_count())
    m = (counts + grid + 32)[:, None]
    err = np.abs(s[:, :D].astype(np.longdouble) - exact)
    tol = m * np.longdouble(2.0**-53) * mag
    bad = err > tol
    assert not bad.any(), f"{name}: {int(bad.sum())} sums outside the bound, worst err/tol {float((err / np.maximum(tol, 1e-300)).max()):.3g}"
    assert (s[~nz, :D] == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("name", [n for n in NAMES if CASES[n][0] in ("grid", "unaligned", "a", "b", "c", "d", "e", "tf32", "sub")])
def test_screening_bound_selftest(name):
    """gsl_kmeans_screen_selftest: stage A's bound against float64 on every (row, centroid) pair.  Rows
    outside the range where the bound is proven take every centroid and are only counted."""
    native = pkg("_native")
    c = get(name)
    K, D = c["cen"].shape
    if not (K >= 16 and 8 <= D <= 64):
        pytest.skip("not a tensor-core shape")
    data = dev_rows(c)
    out = torch.zeros(3, dtype=torch.int64, device=DEV)
    labels = torch.empty(len(c["data"]), dtype=torch.int32, device=DEV)
    cen = torch.from_numpy(c["cen"]).to(DEV)
    native.check(native.lib().gsl_kmeans_screen_selftest(data.data_ptr(), len(c["data"]), D, cen.data_ptr(), K,
                                                         labels.data_ptr(), out.data_ptr(), None))
    torch.cuda.synchronize()
    viol, cand, skip = (int(v) for v in out.tolist())
    print(f"[tc screen] {name}: violations {viol}, candidates per row {cand / len(c['data']):.3f}, rows outside the range {skip}")
    assert viol == 0
    assert np.array_equal(labels.cpu().numpy(), c["labels"])
    if c["group"] in ("grid", "unaligned", "e", "tf32"):
        assert skip == 0, "ordinary data must stay inside the range where the bound is proven"
    if c["group"] in ("a", "b", "c"):
        assert skip > 0
