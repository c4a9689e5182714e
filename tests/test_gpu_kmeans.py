"""Parity of the CUDA K-means path (through the C ABI) with the oracle and the reference's golden
vectors.  Bar: assignments bit-exact except exact distance ties; ordered centroids bit-exact;
fast (float64, shardable) centroids within 1e-5 relative of the reference's float32 mean."""
import contextlib
import io

import numpy as np
import pytest
import torch

from util import KMEANS_CASES, assert_bits_equal, load_kmeans_case, pkg

pytestmark = pytest.mark.gpu
DEV = "cuda"


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


@pytest.mark.parametrize("name", KMEANS_CASES)
def test_golden_vectors_through_the_dropin(name):
    km = pkg("k_means")
    c = load_kmeans_case(name)
    colors = c["colors"].copy()
    buf = io.StringIO()
    np.random.seed(c["seed"])
    with contextlib.redirect_stdout(buf):
        if "points" in c:
            cen, lab, col = km.k_means_with_color(c["points"], c["k"], colors, max_iter=c["max_iter"])
        else:
            cen, lab, col = km.k_means_kd_tree(c["data"], c["k"], colors, max_iter=c["max_iter"])
    assert lab.dtype == np.int64 and cen.dtype == np.float32
    assert np.array_equal(lab, c["labels"])
    assert np.array_equal(cen, c["centroids"]), "ordered update must reproduce NumPy's float32 mean"
    assert col is colors and np.array_equal(col, c["colors_out"])
    mine, ref = buf.getvalue().splitlines(), c["stdout"].splitlines()
    assert len(mine) == len(ref)
    for a, b in zip(mine, ref):                       # iteration indices / "Converged" verbatim,
        if a != b:                                    # shift norms to float32 rounding of the BLAS dot
            assert abs(float(a) - float(b)) <= 2e-6 * max(1.0, abs(float(b))), (a, b)


@pytest.mark.parametrize("name", ["kmeans_color_k10", "kmeans_kdtree_k64_d59"])
def test_golden_vectors_fast_update_within_tolerance(name):
    km = pkg("k_means")
    c = load_kmeans_case(name)
    np.random.seed(c["seed"])
    with contextlib.redirect_stdout(io.StringIO()):
        cen, lab, _ = km.k_means_kd_tree(c["data"], c["k"], c["colors"].copy(), max_iter=c["max_iter"], update="fast")
    rel = np.abs(cen - c["centroids"]).max(axis=1) / np.abs(c["centroids"]).max(axis=1)
    agree = (lab == c["labels"]).mean()
    print(f"[{name}] free-running fast update: centroid rel err max {rel.max():.2e}, label agreement {agree:.5f}")
    assert rel.max() < 1e-5
    assert agree > 0.999


@pytest.mark.parametrize("n,d,k", [(1, 3, 1), (255, 3, 2), (257, 6, 10), (5000, 7, 3), (4099, 8, 17), (20000, 59, 64),
                                   (3001, 61, 5), (9000, 64, 128), (1500, 100, 33)])
def test_step_locked_assignment_and_updates(oracle, n, d, k):
    ops = pkg("ops")
    rng = np.random.default_rng(n + d)
    data = rng.standard_normal((n, d)).astype(np.float32)
    k = min(k, n)
    cen = data[rng.choice(n, k, replace=False)].copy()
    if k > 2:
        cen[k - 1] = 1e6                               # an empty cluster keeps its old centroid
    want, gap = oracle.kmeans_assign(data, cen, want_gap=True)
    lab = ops.kmeans_assign(dev(data), dev(cen))
    lab2, sums = ops.kmeans_step(dev(data), dev(cen))
    torch.cuda.synchronize()
    got = lab.cpu().numpy().astype(np.int64)
    assert np.array_equal(lab2.cpu().numpy(), lab.cpu().numpy())
    bad = got != want
    assert not (bad & (gap > 0)).any(), f"{(bad & (gap > 0)).sum()} mismatches away from exact ties"
    assert not bad.any()                               # ties resolve to the lowest index on both sides
    # counts + float64 sums
    s = sums.cpu().numpy()
    assert np.array_equal(s[:, d], np.bincount(want, minlength=k).astype(np.float64))
    exact = oracle.kmeans_update_f64(data, want, cen)
    new_fast, shift_fast = ops.kmeans_finalize(sums, dev(cen))
    new_ord, shift_ord = ops.kmeans_update_ordered(dev(data), lab, dev(cen))
    ref_new, _ = oracle.kmeans_update(data, want, cen)
    assert_bits_equal(new_ord.cpu().numpy(), ref_new, "ordered update")
    nf = new_fast.cpu().numpy()
    assert np.allclose(nf, exact.astype(np.float32), rtol=0, atol=0) or np.abs(nf - exact).max() <= 1e-7 * np.abs(exact).max()
    scale = np.abs(ref_new).max(axis=1)
    assert (np.abs(nf - ref_new).max(axis=1) <= 1e-5 * scale).all()
    want_shift = np.linalg.norm(ref_new - cen)
    assert abs(float(shift_ord.item()) - want_shift) <= 2e-6 * max(1.0, want_shift)
    assert abs(float(shift_fast.item()) - np.linalg.norm(nf - cen)) <= 2e-6 * max(1.0, want_shift)


def test_screened_assignment_equals_float64_scan(oracle, monkeypatch):
    """The float32 screening + float64 near-tie path must return exactly the labels of the plain
    float64 scan (GSLIFT_KMEANS_EXACT=1) and of the oracle, also on adversarial inputs."""
    ops = pkg("ops")
    rng = np.random.default_rng(12)
    cases = []
    for d, k in [(6, 10), (59, 64), (16, 5), (33, 40), (3, 200)]:
        cen = rng.standard_normal((k, d)).astype(np.float32)
        pts = rng.standard_normal((20000, d)).astype(np.float32)
        # points on / next to bisecting planes of centroid pairs: near ties in float64
        i, j = rng.integers(0, k, 4000), rng.integers(0, k, 4000)
        mid = ((cen[i].astype(np.float64) + cen[j]) / 2).astype(np.float32)
        wob = mid + (rng.standard_normal(mid.shape) * 1e-6).astype(np.float32)
        cases.append((f"normal d{d} k{k}", np.concatenate([pts, mid, wob]), cen))
    cen = (rng.standard_normal((64, 59)) * 0.01 + 1000.0).astype(np.float32)     # far from the origin, tight
    cases.append(("offset", (rng.standard_normal((30000, 59)) * 0.01 + 1000.0).astype(np.float32), cen))
    cen = (rng.standard_normal((10, 6)) * 1e-21).astype(np.float32)               # below float32 range when squared
    cases.append(("tiny", (rng.standard_normal((5000, 6)) * 1e-21).astype(np.float32), cen))
    cen = (rng.standard_normal((10, 6)) * 1e25).astype(np.float32)                # squares overflow float32
    cases.append(("huge", (rng.standard_normal((5000, 6)) * 1e25).astype(np.float32), cen))
    cen = (rng.standard_normal((64, 59)) * 0.01 + 1000.0).astype(np.float32)
    pts = rng.standard_normal((30000, 59)).astype(np.float32) * 0.01 + 1000.0
    pts[::3] = np.nan                                                              # NaN rows -> label 0 like the scan
    pts[1::7, 5] = np.inf
    cases.append(("nonfinite", pts.astype(np.float32), cen))
    for name, data, cen in cases:
        with np.errstate(all="ignore"):
            want, gap = oracle.kmeans_assign(data, cen, want_gap=True)
        monkeypatch.delenv("GSLIFT_KMEANS_EXACT", raising=False)
        monkeypatch.setenv("GSLIFT_KMEANS_TC", "0")                                # float32 CUDA-core screening
        cc = ops.kmeans_assign(dev(data), dev(cen)).cpu().numpy()
        monkeypatch.delenv("GSLIFT_KMEANS_TC", raising=False)                      # tensor-core screening where it applies
        fast = ops.kmeans_assign(dev(data), dev(cen)).cpu().numpy()
        assert np.array_equal(fast, cc), f"{name}: tensor-core and CUDA-core screening disagree on {(fast != cc).sum()} rows"
        fast2 = ops.kmeans_step(dev(data), dev(cen))[0].cpu().numpy()
        monkeypatch.setenv("GSLIFT_KMEANS_EXACT", "1")
        slow = ops.kmeans_assign(dev(data), dev(cen)).cpu().numpy()
        monkeypatch.delenv("GSLIFT_KMEANS_EXACT", raising=False)
        assert np.array_equal(fast, slow), f"{name}: screening changed {(fast != slow).sum()} labels"
        assert np.array_equal(fast, fast2), name
        assert np.array_equal(fast.astype(np.int64), want), f"{name}: {(fast != want).sum()} differ from the oracle (ties {int((gap == 0).sum())})"


def test_tensor_core_screening_bound_holds_on_data():
    """Stage A forwards a candidate set that provably contains the nearest centroid only if its
    error bound holds; the self-test kernel measures the bound against float64 on every
    (row, centroid) pair and reports how many candidates survive."""
    native, scene = pkg("_native"), pkg("scene")
    rng = np.random.default_rng(3)
    sets = []
    data = scene.blob_features(200_000, 59, n_blobs=64, seed=5)
    sets.append(("C5 first iteration (centroids = data rows)", data, data[rng.choice(len(data), 64, replace=False)]))
    lab = np.argmin(((data[:, None, :3] - data[rng.choice(len(data), 64), None, :3][:, 0][None]) ** 2).sum(-1), 1)
    cen = np.stack([data[lab == k].mean(0) if (lab == k).any() else data[k] for k in range(64)]).astype(np.float32)
    sets.append(("C5 converged-like (centroids = blob means)", data, cen))
    off = (rng.standard_normal((100_000, 32)) * 0.05 + 500.0).astype(np.float32)
    sets.append(("far offset, tight", off, off[rng.choice(len(off), 40, replace=False)]))
    wide = (rng.standard_normal((100_000, 8)) * np.array([1e-3, 1, 1e3, 1, 1, 1e2, 1, 1e-2])).astype(np.float32)
    sets.append(("mixed scales D=8", wide, wide[rng.choice(len(wide), 16, replace=False)]))
    for name, x, c in sets:
        out = torch.zeros(3, dtype=torch.int64, device=DEV)
        labels = torch.empty(len(x), dtype=torch.int32, device=DEV)
        dx, dc = dev(x), dev(c)
        native.check(native.lib().gsl_kmeans_screen_selftest(dx.data_ptr(), len(x), x.shape[1], dc.data_ptr(), len(c),
                                                             labels.data_ptr(), out.data_ptr(), None))
        torch.cuda.synchronize()
        viol, cand, skip = (int(v) for v in out.tolist())
        print(f"[tc screen] {name}: bound violations {viol}, candidates per row {cand / len(x):.3f}")
        assert viol == 0
        assert skip == 0, "ordinary data must stay inside the range where the bound is proven"


def test_ties_duplicates_and_determinism(oracle):
    ops = pkg("ops")
    rng = np.random.default_rng(5)
    base = rng.standard_normal((40, 6)).astype(np.float32)
    data = np.repeat(base, 50, axis=0)
    cen = np.concatenate([base[:5], base[:5]])          # every member of 5 blobs ties exactly
    want, gap = oracle.kmeans_assign(data, cen, want_gap=True)
    got = ops.kmeans_assign(dev(data), dev(cen)).cpu().numpy()
    assert np.array_equal(got, want)                    # lowest index on both sides
    assert (gap[:250] == 0).all()
    big = rng.standard_normal((200_003, 59)).astype(np.float32)
    c0 = big[:64].copy()
    a = ops.kmeans_step(dev(big), dev(c0))
    b = ops.kmeans_step(dev(big), dev(c0))
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]), "sums must be bit-reproducible"


def test_unaligned_slice_and_sharded_sums(oracle):
    """Row slices (what a rank owns) need not be 16-byte aligned; per-slice sums add up to the
    whole -- the exchange step of the multi-GPU path, emulated on one device."""
    ops = pkg("ops")
    rng = np.random.default_rng(8)
    data = rng.standard_normal((30011, 59)).astype(np.float32)
    cen = data[rng.choice(len(data), 64, replace=False)]
    d_all, d_cen = dev(data), dev(cen)
    lab_all, sums_all = ops.kmeans_step(d_all, d_cen)
    total = torch.zeros_like(sums_all)
    sharding = pkg("sharding")
    for r in range(3):
        lo, hi = sharding.slice_bounds(len(data), r, 3)
        part = d_all[lo:hi]                              # a view: offset lo*59*4 bytes
        lab, sums = ops.kmeans_step(part, d_cen)
        assert torch.equal(lab, lab_all[lo:hi])
        total += sums
    assert torch.equal(total[:, 59], sums_all[:, 59])
    assert torch.allclose(total, sums_all, rtol=1e-12, atol=0)
    new_a, _ = ops.kmeans_finalize(total, d_cen)
    new_b, _ = ops.kmeans_finalize(sums_all, d_cen)
    assert (new_a - new_b).abs().max().item() <= 1e-6


def test_c5_shape_subsample_step_locked(oracle):
    """K=64, D=59 (config C5) at 1.5M rows: labels vs oracle, fast vs reference mean."""
    ops, scene = pkg("ops"), pkg("scene")
    n = 1_500_000
    data = scene.blob_features(n, 59, n_blobs=64, seed=5)
    np.random.seed(0)
    cen = data[np.random.choice(n, 64, replace=False)]
    d_data = dev(data)
    cur = cen
    for it in range(2):
        want, gap = oracle.kmeans_assign(data, cur, want_gap=True)
        lab, sums = ops.kmeans_step(d_data, dev(cur))
        got = lab.cpu().numpy().astype(np.int64)
        bad = got != want
        assert not (bad & (gap > 0)).any()
        ref_new, counts = oracle.kmeans_update(data, want, cur)
        new_fast = ops.kmeans_finalize(sums, dev(cur))[0].cpu().numpy()
        new_ord = ops.kmeans_update_ordered(d_data, lab, dev(cur))[0].cpu().numpy()
        exact = oracle.kmeans_update_f64(data, want, cur)
        scale = np.abs(ref_new).max(axis=1)
        rel_ref = (np.abs(new_fast - ref_new).max(axis=1) / scale).max()
        rel_exact = (np.abs(new_fast - exact).max(axis=1) / scale).max()
        print(f"[C5 1.5M it{it}] ties {int((gap == 0).sum())}, mismatches {int(bad.sum())}, largest cluster {counts.max()}, "
              f"fast vs reference f32 mean {rel_ref:.2e}, fast vs exact mean {rel_exact:.2e}")
        assert bad.sum() == 0
        assert_bits_equal(new_ord, ref_new, f"ordered update, iteration {it}")
        ref_drift = (np.abs(ref_new - exact).max(axis=1) / scale).max()      # the reference's own float32 accumulation error
        print(f"[C5 1.5M it{it}] reference f32 mean vs exact mean {ref_drift:.2e}")
        # north_star asks for 1e-5 against the reference.  The fast update is the exact mean rounded once
        # (< 1e-7), so its distance from the reference IS the reference's drift (SURVEY H6), which exceeds
        # 1e-5 on clusters of ~1e5 members; that is asserted as such instead of loosening a constant.
        assert rel_exact < 1e-7 and rel_ref <= ref_drift + 2e-7
        cur = ref_new


def test_fused_exchange_single_rank_equals_three_step_form():
    """gsl_kmeans_step_exchange on one rank (the exchange pushes into its own buffer) must give
    exactly what step + finalize give: same labels, same float64 totals, same centroids and shift,
    over several calls (parity of the slots alternates) and for an empty shard."""
    ops = pkg("ops")
    rng = np.random.default_rng(21)
    for n, d, k in ((40_000, 59, 64), (5_000, 6, 10), (777, 33, 17)):
        data = rng.standard_normal((n, d)).astype(np.float32)
        cen = dev(data[rng.choice(n, k, replace=False)])
        d_data = dev(data)
        xch = ops.KMeansExchange(k, d, d_data.device)
        lab_x = torch.empty(n, dtype=torch.int32, device=DEV)
        for it in range(3):
            lab, sums = ops.kmeans_step(d_data, cen)
            new, shift = ops.kmeans_finalize(sums, cen)
            new_x, shift_x = xch.step(d_data, cen, lab_x)
            assert torch.equal(lab_x, lab) and torch.equal(xch.sums, sums)
            assert torch.equal(new_x, new) and torch.equal(shift_x, shift)
            cen = new
        empty = torch.empty((0, d), dtype=torch.float32, device=DEV)
        new_e, shift_e = xch.step(empty, cen, torch.empty(0, dtype=torch.int32, device=DEV))
        assert torch.equal(new_e, cen) and float(shift_e.item()) == 0.0 and float(xch.sums.abs().sum().item()) == 0.0


_MGPU_WORKER = r'''
import os, sys, importlib
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
gs = importlib.import_module("3d_gaussian_splatting_project_b200")
ops, sharding, km = gs.ops, gs.sharding, gs.k_means
rank, world, local = sharding.init_from_env("nccl")
dev = torch.device("cuda", local)
n, d, k = 400_003, 59, 64
data = gs.scene.blob_features(n, d, n_blobs=64, seed=5)
np.random.seed(0)
cen0 = torch.from_numpy(data[np.random.choice(n, k, replace=False)]).to(dev)
lo, hi = sharding.slice_bounds(n, rank, world)
mine = torch.from_numpy(data[lo:hi]).to(dev)
xch = ops.KMeansExchange(k, d, dev)
lab = torch.empty(hi - lo, dtype=torch.int32, device=dev)
cen = cen0.clone()
for it in range(6):
    # three-step form: reduce kernel, NCCL all-reduce, finalize kernel
    lab_n, sums_n = ops.kmeans_step(mine, cen)
    dist.all_reduce(sums_n)
    new_n, shift_n = ops.kmeans_finalize(sums_n, cen)
    # fused form over peer memory
    new_x, shift_x = xch.step(mine, cen, lab)
    assert torch.equal(lab, lab_n)
    assert torch.equal(xch.sums[:, d], sums_n[:, d]), "member counts differ"
    assert torch.allclose(xch.sums, sums_n, rtol=1e-13, atol=0), (xch.sums - sums_n).abs().max().item()
    assert (new_x - new_n).abs().max().item() <= 1e-6 and abs(float(shift_x) - float(shift_n)) <= 1e-6
    # every rank must hold bit-identical totals and centroids (rank-ordered sum)
    gathered = [torch.empty_like(new_x) for _ in range(world)]
    dist.all_gather(gathered, new_x)
    assert all(torch.equal(g, gathered[0]) for g in gathered), "ranks disagree on the centroids"
    cen = new_x
# the drop-in loop on shards == the same loop on one device holding everything
cen_s, lab_s, it_s = km.lloyd(mine, cen0, max_iter=4, tol=0.0, verbose=False)
if rank == 0:
    full = torch.from_numpy(data).to(dev)
dist.barrier()
whole = sharding.gather_labels(lab_s, n, rank, world)
if rank == 0:
    lab1, sums1 = ops.kmeans_step(full, cen_s)      # labels under the final centroids, one device
    assert torch.equal(whole, lab1), int((whole != lab1).sum())
torch.cuda.synchronize(); dist.barrier(); dist.destroy_process_group()
print("ok", rank)
'''


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs on one node")
def test_fused_exchange_over_peer_memory_two_ranks(tmp_path):
    """One process per GPU: the fused exchange kernel against NCCL all-reduce, step by step."""
    import os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = tmp_path / "mgpu_worker.py"
    script.write_text(_MGPU_WORKER)
    n = min(torch.cuda.device_count(), 8)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
                          "--master-addr", "127.0.0.1", "--master-port", "29741", str(script), root],
                         capture_output=True, text=True, env=env, timeout=600)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert out.stdout.count("ok") == n
