"""Parity of the CUDA lifting path (through the C ABI) with the oracle and the reference's
golden vectors.  Bar: labels bit-exact; the only tolerated differences are Gaussians with a
projection within 1e-4 px of a pixel boundary (north_star), whose count is reported."""
import contextlib
import io
import os

import numpy as np
import pytest
import torch

from util import LIFT_CASES, load_lift_case, pkg

pytestmark = pytest.mark.gpu
DEV = "cuda"


def gpu_lift(pos, cameras, maps_list, sizes, **kw):
    ops = pkg("ops")
    shapes = [m.shape for m in maps_list]
    views = ops.make_views(cameras, shapes, sizes)
    flat = np.concatenate([np.ascontiguousarray(m, np.int32).reshape(-1) for m in maps_list]) if maps_list else np.zeros(0, np.int32)
    packed = ops.pack_labels(torch.from_numpy(flat).to(DEV), shapes) if maps_list else torch.zeros(0, dtype=torch.uint8, device=DEV)
    res = ops.lift_votes(torch.from_numpy(np.ascontiguousarray(pos, np.float32)).to(DEV), views, packed, **kw)
    torch.cuda.synchronize()
    return res


def compare(got, want, near=None):
    bad = got != want
    if near is not None:
        outside = bad & (near == 0)
        assert not outside.any(), f"{outside.sum()} mismatches away from any pixel boundary"
    else:
        assert not bad.any(), f"{bad.sum()} of {len(want)} labels differ"
    return int(bad.sum())


@pytest.mark.parametrize("name", LIFT_CASES)
def test_golden_vectors_from_the_verbatim_reference(name):
    c = load_lift_case(name)
    got = gpu_lift(c["pos"], c["cameras"], c["maps"], c["sizes"]).cpu().numpy()
    assert got.dtype == np.int32
    compare(got, c["labels"])


@pytest.mark.parametrize("name", ["lift_lookat_regions", "lift_bundled_halfres"])
def test_dropin_assign_labels_end_to_end(name, tmp_path):
    """Through the reference-facing function: PNG probes, per-view prints, segmenter hook."""
    from PIL import Image
    dls = pkg("deep_learning_segmentation")
    c = load_lift_case(name)
    cams = [dict(cam) for cam in c["cameras"]]
    by_name = {cam["img_name"]: i for i, cam in enumerate(cams)}
    for cam, (w, h) in zip(cams, c["sizes"]):
        Image.new("L", (w, h)).save(tmp_path / (cam["img_name"] + ".png"))
    ghost = dict(cams[1], img_name="not_on_disk")          # skipped with a warning (dls:257-259)
    cams_in = cams[:1] + [ghost] + cams[1:]
    g = np.zeros(len(c["pos"]), dls.GAUSSIAN_DTYPE)
    g["position"] = c["pos"]
    seg = lambda path, out_dir, model_type: c["maps"][by_name[os.path.splitext(os.path.basename(path))[0]]]
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        labels = dls.assign_labels(g, cams_in, str(tmp_path), str(tmp_path / "out"), segmenter=seg)
    lines = buf.getvalue().splitlines()
    assert lines[1] == "Warning: Image not_on_disk not found"
    assert sum(l.startswith("Processing image") for l in lines) == len(cams)
    assert labels.dtype == np.int32
    compare(labels, c["labels"])
    # precomputed <img>_segmap.npy files (what the reference's segment_image leaves behind, dls:165)
    os.makedirs(tmp_path / "pre", exist_ok=True)
    for cam, m in zip(cams, c["maps"]):
        np.save(tmp_path / "pre" / f"{cam['img_name']}_segmap.npy", m)
    # ... are reused only on request (the reference always recomputes them): without the switch
    # and without a segmenter the call must ask for one
    os.environ.pop("GSLIFT_REUSE_SEGMAPS", None)
    os.environ.pop("GSLIFT_REFERENCE_DIR", None)
    with contextlib.redirect_stdout(io.StringIO()), pytest.raises(RuntimeError, match="no segmenter"):
        dls.assign_labels(g, cams, str(tmp_path), str(tmp_path / "pre"))
    os.environ["GSLIFT_REUSE_SEGMAPS"] = "1"
    try:
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf):
            labels2 = dls.assign_labels(g, cams, str(tmp_path), str(tmp_path / "pre"))
    finally:
        del os.environ["GSLIFT_REUSE_SEGMAPS"]
    assert buf.getvalue().count("Using precomputed segmentation map") == len(cams)
    compare(labels2, c["labels"])


def _scene(n, v, w, h, seed, block=16):
    scene = pkg("scene")
    cams = scene.lookat_cameras(v, width=w, height=h, seed=seed)
    pos = scene.gaussian_cloud(n, 1.5, seed=seed + 1)
    maps = scene.block_label_maps(v, h, w, block=block, seed=seed + 2)
    return cams, pos, maps


@pytest.mark.parametrize("n,v,w,h", [(1, 1, 64, 48), (31, 3, 64, 48), (1000, 5, 320, 200), (70001, 37, 640, 360), (300000, 24, 960, 540)])
def test_random_scenes_against_oracle(oracle, n, v, w, h):
    cams, pos, maps = _scene(n, v, w, h, seed=100 + v)
    shapes = [(h, w)] * v
    want, near, vis = oracle.lift_votes(pos, oracle.make_views(cams, shapes), maps, eps=1e-4, want_near=True)
    got, gnear = gpu_lift(pos, cams, list(maps), None, want_near=True, near_eps=1e-4)
    got, gnear = got.cpu().numpy(), gnear.cpu().numpy()
    flips = compare(got, want, near)
    assert np.array_equal(gnear, near), "near-boundary set differs from the oracle's"
    print(f"[lift {n}x{v}] visible pairs {vis}, near-boundary Gaussians {int(near.sum())}, label flips {flips}")
    assert flips == 0            # same dgemv formula on both sides: expect none even inside the band


def test_shared_reciprocal_division_is_ieee_exact():
    """The gather kernel divides fx*X and fy*Y by Z with one shared reciprocal; the result
    must equal IEEE-754 division bit for bit, on ordinary and on extreme operands."""
    native = pkg("_native")
    rng = np.random.default_rng(17)
    n = 1 << 22
    def draw(kind):
        if kind == "scene":
            return rng.standard_normal(n) * rng.choice([1e-3, 1.0, 50.0, 4000.0], n)
        bits = rng.integers(0, 2**63, n, dtype=np.int64) | (rng.integers(0, 2, n, dtype=np.int64) << 63)
        return bits.view(np.float64)
    for kind in ("scene", "bits"):
        a1, a2, b = draw(kind), draw(kind), draw(kind)
        if kind == "bits":
            b[:8] = [0.0, -0.0, np.inf, -np.inf, np.nan, 5e-324, 1e308, -1e-308]
            a1[:8] = [1.0, 0.0, np.inf, 1.0, 1.0, 5e-324, 1e308, 1e308]
        bad = torch.zeros(1, dtype=torch.int64, device=DEV)
        t = [torch.from_numpy(x).to(DEV) for x in (a1, a2, b)]
        native.check(native.lib().gsl_div_selftest(t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), n, bad.data_ptr(), None))
        torch.cuda.synchronize()
        assert int(bad.item()) == 0, f"{int(bad.item())} of {n} quotients differ from IEEE division ({kind})"


def test_ordering_and_culling_do_not_change_results(oracle, monkeypatch):
    """Spatial ordering + per-tile frustum culling (GSLIFT_LIFT_ORDER, default on) is an
    execution-order change only: same labels and same near-boundary set as the plain sweep,
    also when most pairs are invisible (bundled cameras) and with non-finite positions."""
    c = load_lift_case("lift_bundled_halfres")
    rng = np.random.default_rng(4)
    pos = (rng.standard_normal((150_000, 3)) * 2.0).astype(np.float32)
    pos[::5000] = np.nan
    pos[7::9000, 1] = np.inf
    maps = [c["maps"][i % len(c["maps"])] for i in range(len(c["cameras"]))]
    with np.errstate(all="ignore"):
        want, near, vis = oracle.lift_votes(pos, oracle.make_views(c["cameras"], c["shapes"], c["sizes"]), c["flat"],
                                            eps=1e-4, want_near=True)
    out = {}
    for flag in ("1", "0"):
        monkeypatch.setenv("GSLIFT_LIFT_ORDER", flag)
        lab, nr = gpu_lift(pos, c["cameras"], maps, c["sizes"], want_near=True, near_eps=1e-4)
        out[flag] = (lab.cpu().numpy(), nr.cpu().numpy())
    monkeypatch.delenv("GSLIFT_LIFT_ORDER", raising=False)
    assert np.array_equal(out["1"][0], out["0"][0]) and np.array_equal(out["1"][1], out["0"][1])
    compare(out["1"][0], want)
    assert np.array_equal(out["1"][1], near)
    print(f"[order/cull] bundled cameras: {vis / (len(pos) * len(c['cameras'])):.1%} of pairs visible")


def test_many_views_and_key_widths(oracle):
    cams, pos, maps = _scene(5000, 11, 160, 90, seed=7)
    want, _, _ = oracle.lift_votes(pos, oracle.make_views(cams, [(90, 160)] * 11), maps)
    compare(gpu_lift(pos, cams, list(maps), None).cpu().numpy(), want)
    # many windows, the last one partial (401 = 25 * 16 + 1); many tiny maps
    cams, pos, maps = _scene(3000, 401, 48, 32, seed=9, block=4)
    want, _, _ = oracle.lift_votes(pos, oracle.make_views(cams, [(32, 48)] * 401), maps)
    compare(gpu_lift(pos, cams, list(maps), None).cpu().numpy(), want)
    # 256 <= V <= 508 counts with 16-bit word-resolution keys; the 32-bit keys must agree, also on a
    # tie-heavy scene (few labels, so equal counts with first sightings inside one group of four views are common)
    scene = pkg("scene")
    few = np.stack([scene.block_label_map(32, 48, 4, 0, 2, 700 + i) for i in range(401)])
    want_few, _, _ = oracle.lift_votes(pos, oracle.make_views(cams, [(32, 48)] * 401), few)
    compare(gpu_lift(pos, cams, list(few), None).cpu().numpy(), want_few)
    os.environ["GSLIFT_MAJORITY_WIDE"] = "1"
    try:
        compare(gpu_lift(pos, cams, list(few), None).cpu().numpy(), want_few)
    finally:
        del os.environ["GSLIFT_MAJORITY_WIDE"]


def test_rescaled_and_ragged_maps(oracle):
    """Different seg-map size per view, image size != map size != camera size (SURVEY H4)."""
    scene = pkg("scene")
    cams = scene.lookat_cameras(6, width=800, height=450, seed=21)
    pos = scene.gaussian_cloud(20000, 1.5, seed=22)
    shapes = [(450, 800), (225, 400), (100, 333), (450, 800), (77, 51), (900, 1600)]
    sizes = [(800, 450), (800, 450), (640, 360), (400, 225), (800, 450), (800, 450)]
    maps = [scene.block_label_map(h, w, 8, -1, 149, 300 + i) for i, (h, w) in enumerate(shapes)]
    flat = np.concatenate([m.reshape(-1) for m in maps])
    want, _, _ = oracle.lift_votes(pos, oracle.make_views(cams, shapes, sizes), flat)
    compare(gpu_lift(pos, cams, maps, sizes).cpu().numpy(), want)


def test_empty_inputs_and_label_range():
    ops = pkg("ops")
    cams, pos, maps = _scene(100, 2, 64, 48, seed=3)
    out = gpu_lift(pos[:0], cams, list(maps), None)
    assert out.numel() == 0
    none = ops.lift_votes(torch.from_numpy(pos).to(DEV), ops.make_views([], []), torch.zeros(0, dtype=torch.uint8, device=DEV))
    assert (none.cpu().numpy() == -1).all()            # no views: nothing visible (dls:306)
    bad = torch.full((8, 8), 1000, dtype=torch.int32, device=DEV)
    with pytest.raises(ValueError):
        ops.pack_labels(bad)
    assert ops.label_range(torch.tensor([5, -3, 77], dtype=torch.int32, device=DEV)) == (-3, 77)
    dls, scene = pkg("deep_learning_segmentation"), pkg("scene")
    maps0 = [scene.block_label_map(48, 64, 4, 0, 149, 50 + i) for i in range(2)]   # no -1 label
    shifted = [m + 1000 for m in maps0]                # ids outside the default window: remapped
    got = dls.lift_labels(pos, cams, shifted)
    ref = dls.lift_labels(pos, cams, maps0)
    assert (ref >= 0).any() and np.array_equal(np.where(ref == -1, -1, ref + 1000), got)
    # no Gaussians, or no views, through lift_labels: -1 labels of the right length, a zero mask
    for p, cc, mm in ((pos[:0], cams, list(maps)), (pos, [], [])):
        labels = dls.lift_labels(p, cc, mm)
        assert labels.dtype == np.int32 and labels.shape == (len(p),) and (labels == -1).all()
        labels, near = dls.lift_labels(p, cc, mm, want_near=True)
        assert labels.shape == near.shape == (len(p),) and (labels == -1).all() and not near.any()


def test_full_size_c3_properties_and_oracle(oracle):
    """BASELINE config C3 shape (1M x 200 views, 1920x1080): slicing invariance (the multi-GPU
    sharding property), permutation equivariance, determinism; and the oracle on a 1/8 slice."""
    scene, ops = pkg("scene"), pkg("ops")
    n, v, w, h = 1_000_000, 200, 1920, 1080
    cams = scene.lookat_cameras(v, width=w, height=h, seed=3)
    pos = scene.gaussian_cloud(n, 1.5, seed=3)
    views = ops.make_views(cams, [(h, w)] * v)
    pb = ops.packed_map_bytes(h, w)
    packed = torch.empty(v * pb, dtype=torch.uint8, device=DEV)
    maps = scene.block_label_maps(v, h, w, block=32, seed=1000)
    for v0 in range(0, v, 8):                          # stage + pack 8 maps at a time
        ops.pack_labels(torch.from_numpy(maps[v0:v0 + 8]).to(DEV), out=packed[v0 * pb:(v0 + 8) * pb])
    d_pos = torch.from_numpy(pos).to(DEV)
    full = ops.lift_votes(d_pos, views, packed).cpu().numpy()
    again = ops.lift_votes(d_pos, views, packed).cpu().numpy()
    assert np.array_equal(full, again)
    # float32 screening and ordering+culling (both default) are execution strategies only
    for var, val in (("GSLIFT_LIFT_F64", "1"), ("GSLIFT_LIFT_ORDER", "0")):
        os.environ[var] = val
        try:
            plain = ops.lift_votes(d_pos, views, packed).cpu().numpy()
        finally:
            del os.environ[var]
        assert np.array_equal(plain, full), f"{var}={val} changes {(plain != full).sum()} labels"
    lo, hi = 375_000, 500_000                           # rank 3 of 8
    part = ops.lift_votes(d_pos[lo:hi].contiguous(), views, packed).cpu().numpy()
    assert np.array_equal(part, full[lo:hi])
    perm = np.random.default_rng(0).permutation(n)
    shuffled = ops.lift_votes(torch.from_numpy(pos[perm]).to(DEV), views, packed).cpu().numpy()
    assert np.array_equal(shuffled, full[perm])
    # oracle on the same slice, all 200 views
    want, near, vis = oracle.lift_votes(pos[lo:hi], oracle.make_views(cams, [(h, w)] * v), maps, eps=1e-4, want_near=True)
    flips = compare(part, want, near)
    print(f"[C3 slice] {hi - lo} Gaussians x {v} views: visible pairs {vis} ({vis / ((hi - lo) * v):.1%}), "
          f"near-boundary Gaussians {int(near.sum())}, flips {flips}")
    assert flips == 0


def test_float32_screening_hard_cases_against_oracle(oracle):
    """Inputs chosen to sit on the float32 screening's decision edges: points on and next to the
    camera plane (z ~ 0), projections a hair from pixel edges and from the image border, huge and
    tiny coordinates (the bound turns NaN and everything is re-evaluated in float64), views far
    from the origin (large |t|: loose bound, many re-evaluations), mixed frame sizes in one window.
    The float32-screened sweep, the float64 sweep and the oracle must agree label for label."""
    scene = pkg("scene")
    rng = np.random.default_rng(77)
    cams = scene.lookat_cameras(20, width=640, height=360, seed=31)
    for i, c in enumerate(cams[:6]):                       # push six cameras far away: |t| grows, z stays positive
        c["position"] = [float(v) * (50.0 + 400.0 * i) for v in c["position"]]
    for c in cams[6:9]:                                    # other frame sizes inside the same 16-view window
        c["width"], c["height"] = 320, 200
    shapes = [(int(c["height"]), int(c["width"])) for c in cams]
    maps = [scene.block_label_map(h, w, 1, -1, 149, 900 + i) for i, (h, w) in enumerate(shapes)]   # every pixel its own label
    n = 60_000
    pos = (rng.standard_normal((n, 3)) * 1.5).astype(np.float32)
    views64 = oracle.make_views(cams, shapes)
    # points constructed to project onto exact pixel edges of camera 10 (then nudged by a few float32 ulps)
    R = np.array(cams[10]["rotation"]); p = np.array(cams[10]["position"])
    k = 4000
    px = rng.integers(0, 641, k).astype(np.float64); py = rng.integers(0, 361, k).astype(np.float64)
    z = rng.uniform(3.0, 9.0, k)
    cam_pts = np.stack([(px - 320.0) * z / cams[10]["fx"], (py - 180.0) * z / cams[10]["fy"], z], axis=1)
    world = (np.linalg.inv(R) @ cam_pts.T).T + p
    pos[:k] = world.astype(np.float32)
    pos[k:2 * k] = np.nextafter(pos[:k], np.float32(np.inf))
    pos[2 * k:3 * k] = np.nextafter(pos[:k], np.float32(-np.inf))
    # points on the camera plane of camera 11 (z ~ 0 within rounding)
    R = np.array(cams[11]["rotation"]); p = np.array(cams[11]["position"])
    plane = np.stack([rng.uniform(-3, 3, 2000), rng.uniform(-3, 3, 2000), rng.uniform(-1e-6, 1e-6, 2000)], axis=1)
    pos[3 * k:3 * k + 2000] = ((np.linalg.inv(R) @ plane.T).T + p).astype(np.float32)
    pos[20000:20050] *= np.float32(1e20)                   # beyond the sanity limit of the float32 path
    pos[20050:20100] *= np.float32(1e-30)
    pos[20100] = [np.inf, 0.0, 0.0]; pos[20101] = [np.nan, 1.0, 1.0]; pos[20102] = [3e38, -3e38, 3e38]
    flat = np.concatenate([m.reshape(-1) for m in maps])
    with np.errstate(all="ignore"):
        want, near, vis = oracle.lift_votes(pos, views64, flat, eps=1e-4, want_near=True)
    got = gpu_lift(pos, cams, maps, None).cpu().numpy()
    os.environ["GSLIFT_LIFT_F64"] = "1"
    try:
        got64 = gpu_lift(pos, cams, maps, None).cpu().numpy()
    finally:
        del os.environ["GSLIFT_LIFT_F64"]
    assert np.array_equal(got, got64), f"float32-screened and float64 sweeps differ on {(got != got64).sum()} labels"
    flips = compare(got, want, near)
    print(f"[screening edges] visible pairs {vis}, near-boundary Gaussians {int(near.sum())}, flips {flips}")
    assert flips == 0


@pytest.mark.parametrize("fraction", ["0", "0.5", "1"])
def test_hybrid_staging_host_narrowed_views_give_the_same_labels(oracle, monkeypatch, fraction):
    """lift_labels from host maps: views narrowed to 1-byte codes on the host (gsl_host_pack_labels
    + gsl_tile_codes) and views that cross as int32 (gsl_pack_labels) must give the oracle's labels
    for every split, with ragged map shapes (scalar tile path), int64 / non-contiguous NumPy maps,
    CPU tensors, and 40 views (3 windows, the last one partial)."""
    dls, scene = pkg("deep_learning_segmentation"), pkg("scene")
    v = 40
    cams = scene.lookat_cameras(v, width=320, height=200, seed=41)
    pos = scene.gaussian_cloud(30_000, 1.5, seed=42)
    shapes = [(200, 320) if i % 3 else (111, 203) for i in range(v)]
    sizes = [(320, 200) if i % 3 else (301, 155) for i in range(v)]
    base = [scene.block_label_map(h, w, 4, -1, 149, 800 + i) for i, (h, w) in enumerate(shapes)]
    maps = []
    for i, m in enumerate(base):
        if i % 4 == 1:
            maps.append(m.astype(np.int64))                      # converted on the host
        elif i % 4 == 2:
            maps.append(np.asfortranarray(m))                    # not C-contiguous
        elif i % 4 == 3:
            maps.append(torch.from_numpy(m.copy()))              # CPU tensor
        else:
            maps.append(m)
    flat = np.concatenate([m.reshape(-1) for m in base])
    want, _, _ = oracle.lift_votes(pos, oracle.make_views(cams, shapes, sizes), flat)
    monkeypatch.setenv("GSLIFT_HOST_STAGE", fraction)
    got = dls.lift_labels(pos, cams, maps, sizes)
    compare(got, want)


@pytest.mark.parametrize("fraction", ["0", "0.5"])
def test_lift_labels_from_rows_of_one_pinned_tensor(oracle, monkeypatch, fraction):
    """The benchmark's call: pinned CPU positions, maps as rows of one pinned int32 tensor (they
    cross in coalesced copies), 48 views = three 16-view chunks, so that with a host share of 0.5
    one chunk crosses as int32 and two are narrowed on the host.  The byte counts of
    last_call_stats follow the split."""
    dls = pkg("deep_learning_segmentation")
    v, w, h = 48, 320, 200
    cams, pos, maps = _scene(30_000, v, w, h, seed=91)
    want, _, _ = oracle.lift_votes(pos, oracle.make_views(cams, [(h, w)] * v), maps)
    rows = torch.from_numpy(maps).pin_memory()
    monkeypatch.setenv("GSLIFT_HOST_STAGE", fraction)
    got = dls.lift_labels(torch.from_numpy(pos).pin_memory(), cams, [rows[i] for i in range(v)], None, device=DEV)
    compare(got, want)
    st = dls.last_call_stats
    as_int32, narrowed = st["views_as_int32"], st["views_narrowed_on_host"]
    assert as_int32 + narrowed == v and (as_int32, narrowed) == ((v, 0) if fraction == "0" else (16, 32))
    assert st["h2d_bytes"] == 4 * as_int32 * h * w + narrowed * h * w + 12 * len(pos)
    assert st["d2h_bytes"] == 4 * len(pos) and st["label_passes"] == 1


def test_lift_labels_explicit_code_window(oracle):
    """label_min and n_classes given together: the maps are packed with that window and the labels
    are the oracle's; a map value outside the window raises, and so does giving only one of the two."""
    dls = pkg("deep_learning_segmentation")
    v, w, h = 20, 320, 200
    cams, pos, maps = _scene(20_000, v, w, h, seed=81)
    want, _, _ = oracle.lift_votes(pos, oracle.make_views(cams, [(h, w)] * v), maps)
    compare(dls.lift_labels(pos, cams, list(maps), label_min=-1, n_classes=151), want)
    for bad_value in (150, -2):
        bad = maps.copy()
        bad[17, 5, 9] = bad_value
        with pytest.raises(ValueError, match="outside"):
            dls.lift_labels(pos, cams, list(bad), label_min=-1, n_classes=151)
    for half in ({"label_min": -1}, {"n_classes": 151}):
        with pytest.raises(ValueError, match="label_min and n_classes"):
            dls.lift_labels(pos, cams, list(maps), **half)


def test_lift_labels_want_near_equals_lift_votes():
    """want_near=True through lift_labels: labels and near-boundary mask of ops.lift_votes."""
    dls = pkg("deep_learning_segmentation")
    cams, pos, maps = _scene(40_000, 21, 320, 200, seed=83)
    labels, near = dls.lift_labels(pos, cams, list(maps), want_near=True, near_eps=1e-4)
    want, want_near = gpu_lift(pos, cams, list(maps), None, want_near=True, near_eps=1e-4)
    assert labels.dtype == np.int32 and near.dtype == np.uint8
    assert np.array_equal(labels, want.cpu().numpy()) and np.array_equal(near, want_near.cpu().numpy())
    assert near.any()


def test_more_than_255_distinct_labels(oracle):
    """The reference's vote dict takes any int32 label (dls:288-295): 1000 instance ids spread
    over the whole int32 range are lifted in passes of 254 dense ids and merged by vote key.
    Checked against the pure-Python restatement of the reference loop (dict of dicts)."""
    dls, scene = pkg("deep_learning_segmentation"), pkg("scene")
    v = 24
    cams = scene.lookat_cameras(v, width=320, height=200, seed=51)
    pos = scene.gaussian_cloud(3000, 1.5, seed=52)
    rng = np.random.default_rng(53)
    ids = np.unique(rng.integers(-2**31, 2**31 - 1, 1000, dtype=np.int64)).astype(np.int32)
    ids[0] = -1                                            # the "no segment" value is just another label
    # big regions, so that counts tie often and the first sighting decides -- also across passes
    maps = [ids[scene.block_label_map(200, 320, 40, 0, len(ids) - 1, 600 + i)] for i in range(v)]
    got = dls.lift_labels(pos, cams, maps)
    present = np.unique(np.concatenate([m.reshape(-1) for m in maps]))
    assert dls.last_call_stats["label_passes"] == -(-len(present) // 254) >= 2
    want = oracle.lift_votes_py(pos, cams, maps)
    compare(got, want)
    assert len(np.unique(got)) > 100


def test_device_resident_maps_written_just_before_the_call(oracle):
    """Maps that are CUDA tensors still being produced on the current stream when lift_labels is
    called (a segmenter running on the GPU): the staging streams must wait for them."""
    dls, scene = pkg("deep_learning_segmentation"), pkg("scene")
    v = 40
    cams = scene.lookat_cameras(v, width=640, height=360, seed=61)
    pos = scene.gaussian_cloud(50_000, 1.5, seed=62)
    host = [scene.block_label_map(360, 640, 8, -1, 149, 900 + i) for i in range(v)]
    want, _, _ = oracle.lift_votes(pos, oracle.make_views(cams, [(360, 640)] * v), np.stack(host))
    staged = [torch.from_numpy(m).to(DEV) for m in host]
    torch.cuda.synchronize()
    for rep in range(3):
        spin = torch.empty(64 << 20, dtype=torch.float32, device=DEV)
        for _ in range(20):
            spin.mul_(1.0001)                              # keep the stream busy ahead of the writes
        dev_maps = [(m * 1) for m in staged]               # produced asynchronously, right before the call
        got = dls.lift_labels(pos, cams, dev_maps)
        compare(got, want)


_MGPU_LIFT_WORKER = r'''
import os, sys, importlib
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
gs = importlib.import_module("3d_gaussian_splatting_project_b200")
from oracle import oracle as orc
sharding, dls, scene = gs.sharding, gs.deep_learning_segmentation, gs.scene
rank, world, local = sharding.init_from_env("nccl")
dev = torch.device("cuda", local)
v, w, h, n = 70, 640, 360, 120_001
cams = scene.lookat_cameras(v, width=w, height=h, seed=71)
pos = scene.gaussian_cloud(n, 1.5, seed=72)
maps = [scene.block_label_map(h, w, 8, -1, 149, 1000 + i) for i in range(v)]
lo, hi = sharding.slice_bounds(n, rank, world)
for rep in range(2):                                   # the second call reuses the symmetric-memory buffer
    mine = dls.lift_labels(pos[lo:hi], cams, maps, device=dev)
    whole = sharding.gather_labels(torch.from_numpy(mine).to(dev), n, rank, world)
    if rank == 0:
        want, _, _ = orc.lift_votes(pos, orc.make_views(cams, [(h, w)] * v), np.stack(maps))
        got = whole.cpu().numpy()
        assert np.array_equal(got, want), int((got != want).sum())
    if os.environ.get("GSLIFT_STAGE_EXCHANGE") != "nccl":
        assert dls.last_call_stats["h2d_bytes"] < 4 * w * h * (v // world + 1) + 12 * (hi - lo) + 64, dls.last_call_stats
torch.cuda.synchronize(); dist.barrier(); dist.destroy_process_group()
print("ok", rank)
'''


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs on one node")
@pytest.mark.parametrize("exchange", ["symm", "nccl"])
def test_sharded_staging_and_lifting_on_several_ranks(tmp_path, exchange):
    """One process per GPU through lift_labels: every rank uploads and packs only its block of
    views and pushes the packed chunks into all ranks' buffers over peer memory (or broadcasts them
    with NCCL); each rank lifts its slice of the Gaussians; gathered labels == the oracle's."""
    import subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = tmp_path / "mgpu_lift_worker.py"
    script.write_text(_MGPU_LIFT_WORKER)
    n = min(torch.cuda.device_count(), 8)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", GSLIFT_STAGE_EXCHANGE=exchange)
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
                          "--master-addr", "127.0.0.1", "--master-port", "29743", str(script), root],
                         capture_output=True, text=True, env=env, timeout=600)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert out.stdout.count("ok") == n
