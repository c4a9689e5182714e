"""The majority kernel counts sheet words in whole batches of 16 (unpredicated loads) and one
partial batch.  View counts on both sides of the batch edges, for the 16-bit view-resolution keys
(V <= 255), the 16-bit word-resolution keys (256 <= V <= 508) and the 32-bit keys, against the
oracle -- on scenes with few labels, where the two votes of a pair often name the same slot and
counts tie often."""
import numpy as np
import pytest
import torch

from util import pkg

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _lift(pos, cams, maps):
    ops = pkg("ops")
    shapes = [m.shape for m in maps]
    views = ops.make_views(cams, shapes)
    flat = np.concatenate([np.ascontiguousarray(m, np.int32).reshape(-1) for m in maps])
    packed = ops.pack_labels(torch.from_numpy(flat).to(DEV), shapes)
    out = ops.lift_votes(torch.from_numpy(np.ascontiguousarray(pos, np.float32)).to(DEV), views, packed)
    torch.cuda.synchronize()
    return out.cpu().numpy()


# sheet words = ceil(V / 4): 15, 16, 17 | 32, 33 | 64, 65 | 80, 81 -- no whole batch, one whole batch
# and no partial one, whole batches with and without a partial one
@pytest.mark.parametrize("v", [60, 64, 65, 128, 129, 256, 260, 320, 321])
@pytest.mark.parametrize("wide", [False, True])
def test_view_counts_around_batch_edges(oracle, monkeypatch, v, wide):
    scene = pkg("scene")
    cams = scene.lookat_cameras(v, width=48, height=32, seed=800 + v)
    pos = scene.gaussian_cloud(3000, 1.5, seed=801 + v)
    maps = [scene.block_label_map(32, 48, 4, 0, 2, 900 + v + i) for i in range(v)]
    want, _, _ = oracle.lift_votes(pos, oracle.make_views(cams, [(32, 48)] * v), np.stack(maps))
    if wide:
        monkeypatch.setenv("GSLIFT_MAJORITY_WIDE", "1")
    got = _lift(pos, cams, maps)
    bad = got != want
    assert not bad.any(), f"{bad.sum()} of {len(want)} labels differ"


def test_best_keys_merge_across_passes_with_whole_batches(oracle):
    """Winning keys (`best`) of label passes over 70 views (17 sheet words: one whole batch and a
    partial one) merge to the reference's answer."""
    dls, scene = pkg("deep_learning_segmentation"), pkg("scene")
    v = 70
    cams = scene.lookat_cameras(v, width=160, height=100, seed=61)
    pos = scene.gaussian_cloud(1000, 1.5, seed=62)
    rng = np.random.default_rng(63)
    ids = np.unique(rng.integers(-2**31, 2**31 - 1, 600, dtype=np.int64)).astype(np.int32)
    maps = [ids[scene.block_label_map(100, 160, 20, 0, len(ids) - 1, 700 + i)] for i in range(v)]
    got = dls.lift_labels(pos, cams, maps)
    assert dls.last_call_stats["label_passes"] >= 2
    want = oracle.lift_votes_py(pos, cams, maps)
    bad = got != want
    assert not bad.any(), f"{bad.sum()} of {len(want)} labels differ"
