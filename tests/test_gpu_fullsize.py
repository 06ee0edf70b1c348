"""Size-independent properties at BASELINE.json's full size (C3: 10M rows x 200 features, 256 bins,
depth 8), where the CPU oracle would take minutes per tree: conservation of row counts and of the
fixed-point sums across every split, exactness of sibling subtraction, run-to-run determinism,
monotone training loss, and an exact check of the root histogram against numpy."""
import numpy as np
import pytest

import ydf_b200
from tests.util import quantize_g

pytestmark = pytest.mark.gpu

W = dict(rows=10_000_000, features=200, max_depth=8, bins=256, informative=20)


@pytest.fixture(scope="module")
def data():
    import bench
    return bench.make_data(W, device=0)


def _train(data, iters, **kw):
    bins, nb, na, y = data
    ds = ydf_b200.Dataset(bins, nb, na)
    cfg = ydf_b200.default_config(max_depth=W["max_depth"], num_trees=iters, **kw)
    gbt = ydf_b200.Gbt(ds, cfg)
    gbt.set_labels(y)
    gbt.train(iters)
    trees = [gbt.get_tree(i) for i in range(iters)]
    losses = [gbt.train_loss(i)[0] for i in range(iters)]
    return ds, gbt, trees, losses


def _check_tree(t, n_rows):
    assert t[0]["num_examples"] == n_rows
    for nd in t:
        if nd["feature"] >= 0:
            pos, neg = t[nd["pos_child"]], t[nd["neg_child"]]
            # row conservation across the partition (SplitExamplesInPlace count check, training.cc:5269-5303)
            assert pos["num_examples"] == nd["num_pos_examples"]
            assert pos["num_examples"] + neg["num_examples"] == nd["num_examples"]
            assert pos["num_examples"] >= 5 and neg["num_examples"] >= 5  # min_examples in the split search
            assert pos["depth"] == nd["depth"] + 1 and nd["depth"] < W["max_depth"]
            # linearity of the statistics: a node's sums are the sums of its children's (fixed point: exact
            # up to the final int->double conversion)
            for s in range(3):
                tot = pos["stat"][s] + neg["stat"][s]
                assert abs(tot - nd["stat"][s]) <= 1e-9 * max(1.0, abs(nd["stat"][s])), (s, tot, nd["stat"][s])
            assert nd["split_score"] > 0
    leaves = t[t["feature"] < 0]
    assert leaves["num_examples"].sum() == n_rows
    assert len(t) <= 2 ** W["max_depth"] - 1


def test_full_size_properties_and_exact_root_histogram(data):
    bins, nb, na, y = data
    n = bins.shape[1]
    ds, gbt, trees, losses = _train(data, 3)
    for t in trees:
        _check_tree(t, n)
    assert len(trees[0]) == 255  # 10M informative rows fill depth 8
    assert losses[0] > losses[1] > losses[2]
    # sibling subtraction off: bit-identical trees and predictions (integer histograms => exact subtraction)
    pred = gbt.get_predictions()
    gbt.close(); ds.close()
    ds2, gbt2, trees2, losses2 = _train(data, 3, sibling_subtraction=0)
    assert [t.tobytes() for t in trees] == [t.tobytes() for t in trees2]
    assert losses == losses2
    assert pred.tobytes() == gbt2.get_predictions().tobytes()
    # root histogram of two features against numpy, bin for bin
    rng = np.random.default_rng(0)
    g = (rng.uniform(-1, 1, size=n) * 0.999).astype(np.float32)   # binomial: P = 1
    gbt2.debug_capture_histograms(True)
    gbt2.train_tree_on_gradients(g, np.full(n, 0.25, np.float32))
    root = gbt2.debug_level_histograms(0)
    assert root["layout"] == "root_sum" and root["g_pow2"] == 1.0 and root["num_slots"] == 1
    q = quantize_g(g, 0)
    for f in (0, 199):
        want_c = np.bincount(bins[f], minlength=256)
        want_s = np.bincount(bins[f], weights=q, minlength=256).astype(np.int64)
        np.testing.assert_array_equal(root["cnt"][0, f], want_c)
        np.testing.assert_array_equal(root["sum"][0, f].astype(np.int64), want_s)
        assert root["cnt"][0, f].sum() == n
    gbt2.close(); ds2.close()
