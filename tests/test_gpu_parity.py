"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on the same inputs.

Bar: bit-exact for integer / index work (features, thresholds, counts, row ids); 1e-5 relative on
split scores and 1e-5 absolute on leaf values (BASELINE.json north_star tolerance).
"""
import numpy as np
import pytest

import ydf_b200
from oracle import oracle as O
from tests.util import check_captured_levels, compare_trees, first_divergence, synth

pytestmark = pytest.mark.gpu


def _oracle_cfg(cfg):
    o = O.default_config()
    for k, _ in cfg._fields_:
        if k != "reserved":
            setattr(o, k, getattr(cfg, k))
    return o


def _mk(bins, nb, na, **kw):
    ds = ydf_b200.Dataset(bins, nb, na)
    cfg = ydf_b200.default_config(**kw)
    return ds, ydf_b200.Gbt(ds, cfg), cfg


def test_kat_train_tree_discretized_numerical():
    # learner/decision_tree/training_test.cc:193-267.  Newton leaf with h = 1, shrinkage 1, l2 0 is
    # the label mean, i.e. the plain regression leaf of the reference test.
    f1 = np.array([1, 2, 3, 4, 3, 4], dtype=np.uint8)
    f2 = np.array([1, 2, 1, 1, 2, 2], dtype=np.uint8)
    label = np.array([0, 0, 1, 1, 1.5, 1.5], dtype=np.float32)
    ds, gbt, cfg = _mk(np.stack([f1, f2]), [5, 3], [0, 0], loss=1, max_depth=8, min_examples=1,
                       shrinkage=1.0)
    t = gbt.train_tree_on_gradients(label)
    assert len(t) == 5
    root = t[0]
    assert root["feature"] == 0 and root["threshold_bin"] == 3
    assert root["num_examples"] == 6 and root["num_pos_examples"] == 4
    assert abs(root["split_score"] - 0.347222) < 1e-6
    assert abs(root["leaf_value"] - 0.833333) < 1e-6
    pos = t[root["pos_child"]]
    assert t[root["neg_child"]]["feature"] == -1 and abs(t[root["neg_child"]]["leaf_value"]) < 1e-7
    assert pos["feature"] == 1 and pos["threshold_bin"] == 2 and pos["num_pos_examples"] == 2
    assert abs(pos["split_score"] - 0.0625) < 1e-7
    assert abs(t[pos["pos_child"]]["leaf_value"] - 1.5) < 1e-6
    assert abs(t[pos["neg_child"]]["leaf_value"] - 1.0) < 1e-6


def test_kat_bucket_interpolation_and_hessian_score():
    # decision_tree_test.cc:2593-2626 (threshold 3 by interpolation over the empty bins 2,3)
    col = np.array([[0, 1, 4, 5]], dtype=np.uint8)
    ds, gbt, cfg = _mk(col, [6], [0], loss=1, max_depth=2, min_examples=1, shrinkage=1.0)
    t = gbt.train_tree_on_gradients(np.array([0, 0, 1, 1], np.float32))
    assert t[0]["threshold_bin"] == 3 and t[0]["num_pos_examples"] == 2 and t[0]["na_value"] == 0
    # decision_tree_test.cc:3052-3084: hessian gain, g = {-10,-10,10,10}, h = 1 -> score 400
    col = np.array([[0, 1, 2, 3]], dtype=np.uint8)
    ds, gbt, cfg = _mk(col, [4], [0], loss=1, max_depth=2, min_examples=1, use_hessian_gain=1)
    t = gbt.train_tree_on_gradients(np.array([-10, -10, 10, 10], np.float32))
    assert t[0]["threshold_bin"] == 2 and t[0]["num_pos_examples"] == 2
    assert abs(t[0]["split_score"] - 400.0) < 1e-3


def test_kat_split_examples_in_place():
    # training_test.cc:826-860
    ds = ydf_b200.Dataset(np.array([[0, 2, 1, 3]], np.uint8), [4], [0])
    pos, neg = ds.partition_rows([0, 1, 2, 3], 0, 2)
    assert pos.tolist() == [1, 3] and neg.tolist() == [0, 2]


@pytest.mark.parametrize("n", [1, 777, 4096, 70001])
def test_partition_rows_matches_oracle(n):
    rng = np.random.default_rng(n)
    col = rng.integers(0, 50, size=(1, max(n, 4))).astype(np.uint8)
    ds = ydf_b200.Dataset(col, [50], [0])
    rows = np.sort(rng.choice(col.shape[1], size=n, replace=False)).astype(np.uint32)
    pos, neg = ds.partition_rows(rows, 0, 23)
    opos, oneg = O.partition(col[0].astype(np.uint16), 23, False, rows)
    np.testing.assert_array_equal(pos, opos)
    np.testing.assert_array_equal(neg, oneg)
    assert np.all(np.diff(pos.astype(np.int64)) > 0) and np.all(np.diff(neg.astype(np.int64)) > 0)


@pytest.mark.parametrize("n", [5000, 70000])
def test_level_histograms_match_numpy(n):
    """Every level histogram of a grown tree equals the numpy restatement bin for bin (tests/test_gpu_hist_exact.py
    holds each layout to it)."""
    bins, nb, na, y = synth(n, 4, seed=3)
    ds, gbt, cfg = _mk(bins, nb, na, loss=1, max_depth=4)
    rng = np.random.default_rng(0)
    g = rng.normal(size=n).astype(np.float32)
    gbt.debug_capture_histograms(True)
    tree = gbt.train_tree_on_gradients(g)
    assert len(tree) > 7
    caps = check_captured_levels(gbt, tree, bins, ["root_sum", "packed", "packed"])
    assert caps[0]["cnt"][0].sum(axis=1).tolist() == [n] * 4


CASES = [
    dict(n=20000, f=8, kw=dict(loss=1, max_depth=6)),
    dict(n=20000, f=8, kw=dict(loss=1, max_depth=6, use_hessian_gain=1)),
    dict(n=50000, f=12, kw=dict(loss=0, max_depth=8, min_examples=5)),
    dict(n=50000, f=12, kw=dict(loss=0, max_depth=8, use_hessian_gain=1, l2_regularization=1.0)),
    dict(n=30011, f=5, kw=dict(loss=0, max_depth=5, min_examples=50, in_split_min_examples_check=0)),
    dict(n=9000, f=3, kw=dict(loss=1, max_depth=9, min_examples=1)),
    dict(n=9000, f=3, kw=dict(loss=1, max_depth=7, use_hessian_gain=1, l1_regularization=0.5,
                              hessian_split_score_subtract_parent=1)),
    # sparse deep levels: most nodes stop early, so levels 4+ have far fewer children than 2^(level+1)
    # (regression test: the partition kernel's accumulator layout must follow the launch's shared memory)
    dict(n=6000, f=4, kw=dict(loss=0, max_depth=9, min_examples=400)),
    dict(n=3000, f=2, kw=dict(loss=1, max_depth=9, min_examples=300)),
]


@pytest.mark.parametrize("case", CASES, ids=[str(i) for i in range(len(CASES))])
def test_tree_on_gradients_matches_oracle(case):
    """decision_tree::Train seam: same g/h in, same tree out."""
    n, f, kw = case["n"], case["f"], case["kw"]
    task = "binary" if kw["loss"] == 0 else "regression"
    bins, nb, na, y = synth(n, f, seed=11, task=task, bins=64)
    ds, gbt, cfg = _mk(bins, nb, na, **kw)
    rng = np.random.default_rng(5)
    if kw["loss"] == 0:
        p = 1 / (1 + np.exp(-rng.normal(size=n)))
        g = ((y == 2) - p).astype(np.float32)
        h = (p * (1 - p)).astype(np.float32)
    else:
        g = (y - y.mean() + 0.1 * rng.normal(size=n)).astype(np.float32)
        h = np.ones(n, np.float32)
    got = gbt.train_tree_on_gradients(g, h)
    want = O.train_tree(bins, nb, na, g, h, _oracle_cfg(cfg), num_threads=4)
    if kw.get("use_hessian_gain"):
        # The reference sums hessian-gain buckets in float32, sequentially: its own scores carry
        # ~1e-6..1e-4 relative rounding noise (amplified by l1 / small nodes).  Structure must match
        # the reference arithmetic exactly; scores are held to 1e-5 against the exact-bucket variant
        # of the oracle and to 2e-4 against the float one.
        errs = compare_trees(got, want, score_rtol=2e-4)
        assert not errs, errs[:10]
        O.set_hessian_buckets_double(True)
        try:
            want_exact = O.train_tree(bins, nb, na, g, h, _oracle_cfg(cfg), num_threads=4)
        finally:
            O.set_hessian_buckets_double(False)
        # subtract_parent turns the score into a small difference of large terms, which amplifies
        # the 24-bit gradient quantisation (DESIGN.md §3): 1e-4 there, 1e-5 otherwise.
        errs = compare_trees(got, want_exact, score_rtol=1e-5)
        assert not errs, errs[:10]
    else:
        errs = compare_trees(got, want)
        assert not errs, errs[:10]
    assert len(got) > 3


@pytest.mark.parametrize("sib", [0, 1])
@pytest.mark.parametrize("loss,hess", [(0, 0), (0, 1), (1, 0)])
def test_gbt_loop_matches_oracle(loss, hess, sib):
    """Whole boosting loop, free-running, first 20 trees + losses."""
    n, f, iters = 40000, 10, 20
    bins, nb, na, y = synth(n, f, seed=21, task="binary" if loss == 0 else "regression", bins=128)
    ds, gbt, cfg = _mk(bins, nb, na, loss=loss, use_hessian_gain=hess, max_depth=6, num_trees=iters,
                       sibling_subtraction=sib)
    gbt.set_labels(y)
    gbt.train(iters)
    ref = O.gbt_train(bins, nb, na, y, _oracle_cfg(cfg), iters, num_threads=4)
    assert abs(gbt.initial_prediction() - O.initial_prediction(loss, y)) == 0
    got_trees = [gbt.get_tree(i) for i in range(iters)]
    t, errs = first_divergence(got_trees, ref["trees"])
    assert t is None, (t, errs[:10])
    for i in range(iters):
        l, s = gbt.train_loss(i)
        assert abs(l - ref["loss"][i]) <= 1e-5 * abs(ref["loss"][i]), (i, l, ref["loss"][i])
        assert abs(s - ref["secondary"][i]) <= 1e-5
    np.testing.assert_allclose(gbt.get_predictions(), ref["predictions"], rtol=0, atol=2e-5)


def test_sibling_subtraction_is_bit_identical():
    bins, nb, na, y = synth(60000, 9, seed=33, bins=255)
    out = []
    for sib in (0, 1):
        ds, gbt, cfg = _mk(bins, nb, na, max_depth=7, num_trees=5, sibling_subtraction=sib)
        gbt.set_labels(y)
        gbt.train(5)
        out.append([gbt.get_tree(i).tobytes() for i in range(5)] + [gbt.get_predictions().tobytes()])
    assert out[0] == out[1]


def test_reruns_are_bit_identical():
    bins, nb, na, y = synth(50000, 6, seed=44)
    out = []
    for _ in range(2):
        ds, gbt, cfg = _mk(bins, nb, na, max_depth=6, num_trees=4)
        gbt.set_labels(y)
        gbt.train(4)
        out.append([gbt.get_tree(i).tobytes() for i in range(4)])
    assert out[0] == out[1]


def test_edge_cases():
    # fewer rows than min_examples: a single leaf (training.cc:4909)
    bins = np.array([[0, 1, 1, 0]], np.uint8)
    ds, gbt, cfg = _mk(bins, [2], [0], loss=1, min_examples=5, num_trees=2)
    gbt.set_labels(np.array([1, 2, 3, 4], np.float32))
    gbt.train(2)
    t = gbt.get_tree(0)
    assert len(t) == 1 and t[0]["feature"] == -1 and t[0]["num_examples"] == 4
    ref = O.gbt_train(bins, [2], [0], np.array([1, 2, 3, 4], np.float32), _oracle_cfg(cfg), 2)
    assert not compare_trees(t, ref["trees"][0])
    # max_depth = 1: root only
    ds, gbt, cfg = _mk(bins, [2], [0], loss=1, min_examples=1, max_depth=1, num_trees=1)
    gbt.set_labels(np.array([1, 2, 3, 4], np.float32))
    gbt.train(1)
    assert len(gbt.get_tree(0)) == 1
    # constant feature + constant gradients: no split has a positive score
    bins = np.zeros((2, 1000), np.uint8)
    bins[1] = np.arange(1000) % 7
    ds, gbt, cfg = _mk(bins, [4, 7], [0, 0], loss=1, min_examples=1, max_depth=4)
    t = gbt.train_tree_on_gradients(np.ones(1000, np.float32))
    assert len(t) == 1
    # error behaviour: labels outside {1,2}, wrong length
    ds, gbt, cfg = _mk(bins, [4, 7], [0, 0])
    with pytest.raises(ydf_b200.YggError):
        gbt.set_labels(np.zeros(1000, np.int32))
    with pytest.raises(ydf_b200.YggError):
        gbt.set_labels(np.ones(10, np.int32))
    with pytest.raises(ydf_b200.YggError):
        gbt.step()  # labels not set


def test_learner_end_to_end_small():
    bins_unused, nb, na, y = synth(1000, 2, seed=1)
    rng = np.random.default_rng(0)
    x0, x1 = rng.normal(size=20000).astype(np.float32), rng.normal(size=20000).astype(np.float32)
    lab = np.where(x0 + 0.5 * x1 + 0.2 * rng.normal(size=20000) > 0, "pos", "neg")
    data = {"x0": x0, "x1": x1, "y": lab}
    learner = ydf_b200.GradientBoostedTreesLearner(
        label="y", discretize_numerical_columns=True, validation_ratio=0.0, early_stopping="NONE",
        num_trees=20, max_depth=4)
    model = learner.train(data)
    ev = model.evaluate(data)
    assert model.num_trees() == 20 and ev["accuracy"] > 0.9
    assert model.training_logs[-1]["loss"] < model.training_logs[0]["loss"]


@pytest.mark.parametrize("label_data", [np.array([20, 20, 20, -10, -10]), np.array([-10, -10, 20, 20, 20]),
                                        np.array(["f", "f", "f", "x", "x"]), np.array(["x", "x", "x", "f", "f"])])
def test_reference_label_classes_order(label_data):
    """gradient_boosted_trees_learner_test.py:383-413 (test_label_classes_order_int / _str), with the
    discretized splitter: the classes are the sorted unique label values, as strings."""
    data = {"f": np.arange(5), "label": label_data}
    model = ydf_b200.GradientBoostedTreesLearner(label="label", min_examples=1, num_trees=1, validation_ratio=0.0,
                                                 discretize_numerical_columns=True).train(data)
    np.testing.assert_equal(np.array(model.label_classes()), np.unique(label_data).astype(str))
    assert model.num_trees() == 1


@pytest.mark.parametrize("mode,threads", [(2, 4), (1, 4)])
def test_tie_break_follows_the_candidate_shuffle(mode, threads):
    """a5: between features whose best splits have EQUAL float scores the reference takes the first in the order of
    its per-node std::shuffle of the candidates on the learner's mt19937 (GetCandidateAttributes,
    training.cc:4293-4306; one more word per feature job with the concurrent manager, :1658), nodes visited
    depth-first, positive child first.  Twin columns (exact copies) tie at every node they win; with
    cfg.candidate_shuffle the engine replays the stream on its finished trees and must name the same twin as the
    oracle, which follows the stream while it grows the tree (and reproduces the reference's golden models with it)."""
    base, nb, na, y = synth(40000, 6, seed=21, bins=64)
    # features 0..5, then copies of 0, 2 and 0 again: three-way and two-way ties
    bins = np.ascontiguousarray(np.concatenate([base, base[[0, 2, 0]]]))
    nb = np.concatenate([nb, nb[[0, 2, 0]]]).astype(np.int32)
    na = np.concatenate([na, na[[0, 2, 0]]]).astype(np.int32)
    ds, gbt, cfg = _mk(bins, nb, na, max_depth=6, num_trees=6, candidate_shuffle=mode, split_jobs_draw_seeds=int(threads > 1))
    gbt.set_labels(y)
    gbt.train(6)
    ref = O.gbt_train(bins, nb, na, y, _oracle_cfg(cfg), 6, num_threads=threads, shuffle_candidates=mode)
    renamed, unresolved = gbt.tie_stats()
    assert unresolved == 0 and renamed > 0
    n_twin_splits = 0
    for i in range(6):
        got, want = gbt.get_tree(i), ref["trees"][i]
        errs = compare_trees(got, want)
        assert not errs, (i, errs[:5])
        n_twin_splits += int(np.isin(want["feature"], [0, 2, 6, 7, 8]).sum())
    assert n_twin_splits > 10
    # without the replay the engine keeps the lowest index of every tie
    ds2, gbt2, _ = _mk(bins, nb, na, max_depth=6, num_trees=2)
    gbt2.set_labels(y)
    gbt2.train(2)
    assert not np.isin(gbt2.get_tree(0)["feature"], [6, 7, 8]).any()


@pytest.mark.parametrize("loss,shuffle", [(0, 0), (1, 0), (0, 2)])
def test_stochastic_gradient_boosting_matches_oracle(loss, shuffle):
    """N3: subsample < 1 (SampleTrainingExamples, gradient_boosted_trees.cc:2932-2956).  Every iteration draws one word
    of the learner's mt19937 per row BEFORE its tree (and after the candidate shuffles of the previous tree when those
    are replayed); the tree is trained on the drawn rows, every row gets the prediction update.  Same rows, same trees,
    same losses as the oracle, whose draw is pinned on the reference's gbt_adult_subsampling golden."""
    bins, nb, na, y = synth(50000, 10, seed=5, bins=64, task="binary" if loss == 0 else "regression")
    ds, gbt, cfg = _mk(bins, nb, na, loss=loss, max_depth=5, num_trees=8, subsample=0.6, candidate_shuffle=shuffle,
                       split_jobs_draw_seeds=int(shuffle != 0))
    gbt.set_labels(y)
    gbt.train(8)
    ref = O.gbt_train(bins, nb, na, y, _oracle_cfg(cfg), 8, num_threads=4, shuffle_candidates=shuffle)
    for i in range(8):
        got, want = gbt.get_tree(i), ref["trees"][i]
        assert got[0]["num_examples"] == want[0]["num_examples"] != 50000   # the root holds the drawn rows only
        errs = compare_trees(got, want)
        assert not errs, (i, errs[:5])
        assert abs(gbt.train_loss(i)[0] - ref["loss"][i]) <= 1e-5 * abs(ref["loss"][i])
    np.testing.assert_allclose(gbt.get_predictions(), ref["predictions"], rtol=0, atol=2e-5)


def test_exact_threshold_rule_matches_oracle():
    """N4: numerical columns with one bucket per distinct value carry their bucket VALUES (ygg_dataset_set_bucket_values);
    the engine then places the threshold like the reference's exact splitter — MidThreshold of the two values PRESENT in
    the node around the cut (splitter_accumulator.h:213-232, utils.h:103-109) — instead of the middle of the empty buckets:
    same partition of the training rows, but the bin threshold, na_value and float threshold of the reference.  Checked
    against the oracle's restatement of that rule (oracle_set_bucket_values), which reproduces the reference's default
    PYDF runs from scratch (tests/test_reference_replay.py)."""
    rng = np.random.default_rng(3)
    n = 30000
    # integer-valued columns with gaps (squares, multiples of 3, ...): deep nodes see few of the 40..120 distinct values
    raw = [np.round(rng.normal(size=n) * s) ** 2 for s in (4, 6, 8)] + [rng.integers(0, 40, size=n) * 3.0, rng.integers(0, 100, size=n) * 1.5 - 20]
    cols = [ydf_b200.dataspec.infer_column_lossless(f"x{j}", x.astype(np.float32)) for j, x in enumerate(raw)]
    assert all(c is not None for c in cols)
    bins = np.stack([c.encode(x.astype(np.float32)) for c, x in zip(cols, raw)])
    nb = np.array([c.num_bins for c in cols], np.int32)
    na = np.array([c.na_bin for c in cols], np.int32)
    y = ((raw[0] > 20) ^ (raw[3] > 60) ^ (rng.random(n) < 0.2)).astype(np.int32) + 1
    ds = ydf_b200.Dataset(bins, nb, na)
    for f, c in enumerate(cols):
        ds.set_bucket_values(f, c.bucket_values, c.mean)
    cfg = ydf_b200.default_config(max_depth=7, num_trees=5)
    gbt = ydf_b200.Gbt(ds, cfg)
    gbt.set_labels(y)
    gbt.train(5)
    O.set_bucket_values([c.bucket_values for c in cols], [c.mean for c in cols])
    try:
        ref = O.gbt_train(bins, nb, na, y, _oracle_cfg(cfg), 5, num_threads=2)
    finally:
        O.set_bucket_values(None)
    moved = 0
    for i in range(5):
        got, want = gbt.get_tree(i), ref["trees"][i]
        # (the label is mostly noise below depth 3: scores of 6e-5 on nodes of a few hundred rows, where the 24-bit
        # gradients show up at 1e-5 relative)
        errs = compare_trees(got, want)
        assert not errs, (i, errs[:5])
        sp = want["feature"] >= 0
        np.testing.assert_array_equal(got["threshold_value"][sp], want["threshold_value"][sp])   # the float threshold, bit for bit
        for nd in want[sp]:   # the rule moved the bin threshold off the interpolated one somewhere
            moved += int(cols[nd["feature"]].bucket_values[nd["threshold_bin"]] != nd["threshold_value"])
    assert moved > 0


@pytest.mark.parametrize("loss,max_nodes", [(0, 31), (1, 12), (0, -1)])
def test_best_first_global_growth_matches_oracle(loss, max_nodes):
    """N3: growing_strategy = BEST_FIRST_GLOBAL (GrowTreeBestFirstGlobal, training.cc:4499-4656): the candidate with the largest
    split_score * n is split next until max_num_nodes leaves exist; root depth 0.  The engine replays the reference's priority
    queue on its level-wise tree (a node's best split does not depend on when it is found); the oracle grows node by node like
    the reference, and reproduces the golden metrics of its LeafWiseGrow test."""
    bins, nb, na, y = synth(40000, 10, seed=8, bins=64, task="binary" if loss == 0 else "regression")
    ds, gbt, cfg = _mk(bins, nb, na, loss=loss, max_depth=6, num_trees=6, growing_strategy=1, max_num_nodes=max_nodes)
    gbt.set_labels(y)
    gbt.train(6)
    O.set_growing_strategy(True, max_nodes)
    try:
        ref = O.gbt_train(bins, nb, na, y, _oracle_cfg(cfg), 6, num_threads=2)
    finally:
        O.set_growing_strategy(False)
    for i in range(6):
        got, want = gbt.get_tree(i), ref["trees"][i]
        if max_nodes > 0:
            assert int((want["feature"] < 0).sum()) == max_nodes   # informative data: the leaf budget is used up
        assert int(want["depth"].max()) <= 7                      # root depth 0: one level more than the local growth
        errs = compare_trees(got, want)
        assert not errs, (i, errs[:5])
        assert abs(gbt.train_loss(i)[0] - ref["loss"][i]) <= 1e-5 * abs(ref["loss"][i])
    np.testing.assert_allclose(gbt.get_predictions(), ref["predictions"], rtol=0, atol=2e-5)


@pytest.mark.parametrize("depth,hessian", [(10, 0), (9, 1), (10, 1)])
def test_deep_trees_with_multi_pass_levels_match_oracle(depth, hessian):
    """max_depth 10 (9 with hessian histograms) needs more histogram slots at its last level(s) than shared memory holds:
    those levels are accumulated in several k_hist launches, each over a window of slots (rows of the other windows land in a
    dummy slot).  Same trees as the oracle, which has no depth limit (decision_tree.proto:30-32)."""
    bins, nb, na, y = synth(200000, 12, seed=13, bins=64)
    ds, gbt, cfg = _mk(bins, nb, na, max_depth=depth, num_trees=2, use_hessian_gain=hessian, min_examples=5)
    gbt.set_labels(y)
    gbt.train(2)
    O.set_hessian_buckets_double(bool(hessian))
    try:
        ref = O.gbt_train(bins, nb, na, y, _oracle_cfg(cfg), 2, num_threads=4)
    finally:
        O.set_hessian_buckets_double(False)
    for i in range(2):
        got, want = gbt.get_tree(i), ref["trees"][i]
        assert int(want["depth"].max()) == depth and len(want) > (1 << (depth - 1))
        errs = compare_trees(got, want)
        assert not errs, (i, errs[:5])
