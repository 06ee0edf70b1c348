"""Every histogram layout of the training loop held to an exact integer reference, level by level.

The engine's histograms are integer sums of 24-bit quantised gradients (DESIGN.md §3), so they can be restated
exactly: quantise the gradients as the engine intends (P = the smallest power of two strictly above max|g|), route
every row through the returned tree, and bincount q, hq and the counts per (slot, feature, bin).  Tree-level parity
cannot see a wrong bin unless it changes which split wins; this file compares the planes themselves, as the level
loop computed them (ygg_gbt_debug_capture_histograms), for every layout configure_launches can pick: the root's carry
plane, the packed words on both sides of their bound, the carry-detecting fallback with and without the hessian
planes, the windowed deep levels, sampled and weighted roots and row shards.  Each case asserts the layout it expects,
so that a case cannot silently stop covering the path it names.
"""
import numpy as np
import pytest

import ydf_b200
from oracle import oracle as O
from tests.util import Q_BIAS, Q_MAX, check_captured_levels as check_levels, synth

pytestmark = pytest.mark.gpu


def _gbt(bins, nb, na, ft=None, **kw):
    ds = ydf_b200.Dataset(bins, nb, na, feature_types=ft)
    gbt = ydf_b200.Gbt(ds, ydf_b200.default_config(**kw))
    gbt.debug_capture_histograms(True)
    return ds, gbt


def _grad(bins, seed, scale=1.0):
    """Regression gradients with structure on the first features, quantised to multiples of 2^-10 (so that any
    power-of-two scaling of them is exact in float32)."""
    rng = np.random.default_rng(seed)
    f = bins.shape[0]
    g = rng.normal(size=bins.shape[1])
    for j in range(min(f, 3)):
        g += (bins[j].astype(np.float64) / max(1, bins[j].max()) - 0.5) * (3 - j)
    return (np.rint(g * 1024) / 1024 * scale).astype(np.float32)


# ---- root: the low word + carry plane, counts from k_root_counts -------------------------------------------------

@pytest.mark.parametrize("n", [1, 3, 4097, 8191, 8192, 8193, 127 * 8192 + 1])
def test_root_sum_row_count_edges(n, monkeypatch):
    if n == 127 * 8192 + 1:
        monkeypatch.setenv("YGG_HIST_CHUNK_BLOCKS", "127")   # two work items, the second holds one row
    bins, nb, na, _ = synth(max(n, 8), 3, seed=n % 1000, bins=64)
    bins = np.ascontiguousarray(bins[:, :n])
    ds, gbt = _gbt(bins, nb, na, loss=1, max_depth=2, min_examples=1)
    g = _grad(bins, n)
    tree = gbt.train_tree_on_gradients(g)
    caps = check_levels(gbt, tree, bins, ["root_sum"])
    assert caps[0]["num_slots"] == 1 and int(caps[0]["cnt"][0, 0].sum()) == n
    if n == 127 * 8192 + 1:
        assert caps[0]["chunk_blocks"] == 127


# ---- packed words: partial feature groups, edge bin counts, categorical columns ----------------------------------

def _packed_case(F):
    """F columns of 256, 2 and 255 bins, the last bin of each populated, every 4th column categorical: one tree of
    depth 5 on them.  Returns (bins, nbs, tree, captures of its 4 levels, which must be root_sum, packed, packed,
    packed)."""
    n = 50000
    rng = np.random.default_rng(F)
    nbs = [(256, 2, 255)[j % 3] for j in range(F)]
    bins = np.stack([rng.integers(0, k, size=n) for k in nbs]).astype(np.uint8)
    for j, k in enumerate(nbs):
        bins[j, rng.choice(n, 50, replace=False)] = k - 1     # the last bin (255 for 256 bins) is populated
    ft = np.array([1 if (j % 4 == 3) else 0 for j in range(F)], np.int32)   # every 4th column categorical
    ds, gbt = _gbt(bins, np.array(nbs, np.int32), np.zeros(F, np.int32), ft=ft, loss=1, max_depth=5)
    g = _grad(bins, F)
    tree = gbt.train_tree_on_gradients(g)
    caps = check_levels(gbt, tree, bins, ["root_sum"] + ["packed"] * 3)
    return bins, nbs, tree, caps


@pytest.mark.parametrize("F", [1, 7, 9])
def test_packed_feature_groups_and_bins(F):
    bins, nbs, tree, caps = _packed_case(F)
    assert len(tree) > 7
    for j, k in enumerate(nbs):
        assert caps[0]["cnt"][0, j, k - 1] >= 50


def test_retired_switches_are_ignored(monkeypatch):
    """The layout of every level follows from the configuration alone: the environment switches that once selected
    the feature-lane kernel (YGG_HIST2) or turned the root's and the packed layouts off change nothing."""
    def run():
        _, _, tree, caps = _packed_case(9)
        return tree.tobytes(), [(c["chunk_blocks"], c["features_per_item"], c["smem_slots"]) for c in caps]

    base = run()
    monkeypatch.setenv("YGG_HIST2", "1")
    monkeypatch.setenv("YGG_HIST_ROOT_SUM", "0")
    monkeypatch.setenv("YGG_HIST_PACKED", "0")
    assert run() == base


@pytest.mark.parametrize("heavy", [8191, 8192])
def test_packed_bound_both_sides(heavy):
    """One 8192-row block: a bin that holds 8191 rows keeps the packed words (13-bit count), 8192 rows fall back."""
    n = 8192
    rng = np.random.default_rng(heavy)
    col = np.zeros(n, np.uint8)
    col[rng.choice(n, n - heavy, replace=False)] = 1
    bins = np.stack([rng.integers(0, 64, size=n).astype(np.uint8), col, rng.integers(0, 16, size=n).astype(np.uint8)])
    ds, gbt = _gbt(bins, np.array([64, 2, 16], np.int32), np.zeros(3, np.int32), loss=1, max_depth=4)
    tree = gbt.train_tree_on_gradients(_grad(bins, heavy))
    layout = "packed" if heavy == 8191 else "shared"
    check_levels(gbt, tree, bins, ["root_sum", layout, layout])


def test_shared_fallback_at_large_n():
    """4,194,304 rows: the packed bound is checked on 8-block sub-chunks; a balanced binary column puts ~32768 rows
    of a sub-chunk in one bin, so every level below the root falls back to the carry-detecting layout."""
    n = 1 << 22
    rng = np.random.default_rng(4)
    bins = np.stack([rng.integers(0, 2, size=n), rng.integers(0, 64, size=n)]).astype(np.uint8)
    ds, gbt = _gbt(bins, np.array([2, 64], np.int32), np.zeros(2, np.int32), loss=1, max_depth=4)
    tree = gbt.train_tree_on_gradients(_grad(bins, 4))
    check_levels(gbt, tree, bins, ["root_sum", "shared", "shared"])


def test_carry_field_near_its_limit(monkeypatch):
    """127-block work items of rows whose q is 2^24 - 1: a level-1 bin of the shared layout receives 1,040,384 such
    rows, ~4063 carries in its 12-bit field (limit 4095); the root's carry plane gets the same rows."""
    monkeypatch.setenv("YGG_HIST_CHUNK_BLOCKS", "127")
    half = 127 * 8192
    n = 2 * half
    rows = np.arange(n)
    bins = np.stack([(rows >= half).astype(np.uint8), np.zeros(n, np.uint8),
                     (rows % 64).astype(np.uint8)])
    g = np.where(rows < half, np.float32(1 - 2.0 ** -24), np.float32(-(1 - 2.0 ** -24))).astype(np.float32)
    ds, gbt = _gbt(bins, np.array([2, 2, 64], np.int32), np.zeros(3, np.int32), loss=1, max_depth=3,
                   sibling_subtraction=0)
    tree = gbt.train_tree_on_gradients(g)
    assert tree[0]["feature"] == 0 and tree[0]["num_pos_examples"] == half
    caps = check_levels(gbt, tree, bins, ["root_sum", "shared"], g_pow2=1.0)
    for c in caps:
        assert c["chunk_blocks"] == 127
    top = int(caps[1]["sum"][:, 1, 0].max())
    assert top == half * Q_MAX and top >> 32 >= 4060


# ---- hessian / weight planes -------------------------------------------------------------------------------------

def test_hessian_planes_quarter():
    """h = 1/4 on every row with h_pow2 = 1/4: every hq is 2^24, so the hessian low word carries once per 256 rows."""
    n = 30000
    bins, nb, na, y = synth(n, 6, seed=8, bins=64)
    ds, gbt = _gbt(bins, nb, na, loss=0, max_depth=5, use_hessian_gain=1)
    rng = np.random.default_rng(8)
    g = (np.where(y == 2, 0.5, -0.5) * rng.random(n)).astype(np.float32)
    tree = gbt.train_tree_on_gradients(g, np.full(n, 0.25, np.float32))
    caps = check_levels(gbt, tree, bins, ["shared_hess"] * 4, g_pow2=1.0, h2_pow2=0.25)
    assert np.array_equal(caps[0]["hsum"], caps[0]["cnt"].astype(np.uint64) << np.uint64(24))


def test_balanced_binomial_iteration_zero_hessian():
    """Balanced labels: iteration 0 has p = 1/2 on every row, h = 1/4 exactly."""
    n = 20000
    bins, nb, na, y = synth(n, 5, seed=9, bins=64)
    y = np.where(np.arange(n) % 2 == 0, 1, 2).astype(np.int32)
    ds, gbt = _gbt(bins, nb, na, loss=0, max_depth=4, use_hessian_gain=1, num_trees=1)
    gbt.set_labels(y)
    gbt.train(1)
    caps = check_levels(gbt, gbt.get_tree(0), bins, ["shared_hess"] * 3, g_pow2=1.0, h2_pow2=0.25)
    assert np.all(caps[0]["h2"] == 0.25)


# ---- windowed deep levels ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("depth,hess", [(10, 0), (9, 1), (10, 1)])
def test_multi_window_levels(depth, hess):
    n = 120000
    bins, nb, na, y = synth(n, 5, seed=depth + hess, bins=64)
    kw = dict(loss=1, max_depth=depth, min_examples=2) if not hess else dict(loss=0, max_depth=depth, use_hessian_gain=1,
                                                                             min_examples=2)
    ds, gbt = _gbt(bins, nb, na, **kw)
    rng = np.random.default_rng(depth)
    g = _grad(bins, depth)
    if hess:
        p = (1 / (1 + np.exp(-rng.normal(size=n)))).astype(np.float32)
        g = ((y == 2) - p).astype(np.float32)
        tree = gbt.train_tree_on_gradients(g, (p * (1 - p)).astype(np.float32))
    else:
        tree = gbt.train_tree_on_gradients(g)
    caps = check_levels(gbt, tree, bins, [None] * (depth - 1), g_pow2=1.0 if hess else None)
    multi = [c for c in caps if c["layout"].endswith("_multi")]
    assert multi and all(c["passes"] > 1 for c in multi)
    assert multi[-1]["layout"] == ("shared_hess_multi" if hess else "packed_multi")
    assert max(c["num_slots"] for c in multi) > multi[-1]["smem_slots"]   # the windows really split the slots


# ---- sampled roots, GOSS, example weights --------------------------------------------------------------------------

@pytest.mark.parametrize("mode", ["subsample", "goss", "weights"])
def test_sampled_and_weighted_iterations(mode):
    n = 40000
    bins, nb, na, y = synth(n, 6, seed=12, bins=128)
    kw = dict(loss=0, max_depth=5, num_trees=2)
    if mode == "subsample":
        kw["subsample"] = 0.6
    elif mode == "goss":
        kw.update(goss_alpha=0.2, goss_beta=0.1)
    ds, gbt = _gbt(bins, nb, na, **kw)
    if mode == "weights":
        w = np.random.default_rng(3).uniform(0.1, 3.0, size=n).astype(np.float32)
        gbt.set_weights(w)
    gbt.set_labels(y)
    gbt.train(2)
    hist_hess = mode != "subsample"
    layouts = (["shared_hess"] * 4) if hist_hess else (["packed"] * 4)
    caps = check_levels(gbt, gbt.get_tree(1), bins, layouts, g_pow2=1.0 if mode == "subsample" else None)
    sel = caps[0]["selected"]
    if mode == "weights":
        assert sel.all() and np.array_equal(caps[0]["h2"], w)
        assert caps[0]["h2_pow2"] == 4.0
    else:
        assert 0 < sel.sum() < n


# ---- row shards ----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("scatter", [0, 1])
def test_row_shard_planes_sum_to_single_rank(scatter):
    from tests.test_gpu_sharding import FakeComm, _run_ranks
    n, f, world = 30000, 5, 2
    bins, nb, na, y = synth(n, f, seed=31, task="regression", bins=64)
    kw = dict(loss=1, max_depth=5, num_trees=1)
    ds, gbt = _gbt(bins, nb, na, **kw)
    gbt.set_labels(y)
    gbt.train(1)
    tree = gbt.get_tree(0)
    single = check_levels(gbt, tree, bins, ["root_sum"] + [None] * 3)
    init = gbt.initial_prediction()
    comm = FakeComm(world)

    def rank_main(r):
        r0, r1 = (n * r) // world, (n * (r + 1)) // world
        d = ydf_b200.Dataset(bins[:, r0:r1], nb, na)
        gb = ydf_b200.Gbt(d, ydf_b200.default_config(**kw))
        gb.debug_capture_histograms(True)
        gb.set_labels(y[r0:r1])
        if scatter:
            gb.set_row_shard_scatter(r, world, n, init, allreduce=comm.allreduce(r), reducescatter=comm.reducescatter(r),
                                     allgather=comm.allgather(r))
        else:
            gb.set_row_shard(r, world, n, init, comm.allreduce(r))
        gb.train(1)
        assert gb.get_tree(0).tobytes() == tree.tobytes()
        return [gb.debug_level_histograms(l) for l in range(4)]

    res = _run_ranks(world, rank_main, comm)
    for l in range(4):
        for k in ("sum", "cnt"):
            tot = sum(res[r][l][k].astype(np.int64) for r in range(world))
            assert np.array_equal(tot, single[l][k].astype(np.int64)), (l, k)
        assert all(np.array_equal(res[r][l]["slot_node"], single[l]["slot_node"]) for r in range(world))


# ---- gradient = +P -------------------------------------------------------------------------------------------------

def test_gradient_equal_to_a_power_of_two():
    """max|g| = 2^-1 exactly: P must be 2^0, or the row with g = +P is clamped one unit short."""
    n = 20000
    bins, nb, na, _ = synth(n, 4, seed=41, bins=64)
    rng = np.random.default_rng(41)
    g = (rng.integers(-64, 65, size=n) / 128.0).astype(np.float32)   # multiples of 2^-7 in [-1/2, 1/2]
    g[0] = 0.5
    ds, gbt = _gbt(bins, nb, na, loss=1, max_depth=4)
    tree = gbt.train_tree_on_gradients(g)
    check_levels(gbt, tree, bins, ["root_sum", "packed", "packed"], g_pow2=1.0)


def test_squared_error_on_balanced_labels():
    """Squared error on balanced 0/1 labels: iteration 0 has residuals of exactly +-1/2."""
    n = 20000
    bins, nb, na, _ = synth(n, 4, seed=42, bins=64)
    y = (np.arange(n) % 2).astype(np.float32)
    ds, gbt = _gbt(bins, nb, na, loss=1, max_depth=4, num_trees=1)
    gbt.set_labels(y)
    gbt.train(1)
    caps = check_levels(gbt, gbt.get_tree(0), bins, ["root_sum", "packed", "packed"], g_pow2=1.0)
    assert np.abs(caps[0]["g"]).max() == 0.5
    # the residuals +-1/2 cancel exactly, and so must their codes 2^23 +- 2^22: every feature's root histogram sums to
    # n * 2^23 (with P = 1/2, +1/2 would be clamped to 2^24 - 1 and the sum would fall n / 2 short)
    assert np.all(caps[0]["sum"].astype(np.int64).sum(axis=2) == n * Q_BIAS)


# ---- gradient scale sweep ------------------------------------------------------------------------------------------

def _oracle_cfg(cfg):
    o = O.default_config()
    for k, _ in cfg._fields_:
        if k != "reserved":
            setattr(o, k, getattr(cfg, k))
    return o


STRUCT = ("feature", "threshold_bin", "na_value", "depth", "neg_child", "pos_child", "num_examples", "num_pos_examples",
          "condition_type")


@pytest.fixture(scope="module")
def sweep_data():
    n = 30000
    bins, nb, na, _ = synth(n, 6, seed=51, bins=64)
    ds, gbt = _gbt(bins, nb, na, loss=1, max_depth=5)
    g = _grad(bins, 51)
    tree0 = gbt.train_tree_on_gradients(g)
    caps0 = check_levels(gbt, tree0, bins, ["root_sum"] + ["packed"] * 3)
    return bins, nb, na, g, ds, gbt, tree0, caps0


@pytest.mark.parametrize("k", [-110, -100, -60, -52, 0, 30, 50])
def test_gradient_scale_sweep(k, sweep_data):
    """g * 2^k: the integer planes and the tree structure do not move; leaves and stat[0] scale by 2^k, scores and
    stat[1] by 2^2k, against the oracle on the same scaled inputs (where float g^2 underflows, both take the float
    product).  Split scores are floats (NodeCondition.split_score): once they scale below the smallest normal float
    (k <= -100 here) neither the reference nor the engine finds a split, and only the root's planes are compared."""
    bins, nb, na, g, ds, gbt, tree0, caps0 = sweep_data
    gk = (g.astype(np.float64) * 2.0 ** k).astype(np.float32)
    assert np.array_equal(gk.astype(np.float64) * 2.0 ** -k, g.astype(np.float64))   # the scaling is exact
    tree = gbt.train_tree_on_gradients(gk)
    caps = check_levels(gbt, tree, bins, [c["layout"] for c in caps0])
    assert caps[0]["g_pow2"] == caps0[0]["g_pow2"] * 2.0 ** k
    scores0 = tree0["split_score"][tree0["feature"] >= 0].astype(np.float64)
    in_range = scores0.min() * 2.0 ** (2 * k) >= np.finfo(np.float32).tiny
    assert in_range or k <= -100
    for a, b in zip(caps if in_range else caps[:1], caps0):
        for key in ("sum", "cnt", "slot_node"):
            assert np.array_equal(a[key], b[key]), (k, key)
    if in_range:
        for key in STRUCT:
            assert np.array_equal(tree[key], tree0[key]), (k, key)
    else:
        assert len(tree) == 1
    want = O.train_tree(bins, nb, na, gk, np.ones(len(gk), np.float32), _oracle_cfg(gbt.cfg), num_threads=4)
    for key in STRUCT:
        assert np.array_equal(tree[key], want[key]), (k, key)
    s1, s2 = 2.0 ** k, 2.0 ** (2 * k)
    tiny = 2.0 ** -149
    n_ex = tree["num_examples"].astype(np.float64)
    for i in range(len(tree)):
        got, ref = tree[i], want[i]
        assert abs(float(got["split_score"]) - float(ref["split_score"])) <= 1e-5 * abs(float(ref["split_score"])) + tiny, (k, i)
        assert abs(float(got["leaf_value"]) - float(ref["leaf_value"])) <= 1e-5 * s1 + tiny, (k, i)
        assert abs(got["stat"][0] - ref["stat"][0]) <= max(1e-6 * abs(ref["stat"][0]), 2e-8 * n_ex[i] * s1), (k, i)
        assert abs(got["stat"][1] - ref["stat"][1]) <= max(1e-6 * abs(ref["stat"][1]), 2e-8 * n_ex[i] * s2, 1e-300), (k, i)
        assert got["stat"][2] == ref["stat"][2], (k, i)
