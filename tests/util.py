"""Shared helpers for the parity tests: synthetic data (SURVEY.md §8d generator), tree comparison."""
import math

import numpy as np


def synth(n, f, seed=1234, informative=None, task="binary", bins=255, sample=100000):
    """X ~ N(0,1) [f, n]; y = 1[sum_j w_j x_j + 0.5 x0 x1 + 0.3 sin(3 x2) + eps > 0] (binary) or the
    margin itself (regression).  Returns (bins uint8 [f, n], num_bins, na_bin, labels)."""
    import ydf_b200
    rng = np.random.default_rng(seed)
    informative = informative or min(10, f)
    w = rng.normal(size=informative)
    margin = np.zeros(n, dtype=np.float64)
    out = np.empty((f, n), dtype=np.uint8)
    nb, na = [], []
    cols = {}
    for j in range(f):
        x = rng.normal(size=n).astype(np.float32)
        if j < informative:
            margin += w[j] * x
        if j < 3:
            cols[j] = x
        b, mean = ydf_b200.discretize_boundaries(x[:sample], bins, 3)
        nbin = len(b) + 1
        nab = int(np.searchsorted(b, np.float32(mean), side="right"))
        out[j] = ydf_b200.discretize_encode(x, b, nab)
        nb.append(nbin)
        na.append(nab)
    if f >= 3:
        margin += 0.5 * cols[0] * cols[1] + 0.3 * np.sin(3 * cols[2])
    margin += rng.normal(scale=0.5, size=n)
    if task == "binary":
        y = (margin > 0).astype(np.int32) + 1
    else:
        y = margin.astype(np.float32)
    return out, np.array(nb, np.int32), np.array(na, np.int32), y


def synth_mixed(n, f_num, cat_sizes, seed=77, task="binary", bins=64):
    """Numerical features as in synth() plus one categorical feature per entry of `cat_sizes`
    (number_of_unique_values incl. index 0 = <OOD>; skewed frequencies, some categories empty, a
    per-category effect on the margin).  Returns (bins, num_bins, na_bin, feature_type, labels)."""
    b, nb, na, _ = synth(n, f_num, seed=seed, task="regression", bins=bins)
    rng = np.random.default_rng(seed + 1)
    margin = np.zeros(n)
    for j in range(min(f_num, 4)):
        margin += rng.normal() * (b[j].astype(np.float64) / nb[j] - 0.5) * 3
    cols, cnb, cna = [], [], []
    for k in cat_sizes:
        p = 1.0 / np.arange(1, k + 1) ** 1.1
        p[0] = p[-1] * 0.5                      # <OOD> is rare
        if k > 8:
            p[rng.choice(np.arange(1, k), size=max(1, k // 10), replace=False)] = 0.0  # unseen categories
        p /= p.sum()
        c = rng.choice(k, size=n, p=p).astype(np.uint8)
        effect = rng.normal(size=k)
        effect[rng.random(k) < 0.3] = 0.0
        margin += effect[c]
        cols.append(c)
        cnb.append(k)
        cna.append(int(np.bincount(c, minlength=k)[1:].argmax()) + 1 if k > 1 else 0)
    margin += rng.normal(scale=0.7, size=n)
    allb = np.concatenate([b, np.stack(cols)]) if cols else b
    ft = np.array([0] * f_num + [1] * len(cat_sizes), np.int32)
    # interleave so that shards / candidate order mix both kinds
    order = rng.permutation(len(ft))
    y = (margin > np.median(margin)).astype(np.int32) + 1 if task == "binary" else margin.astype(np.float32)
    return (np.ascontiguousarray(allb[order]), np.concatenate([nb, cnb]).astype(np.int32)[order],
            np.concatenate([na, cna]).astype(np.int32)[order], ft[order], y)


def compare_trees(a, b, score_rtol=1e-5, leaf_atol=1e-5, stat_rtol=1e-6, stat_atol_per_row=2e-8):
    """a, b: node arrays (pre-order).  Returns a list of mismatch strings (empty = parity)."""
    errs = []
    if len(a) != len(b):
        return [f"node count {len(a)} != {len(b)}"]
    for i, (x, y) in enumerate(zip(a, b)):
        for k in ("feature", "threshold_bin", "na_value", "depth", "neg_child", "pos_child",
                  "num_examples", "num_pos_examples", "condition_type"):
            if x[k] != y[k]:
                errs.append(f"node {i}: {k} {x[k]} != {y[k]}")
        if not np.array_equal(x["cat_mask"], y["cat_mask"]):
            errs.append(f"node {i}: cat_mask {x['cat_mask']} != {y['cat_mask']}")
        if abs(float(x["split_score"]) - float(y["split_score"])) > score_rtol * max(1e-30, abs(float(y["split_score"]))):
            errs.append(f"node {i}: split_score {x['split_score']} vs {y['split_score']}")
        if abs(float(x["leaf_value"]) - float(y["leaf_value"])) > leaf_atol:
            errs.append(f"node {i}: leaf_value {x['leaf_value']} vs {y['leaf_value']}")
        for s in range(3):
            d = abs(float(x["stat"][s]) - float(y["stat"][s]))
            # sums over n rows: 1e-6 relative, or 2e-8 per row (fixed-point resolution / 1-ulp
            # differences of the per-row gradients between devices)
            if d > max(stat_rtol * abs(float(y["stat"][s])), stat_atol_per_row * float(y["num_examples"]), 1e-9):
                errs.append(f"node {i}: stat[{s}] {x['stat'][s]} vs {y['stat'][s]}")
    return errs


def prune_noise_splits(tree, eps):
    """Collapses every split with split_score <= eps into a leaf (pre-order array in, pre-order array
    out).  On a pure node (constant gradients) the reference's double-precision variance arithmetic
    leaves +-1e-16 of rounding noise, so whether it still "splits" such a node into children with
    identical leaf values depends on the accumulation order; the GPU's integer sums give exactly 0
    (DESIGN.md §6).  Predictions are unaffected either way."""
    out = []

    def walk(i):
        nd = tree[i].copy()
        me = len(out)
        out.append(nd)
        if nd["feature"] >= 0 and nd["split_score"] <= eps:
            for k, v in (("feature", -1), ("threshold_bin", 0), ("na_value", 0), ("split_score", 0.0),
                         ("num_pos_examples", 0), ("condition_type", 0), ("neg_child", -1), ("pos_child", -1)):
                nd[k] = v
            nd["cat_mask"] = 0
        elif nd["feature"] >= 0:
            nd["neg_child"] = len(out)
            walk(int(tree[i]["neg_child"]))
            nd["pos_child"] = len(out)
            walk(int(tree[i]["pos_child"]))
        out[me] = nd

    walk(0)
    return np.array(out, dtype=tree.dtype)


def drop_absent_categories(tree, bins):
    """Clears, in every categorical split, the mask bits of categories that no row of the node carries.
    Such categories have empty buckets (sort key 0); they can only change sides when a NON-empty bucket's key
    is exactly 0 as well (gradient sums that cancel exactly, e.g. iteration 0 of the multinomial loss with
    p = 1/K), which the 24-bit quantised sums do not reproduce bit for bit (DESIGN.md §6).  Training rows are
    unaffected by where absent categories go."""
    out = tree.copy()

    def walk(i, rows):
        nd = out[i]
        if nd["feature"] < 0:
            return
        b = bins[nd["feature"], rows].astype(np.int64)
        if nd["condition_type"] == 1:
            present = np.zeros(8, np.uint32)
            for c in np.unique(b):
                present[c >> 5] |= np.uint32(1) << np.uint32(c & 31)
            out[i]["cat_mask"] = nd["cat_mask"] & present
            go = ((nd["cat_mask"][b >> 5] >> (b & 31).astype(np.uint32)) & 1) != 0
        else:
            go = b >= nd["threshold_bin"]
        walk(int(nd["neg_child"]), rows[~go])
        walk(int(nd["pos_child"]), rows[go])

    walk(0, np.arange(bins.shape[1]))
    return out


def first_divergence(trees_a, trees_b, prune_noise=None, present_in=None, **kw):
    for t, (a, b) in enumerate(zip(trees_a, trees_b)):
        if prune_noise is not None:
            a, b = prune_noise_splits(a, prune_noise), prune_noise_splits(b, prune_noise)
        if present_in is not None:
            a, b = drop_absent_categories(a, present_in), drop_absent_categories(b, present_in)
        e = compare_trees(a, b, **kw)
        if e:
            return t, e
    return None, []


def predict_raw(trees, initial_prediction, bins):
    """Sum of the leaves reached by every column of `bins` ([F, n] bucket / dictionary codes) — numpy walk of
    ydf_b200.NODE_DTYPE trees (DiscretizedHigher and Contains conditions)."""
    n = bins.shape[1]
    rows = np.arange(n)
    raw = np.full(n, initial_prediction, np.float32)
    for t in trees:
        node = np.zeros(n, np.int64)
        while True:
            f = t["feature"][node]
            act = np.nonzero(f >= 0)[0]
            if len(act) == 0:
                break
            nd = node[act]
            v = bins[f[act], rows[act]].astype(np.int64)
            in_set = ((t["cat_mask"][nd, v >> 5] >> (v & 31).astype(np.uint32)) & 1) != 0
            go = np.where(t["condition_type"][nd] == 1, in_set, v >= t["threshold_bin"][nd])
            node[act] = np.where(go, t["pos_child"][nd], t["neg_child"][nd])
        raw += t["leaf_value"][node]
    return raw


# ---- exact restatement of the level histograms (ygg_gbt_debug_level_histograms) --------------------------------

Q_BIAS = 1 << 23
Q_MAX = (1 << 24) - 1


def g_pow2_exp(g):
    """e of P = 2^e, the smallest power of two strictly above max|g| (P = 1 when every g is 0)."""
    m = float(np.max(np.abs(g.astype(np.float64)))) if len(g) else 0.0
    return 0 if m == 0.0 else math.frexp(m)[1]   # m = f * 2^e, 0.5 <= f < 1: 2^(e-1) <= m < 2^e


def quantize_g(g, e):
    """q = clip(rint(g * 2^(23-e)) + 2^23, 0, 2^24 - 1), exact in float64 (a power-of-two scale of a float32)."""
    t = np.rint(g.astype(np.float32).astype(np.float64) * 2.0 ** (23 - e)) + Q_BIAS
    return np.clip(t, 0, Q_MAX).astype(np.int64)


def quantize_h2(v, h2_pow2):
    """The second plane (hessians or weights): [0, 2^24] inclusive."""
    return np.minimum(np.rint(v.astype(np.float32).astype(np.float64) * (2.0 ** 24 / float(h2_pow2))), 1 << 24).astype(np.int64)


def node_per_level(tree, bins, levels):
    """[levels, n]: the node (index in `tree`) each row sits in at every level, -1 once it has reached a leaf."""
    n = bins.shape[1]
    rows = np.arange(n)
    node = np.zeros(n, np.int64)
    alive = np.ones(n, bool)
    out = np.full((levels, n), -1, np.int64)
    for l in range(levels):
        out[l, alive] = node[alive]
        f = tree["feature"][node]
        alive &= f >= 0
        act = np.nonzero(alive)[0]
        nd = node[act]
        v = bins[f[act], rows[act]].astype(np.int64)
        in_set = ((tree["cat_mask"][nd, v >> 5] >> (v & 31).astype(np.uint32)) & 1) != 0
        go = np.where(tree["condition_type"][nd] == 1, in_set, v >= tree["threshold_bin"][nd])
        node[act] = np.where(go, tree["pos_child"][nd], tree["neg_child"][nd])
    return out


def expected_planes(cap, tree, bins, node_at_level, q, hq=None):
    """int64 [slot, feature, 256] sums of q, hq and counts over the rows of every slot's node (sampled rows only)."""
    S, F = cap["num_slots"], cap["num_features"]
    slot_of_node = np.full(len(tree), -1, np.int64)
    slot_of_node[cap["slot_node"]] = np.arange(S)
    rs = np.where(node_at_level >= 0, slot_of_node[np.maximum(node_at_level, 0)], -1)
    rs[~cap["selected"]] = -1
    m = rs >= 0
    out = {k: np.zeros((S, F, 256), np.int64) for k in ("sum", "hsum", "cnt")}
    for fl in range(F):
        key = rs[m] * 256 + bins[cap["feature_begin"] + fl][m].astype(np.int64)
        out["cnt"][:, fl] = np.bincount(key, minlength=S * 256).reshape(S, 256)
        # float64 bincount weights are exact here: every sum stays below 2^53
        out["sum"][:, fl] = np.bincount(key, weights=q[m], minlength=S * 256).reshape(S, 256).astype(np.int64)
        if hq is not None:
            out["hsum"][:, fl] = np.bincount(key, weights=hq[m], minlength=S * 256).reshape(S, 256).astype(np.int64)
    return out


def _first_diff(name, got, want):
    bad = np.argwhere(got.astype(np.int64) != want)
    s, f, b = bad[0]
    return (f"{name}: {len(bad)} bins differ, first at slot {s} feature {f} bin {b}: "
            f"{int(got[s, f, b])} != {int(want[s, f, b])}")


def check_captured_levels(gbt, tree, bins, layouts, g_pow2=None, h2_pow2=None):
    """Compares every level of the last tree `gbt` grew with the histogram capture on (Gbt.debug_capture_histograms)
    with the numpy restatement, for equality.  layouts[l] = the layout level l must have run with (None: not asserted);
    there must be exactly len(layouts) levels.  g_pow2 / h2_pow2: the scales the planes must have used (default for
    g_pow2: the smallest power of two strictly above max|g|).  Returns the captures."""
    import ydf_b200
    caps = [gbt.debug_level_histograms(l) for l in range(len(layouts))]
    try:
        gbt.debug_level_histograms(len(layouts))
        raise AssertionError(f"more than {len(layouts)} histogram levels were captured")
    except ydf_b200.YggError:
        pass
    c0 = caps[0]
    # P: the smallest power of two above max|g| over all rows of the iteration (sampled or not); the binomial loss
    # without weights has |g| <= 1 and uses P = 1: the caller passes g_pow2 = 1
    want_p = 2.0 ** g_pow2_exp(c0["g"]) if g_pow2 is None else g_pow2
    assert c0["g_pow2"] == want_p, (c0["g_pow2"], want_p)
    if h2_pow2 is not None:
        assert c0["h2_pow2"] == h2_pow2
    q = quantize_g(c0["g"], int(round(math.log2(c0["g_pow2"]))))
    hq = quantize_h2(c0["h2"], c0["h2_pow2"]) if c0["has_hsum"] else None
    at = node_per_level(tree, bins, len(layouts))
    for l, cap in enumerate(caps):
        if layouts[l] is not None:
            assert cap["layout"] == layouts[l], (l, cap["layout"], layouts[l], cap)
        want = expected_planes(cap, tree, bins, at[l], q, hq)
        assert np.array_equal(cap["cnt"], want["cnt"]), f"level {l}: " + _first_diff("cnt", cap["cnt"], want["cnt"])
        assert np.array_equal(cap["sum"], want["sum"]), f"level {l}: " + _first_diff("sum", cap["sum"], want["sum"])
        if hq is not None:
            assert np.array_equal(cap["hsum"], want["hsum"]), f"level {l}: " + _first_diff("hsum", cap["hsum"], want["hsum"])
        # cross-check with the partition: every feature of a slot counts its node's rows
        per_feature = cap["cnt"].astype(np.int64).sum(axis=2)
        assert np.array_equal(per_feature, np.repeat(tree["num_examples"][cap["slot_node"]][:, None], cap["num_features"], 1))
    return caps
