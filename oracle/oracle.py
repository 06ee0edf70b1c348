"""ctypes front-end of the CPU oracle (TEST INFRASTRUCTURE — see ygg_oracle.cc's header).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module.  The product package never does.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


class GbtConfig(C.Structure):
    """Mirror of ygg_gbt_config (include/ygg_b200.h)."""
    _fields_ = [
        ("abi_version", C.c_int32), ("loss", C.c_int32), ("num_trees", C.c_int32),
        ("shrinkage", C.c_float), ("max_depth", C.c_int32), ("min_examples", C.c_int32),
        ("in_split_min_examples_check", C.c_int32), ("use_hessian_gain", C.c_int32),
        ("l1_regularization", C.c_float), ("l2_regularization", C.c_float),
        ("l2_regularization_categorical", C.c_float), ("clamp_leaf_logit", C.c_float),
        ("hessian_split_score_subtract_parent", C.c_int32), ("random_seed", C.c_uint32),
        ("subsample", C.c_float), ("validation_ratio", C.c_float),
        ("sibling_subtraction", C.c_int32), ("early_stopping", C.c_int32),
        ("early_stopping_num_trees_look_ahead", C.c_int32), ("early_stopping_initial_iteration", C.c_int32),
        ("num_classes", C.c_int32), ("candidate_shuffle", C.c_int32), ("rng_words_consumed", C.c_uint32),
        ("split_jobs_draw_seeds", C.c_int32), ("growing_strategy", C.c_int32), ("max_num_nodes", C.c_int32),
        ("goss_alpha", C.c_float), ("goss_beta", C.c_float),
    ]


class Node(C.Structure):
    """Mirror of ygg_node (include/ygg_b200.h)."""
    _fields_ = [
        ("feature", C.c_int32), ("threshold_bin", C.c_int32), ("na_value", C.c_int32),
        ("depth", C.c_int32), ("neg_child", C.c_int32), ("pos_child", C.c_int32),
        ("split_score", C.c_float), ("leaf_value", C.c_float),
        ("num_examples", C.c_int64), ("num_pos_examples", C.c_int64),
        ("stat", C.c_double * 3), ("condition_type", C.c_int32), ("threshold_value", C.c_float),
        ("cat_mask", C.c_uint32 * 8),
    ]


NODE_DTYPE = np.dtype([
    ("feature", "<i4"), ("threshold_bin", "<i4"), ("na_value", "<i4"), ("depth", "<i4"),
    ("neg_child", "<i4"), ("pos_child", "<i4"), ("split_score", "<f4"), ("leaf_value", "<f4"),
    ("num_examples", "<i8"), ("num_pos_examples", "<i8"), ("stat", "<f8", (3,)),
    ("condition_type", "<i4"), ("threshold_value", "<f4"), ("cat_mask", "<u4", (8,)),
])
assert NODE_DTYPE.itemsize == C.sizeof(Node)

LOSS_BINOMIAL = 0
LOSS_SQUARED_ERROR = 1


def default_config(**kw):
    """Proto defaults (gradient_boosted_trees.proto:35-278, decision_tree.proto:32-108)."""
    cfg = GbtConfig()
    cfg.abi_version = 3
    cfg.max_num_nodes = 31
    cfg.loss = LOSS_BINOMIAL
    cfg.num_trees = 300
    cfg.shrinkage = 0.1
    cfg.max_depth = 6
    cfg.min_examples = 5
    cfg.in_split_min_examples_check = 1
    cfg.use_hessian_gain = 0
    cfg.l1_regularization = 0.0
    cfg.l2_regularization = 0.0
    cfg.l2_regularization_categorical = 1.0
    cfg.clamp_leaf_logit = 5.0
    cfg.hessian_split_score_subtract_parent = 0
    cfg.random_seed = 123456
    cfg.subsample = 1.0
    cfg.validation_ratio = 0.0
    cfg.sibling_subtraction = 1
    cfg.early_stopping = 2                          # VALIDATION_LOSS_INCREASE
    cfg.early_stopping_num_trees_look_ahead = 30
    cfg.early_stopping_initial_iteration = 10
    for k, v in kw.items():
        if not hasattr(cfg, k):
            raise AttributeError(k)
        setattr(cfg, k, v)
    return cfg


_NATIVE_FLAGS = ["-O3", "-march=native", "-std=c++17", "-fPIC", "-pthread", "-fno-fast-math", "-ffp-contract=off",
                 "-shared"]


def _native_path(src):
    """Where the -march=native build lives: a private directory under the system's temporary directory, named after
    the sources and flags, so that building it at run time never writes into the source tree (which may be
    read-only) and an edit of the sources gives a new file."""
    import hashlib
    import tempfile
    h = hashlib.sha256(" ".join(_NATIVE_FLAGS).encode())
    for p in (src, os.path.join(_HERE, "..", "include", "ygg_b200.h")):
        with open(p, "rb") as f:
            h.update(f.read())
    d = os.path.join(tempfile.gettempdir(), "ygg_oracle_%d" % os.getuid())
    os.makedirs(d, mode=0o700, exist_ok=True)
    if os.stat(d).st_uid != os.getuid():
        raise PermissionError("%s belongs to another user" % d)
    return os.path.join(d, "libygg_oracle_native_%s.so" % h.hexdigest()[:16])


def build(force=False, native=False):
    """Builds the restatement.  native=True: a second library compiled with -march=native for this host (see
    _native_path for where it goes), for the timed CPU legs of bench.py (SURVEY.md §8d); the portable in-tree
    build is what the tests load, because it may run on a host with another CPU than the one that built it."""
    src = os.path.join(_HERE, "ygg_oracle.cc")
    if native:
        so = _native_path(src)
        if force or not os.path.exists(so):
            tmp = so + ".%d.tmp" % os.getpid()
            subprocess.check_call(["g++"] + _NATIVE_FLAGS + ["-o", tmp, src], stdout=subprocess.DEVNULL)
            os.replace(tmp, so)
        return so
    so = os.path.join(_HERE, "libygg_oracle.so")
    if force or not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-B", "libygg_oracle.so"], stdout=subprocess.DEVNULL)
    return so


_NATIVE = False


def use_native_build():
    """Switches this process to the -march=native build (before the first call).  Returns a description of the
    build in use; falls back to the portable one when the box has no compiler."""
    global _NATIVE, _LIB
    if _LIB is not None and not _NATIVE:
        _LIB = None
    try:
        build(native=True)
        _NATIVE = True
        return "g++ -O3 -march=native (built on this host)"
    except Exception as e:  # noqa: BLE001
        _NATIVE = False
        return "g++ -O3, portable x86-64 (native build failed: %s)" % type(e).__name__


def lib():
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(build(native=True) if _NATIVE else build())
        L = _LIB
        L.oracle_find_split.restype = C.c_int
        L.oracle_partition.restype = C.c_int64
        L.oracle_train_tree.restype = C.c_int32
        L.oracle_initial_prediction.restype = C.c_float
        L.oracle_gbt_train.restype = C.c_int32
        L.oracle_max_threads.restype = C.c_int32
    return _LIB


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t)) if a is not None else None


CATEGORY_SORT_LIBSTDCXX, CATEGORY_SORT_STABLE, CATEGORY_SORT_LIBCXX_CLASSIC, CATEGORY_SORT_LIBCXX = 0, 1, 2, 3


def set_stable_category_sort(enabled):
    """Order of category buckets with EQUAL keys: False / 0 = libstdc++'s std::sort, True / 1 = stable (by index, what the
    GPU does), 2 = libc++'s std::sort up to LLVM 15, 3 = libc++'s std::sort from LLVM 16 on — the one the reference's goldens
    follow (tests/test_reference_replay.py)."""
    lib().oracle_set_stable_category_sort(C.c_int32(int(enabled)))


def set_bucket_values(values=None, na_replacement=None):
    """Exact numerical threshold rule (oracle_set_bucket_values): values[f] = float32 array of the bucket values of
    feature f (empty / None for a categorical feature), na_replacement[f] = column mean.  None removes the rule.
    With the rule, split nodes carry the float threshold in `threshold_value`."""
    if values is None:
        lib().oracle_set_bucket_values(C.c_int32(0), None, None, None)
        return
    flat = np.concatenate([np.asarray(v, np.float32) if v is not None else np.zeros(0, np.float32) for v in values] + [np.zeros(0, np.float32)])
    offs = np.zeros(len(values) + 1, np.int64)
    offs[1:] = np.cumsum([0 if v is None else len(v) for v in values])
    na = np.ascontiguousarray(na_replacement, dtype=np.float32)
    flat = np.ascontiguousarray(flat, dtype=np.float32)
    lib().oracle_set_bucket_values(C.c_int32(len(values)), _p(flat, C.c_float), _p(offs, C.c_int64), _p(na, C.c_float))


def set_categorical_random(enabled=False, num_trial_exponent=2.0, max_num_trials=5000):
    """categorical_algorithm RANDOM (ScanSplitsRandomBuckets) instead of CART for every categorical feature."""
    lib().oracle_set_categorical_random(C.c_int32(int(enabled)), C.c_float(num_trial_exponent), C.c_int32(max_num_trials))


def set_growing_strategy(best_first_global=False, max_num_nodes=31):
    """growing_strategy of every tree trainer of the oracle: LOCAL (default) or BEST_FIRST_GLOBAL (training.cc:4499-4656)."""
    lib().oracle_set_growing_strategy(C.c_int32(int(best_first_global)), C.c_int32(int(max_num_nodes)))


def set_weights(weights=None):
    """Example weights (one float32 per row of the dataset later handed to gbt_train / gbt_train_validated / train_tree);
    None = unweighted.  Variance gain, binomial / squared-error losses (LabelNumericalBucket<weighted=true>,
    SetLeafValueWithNewtonRaphsonStep<true>, weighted losses and initial predictions)."""
    if weights is None:
        lib().oracle_set_weights(None, C.c_int64(0))
        return
    w = np.ascontiguousarray(weights, dtype=np.float32)
    lib().oracle_set_weights(_p(w, C.c_float), C.c_int64(len(w)))


def set_goss_stable_sort(enabled):
    """GOSS: rows with EQUAL |gradient| ordered by row index (stable sort; what the engine's device sort gives) instead of
    by the standard library's std::sort."""
    lib().oracle_set_goss_stable_sort(C.c_int32(int(enabled)))


def goss_sample(gradient, alpha, beta, rng, weights=None):
    """SampleTrainingExamplesWithGoss on its own -> (selected row ids in the reference's order, weights)."""
    g = np.ascontiguousarray(gradient, dtype=np.float32)
    w = np.ones(len(g), np.float32) if weights is None else np.array(weights, dtype=np.float32)
    sel = np.zeros(len(g) + 1, np.uint32)
    k = lib().oracle_goss_sample(_p(g, C.c_float), C.c_int64(len(g)), C.c_float(alpha), C.c_float(beta), rng._h,
                                 _p(sel, C.c_uint32), _p(w, C.c_float))
    return sel[:k].copy(), w


def set_validated_shuffle_mode(mode):
    """Candidate shuffle of gbt_train_validated: SHUFFLE_NONE / SHUFFLE_LIBSTDCXX / SHUFFLE_LIBCXX."""
    lib().oracle_set_validated_shuffle_mode(C.c_int32(int(mode)))


def set_hessian_buckets_double(enabled):
    """Cross-check mode: exact (double) hessian-gain buckets instead of the reference's float."""
    lib().oracle_set_hessian_buckets_double(C.c_int32(int(enabled)))


class Rng:
    """std::mt19937 + libstdc++'s std::shuffle, to follow the learner's random stream (oracle_rng_*)."""

    def __init__(self, seed):
        L = lib()
        L.oracle_rng_create.restype = C.c_void_p
        self._h = C.c_void_p(L.oracle_rng_create(C.c_uint32(seed)))
        self.position = 0   # engine words drawn so far (None once a call drew an unknown number)

    def discard(self, n):
        lib().oracle_rng_discard(self._h, C.c_uint64(n))
        if self.position is not None:
            self.position += int(n)

    def clone(self):
        L = lib()
        L.oracle_rng_clone.restype = C.c_void_p
        other = Rng.__new__(Rng)
        other._h = C.c_void_p(L.oracle_rng_clone(self._h))
        other.position = self.position
        return other

    def next(self):
        L = lib()
        L.oracle_rng_next.restype = C.c_uint32
        if self.position is not None:
            self.position += 1
        return int(L.oracle_rng_next(self._h))

    def shuffle_libcxx(self, n):
        """The order libc++'s std::shuffle gives to 0..n-1 (llvm libcxx/include/__algorithm/shuffle.h: for each position
        draw i in [0, d] with uniform_int_distribution = low w bits of one engine word, rejected while >= d + 1)."""
        v = list(range(n))
        d = n - 1
        first = 0
        while first < n - 1:
            rp = d + 1
            w = rp.bit_length() - 1
            if rp & ((1 << w) - 1):
                w += 1
            while True:
                u = self.next() & ((1 << w) - 1)
                if u < rp:
                    break
            if u:
                v[first], v[first + u] = v[first + u], v[first]
            first += 1
            d -= 1
        return v

    def shuffle(self, n):
        """-> the order libstdc++'s std::shuffle gives to 0..n-1."""
        v = np.arange(n, dtype=np.int32)
        self.position = None
        lib().oracle_rng_shuffle(self._h, _p(v, C.c_int32), C.c_int32(n))
        return v.tolist()

    def __del__(self):
        if getattr(self, "_h", None):
            lib().oracle_rng_destroy(self._h)
            self._h = None


def max_threads():
    return int(lib().oracle_max_threads())


def as_u16_columns(bins):
    """bins: [F, N] integer array (column-major storage == C-contiguous [F][N])."""
    b = np.ascontiguousarray(bins, dtype=np.uint16)
    assert b.ndim == 2
    return b


def find_split(column, num_bins, na_bin, rows, gradients, hessians=None, parent_stat=None,
               use_hessian_gain=False, min_num_obs=1, l1=0.0, l2=0.0, subtract_parent=False,
               initial_split_score=0.0, categorical=False):
    column = np.ascontiguousarray(column, dtype=np.uint16)
    rows = np.ascontiguousarray(rows, dtype=np.uint32)
    g = np.ascontiguousarray(gradients, dtype=np.float32)
    h = None if hessians is None else np.ascontiguousarray(hessians, dtype=np.float32)
    if parent_stat is None:
        gs = g[rows].astype(np.float64)
        if use_hessian_gain:
            parent_stat = [gs.sum(), float(h[rows].astype(np.float64).sum()), float(len(rows))]
        else:
            g2 = (g[rows] * g[rows]).astype(np.float64)
            parent_stat = [gs.sum(), g2.sum(), float(len(rows))]
    ps = np.asarray(parent_stat, dtype=np.float64)
    thr, na = C.c_int32(), C.c_int32()
    score, npos = C.c_float(), C.c_int64()
    mask = np.zeros(8, dtype=np.uint32)
    r = lib().oracle_find_split(
        _p(column, C.c_uint16), C.c_int64(len(column)), C.c_int32(num_bins), C.c_int32(na_bin),
        _p(rows, C.c_uint32), C.c_int64(len(rows)), _p(g, C.c_float), _p(h, C.c_float),
        _p(ps, C.c_double), C.c_int32(int(use_hessian_gain)), C.c_int32(min_num_obs),
        C.c_double(l1), C.c_double(l2), C.c_int32(int(subtract_parent)),
        C.c_float(initial_split_score), C.byref(thr), C.byref(na), C.byref(score), C.byref(npos),
        C.c_int32(int(categorical)), _p(mask, C.c_uint32))
    pos_set = [c for c in range(256) if (int(mask[c >> 5]) >> (c & 31)) & 1]
    return dict(result=r, threshold=thr.value, na_value=bool(na.value), split_score=score.value,
                num_pos=npos.value, positive_categories=pos_set)


def partition(column, threshold, na_value, rows):
    column = np.ascontiguousarray(column, dtype=np.uint16)
    rows = np.ascontiguousarray(rows, dtype=np.uint32)
    out = np.empty_like(rows)
    n_pos = lib().oracle_partition(_p(column, C.c_uint16), C.c_int32(threshold),
                                   C.c_int32(int(na_value)), _p(rows, C.c_uint32),
                                   C.c_int64(len(rows)), _p(out, C.c_uint32))
    return out[:n_pos], out[n_pos:]


def _ft(feature_type):
    return None if feature_type is None else np.ascontiguousarray(feature_type, dtype=np.int32)


def train_tree(bins, num_bins, na_bin, gradients, hessians, cfg, num_threads=1,
               shuffle_candidates=False, leaf_mode=0, capacity=1 << 16, feature_type=None):
    b = as_u16_columns(bins)
    F, N = b.shape
    nb = np.ascontiguousarray(num_bins, dtype=np.int32)
    na = np.ascontiguousarray(na_bin, dtype=np.int32)
    g = np.ascontiguousarray(gradients, dtype=np.float32)
    h = None if hessians is None else np.ascontiguousarray(hessians, dtype=np.float32)
    out = np.zeros(capacity, dtype=NODE_DTYPE)
    n = lib().oracle_train_tree(_p(b, C.c_uint16), C.c_int64(N), C.c_int32(F), _p(nb, C.c_int32),
                                _p(na, C.c_int32), _p(g, C.c_float), _p(h, C.c_float),
                                C.byref(cfg), C.c_int32(num_threads),
                                C.c_int32(int(shuffle_candidates)), C.c_int32(leaf_mode),
                                out.ctypes.data_as(C.POINTER(Node)), C.c_int32(capacity),
                                _p(_ft(feature_type), C.c_int32))
    if n < 0:
        raise RuntimeError("oracle_train_tree: capacity too small")
    return out[:n].copy()


SHUFFLE_NONE, SHUFFLE_LIBSTDCXX, SHUFFLE_LIBCXX = 0, 1, 2


def train_tree_rng(bins, num_bins, na_bin, gradients, hessians, cfg, rng, shuffle=SHUFFLE_LIBCXX, num_threads=4,
                   capacity=1 << 16, feature_type=None):
    """train_tree drawing the per-node candidate shuffles (+ one seed per feature job) from the caller's Rng."""
    b = as_u16_columns(bins)
    F, N = b.shape
    nb = np.ascontiguousarray(num_bins, dtype=np.int32)
    na = np.ascontiguousarray(na_bin, dtype=np.int32)
    g = np.ascontiguousarray(gradients, dtype=np.float32)
    h = None if hessians is None else np.ascontiguousarray(hessians, dtype=np.float32)
    out = np.zeros(capacity, dtype=NODE_DTYPE)
    assert num_threads > 1, "the seed draws belong to the concurrent manager"
    n = lib().oracle_train_tree_rng(_p(b, C.c_uint16), C.c_int64(N), C.c_int32(F), _p(nb, C.c_int32), _p(na, C.c_int32),
                                    _p(g, C.c_float), _p(h, C.c_float), C.byref(cfg), C.c_int32(num_threads),
                                    C.c_int32(shuffle), rng._h, out.ctypes.data_as(C.POINTER(Node)),
                                    C.c_int32(capacity), _p(_ft(feature_type), C.c_int32))
    if n < 0:
        raise RuntimeError("oracle_train_tree_rng: capacity too small")
    return out[:n].copy()


def initial_prediction(loss, labels, weights=None):
    w = None if weights is None else np.ascontiguousarray(weights, dtype=np.float32)
    fn = lib().oracle_initial_prediction_w
    fn.restype = C.c_float
    if loss == LOSS_BINOMIAL:
        l = np.ascontiguousarray(labels, dtype=np.int32)
        return float(fn(C.c_int32(loss), _p(l, C.c_int32), None, _p(w, C.c_float), C.c_int64(len(l))))
    l = np.ascontiguousarray(labels, dtype=np.float32)
    return float(fn(C.c_int32(loss), None, _p(l, C.c_float), _p(w, C.c_float), C.c_int64(len(l))))


def update_gradients(loss, labels, predictions):
    p = np.ascontiguousarray(predictions, dtype=np.float32)
    g = np.empty_like(p)
    h = np.empty_like(p)
    li = lf = None
    if loss == LOSS_BINOMIAL:
        li = np.ascontiguousarray(labels, dtype=np.int32)
    else:
        lf = np.ascontiguousarray(labels, dtype=np.float32)
    lib().oracle_update_gradients(C.c_int32(loss), _p(li, C.c_int32), _p(lf, C.c_float),
                                  _p(p, C.c_float), C.c_int64(len(p)), _p(g, C.c_float),
                                  _p(h, C.c_float))
    return g, h


def loss_value(loss, labels, predictions, weights=None):
    p = np.ascontiguousarray(predictions, dtype=np.float32)
    w = None if weights is None else np.ascontiguousarray(weights, dtype=np.float32)
    li = lf = None
    if loss == LOSS_BINOMIAL:
        li = np.ascontiguousarray(labels, dtype=np.int32)
    else:
        lf = np.ascontiguousarray(labels, dtype=np.float32)
    a, b = C.c_float(), C.c_float()
    lib().oracle_loss_w(C.c_int32(loss), _p(li, C.c_int32), _p(lf, C.c_float), _p(p, C.c_float), _p(w, C.c_float),
                        C.c_int64(len(p)), C.byref(a), C.byref(b))
    return a.value, b.value


def gbt_train(bins, num_bins, na_bin, labels, cfg, num_iters, num_threads=1,
              shuffle_candidates=False, predictions=None, want_gradients=False, feature_type=None):
    """Runs the boosting loop.  Returns dict(trees=[node arrays], loss, secondary, predictions)."""
    b = as_u16_columns(bins)
    F, N = b.shape
    nb = np.ascontiguousarray(num_bins, dtype=np.int32)
    na = np.ascontiguousarray(na_bin, dtype=np.int32)
    li = lf = None
    if cfg.loss == LOSS_BINOMIAL:
        li = np.ascontiguousarray(labels, dtype=np.int32)
    else:
        lf = np.ascontiguousarray(labels, dtype=np.float32)
    init = predictions is None
    pred = np.zeros(N, dtype=np.float32) if init else np.array(predictions, dtype=np.float32)
    max_nodes = (2 << max(1, cfg.max_depth)) if cfg.max_depth > 0 else 1 << 16   # (best-first trees are one level deeper)
    cap = int(num_iters) * max_nodes
    nodes = np.zeros(cap, dtype=NODE_DTYPE)
    offs = np.zeros(num_iters + 1, dtype=np.int64)
    loss = np.zeros(num_iters, dtype=np.float32)
    sec = np.zeros(num_iters, dtype=np.float32)
    g = np.zeros(N, dtype=np.float32) if want_gradients else None
    h = np.zeros(N, dtype=np.float32) if want_gradients else None
    r = lib().oracle_gbt_train(
        _p(b, C.c_uint16), C.c_int64(N), C.c_int32(F), _p(nb, C.c_int32), _p(na, C.c_int32),
        _p(li, C.c_int32), _p(lf, C.c_float), C.byref(cfg), C.c_int32(num_iters),
        C.c_int32(num_threads), C.c_int32(int(shuffle_candidates)), C.c_int32(int(init)),
        _p(pred, C.c_float), nodes.ctypes.data_as(C.POINTER(Node)), C.c_int64(cap),
        _p(offs, C.c_int64), _p(loss, C.c_float), _p(sec, C.c_float), _p(g, C.c_float),
        _p(h, C.c_float), _p(_ft(feature_type), C.c_int32))
    if r == -2:
        raise NotImplementedError("oracle: example weights with hessian gain / multinomial loss are not restated")
    if r < 0:
        raise RuntimeError("oracle_gbt_train: node capacity too small")
    trees = [nodes[offs[i]:offs[i + 1]].copy() for i in range(num_iters)]
    return dict(trees=trees, loss=loss, secondary=sec, predictions=pred, gradients=g, hessians=h)


def gbt_train_validated(bins, num_bins, na_bin, labels, cfg, validation_ratio, num_threads=1, feature_type=None):
    """The learner loop with the validation hold-out and early stopping (oracle_gbt_train_validated).
    `bins` / `labels` are the FULL dataset.  Returns dict(in_training, trees (final model), train_loss,
    valid_loss, valid_secondary (per logged iteration), validation_loss, early_stopping_triggered)."""
    b = as_u16_columns(bins)
    F, N = b.shape
    nb = np.ascontiguousarray(num_bins, dtype=np.int32)
    na = np.ascontiguousarray(na_bin, dtype=np.int32)
    li = lf = None
    if cfg.loss in (LOSS_BINOMIAL, 2):   # 2 = LOSS_MULTINOMIAL: K = cfg.num_classes trees per iteration
        li = np.ascontiguousarray(labels, dtype=np.int32)
    else:
        lf = np.ascontiguousarray(labels, dtype=np.float32)
    iters = int(cfg.num_trees)
    T = iters * (int(cfg.num_classes) if cfg.loss == 2 else 1)
    cap = T * max(1 << (max(1, cfg.max_depth) + 1), 64)   # BEST_FIRST_GLOBAL trees start at depth 0
    nodes = np.zeros(cap, dtype=NODE_DTYPE)
    offs = np.zeros(T + 1, dtype=np.int64)
    mask = np.zeros(N, dtype=np.uint8)
    tl, vl, vs = (np.zeros(iters, dtype=np.float32) for _ in range(3))
    n_entries, trig, fvl = C.c_int32(), C.c_int32(), C.c_float()
    fn = lib().oracle_gbt_train_validated
    fn.restype = C.c_int32
    r = fn(_p(b, C.c_uint16), C.c_int64(N), C.c_int32(F), _p(nb, C.c_int32), _p(na, C.c_int32),
           _p(li, C.c_int32), _p(lf, C.c_float), C.byref(cfg), C.c_float(validation_ratio), C.c_int32(num_threads),
           _p(_ft(feature_type), C.c_int32), _p(mask, C.c_uint8), nodes.ctypes.data_as(C.POINTER(Node)),
           C.c_int64(cap), _p(offs, C.c_int64), _p(tl, C.c_float), _p(vl, C.c_float), _p(vs, C.c_float),
           C.byref(n_entries), C.byref(fvl), C.byref(trig))
    if r == -2:
        raise NotImplementedError("oracle: example weights with hessian gain / multinomial loss are not restated")
    if r < 0:
        raise RuntimeError("oracle_gbt_train_validated: node capacity too small")
    k = n_entries.value
    return dict(in_training=mask.astype(bool), trees=[nodes[offs[i]:offs[i + 1]].copy() for i in range(r)],
                train_loss=tl[:k], valid_loss=vl[:k], valid_secondary=vs[:k], num_entries=k,
                validation_loss=fvl.value, early_stopping_triggered=bool(trig.value))


LOSS_MULTINOMIAL = 2


def mc_update_gradients(labels, K, predictions):
    """predictions [n, K] -> (gradient [K, n], hessian [K, n])."""
    l = np.ascontiguousarray(labels, dtype=np.int32)
    p = np.ascontiguousarray(predictions, dtype=np.float32)
    n = len(l)
    g, h = np.zeros((K, n), np.float32), np.zeros((K, n), np.float32)
    lib().oracle_mc_update_gradients(_p(l, C.c_int32), C.c_int32(K), _p(p, C.c_float), C.c_int64(n),
                                     _p(g, C.c_float), _p(h, C.c_float))
    return g, h


def mc_loss(labels, K, predictions, weights=None):
    l = np.ascontiguousarray(labels, dtype=np.int32)
    p = np.ascontiguousarray(predictions, dtype=np.float32)
    w = None if weights is None else np.ascontiguousarray(weights, dtype=np.float32)
    a, b = C.c_float(), C.c_float()
    lib().oracle_mc_loss_w(_p(l, C.c_int32), C.c_int32(K), _p(p, C.c_float), _p(w, C.c_float), C.c_int64(len(l)), C.byref(a), C.byref(b))
    return a.value, b.value


def gbt_train_mc(bins, num_bins, na_bin, labels, cfg, num_iters, num_threads=1, feature_type=None):
    """Multinomial boosting loop: K = cfg.num_classes trees per iteration (iteration-major, class-minor)."""
    b = as_u16_columns(bins)
    F, N = b.shape
    K = int(cfg.num_classes)
    nb = np.ascontiguousarray(num_bins, dtype=np.int32)
    na = np.ascontiguousarray(na_bin, dtype=np.int32)
    l = np.ascontiguousarray(labels, dtype=np.int32)
    cap = int(num_iters) * K * (1 << max(1, cfg.max_depth))
    nodes = np.zeros(cap, dtype=NODE_DTYPE)
    offs = np.zeros(num_iters * K + 1, dtype=np.int64)
    pred = np.zeros((N, K), np.float32)
    loss, sec = np.zeros(num_iters, np.float32), np.zeros(num_iters, np.float32)
    fn = lib().oracle_gbt_train_mc
    fn.restype = C.c_int32
    r = fn(_p(b, C.c_uint16), C.c_int64(N), C.c_int32(F), _p(nb, C.c_int32), _p(na, C.c_int32), _p(l, C.c_int32),
           C.byref(cfg), C.c_int32(num_iters), C.c_int32(num_threads), _p(_ft(feature_type), C.c_int32),
           _p(pred, C.c_float), nodes.ctypes.data_as(C.POINTER(Node)), C.c_int64(cap), _p(offs, C.c_int64),
           _p(loss, C.c_float), _p(sec, C.c_float))
    if r == -2:
        raise NotImplementedError("oracle: example weights with hessian gain are not restated")
    if r < 0:
        raise RuntimeError("oracle_gbt_train_mc: node capacity too small")
    return dict(trees=[nodes[offs[i]:offs[i + 1]].copy() for i in range(r)], loss=loss, secondary=sec, predictions=pred)
