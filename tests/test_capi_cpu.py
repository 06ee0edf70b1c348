"""CPU-side checks: the C-ABI library loads, exports every declared symbol, validates its
arguments, fails loudly without a device, and the host binning rule matches a numpy restatement."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import ydf_b200
from ydf_b200 import _capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    names = set()
    for hdr in ("ygg_b200.h", "ygg_b200_dataspec.h", "ygg_b200_model.h", "ygg_b200_comm.h"):
        text = open(os.path.join(ROOT, "include", hdr)).read()
        text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
        names |= set(re.findall(r"\b(ygg_[a-z0-9_]+)\s*\(", text))
    names -= {"ygg_allgather_fn"}
    return names


def test_library_exports_every_declared_symbol_of_abi_4():
    L = ydf_b200.lib()
    declared = _declared_symbols()
    assert len(declared) >= 25
    for name in sorted(declared):
        assert hasattr(L, name), name
    assert L.ygg_abi_version() == 4


def test_comm_bootstrap_without_device():
    """The NCCL binding resolves at run time (dlopen); the unique id needs no GPU, a communicator does."""
    try:
        uid = ydf_b200.Comm.unique_id()
    except ydf_b200.YggError as e:  # a box without any libnccl.so.2: loud, not silent
        assert "NCCL is not available" in str(e)
        return
    assert len(uid) == 128 and any(uid)
    with pytest.raises(ydf_b200.YggError):
        ydf_b200.Comm(uid, 3, 2, 0)  # rank outside the world


def test_config_defaults_match_reference_protos():
    # gradient_boosted_trees.proto:35-278, decision_tree.proto:32-108, gradient_boosted_trees.cc:3243-3249
    cfg = ydf_b200.default_config()
    assert cfg.num_trees == 300 and abs(cfg.shrinkage - 0.1) < 1e-7
    assert cfg.max_depth == 6 and cfg.min_examples == 5 and cfg.in_split_min_examples_check == 1
    assert cfg.use_hessian_gain == 0 and cfg.l1_regularization == 0 and cfg.l2_regularization == 0
    assert cfg.clamp_leaf_logit == 5 and cfg.hessian_split_score_subtract_parent == 0
    assert cfg.random_seed == 123456 and cfg.subsample == 1 and cfg.validation_ratio == 0
    # gradient_boosted_trees.proto:150-182 (validation rows are attached explicitly: ygg_gbt_set_validation_*)
    assert cfg.early_stopping == 2 and cfg.early_stopping_num_trees_look_ahead == 30
    assert cfg.early_stopping_initial_iteration == 10


def test_argument_validation_and_loud_failure_without_device():
    with pytest.raises(ydf_b200.YggError) as e:
        ydf_b200.Dataset(np.zeros((1, 4), np.uint8), [300], [0])
    assert e.value.code == 1  # INVALID_ARGUMENT before any device work
    with pytest.raises(ydf_b200.YggError) as e:
        ydf_b200.Dataset(np.zeros((1, 4), np.uint8), [4], [7])
    assert e.value.code == 1
    if ydf_b200.device_count() == 0:
        with pytest.raises(ydf_b200.YggError) as e:
            ydf_b200.Dataset(np.zeros((2, 10), np.uint8), [2, 2], [0, 0])
        assert e.value.code == 2  # NO_DEVICE: there is no CPU fallback
        assert "no CPU fallback" in str(e.value)


def test_histogram_capture_validates_arguments():
    L = ydf_b200.lib()
    assert L.ygg_gbt_debug_capture_histograms(None, C.c_int32(1)) == 1
    info = _capi.HistLevelInfo()
    assert L.ygg_gbt_debug_level_histograms(None, C.c_int32(0), C.byref(info), None, None, None, None, C.c_int32(0)) == 1
    assert C.sizeof(_capi.HistLevelInfo) == 80   # sizeof(ygg_hist_level_info), include/ygg_b200.h


def test_histogram_reference_quantiser():
    """The restatement the GPU histogram tests compare with: P strictly above max|g|, clamped 24-bit codes."""
    from tests.util import Q_BIAS, Q_MAX, g_pow2_exp, quantize_g, quantize_h2
    assert g_pow2_exp(np.float32([0.5, -0.25])) == 0 and g_pow2_exp(np.float32([-0.5])) == 0
    assert g_pow2_exp(np.zeros(3, np.float32)) == 0 and g_pow2_exp(np.float32([2.0 ** -140])) == -139
    assert g_pow2_exp(np.float32([0.75])) == 0 and g_pow2_exp(np.float32([1.0])) == 1
    below = np.nextafter(np.float32(1), np.float32(0))
    assert quantize_g(np.float32([0.5, -0.5, 0.0, below, -below]), 0).tolist() == \
        [Q_BIAS + (1 << 22), Q_BIAS - (1 << 22), Q_BIAS, Q_MAX, 0]
    assert quantize_g(np.float32([2.0 ** -120]), -119).tolist() == [Q_BIAS + (1 << 22)]
    assert quantize_h2(np.float32([0.25, 0.125, 0.0]), 0.25).tolist() == [1 << 24, 1 << 23, 0]


def test_learner_rejects_options_outside_the_path():
    L = ydf_b200.GradientBoostedTreesLearner
    # exact splitter (discretize_numerical_columns=False, the reference's default): reproduced with one bucket per distinct
    # value, refused — not approximated — for a column with more than 255 of them, before anything touches the device
    with pytest.raises(NotImplementedError, match="more than 255 distinct values"):
        L(label="y").train({"x": np.arange(1000, dtype=np.float32), "y": np.arange(1000) % 2})
    L(label="y", discretize_numerical_columns=True)  # reference defaults: validation_ratio=0.1, LOSS_INCREASE
    with pytest.raises(NotImplementedError):
        L(label="y", discretize_numerical_columns=True, validation_interval_in_trees=5)
    with pytest.raises(ValueError):
        L(label="y", discretize_numerical_columns=True, validation_ratio=1.5)
    # stochastic gradient boosting is on the path (SampleTrainingExamples); GOSS is not
    assert L(label="y", discretize_numerical_columns=True, validation_ratio=0.0, early_stopping="NONE", subsample=0.5).cfg.subsample == 0.5
    # ... and so is GOSS (variance gain); SELGB (ranking) is not
    g = L(label="y", discretize_numerical_columns=True, sampling_method="GOSS")
    assert abs(g.cfg.goss_alpha - 0.2) < 1e-7 and abs(g.cfg.goss_beta - 0.1) < 1e-7 and g.cfg.subsample == 1.0
    with pytest.raises(NotImplementedError):
        L(label="y", discretize_numerical_columns=True, sampling_method="GOSS", use_hessian_gain=True)
    with pytest.raises(NotImplementedError):
        L(label="y", discretize_numerical_columns=True, sampling_method="SELGB")
    with pytest.raises(ValueError):
        L(label="y", discretize_numerical_columns=True, subsample=0.0)
    with pytest.raises(ValueError):
        L(label="y", discretize_numerical_columns=True, tie_break="RANDOM")
    # example weights: on the path for the variance gain, refused with hessian gain
    assert L(label="y", discretize_numerical_columns=True, weights="w").weights == "w"
    with pytest.raises(NotImplementedError):
        L(label="y", discretize_numerical_columns=True, weights="w", use_hessian_gain=True)
    L(label="y", discretize_numerical_columns=True, validation_ratio=0.0, early_stopping="NONE")


def _np_boundaries(values, max_bins, min_obs):
    """numpy/python restatement of GenDiscretizedBoundaries (dataset/data_spec.cc:854-986)."""
    v = values[~np.isnan(values)].astype(np.float32)
    mean = float(v.astype(np.float64).sum() / len(v))
    uniq, counts = np.unique(v, return_counts=True)
    special = [np.float32(0.0), np.float32(mean)]
    inb = sum(1 for s in special if uniq[0] < s < uniq[-1])
    mb = max(1, max_bins - 2 - inb)
    max_boundaries = mb - 1
    bounds = []
    if len(uniq) > mb:
        total = int(counts.sum())
        # total < min_obs makes the reference divide by zero (data_spec.cc:900-903); the library clamps to one bin
        mb = max(1, min(mb, total // min_obs))
        large = total // mb
        is_large = counts >= large
        rem_bins = mb - int(is_large.sum())
        remaining = total - int(counts[is_large].sum())
        rem_bins = max(rem_bins, 1)
        cur = remaining // rem_bins
        running = 0
        made = 0
        for i in range(len(uniq) - 1):
            if not is_large[i]:
                remaining -= int(counts[i])
            running += int(counts[i])
            if is_large[i] or running >= cur or (is_large[i + 1] and running >= max(1, cur // 2)):
                bounds.append(np.float32((uniq[i] + uniq[i + 1]) / np.float32(2)))
                made += 1
                if made >= max_boundaries:
                    break
                running = 0
                if not is_large[i]:
                    rem_bins = max(1, rem_bins - 1)
                    cur = remaining // rem_bins
    else:
        running = 0
        for i in range(len(uniq) - 1):
            running += int(counts[i])
            if running >= min_obs:
                bounds.append(np.float32((uniq[i] + uniq[i + 1]) / np.float32(2)))
                running = 0
    for s in special:
        lo = np.nextafter(s, s - np.float32(1), dtype=np.float32)
        hi = np.nextafter(s, s + np.float32(1), dtype=np.float32)
        if not bounds:
            bounds += [lo, hi]
            continue
        bounds = [b for b in bounds if not (lo <= b <= hi)]
        if not bounds:
            # every boundary was inside the special bucket (e.g. a constant 0 column: the second special value,
            # the mean, equals the first).  The reference dereferences min_element of an empty vector here
            # (undefined behaviour, data_spec.cc:95-98); the library keeps the one special bucket.
            bounds = [lo, hi]
            continue
        mn, mx = min(bounds), max(bounds)
        if mn < hi:
            bounds.append(lo)
        if mx > lo:
            bounds.append(hi)
    return np.array(sorted(bounds), dtype=np.float32), mean


@pytest.mark.parametrize("case", ["normal", "few_values", "skewed", "with_nan"])
def test_binning_rule(case):
    rng = np.random.default_rng(7)
    if case == "normal":
        v = rng.normal(size=20000).astype(np.float32)
    elif case == "few_values":
        v = rng.integers(0, 12, size=5000).astype(np.float32)
    elif case == "skewed":
        v = np.concatenate([np.zeros(6000), rng.exponential(size=6000), np.full(3000, 7.5)]).astype(np.float32)
    else:
        v = rng.normal(size=8000).astype(np.float32)
        v[rng.random(8000) < 0.05] = np.nan
    for max_bins in (255, 256, 16):
        got, mean = ydf_b200.discretize_boundaries(v, max_bins, 3)
        want, wmean = _np_boundaries(v, max_bins, 3)
        assert abs(mean - wmean) < 1e-12 * max(1, abs(wmean))
        np.testing.assert_array_equal(got, want)
        assert len(got) + 1 <= max_bins
        na_bin = int(np.searchsorted(got, np.float32(mean), side="right"))
        enc = ydf_b200.discretize_encode(v, got, na_bin)
        ref = np.searchsorted(got, v, side="right")
        ref[np.isnan(v)] = na_bin
        np.testing.assert_array_equal(enc, ref.astype(np.uint8))
        # special values: 0 and the mean own a one-value bin
        if case != "few_values":
            assert ydf_b200.discretize_encode(np.array([0.0], np.float32), got, 0)[0] != \
                ydf_b200.discretize_encode(np.array([1e-3], np.float32), got, 0)[0]


def test_product_never_touches_the_oracle():
    """The oracle is test infrastructure: nothing under the package (Python, C++, CUDA, headers) nor the C-ABI headers may
    import, include, link or name it, and the shared library must not depend on libygg_oracle."""
    import os
    import re
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    pkg = os.path.join(root, "yggdrasil-decision-forests_b200")
    offenders = []
    for base in (pkg, os.path.join(root, "include")):
        for d, _, files in os.walk(base):
            for f in files:
                if f.endswith((".py", ".cc", ".cu", ".cuh", ".h", ".hpp")):
                    text = open(os.path.join(d, f), errors="replace").read()
                    if re.search(r"(?i)\boracle\b|ygg_oracle", text):
                        offenders.append(os.path.relpath(os.path.join(d, f), root))
    assert not offenders, offenders
    so = os.path.join(pkg, "libygg_b200.so")
    if os.path.exists(so):
        needed = subprocess.run(["readelf", "-d", so], capture_output=True, text=True).stdout
        assert "oracle" not in needed
