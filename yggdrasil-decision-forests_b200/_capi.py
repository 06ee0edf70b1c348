"""ctypes binding of libygg_b200.so (include/ygg_b200.h).  No torch types cross this boundary."""
import ctypes as C
import os

import numpy as np

from . import _build

_LIB = None


class YggError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"[ygg status {code}] {msg}")
        self.code = code


class GbtConfig(C.Structure):
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


NODE_DTYPE = np.dtype([
    ("feature", "<i4"), ("threshold_bin", "<i4"), ("na_value", "<i4"), ("depth", "<i4"),
    ("neg_child", "<i4"), ("pos_child", "<i4"), ("split_score", "<f4"), ("leaf_value", "<f4"),
    ("num_examples", "<i8"), ("num_pos_examples", "<i8"), ("stat", "<f8", (3,)),
    ("condition_type", "<i4"), ("threshold_value", "<f4"), ("cat_mask", "<u4", (8,)),
])
assert NODE_DTYPE.itemsize == 112  # sizeof(ygg_node), include/ygg_b200.h

FEATURE_DISCRETIZED_NUMERICAL = 0
FEATURE_CATEGORICAL = 1

# enum ygg_hist_layout
HIST_LAYOUTS = ("root_sum", "packed", "shared", "shared_hess", "packed_multi", "shared_multi", "shared_hess_multi")


class HistLevelInfo(C.Structure):
    _fields_ = [
        ("layout", C.c_int32), ("features_per_item", C.c_int32), ("smem_slots", C.c_int32), ("passes", C.c_int32),
        ("chunk_blocks", C.c_int32), ("reserved", C.c_int32), ("num_slots", C.c_int32), ("feature_begin", C.c_int32),
        ("num_features", C.c_int32), ("has_hsum", C.c_int32), ("g_pow2", C.c_float), ("h2_pow2", C.c_float),
        ("n_rows", C.c_int64), ("g", C.POINTER(C.c_float)), ("h2", C.POINTER(C.c_float)), ("selected", C.POINTER(C.c_uint8)),
    ]

ALLGATHER_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p)
ALLREDUCE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p)
REDUCESCATTER_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p)

EXPORTS = [
    "ygg_abi_version", "ygg_last_error", "ygg_device_count", "ygg_dataset_create",
    "ygg_dataset_set_feature_types", "ygg_dataset_destroy", "ygg_dataset_num_rows", "ygg_dataset_num_features",
    "ygg_gbt_config_init", "ygg_gbt_create", "ygg_gbt_destroy", "ygg_gbt_set_labels_i32",
    "ygg_gbt_set_labels_f32", "ygg_gbt_set_weights_f32", "ygg_gbt_set_validation_weights_f32", "ygg_gbt_set_feature_shard", "ygg_gbt_set_row_shard", "ygg_gbt_set_row_shard_scatter", "ygg_feature_shard",
    "ygg_merge_shard_best", "ygg_gbt_initial_prediction",
    "ygg_gbt_train", "ygg_gbt_train_timed", "ygg_gbt_step", "ygg_gbt_sync", "ygg_gbt_num_trees", "ygg_gbt_get_tree",
    "ygg_gbt_train_loss", "ygg_gbt_get_predictions", "ygg_gbt_set_predictions", "ygg_gbt_predict",
    "ygg_tree_train_on_gradients", "ygg_gbt_debug_capture_histograms", "ygg_gbt_debug_level_histograms", "ygg_partition_rows",
    "ygg_gbt_set_profiling", "ygg_gbt_get_profile", "ygg_gbt_save_ydf",
    "ygg_discretize_boundaries", "ygg_discretize_encode", "ygg_model_write_ydf",
    "ygg_validation_split_mask", "ygg_dataset_split_rows", "ygg_gbt_set_validation_i32",
    "ygg_gbt_set_validation_f32", "ygg_gbt_validation_loss", "ygg_gbt_num_iterations", "ygg_gbt_final_validation",
    "ygg_gen_discretized_boundaries", "ygg_dataset_builder_create", "ygg_dataset_builder_add_numerical",
    "ygg_dataset_builder_add_numerical_async", "ygg_dataset_builder_get_numerical",
    "ygg_dataset_builder_add_bins", "ygg_dataset_builder_finish", "ygg_dataset_builder_destroy",
    "ygg_dataset_get_bins", "ygg_dataset_set_bucket_values", "ygg_gbt_tie_stats", "ygg_gbt_set_tie_rng_position",
    "ygg_gbt_best_split_window_bytes", "ygg_gbt_set_best_split_window", "ygg_comm_window_create",
    "ygg_comm_unique_id", "ygg_comm_create", "ygg_comm_destroy", "ygg_comm_allreduce", "ygg_comm_allgather", "ygg_comm_reducescatter",
]


def lib():
    """Loads (building if stale) the native library.  There is no fallback: if the library
    cannot be built or loaded this raises."""
    global _LIB
    if _LIB is None:
        path = _build.build()
        L = C.CDLL(path)
        L.ygg_last_error.restype = C.c_char_p
        L.ygg_dataset_num_rows.restype = C.c_int64
        L.ygg_gbt_config_init.restype = None
        for name in EXPORTS:
            getattr(L, name)  # fail loudly on a missing symbol
        _LIB = L
    return _LIB


def check(status):
    if status != 0:
        raise YggError(status, lib().ygg_last_error().decode("utf-8", "replace"))


def ptr(a, t):
    return a.ctypes.data_as(C.POINTER(t)) if a is not None else None


def default_config(**kw):
    cfg = GbtConfig()
    lib().ygg_gbt_config_init(C.byref(cfg))
    for k, v in kw.items():
        if not hasattr(cfg, k):
            raise AttributeError(k)
        setattr(cfg, k, v)
    return cfg


class Dataset:
    """Device-resident bucketised dataset (ygg_dataset)."""

    def __init__(self, bins, num_bins, na_bin, device=0, feature_types=None):
        b = np.asarray(bins)
        # a row slice of a larger [F, N] matrix is taken in place (column_stride = the parent's N)
        if not (b.dtype == np.uint8 and b.ndim == 2 and b.strides[1] == 1 and b.strides[0] >= b.shape[1]):
            b = np.ascontiguousarray(bins, dtype=np.uint8)
        assert b.ndim == 2, "bins must be [n_features, n_rows] (column-major storage)"
        self.n_features, self.n_rows = b.shape
        self.num_bins = np.ascontiguousarray(num_bins, dtype=np.int32)
        self.na_bin = np.ascontiguousarray(na_bin, dtype=np.int32)
        assert len(self.num_bins) == self.n_features and len(self.na_bin) == self.n_features
        self.handle = C.c_void_p()
        self.h2d_bytes = self.n_features * self.n_rows
        # (the stride of a length-1 axis is arbitrary in numpy: a single-feature matrix has no second column to reach)
        col_stride = b.strides[0] if self.n_features > 1 else max(int(b.strides[0]), self.n_rows)
        check(lib().ygg_dataset_create(C.byref(self.handle), C.c_int64(self.n_rows),
                                       C.c_int32(self.n_features), C.cast(b.ctypes.data, C.POINTER(C.c_uint8)),
                                       C.c_int64(col_stride), ptr(self.num_bins, C.c_int32),
                                       ptr(self.na_bin, C.c_int32), C.c_int32(device)))
        self.feature_types = np.zeros(self.n_features, np.int32)
        if feature_types is not None:
            self.set_feature_types(feature_types)

    def set_bucket_values(self, feature, values, na_replacement):
        """Exact threshold rule for a numerical feature with one bucket per distinct value: values[b] = value of bucket b,
        na_replacement = the column mean."""
        v = np.ascontiguousarray(values, dtype=np.float32)
        check(lib().ygg_dataset_set_bucket_values(self.handle, C.c_int32(int(feature)), ptr(v, C.c_float), C.c_int32(len(v)),
                                                  C.c_float(float(np.float32(na_replacement)))))

    def set_feature_types(self, feature_types):
        """feature_types[f]: FEATURE_DISCRETIZED_NUMERICAL or FEATURE_CATEGORICAL."""
        ft = np.ascontiguousarray(feature_types, dtype=np.int32)
        check(lib().ygg_dataset_set_feature_types(self.handle, ptr(ft, C.c_int32), C.c_int32(len(ft))))
        self.feature_types = ft

    def close(self):
        if self.handle:
            lib().ygg_dataset_destroy(self.handle)
            self.handle = C.c_void_p()

    def split_rows(self, select):
        """-> (Dataset of the rows with select != 0, Dataset of the others), gathered on the device."""
        m = np.ascontiguousarray(select, dtype=np.uint8)
        assert m.shape == (self.n_rows,)
        a, b = C.c_void_p(), C.c_void_p()
        check(lib().ygg_dataset_split_rows(self.handle, ptr(m, C.c_uint8), C.byref(a), C.byref(b)))
        out = []
        for hnd, n in ((a, int(m.astype(bool).sum())), (b, int(len(m) - m.astype(bool).sum()))):
            d = Dataset.__new__(Dataset)
            d.handle, d.n_features, d.n_rows = hnd, self.n_features, n
            d.num_bins, d.na_bin, d.feature_types, d.h2d_bytes = self.num_bins, self.na_bin, self.feature_types, 0
            out.append(d)
        return out[0], out[1]

    def get_bins(self, feature):
        out = np.empty(self.n_rows, np.uint8)
        check(lib().ygg_dataset_get_bins(self.handle, C.c_int32(feature), ptr(out, C.c_uint8)))
        return out

    def partition_rows(self, rows, feature, threshold_bin):
        rows = np.ascontiguousarray(rows, dtype=np.uint32)
        out = np.empty_like(rows)
        n_pos = C.c_int64()
        check(lib().ygg_partition_rows(self.handle, ptr(rows, C.c_uint32), C.c_int64(len(rows)),
                                       C.c_int32(feature), C.c_int32(threshold_bin),
                                       ptr(out, C.c_uint32), C.byref(n_pos)))
        return out[:n_pos.value], out[n_pos.value:]

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DatasetBuilder:
    """Column-by-column construction of a device-resident dataset with ON-GPU binning of the float32
    columns (include/ygg_b200_dataspec.h, csrc/ygg_binning.cu)."""

    def __init__(self, n_rows, n_features, device=0):
        self.handle = C.c_void_p()
        self.n_rows, self.n_features, self.device = int(n_rows), int(n_features), device
        self.num_bins = np.ones(n_features, np.int32)
        self.na_bin = np.zeros(n_features, np.int32)
        self.feature_types = np.zeros(n_features, np.int32)
        self.h2d_bytes = 0
        check(lib().ygg_dataset_builder_create(C.byref(self.handle), C.c_int64(n_rows), C.c_int32(n_features),
                                               C.c_int32(device)))

    def add_numerical(self, feature, values, maximum_num_bins=255, min_obs_in_bins=3, n_stats_rows=0):
        """-> (boundaries float32, mean, na_bin, num_missing); the column is binned on the GPU."""
        v = np.ascontiguousarray(values, dtype=np.float32)
        assert v.shape == (self.n_rows,)
        bounds = np.empty(256, np.float32)
        nb, mean, na, miss = C.c_int32(), C.c_double(), C.c_int32(), C.c_int64()
        check(lib().ygg_dataset_builder_add_numerical(
            self.handle, C.c_int32(feature), ptr(v, C.c_float), C.c_int64(n_stats_rows),
            C.c_int32(maximum_num_bins), C.c_int32(min_obs_in_bins), ptr(bounds, C.c_float), C.c_int32(256),
            C.byref(nb), C.byref(mean), C.byref(na), C.byref(miss)))
        self.num_bins[feature], self.na_bin[feature] = nb.value + 1, na.value
        self.h2d_bytes += v.nbytes
        return bounds[:nb.value].copy(), mean.value, na.value, miss.value

    def add_numerical_async(self, feature, values, maximum_num_bins=255, min_obs_in_bins=3, n_stats_rows=0):
        """Enqueues the column and returns; collect with get_numerical (or finish).  The array is kept
        alive by the builder until then."""
        v = np.ascontiguousarray(values, dtype=np.float32)
        assert v.shape == (self.n_rows,)
        self._pending = getattr(self, "_pending", {})
        self._pending[feature] = v
        check(lib().ygg_dataset_builder_add_numerical_async(
            self.handle, C.c_int32(feature), ptr(v, C.c_float), C.c_int64(n_stats_rows),
            C.c_int32(maximum_num_bins), C.c_int32(min_obs_in_bins)))
        self.h2d_bytes += v.nbytes

    def get_numerical(self, feature):
        bounds = np.empty(256, np.float32)
        nb, mean, na, miss = C.c_int32(), C.c_double(), C.c_int32(), C.c_int64()
        check(lib().ygg_dataset_builder_get_numerical(self.handle, C.c_int32(feature), ptr(bounds, C.c_float),
                                                      C.c_int32(256), C.byref(nb), C.byref(mean), C.byref(na),
                                                      C.byref(miss)))
        getattr(self, "_pending", {}).pop(feature, None)
        self.num_bins[feature], self.na_bin[feature] = nb.value + 1, na.value
        return bounds[:nb.value].copy(), mean.value, na.value, miss.value

    def add_bins(self, feature, bins, num_bins, na_bin, feature_type=0):
        b = np.ascontiguousarray(bins, dtype=np.uint8)
        assert b.shape == (self.n_rows,)
        check(lib().ygg_dataset_builder_add_bins(self.handle, C.c_int32(feature), ptr(b, C.c_uint8),
                                                 C.c_int32(num_bins), C.c_int32(na_bin), C.c_int32(feature_type)))
        self.num_bins[feature], self.na_bin[feature], self.feature_types[feature] = num_bins, na_bin, feature_type
        self.h2d_bytes += b.nbytes

    def finish(self):
        """-> Dataset (the builder is consumed)."""
        for f in list(getattr(self, "_pending", {})):
            self.get_numerical(f)
        out = C.c_void_p()
        check(lib().ygg_dataset_builder_finish(self.handle, C.byref(out)))
        self.handle = C.c_void_p()
        ds = Dataset.__new__(Dataset)
        ds.handle = out
        ds.n_features, ds.n_rows = self.n_features, self.n_rows
        ds.num_bins, ds.na_bin, ds.feature_types = self.num_bins, self.na_bin, self.feature_types
        ds.h2d_bytes = self.h2d_bytes
        return ds

    def close(self):
        if self.handle:
            lib().ygg_dataset_builder_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def validation_split_mask(random_seed, n_rows, validation_ratio):
    """ExtractValidationDataset's row draw: True = training row."""
    m = np.empty(n_rows, np.uint8)
    check(lib().ygg_validation_split_mask(C.c_uint32(random_seed), C.c_int64(n_rows), C.c_float(validation_ratio),
                                          ptr(m, C.c_uint8)))
    return m.astype(bool)


def gen_discretized_boundaries(values, counts, maximum_num_bins, min_obs_in_bins, special_values=()):
    """GenDiscretizedBoundaries on explicit (unique value, count) candidates (host)."""
    v = np.ascontiguousarray(values, dtype=np.float32)
    c = np.ascontiguousarray(counts, dtype=np.int64)
    sp = np.ascontiguousarray(special_values, dtype=np.float32)
    out = np.empty(len(v) + 2 * len(sp) + 4, np.float32)
    n = C.c_int32()
    st = lib().ygg_gen_discretized_boundaries(ptr(v, C.c_float), ptr(c, C.c_int64), C.c_int64(len(v)),
                                              C.c_int32(maximum_num_bins), C.c_int32(min_obs_in_bins),
                                              ptr(sp, C.c_float), C.c_int32(len(sp)), ptr(out, C.c_float),
                                              C.c_int32(len(out)), C.byref(n))
    if st != 0:
        raise YggError(st, "ygg_gen_discretized_boundaries: invalid argument")
    return out[:n.value].copy()


class Comm:
    """NCCL communicator owned by the native library (include/ygg_b200_comm.h): the collectives of the
    level loop are issued from C++ on the engine's stream.  `unique_id()` on rank 0, ship the 128 bytes
    to the other ranks (e.g. torch.distributed.broadcast), then Comm(id, rank, world, device)."""

    def __init__(self, unique_id: bytes, rank: int, world: int, device: int = 0):
        assert len(unique_id) == 128
        self.handle = C.c_void_p()
        self.rank, self.world = rank, world
        buf = (C.c_uint8 * 128).from_buffer_copy(unique_id)
        check(lib().ygg_comm_create(C.byref(self.handle), buf, C.c_int32(rank), C.c_int32(world),
                                    C.c_int32(device)))

    @staticmethod
    def unique_id() -> bytes:
        buf = (C.c_uint8 * 128)()
        check(lib().ygg_comm_unique_id(buf))
        return bytes(buf)

    @classmethod
    def from_torch_distributed(cls, device: int):
        """Bootstraps over an initialised torch.distributed process group (any backend)."""
        import torch
        import torch.distributed as dist
        rank, world = dist.get_rank(), dist.get_world_size()
        dev = torch.device(f"cuda:{device}") if dist.get_backend() == "nccl" else torch.device("cpu")
        t = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            t.copy_(torch.frombuffer(bytearray(cls.unique_id()), dtype=torch.uint8))
        dist.broadcast(t, src=0)
        return cls(bytes(t.cpu().numpy().tobytes()), rank, world, device)

    def close(self):
        if self.handle:
            lib().ygg_comm_destroy(self.handle)
            self.handle = C.c_void_p()


class Gbt:
    """Boosting state on one GPU (ygg_gbt)."""

    def __init__(self, dataset, cfg):
        self.dataset = dataset
        self.cfg = cfg
        self.handle = C.c_void_p()
        self._cb = None
        check(lib().ygg_gbt_create(C.byref(self.handle), dataset.handle, C.byref(cfg)))

    def close(self):
        if self.handle:
            lib().ygg_gbt_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_labels(self, labels):
        if self.cfg.loss in (0, 2):   # binomial {1, 2} / multinomial {1..K}
            l = np.ascontiguousarray(labels, dtype=np.int32)
            check(lib().ygg_gbt_set_labels_i32(self.handle, ptr(l, C.c_int32), C.c_int64(len(l))))
        else:
            l = np.ascontiguousarray(labels, dtype=np.float32)
            check(lib().ygg_gbt_set_labels_f32(self.handle, ptr(l, C.c_float), C.c_int64(len(l))))

    def set_weights(self, weights):
        """Example weights of the training rows (before set_labels): weighted histograms, leaves, losses, initial predictions."""
        w = np.ascontiguousarray(weights, dtype=np.float32)
        check(lib().ygg_gbt_set_weights_f32(self.handle, ptr(w, C.c_float), C.c_int64(len(w))))

    def set_validation(self, dataset, labels, weights=None):
        """Held-out rows (same features / binning): validation loss per iteration + cfg.early_stopping."""
        self._set_validation(dataset, labels)
        if weights is not None:
            w = np.ascontiguousarray(weights, dtype=np.float32)
            check(lib().ygg_gbt_set_validation_weights_f32(self.handle, ptr(w, C.c_float), C.c_int64(len(w))))

    def _set_validation(self, dataset, labels):
        self._valid = dataset
        if self.cfg.loss in (0, 2):
            l = np.ascontiguousarray(labels, dtype=np.int32)
            check(lib().ygg_gbt_set_validation_i32(self.handle, dataset.handle, ptr(l, C.c_int32), C.c_int64(len(l))))
        else:
            l = np.ascontiguousarray(labels, dtype=np.float32)
            check(lib().ygg_gbt_set_validation_f32(self.handle, dataset.handle, ptr(l, C.c_float), C.c_int64(len(l))))

    def validation_loss(self, it):
        a, b = C.c_float(), C.c_float()
        check(lib().ygg_gbt_validation_loss(self.handle, C.c_int32(it), C.byref(a), C.byref(b)))
        return a.value, b.value

    def num_iterations(self):
        return int(lib().ygg_gbt_num_iterations(self.handle))

    def final_validation(self):
        """-> (Header.validation_loss, Header.early_stopping_triggered)."""
        a, t = C.c_float(), C.c_int32()
        check(lib().ygg_gbt_final_validation(self.handle, C.byref(a), C.byref(t)))
        return a.value, bool(t.value)

    def set_feature_shard(self, begin, end, rank, world, allgather=None):
        """allgather: a Comm (NCCL, called from C++ without touching Python), or a Python callable
        allgather(send_ptr, recv_ptr, nbytes, stream_ptr) -> int, called once per tree level."""
        if isinstance(allgather, Comm):
            self._comm = allgather
            fn = C.cast(lib().ygg_comm_allgather, ALLGATHER_FN)
            check(lib().ygg_gbt_set_feature_shard(self.handle, C.c_int32(begin), C.c_int32(end),
                                                  C.c_int32(rank), C.c_int32(world), fn, allgather.handle))
            return
        if allgather is not None:
            def _cb(ctx, send, recv, nbytes, stream):
                try:
                    return int(allgather(send, recv, nbytes, stream) or 0)
                except Exception:  # never let an exception cross the C boundary
                    import traceback
                    traceback.print_exc()
                    return 1
            self._cb = ALLGATHER_FN(_cb)
            fn = self._cb
        else:
            fn = C.cast(None, ALLGATHER_FN)
        check(lib().ygg_gbt_set_feature_shard(self.handle, C.c_int32(begin), C.c_int32(end),
                                              C.c_int32(rank), C.c_int32(world), fn, None))

    def set_row_shard_scatter(self, rank, world, n_rows_global, initial_prediction, comm=None, allreduce=None,
                              reducescatter=None, allgather=None):
        """Row shards with one reduce-scatter (by feature chunk) + one all-gather of the best splits per level.
        Pass a Comm (NCCL from C++), or three Python callables (same conventions as set_row_shard /
        set_feature_shard; reducescatter(buf_ptr, count_per_rank, dtype, op, stream_ptr))."""
        if comm is not None:
            self._comm = comm
            fns = (C.cast(lib().ygg_comm_allreduce, ALLREDUCE_FN), C.cast(lib().ygg_comm_reducescatter, REDUCESCATTER_FN),
                   C.cast(lib().ygg_comm_allgather, ALLGATHER_FN))
            ctx = comm.handle
        elif allreduce is None:
            fns = (C.cast(None, ALLREDUCE_FN), C.cast(None, REDUCESCATTER_FN), C.cast(None, ALLGATHER_FN))
            ctx = None
        else:
            def wrap(fn, nargs):
                def _cb(ctx, *a):
                    try:
                        return int(fn(*a) or 0)
                    except Exception:
                        import traceback
                        traceback.print_exc()
                        return 1
                return _cb
            self._cbs = (ALLREDUCE_FN(wrap(allreduce, 5)), REDUCESCATTER_FN(wrap(reducescatter, 5)),
                         ALLGATHER_FN(wrap(allgather, 4)))
            fns, ctx = self._cbs, None
        check(lib().ygg_gbt_set_row_shard_scatter(self.handle, C.c_int32(rank), C.c_int32(world),
                                                  C.c_int64(n_rows_global), C.c_float(initial_prediction),
                                                  fns[0], fns[1], fns[2], ctx))

    def set_row_shard(self, rank, world, n_rows_global, initial_prediction, allreduce=None):
        """allreduce: a Comm (NCCL from C++), or a Python callable
        allreduce(buf_ptr, count, dtype, op, stream_ptr) -> int; dtype 0=u32 1=u64 2=f64, op 0=sum 1=max."""
        if isinstance(allreduce, Comm):
            self._comm = allreduce
            fn = C.cast(lib().ygg_comm_allreduce, ALLREDUCE_FN)
            check(lib().ygg_gbt_set_row_shard(self.handle, C.c_int32(rank), C.c_int32(world),
                                              C.c_int64(n_rows_global), C.c_float(initial_prediction), fn,
                                              allreduce.handle))
            return
        if allreduce is not None:
            def _cb(ctx, buf, count, dtype, op, stream):
                try:
                    return int(allreduce(buf, count, dtype, op, stream) or 0)
                except Exception:
                    import traceback
                    traceback.print_exc()
                    return 1
            self._cb = ALLREDUCE_FN(_cb)
            fn = self._cb
        else:
            fn = C.cast(None, ALLREDUCE_FN)
        check(lib().ygg_gbt_set_row_shard(self.handle, C.c_int32(rank), C.c_int32(world),
                                          C.c_int64(n_rows_global), C.c_float(initial_prediction), fn, None))

    def initial_prediction(self):
        v = C.c_float()
        check(lib().ygg_gbt_initial_prediction(self.handle, C.byref(v)))
        return v.value

    def train(self, num_iters, stop_flag=None):
        check(lib().ygg_gbt_train(self.handle, C.c_int32(num_iters), stop_flag))

    def train_timed(self, num_iters):
        """Returns (device milliseconds, kernel launches) for `num_iters` iterations."""
        ms, n = C.c_double(), C.c_int64()
        check(lib().ygg_gbt_train_timed(self.handle, C.c_int32(num_iters), C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def step(self):
        check(lib().ygg_gbt_step(self.handle))

    def sync(self):
        check(lib().ygg_gbt_sync(self.handle))

    def num_trees(self):
        return int(lib().ygg_gbt_num_trees(self.handle))

    def use_peer_windows(self, comm):
        """Best-split exchange over NVLink peer memory (ygg_gbt_set_best_split_window) instead of the all-gather."""
        L = lib()
        L.ygg_gbt_best_split_window_bytes.restype = C.c_int64
        nbytes = int(L.ygg_gbt_best_split_window_bytes(self.handle))
        peers = (C.c_void_p * comm.world)()
        check(L.ygg_comm_window_create(comm.handle, C.c_int64(nbytes), peers))
        check(L.ygg_gbt_set_best_split_window(self.handle, peers, C.c_int32(comm.world)))

    def set_tie_rng_position(self, words):
        check(lib().ygg_gbt_set_tie_rng_position(self.handle, C.c_uint64(int(words))))

    def tie_stats(self):
        """(renamed, unresolved) tied nodes of the trees trained so far (cfg.candidate_shuffle != 0)."""
        a, b = C.c_int64(), C.c_int64()
        check(lib().ygg_gbt_tie_stats(self.handle, C.byref(a), C.byref(b)))
        return a.value, b.value

    def get_tree(self, it):
        cap = (1 << (self.cfg.max_depth + (1 if self.cfg.growing_strategy == 1 else 0)))   # best-first: root depth 0
        out = np.zeros(cap, dtype=NODE_DTYPE)
        n = C.c_int32()
        check(lib().ygg_gbt_get_tree(self.handle, C.c_int32(it), out.ctypes.data_as(C.c_void_p),
                                     C.c_int32(cap), C.byref(n)))
        return out[:n.value].copy()

    def train_loss(self, it):
        a, b = C.c_float(), C.c_float()
        check(lib().ygg_gbt_train_loss(self.handle, C.c_int32(it), C.byref(a), C.byref(b)))
        return a.value, b.value

    def get_predictions(self):
        """Training predictions: [n]; multinomial loss: [n, K] (the engine holds them as K planes)."""
        k = self.cfg.num_classes if self.cfg.loss == 2 else 1
        out = np.empty(self.dataset.n_rows * k, dtype=np.float32)
        check(lib().ygg_gbt_get_predictions(self.handle, ptr(out, C.c_float), C.c_int64(len(out))))
        return out if k == 1 else np.ascontiguousarray(out.reshape(k, self.dataset.n_rows).T)

    def predict(self, dataset):
        """Raw scores of the trained model on `dataset` (same features / binning): [n], or [n, K] for the multinomial loss
        (the layout of get_predictions)."""
        n = int(lib().ygg_dataset_num_rows(dataset.handle))
        K = int(self.cfg.num_classes) if self.cfg.loss == 2 else 1
        out = np.empty(n * K, dtype=np.float32)
        check(lib().ygg_gbt_predict(self.handle, dataset.handle, ptr(out, C.c_float), C.c_int64(n * K)))
        return out if K == 1 else np.ascontiguousarray(out.reshape(K, n).T)

    def set_predictions(self, pred):
        p = np.ascontiguousarray(pred, dtype=np.float32)
        check(lib().ygg_gbt_set_predictions(self.handle, ptr(p, C.c_float), C.c_int64(len(p))))

    def train_tree_on_gradients(self, g, h=None):
        g = np.ascontiguousarray(g, dtype=np.float32)
        h = None if h is None else np.ascontiguousarray(h, dtype=np.float32)
        cap = (1 << (self.cfg.max_depth + (1 if self.cfg.growing_strategy == 1 else 0)))
        out = np.zeros(cap, dtype=NODE_DTYPE)
        n = C.c_int32()
        check(lib().ygg_tree_train_on_gradients(self.handle, ptr(g, C.c_float), ptr(h, C.c_float),
                                                out.ctypes.data_as(C.c_void_p), C.c_int32(cap),
                                                C.byref(n)))
        return out[:n.value].copy()

    def debug_capture_histograms(self, enabled=True):
        """While enabled, every tree grown records the slot histograms of each of its levels (debug_level_histograms)."""
        check(lib().ygg_gbt_debug_capture_histograms(self.handle, C.c_int32(int(enabled))))

    def debug_level_histograms(self, level):
        """The capture of `level` of the last tree grown with the capture on -> dict: the launch configuration
        (ygg_hist_level_info, "layout" as a name of HIST_LAYOUTS), the quantiser's inputs "g", "h2", "selected" [n_rows],
        and the planes "sum", "hsum" (None without a second plane), "cnt" as [slot, feature, 256] arrays (uint64 / uint32)
        with "slot_node" [slot] = the slot's node in the returned tree array."""
        info = HistLevelInfo()
        check(lib().ygg_gbt_debug_level_histograms(self.handle, C.c_int32(level), C.byref(info), None, None, None, None,
                                                   C.c_int32(0)))
        n, S, F = info.n_rows, info.num_slots, info.num_features
        g, h2, sel = np.empty(n, np.float32), np.empty(n, np.float32), np.empty(n, np.uint8)
        info.g, info.h2, info.selected = ptr(g, C.c_float), ptr(h2, C.c_float), ptr(sel, C.c_uint8)
        s = np.zeros((S, F, 256), np.uint64)
        hs = np.zeros((S, F, 256), np.uint64) if info.has_hsum else None
        c = np.zeros((S, F, 256), np.uint32)
        sn = np.zeros(S, np.int32)
        check(lib().ygg_gbt_debug_level_histograms(self.handle, C.c_int32(level), C.byref(info), ptr(s, C.c_uint64),
                                                   ptr(hs, C.c_uint64), ptr(c, C.c_uint32), ptr(sn, C.c_int32),
                                                   C.c_int32(S)))
        out = {k: getattr(info, k) for k, _ in HistLevelInfo._fields_ if k not in ("g", "h2", "selected")}
        out["layout"] = HIST_LAYOUTS[info.layout]
        out.update(g=g, h2=h2, selected=sel.astype(bool), sum=s, hsum=hs, cnt=c, slot_node=sn)
        return out

    def set_profiling(self, enabled=True):
        check(lib().ygg_gbt_set_profiling(self.handle, C.c_int32(int(enabled))))

    def get_profile(self, name):
        ms, n = C.c_double(), C.c_int64()
        check(lib().ygg_gbt_get_profile(self.handle, name.encode(), C.byref(ms), C.byref(n)))
        return ms.value, n.value


SHARD_BEST_DTYPE = np.dtype([("score", "<f4"), ("feature", "<i4"), ("threshold_bin", "<i4"),
                             ("num_pos_examples", "<i4"), ("condition_type", "<i4"), ("na_value", "<i4"),
                             ("cat_mask", "<u4", (8,))])
assert SHARD_BEST_DTYPE.itemsize == 56  # sizeof(ygg_shard_best)


def feature_shard(n_features, rank, world):
    b, e = C.c_int32(), C.c_int32()
    check(lib().ygg_feature_shard(C.c_int32(n_features), C.c_int32(rank), C.c_int32(world),
                                  C.byref(b), C.byref(e)))
    return b.value, e.value


def merge_shard_best(records):
    """records: [world, nodes] array of SHARD_BEST_DTYPE -> [nodes]."""
    r = np.ascontiguousarray(records, dtype=SHARD_BEST_DTYPE)
    world, nodes = r.shape
    out = np.zeros(nodes, dtype=SHARD_BEST_DTYPE)
    check(lib().ygg_merge_shard_best(r.ctypes.data_as(C.c_void_p), C.c_int32(world), C.c_int32(nodes),
                                     out.ctypes.data_as(C.c_void_p)))
    return out


def device_count():
    return int(lib().ygg_device_count())


def discretize_boundaries(values, maximum_num_bins=255, min_obs_in_bins=3):
    v = np.ascontiguousarray(values, dtype=np.float32)
    out = np.zeros(max(2, maximum_num_bins + 4), dtype=np.float32)
    n = C.c_int32()
    mean = C.c_double()
    check(lib().ygg_discretize_boundaries(ptr(v, C.c_float), C.c_int64(len(v)),
                                          C.c_int32(maximum_num_bins), C.c_int32(min_obs_in_bins),
                                          ptr(out, C.c_float), C.c_int32(len(out)), C.byref(n),
                                          C.byref(mean)))
    return out[:n.value].copy(), mean.value


def discretize_encode(values, boundaries, na_bin):
    v = np.ascontiguousarray(values, dtype=np.float32)
    b = np.ascontiguousarray(boundaries, dtype=np.float32)
    out = np.empty(len(v), dtype=np.uint8)
    check(lib().ygg_discretize_encode(ptr(v, C.c_float), C.c_int64(len(v)), ptr(b, C.c_float),
                                      C.c_int32(len(b)), C.c_int32(na_bin), ptr(out, C.c_uint8)))
    return out
