#!/usr/bin/env python
"""bench.py — boosting iterations/second of the GBT histogram split finder (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c3|c2] [--dump-outputs DIR]

A "step" is one boosting iteration (one tree) over the resident synthetic matrix.  Default workload
is BASELINE.json's headline configuration C3: 10M rows x 200 numerical features, 256 bins,
max_depth 8, binomial log-likelihood, variance gain (the reference's default split score).
One JSON line is printed by rank 0.  See DESIGN.md §7 for every field's definition.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: rows, features, max_depth, bins, informative features
    "c3": dict(rows=10_000_000, features=200, max_depth=8, bins=256, informative=20),
    "c2": dict(rows=1_000_000, features=50, max_depth=6, bins=255, informative=10),
    "tiny": dict(rows=200_000, features=16, max_depth=6, bins=255, informative=8),
    # BASELINE configs[4], within what the engine supports: 100 numerical + 50 categorical features (Zipf(1.2)
    # frequencies, cardinalities log-uniform in [100, 256] — the reference's config goes to 2000, which needs
    # the random-mask splitter, DESIGN.md §9), regression.  Not the headline metric: use --workload c5.
    "c5": dict(rows=10_000_000, features=150, categorical=50, max_depth=8, bins=256, informative=20, loss=1),
}
METRIC = "GBT boosting iters/sec, 10M rows x 200 num feats"   # BASELINE.json's metric (workload c3)


def _rows_name(n):
    return f"{n // 1_000_000}M" if n % 1_000_000 == 0 else (f"{n // 1000}k" if n % 1000 == 0 else str(n))


def metric_name(w):
    if w.get("categorical"):
        return (f"GBT boosting iters/sec, {_rows_name(w['rows'])} rows x {w['features'] - w['categorical']} num + "
                f"{w['categorical']} categorical feats, regression")
    if w["rows"] == 10_000_000 and w["features"] == 200:
        return METRIC
    return f"GBT boosting iters/sec, {_rows_name(w['rows'])} rows x {w['features']} num feats"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


class _near_gpu:
    """Context manager: run on the CPUs that are local to GPU `device` (sysfs local_cpulist of its PCI function); the
    previous affinity is restored on exit.  Best effort: any failure leaves the affinity alone."""

    def __init__(self, device):
        self.device, self.saved = device, None

    def __enter__(self):
        if self.device is None or not hasattr(os, "sched_setaffinity"):
            return self
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            index = int(visible.split(",")[self.device]) if visible and visible.split(",")[self.device].isdigit() else self.device
            bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(index)).busId
            bus = bus.decode() if isinstance(bus, bytes) else bus
            path = "/sys/bus/pci/devices/%s/local_cpulist" % bus[-12:].lower()
            cpus = set()
            for part in open(path).read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
            allowed = os.sched_getaffinity(0)
            cpus &= allowed
            if cpus:
                self.saved = allowed
                os.sched_setaffinity(0, cpus)
        except Exception:  # noqa: BLE001
            self.saved = None
        return self

    def __exit__(self, *exc):
        if self.saved is not None:
            os.sched_setaffinity(0, self.saved)
        return False


# ------------------------------------------------------------------------------------------------
# synthetic data (SURVEY.md §8d): X ~ N(0,1), y = 1[sum_j w_j x_j + 0.5 x0 x1 + 0.3 sin(3 x2) + eps > 0]
def make_data(w, device=None, binning=None):
    """Returns host arrays (bins uint8 [F, N] pinned if CUDA, num_bins, na_bin, labels int32 {1,2}).
    Columns are generated and bucketised with torch on the GPU when there is one (seconds instead
    of minutes); the result lives in HOST memory, which is what both arms start from.
    `binning`: the module whose discretize_boundaries() gives the boundaries — the product's host rule for
    our arm, oracle/binning.py (numpy restatement, bit-identical: tests/test_binning_kat.py) for the reference
    arm, which must not load the product library."""
    import torch
    if binning is None:
        import ydf_b200 as binning
    n, f = w["rows"], w["features"]
    use_cuda = device is not None and torch.cuda.is_available()
    dev = torch.device(f"cuda:{device}") if use_cuda else torch.device("cpu")
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234)
    wrng = np.random.default_rng(1234)
    wvec = wrng.normal(size=w["informative"])
    # pinned pages are placed where the allocating thread runs: allocate them on the GPU's own NUMA node (an upload that
    # crosses the socket interconnect ran at 12-17 GB/s on some boxes of the pool, 50 GB/s locally)
    with _near_gpu(device if use_cuda else None):
        bins = torch.empty((f, n), dtype=torch.uint8, pin_memory=use_cuda)
    margin = torch.zeros(n, dtype=torch.float32, device=dev)
    num_bins, na_bin = [], []
    x01 = {}
    n_cat = w.get("categorical", 0)
    w["feature_types"] = None if not n_cat else [0] * (f - n_cat) + [1] * n_cat
    for j in range(f):
        if j >= f - n_cat:
            # categorical column: dictionary indices 1..k-1 by decreasing Zipf(1.2) frequency (index 0 = OOD, unused),
            # 5 % missing -> most_frequent_value = 1, a random effect N(0, 0.3^2) per category on the target
            k = int(round(float(np.exp(wrng.uniform(np.log(100), np.log(256))))))
            pk = 1.0 / np.arange(1, k) ** 1.2
            cdf = torch.from_numpy(np.cumsum(pk / pk.sum())).to(dev, torch.float32)
            u = torch.rand(n, generator=gen, device=dev)
            c = (torch.bucketize(u, cdf, right=True).clamp_(max=k - 2) + 1).to(torch.int64)
            eff = torch.from_numpy(wrng.normal(scale=0.3, size=k).astype(np.float32)).to(dev)
            margin += eff[c]
            miss = torch.rand(n, generator=gen, device=dev) < 0.05
            c[miss] = 1
            bins[j].copy_(c.to(torch.uint8))
            num_bins.append(k)
            na_bin.append(1)
            continue
        x = torch.randn(n, generator=gen, device=dev, dtype=torch.float32)
        sample = x[:100_000].cpu().numpy()
        b, mean = binning.discretize_boundaries(sample, w["bins"], 3)
        nb = len(b) + 1
        nab = int(np.searchsorted(b, np.float32(mean), side="right"))
        bt = torch.from_numpy(b).to(dev)
        enc = torch.bucketize(x, bt, right=True).to(torch.uint8)  # upper_bound, data_spec.cc:1006-1018
        bins[j].copy_(enc)
        num_bins.append(nb)
        na_bin.append(nab)
        if j < w["informative"]:
            margin += float(wvec[j]) * x
        if j < 3:
            x01[j] = x
    if f >= 3:
        margin += 0.5 * x01[0] * x01[1] + 0.3 * torch.sin(3 * x01[2])
    margin += 0.5 * torch.randn(n, generator=gen, device=dev, dtype=torch.float32)
    if w.get("loss", 0) == 1:
        labels = margin.cpu().numpy().astype(np.float32)      # regression target
    else:
        labels = (margin > 0).to(torch.int32).cpu().numpy() + 1
    if use_cuda:
        torch.cuda.synchronize()
    return bins.numpy(), np.array(num_bins, np.int32), np.array(na_bin, np.int32), labels


class ClockSampler:
    """Samples SM clocks / throttle reasons of the job's GPUs during the timed region
    (B200_PROFILING.md clocks line).  NVML in-process (the source nvidia-smi itself reads); one
    sampler on rank 0 covers every GPU of the job, so no rank forks a subprocess while timing."""
    REASONS = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
               "sw_power_cap": 0x4}

    def __init__(self, gpus):
        self.gpus = list(gpus)
        self.rows = []
        self.first = 0
        self.stop_flag = threading.Event()
        self.t = None

    def start(self):
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            self.nv = pynvml
            self.handles = []
            for i in self.gpus:  # CUDA ordinal -> NVML handle through the PCI bus id
                pr = torch.cuda.get_device_properties(i)
                bus = "%08X:%02X:%02X.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
                try:
                    self.handles.append(pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode()))
                except Exception:
                    self.handles.append(pynvml.nvmlDeviceGetHandleByIndex(i))
        except Exception:
            self.nv = None
            return
        self.t = threading.Thread(target=self._loop, daemon=True)
        self.t.start()

    def _sample(self):
        nv = self.nv
        for h in self.handles:
            try:
                self.rows.append((nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM),
                                  nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM),
                                  nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)))
            except Exception:
                pass

    def _loop(self):
        while not self.stop_flag.is_set():
            self._sample()
            self.stop_flag.wait(0.05)

    def mark(self):
        """Samples taken before this call (warm-up) are dropped from the summary."""
        self.first = len(self.rows)

    def stop(self):
        if self.t is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["NVML unavailable"]}
        self._sample()
        self.stop_flag.set()
        self.t.join(timeout=2)
        rows = self.rows[self.first:]
        reasons = sorted(n for n, bit in self.REASONS.items() if any(r[2] & bit for r in rows))
        return {"sm_mhz": float(np.median([r[0] for r in rows])) if rows else None,
                "sm_max_mhz": float(max(r[1] for r in rows)) if rows else None, "samples": len(rows),
                "reasons": reasons, "source": "NVML, sampled on rank 0 for all GPUs of the job"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p))["hbm_gbs"], "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def gbt_config(w, steps_total):
    import ydf_b200
    return ydf_b200.default_config(loss=w.get("loss", 0), num_trees=steps_total, max_depth=w["max_depth"],
                                   shrinkage=0.1, min_examples=5, use_hessian_gain=int(w.get("hessian", 0)))


def hist_bytes_per_level(w, f_local=None):
    # SURVEY.md §8d: one level reads every active row of every feature once: N * (F*1 B + 4 B
    # gradient + 4 B row/node id).  The kernel's own traffic is N * (F + 4) (a packed 4-byte
    # rowinfo word per row), re-read per feature group from L2.
    f = w["features"] if f_local is None else f_local
    return w["rows"] * (f + 8 + (4 if w.get("hessian") else 0))   # + 4 B hessian per row with hessian gain


# ------------------------------------------------------------------------------------------------
# CPU legs.  Everything below runs the oracle port (oracle/ygg_oracle.cc) or, when importable, the real YDF.
def workload_text(name, w):
    loss = "squared error" if w.get("loss", 0) == 1 else "binomial log-likelihood"
    gain = "hessian" if w.get("hessian") else "variance"
    cat = f", {w['categorical']} of the features categorical (100-256 values, CART)" if w.get("categorical") else ""
    return f"{name}: {w['rows']}x{w['features']} u8 bins({w['bins']}), GBT depth {w['max_depth']}, {loss}, {gain} gain{cat}"


class CpuPort:
    """The oracle port on ALL rows of the workload, all host threads, one boosting iteration per call
    (gradients -> tree -> prediction update -> training loss, as gradient_boosted_trees.cc:1428-1580).
    Set-up (u16 copy of the matrix: the reference's storage type, dataset/data_spec.h:45-48) is outside the timing."""

    def __init__(self, w, bins, num_bins, na_bin, labels, threads=None):
        from oracle import oracle as O
        self.O = O
        self.build = O.use_native_build()
        self.threads = threads or O.max_threads()
        self.cfg = O.default_config(loss=w.get("loss", 0), max_depth=w["max_depth"], shrinkage=0.1, min_examples=5,
                                    use_hessian_gain=int(w.get("hessian", 0)))
        self.ft = w.get("feature_types")
        self.b16 = np.ascontiguousarray(bins, dtype=np.uint16)
        self.nb, self.na, self.labels = num_bins, na_bin, labels
        self.pred = None
        self.trees, self.loss, self.seconds = [], [], []
        self.stable_sort = any(t == 1 for t in (self.ft or []))
        if self.stable_sort:
            O.set_stable_category_sort(True)   # the order the engine's in-kernel sort gives to equal keys (DESIGN.md §6)

    def close(self):
        if self.stable_sort:
            self.O.set_stable_category_sort(False)
            self.stable_sort = False
        self.b16 = None

    def step(self):
        t0 = time.perf_counter()
        r = self.O.gbt_train(self.b16, self.nb, self.na, self.labels, self.cfg, 1, num_threads=self.threads,
                             predictions=self.pred, feature_type=self.ft)
        dt = time.perf_counter() - t0
        self.pred = r["predictions"]
        self.trees.append(r["trees"][0])
        self.loss.append(float(r["loss"][0]))
        self.seconds.append(dt)
        return dt

    def baseline(self, first, w):
        sec = self.seconds[first:]
        v = len(sec) / sum(sec)
        return {"value": v, "unit": "iters/s", "cores": self.threads, "kind": "port",
                "sample": f"{len(sec)} full boosting iterations on ALL {w['rows']} rows x {w['features']} features "
                          f"(no sampling, no extrapolation), {self.threads} threads, {self.build}",
                "seconds_per_iteration": [round(x, 4) for x in sec]}


def tree_hash(trees):
    """sha256 over what defines the trees: structure, counts, float bits of scores and leaf values."""
    import hashlib
    h = hashlib.sha256()
    for t in trees:
        for k in ("feature", "threshold_bin", "na_value", "num_examples", "num_pos_examples", "condition_type",
                  "split_score", "leaf_value", "cat_mask"):
            h.update(np.ascontiguousarray(t[k]).tobytes())
    return h.hexdigest()[:16]


def parity_block(gpu_trees, cpu_trees, gpu_loss, cpu_loss, score_rel=1e-5, note=None):
    """SURVEY.md §8(d) 'parity check in the same run': per node (feature, threshold bin, na_value, counts) exact,
    split_score relative, leaf value absolute, training loss relative."""
    out = {"trees_compared": len(cpu_trees), "structure_mismatches": 0, "nodes_compared": 0, "max_score_rel_err": 0.0,
           "max_leaf_abs_err": 0.0, "max_loss_rel_err": 0.0, "tolerance": {"score_rel": score_rel, "leaf_abs": 1e-5},
           "checker": "oracle port (oracle/ygg_oracle.cc), same rows, closed loop from iteration 0"}
    if note:
        out["note"] = note
    for a, b in zip(gpu_trees, cpu_trees):
        if len(a) != len(b):
            out["structure_mismatches"] += abs(len(a) - len(b)) + 1
            continue
        out["nodes_compared"] += len(a)
        for k in ("feature", "threshold_bin", "na_value", "num_examples", "num_pos_examples", "condition_type"):
            out["structure_mismatches"] += int(np.count_nonzero(a[k] != b[k]))
        out["structure_mismatches"] += int(np.count_nonzero((a["cat_mask"] != b["cat_mask"]).any(axis=1)))
        sp = b["feature"] >= 0
        if sp.any():
            rel = np.abs(a["split_score"][sp].astype(np.float64) - b["split_score"][sp]) / np.maximum(np.abs(b["split_score"][sp]), 1e-30)
            out["max_score_rel_err"] = max(out["max_score_rel_err"], float(rel.max()))
        out["max_leaf_abs_err"] = max(out["max_leaf_abs_err"], float(np.abs(a["leaf_value"].astype(np.float64) - b["leaf_value"]).max()))
    for x, y in zip(gpu_loss, cpu_loss):
        out["max_loss_rel_err"] = max(out["max_loss_rel_err"], abs(x - y) / max(abs(y), 1e-30))
    out["ok"] = bool(out["structure_mismatches"] == 0 and out["max_score_rel_err"] <= score_rel and out["max_leaf_abs_err"] <= 1e-5)
    return out


def try_real_ydf(w, bins, labels, steps):
    """BASELINE.md §4 step 1: if the real YDF is importable on this box, time IT (the unmodified reference, CPU)."""
    try:
        import ydf  # noqa: F401
    except Exception as e:  # noqa: BLE001
        return None, f"import ydf failed: {type(e).__name__}"
    try:
        import pandas as pd
        # the bucket indices as numerical columns: 256 distinct integers per column, discretized again by YDF
        # into one bucket per value = the same candidate cuts as the u8 matrix
        df = pd.DataFrame({f"f{j}": bins[j].astype(np.float32) for j in range(bins.shape[0])})
        df["label"] = labels
        task = ydf.Task.REGRESSION if w.get("loss", 0) == 1 else ydf.Task.CLASSIFICATION
        learner = ydf.GradientBoostedTreesLearner(
            label="label", task=task, num_trees=steps, max_depth=w["max_depth"], shrinkage=0.1, min_examples=5,
            discretize_numerical_columns=True, num_discretized_numerical_bins=256, validation_ratio=0.0,
            early_stopping="NONE", use_hessian_gain=bool(w.get("hessian", 0)), num_threads=os.cpu_count())
        t0 = time.perf_counter()
        learner.train(df)
        dt = time.perf_counter() - t0
        return {"value": steps / dt, "seconds": dt, "cores": os.cpu_count()}, "ydf " + getattr(ydf, "__version__", "?")
    except Exception as e:  # noqa: BLE001
        return None, f"ydf present but the run failed: {type(e).__name__}: {e}"


def run_reference(args, w):
    """--impl reference: the reference's CPU path on the box's host cores, SAME configuration as our arm: all rows,
    K timed full-size boosting iterations after W warm-up iterations.  The real YDF when importable, else the
    oracle port.  The product library is never loaded in this process."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from oracle import binning
    dev = 0 if torch.cuda.is_available() else None
    bins, nb, na, labels = make_data(w, dev, binning=binning)
    K, W = max(1, args.steps), max(0, args.warmup)
    ydf_res, ydf_note = try_real_ydf(w, bins, labels, K) if not args.no_ydf_probe else (None, "probe disabled")
    t_wall = time.perf_counter()
    if ydf_res is not None:
        v = ydf_res["value"]
        cpu = {"value": v, "unit": "iters/s", "cores": ydf_res["cores"], "kind": "reference",
               "sample": f"{K} trees by {ydf_note} on all rows, training time / trees"}
        steps_done, warm_done = K, 0
    else:
        port = CpuPort(w, bins, nb, na, labels)
        cap_s = float(os.environ.get("YGG_BENCH_REF_MAX_S", "600"))
        warm_done = 0
        for _ in range(W):
            port.step()
            warm_done += 1
            if sum(port.seconds) > cap_s / 4:
                break
        steps_done = 0
        for _ in range(K):
            port.step()
            steps_done += 1
            if sum(port.seconds) > cap_s:   # safety net only; the default sizes finish far below it
                break
        cpu = port.baseline(warm_done, w)
        v = cpu["value"]
    line = {"impl": "reference", "reference_kind": cpu["kind"], "ydf_probe": ydf_note, "same_config": True,
            "rows_sampled_fraction": 1.0,
            "metric": metric_name(w), "value": v, "unit": "iters/s", "n_gpus": args.gpus,
            "steps": steps_done, "warmup": warm_done, "ms_per_step": 1000.0 / v, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_text(args.workload, w)},
            "cpu_baseline": cpu,
            "e2e": {"value": v, "unit": "iters/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "wall_s": time.perf_counter() - t_wall}
    emit(line)


# ------------------------------------------------------------------------------------------------
def run_ours(args, w):
    import torch
    import ydf_b200
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available() or ydf_b200.device_count() == 0:
        raise SystemExit("bench.py: no CUDA device — the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    K, W = args.steps, max(3, args.warmup)
    bins, nb, na, labels = make_data(w, local_rank)
    F = w["features"]
    f_begin, f_end = (F * rank) // world, (F * (rank + 1)) // world

    class _Buf:  # device pointer -> torch tensor via the CUDA array interface
        def __init__(self, p, n, typestr):
            self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (p, False), "version": 2}

    def allgather(send, recv, nbytes, stream):
        with torch.cuda.stream(torch.cuda.ExternalStream(stream)):
            r = torch.as_tensor(_Buf(recv, nbytes * world, "|u1"), device=f"cuda:{local_rank}")
            dist.all_gather_into_tensor(r, r[rank * nbytes:(rank + 1) * nbytes])
        return 0

    def allreduce(buf, count, dtype, op, stream):
        # two's-complement sums of u32/u64 are bit-identical to the unsigned sums; max is only used on
        # the bits of a non-negative float
        typestr = {0: "<i4", 1: "<i8", 2: "<f8"}[dtype]
        with torch.cuda.stream(torch.cuda.ExternalStream(stream)):
            t = torch.as_tensor(_Buf(buf, count, typestr), device=f"cuda:{local_rank}")
            dist.all_reduce(t, op=dist.ReduceOp.SUM if op == 0 else dist.ReduceOp.MAX)
        return 0

    comm = None
    if world > 1 and args.comm == "nccl":
        # the production path: NCCL called from C++ on the engine's stream (include/ygg_b200_comm.h);
        # torch.distributed only bootstraps the unique id and provides the timing barrier
        comm = ydf_b200.Comm.from_torch_distributed(local_rank)
    row_mode = world > 1 and args.shard == "rows"
    n_all = bins.shape[1]
    r0, r1 = (n_all * rank) // world, (n_all * (rank + 1)) // world
    my_bins = bins[:, r0:r1] if row_mode else bins
    my_labels = labels[r0:r1] if row_mode else labels
    if w.get("loss", 0) == 1:
        init_pred = float(np.float32(labels.astype(np.float64).mean()))   # loss_imp_mean_square_error.cc:56-88
    else:
        ratio = float((labels == 2).mean(dtype=np.float64))
        init_pred = float(np.float32(np.log(ratio / (1.0 - ratio))))  # loss_imp_binomial.cc:65-99 on the whole job

    def make_gbt(dataset, total):
        g = ydf_b200.Gbt(dataset, gbt_config(w, total))
        g.set_labels(my_labels)
        if world > 1:
            if row_mode:
                if comm is not None and args.scatter:
                    g.set_row_shard_scatter(rank, world, n_all, init_pred, comm)
                    if args.p2p:
                        g.use_peer_windows(comm)   # best splits over NVLink peer memory inside k_select_global
                else:
                    g.set_row_shard(rank, world, n_all, init_pred, comm or allreduce)
            else:
                g.set_feature_shard(f_begin, f_end, rank, world, comm or allgather)
                if comm is not None and args.p2p:
                    g.use_peer_windows(comm)
        return g

    # ---- device-resident throughput ("value") ----
    dataset = ydf_b200.Dataset(my_bins, nb, na, device=local_rank, feature_types=w.get("feature_types"))
    gbt = make_gbt(dataset, W + K + K + 1)
    sampler = ClockSampler(range(world) if rank == 0 else [])   # one in-process NVML sampler for the whole job
    sampler.start()          # started before the warm-up so that its start-up cost is outside the timed region
    gbt.train_timed(W)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.mark()
    ms, launches = gbt.train_timed(K)
    torch.cuda.synchronize()
    clocks = sampler.stop()
    t = torch.tensor([ms], dtype=torch.float64, device=f"cuda:{local_rank}")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = K / (ms / 1000.0)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, gbt)

    # ---- per-kernel device time for the roofline (separate profiled run of K steps) ----
    gbt.set_profiling(True)
    ms_profiled, _ = gbt.train_timed(K)
    prof = {k: gbt.get_profile(k) for k in ["grad", "hist", "scan", "select", "partition", "allreduce"] +
            [f"hist_L{i}" for i in range(w["max_depth"] - 1)]}
    gbt.set_profiling(False)
    hist_ms, hist_launches = prof["hist"]
    levels = w["max_depth"] - 1
    if row_mode:
        bytes_per_launch = (r1 - r0) * (F + 8)
    else:
        bytes_per_launch = hist_bytes_per_level(w, f_end - f_begin)
    n_hist_kernels = K * levels
    hist_ms_per_launch = hist_ms / n_hist_kernels
    peak, peak_src = peaks()
    achieved = bytes_per_launch / (hist_ms_per_launch * 1e-3) / 1e9
    # the first P trees of this handle are the model's first P trees (the warm-up started at iteration 0)
    P = parity_trees(args, w)
    trees = [gbt.get_tree(i) for i in range(min(max(3, P), gbt.num_trees()))]
    first_losses = [gbt.train_loss(i)[0] for i in range(min(P, gbt.num_trees()))]
    loss_last = gbt.train_loss(gbt.num_trees() - 1)
    gbt.close()
    dataset.close()

    # ---- end to end through the C ABI from host buffers ("e2e") ----
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    d2 = ydf_b200.Dataset(my_bins, nb, na, device=local_rank, feature_types=w.get("feature_types"))  # H2D of the bucketised matrix (this rank's shard)
    t1 = time.perf_counter()
    g2 = make_gbt(d2, K)                                       # H2D of the labels
    t2 = time.perf_counter()
    g2.train(K)
    t3 = time.perf_counter()
    d2h = 0
    for i in range(K):
        d2h += g2.get_tree(i).nbytes                           # D2H of every tree
    l_e2e = g2.train_loss(K - 1)
    d2h += 8
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    e2e_phases = {"dataset_create_s": t1 - t0, "gbt_create_labels_s": t2 - t1, "train_s": t3 - t2,
                  "fetch_trees_s": e2e_s - (t3 - t0)}
    te = torch.tensor([e2e_s], dtype=torch.float64, device=f"cuda:{local_rank}")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_s = float(te.item())
    h2d = (my_bins.shape[0] * my_bins.shape[1] + my_labels.nbytes) * (world if row_mode else 1)
    g2.close()
    d2.close()

    # ---- CPU leg in the same run (N = 1, rank 0): the oracle port grows the first P trees on ALL rows; its trees
    # are the parity checker of the GPU's first P trees, its clock is the cpu_baseline ----
    cpu = parity = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and P > 0:
        port = CpuPort(w, bins, nb, na, labels)
        for _ in range(P):
            port.step()
        cpu = port.baseline(0, w)
        if w.get("hessian"):
            # the reference sums its hessian-gain buckets in float32 in row order: ITS scores carry 1e-6..1e-3 of
            # order-dependent noise at these sizes (tests/test_gpu_baseline_parity.py holds the engine to 1e-5 against
            # exact buckets); the port timed here is the reference arithmetic, so the score bar is the noise's
            parity = parity_block(trees[:P], port.trees, first_losses, port.loss, score_rel=2e-3,
                                  note="hessian gain: float32 bucket sums in the reference arithmetic (order-dependent)")
        else:
            parity = parity_block(trees[:P], port.trees, first_losses, port.loss)
        port.close()

    if rank == 0:
        line = {
            "metric": metric_name(w), "value": value, "unit": "iters/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "strong" if world > 1 else "weak",
            "vs_baseline": None, "dtype": "int64 fixed-point sums (q24 gradients), f64 split scores",
            "data": "synthetic",
            "config": {"workload": workload_text(args.workload, w) + ", sibling subtraction",
                       "parallelism": ((f"row-shard x{world}, NCCL reduce-scatter of the integer level histograms by feature chunk, sharded scan, "
                                         f"best splits exchanged over NVLink peer memory inside k_select_global" + ("" if args.p2p else " (off: NCCL all-gather)") if (comm is not None and args.scatter) else
                                         f"row-shard x{world}, NCCL all-reduce of the integer level histograms") if row_mode
                                       else f"feature-shard x{world}, NCCL all-gather of best splits") if world > 1 else "single GPU",
                       "collectives": ("NCCL from C++ on the engine stream (ygg_b200_comm.h)" if comm is not None else
                                       "torch.distributed from Python callbacks") if world > 1 else "none",
                       "l2_flush": "inputs (2 GB bins + 40 MB rowinfo per level) exceed the 126 MB L2",
                       "timing": "CUDA events on the engine stream, max over ranks"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "k_hist", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "peak_source": peak_src,
                         # dram__bytes_read.sum + dram__bytes_write.sum per launch of the committed ncu capture of this
                         # workload (profiles/k_hist_traffic.json, written from the .ncu-rep by tools/ncu_traffic.py)
                         "traffic": measured_traffic(args, w, world),
                         "bytes_per_launch": bytes_per_launch, "ms_per_launch": hist_ms_per_launch,
                         "launches": n_hist_kernels},
            "kernel_ms_per_step": {k: v[0] / K for k, v in prof.items()},
            "ms_per_step_profiled_pass": ms_profiled / K,
            "e2e": {"value": K / e2e_s, "unit": "iters/s", "h2d_bytes_per_step": h2d / K,
                    "d2h_bytes_per_step": d2h / K, "seconds": e2e_s, "phases": e2e_phases,
                    "includes": "dataset H2D, labels H2D, K iterations, trees + loss D2H"},
            "train_loss_last": loss_last[0], "e2e_train_loss_last": l_e2e[0],
            "tree0_nodes": int(len(trees[0])) if trees else 0,
            # identical at every N when the trees are (integer histograms: rank-count invariant by construction)
            "tree_hash": {"trees": len(trees), "sha256_16": tree_hash(trees)},
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
            line["parity"] = parity
        emit(line)
    if world > 1:
        dist.barrier()
        if comm is not None:
            comm.close()
        dist.destroy_process_group()


DUMP_MAX_PREDICTIONS = 15_000_000   # 60 MB of float32: every row of the 10M-row workloads; the tree adds < 0.1 MB


def dump_outputs(out_dir, gbt):
    """Writes what the last timed iteration gave its caller, as float64 / float32 .npy files in `out_dir`: the tree
    (tree_<field>.npy, one file per field of NODE_DTYPE but threshold_value, which include/ygg_b200.h defines as NaN
    on every node of a dataset without bucket values, as here: threshold_bin holds the split), its training loss and
    secondary metric (train_loss.npy) and
    the training predictions after it (predictions.npy; rank 0's rows when the rows are sharded).  Of more than
    DUMP_MAX_PREDICTIONS predictions, those of DUMP_MAX_PREDICTIONS rows drawn with a fixed seed are kept, in row
    order: the same rows in every run with the same number of rows."""
    os.makedirs(out_dir, exist_ok=True)
    it = gbt.num_trees() - 1
    tree = gbt.get_tree(it)
    for k in tree.dtype.names:
        if k == "threshold_value":
            continue
        np.save(os.path.join(out_dir, f"tree_{k}.npy"), tree[k].astype(np.float64))
    np.save(os.path.join(out_dir, "train_loss.npy"), np.array(gbt.train_loss(it), np.float64))
    pred = gbt.get_predictions()
    if len(pred) > DUMP_MAX_PREDICTIONS:
        pred = pred[np.sort(np.random.default_rng(0).choice(len(pred), DUMP_MAX_PREDICTIONS, replace=False))]
    np.save(os.path.join(out_dir, "predictions.npy"), pred.astype(np.float32))
    log(f"bench.py: outputs of iteration {it} written to {out_dir}")


def parity_trees(args, w):
    """Trees compared with the oracle in the same run: 20 at C2 (SURVEY.md §8d), 2 at the 10M-row workloads (a CPU
    iteration takes seconds there)."""
    if args.parity_trees is not None:
        return max(0, args.parity_trees)
    return 2 if w["rows"] * w["features"] > 200_000_000 else 20


def measured_traffic(args, w, world):
    if world != 1 or args.rows or args.features:
        return None
    p = os.path.join(ROOT, "profiles", "k_hist_traffic.json")
    if not os.path.exists(p):
        return None
    key = args.workload + ("_hessian" if w.get("hessian") else "")
    rec = json.load(open(p)).get(key)
    return None if rec is None else rec["dram_bytes_per_launch"]


_REAL_STDOUT = None


def emit(line: dict):
    """The ONE JSON line goes to the process's original stdout; everything else any library prints
    (NCCL's version banner, torchrun notices) has been redirected to stderr in main()."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)  # fd 1 -> stderr for the rest of the run
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--rows", type=int, default=None)
    ap.add_argument("--features", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--parity-trees", type=int, default=None,
                    help="first trees compared with the oracle in the same run (default: 20 at C2, 2 at 10M rows)")
    ap.add_argument("--no-ydf-probe", action="store_true", help="reference arm: do not try `import ydf`")
    ap.add_argument("--use-hessian-gain", action="store_true",
                    help="hessian gain instead of the reference default (variance gain): one more histogram word per bin")
    ap.add_argument("--scatter", type=int, default=1,
                    help="row shards: 1 = reduce-scatter by feature chunk + sharded scan + all-gather of the bests "
                         "(default), 0 = one all-reduce of the level histograms and a replicated scan")
    ap.add_argument("--p2p", type=int, default=1,
                    help="N>1: 1 = the best splits of a level are exchanged by k_select_global itself over NVLink peer memory "
                         "(CUDA IPC windows; default), 0 = NCCL all-gather")
    ap.add_argument("--comm", default="nccl", choices=["nccl", "torch"],
                    help="N>1: collectives issued by the native library through NCCL (default) or by "
                         "torch.distributed from Python callbacks (A/B)")
    ap.add_argument("--shard", default="rows", choices=["rows", "features"],
                    help="multi-GPU decomposition: rows (histogram all-reduce) or features (best-split all-gather)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the tree, training loss and predictions of the last timed iteration to DIR as .npy "
                         "(at most 64 MB), to compare two builds on the same seeded inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps the GPU path (--impl ours)")
    w = dict(WORKLOADS[args.workload])
    if args.rows:
        w["rows"] = args.rows
    if args.features:
        w["features"] = args.features
        w["informative"] = min(w["informative"], args.features)
    if args.use_hessian_gain:
        w["hessian"] = 1
    if args.impl == "reference":
        run_reference(args, w)
    else:
        run_ours(args, w)


if __name__ == "__main__":
    main()
