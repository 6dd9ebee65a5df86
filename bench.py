#!/usr/bin/env python
"""Benchmark of the sknnr query-time hot path (kneighbors + predict, k=7) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Headline workload (BASELINE.json configs[2], "C3"): EuclideanKNNRegressor, 10M query rows x
50k reference plots x 32 features, k=7, predict(weights="distance") over 8 targets; synthetic
N(0,1) data with the seeds of BASELINE.md section 3.  One "step" = one pass of the hot path
over the whole 10M-row query batch of a rank.  N > 1: every rank holds the full reference set
and its own 10M-row shard (weak scaling); every rank's rows land in rank 0's result arrays
(CUDA IPC mapping) over NVLink inside the timed region: as per-chunk copy-engine peer copies
under the next chunks' kernels (default), or stored by the finishing kernels themselves
(--gather fused; the mode not chosen is timed right behind the headline as `gather_alt`).

`value`   : device-resident inputs/outputs (queries/s, whole job).
`e2e`     : the same through the host-buffer C-ABI call, pinned host inputs/outputs, H2D/D2H
            copies inside the timed region.
`e2e_estimator`: the same through `EuclideanKNNRegressor.predict(X)` on an ordinary (pageable)
            NumPy array - the call a user of the drop-in makes.
`roofline`: the dominant kernel (fused FP16 tcgen05 distance + top-k filter) against the measured
            dense 16-bit tensor peak of MEASURED_PEAKS.json (plus a cuBLAS TF32 figure measured here).
`c5`, `c4`: sub-records for BASELINE.json configs[4] (Mahalanobis, 100M x 50k x 64, rows split
            over the ranks) and configs[3] (RFNN, 500 trees, 20k plots, raw rows -> forest walk ->
            Hamming search), each with its own roofline and CPU baseline.
`cpu_baseline` / `--impl reference`: the UNMODIFIED reference package (oracle/_ref/sknnr, installed
            by __graft_entry__.build()) on the box's host cores, on a bounded sample.

--steps K sets the number of timed steps of every leg.  --dump-outputs DIR writes, after each leg's
timed steps, what its last step returned - (dist, idx, pred) of a fixed, seeded sample of rows and the
sample's row numbers - as DIR/<leg>_<name>.npy in float64 (64 MB in all at most).  The inputs depend on
the arguments only, so two builds can be compared output for output.
"""

from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "query-neighbors/sec (kneighbors+predict, k=7)"
UNIT = "queries/s"
LANE_OPS_PEAK = 148 * 128 * 1.965e9      # SURVEY.md section 8d: integer lane-ops/s of one B200


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n-queries", type=int, default=10_000_000)
    ap.add_argument("--n-ref", type=int, default=50_000)
    ap.add_argument("--dim", type=int, default=32)
    ap.add_argument("--n-out", type=int, default=8)
    ap.add_argument("--k", type=int, default=7)
    ap.add_argument("--cpu-sample", type=int, default=600_000)
    ap.add_argument("--ref-sample", type=int, default=400_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-est", action="store_true")
    ap.add_argument("--no-c4", action="store_true")
    ap.add_argument("--no-c5", action="store_true")
    ap.add_argument("--no-peaks", action="store_true")
    ap.add_argument("--only", default="", help="c3 | c4 | c5: run one workload alone (profiling)")
    ap.add_argument("--c5-rows", type=int, default=100_000_000)
    ap.add_argument("--c4-rows", type=int, default=2_000_000)
    ap.add_argument("--engine", type=int, default=0)
    ap.add_argument("--kc", type=int, default=0)
    ap.add_argument("--tc-seed-stride", type=int, default=-1)
    ap.add_argument("--tc-streams", type=int, default=0)
    ap.add_argument("--tc-debug", type=int, default=0)
    ap.add_argument("--chunk-rows", type=int, default=0)
    ap.add_argument("--host-slots", type=int, default=0)
    ap.add_argument("--opt", action="append", default=[], metavar="NAME=VALUE",
                    help="library option for an experiment (sknnr_set_option), repeatable")
    ap.add_argument("--no-gather-ab", action="store_true", help="N > 1: do not time the other gather mode as well")
    ap.add_argument("--gather", default="auto", choices=["auto", "fused", "copy"],
                    help="N > 1: how a rank's rows reach rank 0's arrays - fused = the finishing kernels store "
                         "over NVLink; copy = per-chunk copy-engine peer copies on the chunk's stream")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write a seeded sample of each leg's last timed step's results to DIR/<leg>_<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes what this project's timed path returns; --impl reference has no such path")
    if a.gather == "auto":
        # measured on 8 GPUs (profiles/r02_multi_gpu_gather.md): copy 83.4 ms per step against 88.6 fused and
        # 82.4 on one GPU - the ranks run in step, so seven ranks' finishing kernels store into rank 0 at
        # once (7 x ~195 GB/s against 900 GB/s of NVLink ingress) while the copy engines spread the same
        # bytes under the next chunks' search kernels
        a.gather = "copy"
    if a.only:
        a.no_c4 = a.no_c4 or a.only != "c4"
        a.no_c5 = a.no_c5 or a.only != "c5"
        if a.only != "c3":
            a.no_e2e = a.no_est = a.no_cpu_baseline = a.no_peaks = True
    return a


def workload_name(a):
    return (f"C3 EuclideanKNNRegressor {a.n_queries} queries x {a.n_ref} reference plots x "
            f"{a.dim} features, k={a.k}, predict(weights='distance') over {a.n_out} targets")


def config_of(a):
    """The same keys in both arms (the driver compares them)."""
    return {"workload": workload_name(a), "n_ref": a.n_ref, "dim": a.dim, "k": a.k,
            "queries_per_gpu": a.n_queries,
            "l2": f"inputs {a.n_queries * a.dim * 8 / 1e9:.2f} GB per step exceed the 126 MB L2 (no flush needed)",
            "multi_gpu": "queries sharded, reference set replicated, every rank's results land in rank 0's result "
                         "arrays over NVLink (CUDA IPC mapping) inside the timed region - per-chunk copy-engine "
                         "peer copies under the next chunks' kernels (--gather copy, the default) or stores of "
                         "the finishing kernels themselves (--gather fused, timed beside it as gather_alt); "
                         "NCCL carries the barriers and the out-of-band verification gather"}


# ------------------------------------------------------------------------------------------
# synthetic data (BASELINE.md section 3)
# ------------------------------------------------------------------------------------------
def make_reference_set(a):
    """C3: refs seed 0, y seed 1."""
    R = np.random.default_rng(0).standard_normal((a.n_ref, a.dim))
    y = np.random.default_rng(1).standard_normal((a.n_ref, a.n_out))
    return R, y


def query_block(dim, block, rows, rank=0):
    """Queries: N(0,1) in 1M-row blocks from SeedSequence(2).spawn (rank-offset per GPU)."""
    ss = np.random.SeedSequence(2).spawn(block + 1 + 1000 * rank)[-1]
    return np.random.default_rng(ss).standard_normal((rows, dim))


def c5_mixing(dim=64):
    """Fixed seed-3 mixing matrix: X = G @ A has correlated features, so the whitening is not trivial."""
    A = np.random.default_rng(3).standard_normal((dim, dim)) / np.sqrt(dim)
    return A + np.eye(dim)


def c5_reference_set(n_ref=50_000, dim=64, n_out=8):
    A = c5_mixing(dim)
    R = np.random.default_rng(0).standard_normal((n_ref, dim)) @ A
    y = np.random.default_rng(1).standard_normal((n_ref, n_out))
    return R, y, A


def c4_training_set(n_ref=20_000, dim=16, n_targets=10):
    X = np.random.default_rng(0).standard_normal((n_ref, dim))
    y = X[:, :n_targets] * 2.0 + np.random.default_rng(1).standard_normal((n_ref, n_targets))
    return X, y


# ------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-i", str(self.gpu), "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)),
                "power_w_max": float(max(pw)), "samples": len(sm), "reasons": sorted(reasons)}


def usable_cores():
    try:
        return max(len(os.sched_getaffinity(0)), 1)
    except AttributeError:
        return max(os.cpu_count() or 1, 1)


# ------------------------------------------------------------------------------------------
# the reference arm: the unmodified package from oracle/_ref (see __graft_entry__.install_reference)
# ------------------------------------------------------------------------------------------
def import_reference():
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "sknnr")):
        return None
    if ref_dir not in sys.path:
        sys.path.insert(0, ref_dir)
    import sknnr

    assert os.path.realpath(sknnr.__file__).startswith(os.path.realpath(ref_dir)), sknnr.__file__
    return sknnr


class ReferenceC3:
    """`EuclideanKNNRegressor(n_neighbors=k, weights="distance", algorithm="brute")` of the
    reference, fitted once (ref:src/sknnr/_euclidean.py:55-56); a step is the stock way to obtain
    what one call of ours returns: `kneighbors(X)` (dist, idx) then `predict(X)`
    (ref:src/sknnr/_base.py:285-352).  Falls back to the oracle port when oracle/_ref is absent."""

    def __init__(self, a):
        from threadpoolctl import threadpool_limits

        self.a = a
        self.limits = threadpool_limits
        self.ref = import_reference()
        R, y = make_reference_set(a)
        with self.limits(limits=usable_cores()):
            if self.ref is not None:
                self.kind = "reference"
                self.est = self.ref.EuclideanKNNRegressor(n_neighbors=a.k, weights="distance",
                                                          algorithm="brute").fit(R, y)
            else:
                from sklearn.neighbors import KNeighborsRegressor

                self.kind = "port"
                self.mean, self.scale = R.mean(axis=0), R.std(axis=0, ddof=1)
                self.y = y
                self.est = KNeighborsRegressor(n_neighbors=a.k, algorithm="brute",
                                               weights="distance").fit((R - self.mean) / self.scale, y)

    def step(self, rows):
        """-> (seconds of kneighbors, seconds of predict)"""
        Q = query_block(self.a.dim, 0, rows)
        # every host thread the process may use, whatever OMP_NUM_THREADS says (torchrun exports
        # OMP_NUM_THREADS=1 to its workers, which would make this a one-core number)
        with self.limits(limits=usable_cores()):
            if self.kind == "reference":
                t0 = time.perf_counter()
                self.est.kneighbors(Q)
                t1 = time.perf_counter()
                self.est.predict(Q)
                t2 = time.perf_counter()
            else:
                from oracle import sknnr_oracle as orc

                t0 = time.perf_counter()
                Z = orc.affine_project(Q, self.mean, self.scale, None)
                dist, idx = self.est.kneighbors(Z)
                dist, idx = orc.deterministic_order(dist, idx)
                t1 = time.perf_counter()
                orc.weighted_average(self.y, idx, orc.get_weights(dist, "distance"))
                t2 = time.perf_counter()
        return t1 - t0, t2 - t1

    def describe(self, rows, t_kn, t_pr):
        import sklearn

        if self.kind == "reference":
            what = (f"unmodified sknnr {self.ref.__version__} from oracle/_ref: EuclideanKNNRegressor(n_neighbors="
                    f"{self.a.k}, weights='distance', algorithm='brute').kneighbors(X) {t_kn:.2f} s + .predict(X) "
                    f"{t_pr:.2f} s (predict repeats the search: the stock API has no call that returns both)")
        else:
            what = ("oracle port (oracle/_ref absent): scikit-learn brute KNeighborsRegressor + sknnr "
                    f"ordering/predict glue, search {t_kn:.2f} s + predict {t_pr:.2f} s")
        return (f"{rows} of {self.a.n_queries} query rows per step (brute cost is linear in n_q); {what}; "
                f"scikit-learn {sklearn.__version__}")


def run_reference(a, rank):
    if rank != 0:
        return
    rows = min(a.ref_sample, a.n_queries)
    leg = ReferenceC3(a)
    for _ in range(a.warmup):
        leg.step(min(rows, 20_000))
    t_kn = t_pr = 0.0
    for _ in range(a.steps):
        x, y = leg.step(rows)
        t_kn += x
        t_pr += y
    total = t_kn + t_pr
    value = rows * a.steps / total
    threads = usable_cores()
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * total / a.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": config_of(a),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "os_cpu_count": os.cpu_count(),
                         "kind": leg.kind, "sample": leg.describe(rows, t_kn / a.steps, t_pr / a.steps),
                         "kneighbors_only_qps": rows * a.steps / t_kn, "predict_only_qps": rows * a.steps / t_pr},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------
class SharedResults:
    """Result arrays of the whole job in rank 0's HBM, mapped into every rank (CUDA IPC): each
    rank's query call writes its block of rows directly, over NVLink for ranks > 0."""

    def __init__(self, lib, L, dev_index, rank, world, rows_per_rank, k, n_out):
        import torch.distributed as dist

        self.lib, self.L, self.dev, self.rank, self.world = lib, L, dev_index, rank, world
        self.rows = rows_per_rank
        self.sizes = [k * 8, k * 8, n_out * 8]          # bytes per row: dist f64, idx i64, pred f64
        self.base = [C.c_void_p(None) for _ in self.sizes]
        self.mapped = world > 1 and rank != 0
        handles = [None, None, None]
        if rank == 0:
            for i, sz in enumerate(self.sizes):
                L.check(lib.sknnr_device_alloc(dev_index, C.byref(self.base[i]), world * rows_per_rank * sz))
            if world > 1:
                for i in range(3):
                    buf = (C.c_ubyte * 64)()
                    L.check(lib.sknnr_ipc_export(dev_index, self.base[i], buf))
                    handles[i] = bytes(buf)
        if world > 1:
            box = [handles]
            dist.broadcast_object_list(box, src=0)
            handles = box[0]
            if rank != 0:
                for i in range(3):
                    buf = (C.c_ubyte * 64).from_buffer_copy(handles[i])
                    L.check(lib.sknnr_ipc_open(dev_index, buf, C.byref(self.base[i])))

    def ptr(self, i, rank=None):
        r = self.rank if rank is None else rank
        return self.base[i].value + r * self.rows * self.sizes[i]

    def to_host(self, i, rank, rows, dtype, width):
        """rows of rank `rank` (rank 0 only)."""
        out = np.empty((rows, width), dtype=dtype)
        self.L.check(self.lib.sknnr_device_copy(self.dev, out.ctypes.data_as(C.c_void_p),
                                                C.c_void_p(self.ptr(i, rank)), out.nbytes, 2, None))
        return out

    def rows_to_host(self, rows, k, n_out):
        """(dist, idx, pred) of the job-wide row numbers `rows`, gathered on the device so that only those
        rows are copied (rank 0 only).  The arrays are the library's allocations, seen by torch through the
        CUDA array interface."""
        import torch

        sel = torch.from_numpy(rows).to(torch.device("cuda", self.dev))
        out = []
        for i, typestr, width in ((0, "<f8", k), (1, "<i8", k), (2, "<f8", n_out)):
            iface = {"data": (self.base[i].value, False), "shape": (self.world * self.rows, width),
                     "typestr": typestr, "strides": None, "version": 3}
            whole = torch.as_tensor(type("LibraryArray", (), {"__cuda_array_interface__": iface})())
            out.append(whole[sel].cpu().numpy())
        return out

    def close(self):
        for i in range(3):
            if self.base[i].value:
                if self.mapped:
                    self.lib.sknnr_ipc_close(self.dev, self.base[i])
                else:
                    self.lib.sknnr_device_free(self.dev, self.base[i])
                self.base[i] = C.c_void_p(None)


DUMP_BYTES = {"c3": 32_000_000, "c5": 15_000_000, "c4": 15_000_000}     # --dump-outputs: under 64 MB in all


def dump_outputs(a, leg, n_rows, k, n_out, fetch):
    """--dump-outputs: DIR/<leg>_{rows,dist,idx,pred}.npy for a fixed, seeded sample of the `n_rows` result
    rows (all of them when they fit DUMP_BYTES[leg]); `fetch(rows)` returns (dist, idx, pred) of those rows.
    Everything is stored as float64 (indices and row numbers are exact in it)."""
    m = DUMP_BYTES[leg] // (8 * (1 + 2 * k + n_out))
    if m >= n_rows:
        rows = np.arange(n_rows)
    else:
        rows = np.unique(np.random.default_rng(20261020).integers(0, n_rows, size=m))
    os.makedirs(a.dump_outputs, exist_ok=True)
    for name, arr in zip(("rows", "dist", "idx", "pred"), (rows, *fetch(rows))):
        np.save(os.path.join(a.dump_outputs, f"{leg}_{name}.npy"), np.asarray(arr, dtype=np.float64))


def measure_gemm_peaks(dev):
    """cuBLAS dense GEMM throughput measured in this run (8192^3): burst = best of 10, sustained = a
    2 s back-to-back loop.  TF32 (allow_tf32) is what round 1's kernel ran on; FP16 is the pipe the
    kernel uses now (the driver's MEASURED_PEAKS.json holds the bf16 figure)."""
    import torch

    out = {}
    n = 8192
    for name, dt, tf32 in (("tf32", torch.float32, True), ("fp16", torch.float16, False)):
        torch.backends.cuda.matmul.allow_tf32 = tf32
        a = torch.randn((n, n), device=dev, dtype=dt)
        b = torch.randn((n, n), device=dev, dtype=dt)
        for _ in range(3):
            a @ b
        torch.cuda.synchronize(dev)
        best = float("inf")
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            a @ b
            e1.record()
            torch.cuda.synchronize(dev)
            best = min(best, e0.elapsed_time(e1))
        out[f"{name}_tflops_burst"] = 2.0 * n ** 3 / (best * 1e-3) / 1e12
        iters = max(10, int(2000.0 / best))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            a @ b
        e1.record()
        torch.cuda.synchronize(dev)
        out[f"{name}_tflops_sustained"] = 2.0 * n ** 3 * iters / (e0.elapsed_time(e1) * 1e-3) / 1e12
        del a, b
    torch.backends.cuda.matmul.allow_tf32 = False
    out["how"] = "torch.matmul 8192^3 (cuBLAS), CUDA events: best of 10 and a 2 s back-to-back loop"
    return out


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f)
    except OSError:
        return {}


def tensor_roofline(flops, search_ms, n_launches, peaks, gemm, traffic_per_row, rows_per_launch, note):
    """roofline object of the fused tcgen05 distance + top-k kernel.  The contraction runs on the
    16-bit (FP16 operand, FP32 accumulate) tensor pipe, so the denominator is the measured dense
    bf16/fp16 figure; the TF32-basis fraction (round 1's denominator) is kept beside it."""
    achieved = flops / (search_ms * 1e-3) / 1e12 if search_ms > 0 else None
    peak16 = peaks.get("bf16_tflops_sustained")
    src = "MEASURED_PEAKS.json bf16_tflops_sustained (dense 16-bit tensor pipe, sustained), of measured"
    if peak16 is None:
        peak16, src = 1400.0, "fallback 1400 dense bf16 sustained (B200_PROFILING.md), of fallback"
    r = {"kernel": "search_tc_kernel", "bound": "tensor", "achieved": achieved, "peak": peak16, "unit": "TFLOP/s",
         "frac": (achieved / peak16) if achieved else None, "peak_source": src,
         "frac_tf32_basis": (achieved / (peak16 / 2.0)) if achieved else None,
         "traffic": traffic_per_row * rows_per_launch if traffic_per_row else None,
         "algorithmic_flops_per_launch": flops / max(n_launches, 1), "launches_per_step": n_launches,
         "kernel_ms_per_step": search_ms, "note": note}
    if gemm:
        r["cublas_measured_here"] = gemm
        if achieved and gemm.get("tf32_tflops_sustained"):
            r["frac_vs_cublas_tf32_sustained"] = achieved / gemm["tf32_tflops_sustained"]
        if achieved and gemm.get("fp16_tflops_sustained"):
            r["frac_vs_cublas_fp16_sustained"] = achieved / gemm["fp16_tflops_sustained"]
    return r


TC_NOTE = ("algorithmic FLOPs 2*d'*n_q*n_ref over the CUDA-event time of the search kernel launches of one "
           "device-resident step.  The kernel contracts FP16 operands (11-bit significand, the precision of TF32, "
           "at twice its rate) with FP32 accumulation in TMEM; it is bound by the selection epilogue (every score "
           "is read out of TMEM and compared: TMEM capacity x slot round-trip latency), not by the tensor pipe - "
           "see DESIGN.md section 4")


def run_ours(a, rank, world, local_rank):
    import torch

    from sknnr_b200 import _lib as L
    from sknnr_b200._engine import KNNIndex

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    lib = L.load()
    L.set_option("timing", 1)
    for name, v in (("engine", a.engine), ("kc", a.kc), ("tc_streams", a.tc_streams), ("tc_debug", a.tc_debug),

                    ("chunk_rows", a.chunk_rows), ("host_slots", a.host_slots)):
        if v:
            L.set_option(name, v)
    if a.tc_seed_stride >= 0:
        L.set_option("tc_seed_stride", a.tc_seed_stride)
    for item in a.opt:
        name, _, v = item.partition("=")
        L.set_option(name, int(v))
    stream = torch.cuda.current_stream(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(v):
        if world > 1:
            t = torch.tensor([v], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return v

    def timed(fn, steps):
        """K calls of fn bracketed by barrier + synchronize, CUDA events on the launching stream, max over ranks."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    peaks = load_peaks()
    gemm = None
    line = None

    def note(msg):
        if rank == 0:
            print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)

    if a.only in ("", "c3"):
        line = bench_c3(a, rank, world, local_rank, dev, stream, lib, L, KNNIndex, barrier, timed, max_over_ranks,
                        peaks, dist)
        if rank == 0 and not a.no_peaks:
            gemm = measure_gemm_peaks(dev)
            line["roofline"] = tensor_roofline(**line.pop("_roof"), peaks=peaks, gemm=gemm)
        elif rank == 0:
            line["roofline"] = tensor_roofline(**line.pop("_roof"), peaks=peaks, gemm=None)
    barrier()
    note("c3 done: " + (json.dumps({k_: line.get(k_) for k_ in ("value", "ms_per_step", "e2e", "e2e_estimator")}) if line else ""))
    c5 = c4 = None
    if not a.no_c5:
        c5 = bench_c5(a, rank, world, local_rank, dev, stream, lib, L, barrier, timed, peaks, gemm, dist)
    barrier()
    note("c5 done: " + json.dumps(c5)[:600])
    if not a.no_c4:
        c4 = bench_c4(a, rank, world, local_rank, dev, stream, lib, L, barrier, timed, dist)
    if rank != 0:
        return
    if line is None:
        line = {"metric": METRIC, "unit": UNIT, "n_gpus": world, "note": f"--only {a.only}"}
    line["c5"] = c5
    line["c4"] = c4
    print(json.dumps(line), flush=True)


def bench_c3(a, rank, world, local_rank, dev, stream, lib, L, KNNIndex, barrier, timed, max_over_ranks, peaks, dist):
    import torch

    R, y = make_reference_set(a)
    mean, scale = R.mean(axis=0), R.std(axis=0, ddof=1)
    index = KNNIndex((R - mean) / scale, mean, scale, None, y, device=local_rank)

    # queries: host pinned (e2e leg) and device resident (value leg), float64 like the reference's inputs
    n_q, d, k, n_out = a.n_queries, a.dim, a.k, a.n_out
    X_host = torch.empty((n_q, d), dtype=torch.float64, pin_memory=True)
    xh = X_host.numpy()
    blk = 1_000_000
    for b, s in enumerate(range(0, n_q, blk)):
        rows = min(blk, n_q - s)
        xh[s:s + rows] = query_block(d, b, rows, rank)
    X_dev = X_host.to(dev, non_blocking=False)
    shared = SharedResults(lib, L, local_rank, rank, world, n_q, k, n_out)

    def step_device():
        index.query_device(X_dev.data_ptr(), False, n_q, d, k, dist_ptr=shared.ptr(0), idx_ptr=shared.ptr(1),
                           pred_ptr=shared.ptr(2), weights="distance", row_offset=rank * n_q,
                           stream=stream.cuda_stream)

    def step_copy():
        # synchronous call on device pointers: chunks pipeline over the library's slot streams and every
        # chunk's results travel to rank 0's arrays as copy-engine peer copies under the next chunks' kernels
        L.check(lib.sknnr_kneighbors(index._h, C.c_void_p(X_dev.data_ptr()), L.F64, n_q, d, rank * n_q, k,
                                     L.DETERMINISTIC, 10, C.c_void_p(shared.ptr(0)), C.c_void_p(shared.ptr(1)),
                                     L.W_DISTANCE, C.c_void_p(shared.ptr(2)), None))

    step_timed = step_copy if (world > 1 and a.gather == "copy") else step_device
    for _ in range(a.warmup):
        step_timed()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_total = timed(step_timed, a.steps)
    clocks = sampler.stop() if rank == 0 else None
    value = world * n_q * a.steps / (ms_total * 1e-3)
    barrier()
    if a.dump_outputs and rank == 0:
        dump_outputs(a, "c3", world * n_q, k, n_out, lambda rows: shared.rows_to_host(rows, k, n_out))
    headline_launches = int(index.stats()["kernel_launches"])   # of one headline step (this rank)

    # out-of-band verification of the fused gather: every rank repeats its block into local memory and
    # NCCL gathers those; rank 0 compares them with what the ranks stored into its arrays over NVLink
    def verify_gather():
        loc = [torch.empty((n_q, k), dtype=torch.float64, device=dev), torch.empty((n_q, k), dtype=torch.int64, device=dev),
               torch.empty((n_q, n_out), dtype=torch.float64, device=dev)]
        index.query_device(X_dev.data_ptr(), False, n_q, d, k, dist_ptr=loc[0].data_ptr(), idx_ptr=loc[1].data_ptr(),
                           pred_ptr=loc[2].data_ptr(), weights="distance", row_offset=rank * n_q,
                           stream=stream.cuda_stream)
        barrier()
        ok = True
        for i, t in enumerate(loc):
            parts = [torch.empty_like(t) for _ in range(world)] if rank == 0 else None
            dist.gather(t, parts, dst=0)
            if rank == 0:
                for r in range(world):
                    got = shared.to_host(i, r, 4096, np.float64 if i != 1 else np.int64, t.shape[1])
                    tail = parts[r][:4096].cpu().numpy()
                    ok = ok and bool(np.array_equal(got, tail))
            del parts
        del loc
        assert rank != 0 or ok, "rows that arrived over NVLink differ from the NCCL-gathered blocks"
        return ok

    gather_ok = verify_gather() if world > 1 else None
    # the other way of getting the results to rank 0, timed the same way right behind the headline
    # (fused: the finishing kernels store over NVLink; copy: every chunk's results leave as copy-engine
    # peer copies under the next chunks' kernels)
    gather_alt = None
    if world > 1 and not a.no_gather_ab:
        alt = step_device if step_timed is step_copy else step_copy
        alt()
        ms_alt = timed(alt, a.steps)
        gather_alt = {"mode": "fused" if a.gather == "copy" else "copy",
                      "value": world * n_q * a.steps / (ms_alt * 1e-3), "ms_per_step": ms_alt / a.steps,
                      "verified": verify_gather()}

    # dominant-kernel timing: one more device-resident step; the library brackets every search
    # kernel launch with CUDA events on the launching stream (option "timing") and the stats
    # query sums them.  (The host-buffer call below overlaps chunks on several streams, so its
    # per-kernel brackets would include waiting for the other streams' kernels.)
    step_device()
    barrier()
    dev_stats = index.stats()
    cascade = index.cascade_counts()
    search_ms = dev_stats["search_ms"]

    # e2e through the host-buffer call (pinned host in/out, copies inside the timed region)
    e2e = e2e_est = None
    stats = dev_stats
    if not a.no_e2e:
        h_dist = torch.empty((n_q, k), dtype=torch.float64, pin_memory=True)
        h_idx = torch.empty((n_q, k), dtype=torch.int64, pin_memory=True)
        h_pred = torch.empty((n_q, n_out), dtype=torch.float64, pin_memory=True)

        def step_host():
            L.check(index._lib.sknnr_kneighbors(
                index._h, C.c_void_p(X_host.data_ptr()), L.F64, n_q, d, rank * n_q, k,
                L.DETERMINISTIC, 10, C.c_void_p(h_dist.data_ptr()), C.c_void_p(h_idx.data_ptr()),
                L.W_DISTANCE, C.c_void_p(h_pred.data_ptr()), None))

        step_host()
        barrier()
        t0 = time.perf_counter()
        e2e_steps = a.steps
        for _ in range(e2e_steps):
            step_host()
        barrier()
        dt = max_over_ranks(time.perf_counter() - t0)
        stats = index.stats()
        e2e = {"value": world * n_q * e2e_steps / dt, "unit": UNIT,
               "h2d_bytes_per_step": int(stats["h2d_bytes"]), "d2h_bytes_per_step": int(stats["d2h_bytes"]),
               "steps": e2e_steps, "timer": "host wall clock around the synchronous C-ABI call (pinned buffers)"}
        # device-path results must equal host-path results bit for bit
        mine = shared.to_host(1, rank, n_q, np.int64, k) if rank == 0 else None
        assert rank != 0 or np.array_equal(mine, h_idx.numpy()), "device and host paths disagree"
        del h_dist, h_idx, h_pred, mine

    # e2e through the estimator surface: the drop-in call on an ordinary NumPy array
    if not a.no_est:
        from sknnr_b200 import EuclideanKNNRegressor

        est = EuclideanKNNRegressor(n_neighbors=k, weights="distance").fit(R, y)
        X_np = np.array(xh, copy=True)           # pageable, like any user array
        for _ in range(2):                       # warm-up: staging buffers and result blocks exist afterwards
            pred = est.predict(X_np)
        barrier()
        t0 = time.perf_counter()
        est_steps = a.steps
        per_call = []
        for _ in range(est_steps):
            t1 = time.perf_counter()
            pred = est.predict(X_np)
            per_call.append(round((time.perf_counter() - t1) * 1e3, 2))
        barrier()
        dt = max_over_ranks(time.perf_counter() - t0)
        e2e_est = {"value": world * n_q * est_steps / dt, "unit": UNIT, "steps": est_steps,
                   "call": "sknnr_b200.EuclideanKNNRegressor(n_neighbors=7, weights='distance').predict(X), "
                           "X a pageable float64 ndarray, result a new float64 ndarray; host wall clock",
                   "h2d_bytes_per_step": int(n_q * d * 8), "d2h_bytes_per_step": int(n_q * n_out * 8),
                   "per_call_ms": per_call}
        if rank == 0 and not a.no_e2e:
            ref_pred = shared.to_host(2, 0, 4096, np.float64, n_out)
            assert np.array_equal(pred[:4096], ref_pred), "estimator and C-ABI predictions disagree"
        del X_np, pred, est

    cpu = None
    if rank == 0 and not a.no_cpu_baseline and world == 1:
        leg = ReferenceC3(a)
        rows = min(a.cpu_sample, n_q)
        leg.step(min(rows, 20_000))
        t_kn, t_pr = leg.step(rows)
        cpu = {"value": rows / (t_kn + t_pr), "unit": UNIT, "cores": usable_cores(), "os_cpu_count": os.cpu_count(),
               "kind": leg.kind, "sample": leg.describe(rows, t_kn, t_pr),
               "kneighbors_only_qps": rows / t_kn, "predict_only_qps": rows / t_pr}
    shared.close()
    if rank != 0:
        return None
    engine = int(stats.get("engine", 0))
    dpad = (d + 7) // 8 * 8
    flops = 2.0 * d * n_q * a.n_ref                      # algorithmic: 2 * d' * n_q * n_ref
    chunk_dev = 2 * (a.chunk_rows if a.chunk_rows > 0 else (1 << 20))
    n_chunks = max(1, -(-n_q // chunk_dev))
    hbm = {"algorithmic_bytes_per_step": n_q * (8 * d + k * 16 + 8 * n_out) + 4 * a.n_ref * dpad,
           "peak_gbs": peaks.get("hbm_gbs"), "peak_source": "MEASURED_PEAKS.json" if peaks else "absent"}
    if hbm["peak_gbs"]:
        hbm["achieved_gbs_whole_step"] = hbm["algorithmic_bytes_per_step"] / (ms_total / a.steps * 1e-3) / 1e9
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": ms_total / a.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None,
        "dtype": ("f16 operands / f32 accumulate filter + f64 refine" if engine == L.ENGINE_TENSOR
                  else "f32 filter + f64 refine"),
        "data": "synthetic", "config": config_of(a),
        "_roof": dict(flops=flops, search_ms=search_ms, n_launches=n_chunks,
                      # dram__bytes_read.sum + dram__bytes_write.sum of one 2^20-row launch, ncu --set full
                      # (profiles/r02_search_tc_*.md), per row
                      traffic_per_row=(TC_TRAFFIC_PER_ROW if d == 32 else None), rows_per_launch=n_q / n_chunks,
                      note=TC_NOTE),
        "hbm": hbm, "cpu_baseline": cpu, "e2e": e2e, "e2e_estimator": e2e_est,
        "gpu_launches": headline_launches * a.steps,
        "fallback_rows_per_step": int(dev_stats["n_fallback"]), "cascade_rows_per_step": cascade,
        "gather_verified": gather_ok,
        "fused_gather_verified": (gather_ok if a.gather == "fused" else (gather_alt or {}).get("verified")),
        "gather": (a.gather if world > 1 else None), "gather_alt": gather_alt,
        "clocks": clocks,
    }
    return line


TC_TRAFFIC_PER_ROW = 150.8e6 / float(1 << 20)     # profiles/r02_search_tc_final2.md: 106.0 MB read + 44.8 MB written


def bench_c5(a, rank, world, local_rank, dev, stream, lib, L, barrier, timed, peaks, gemm, dist):
    """BASELINE.json configs[4]: MahalanobisKNNRegressor, 100M-pixel map x 50k plots x 64 features, k=7,
    rows split over the ranks (strong scaling), a real 64x64 whitening projector
    (ref:src/sknnr/transformers/_mahalanobis_transformer.py:47-55), queries generated on the device."""
    import torch

    from sknnr_b200 import MahalanobisKNNRegressor

    n_ref, dim, n_out, k = 50_000, 64, 8, 7
    Rraw, y, A = c5_reference_set(n_ref, dim, n_out)
    est = MahalanobisKNNRegressor(n_neighbors=k, weights="distance").fit(Rraw, y)
    index = est.regressor_._get_index()
    total = a.c5_rows
    per = -(-total // world)
    lo, hi = min(rank * per, total), min((rank + 1) * per, total)
    n_q = hi - lo
    # correlated raw features X = G @ A, generated block-wise on the device (float64, like the reference's input)
    X = torch.empty((n_q, dim), dtype=torch.float64, device=dev)
    At = torch.from_numpy(A).to(dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(5 + rank)
    blk = 4_000_000
    for s in range(0, n_q, blk):
        e = min(n_q, s + blk)
        torch.matmul(torch.randn((e - s, dim), dtype=torch.float64, device=dev, generator=gen), At, out=X[s:e])
    shared = SharedResults(lib, L, local_rank, rank, world, per, k, n_out)

    def step():
        index.query_device(X.data_ptr(), False, n_q, dim, k, dist_ptr=shared.ptr(0), idx_ptr=shared.ptr(1),
                           pred_ptr=shared.ptr(2), weights="distance", row_offset=lo, stream=stream.cuda_stream)

    step()
    steps = a.steps
    ms = timed(step, steps)
    if a.dump_outputs:
        if rank == 0:
            dump_outputs(a, "c5", total, k, n_out, lambda rows: shared.rows_to_host(rows, k, n_out))
        barrier()      # the next step() of the other ranks stores into the arrays read here
    step()
    barrier()
    st = index.stats()
    cascade = index.cascade_counts()
    rec = None
    if rank == 0:
        # parity on a sample, outside the timed region: the first rows of rank 0 against the oracle
        from oracle import sknnr_oracle as orc

        m = 2000
        Xs = X[:m].cpu().numpy()
        d_g = shared.to_host(0, 0, m, np.float64, k)
        i_g = shared.to_host(1, 0, m, np.int64, k)
        p_g = shared.to_host(2, 0, m, np.float64, n_out)
        center, scale, proj, _ = est.transformer_._affine()
        state = orc.FittedState("euclidean", fit_Z=np.asarray(est.regressor_._fit_X), y=y, center=center, scale=scale,
                                proj=proj)
        d_o, i_o = orc.kneighbors(state, Xs, k=k, row_offset=0)
        orc.assert_tie_aware_equal(d_g, i_g, d_o, i_o, rtol=1e-5, atol=1e-7)
        same = (i_g == i_o).all(axis=1)
        np.testing.assert_allclose(p_g[same], orc.weighted_average(y, i_o, orc.get_weights(d_o, "distance"))[same],
                                   rtol=1e-5, atol=1e-8)
        flops = 2.0 * dim * n_q * n_ref
        chunk_dev = 2 * (a.chunk_rows if a.chunk_rows > 0 else (1 << 20))
        n_chunks = max(1, -(-n_q // chunk_dev))
        rec = {"workload": f"C5 MahalanobisKNNRegressor {total} queries x {n_ref} reference plots x {dim} features, "
                           f"k={k}, predict(weights='distance') over {n_out} targets, rows split over {world} GPU(s)",
               "metric": METRIC, "value": total * steps / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": steps,
               "ms_per_step": ms / steps, "scaling": "strong", "rows_per_gpu": per,
               "roofline": tensor_roofline(flops, st["search_ms"], n_chunks, peaks, gemm, None, n_q / n_chunks,
                                           TC_NOTE + " (rank 0's launches)"),
               "fallback_rows_per_step_rank0": int(st["n_fallback"]), "cascade_rows_per_step_rank0": cascade,
               "parity_sample_rows": m,
               "gpu_launches": int(st["kernel_launches"] * steps)}
        if not a.no_cpu_baseline and world == 1:
            rec["cpu_baseline"] = cpu_c5(a, Rraw, y, A, k)
    shared.close()
    del X
    torch.cuda.empty_cache()
    return rec


def cpu_c5(a, Rraw, y, A, k, rows=200_000):
    from threadpoolctl import threadpool_limits

    ref = import_reference()
    if ref is None:
        return None
    Q = np.random.default_rng(7).standard_normal((rows, A.shape[0])) @ A
    with threadpool_limits(limits=usable_cores()):
        est = ref.MahalanobisKNNRegressor(n_neighbors=k, weights="distance", algorithm="brute").fit(Rraw, y)
        est.kneighbors(Q[:5000])
        t0 = time.perf_counter()
        est.kneighbors(Q)
        t1 = time.perf_counter()
        est.predict(Q)
        t2 = time.perf_counter()
    return {"value": rows / (t2 - t0), "unit": UNIT, "cores": usable_cores(), "os_cpu_count": os.cpu_count(),
            "kind": "reference", "kneighbors_only_qps": rows / (t1 - t0), "predict_only_qps": rows / (t2 - t1),
            "sample": f"{rows} query rows; unmodified sknnr MahalanobisKNNRegressor(n_neighbors={k}, weights='distance', "
                      f"algorithm='brute').kneighbors(X) {t1 - t0:.2f} s + .predict(X) {t2 - t1:.2f} s"}


def bench_c4(a, rank, world, local_rank, dev, stream, lib, L, barrier, timed, dist):
    """BASELINE.json configs[3]: RFNNRegressor, 500 trees (10 forests x 50), 20k plots, raw query rows ->
    forest walk -> 16-bit node codes -> bit-exact Hamming search -> predict, one device call
    (ref:src/sknnr/_rfnn.py:216-239, ref:src/sknnr/_weighted_trees.py:46-59)."""
    import torch

    from sknnr_b200 import RFNNRegressor

    n_ref, dim, n_t, k = 20_000, 16, 10, 7
    Xr, yr = c4_training_set(n_ref, dim, n_t)
    t0 = time.perf_counter()
    est = RFNNRegressor(n_estimators=50, random_state=0, n_neighbors=k, n_jobs=-1).fit(Xr, yr)
    fit_s = time.perf_counter() - t0
    reg = est.regressor_
    index = reg._get_index()
    forest = est.transformer_._forest_index(reg.__dict__.get("_node_tables"))
    n_trees = index.n_trees
    n_q = a.c4_rows
    gen = torch.Generator(device=dev)
    gen.manual_seed(11 + rank)
    X = torch.randn((n_q, dim), dtype=torch.float64, device=dev, generator=gen)
    o_dist = torch.empty((n_q, k), dtype=torch.float64, device=dev)
    o_idx = torch.empty((n_q, k), dtype=torch.int64, device=dev)
    o_pred = torch.empty((n_q, n_t), dtype=torch.float64, device=dev)

    def step():
        L.check(lib.sknnr_hamming_kneighbors_forest(
            index._h, forest._h, C.c_void_p(X.data_ptr()), L.F64, n_q, dim, rank * n_q, k,
            L.DETERMINISTIC | L.DEVICE_PTRS, 10, C.c_void_p(o_dist.data_ptr()), C.c_void_p(o_idx.data_ptr()),
            L.W_UNIFORM, C.c_void_p(o_pred.data_ptr()), C.c_void_p(stream.cuda_stream)))

    step()
    steps = a.steps
    ms = timed(step, steps)
    if a.dump_outputs and rank == 0:
        dump_outputs(a, "c4", n_q, k, n_t, lambda rows: [t[torch.from_numpy(rows).to(dev)].cpu().numpy()
                                                         for t in (o_dist, o_idx, o_pred)])
    step()
    barrier()
    st = index.stats()
    if rank != 0:
        return None
    # parity on a sample, outside the timed region: node IDs from scikit-learn's own apply, neighbours
    # and distances from the oracle's canonical (distance, index) ranking - bit-exact
    from oracle import sknnr_oracle as orc

    m = 300
    Xs = X[:m].cpu().numpy()
    ids_ref = np.asarray(reg._fit_X).astype(np.int64)
    ids_q = np.hstack([e_.apply(Xs.astype(np.float32)) for e_ in est.transformer_.estimators_]).astype(np.int64)
    state = orc.FittedState("hamming", fit_Z=ids_ref, y=yr, hamming_w=est.hamming_weights_)
    d_o, i_o = orc.kneighbors(state, ids_q, k=k, row_offset=0)
    assert np.array_equal(o_idx[:m].cpu().numpy(), i_o), "C4: neighbour indices differ from the oracle"
    assert np.array_equal(o_dist[:m].cpu().numpy(), d_o), "C4: distances differ from the oracle"
    np.testing.assert_allclose(o_pred[:m].cpu().numpy(), orc.weighted_average(yr, i_o), rtol=1e-12)
    compares = float(n_q) * n_ref * n_trees
    search_ms = st["search_ms"]
    achieved = compares / (search_ms * 1e-3) / 1e12 if search_ms > 0 else None
    rec = {"workload": f"C4 RFNNRegressor(n_estimators=50) x {n_t} targets = {n_trees} trees, {n_q} raw query rows per "
                       f"GPU x {n_ref} plots x {dim} features, k={k}, predict (uniform) over {n_t} targets",
           "metric": METRIC, "value": world * n_q * steps / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": steps,
           "ms_per_step": ms / steps, "scaling": "weak", "fit_seconds": fit_s,
           "roofline": {"kernel": "hamming_search_kernel", "bound": "integer ALU (HSET2 issue rate)",
                        "achieved": achieved, "peak": LANE_OPS_PEAK / 1e12, "unit": "T ID-compares/s",
                        "frac": (achieved / (LANE_OPS_PEAK / 1e12)) if achieved else None,
                        "peak_source": "148 SMs x 128 lanes x 1.965 GHz lane-ops/s (SURVEY.md section 8d); the kernel "
                                       "compares two 16-bit node IDs per lane-instruction",
                        "kernel_ms_per_step": search_ms, "search_share_of_step": search_ms / (ms / steps),
                        "traffic": None},
           "parity_sample_rows": m, "gpu_launches": int(st["kernel_launches"] * steps)}
    if not a.no_cpu_baseline and world == 1:
        rec["cpu_baseline"] = cpu_c4(Xr, yr, k)
    return rec


def cpu_c4(Xr, yr, k, rows=2000):
    """The reference's RFNN query path on the host.  Its fit() ends with two leave-one-out self-queries
    (n_ref^2 x 500 trees through SciPy's single-threaded cdist: minutes at 20k plots,
    ref:src/sknnr/_base.py:37-40); they are not on the timed path, so they are switched off while
    fitting.  kneighbors / predict below are the unmodified reference."""
    from threadpoolctl import threadpool_limits

    ref = import_reference()
    if ref is None:
        return None
    from sknnr import _base as ref_base

    Q = np.random.default_rng(13).standard_normal((rows, Xr.shape[1]))
    saved = ref_base.IndependentPredictorMixin._set_independent_prediction_attributes

    def skip_self_query(self, y):
        self.independent_prediction_ = None
        self.independent_score_ = None

    ref_base.IndependentPredictorMixin._set_independent_prediction_attributes = skip_self_query
    try:
        with threadpool_limits(limits=usable_cores()):
            est = ref.RFNNRegressor(n_estimators=50, random_state=0, n_neighbors=k, n_jobs=-1).fit(Xr, yr)
    finally:
        ref_base.IndependentPredictorMixin._set_independent_prediction_attributes = saved
    out = {}
    for label, nj in (("n_jobs=None", None), ("n_jobs=-1", -1)):
        est.regressor_.n_jobs = nj
        for f_ in est.transformer_.estimators_:
            f_.n_jobs = nj
        with threadpool_limits(limits=usable_cores()):
            t0 = time.perf_counter()
            est.kneighbors(Q)
            t1 = time.perf_counter()
            est.predict(Q)
            t2 = time.perf_counter()
        out[label] = {"qps": rows / (t2 - t0), "kneighbors_s": t1 - t0, "predict_s": t2 - t1}
    best = max(v["qps"] for v in out.values())
    return {"value": best, "unit": UNIT, "cores": usable_cores(), "os_cpu_count": os.cpu_count(), "kind": "reference",
            "by_n_jobs": out,
            "sample": f"{rows} raw query rows; unmodified sknnr RFNNRegressor(n_estimators=50, random_state=0).kneighbors(X) "
                      "+ .predict(X) (forest apply + scipy cdist_hamming), value = the faster of n_jobs=None / -1; the "
                      "fit-time leave-one-out self-queries were skipped (not on the timed path)"}


def main():
    a = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if a.impl == "reference":
        run_reference(a, rank)
        return
    run_ours(a, rank, world, local_rank)
    if world > 1:
        import torch.distributed as dist

        dist.destroy_process_group()


if __name__ == "__main__":
    main()
