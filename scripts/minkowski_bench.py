"""Throughput of the Manhattan / Chebyshev searches next to the Euclidean one (GPU).

C3-shaped data (BASELINE.md section 3, the seeds `bench.py` uses): 50 000 plots x 32 features, 8
targets, N(0, 1), standardised as EuclideanKNNRegressor does; queries N(0, 1) in 1M-row blocks; k = 7,
weights="distance", deterministic ordering.  Legs per metric:

  device   the queries held on the device (10M rows), sknnr_kneighbors on device pointers
  e2e      est.predict(X) of an EuclideanKNNRegressor(metric=...) on a 2M-row NumPy array
  exact    engine=EXACT on a subsample (the filter's advantage), capped in time
  cpu      scikit-learn's brute KNeighborsRegressor with the same metric on a 20k-row subsample

and, for the FP32 filter, its share of the FP32-pipe issue bound: element pairs / s of the search
kernel alone (CUDA events, `sknnr_set_option("timing", 1)`) against the measured FFMA2 issue rate
(`sknnr_measure_fp32_peak`) divided by the inner loop's FP32-pipe instructions per element pair.
One JSON document goes to stdout (and to --out); the GPU's name and power limit are read in the
same process.  Needs a CUDA device: without one it fails.

    python scripts/minkowski_bench.py [--queries N] [--e2e-rows N] [--exact-rows N] [--cpu-rows N]
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# FP32-pipe instructions per (query, plot, feature) in the search kernel's inner loop (cuobjdump -sass of
# search_simt_kernel): Euclidean one FFMA2 per two pairs; Manhattan one FADD2 (two differences) and one
# FADD2 (|t| accumulated) per two pairs; Chebyshev one FADD2 and two FMNMX per two pairs
INSTR_PER_PAIR = {"euclidean": 0.5, "manhattan": 1.0, "chebyshev": 1.5}
ESTIMATOR_KW = {"euclidean": {}, "manhattan": {"p": 1}, "chebyshev": {"metric": "chebyshev"}}


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                       capture_output=True, text=True)
    return r.stdout.strip()


def reference_set(n_ref, dim, n_out):
    R = np.random.default_rng(0).standard_normal((n_ref, dim))
    y = np.random.default_rng(1).standard_normal((n_ref, n_out))
    return R, y


def query_block(dim, block, rows):
    ss = np.random.SeedSequence(2).spawn(block + 1)[-1]
    return np.random.default_rng(ss).standard_normal((rows, dim))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--queries", type=int, default=10_000_000)
    ap.add_argument("--n-ref", type=int, default=50_000)
    ap.add_argument("--dim", type=int, default=32)
    ap.add_argument("--n-out", type=int, default=8)
    ap.add_argument("--k", type=int, default=7)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--e2e-rows", type=int, default=2_000_000)
    ap.add_argument("--exact-rows", type=int, default=200_000)
    ap.add_argument("--exact-seconds", type=float, default=60.0, help="time cap of each exact leg")
    ap.add_argument("--cpu-rows", type=int, default=20_000)
    ap.add_argument("--metrics", default="euclidean,manhattan,chebyshev")
    ap.add_argument("--out", default="")
    a = ap.parse_args()

    import torch

    import sknnr_b200 as S
    from sknnr_b200 import _lib as L
    from sknnr_b200._engine import KNNIndex

    if not torch.cuda.is_available() or L.device_count() == 0:
        raise SystemExit("minkowski_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream(dev)
    res = {"gpu": gpu_info(), "shape": {"n_ref": a.n_ref, "dim": a.dim, "n_out": a.n_out, "k": a.k,
                                         "queries": a.queries}}
    peak = L.measure_fp32_peak(0)
    res["fp32_ffma2_tflops"] = peak
    issue_rate = peak * 1e12 / 4          # FFMA2 lane-instructions / s (one FFMA2 = two FMAs = 4 FLOP)

    R, y = reference_set(a.n_ref, a.dim, a.n_out)
    mean, scale = R.mean(axis=0), R.std(axis=0, ddof=1)
    Z = (R - mean) / scale
    X_host = torch.empty((a.queries, a.dim), dtype=torch.float64, pin_memory=True)
    xh = X_host.numpy()
    for b, s in enumerate(range(0, a.queries, 1_000_000)):
        rows = min(1_000_000, a.queries - s)
        xh[s:s + rows] = query_block(a.dim, b, rows)
    X_dev = X_host.to(dev)
    n_q, k = a.queries, a.k
    o_d = torch.empty((n_q, k), dtype=torch.float64, device=dev)
    o_i = torch.empty((n_q, k), dtype=torch.int64, device=dev)
    o_p = torch.empty((n_q, a.n_out), dtype=torch.float64, device=dev)

    def device_call(ix, rows):
        ix.query_device(X_dev.data_ptr(), False, rows, a.dim, k, dist_ptr=o_d.data_ptr(), idx_ptr=o_i.data_ptr(),
                        pred_ptr=o_p.data_ptr(), weights="distance", stream=stream.cuda_stream)

    def timed(fn, steps):
        ts = []
        for _ in range(steps):
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize(dev)
            ts.append(time.perf_counter() - t0)
        return ts

    legs = {}
    for metric in a.metrics.split(","):
        out = legs[metric] = {}
        ix = KNNIndex(Z, mean, scale, None, y, metric=metric)
        pairs = float(a.n_ref) * a.dim
        # device-resident throughput (warm-up: one full step, every shape of the timed window)
        device_call(ix, n_q)
        ts = timed(lambda: device_call(ix, n_q), a.steps)
        t = min(ts)
        out["device"] = {"seconds": ts, "queries_per_s": n_q / t, "element_pairs_per_s": n_q * pairs / t,
                         "engine": int(ix.stats()["engine"]), "cascade": ix.cascade_counts()}
        # the search kernel alone (events around it), one more step
        L.set_option("timing", 1)
        try:
            device_call(ix, n_q)
            torch.cuda.synchronize(dev)
            search_s = ix.stats()["search_ms"] * 1e-3
        finally:
            L.set_option("timing", 0)
        out["search_kernel"] = {"seconds": search_s, "element_pairs_per_s": n_q * pairs / search_s}
        if metric != "euclidean":
            bound = issue_rate / INSTR_PER_PAIR[metric]
            out["search_kernel"]["fp32_issue_bound_pairs_per_s"] = bound
            out["search_kernel"]["share_of_issue_bound"] = n_q * pairs / search_s / bound
            out["device"]["share_of_issue_bound_whole_call"] = n_q * pairs / t / bound
        else:
            # the Euclidean comparison point of the FP32 kernel: the same data through engine=SIMT
            L.set_option("engine", L.ENGINE_SIMT)
            L.set_option("timing", 1)
            try:
                device_call(ix, n_q)
                torch.cuda.synchronize(dev)
                ts_simt = timed(lambda: device_call(ix, n_q), 1)
                search_s = ix.stats()["search_ms"] * 1e-3
            finally:
                L.set_option("engine", L.ENGINE_AUTO)
                L.set_option("timing", 0)
            bound = issue_rate / INSTR_PER_PAIR["euclidean"]
            out["simt_engine"] = {"seconds": ts_simt, "queries_per_s": n_q / ts_simt[0], "search_seconds": search_s,
                                  "share_of_issue_bound": n_q * pairs / search_s / bound}
        # the filter's advantage: the exhaustive float64 kernel alone, on a subsample
        L.set_option("engine", L.ENGINE_EXACT)
        try:
            device_call(ix, 1000)
            torch.cuda.synchronize(dev)
            done, t0, step = 0, time.perf_counter(), 10_000
            while done < min(a.exact_rows, n_q) and time.perf_counter() - t0 < a.exact_seconds:
                rows = min(step, a.exact_rows - done)
                ix.query_device(X_dev[done:].data_ptr(), False, rows, a.dim, k, dist_ptr=o_d.data_ptr(),
                                idx_ptr=o_i.data_ptr(), pred_ptr=o_p.data_ptr(), weights="distance",
                                row_offset=done, stream=stream.cuda_stream)
                torch.cuda.synchronize(dev)
                done += rows
            te = time.perf_counter() - t0
        finally:
            L.set_option("engine", L.ENGINE_AUTO)
        out["exact"] = {"rows": done, "seconds": te, "queries_per_s": done / te,
                        "filtered_speedup": (n_q / t) / (done / te)}
        ix.close()
        # end to end through the estimator on a pageable NumPy array
        est = S.EuclideanKNNRegressor(n_neighbors=k, weights="distance", **ESTIMATOR_KW[metric]).fit(R, y)
        Xe = np.ascontiguousarray(xh[:a.e2e_rows])
        est.predict(Xe[:100_000])
        ts = []
        for _ in range(a.steps):
            t0 = time.perf_counter()
            est.predict(Xe)
            ts.append(time.perf_counter() - t0)
        out["e2e_estimator"] = {"rows": len(Xe), "seconds": ts, "queries_per_s": len(Xe) / min(ts)}
        del est
        # scikit-learn's brute search on the host, same metric
        from sklearn.neighbors import KNeighborsRegressor
        from threadpoolctl import threadpool_info

        reg = KNeighborsRegressor(n_neighbors=k, weights="distance", algorithm="brute", metric=metric,
                                  n_jobs=-1).fit(Z, y)
        Xc = (xh[:a.cpu_rows] - mean) / scale
        t0 = time.perf_counter()
        reg.predict(Xc)
        tc = time.perf_counter() - t0
        out["cpu_sklearn"] = {"rows": len(Xc), "seconds": tc, "queries_per_s": len(Xc) / tc,
                              "host_cpus": len(os.sched_getaffinity(0)),
                              "openmp_threads": [p.get("num_threads") for p in threadpool_info()
                                                 if p.get("user_api") == "openmp"]}
        print(json.dumps({metric: out}), flush=True)
    res["legs"] = legs
    res["gpu_after"] = gpu_info()
    doc = json.dumps(res, indent=1)
    print(doc)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(doc)


if __name__ == "__main__":
    main()
