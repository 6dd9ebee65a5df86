"""Integer query inputs against the same values in floating point (GPU).

C3-shaped data (BASELINE.md section 3): 50 000 plots x 32 features, 8 targets, k = 7,
weights="distance", an EuclideanKNNRegressor.  Plots and queries are round(N(0, 1) * 1000), the
queries held as int16 (scaled reflectance) and, for the comparison, as the same values in float64 /
float32.  Legs, each timed alternately per dtype after one warm-up call of every variant:

  predict   est.predict(X) on a pageable 10M-row array
  pinned    the index's host-buffer call (sknnr_kneighbors) on page-locked X and result arrays
  raster    predict_raster on a [32, 2500, 4000] image with 5 % nodata pixels (int16 / float32 / float64)
  rfnn      RFNNRegressor (C4 shape: 20 000 plots x 16 features, 10 targets) est.predict on 2M rows

Every leg asserts that the integer and the float outputs are bit-identical.  Per call it reports the
host wall clock (the calls are synchronous), queries / s and the bytes the library copied to and from
the device (``sknnr_stats``).  The script only uses the public surface, so the same file run against
an older build of the project gives that build's numbers for the same inputs.  One JSON document goes
to stdout (and to --out); the GPU's name and power limit are read in the same process.  Needs a CUDA
device: without one it fails.

    python scripts/int_input_bench.py [--rows N] [--steps N] [--legs predict,pinned,raster,rfnn]
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                       capture_output=True, text=True)
    return r.stdout.strip()


def scaled_int16(rng, shape):
    return np.rint(rng.standard_normal(shape) * 1000.0).astype(np.int16)


def run_leg(variants, steps, rows, index_of):
    """variants: {name: call}.  One warm-up call each, then `steps` rounds alternating the variants.
    Returns the per-variant record and the last output of each."""
    outs = {}
    for name, call in variants.items():
        outs[name] = call()
    times = {name: [] for name in variants}
    stats = {}
    for _ in range(steps):
        for name, call in variants.items():
            t0 = time.perf_counter()
            outs[name] = call()
            times[name].append(time.perf_counter() - t0)
            stats[name] = index_of().stats()
    rec = {}
    for name, ts in times.items():
        med = statistics.median(ts)
        rec[name] = {"times_s": [round(t, 5) for t in ts], "median_s": round(med, 5),
                     "spread_s": round(max(ts) - min(ts), 5), "queries_per_s_M": round(rows / med / 1e6, 2),
                     "h2d_bytes": int(stats[name]["h2d_bytes"]), "d2h_bytes": int(stats[name]["d2h_bytes"])}
    return rec, outs


def assert_same(outs, leg):
    names = list(outs)
    for n in names[1:]:
        a, b = outs[names[0]], outs[n]
        assert a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a, b, equal_nan=True), \
            f"{leg}: {names[0]} and {n} outputs differ"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--n-ref", type=int, default=50_000)
    ap.add_argument("--dim", type=int, default=32)
    ap.add_argument("--n-out", type=int, default=8)
    ap.add_argument("--k", type=int, default=7)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--raster", default="2500x4000", help="image height x width")
    ap.add_argument("--rfnn-rows", type=int, default=2_000_000)
    ap.add_argument("--rfnn-trees", type=int, default=50, help="trees per target forest")
    ap.add_argument("--legs", default="predict,pinned,raster,rfnn")
    ap.add_argument("--out", default="")
    a = ap.parse_args()

    import sknnr_b200 as S
    from sknnr_b200 import _lib as L
    from sknnr_b200._engine import pinned_empty

    if L.device_count() < 1:
        raise SystemExit("int_input_bench.py needs a CUDA device")
    legs = set(a.legs.split(","))
    doc = {"gpu": gpu_info(), "rows": a.rows, "n_ref": a.n_ref, "dim": a.dim, "k": a.k, "steps": a.steps,
           "queries": "round(N(0,1) * 1000)", "legs": {}}

    R = scaled_int16(np.random.default_rng(0), (a.n_ref, a.dim)).astype(np.float64)
    y = np.random.default_rng(1).standard_normal((a.n_ref, a.n_out))
    t0 = time.perf_counter()
    est = S.EuclideanKNNRegressor(n_neighbors=a.k, weights="distance").fit(R, y)
    doc["fit_s"] = round(time.perf_counter() - t0, 3)
    ix = est.regressor_._get_index()
    index_of = lambda: ix  # noqa: E731

    Xi = scaled_int16(np.random.default_rng(2), (a.rows, a.dim))
    if "predict" in legs:
        Xf = Xi.astype(np.float64)
        rec, outs = run_leg({"int16": lambda: est.predict(Xi), "float64": lambda: est.predict(Xf)},
                            a.steps, a.rows, index_of)
        assert_same(outs, "predict")
        doc["legs"]["predict"] = rec
        del Xf, outs
    if "pinned" in legs:
        Xip = pinned_empty(Xi.shape, np.int16)
        Xip[:] = Xi
        Xfp = pinned_empty(Xi.shape, np.float64)
        Xfp[:] = Xi
        preds = {n: pinned_empty((a.rows, a.n_out)) for n in ("int16", "float64")}

        def call(X, name):
            ix.query(X, a.k, weights="distance", with_pred=True, return_distance=False, return_index=False,
                     out=(None, None, preds[name]))
            return preds[name]

        rec, outs = run_leg({"int16": lambda: call(Xip, "int16"), "float64": lambda: call(Xfp, "float64")},
                            a.steps, a.rows, index_of)
        assert_same(outs, "pinned")
        doc["legs"]["pinned"] = rec
        del Xip, Xfp, preds, outs
    del Xi

    if "raster" in legs:
        H, W = (int(v) for v in a.raster.split("x"))
        rng = np.random.default_rng(3)
        img = scaled_int16(rng, (a.dim, H, W))
        holes = rng.random((H, W)) < 0.05
        band = rng.integers(0, a.dim, int(holes.sum()))
        hy, hx = np.nonzero(holes)
        img[band, hy, hx] = -32768                 # nodata: no value of round(N(0,1) * 1000) reaches it
        img32, img64 = img.astype(np.float32), img.astype(np.float64)
        rec, outs = run_leg({"int16": lambda: S.predict_raster(est, img, nodata=-32768),
                             "float32": lambda: S.predict_raster(est, img32, nodata=-32768),
                             "float64": lambda: S.predict_raster(est, img64, nodata=-32768)},
                            a.steps, H * W, index_of)
        assert_same(outs, "raster")
        rec["nodata_pixels"] = int(holes.sum())
        doc["legs"]["raster"] = rec
        del img, img32, img64, outs

    if "rfnn" in legs:
        n4, d4, t4 = 20_000, 16, 10
        X4 = np.random.default_rng(0).standard_normal((n4, d4))
        y4 = X4[:, :t4] * 2.0 + np.random.default_rng(1).standard_normal((n4, t4))
        X4 = np.rint(X4 * 1000.0)
        t0 = time.perf_counter()
        rf = S.RFNNRegressor(n_estimators=a.rfnn_trees, random_state=0, n_neighbors=a.k, n_jobs=-1).fit(X4, y4)
        Qi = scaled_int16(np.random.default_rng(4), (a.rfnn_rows, d4))
        Qf = Qi.astype(np.float64)
        rix = rf.regressor_._get_index()
        rec, outs = run_leg({"int16": lambda: rf.predict(Qi), "float64": lambda: rf.predict(Qf)},
                            a.steps, a.rfnn_rows, lambda: rix)
        assert_same(outs, "rfnn")
        rec["fit_s"] = round(time.perf_counter() - t0, 3)
        rec["trees"] = a.rfnn_trees * t4
        doc["legs"]["rfnn"] = rec

    text = json.dumps(doc, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
