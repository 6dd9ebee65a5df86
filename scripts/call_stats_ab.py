"""Per-call counters of two builds of the library, entry point by entry point (GPU).

Makes one call of each entry point on small seeded inputs and records, after every call, the index's
``stats()`` (queries, uncertified rows, kernel launches, bytes copied each way, engine) and, for a
float index, ``cascade_counts()``, plus a digest of the call's outputs.  Small chunk sizes make every
call run several chunks, so the host pipeline, its ramp, the slot rotation and the raster look-ahead
all take part.  Entry points: host-buffer and device-pointer kneighbors on float64 / float32 / int16
rows, SKNNR_EXCLUDE_SELF, SKNNR_CHECK_FINITE (clean and with a NaN), a k beyond the filtered engines,
raster calls of both index kinds, Hamming queries on node codes (host and device pointers, equal and
unequal tree weights, 16-bit and wide indexes of the same node IDs) and through a device forest walk,
transform and both weighted averages.

    python scripts/call_stats_ab.py LIB_A LIB_B [--repeats N] [--out FILE]

runs the calls N times against each library, alternating (``SKNNR_B200_LIB``, one process per run),
and exits with 1 if a value is the same in every run of each library but differs between the two.
A value that differs between runs of one library is listed apart, with every run's value: the
tensor engine's first-pass failure count can (its two candidate streams of a query read each other's
thresholds while both run), although the results it leaves are certified and bit-identical.
``python scripts/call_stats_ab.py --record`` prints the records of the library the package loads.
Needs a CUDA device: without one it fails.
"""

from __future__ import annotations

import argparse
import hashlib
import itertools
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def digest(*arrays):
    h = hashlib.sha1()
    for a in arrays:
        if a is not None:
            h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def record() -> dict:
    import torch
    from sklearn.ensemble import RandomForestRegressor

    from sknnr_b200 import _lib as L
    from sknnr_b200._engine import ForestIndex, HammingIndex, KNNIndex

    L.set_option("chunk_rows", 8192)
    L.set_option("stage_rows", 4096)
    rng = np.random.default_rng(20)
    out = {}

    # ---- float index: 20 000 plots, 16 features, projected to 12, 3 targets
    n_ref, d_in, d_out, n_q, k = 20_000, 16, 12, 60_000, 7
    R = np.rint(rng.standard_normal((n_ref, d_in)) * 1000.0)
    center, scale = R.mean(0), R.std(0)
    proj = rng.standard_normal((d_in, d_out))
    ix = KNNIndex(((R - center) / scale) @ proj, center, scale, proj, rng.standard_normal((n_ref, 3)))
    X = np.rint(rng.standard_normal((n_q, d_in)) * 1000.0)

    def keep(name, res, index, cascade):
        rec = {f"stats.{f}": v for f, v in index.stats().items()}
        if cascade:
            rec.update({f"cascade.{f}": v for f, v in index.cascade_counts().items()})
        rec["out"] = digest(*(res if isinstance(res, tuple) else (res,)))
        out[name] = rec

    def knn(name, call):
        keep(name, call(), ix, True)

    for dt in (np.float64, np.float32, np.int16):
        Xd = X.astype(dt)
        knn(f"knn_host_{np.dtype(dt).name}", lambda: ix.query(Xd, k, weights="distance", with_pred=True))
        xd = torch.from_numpy(Xd).cuda()
        res = [torch.empty((n_q, k), dtype=torch.float64, device="cuda"),
               torch.empty((n_q, k), dtype=torch.int64, device="cuda"),
               torch.empty((n_q, 3), dtype=torch.float64, device="cuda")]

        def dev():
            ix.query_device(xd.data_ptr(), False, n_q, d_in, k, dist_ptr=res[0].data_ptr(),
                            idx_ptr=res[1].data_ptr(), pred_ptr=res[2].data_ptr(), weights="uniform",
                            stream=torch.cuda.current_stream().cuda_stream, x_dtype=dt)
            torch.cuda.synchronize()
            return tuple(t.cpu().numpy() for t in res)

        knn(f"knn_device_{np.dtype(dt).name}", dev)
    knn("knn_exclude_self", lambda: ix.query(None, k, exclude_self=True, weights="uniform", with_pred=True))
    knn("knn_check_finite", lambda: ix.query(X, k, check_finite=True))
    Xn = X.copy()
    Xn[12345, 3] = np.nan

    def nonfinite():
        try:
            ix.query(Xn, k, check_finite=True)
        except L.NonFiniteInput:
            return np.array([1])
        return np.array([0])

    knn("knn_check_finite_nan", nonfinite)
    knn("knn_large_k", lambda: ix.query(X[:5000], 40))
    bands = np.ascontiguousarray(np.rint(rng.standard_normal((d_in, 50_000)) * 1000.0).astype(np.int16))
    bands[:, rng.random(50_000) < 0.1] = -9999
    knn("raster_int16", lambda: ix.query_raster(bands, k, nodata=-9999, weights="distance", with_pred=True))
    knn("raster_float64", lambda: ix.query_raster(bands.astype(np.float64), k, nodata=-9999))
    knn("transform", lambda: ix.transform(X[:30_000]))
    d, i, _ = ix.query(X[:30_000], k)
    knn("weighted_average", lambda: ix.weighted_average(i, 1.0 / (1.0 + d)))
    ix.close()

    # ---- tree-node index: a random forest's node IDs as codes
    n_ref, n_feat, n_q, k = 8_000, 10, 40_000, 5
    Rf = rng.standard_normal((n_ref, n_feat))
    y = Rf[:, :2] @ rng.standard_normal((2, 2)) + 0.1 * rng.standard_normal((n_ref, 2))
    rf = RandomForestRegressor(n_estimators=40, max_depth=8, random_state=0).fit(Rf, y)
    forest = ForestIndex([e.tree_ for e in rf.estimators_], n_feat)
    codes = forest.apply(Rf).astype(np.uint16)
    Xf = rng.standard_normal((n_q, n_feat))
    qcodes = forest.apply(Xf).astype(np.uint16)
    out["forest_apply"] = {"out": digest(qcodes)}
    tree_weights = (("equal", np.full(40, 1.0 / 40)), ("unequal", rng.uniform(0.5, 1.5, 40)))
    # the wide legs: the same node IDs as exact u32 codes (wide mode's filter and re-rank)
    for (wname, w), wide in itertools.product(tree_weights, (False, True)):
        hq = qcodes.astype(np.uint32) if wide else qcodes
        hx = HammingIndex(codes.astype(np.uint32) if wide else codes, w, y)

        def ham(name, call):
            keep(f"hamming_{'wide_' if wide else ''}{wname}_{name}", call(), hx, False)

        ham("codes_host", lambda: hx.query(hq, k, weights="distance", with_pred=True))
        qd = torch.from_numpy(qcodes.astype(np.int32 if wide else np.int16)).cuda()
        res = [torch.empty((n_q, k), dtype=torch.float64, device="cuda"),
               torch.empty((n_q, k), dtype=torch.int64, device="cuda")]

        def hdev():
            hx.query_device(qd.data_ptr(), n_q, 40, k, dist_ptr=res[0].data_ptr(), idx_ptr=res[1].data_ptr(),
                            stream=torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
            return tuple(t.cpu().numpy() for t in res)

        ham("codes_device", hdev)
        ham("exclude_self", lambda: hx.query(None, k, exclude_self=True))
        ham("forest_float64", lambda: hx.query_forest(forest, Xf, k, weights="uniform", with_pred=True))
        ham("forest_int16", lambda: hx.query_forest(forest, np.rint(Xf * 100).astype(np.int16), k))
        fb = np.ascontiguousarray(rng.standard_normal((n_feat, 30_000)))
        fb[:, rng.random(30_000) < 0.1] = np.nan
        ham("raster_forest", lambda: hx.query_raster_forest(forest, fb, k, weights="distance", with_pred=True))
        hd, hi, _ = hx.query(hq[:10_000], k)
        ham("weighted_average", lambda: hx.weighted_average(hi, 1.0 / (1.0 + hd)))
        hx.close()
    forest.close()
    return out


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("libs", nargs="*", help="two library builds to compare")
    ap.add_argument("--record", action="store_true", help="print this process's records and exit")
    ap.add_argument("--repeats", type=int, default=3, help="runs per library (default 3)")
    ap.add_argument("--out", help="also write the comparison to this JSON file")
    a = ap.parse_args()
    if a.record:
        print(json.dumps(record()))
        return 0
    if len(a.libs) != 2 or a.repeats < 1:
        ap.error("give two library paths and --repeats >= 1, or --record")
    runs = {lib: [] for lib in a.libs}
    for _ in range(a.repeats):
        for lib in a.libs:
            env = dict(os.environ, SKNNR_B200_LIB=os.path.abspath(lib))
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--record"], env=env,
                               capture_output=True, text=True, check=True)
            runs[lib].append(json.loads(r.stdout.strip().splitlines()[-1]))
    first = runs[a.libs[0]][0]
    differ, varying = {}, {}
    for call in sorted(set().union(*(r.keys() for rs in runs.values() for r in rs))):
        for field in sorted(set().union(*(r.get(call, {}).keys() for rs in runs.values() for r in rs))):
            vals = {lib: [r.get(call, {}).get(field) for r in rs] for lib, rs in runs.items()}
            seen = [json.dumps(v) for vs in vals.values() for v in vs]
            if len(set(seen)) == 1:
                continue
            steady = all(len({json.dumps(v) for v in vs}) == 1 for vs in vals.values())
            (differ if steady else varying)[f"{call} {field}"] = vals
    doc = {"libs": a.libs, "repeats": a.repeats, "calls": len(first), "differ": differ,
           "varying_within_a_build": varying, "records": first}
    text = json.dumps(doc, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")
    return 1 if differ else 0


if __name__ == "__main__":
    sys.exit(main())
