"""Wide Hamming mode next to the 16-bit one at the same shape (GPU).

n_ref = 100 000 plots x T = 500 trees, 1M queries, k = 7, equal tree weights.  The node IDs mimic a
forest's: plots and queries are points of the unit square, and every tree is a grid of square leaves,
rotated and shifted at random, whose cell number is the node ID - so a query shares leaves with the
plots near it.  The wide leg's cells (side 0.003) give about 66 000 distinct IDs per tree among the
plots, 1.5 plots per leaf: more than 16-bit codes reach, so the index keeps exact 32-bit codes behind
the hashed 16-bit filter.  At that leaf size a query's 7th neighbour typically shares a leaf in no
tree or one, where hash collisions (about one per 31 743 tree pairs) outnumber true matches, which
is the hard case of the certificate (DESIGN.md section 5).  The narrow leg's cells (side 0.0065)
give about 23 500 IDs per tree, which fit.  Per leg:

  queries/s          one host-buffer HammingIndex.query of all rows (codes in, neighbours out)
  ID-compares/s      n_q x n_ref x T over the search kernel's time (CUDA events, option "timing")
  certified share    rows the float64 re-rank certified; exhaustive share: rows the exhaustive kernel took
  oracle             200 rows compared bit for bit with the oracle's SciPy-equal distances

and scikit-learn's brute Hamming search (the reference) on a sample of the wide queries.  One JSON
document goes to stdout (and to --out); the GPU's name and power limit are read in the same process.
Needs a CUDA device: without one it fails.

    python scripts/hamming_wide_bench.py [--queries N] [--cpu-rows N] [--out FILE]
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

N_REF, T, K = 100_000, 500, 7


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                       capture_output=True, text=True)
    return r.stdout.strip()


def node_ids(points, cell, T, seed):
    """[n, T] int64: the cell of every point in each tree's rotated, shifted grid of side `cell`."""
    rng = np.random.default_rng(seed)
    out = np.empty((len(points), T), dtype=np.int64)
    for t in range(T):
        th = rng.uniform(0, np.pi / 2)
        c, s = np.cos(th), np.sin(th)
        u = (points[:, 0] * c - points[:, 1] * s + 1.0 + rng.uniform(0, cell)) // cell
        v = (points[:, 0] * s + points[:, 1] * c + rng.uniform(0, cell)) // cell
        out[:, t] = u.astype(np.int64) * 100_000 + v.astype(np.int64)
    return out


def data(cell, n_q):
    rng = np.random.default_rng(0)
    R = node_ids(rng.random((N_REF, 2)), cell, T, 1)
    Q = node_ids(rng.random((n_q, 2)), cell, T, 1)    # the same trees (seed 1)
    return R, Q


def leg(name, cell, n_q):
    from oracle import sknnr_oracle as orc
    from sknnr_b200 import _lib as L
    from sknnr_b200._base import _encode_nodes, _node_code_tables
    from sknnr_b200._engine import HammingIndex

    R, Q = data(cell, n_q)
    distinct = min(len(np.unique(R[:, t])) for t in range(4))
    tables = _node_code_tables(R)
    Rc, Qc = _encode_nodes(R, tables), _encode_nodes(Q, tables)
    w = np.full(T, 1.0 / T)
    ix = HammingIndex(Rc, w, device=0)
    ix.query(Qc[:50_000], K)                                   # warm-up
    L.set_option("timing", 1)
    try:
        t0 = time.perf_counter()
        d, i, _ = ix.query(Qc, K)
        dt = time.perf_counter() - t0
        st = ix.stats()
    finally:
        L.set_option("timing", 0)
    cc = ix.cascade_counts()
    r0 = n_q // 3
    rows = slice(r0, r0 + 200)       # (the ordering key holds the query's row number: row_offset)
    st_o = orc.FittedState("hamming", fit_Z=R, y=np.zeros((N_REF, 1)), hamming_w=w)
    d_o, i_o = orc.kneighbors(st_o, Q[rows], k=K, row_offset=r0)
    return {
        "leg": name, "wide": bool(ix.wide), "distinct_ids_per_tree_min_of_4": int(distinct),
        "n_ref": N_REF, "T": T, "n_q": n_q, "k": K,
        "queries_per_s": n_q / dt, "call_s": dt,
        "search_ms": st["search_ms"],
        "id_compares_per_s": n_q * N_REF * T / (st["search_ms"] * 1e-3) if st["search_ms"] else None,
        "certified_share": (1.0 - cc["uncertified"] / n_q) if ix.wide else None,
        "exhaustive_share": cc["to_exact"] / n_q,
        "oracle_rows_bit_equal": bool(np.array_equal(d[rows], d_o) and np.array_equal(i[rows], i_o)),
    }, (R, Q, w)


def reference_rate(R, Q, w, rows):
    from sklearn.neighbors import KNeighborsRegressor

    ref = KNeighborsRegressor(n_neighbors=K, metric="hamming", metric_params={"w": w}, algorithm="brute",
                              n_jobs=-1).fit(R, np.zeros(len(R)))
    t0 = time.perf_counter()
    ref.kneighbors(Q[:rows])
    return rows / (time.perf_counter() - t0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--queries", type=int, default=1_000_000)
    ap.add_argument("--cpu-rows", type=int, default=100)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    out = {"gpu": gpu_info(), "legs": []}
    wide, (R, Q, w) = leg("wide", 0.003, a.queries)
    out["legs"].append(wide)
    print(json.dumps(wide), flush=True)
    out["reference_queries_per_s"] = reference_rate(R, Q, w, a.cpu_rows)
    del R, Q
    narrow, _ = leg("narrow", 0.0065, a.queries)
    out["legs"].append(narrow)
    print(json.dumps(narrow), flush=True)
    out["wide_over_narrow_queries_per_s"] = wide["queries_per_s"] / narrow["queries_per_s"]
    print(json.dumps(out, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
