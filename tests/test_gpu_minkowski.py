"""GPU tests of the Manhattan / Chebyshev searches (metric="manhattan" / p=1, "chebyshev" / p=inf).

The reference is scikit-learn's own brute search: its distances come from ManhattanDistance64 /
ChebyshevDistance64, which `DistanceMetric.get_metric(...).pairwise` runs as well.  `_reference`
takes the k nearest by (distance, index) from that matrix, i.e. the lowest index wins every tie at
the k-th position, then applies sknnr's glue (self exclusion, deterministic ordering).  The device's
distances must equal it bit for bit."""

import numpy as np
import pytest
from sklearn.metrics import DistanceMetric, r2_score
from sklearn.neighbors import KNeighborsRegressor

from oracle import sknnr_oracle as orc
from tests.conftest import load_golden, yaimpute_weights

pytestmark = pytest.mark.gpu

METRICS = ["manhattan", "chebyshev"]
SPELLINGS = [("manhattan", {"metric": "manhattan"}), ("manhattan", {"metric": "cityblock"}),
             ("manhattan", {"metric": "l1"}), ("manhattan", {"p": 1}),
             ("chebyshev", {"metric": "chebyshev"}), ("chebyshev", {"metric": "infinity"}),
             ("chebyshev", {"p": np.inf})]


def _reference(metric, R, Q, k, deterministic=True):
    """(dist, idx) of a kneighbors call; Q=None is the X=None self-query."""
    self_query = Q is None
    D = DistanceMetric.get_metric(metric).pairwise(R if self_query else np.asarray(Q, dtype=np.float64), R)
    kk = k + 1 if self_query else k
    idx = np.argsort(D, axis=1, kind="stable")[:, :kk]    # stable: equal distances keep index order
    dist = np.take_along_axis(D, idx, axis=1)
    if self_query:
        dist, idx = orc.exclude_self(dist, idx)
    if deterministic:
        dist, idx = orc.deterministic_order(dist, idx)
    return dist, idx


def _assert_sklearn_agrees(metric, R, y, Q, k):
    """scikit-learn's KNeighborsRegressor returns the same distances as `_reference`; its indices may
    differ only among references tied with the k-th distance."""
    reg = KNeighborsRegressor(n_neighbors=k, algorithm="brute", metric=metric).fit(R, y)
    sd, si = reg.kneighbors(Q)
    rd, ri = _reference(metric, R, Q, k, deterministic=False)
    np.testing.assert_array_equal(sd, rd)
    kth = rd[:, -1:]
    for r in np.flatnonzero((si != ri).any(axis=1)):
        inside = rd[r] < kth[r]
        assert set(si[r][inside]) == set(ri[r][inside]), r


def _pred(y, dist, idx, weights):
    return orc.weighted_average(y, idx, orc.get_weights(dist, weights))


def _data(n_ref, n_q, d, seed, offset=0.0, grid=False, dup=True, n_out=3):
    rng = np.random.default_rng(seed)
    if grid:   # integer features: exact distance ties everywhere, at the k-th position included
        R = rng.integers(0, 4, (n_ref, d)).astype(np.float64)
        Q = rng.integers(0, 4, (n_q, d)).astype(np.float64)
    else:
        R = rng.standard_normal((n_ref, d))
        Q = rng.standard_normal((n_q, d))
    if dup and n_ref >= 8:
        R[n_ref // 2: n_ref // 2 + 4] = R[:4]          # duplicated plots
        Q[: min(n_q, 6)] = R[rng.integers(0, n_ref, min(n_q, 6))]   # queries on plots: zero distances
    R += offset
    Q += offset
    y = rng.standard_normal((n_ref, n_out))
    return R, Q, y


def _index(R, y, metric):
    from sknnr_b200._engine import KNNIndex

    return KNNIndex(R, None, None, None, y, metric=metric)


# ---- the raw estimator, every spelling of the two metrics ------------------------------------
@pytest.mark.parametrize("grid", [False, True])
@pytest.mark.parametrize(("metric", "kw"), SPELLINGS)
def test_raw_estimator_bit_identical_to_scikit_learn(metric, kw, grid):
    import pandas as pd

    import sknnr_b200 as S

    k = 5
    R, Q, y = _data(900, 300, 6, seed=11, offset=0.0 if grid else 5e5, grid=grid)
    _assert_sklearn_agrees(metric, R, y, Q, k)
    est = S.RawKNNRegressor(n_neighbors=k, **kw).fit(R, y)
    assert est._metric_kind() == metric
    rd, ri = _reference(metric, R, Q, k)
    d, i = est.kneighbors(Q)
    np.testing.assert_array_equal(d, rd)
    np.testing.assert_array_equal(i, ri)
    sd, si = _reference(metric, R, None, k)
    d, i = est.kneighbors()
    np.testing.assert_array_equal(d, sd)
    np.testing.assert_array_equal(i, si)
    np.testing.assert_allclose(est.independent_prediction_, _pred(y, sd, si, "uniform"), rtol=1e-12, atol=1e-14)
    assert est.independent_score_ == pytest.approx(r2_score(y, _pred(y, sd, si, "uniform")), rel=1e-12)
    np.testing.assert_allclose(est.predict(Q), _pred(y, rd, ri, "uniform"), rtol=1e-12, atol=1e-14)
    for w in ("distance", yaimpute_weights):
        ew = S.RawKNNRegressor(n_neighbors=k, weights=w, **kw).fit(R, y)
        np.testing.assert_allclose(ew.predict(Q), _pred(y, rd, ri, w), rtol=1e-12, atol=1e-14)
        np.testing.assert_allclose(ew.independent_prediction_, _pred(y, sd, si, w), rtol=1e-12, atol=1e-14)
    # dataframe index crosswalk
    ids = np.arange(len(R)) * 7 + 1000
    ef = S.RawKNNRegressor(n_neighbors=k, **kw).fit(pd.DataFrame(R, index=ids), y)
    d, i = ef.kneighbors(pd.DataFrame(Q), return_dataframe_index=True)
    np.testing.assert_array_equal(d, rd)
    np.testing.assert_array_equal(i, ids[ri])


# ---- adversarial shapes through the index: every engine of the cascade -----------------------
# d = 113 (dpad 120) is one past what the FP32 kernel's shared memory holds with lists of 16;
# k + 1 > 32 (k = 32 with the self-query, k = 40) is the exhaustive kernel's alone
CASES = [
    # metric, n_ref, n_q, d, k, self_query, offset, f32, grid
    ("manhattan", 1000, 700, 1, 7, False, 0.0, False, False),
    ("chebyshev", 1000, 700, 1, 7, True, 0.0, False, False),
    ("manhattan", 1000, 700, 7, 1, False, 5e5, False, False),
    ("chebyshev", 1000, 700, 7, 15, True, 5e5, False, False),
    ("manhattan", 1000, 700, 32, 15, True, 0.0, True, False),
    ("chebyshev", 1000, 700, 32, 31, False, 0.0, False, False),
    ("manhattan", 1000, 700, 64, 31, False, 5e5, False, False),
    ("chebyshev", 1000, 700, 64, 7, False, 0.0, True, False),
    ("manhattan", 1000, 300, 113, 7, True, 0.0, False, False),
    ("chebyshev", 1000, 300, 113, 7, False, 5e5, False, False),
    ("manhattan", 37, 200, 7, 7, True, 0.0, False, False),
    ("chebyshev", 37, 200, 32, 1, False, 0.0, False, False),
    ("manhattan", 1000, 400, 7, 32, True, 0.0, False, False),
    ("chebyshev", 1000, 400, 7, 32, True, 0.0, False, False),
    ("manhattan", 1000, 400, 7, 40, False, 5e5, False, False),
    ("chebyshev", 1000, 400, 7, 40, True, 0.0, False, False),
    ("manhattan", 1000, 700, 5, 7, False, 0.0, False, True),
    ("chebyshev", 1000, 700, 5, 7, True, 0.0, False, True),
    ("manhattan", 1000, 700, 5, 31, True, 0.0, True, True),
    ("chebyshev", 1000, 700, 5, 15, False, 0.0, True, True),
]


@pytest.mark.parametrize(("metric", "n_ref", "n_q", "d", "k", "self_query", "offset", "f32", "grid"), CASES)
def test_adversarial_shapes_bit_identical(metric, n_ref, n_q, d, k, self_query, offset, f32, grid):
    R, Q, y = _data(n_ref, n_q, d, seed=d * 100 + k, offset=offset, grid=grid)
    if f32:
        Q = Q.astype(np.float32)
    ix = _index(R, y, metric)
    for weights in ("uniform", "distance"):
        if self_query:
            dd, ii, pp = ix.query(None, k, exclude_self=True, weights=weights, with_pred=True)
            rd, ri = _reference(metric, R, None, k)
        else:
            dd, ii, pp = ix.query(Q, k, transformed=True, weights=weights, with_pred=True)
            rd, ri = _reference(metric, R, Q, k)
        np.testing.assert_array_equal(dd, rd)
        np.testing.assert_array_equal(ii, ri)
        np.testing.assert_allclose(pp, _pred(y, rd, ri, weights), rtol=1e-12, atol=1e-14)


def test_engines_agree_and_the_fp32_filter_does_the_work():
    from sknnr_b200 import _lib as L

    rng = np.random.default_rng(5)
    for case in range(20):
        metric = METRICS[case % 2]
        n_ref = int(rng.integers(20, 3000))
        d = int(rng.integers(1, 70))
        k = int(rng.integers(1, min(n_ref, 31)))
        offset = [0.0, 5e5, -3.0][case % 3]
        R, Q, y = _data(n_ref, int(rng.integers(1, 900)), d, seed=1000 + case, offset=offset,
                        grid=case % 5 == 4)
        ix = _index(R, y, metric)
        # (lists of 32 candidates, k >= 16, leave shared memory for 64 features: beyond, SIMT means exhaustive)
        fits = k <= 15 or -(-d // 8) * 8 <= 64
        out = {}
        try:
            for engine in (L.ENGINE_SIMT, L.ENGINE_EXACT):
                L.set_option("engine", engine)
                out[engine] = ix.query(Q, k, transformed=True, weights="distance", with_pred=True)
                st = ix.stats()
                assert st["engine"] == (engine if fits else L.ENGINE_EXACT), (case, st)
                if engine == L.ENGINE_SIMT and fits:
                    assert ix.cascade_counts()["to_fp32"] == len(Q)
        finally:
            L.set_option("engine", L.ENGINE_AUTO)
        for a, b in zip(out[L.ENGINE_SIMT], out[L.ENGINE_EXACT]):
            np.testing.assert_array_equal(a, b)
        rd, ri = _reference(metric, R, Q, k)
        np.testing.assert_array_equal(out[L.ENGINE_EXACT][0], rd)
        np.testing.assert_array_equal(out[L.ENGINE_EXACT][1], ri)

    # C3-like data: N(0, 1), 50k plots, 32 features, k = 7 - the FP32 filter certifies > 99 % of the rows
    R, Q, y = _data(50_000, 20_000, 32, seed=7, dup=False)
    for metric in METRICS:
        ix = _index(R, y, metric)
        for engine in (L.ENGINE_AUTO, L.ENGINE_TENSOR):   # (no tensor engine for these metrics: both pick SIMT)
            try:
                L.set_option("engine", engine)
                d, i, _ = ix.query(Q, 7, transformed=True)
            finally:
                L.set_option("engine", L.ENGINE_AUTO)
            assert ix.stats()["engine"] == L.ENGINE_SIMT
            cc = ix.cascade_counts()
            assert cc["to_fp32"] == len(Q)
            assert cc["to_exact"] < 0.01 * len(Q), (metric, cc)
        rd, ri = _reference(metric, R, Q[:2000], 7)
        np.testing.assert_array_equal(d[:2000], rd)
        np.testing.assert_array_equal(i[:2000], ri)


def test_huge_magnitudes_fall_back_like_the_exact_engine():
    from sknnr_b200 import _lib as L

    rng = np.random.default_rng(9)
    R, Q, y = _data(3000, 500, 32, seed=9)
    Q[7, :5] = 1e37                      # its FP32 score overflows: the row is never certified
    Q[8] = -3e37
    Rb = R.copy()
    Rb[11, :4] = rng.choice([-1.0, 1.0], 4) * 5e37   # a plot past the FP32 limit: exhaustive-only index
    for metric in METRICS:
        for plots, want_engine in ((R, L.ENGINE_SIMT), (Rb, L.ENGINE_EXACT)):
            ix = _index(plots, y, metric)
            got = ix.query(Q, 7, transformed=True, weights="distance", with_pred=True)
            assert ix.stats()["engine"] == want_engine
            try:
                L.set_option("engine", L.ENGINE_EXACT)
                ref = ix.query(Q, 7, transformed=True, weights="distance", with_pred=True)
            finally:
                L.set_option("engine", L.ENGINE_AUTO)
            for a, b in zip(got, ref):
                np.testing.assert_array_equal(a, b)
            rd, ri = _reference(metric, plots, Q, 7)
            np.testing.assert_array_equal(got[0], rd)
            np.testing.assert_array_equal(got[1], ri)


# ---- transformed estimators: the fused projection in front of the search ----------------------
def _moscow():
    sp = load_golden("moscow_split.npz")
    return sp["X_train"], sp["X_test"], sp["y_train"]


@pytest.mark.parametrize("kw", [{"p": 1}, {"metric": "chebyshev"}])
@pytest.mark.parametrize("name", ["EuclideanKNNRegressor", "MahalanobisKNNRegressor", "MSNRegressor",
                                  "GNNRegressor"])
def test_transformed_estimators_match_scikit_learn_on_the_transformed_data(name, kw):
    import sknnr_b200 as S

    metric = "manhattan" if kw.get("p") == 1 else "chebyshev"
    Xtr, Xte, ytr = _moscow()
    k = 5
    est = getattr(S, name)(n_neighbors=k, **kw).fit(Xtr, ytr)
    Zfit = est.transformer_.transform(Xtr)
    Zte = est.transformer_.transform(Xte)
    _assert_sklearn_agrees(metric, Zfit, ytr, Zte, k)
    rd, ri = _reference(metric, Zfit, Zte, k)
    d, i = est.kneighbors(Xte)
    orc.assert_tie_aware_equal(d, i, rd, ri, rtol=1e-12, atol=1e-12)
    if name == "EuclideanKNNRegressor":
        # (the scaler is the same float64 subtraction and division on both sides: nothing to round differently)
        np.testing.assert_array_equal(d, rd)
    np.testing.assert_allclose(est.predict(Xte), _pred(ytr, rd, ri, "uniform"), rtol=1e-10, atol=1e-12)
    sd, si = _reference(metric, Zfit, None, k)
    d, i = est.kneighbors()
    orc.assert_tie_aware_equal(d, i, sd, si, rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(est.independent_prediction_, _pred(ytr, sd, si, "uniform"), rtol=1e-10, atol=1e-12)
    ed = getattr(S, name)(n_neighbors=k, weights="distance", **kw).fit(Xtr, ytr)
    np.testing.assert_allclose(ed.predict(Xte), _pred(ytr, rd, ri, "distance"), rtol=1e-10, atol=1e-12)


# ---- call paths ----------------------------------------------------------------------------
@pytest.mark.parametrize("metric", METRICS)
def test_host_chunks_device_pointers_and_devices_agree(metric):
    import torch

    from sknnr_b200 import _lib as L
    from sknnr_b200._sharding import MultiDeviceIndex

    R, Q, y = _data(4000, 5000, 12, seed=21, offset=5e5)
    ix = _index(R, y, metric)
    one = ix.query(Q, 7, transformed=True, weights="distance", with_pred=True)
    try:
        L.set_option("chunk_rows", 256)
        many = ix.query(Q, 7, transformed=True, weights="distance", with_pred=True)
    finally:
        L.set_option("chunk_rows", 1 << 20)
    for a, b in zip(one, many):
        np.testing.assert_array_equal(a, b)

    dev = torch.device("cuda", ix.device)
    xq = torch.from_numpy(Q).to(dev)
    dd = torch.empty((len(Q), 7), dtype=torch.float64, device=dev)
    di = torch.empty((len(Q), 7), dtype=torch.int64, device=dev)
    dp = torch.empty((len(Q), y.shape[1]), dtype=torch.float64, device=dev)
    ix.query_device(xq.data_ptr(), False, len(Q), Q.shape[1], 7, dist_ptr=dd.data_ptr(), idx_ptr=di.data_ptr(),
                    pred_ptr=dp.data_ptr(), weights="distance", transformed=True,
                    stream=torch.cuda.current_stream(dev).cuda_stream)
    torch.cuda.synchronize(dev)
    for a, b in zip(one, (dd, di, dp)):
        np.testing.assert_array_equal(a, b.cpu().numpy())

    mi = MultiDeviceIndex(lambda dv: _index(R, y, metric), [0, 0, 0])
    mi.min_rows_per_device = 1000   # split this query over all three handles
    try:
        multi = mi.query(Q, 7, transformed=True, weights="distance", with_pred=True)
        for a, b in zip(one, multi):
            np.testing.assert_array_equal(a, b)
        sd, si, _ = mi.query(None, 7, exclude_self=True)
        rd, ri = _reference(metric, R, None, 7)
        np.testing.assert_array_equal(sd, rd)
        np.testing.assert_array_equal(si, ri)
    finally:
        mi.close()


def test_estimator_on_several_devices_and_nan_queries(monkeypatch):
    import sknnr_b200 as S

    R, Q, y = _data(2000, 3000, 8, seed=4)
    single = S.RawKNNRegressor(n_neighbors=7, p=1).fit(R, y)
    monkeypatch.setenv("SKNNR_B200_DEVICES", "0,0,0")
    multi = S.RawKNNRegressor(n_neighbors=7, p=1).fit(R, y)
    assert type(multi._get_index()).__name__ == "MultiDeviceIndex"
    assert multi._get_index().parts[0].metric == "manhattan"
    for a, b in zip(single.kneighbors(Q), multi.kneighbors(Q)):
        np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(single.independent_prediction_, multi.independent_prediction_)

    Qn = Q.copy()
    Qn[5, 3] = np.nan
    est = S.EuclideanKNNRegressor(n_neighbors=7, metric="chebyshev").fit(R, y)
    for e in (single, est):   # scikit-learn's validation error, as on the Euclidean path
        with pytest.raises(ValueError, match="contains NaN"):
            e.predict(Qn)
        with pytest.raises(ValueError, match="contains NaN"):
            e.kneighbors(Qn)


# ---- rasters ---------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_rasters_of_a_manhattan_estimator_equal_row_queries(dtype):
    import sknnr_b200 as S

    Xtr, Xte, ytr = _moscow()
    rng = np.random.default_rng(3)
    h, w = 37, 53
    pix = Xtr[rng.integers(0, len(Xtr), h * w)] + rng.normal(0, 0.05, (h * w, Xtr.shape[1]))
    pix = pix.astype(dtype)
    pix[rng.random(h * w) < 0.05, 2] = -9999.0
    pix[rng.random(h * w) < 0.05, 4] = np.nan
    image = np.ascontiguousarray(pix.T.reshape(Xtr.shape[1], h, w))
    valid = ~((pix == dtype(-9999.0)).any(1) | np.isnan(pix).any(1))
    for est in (S.EuclideanKNNRegressor(n_neighbors=5, p=1, weights="distance").fit(Xtr, ytr),
                S.RawKNNRegressor(n_neighbors=5, metric="chebyshev").fit(Xtr, ytr)):
        d, i = S.kneighbors_raster(est, image, nodata=-9999.0)
        p = S.predict_raster(est, image, nodata=-9999.0)
        ed, ei = est.kneighbors(pix[valid])
        np.testing.assert_array_equal(d.reshape(5, -1)[:, valid].T, ed)
        np.testing.assert_array_equal(i.reshape(5, -1)[:, valid].T, ei)
        np.testing.assert_array_equal(p.reshape(ytr.shape[1], -1)[:, valid].T, est.predict(pix[valid]))
        assert np.isnan(p.reshape(ytr.shape[1], -1)[:, ~valid]).all()
        assert (i.reshape(5, -1)[:, ~valid] == -1).all()
