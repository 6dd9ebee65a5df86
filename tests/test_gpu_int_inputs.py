"""GPU tests of integer query inputs: uint8, int16, uint16, int32 and int64 arrays and raster bands go to
the device as they are, and every result is bit-identical to the same call on ``X.astype(np.float64)``.

The queries hold each dtype's extremes (and, for int64, values past 2^53, which the device rounds to
float64 as NumPy does).  The call's ``h2d_bytes`` counter shows that the array crossed at its own
element size.  Other integer dtypes (int8, uint32, ...) still take the host conversion to float64."""

import warnings

import numpy as np
import pytest

from sknnr_b200 import _lib as L
from tests.conftest import yaimpute_weights

pytestmark = pytest.mark.gpu

NATIVE = [np.uint8, np.int16, np.uint16, np.int32, np.int64]
KINDS = ["raw", "euclidean", "mahalanobis", "msn", "gnn"]
D = 5


def _ints(dt, shape, rng, extremes=True):
    """Random values of ``dt`` in a moderate range; with ``extremes`` the first rows hold the dtype's
    minimum, maximum and zero (int64: also values past 2^53 that float64 cannot hold exactly)."""
    info = np.iinfo(dt)
    X = rng.integers(max(info.min, -3000), min(info.max, 3000) + 1, size=shape).astype(dt)
    if extremes:
        X[0] = info.min
        X[1] = info.max
        X[2] = 0
        X[3, ::2] = info.max
        X[3, 1::2] = info.min
        if dt == np.int64:
            X[4] = [2**53 + 1, -(2**53) - 3, 2**62 + 12345, -(2**60) - 7, 2**53 + 2][: shape[1]]
    return X


def _fit_data(dt, seed=0, n=400):
    rng = np.random.default_rng(seed)
    X = _ints(dt, (n, D), rng, extremes=False)
    y = rng.random((n, 3)) + 0.1          # positive: CCA (GNN) needs it
    return X, y


def _make(kind, **kw):
    import sknnr_b200 as S

    cls = {"raw": S.RawKNNRegressor, "euclidean": S.EuclideanKNNRegressor,
           "mahalanobis": S.MahalanobisKNNRegressor, "msn": S.MSNRegressor, "gnn": S.GNNRegressor}[kind]
    return cls(**kw)


def _index_of(est):
    return getattr(est, "regressor_", est)._get_index()


def _same(a, b):
    if isinstance(a, tuple):
        assert len(a) == len(b)
        for u, v in zip(a, b):
            _same(u, v)
        return
    assert a.dtype == b.dtype and a.shape == b.shape
    assert np.array_equal(a, b, equal_nan=True)


# ---- the float estimators --------------------------------------------------------------------
@pytest.mark.parametrize("dt", NATIVE, ids=lambda t: np.dtype(t).name)
@pytest.mark.parametrize("kind", KINDS)
def test_float_estimators_integer_query_equals_float64(kind, dt):
    rng = np.random.default_rng(1)
    X, y = _fit_data(dt)
    Q = _ints(dt, (3000, D), rng)
    Qf = Q.astype(np.float64)
    for weights in ("uniform", "distance", yaimpute_weights):
        est = _make(kind, n_neighbors=7, weights=weights).fit(X, y)
        _same(est.predict(Q), est.predict(Qf))
        if weights != "uniform":
            continue
        got = est.kneighbors(Q)
        assert _index_of(est).stats()["h2d_bytes"] == Q.size * Q.itemsize   # no float64 copy went over
        _same(got, est.kneighbors(Qf))
        _same(est.kneighbors(Q, n_neighbors=3, use_deterministic_ordering=False),
              est.kneighbors(Qf, n_neighbors=3, use_deterministic_ordering=False))
        if kind != "raw":
            Z = est.transformer_.transform(Q)
            assert Z.dtype == np.float64
            _same(Z, est.transformer_.transform(Qf))


@pytest.mark.parametrize("kind", KINDS)
def test_int16_dataframe_queries_equal_float64_with_the_same_warnings(kind):
    pd = pytest.importorskip("pandas")
    rng = np.random.default_rng(2)
    X, y = _fit_data(np.int16, seed=2)
    cols = [f"band{i}" for i in range(D)]
    est = _make(kind, n_neighbors=5).fit(pd.DataFrame(X, columns=cols), y)
    Q = _ints(np.int16, (500, D), rng)

    def run(q):
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter("always")
            out = (est.predict(q),) + est.kneighbors(q)
        return out, sorted(str(m.message) for m in w if "feature names" in str(m.message))

    df_i, df_f = pd.DataFrame(Q, columns=cols), pd.DataFrame(Q.astype(np.float64), columns=cols)
    (a, wa), (b, wb) = run(df_i), run(df_f)
    _same(a, b)
    assert wa == wb == []
    (a, wa), (b, wb) = run(Q), run(Q.astype(np.float64))   # no feature names: scikit-learn's warning
    _same(a, b)
    assert wa == wb and len(wa) > 0
    with pytest.raises(ValueError):   # shape errors stay scikit-learn's own
        est.predict(Q[:, :3])


# ---- RFNN / GBNN ---------------------------------------------------------------------------------
@pytest.mark.parametrize("dt", NATIVE, ids=lambda t: np.dtype(t).name)
@pytest.mark.parametrize("kind", ["rfnn", "gbnn"])
def test_tree_estimators_integer_query_equals_float64(kind, dt):
    import sknnr_b200 as S

    rng = np.random.default_rng(3)
    X, y = _fit_data(dt, seed=3)
    Q = _ints(dt, (2000, D), rng)
    Qf = Q.astype(np.float64)
    make = (lambda **kw: S.RFNNRegressor(n_estimators=12, random_state=0, **kw)) if kind == "rfnn" else \
        (lambda **kw: S.GBNNRegressor(n_estimators=12, random_state=0, **kw))
    for weights in ("uniform", "distance"):
        est = make(n_neighbors=5, weights=weights).fit(X, y)
        _same(est.predict(Q), est.predict(Qf))
        if weights == "uniform":
            got = est.kneighbors(Q)
            assert est.regressor_._get_index().stats()["h2d_bytes"] == Q.size * Q.itemsize
            _same(got, est.kneighbors(Qf))
            _same(est.transformer_.transform(Q), est.transformer_.transform(Qf))


@pytest.mark.parametrize(("dt", "base", "spread"), [
    (np.int32, 2**24, 64),              # float32 rounds here: every other integer has no float32 of its own
    (np.int32, -(2**24), 64),
    (np.int64, 2**40, 2**20),
    (np.int64, 2**52, 2**30),           # within 2^53: float64 is exact, float32 rounds once
])
def test_forest_apply_node_ids_equal_scikit_learn(dt, base, spread):
    from sknnr_b200.transformers import RFNodeTransformer

    rng = np.random.default_rng(4)
    X = (base + rng.integers(-spread, spread, size=(600, 4))).astype(dt)
    y = rng.standard_normal((600, 2))
    t = RFNodeTransformer(n_estimators=8, min_samples_leaf=2, random_state=0).fit(X, y)
    Q = (base + rng.integers(-spread, spread, size=(4000, 4))).astype(dt)
    got = t.transform(Q)
    want = np.hstack([e.apply(Q) for e in t.estimators_]).astype(np.int64)
    assert np.array_equal(got, want)
    assert np.array_equal(got, t.transform(Q.astype(np.float64)))


# ---- host calls of many chunks, pinned and device-resident input ----------------------------------
def _affine_index(rng, n_ref=900, d_in=D, d_out=4):
    from sknnr_b200._engine import KNNIndex

    R = rng.integers(-2000, 2000, size=(n_ref, d_in)).astype(np.float64)
    center, scale = R.mean(axis=0), R.std(axis=0)
    proj = rng.standard_normal((d_in, d_out))
    fit_z = ((R - center) / scale) @ proj
    return KNNIndex(fit_z, center, scale, proj, rng.standard_normal((n_ref, 2)))


@pytest.mark.parametrize("dt", NATIVE, ids=lambda t: np.dtype(t).name)
def test_host_call_of_many_chunks_pageable_pinned_and_device_pointer(dt):
    import torch

    from sknnr_b200._engine import pinned_empty

    rng = np.random.default_rng(5)
    ix = _affine_index(rng)
    n_q, k = 20_000, 6
    X = _ints(dt, (n_q, D), rng)
    Xf = pinned_empty((n_q, D))
    Xf[:] = X
    Xp = pinned_empty((n_q, D), dt)
    Xp[:] = X
    Xs = np.ascontiguousarray(np.hstack([X, X[:, :3]]))[:, :D]    # row stride 8 elements
    kw = dict(weights="distance", with_pred=True)
    L.set_option("stage_rows", 1024)
    L.set_option("chunk_rows", 4096)
    try:
        ref = ix.query(Xf, k, **kw)
        for Xin in (X, Xp, Xs):
            _same(ix.query(Xin, k, **kw), ref)
            assert ix.stats()["h2d_bytes"] == n_q * D * np.dtype(dt).itemsize
        _same(ix.transform(X), ix.transform(Xf))
        # device-resident rows, answered on the caller's stream
        x_d = torch.from_numpy(X).cuda()
        outs = [torch.empty((n_q, k), dtype=torch.float64, device="cuda"),
                torch.empty((n_q, k), dtype=torch.int64, device="cuda"),
                torch.empty((n_q, 2), dtype=torch.float64, device="cuda")]
        ix.query_device(x_d.data_ptr(), False, n_q, D, k, dist_ptr=outs[0].data_ptr(), idx_ptr=outs[1].data_ptr(),
                        pred_ptr=outs[2].data_ptr(), weights="distance",
                        stream=torch.cuda.current_stream().cuda_stream, x_dtype=dt)
        torch.cuda.synchronize()
        _same(tuple(t.cpu().numpy() for t in outs), ref)
    finally:
        L.set_option("stage_rows", 1 << 19)
        L.set_option("chunk_rows", 1 << 20)


def test_unknown_dtype_code_is_rejected():
    rng = np.random.default_rng(6)
    ix = _affine_index(rng)
    X = np.zeros((10, D), dtype=np.int16)
    dist = np.empty((10, 3))
    idx = np.empty((10, 3), dtype=np.int64)
    import ctypes as C

    for code in (7, -1, 100):
        with pytest.raises(ValueError, match="x_dtype"):
            L.check(ix._lib.sknnr_kneighbors(ix._h, X.ctypes.data_as(C.c_void_p), code, 10, D, 0, 3, 0, 10,
                                             dist.ctypes.data_as(C.c_void_p), idx.ctypes.data_as(C.c_void_p),
                                             L.W_NONE, None, None))
    with pytest.raises(ValueError):
        ix.query_device(0, False, 10, D, 3, x_dtype=np.int8)


# ---- rasters -------------------------------------------------------------------------------------
RASTER_CASES = [(np.uint8, 200, [None, 200, 200.5, -1]), (np.int16, -9999, [None, -9999, -9999.5, 70000]),
                (np.uint16, 65535, [None, 65535, -9999, 65535.5])]


def _image(dt, fill, rng, H=61, W=97):
    img = _ints(dt, (D, H * W), rng, extremes=False)
    img[:, :4] = np.iinfo(dt).max
    img[:, 4:8] = np.iinfo(dt).min
    holes = rng.random(H * W) < 0.05
    img[rng.integers(0, D, holes.sum()), np.flatnonzero(holes)] = fill
    return img.reshape(D, H, W)


@pytest.mark.parametrize(("dt", "fill", "nodatas"), RASTER_CASES, ids=lambda v: np.dtype(v).name if isinstance(v, type) else None)
@pytest.mark.parametrize("kind", ["euclidean", "gnn", "rfnn"])
def test_raster_integer_bands_equal_float64_image(kind, dt, fill, nodatas):
    import sknnr_b200 as S

    rng = np.random.default_rng(7)
    X, y = _fit_data(dt, seed=7)
    if kind == "rfnn":
        est = S.RFNNRegressor(n_estimators=10, random_state=0, n_neighbors=5).fit(X, y)
    else:
        est = _make(kind, n_neighbors=5, weights="distance").fit(X, y)
    img = _image(dt, fill, rng)
    imgf = img.astype(np.float64)
    for nodata in nodatas:
        a = S.kneighbors_raster(est, img, nodata=nodata)
        assert _index_of(est).stats()["h2d_bytes"] == img.size * img.itemsize
        _same(a, S.kneighbors_raster(est, imgf, nodata=nodata))
        _same(S.predict_raster(est, img, nodata=nodata), S.predict_raster(est, imgf, nodata=nodata))
        masked = (a[1][0] < 0).sum()
        assert masked == (np.any(imgf == nodata, axis=0).sum() if nodata is not None else 0)
    # bands of a larger image: band stride twice the band size, pixels contiguous within a band
    big = np.zeros((2 * D,) + img.shape[1:], dtype=dt)
    big[::2] = img
    _same(S.predict_raster(est, big[::2], nodata=fill), S.predict_raster(est, imgf, nodata=fill))


# ---- several devices -----------------------------------------------------------------------------
@pytest.mark.parametrize("devices", ["0,0", "0,1"])
def test_multi_device_estimators_integer_query_equals_float64(devices, monkeypatch):
    import torch

    import sknnr_b200 as S
    from sknnr_b200._sharding import MultiDeviceIndex

    if devices == "0,1" and torch.cuda.device_count() < 2:
        pytest.skip(f"needs 2 GPUs for SKNNR_B200_DEVICES=0,1, this box has {torch.cuda.device_count()}")
    rng = np.random.default_rng(8)
    X, y = _fit_data(np.int16, seed=8)
    Q = _ints(np.int16, (5000, D), rng)
    single = [S.EuclideanKNNRegressor(n_neighbors=5, weights="distance").fit(X, y),
              S.RFNNRegressor(n_estimators=10, random_state=0).fit(X, y)]
    want = [(e.predict(Q.astype(np.float64)),) + e.kneighbors(Q.astype(np.float64)) for e in single]
    monkeypatch.setenv("SKNNR_B200_DEVICES", devices)
    monkeypatch.setattr(MultiDeviceIndex, "min_rows_per_device", 64)
    multi = [S.EuclideanKNNRegressor(n_neighbors=5, weights="distance").fit(X, y),
             S.RFNNRegressor(n_estimators=10, random_state=0).fit(X, y)]
    for est, w in zip(multi, want):
        assert isinstance(est.regressor_._get_index(), MultiDeviceIndex)
        _same((est.predict(Q),) + est.kneighbors(Q), w)


# ---- dtypes that keep the host conversion --------------------------------------------------------
@pytest.mark.parametrize("dt", [np.int8, np.uint32], ids=lambda t: np.dtype(t).name)
def test_other_integer_types_take_the_float64_path(dt):
    import sknnr_b200 as S

    rng = np.random.default_rng(9)
    info = np.iinfo(dt)
    X = rng.integers(max(info.min, -100), min(info.max, 100) + 1, size=(400, D)).astype(dt)
    y = rng.random((400, 3)) + 0.1
    Q = rng.integers(info.min, info.max, size=(1000, D), endpoint=True).astype(dt)
    Q[0] = info.max
    for kind in ("raw", "euclidean", "gnn"):
        est = _make(kind, n_neighbors=5, weights="distance").fit(X, y)
        _same(est.predict(Q), est.predict(Q.astype(np.float64)))
        _same(est.kneighbors(Q), est.kneighbors(Q.astype(np.float64)))
        assert _index_of(est).stats()["h2d_bytes"] == Q.size * 8
    img = Q[: 30 * 4].T.reshape(D, 30, 4)
    _same(S.predict_raster(est, img), S.predict_raster(est, img.astype(np.float64)))
    assert _index_of(est).stats()["h2d_bytes"] == img.size * 8
