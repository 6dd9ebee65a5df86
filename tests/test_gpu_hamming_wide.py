"""Wide Hamming mode on the device: trees with more than 31,743 distinct node IDs keep exact 32-bit
codes, the 16-bit search runs as a filter on their hashed image, and a float64 re-rank certifies its
candidates.  Every result is compared bit for bit with SciPy's weighted Hamming distances ranked by
stable (distance, index), then sknnr's ordering, or with a 16-bit index of the same codes."""

import numpy as np
import pytest
from scipy.spatial.distance import cdist

from oracle import sknnr_oracle as orc

pytestmark = pytest.mark.gpu

N_IDS = 80000   # per-tree ID range of the bare matrices: ~42k distinct IDs per tree at 60k plots


def _reference(R, Q, w, k, rows=None):
    """Q given: SciPy's neighbours of every row of Q.  Q None: those of the plots ``rows`` among the
    plots themselves, self excluded (X=None)."""
    Qx = R[rows] if Q is None else Q
    D = cdist(np.asarray(Qx, np.float64), np.asarray(R, np.float64), "hamming", w=w)
    kk = k + (1 if Q is None else 0)
    order = np.argsort(D, axis=1, kind="stable")[:, :kk]
    dist, idx = np.take_along_axis(D, order, 1), order.astype(np.int64)
    if Q is not None:
        return orc.deterministic_order(dist, idx)
    out_d, out_i = [], []
    for j, r in enumerate(rows):
        d, i = orc.exclude_self(dist[j:j + 1], idx[j:j + 1], row_offset=int(r))
        d, i = orc.deterministic_order(d, i, row_offset=int(r))
        out_d.append(d)
        out_i.append(i)
    return np.vstack(out_d), np.vstack(out_i)


def _bare_data(seed, n_ref=60000, T=8, n_q=600, id_offset=0):
    """Node-ID matrices with near-duplicate plots, duplicated plots, queries equal to plots, unseen IDs
    and non-integer query values."""
    rng = np.random.default_rng(seed)
    R = rng.integers(0, N_IDS, size=(n_ref, T)).astype(np.int64)
    src = rng.integers(0, n_ref, size=n_ref // 3)
    dst = rng.integers(0, n_ref, size=n_ref // 3)
    R[dst] = R[src]
    R[dst[: n_ref // 6], rng.integers(0, T, n_ref // 6)] = rng.integers(0, N_IDS, n_ref // 6)
    Q = R[rng.integers(0, n_ref, size=n_q)].astype(np.float64)
    flip = rng.random(Q.shape) < 0.3
    Q[flip] = rng.integers(0, N_IDS, int(flip.sum()))
    Q[rng.random(Q.shape) < 0.03] = N_IDS + 7          # unseen
    Q[rng.random(Q.shape) < 0.03] += 0.5               # non-integer: equals no node ID
    R += id_offset
    Q += id_offset
    y = np.column_stack([R[:, 0] % 97, R[:, 1] % 13]).astype(np.float64)
    return R, Q, y


def _raw(k, w=None, weights="uniform"):
    from sknnr_b200 import RawKNNRegressor

    params = None if w is None else {"w": w}
    return RawKNNRegressor(n_neighbors=k, metric="hamming", metric_params=params, weights=weights,
                           algorithm="brute")


@pytest.fixture(scope="module")
def bare():
    return _bare_data(3)


@pytest.mark.parametrize("k", [1, 7, 24, 40])
def test_bare_node_ids_equal_scipy(bare, k):
    R, Q, y = bare
    T = R.shape[1]
    est = _raw(k).fit(R, y)
    ix = est._get_index()
    assert ix.wide
    d, i = est.kneighbors(Q)
    d_o, i_o = _reference(R, Q, np.full(T, 1.0 / T), k)
    np.testing.assert_array_equal(i, i_o)
    assert np.array_equal(d, d_o)
    cc = ix.cascade_counts()
    if k + 8 <= 32:
        assert cc["to_exact"] < Q.shape[0]        # the filter certified rows
    else:
        assert cc["to_exact"] == Q.shape[0]       # k > 24: the exhaustive kernel answers every row
    # X=None on a sample of plots (the self-query answers all of them)
    rows = np.random.default_rng(k).choice(R.shape[0], 300, replace=False)
    d_n, i_n = est.kneighbors()
    d_o, i_o = _reference(R, None, np.full(T, 1.0 / T), k, rows)
    np.testing.assert_array_equal(i_n[rows], i_o)
    assert np.array_equal(d_n[rows], d_o)


@pytest.mark.parametrize("weights", ["uniform", "distance", "callable"])
def test_bare_predict_weights(bare, weights):
    R, Q, y = bare
    T = R.shape[1]
    fn = (lambda d: 1.0 / (d + 0.25)) if weights == "callable" else weights
    est = _raw(7, weights=fn).fit(R, y)
    d_o, i_o = _reference(R, Q, np.full(T, 1.0 / T), 7)
    p_o = orc.weighted_average(y, i_o, orc.get_weights(d_o, fn))
    np.testing.assert_allclose(est.predict(Q), p_o, rtol=1e-12, atol=0)


@pytest.mark.parametrize("k", [5, 40])
def test_bare_unequal_weights_and_ids_beyond_int32(k):
    """GBNN-style unequal weights: the fixed-point filter on hashed codes.  IDs beyond int32 take the
    dense per-tree tables."""
    R, Q, y = _bare_data(11, T=12, n_q=500, id_offset=1 << 40)
    w = np.random.default_rng(2).random(12) + 0.05
    est = _raw(k, w=w).fit(R, y)
    ix = est._get_index()
    assert ix.wide
    d, i = est.kneighbors(Q)
    d_o, i_o = _reference(R, Q, w, k)
    np.testing.assert_array_equal(i, i_o)
    assert np.array_equal(d, d_o)
    rows = np.arange(0, R.shape[0], 191)
    d_n, i_n = est.kneighbors()
    d_o, i_o = _reference(R, None, w, k, rows)
    np.testing.assert_array_equal(i_n[rows], i_o)
    assert np.array_equal(d_n[rows], d_o)


@pytest.mark.parametrize("unequal", [False, True])
def test_adversarial_collisions_reach_the_exhaustive_kernel(unequal):
    """Decoy plots whose IDs collide with the query's under the hash in every tree fill the filter's
    lists with hashed mismatch count 0; the true neighbours lie outside them.  The certificate must
    refuse those rows, and the exhaustive kernel on the exact codes answers them."""
    rng = np.random.default_rng(5)
    n_ids, T, n_ref = 40000, 8, 60000
    R = rng.integers(0, n_ids, size=(n_ref, T)).astype(np.int64)
    for t in range(T):
        R[:n_ids, t] = rng.permutation(n_ids)     # every ID present: ID = its dense code
    n_proto, n_decoy = 200, 30
    P = rng.integers(0, n_ids - 31743, size=(n_proto, T))
    pos = n_ids + rng.permutation(n_ref - n_ids)[: n_proto * (n_decoy + 2)].reshape(n_proto, n_decoy + 2)
    for p in range(n_proto):
        R[pos[p, :n_decoy]] = P[p] + 31743          # collides in every tree, true count T
        for j in range(2):                          # true neighbours: two trees changed
            row = P[p].copy()
            row[rng.choice(T, 2, replace=False)] = rng.integers(0, n_ids, 2)
            R[pos[p, n_decoy + j]] = row
    y = rng.random((n_ref, 1))
    w = rng.random(T) + 0.5 if unequal else None
    est = _raw(5, w=w).fit(R, y)
    ix = est._get_index()
    assert ix.wide
    d, i = est.kneighbors(P.astype(np.float64))
    assert ix.cascade_counts()["to_exact"] >= n_proto // 2
    d_o, i_o = _reference(R, P, np.full(T, 1.0 / T) if w is None else w, 5)
    np.testing.assert_array_equal(i, i_o)
    assert np.array_equal(d, d_o)


@pytest.fixture(scope="module")
def forest_fit():
    from sklearn.datasets import make_friedman1

    from sknnr_b200 import RFNNRegressor

    X, y = make_friedman1(n_samples=62000, n_features=8, noise=0.5, random_state=4)
    X = np.round(X * 1000)            # integer-valued features: the raster bands are int16
    Xtr, ytr, Xq = X[:60000], y[:60000], X[60000:]
    est = RFNNRegressor(n_estimators=2, min_samples_leaf=1, random_state=0).fit(Xtr, ytr)
    return est, Xtr, Xq


def test_forest_with_more_leaves_than_16_bit_codes(forest_fit):
    est, Xtr, Xq = forest_fit
    ids_tr = np.hstack([e.apply(Xtr.astype(np.float32)).reshape(-1, 1)
                        for f in est.transformer_.estimators_ for e in f.estimators_])
    assert max(len(np.unique(ids_tr[:, t])) for t in range(ids_tr.shape[1])) > 31743
    ix = est.regressor_._get_index()
    assert ix.wide
    ids_q = est.transformer_.transform(Xq)
    ref_q = np.hstack([e.apply(Xq.astype(np.float32)).reshape(-1, 1)
                       for f in est.transformer_.estimators_ for e in f.estimators_])
    np.testing.assert_array_equal(ids_q, ref_q)
    np.testing.assert_array_equal(est.transformer_.transform(Xtr), ids_tr)
    d, i = est.kneighbors(Xq)                               # fused: forest walk + wide search
    d_n, i_n = est.regressor_.kneighbors(ids_q)             # node-ID query
    np.testing.assert_array_equal(i, i_n)
    assert np.array_equal(d, d_n)
    d_o, i_o = _reference(ids_tr, ids_q, est.hamming_weights_, 5)
    np.testing.assert_array_equal(i, i_o)
    assert np.array_equal(d, d_o)
    rows = np.arange(0, 60000, 211)
    d_s, i_s = est.kneighbors()
    d_o, i_o = _reference(ids_tr, None, est.hamming_weights_, 5, rows)
    np.testing.assert_array_equal(i_s[rows], i_o)
    assert np.array_equal(d_s[rows], d_o)
    np.testing.assert_array_equal(est.predict(Xq), est.regressor_.predict(ids_q))


def test_forest_raster_int16_equals_row_query(forest_fit):
    from sknnr_b200.raster import kneighbors_raster, predict_raster

    est, _, Xq = forest_fit
    h, w_ = 40, 50
    img = Xq[: h * w_].T.reshape(8, h, w_).astype(np.int16)
    img[3, 5, 7] = -999
    img[0, 20, :] = -999
    valid = ~(img == -999).any(axis=0).ravel()
    d, i = kneighbors_raster(est, img, nodata=-999)
    rows = img.reshape(8, -1).T[valid]
    d_r, i_r = est.kneighbors(rows)
    assert np.array_equal(d.reshape(5, -1)[:, valid].T, d_r)
    np.testing.assert_array_equal(i.reshape(5, -1)[:, valid].T, i_r)
    assert (i.reshape(5, -1)[:, ~valid] == -1).all()
    p = predict_raster(est, img, nodata=-999)
    assert np.array_equal(p.reshape(1, -1)[:, valid].ravel(), est.predict(rows))


@pytest.fixture(scope="module")
def small_forest():
    from sklearn.ensemble import RandomForestRegressor

    from sknnr_b200._engine import ForestIndex

    rng = np.random.default_rng(8)
    X = rng.standard_normal((6000, 6))
    y = X[:, :2] @ rng.standard_normal((2, 2)) + 0.1 * rng.standard_normal((6000, 2))
    rf = RandomForestRegressor(n_estimators=24, max_depth=9, random_state=0).fit(X[:5000], y[:5000])
    forest = ForestIndex([e.tree_ for e in rf.estimators_], 6)   # no code tables: leaves carry their node IDs
    yield forest, X[:5000], y[:5000], X[5000:]
    forest.close()


@pytest.mark.parametrize("k", [1, 7, 40])
@pytest.mark.parametrize("unequal", [False, True])
def test_wide_index_of_16_bit_codes_equals_16_bit_index(small_forest, unequal, k):
    """Node IDs that all fit 16 bits, searched by a 16-bit index and by a wide index of the same IDs as
    u32: distances, indices and predictions are bit-identical, for node-code queries, X=None and the
    forest walk."""
    from sknnr_b200._engine import HammingIndex

    forest, Xr, y, Xq = small_forest
    codes, qcodes = forest.apply(Xr), forest.apply(Xq)
    assert codes.max() < 31743
    T = codes.shape[1]
    w = np.random.default_rng(3).uniform(0.5, 1.5, T) if unequal else np.full(T, 1.0 / T)
    narrow = HammingIndex(codes.astype(np.uint16), w, y)
    wide = HammingIndex(codes.astype(np.uint32), w, y)
    assert wide.wide and not narrow.wide
    try:
        calls = [
            lambda ix, c: ix.query(qcodes.astype(c), k, weights="distance", with_pred=True),
            lambda ix, c: ix.query(None, k, exclude_self=True, weights="uniform", with_pred=True),
            lambda ix, c: ix.query_forest(forest, Xq, k, weights="distance", with_pred=True),
        ]
        for call in calls:
            a, b = call(narrow, np.uint16), call(wide, np.uint32)
            for u, v in zip(a, b):
                assert np.array_equal(u, v)
    finally:
        narrow.close()
        wide.close()


def test_forest_two_devices_equal_one(forest_fit, monkeypatch):
    import torch

    from sknnr_b200 import RFNNRegressor
    from sknnr_b200._sharding import MultiDeviceIndex

    if torch.cuda.device_count() < 2:
        pytest.skip(f"needs 2 GPUs, this box has {torch.cuda.device_count()}")
    est, Xtr, Xq = forest_fit
    y = est.regressor_._y
    monkeypatch.setenv("SKNNR_B200_DEVICES", "0,1")
    monkeypatch.setattr(MultiDeviceIndex, "min_rows_per_device", 256)
    two = RFNNRegressor(n_estimators=2, min_samples_leaf=1, random_state=0).fit(Xtr, y)
    assert isinstance(two.regressor_._get_index(), MultiDeviceIndex)
    assert np.array_equal(two.predict(Xq), est.predict(Xq))
    a, b = two.kneighbors(Xq), est.kneighbors(Xq)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
