"""CPU tests: pin the oracle against the reference's golden vectors and live outputs."""

import numpy as np
import pytest

from oracle import sknnr_oracle as orc
from tests.conftest import FLOAT_CASES, load_golden, state_from_golden, yaimpute_weights

# The reference forms d^2 from the float64 expansion |x|^2 - 2x.y + |y|^2.  On the raw,
# uncentred Moscow features (values ~1e6) that expansion cancels ~9 digits, so the
# reference's own distances carry ~1e-7 relative noise that depends on the BLAS summation
# order; the restatement can only agree to that level there (1e-12 on the scaled spaces).
DIST_RTOL = 1e-6


@pytest.mark.parametrize(("name", "comp"), FLOAT_CASES)
def test_oracle_matches_live_reference_kneighbors(name, comp):
    g = load_golden(f"moscow_{name}_{comp}.npz")
    sp = load_golden("moscow_split.npz")
    st = state_from_golden(g)
    # projection (a1-a4): transformed training plots must equal the reference's _fit_X
    np.testing.assert_allclose(orc.transform(st, sp["X_train"]), g["state_fit_Z"], rtol=1e-9, atol=1e-11)
    # X given
    d, i = orc.kneighbors(st, sp["X_test"], k=5)
    np.testing.assert_array_equal(i, g["live_tgt_nn"])
    np.testing.assert_allclose(d, g["live_tgt_dist"], rtol=DIST_RTOL, atol=1e-12)
    # X=None: k+1, self excluded (a9)
    d, i = orc.kneighbors(st, None, k=5)
    np.testing.assert_array_equal(i, g["live_ref_nn"])
    np.testing.assert_allclose(d, g["live_ref_dist"], rtol=DIST_RTOL, atol=1e-12)
    # dataframe-index crosswalk (ref:src/sknnr/_base.py:177-180)
    np.testing.assert_array_equal(sp["index_train"][i], g["live_ref_ids"])


@pytest.mark.parametrize(("name", "comp"), FLOAT_CASES)
def test_oracle_matches_reference_golden_files(name, comp):
    """ref:tests/test_regressions/*.npz (goldens use algorithm='auto': kd_tree for <=15
    dims, so distances agree to rounding and index order inside exact ties may differ)."""
    g = load_golden(f"moscow_{name}_{comp}.npz")
    sp = load_golden("moscow_split.npz")
    st = state_from_golden(g)
    d, i = orc.kneighbors(st, sp["X_test"], k=5)
    np.testing.assert_array_equal(i, g["refgold_tgt_index_nn"])
    np.testing.assert_allclose(d, g["refgold_tgt_index_dist"], rtol=DIST_RTOL, atol=1e-11)
    np.testing.assert_array_equal(sp["index_train"][i], g["refgold_tgt_ids_nn"])
    d, i = orc.kneighbors(st, None, k=5)
    np.testing.assert_array_equal(i, g["refgold_ref_index_nn"])
    np.testing.assert_allclose(d, g["refgold_ref_index_dist"], rtol=DIST_RTOL, atol=1e-11)
    # predictions: unweighted and the yaImpute callable
    p = orc.predict(st, sp["X_test"], k=5)
    np.testing.assert_allclose(p, g["refgold_tgt_unweighted_pred"], rtol=1e-9, atol=1e-12)
    p = orc.predict(st, sp["X_test"], k=5, weights=yaimpute_weights)
    np.testing.assert_allclose(p, g["refgold_tgt_weighted_pred"], rtol=DIST_RTOL, atol=1e-12)
    p = orc.predict(st, None, k=5)
    np.testing.assert_allclose(p, g["refgold_ref_unweighted_pred"], rtol=1e-9, atol=1e-12)
    assert orc.r2_score_uniform(sp["y_train"], p) == pytest.approx(float(g["refgold_ref_unweighted_score"]), abs=1e-12)
    p = orc.predict(st, None, k=5, weights=yaimpute_weights)
    np.testing.assert_allclose(p, g["refgold_ref_weighted_pred"], rtol=DIST_RTOL, atol=1e-12)
    assert orc.r2_score_uniform(sp["y_train"], p) == pytest.approx(float(g["refgold_ref_weighted_score"]), abs=1e-7)


@pytest.mark.parametrize(("name", "comp"), FLOAT_CASES)
def test_oracle_distance_weights(name, comp):
    g = load_golden(f"moscow_{name}_{comp}.npz")
    sp = load_golden("moscow_split.npz")
    st = state_from_golden(g)
    p = orc.predict(st, sp["X_test"], k=5, weights="distance")
    np.testing.assert_allclose(p, g["live_tgt_pred_distance"], rtol=DIST_RTOL, atol=1e-12)
    p = orc.predict(st, None, k=5, weights="distance")
    np.testing.assert_allclose(p, g["live_ref_pred_distance"], rtol=DIST_RTOL, atol=1e-12)


def test_oracle_config1_swo_msn():
    g = load_golden("c1_swo_msn_k5.npz")
    st = state_from_golden(g)
    d, i = orc.kneighbors(st, None, k=5)
    n_bad = orc.assert_tie_aware_equal(d, i, g["live_ref_dist"], g["live_ref_nn"], rtol=1e-7, atol=1e-9)
    assert n_bad <= 2
    p = orc.weighted_average(st.y, i)
    assert orc.r2_score_uniform(g["y_targets"], p) == pytest.approx(float(g["live_ref_score"]), abs=1e-6)
    d, i = orc.kneighbors(st, g["X"], k=5)
    # self-distance: the reference's expansion gives ~1e-7 instead of 0 -> absolute floor
    np.testing.assert_allclose(d, g["live_self_dist"], rtol=1e-6, atol=1e-6)


def test_oracle_config2_moscow_gnn_independent_score():
    g = load_golden("c2_moscow_gnn_k5.npz")
    st = state_from_golden(g)
    d, i = orc.kneighbors(st, None, k=5)
    np.testing.assert_array_equal(i, g["live_ref_nn"])
    np.testing.assert_allclose(d, g["live_ref_dist"], rtol=1e-9, atol=1e-12)
    p = orc.weighted_average(st.y, i)
    np.testing.assert_allclose(p, g["live_ref_pred"], rtol=1e-9, atol=1e-12)
    assert orc.r2_score_uniform(g["y_targets"], p) == pytest.approx(float(g["live_ref_score"]), abs=1e-12)


# ---- ordering known-answer tests (ref:tests/test_estimators.py:306-378) -------------
def _raw_state(X, y):
    return orc.FittedState(kind="euclidean", fit_Z=np.asarray(X, float), y=np.asarray(y, float))


@pytest.mark.parametrize(("det", "expected"), [(False, [1, 0]), (True, [0, 1])])
def test_oracle_deterministic_ordering(det, expected):
    st = _raw_state(np.array([1e-11, 1e-12, 1.0]).reshape(-1, 1), [0, 1, 2])
    _, idx = orc.kneighbors(st, np.array([[0.0]]), k=2, deterministic=det)
    assert idx[0].tolist() == expected


def test_oracle_uses_index_difference():
    st = _raw_state(np.array([1e-11, 1e-12, 1.0]).reshape(-1, 1), [0, 1, 2])
    _, idx = orc.kneighbors(st, np.array([[0.0], [0.0]]), k=2)
    assert idx.tolist() == [[0, 1], [1, 0]]
    # a sharded caller reproduces row 1 by passing its global offset
    _, idx = orc.kneighbors(st, np.array([[0.0]]), k=2, row_offset=1)
    assert idx.tolist() == [[1, 0]]


@pytest.mark.parametrize(("dec", "expected"), [(8, [2, 1, 0]), (5, [1, 2, 0]), (2, [0, 1, 2])])
def test_oracle_precision_decimals(dec, expected):
    st = _raw_state(np.array([1e-3, 1e-6, 1e-9, 1.0]).reshape(-1, 1), [0, 1, 2, 3])
    _, idx = orc.kneighbors(st, np.array([[0.0]]), k=3, decimals=dec)
    assert idx[0].tolist() == expected


def test_oracle_exclude_self_with_duplicates():
    # >= k+1 exact duplicates: no column equals the row -> column 0 is dropped
    X = np.zeros((6, 2))
    st = _raw_state(X, np.arange(6))
    d, i = orc.kneighbors(st, None, k=2, deterministic=False)
    assert i[5].tolist() == [1, 2]
    assert i[0].tolist() == [1, 2]
    assert np.all(d == 0)


# ---- Hamming ------------------------------------------------------------------------
def test_hamming_c_oracle_is_bit_equal_to_scipy():
    from scipy.spatial.distance import cdist

    rng = np.random.default_rng(0)
    Q = rng.integers(0, 6, size=(37, 53))
    R = rng.integers(0, 6, size=(29, 53))
    for w in (np.full(53, 1.0 / 53), rng.random(53) + 0.1):
        ref = cdist(Q.astype(float), R.astype(float), metric="hamming", w=w)
        assert np.array_equal(orc.hamming_cdist(Q, R, w, use_c=True), ref)
        assert np.array_equal(orc.hamming_cdist(Q, R, w, use_c=False), ref)
    w = np.full(53, 0.1 / 53)
    lut = orc.hamming_lut(w)
    ref = cdist(Q.astype(float), R.astype(float), metric="hamming", w=w)
    m = (Q[:, None, :] != R[None, :, :]).sum(-1)
    assert np.array_equal(lut[m], ref)
    assert np.all(np.diff(lut) > 0)


def test_hamming_oracle_matches_live_rfnn():
    g = load_golden("moscow_rfnn.npz")
    st = orc.FittedState(kind="hamming", fit_Z=g["ids_train"].astype(np.int64), y=g["y"], hamming_w=g["hamming_w"])
    for X, key in ((g["ids_test"].astype(np.int64), "tgt"), (None, "ref")):
        d, i = orc.kneighbors(st, X, k=5)
        # distances are bit-equal; indices may differ only inside boundary ties
        assert np.array_equal(d, g[f"live_{key}_dist"])
        orc.assert_tie_aware_equal(d, i, g[f"live_{key}_dist"], g[f"live_{key}_nn"], rtol=0, atol=0, gap_rtol=0)
    st2 = orc.FittedState(kind="hamming", fit_Z=st.fit_Z, y=st.y, hamming_w=g["hamming_w_nonuniform"])
    d, i = orc.kneighbors(st2, g["ids_test"].astype(np.int64), k=5)
    assert np.array_equal(d, g["live_tgt_dist_nonuniform"])


def test_hamming_oracle_matches_live_gbnn():
    """GBNN (scope row f3): train-improvement tree weights are unequal, so the distance is a genuine
    float64 weighted sum.  The oracle must reproduce the live reference bit for bit, for the
    all-regression model (3500 trees) and the mixed model with a 3-class boosted classifier."""
    g = load_golden("moscow_gbnn.npz")
    for tag in ("", "mixed_"):
        w = g[tag + "hamming_w"]
        assert len(np.unique(w)) > 10 and np.all(w >= 0) and abs(w.sum() - 1.0) < 1e-9
        st = orc.FittedState(kind="hamming", fit_Z=g[tag + "ids_train"].astype(np.int64), y=g[tag + "y"], hamming_w=w)
        for X, key in ((g[tag + "ids_test"].astype(np.int64), "tgt"), (None, "ref")):
            d, i = orc.kneighbors(st, X, k=5)
            assert np.array_equal(d, g[f"{tag}live_{key}_dist"])
            orc.assert_tie_aware_equal(d, i, g[f"{tag}live_{key}_dist"], g[f"{tag}live_{key}_nn"],
                                       rtol=0, atol=0, gap_rtol=0)
        pred = orc.predict(st, g[tag + "ids_test"].astype(np.int64), k=5)
        np.testing.assert_allclose(pred, g[tag + "live_tgt_pred"], rtol=1e-12)


def test_gbnn_live_outputs_agree_with_reference_goldens():
    """The fixture's live outputs against the reference's own stored vectors.  The mixed-forest
    case agrees at the tolerances of ref:tests/test_regressions.py:125-142.  The 35-target case
    does NOT: the stored vectors were written under another scikit-learn build whose boosted trees
    differ (the unmodified reference run in this image misses them by up to 0.035), so that case is
    pinned on the live reference only - the assertion below documents the state of affairs."""
    g = load_golden("moscow_gbnn.npz")
    np.testing.assert_allclose(g["mixed_live_ref_dist"], g["refgold_mixed_ref_dist"], atol=1e-8)
    np.testing.assert_allclose(g["mixed_live_tgt_dist"], g["refgold_mixed_tgt_dist"], atol=1e-2)
    assert g["live_ref_dist"].shape == g["refgold_ref_index_dist"].shape
    assert np.abs(g["live_ref_dist"] - g["refgold_ref_index_dist"]).max() < 0.05


def _installed_reference():
    """The unmodified reference package that build() installs into oracle/_ref (it travels to the GPU
    box with the snapshot); None when it is not there."""
    import os
    import sys

    from tests.conftest import ROOT

    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "sknnr")):
        return None
    if ref_dir not in sys.path:
        sys.path.insert(0, ref_dir)
    import sknnr

    assert os.path.realpath(sknnr.__file__).startswith(os.path.realpath(ref_dir)), sknnr.__file__
    return sknnr


@pytest.mark.parametrize(("est_name", "weights"), [
    ("EuclideanKNNRegressor", "distance"), ("EuclideanKNNRegressor", "uniform"),
    ("MahalanobisKNNRegressor", "distance"), ("RawKNNRegressor", "uniform"),
])
def test_oracle_matches_installed_reference_on_fresh_random_data(est_name, weights):
    """Beyond the committed goldens: the oracle against the unmodified reference run NOW on seeded random
    data - correlated features, duplicated plots (exact ties), queries that coincide with plots
    (zero distances under weights='distance'), and the X=None self-query.  The oracle takes the fitted
    state from the reference's own transformer, so what is compared is the query-time path."""
    sknnr = _installed_reference()
    if sknnr is None:
        pytest.skip("the unmodified reference package is not installed under oracle/_ref/sknnr")
    rng = np.random.default_rng(20260)
    n_ref, d, n_out, k = 600, 6, 3, 5
    A = rng.standard_normal((d, d))
    R = rng.standard_normal((n_ref, d)) @ A + rng.standard_normal(d) * 3.0
    R[50:60] = R[40:50]                                   # duplicated plots: exact distance ties
    y = rng.standard_normal((n_ref, n_out))
    Q = rng.standard_normal((400, d)) @ A
    Q[:20] = R[100:120]                                   # queries on top of plots: zero distances
    est = getattr(sknnr, est_name)(n_neighbors=k, weights=weights).fit(R, y)
    tr = getattr(est, "transformer_", None)
    if est_name == "RawKNNRegressor":
        st = orc.FittedState(kind="euclidean", fit_Z=np.asarray(R, dtype=np.float64), y=y)
    elif est_name == "EuclideanKNNRegressor":
        st = orc.FittedState(kind="euclidean", fit_Z=tr.transform(R), y=y, center=tr.mean_, scale=tr.scale_)
    else:
        st = orc.FittedState(kind="euclidean", fit_Z=tr.transform(R), y=y, center=tr.scaler_.mean_,
                             scale=tr.scaler_.scale_, proj=tr.transform_)
    for X in (Q, None):
        rd, ri = est.kneighbors(X)
        od, oi = orc.kneighbors(st, X, k)
        # (both sides evaluate |x|^2 - 2 x.y + |y|^2 through BLAS: a coincident pair comes out as 0 or as
        # ~1e-8 depending on the GEMM's blocking, hence the absolute tolerance)
        assert orc.assert_tie_aware_equal(od, oi, rd, ri, rtol=1e-7, atol=5e-7) <= 12   # rows that differ only inside a tie
        np.testing.assert_allclose(od, rd, rtol=1e-7, atol=5e-7)
    rp = est.predict(Q)
    op = orc.predict(st, Q, k, weights=weights)
    ok = np.isclose(op, rp, rtol=1e-6, atol=1e-6).all(axis=1)
    # (a prediction may differ only where the k-th place is an exact tie between duplicated plots)
    assert (~ok).sum() <= 12, int((~ok).sum())
    assert ok[:20].all()                                  # zero-distance rows: indicator weights in both


@pytest.mark.parametrize("est_name", ["RFNNRegressor", "GBNNRegressor"])
def test_hamming_oracle_matches_installed_reference_on_fresh_forests(est_name):
    """RFNN (equal tree weights) and GBNN (train-improvement weights) of the unmodified reference,
    fitted NOW on seeded random data: the oracle, given the reference's own node-ID matrices and
    `hamming_weights_`, must return bit-equal distances (integer compares and one float64 sum in SciPy's
    order) and tie-aware equal neighbours, for target rows and for the X=None self-query."""
    sknnr = _installed_reference()
    if sknnr is None:
        pytest.skip("the unmodified reference package is not installed under oracle/_ref/sknnr")
    rng = np.random.default_rng(7)
    n_ref, d, k = 250, 5, 5
    R = rng.standard_normal((n_ref, d))
    y = np.column_stack([R[:, 0] + 0.3 * rng.standard_normal(n_ref), R[:, 1] * R[:, 2], rng.standard_normal(n_ref)])
    Q = rng.standard_normal((120, d))
    kw = dict(n_estimators=12, random_state=3) if est_name == "RFNNRegressor" else dict(n_estimators=8, random_state=3)
    est = getattr(sknnr, est_name)(n_neighbors=k, **kw).fit(R, y)
    tr = est.transformer_
    w = np.asarray(est.hamming_weights_, dtype=np.float64)
    ids_ref = np.asarray(tr.transform(R)).astype(np.int64)
    ids_q = np.asarray(tr.transform(Q)).astype(np.int64)
    assert ids_ref.shape[1] == len(w) and abs(w.sum() - 1.0) < 1e-9
    if est_name == "GBNNRegressor":
        assert len(np.unique(w)) > 3   # genuinely unequal weights
    st = orc.FittedState(kind="hamming", fit_Z=ids_ref, y=y, hamming_w=w)
    for X, ids in ((Q, ids_q), (None, None)):
        rd, ri = est.kneighbors(X)
        od, oi = orc.kneighbors(st, ids, k=k)
        assert np.array_equal(od, rd)
        orc.assert_tie_aware_equal(od, oi, rd, ri, rtol=0, atol=0, gap_rtol=0)
    # few trees = few distinct distances = many exact ties at the k-th place, which the two sides may
    # break differently (tie-aware check above); the averaging step is compared on the reference's own
    # neighbours, the whole prediction on the rows where both picked the same ones
    rd, ri = est.kneighbors(Q)
    od, oi = orc.kneighbors(st, ids_q, k=k)
    rp = est.predict(Q)
    np.testing.assert_allclose(orc.weighted_average(y, ri), rp, rtol=1e-12)
    same = (oi == ri).all(axis=1)
    assert same.sum() >= 20
    np.testing.assert_allclose(orc.predict(st, ids_q, k=k)[same], rp[same], rtol=1e-12)


def _fresh_float_data():
    rng = np.random.default_rng(20260)
    n_ref, d, n_out = 600, 6, 3
    A = rng.standard_normal((d, d))
    R = rng.standard_normal((n_ref, d)) @ A + rng.standard_normal(d) * 3.0
    R[50:60] = R[40:50]                                   # duplicated plots: exact distance ties
    y = rng.standard_normal((n_ref, n_out))
    Q = rng.standard_normal((400, d)) @ A
    Q[:20] = R[100:120]                                   # queries on top of plots: zero distances
    return R, y, Q


@pytest.mark.parametrize(("transformer", "weights"), [
    ("StandardScalerWithDOF", "distance"), ("StandardScalerWithDOF", "uniform"),
    ("MahalanobisTransformer", "distance"), (None, "uniform"),
])
def test_oracle_matches_scikit_learn_on_fresh_random_data(transformer, weights):
    """The data of test_oracle_matches_installed_reference_on_fresh_random_data without the reference
    package: the oracle against scikit-learn's brute KNeighborsRegressor, the code the reference hands its
    transformed plots to (ref:src/sknnr/_base.py:162-164), on the same feature space.  Ties between
    duplicated plots, zero distances under weights='distance' and the X=None self-query."""
    from sklearn.neighbors import KNeighborsRegressor

    import sknnr_b200.transformers as T

    R, y, Q = _fresh_float_data()
    k = 5
    center = scale = proj = None
    if transformer is not None:
        kw = {"ddof": 1} if transformer == "StandardScalerWithDOF" else {}
        center, scale, proj, _ = getattr(T, transformer)(**kw).fit(R, y)._affine()
    st = orc.FittedState(kind="euclidean", fit_Z=orc.affine_project(R, center, scale, proj), y=y,
                         center=center, scale=scale, proj=proj)
    skl = KNeighborsRegressor(n_neighbors=k, weights=weights, algorithm="brute").fit(st.fit_Z, y)
    Zq = orc.affine_project(Q, center, scale, proj)
    for X, Z in ((Q, Zq), (None, None)):
        rd, ri = skl.kneighbors(Z)
        od, oi = orc.kneighbors(st, X, k, deterministic=False)
        orc.assert_tie_aware_equal(od, oi, rd, ri, rtol=1e-7, atol=5e-7)
        # scikit-learn leaves the order of exactly tied plots to its heap: only duplicated plots may trade places
        assert np.isin(oi[oi != ri], np.r_[40:60]).all()
    rp = skl.predict(Zq)
    op = orc.predict(st, Q, k, weights=weights, deterministic=False)
    ok = np.isclose(op, rp, rtol=1e-6, atol=1e-6).all(axis=1)
    assert (~ok).sum() <= 12, int((~ok).sum())
    assert ok[:20].all()


@pytest.mark.parametrize("est_name", ["RFNNRegressor", "GBNNRegressor"])
def test_hamming_oracle_matches_scikit_learn_on_fresh_forests(est_name):
    """The forests of test_hamming_oracle_matches_installed_reference_on_fresh_forests without the
    reference package: node IDs from scikit-learn's own Tree.apply, tree weights from this package's
    fit side (pinned against the reference in test_host.py), and the oracle against scikit-learn's brute
    weighted-Hamming KNeighborsRegressor - bit-equal distances, tie-aware neighbours, X=None included."""
    import warnings

    from sklearn.neighbors import KNeighborsRegressor

    import sknnr_b200 as S

    rng = np.random.default_rng(7)
    n_ref, d, k = 250, 5, 5
    R = rng.standard_normal((n_ref, d))
    y = np.column_stack([R[:, 0] + 0.3 * rng.standard_normal(n_ref), R[:, 1] * R[:, 2], rng.standard_normal(n_ref)])
    Q = rng.standard_normal((120, d))
    est = getattr(S, est_name)(n_neighbors=k, n_estimators=12 if est_name == "RFNNRegressor" else 8, random_state=3)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", FutureWarning)
        est.transformer_ = est._get_transformer().fit(R, y)
    w = est._get_hamming_weights()
    trees = est.transformer_._trees()
    ids_ref = np.stack([t.apply(R.astype(np.float32)) for t in trees], axis=1).astype(np.int64)
    ids_q = np.stack([t.apply(Q.astype(np.float32)) for t in trees], axis=1).astype(np.int64)
    assert ids_ref.shape[1] == len(w) and abs(w.sum() - 1.0) < 1e-9
    if est_name == "GBNNRegressor":
        assert len(np.unique(w)) > 3   # genuinely unequal weights
    st = orc.FittedState(kind="hamming", fit_Z=ids_ref, y=y, hamming_w=w)
    skl = KNeighborsRegressor(n_neighbors=k, metric="hamming", metric_params={"w": w}, algorithm="brute").fit(ids_ref, y)
    for X, ids in ((ids_q, ids_q), (None, None)):
        rd, ri = skl.kneighbors(ids)
        od, oi = orc.kneighbors(st, X, k=k, deterministic=False)
        assert np.array_equal(od, rd)
        orc.assert_tie_aware_equal(od, oi, rd, ri, rtol=0, atol=0, gap_rtol=0)
    rd, ri = skl.kneighbors(ids_q)
    od, oi = orc.kneighbors(st, ids_q, k=k, deterministic=False)
    rp = skl.predict(ids_q)
    np.testing.assert_allclose(orc.weighted_average(y, ri), rp, rtol=1e-12)
    same = (oi == ri).all(axis=1)
    assert same.sum() >= 20
    np.testing.assert_allclose(orc.predict(st, ids_q, k=k, deterministic=False)[same], rp[same], rtol=1e-12)
