"""GPU parity tests: CUDA path (through the C ABI) vs the CPU oracle and golden fixtures."""

import numpy as np
import pytest

from oracle import sknnr_oracle as orc
from tests.conftest import FLOAT_CASES, load_golden, state_from_golden

pytestmark = pytest.mark.gpu

# Stated tolerances (BASELINE.json north_star): distances / predictions within 1e-5 relative,
# with an absolute floor for d -> 0 where the reference's own float64 expansion is noisy.
RTOL = 1e-5


def _index(st):
    from sknnr_b200._engine import KNNIndex

    return KNNIndex(st.fit_Z, st.center, st.scale, st.proj, st.y)


def _atol(st):
    # the reference's expansion error scales with the squared norms of the operands
    z = st.fit_Z
    return 1e-7 * float(np.sqrt((z * z).sum(1).max())) + 1e-12


@pytest.mark.parametrize(("name", "comp"), FLOAT_CASES)
def test_golden_kneighbors_and_predict(name, comp):
    g = load_golden(f"moscow_{name}_{comp}.npz")
    sp = load_golden("moscow_split.npz")
    st = state_from_golden(g)
    ix = _index(st)
    atol = _atol(st)
    # X given: projection + search + ordering
    d, i, p = ix.query(sp["X_test"], 5, weights="uniform", with_pred=True)
    np.testing.assert_array_equal(i, g["refgold_tgt_index_nn"])
    np.testing.assert_allclose(d, g["refgold_tgt_index_dist"], rtol=RTOL, atol=atol)
    np.testing.assert_allclose(p, g["refgold_tgt_unweighted_pred"], rtol=RTOL, atol=1e-8)
    # X=None: k+1 with self excluded, independent prediction and score
    d, i, p = ix.query(None, 5, exclude_self=True, weights="uniform", with_pred=True)
    np.testing.assert_array_equal(i, g["refgold_ref_index_nn"])
    np.testing.assert_allclose(d, g["refgold_ref_index_dist"], rtol=RTOL, atol=atol)
    np.testing.assert_allclose(p, g["refgold_ref_unweighted_pred"], rtol=RTOL, atol=1e-8)
    assert orc.r2_score_uniform(sp["y_train"], p) == pytest.approx(
        float(g["refgold_ref_unweighted_score"]), abs=1e-6)
    # distance weights
    _, _, p = ix.query(sp["X_test"], 5, weights="distance", with_pred=True)
    np.testing.assert_allclose(p, g["live_tgt_pred_distance"], rtol=RTOL, atol=1e-8)
    # callable weights: evaluated on host, averaged on device
    d, i, _ = ix.query(sp["X_test"], 5)
    p = ix.weighted_average(i, 1.0 / (1.0 + d))
    np.testing.assert_allclose(p, g["refgold_tgt_weighted_pred"], rtol=RTOL, atol=1e-8)
    # raw (non-deterministic) ordering is plain ascending distance
    d, i, _ = ix.query(sp["X_test"], 5, deterministic=False)
    np.testing.assert_allclose(d, g["live_tgt_dist_raw"], rtol=RTOL, atol=atol)
    # S2 alone
    np.testing.assert_allclose(ix.transform(sp["X_train"]), g["state_fit_Z"], rtol=1e-9, atol=1e-9)


def test_config1_swo_msn():
    g = load_golden("c1_swo_msn_k5.npz")
    st = state_from_golden(g)
    ix = _index(st)
    d, i, p = ix.query(None, 5, exclude_self=True, weights="uniform", with_pred=True)
    orc.assert_tie_aware_equal(d, i, g["live_ref_dist"], g["live_ref_nn"], rtol=RTOL, atol=_atol(st))
    assert orc.r2_score_uniform(g["y_targets"], p) == pytest.approx(float(g["live_ref_score"]), abs=1e-6)
    d, i, p = ix.query(g["X"], 5, weights="distance", with_pred=True)
    orc.assert_tie_aware_equal(d, i, g["live_self_dist"], g["live_self_nn"], rtol=RTOL, atol=1e-5)
    assert ix.stats()["n_queries"] == 3005


def test_config2_moscow_gnn_independent_score():
    g = load_golden("c2_moscow_gnn_k5.npz")
    st = state_from_golden(g)
    ix = _index(st)
    d, i, p = ix.query(None, 5, exclude_self=True, weights="uniform", with_pred=True)
    np.testing.assert_array_equal(i, g["live_ref_nn"])
    np.testing.assert_allclose(d, g["live_ref_dist"], rtol=RTOL, atol=_atol(st))
    np.testing.assert_allclose(p, g["live_ref_pred"], rtol=RTOL, atol=1e-8)
    assert orc.r2_score_uniform(g["y_targets"], p) == pytest.approx(float(g["live_ref_score"]), abs=1e-6)


def _synthetic(n_ref, n_q, d, n_out=4, seed=0, corr=False):
    rng = np.random.default_rng(seed)
    R = rng.standard_normal((n_ref, d))
    Q = np.random.default_rng(seed + 2).standard_normal((n_q, d))
    if corr:
        A = np.random.default_rng(3).standard_normal((d, d)) / np.sqrt(d)
        R, Q = R @ A, Q @ A
    y = np.random.default_rng(seed + 1).standard_normal((n_ref, n_out))
    return R, Q, y


@pytest.mark.parametrize(("n_ref", "n_q", "d", "k"), [
    (5000, 3000, 32, 7), (777, 1001, 17, 5), (20000, 2048, 64, 7), (300, 257, 3, 1),
    (4096, 512, 40, 15), (5000, 700, 8, 24),
])
def test_synthetic_euclidean_matches_oracle(n_ref, n_q, d, k):
    R, Q, y = _synthetic(n_ref, n_q, d)
    mean, scale = R.mean(0), R.std(0, ddof=1)
    st = orc.FittedState("euclidean", fit_Z=(R - mean) / scale, y=y, center=mean, scale=scale)
    ix = _index(st)
    d_o, i_o = orc.kneighbors(st, Q, k=k)
    p_o = orc.weighted_average(y, i_o, orc.get_weights(d_o, "distance"))
    d_g, i_g, p_g = ix.query(Q, k, weights="distance", with_pred=True)
    orc.assert_tie_aware_equal(d_g, i_g, d_o, i_o, rtol=RTOL, atol=1e-7)
    same = (i_g == i_o).all(axis=1)
    np.testing.assert_allclose(p_g[same], p_o[same], rtol=RTOL, atol=1e-8)
    # float32 queries take the same path (converted to float64 on the device)
    d32, i32, _ = ix.query(Q.astype(np.float32), k)
    assert (i32 == i_o).mean() > 0.99
    # sharded call with row offsets == one call
    h = n_q // 2
    d_a, i_a, _ = ix.query(Q[:h], k)
    d_b, i_b, _ = ix.query(Q[h:], k, row_offset=h)
    np.testing.assert_array_equal(np.vstack([i_a, i_b]), i_g)
    np.testing.assert_array_equal(np.vstack([d_a, d_b]), d_g)


def test_mahalanobis_projection_and_engines_agree():
    from sknnr_b200 import _lib as L

    R, Q, y = _synthetic(6000, 1500, 24, corr=True)
    mean, scale = R.mean(0), R.std(0, ddof=1)
    Rs = (R - mean) / scale
    W = np.linalg.inv(np.linalg.cholesky(np.cov(Rs, rowvar=False)).T)
    st = orc.FittedState("euclidean", fit_Z=Rs @ W, y=y, center=mean, scale=scale, proj=W)
    ix = _index(st)
    d_o, i_o = orc.kneighbors(st, Q, k=7)
    d_g, i_g, _ = ix.query(Q, 7)
    orc.assert_tie_aware_equal(d_g, i_g, d_o, i_o, rtol=RTOL, atol=1e-7)
    assert ix.stats()["engine"] == L.ENGINE_TENSOR      # default first stage: tcgen05 filter
    # every engine is only a filter in front of the same float64 refine: identical results
    for engine in (L.ENGINE_SIMT, L.ENGINE_EXACT, L.ENGINE_TENSOR):
        L.set_option("engine", engine)
        try:
            d_e, i_e, _ = ix.query(Q, 7)
            assert ix.stats()["engine"] == engine
        finally:
            L.set_option("engine", L.ENGINE_AUTO)
        np.testing.assert_array_equal(i_e, i_g)
        np.testing.assert_array_equal(d_e, d_g)


@pytest.mark.parametrize("engine", [1, 2])
def test_ill_conditioned_raw_features_cascade(engine):
    """Raw, uncentred features with huge norms relative to neighbour distances: the TF32 filter
    cannot certify most rows, the cascade hands them to the FP32 engine and the exact kernel,
    and the answers still match the oracle."""
    from sknnr_b200 import _lib as L

    rng = np.random.default_rng(11)
    R = rng.standard_normal((3000, 5)) * np.array([1.0, 50.0, 0.01, 3.0, 1000.0]) + np.array([5e5, 4e6, 10.0, 0.0, 2e4])
    Q = R[rng.integers(0, 3000, 900)] + rng.standard_normal((900, 5)) * np.array([0.3, 20.0, 0.003, 1.0, 300.0])
    st = orc.FittedState("euclidean", fit_Z=R, y=np.zeros((3000, 1)))
    ix = _index(st)
    L.set_option("engine", engine)
    try:
        d_g, i_g, _ = ix.query(Q, 5, transformed=True)
    finally:
        L.set_option("engine", L.ENGINE_AUTO)
    d_o, i_o = orc.kneighbors(st, Q, k=5, transformed=True)
    orc.assert_tie_aware_equal(d_g, i_g, d_o, i_o, rtol=1e-5, atol=1e-3 * float(d_o.mean()))


def test_adversarial_duplicates_offsets_and_self_queries():
    rng = np.random.default_rng(5)
    R = rng.standard_normal((2000, 6))
    R[:, 0] += 500.0 * R[:, 0].std()          # constant-offset feature (mean/std = 500)
    R[100:140] = R[100]                        # 40 exact duplicates (> k+1)
    R[300:303] = R[300]
    y = rng.standard_normal((2000, 3))
    st = orc.FittedState("euclidean", fit_Z=R.copy(), y=y)
    ix = _index(st)
    Q = np.vstack([R[:500], R[100:102] + 1e-9, rng.standard_normal((50, 6)) + R.mean(0)])
    d_o, i_o = orc.kneighbors(st, Q, k=5)
    d_g, i_g, _ = ix.query(Q, 5, transformed=True)
    # the reference's expansion is noisy at d -> 0 with a 500-sigma offset: absolute floor
    orc.assert_tie_aware_equal(d_g, i_g, d_o, i_o, rtol=RTOL, atol=2e-4, gap_rtol=1e-6)
    # exact duplicates: the lowest indices win, exactly like the reference's heap
    assert i_g[100].tolist() == [100, 101, 102, 103, 104]
    assert np.all(d_g[100] == 0)
    # X=None with >= k+1 duplicates drops column 0 when the row itself is not returned
    d_s, i_s, _ = ix.query(None, 5, exclude_self=True, deterministic=False)
    assert i_s[139].tolist() == [101, 102, 103, 104, 105]
    assert i_s[100].tolist() == [101, 102, 103, 104, 105]
    d_so, i_so = orc.kneighbors(st, None, k=5, deterministic=False)
    np.testing.assert_array_equal(i_s[100:140], i_so[100:140])
    assert ix.stats()["n_fallback"] >= 40      # the tie certificate routed them to the exact kernel


def test_ordering_known_answers():
    """ref:tests/test_estimators.py:306-378 through the device epilogue."""
    from sknnr_b200._engine import KNNIndex

    ix = KNNIndex(np.array([1e-11, 1e-12, 1.0]).reshape(-1, 1), y=np.array([0.0, 1.0, 2.0]))
    q = np.array([[0.0], [0.0]])
    assert ix.query(q[:1], 2, deterministic=False)[1][0].tolist() == [1, 0]
    assert ix.query(q[:1], 2, deterministic=True)[1][0].tolist() == [0, 1]
    assert ix.query(q, 2)[1].tolist() == [[0, 1], [1, 0]]
    assert ix.query(q[:1], 2, row_offset=1)[1].tolist() == [[1, 0]]
    ix = KNNIndex(np.array([1e-3, 1e-6, 1e-9, 1.0]).reshape(-1, 1))
    for dec, exp in ((8, [2, 1, 0]), (5, [1, 2, 0]), (2, [0, 1, 2])):
        assert ix.query(np.array([[0.0]]), 3, decimals=dec)[1][0].tolist() == exp


def test_error_behaviour():
    from sknnr_b200._engine import KNNIndex

    ix = KNNIndex(np.random.default_rng(0).standard_normal((10, 3)))
    with pytest.raises(ValueError, match="n_neighbors <= n_samples_fit"):
        ix.query(np.zeros((2, 3)), 11)
    with pytest.raises(ValueError, match="n_neighbors < n_samples_fit"):
        ix.query(None, 10, exclude_self=True)
    with pytest.raises(ValueError, match="features"):
        ix.query(np.zeros((2, 4)), 2)
    d, i, _ = ix.query(np.zeros((0, 3)), 2)
    assert d.shape == (0, 2) and i.shape == (0, 2)


@pytest.mark.parametrize("k", [33, 40, 97, 300])
def test_large_k_matches_oracle(k):
    """ref:src/sknnr/_base.py:162-164 accepts any n_neighbors <= n_samples_fit: beyond 32 the
    exhaustive float64 engine selects and finishes the row with a whole CTA."""
    from sknnr_b200._engine import HammingIndex, KNNIndex

    rng = np.random.default_rng(k)
    n_ref = 301
    R = rng.standard_normal((n_ref, 6))
    R[200:230] = R[:30]                       # exact ties
    y = rng.standard_normal((n_ref, 3))
    Q = np.vstack([R[rng.integers(0, n_ref, 40)], rng.standard_normal((25, 6))])
    st = orc.FittedState("euclidean", fit_Z=R, y=y)
    ix = KNNIndex(R, None, None, None, y)
    for off in (0, 1000):
        d_o, i_o = orc.kneighbors(st, Q, k=k, row_offset=off, transformed=True)
        d_g, i_g, p_g = ix.query(Q, k, transformed=True, weights="distance", with_pred=True, row_offset=off)
        # (the reference's expansion |x|^2 - 2 x.y + |y|^2 returns ~1e-8 for a zero distance)
        orc.assert_tie_aware_equal(d_g, i_g, d_o, i_o, rtol=1e-6, atol=1e-6)
        same = (i_g == i_o).all(axis=1) & (d_o > 1e-6).all(axis=1)
        p_o = orc.weighted_average(y, i_o, orc.get_weights(d_o, "distance"))
        np.testing.assert_allclose(p_g[same], p_o[same], rtol=1e-6, atol=1e-9)
    if k + 1 <= n_ref:
        d_o, i_o = orc.kneighbors(st, None, k=k)
        d_g, i_g, p_g = ix.query(None, k, exclude_self=True, weights="uniform", with_pred=True)
        orc.assert_tie_aware_equal(d_g, i_g, d_o, i_o, rtol=1e-6, atol=1e-6)
    # Hamming: bit-exact (count, index) ranking also for k > 32
    T = 40
    Rc = rng.integers(0, 6, size=(n_ref, T))
    Qc = Rc[rng.integers(0, n_ref, 30)].copy()
    Qc[rng.random(Qc.shape) < 0.3] = 7
    w = np.full(T, 1.0 / T)
    hs = orc.FittedState("hamming", fit_Z=Rc, y=y, hamming_w=w)
    hd_o, hi_o = orc.kneighbors(hs, Qc, k=k)
    hd, hi, _ = HammingIndex(Rc.astype(np.uint16), w, y).query(Qc.astype(np.uint16), k)
    np.testing.assert_array_equal(hi, hi_o)
    assert np.array_equal(hd, hd_o)


# ---- Hamming / RFNN -------------------------------------------------------------------
def _ham_index(codes, w, y=None):
    from sknnr_b200._engine import HammingIndex

    return HammingIndex(codes, w, y)


def test_hamming_golden_rfnn_bit_exact():
    g = load_golden("moscow_rfnn.npz")
    ref = g["ids_train"].astype(np.int64)
    tgt = g["ids_test"].astype(np.int64)
    st = orc.FittedState("hamming", fit_Z=ref, y=g["y"], hamming_w=g["hamming_w"])
    ix = _ham_index(ref.astype(np.uint16), g["hamming_w"], g["y"])
    d_o, i_o = orc.kneighbors(st, tgt, k=5)
    d_g, i_g, p_g = ix.query(tgt.astype(np.uint16), 5, weights="uniform", with_pred=True)
    np.testing.assert_array_equal(i_g, i_o)          # canonical oracle: bit-exact indices
    assert np.array_equal(d_g, d_o)                  # and bit-exact float64 distances
    assert np.array_equal(d_g, g["live_tgt_dist"])   # == the live reference's distances
    orc.assert_tie_aware_equal(d_g, i_g, g["live_tgt_dist"], g["live_tgt_nn"], rtol=0, atol=0, gap_rtol=0)
    np.testing.assert_allclose(p_g, orc.weighted_average(g["y"], i_o), rtol=1e-12)
    d_o, i_o = orc.kneighbors(st, None, k=5)
    d_g, i_g, _ = ix.query(None, 5, exclude_self=True)
    np.testing.assert_array_equal(i_g, i_o)
    assert np.array_equal(d_g, d_o)
    # unequal (user-supplied forest) weights: exact float64 kernel, still bit-exact
    w2 = g["hamming_w_nonuniform"]
    st2 = orc.FittedState("hamming", fit_Z=ref, y=g["y"], hamming_w=w2)
    ix2 = _ham_index(ref.astype(np.uint16), w2, g["y"])
    d_o, i_o = orc.kneighbors(st2, tgt, k=5)
    d_g, i_g, _ = ix2.query(tgt.astype(np.uint16), 5)
    np.testing.assert_array_equal(i_g, i_o)
    assert np.array_equal(d_g, d_o)
    assert np.array_equal(d_g, g["live_tgt_dist_nonuniform"])


@pytest.mark.parametrize(("n_ref", "n_q", "T", "k", "n_codes"), [
    (3000, 1000, 500, 7, 40), (500, 300, 63, 5, 3), (1000, 257, 130, 1, 31743), (2000, 400, 64, 12, 8),
])
def test_hamming_synthetic_bit_exact(n_ref, n_q, T, k, n_codes):
    rng = np.random.default_rng(7)
    R = rng.integers(0, n_codes, size=(n_ref, T))
    # queries resemble references (as forest leaves do) so that small counts occur
    Q = R[rng.integers(0, n_ref, size=n_q)].copy()
    flip = rng.random(Q.shape) < 0.4
    Q[flip] = rng.integers(0, n_codes, size=int(flip.sum()))
    w = np.full(T, 1.0 / T / 3)
    st = orc.FittedState("hamming", fit_Z=R, y=np.zeros((n_ref, 1)), hamming_w=w)
    d_o, i_o = orc.kneighbors(st, Q, k=k)
    ix = _ham_index(R.astype(np.uint16), w)
    d_g, i_g, _ = ix.query(Q.astype(np.uint16), k)
    np.testing.assert_array_equal(i_g, i_o)
    assert np.array_equal(d_g, d_o)


@pytest.mark.parametrize(("streams", "seed_stride", "k", "exclude_self"), [
    (2, 4, 7, False), (2, 0, 7, False), (2, 2, 5, True), (1, 4, 7, False), (1, 8, 12, False),
    (2, 4, 7, True),
])
def test_tensor_engine_configurations_match_oracle(streams, seed_stride, k, exclude_self):
    """The tensor engine's knobs (candidate streams per query, threshold-seeding stride) only change
    how the filter works, never the result: every configuration equals the oracle and the
    exhaustive float64 engine bit for bit.  12k plots = 94 reference tiles, enough for seeding."""
    from sknnr_b200 import _lib as L

    R, Q, y = _synthetic(12000, 1300, 32, seed=5)
    st = orc.FittedState("euclidean", fit_Z=R, y=y)
    ix = _index(st)
    Qx = None if exclude_self else Q
    d_o, i_o = orc.kneighbors(st, Qx, k=k, transformed=True)
    L.set_option("tc_streams", streams)
    L.set_option("tc_seed_stride", seed_stride)
    L.set_option("engine", L.ENGINE_TENSOR)
    try:
        d_g, i_g, _ = ix.query(Qx, k, transformed=True, exclude_self=exclude_self)
        assert ix.stats()["engine"] == L.ENGINE_TENSOR
        L.set_option("engine", L.ENGINE_EXACT)
        d_e, i_e, _ = ix.query(Qx, k, transformed=True, exclude_self=exclude_self)
    finally:
        L.set_option("engine", L.ENGINE_AUTO)
        L.set_option("tc_streams", 0)
        L.set_option("tc_seed_stride", 4)
    orc.assert_tie_aware_equal(d_g, i_g, d_o, i_o, rtol=RTOL, atol=1e-7)
    np.testing.assert_array_equal(i_g, i_e)
    np.testing.assert_array_equal(d_g, d_e)


def test_tensor_engine_duplicates_and_queries_on_plots():
    """Adversarial parity set of SURVEY.md section 8(d): duplicated reference rows (exact ties ->
    lowest index), queries equal to references (zero distances -> indicator weights) and a
    constant-offset feature; the tie rows must come out of the cascade's exact stage identical
    to the oracle."""
    rng = np.random.default_rng(9)
    R = rng.standard_normal((9000, 16))
    R[:, 3] += 500.0
    R[4000:4500] = R[:500]                       # 500 duplicated plots
    off = np.zeros(16)
    off[3] = 500.0
    Q = np.vstack([R[rng.integers(0, 9000, 400)], rng.standard_normal((400, 16)) + off])
    y = rng.standard_normal((9000, 3))
    st = orc.FittedState("euclidean", fit_Z=R, y=y)
    ix = _index(st)
    d_o, i_o = orc.kneighbors(st, Q, k=7, transformed=True)
    d_g, i_g, p_g = ix.query(Q, 7, transformed=True, weights="distance", with_pred=True)
    # (the reference's float64 expansion returns ~1e-5 instead of 0 for a query that IS a plot with
    # a feature offset of 500; ours is exactly 0 -> absolute floor from the operand norms)
    orc.assert_tie_aware_equal(d_g, i_g, d_o, i_o, rtol=RTOL, atol=_atol(st))
    assert (d_g[:400, 0] == 0.0).all()
    same = (i_g == i_o).all(axis=1) & (d_o[:, 0] > 1e-3)
    p_o = orc.weighted_average(y, i_o, orc.get_weights(d_o, "distance"))
    np.testing.assert_allclose(p_g[same], p_o[same], rtol=RTOL, atol=1e-8)
    # zero-distance rows: indicator weights on the coincident plot(s), $SP/sklearn/neighbors/_base.py:107-114
    assert np.isfinite(p_g).all()
    w = (d_g[:400] == 0.0).astype(float)
    np.testing.assert_allclose(p_g[:400], orc.weighted_average(y, i_g[:400], w), rtol=1e-12, atol=1e-12)


# ---- forest walk (scope row f1) -----------------------------------------------------------
@pytest.mark.parametrize("kind", ["regressor", "classifier", "multi"])
def test_forest_apply_bit_exact_with_sklearn(kind):
    """RFNodeTransformer.transform on the device == hstack(est.apply(X)) of scikit-learn
    (ref:src/sknnr/transformers/_tree_node_transformer.py:177-201), for float64 and float32
    inputs, values that sit exactly on thresholds included."""
    from sknnr_b200.transformers import RFNodeTransformer

    rng = np.random.default_rng(4)
    X = rng.standard_normal((1500, 11)) * np.array([1, 10, 0.1, 1000, 1, 1, 5, 1, 1, 1e-3, 1]) + 3.0
    X[:, 6] = np.round(X[:, 6])                      # few distinct values -> thresholds between them
    if kind == "regressor":
        y = X[:, :1] * 2 + rng.standard_normal((1500, 1))
    elif kind == "classifier":
        y = (X[:, 1] > 3).astype(int).astype(str).reshape(-1, 1)
    else:
        y = np.column_stack([X[:, 0] + rng.standard_normal(1500), np.round(X[:, 6]), X[:, 3] * 0.01])
    tr = RFNodeTransformer(n_estimators=23, random_state=1, min_samples_leaf=3).fit(X, y)
    Q = np.vstack([X[:300], rng.standard_normal((700, 11)) * 3 + 3.0])
    # rows that sit exactly on (float32) thresholds of the first trees
    t0 = tr.estimators_[0].estimators_[0].tree_
    inner = np.flatnonzero(t0.children_left >= 0)[:50]
    for j, n in enumerate(inner):
        Q[j, t0.feature[n]] = np.float32(t0.threshold[n])
    want = np.hstack([e.apply(Q) for e in tr.estimators_]).astype(np.int64)
    got = tr.transform(Q)
    assert got.dtype == np.int64 and got.shape == want.shape
    np.testing.assert_array_equal(got, want)
    want32 = np.hstack([e.apply(Q.astype(np.float32)) for e in tr.estimators_]).astype(np.int64)
    np.testing.assert_array_equal(tr.transform(Q.astype(np.float32)), want32)
    with pytest.raises(ValueError):
        tr.transform(np.full((2, 11), 1e300))        # not representable in float32, as est.apply rejects it


def test_rfnn_fused_forest_query_equals_two_step_path():
    """RFNNRegressor.kneighbors / predict on raw features (forest walk fused in front of the Hamming
    search) == Hamming search on the node IDs scikit-learn's apply returns, bit for bit."""
    import sknnr_b200 as S

    rng = np.random.default_rng(8)
    X = rng.standard_normal((900, 9))
    y = np.column_stack([X[:, 0] * 2 + rng.standard_normal(900), X[:, 1] - X[:, 2]])
    Q = rng.standard_normal((400, 9))
    est = S.RFNNRegressor(n_estimators=31, n_neighbors=4, random_state=0, weights="distance").fit(X, y)
    ids_ref = np.hstack([e.apply(X) for e in est.transformer_.estimators_]).astype(np.int64)
    ids_q = np.hstack([e.apply(Q) for e in est.transformer_.estimators_]).astype(np.int64)
    np.testing.assert_array_equal(est.transformer_.transform(X), ids_ref)
    st = orc.FittedState("hamming", fit_Z=ids_ref, y=y, hamming_w=est.hamming_weights_)
    d_o, i_o = orc.kneighbors(st, ids_q, k=4, transformed=True)
    d, i = est.kneighbors(Q)                                   # fused: raw rows in
    np.testing.assert_array_equal(i, i_o)
    np.testing.assert_array_equal(d, d_o)
    d2, i2 = est.regressor_.kneighbors(ids_q)                  # two-step: node IDs in
    np.testing.assert_array_equal(i2, i)
    np.testing.assert_array_equal(d2, d)
    p_o = orc.weighted_average(y, i_o, orc.get_weights(d_o, "distance"))
    np.testing.assert_allclose(est.predict(Q), p_o, rtol=RTOL, atol=1e-10)
    assert est.regressor_._get_index().stats()["kernel_launches"] == 4   # forest + pack + search + finish


# ---- weighted Hamming / GBNN (scope row f3) ------------------------------------------------
def test_hamming_golden_gbnn_weighted_filter_bit_exact():
    """GBNN's train-improvement weights: fixed-point filter + float64 refine + certificate must
    reproduce the oracle and the live reference bit for bit (3500 trees; mixed model 400 trees)."""
    from sknnr_b200 import _lib as L

    g = load_golden("moscow_gbnn.npz")
    for tag in ("", "mixed_"):
        ref = g[tag + "ids_train"].astype(np.int64)
        tgt = g[tag + "ids_test"].astype(np.int64)
        w, y = g[tag + "hamming_w"], g[tag + "y"]
        st = orc.FittedState("hamming", fit_Z=ref, y=y, hamming_w=w)
        ix = _ham_index(ref.astype(np.uint16), w, y)
        d_o, i_o = orc.kneighbors(st, tgt, k=5)
        d_g, i_g, p_g = ix.query(tgt.astype(np.uint16), 5, weights="uniform", with_pred=True)
        assert ix.stats()["engine"] == L.ENGINE_SIMT          # the filter ran, not the exhaustive kernel
        np.testing.assert_array_equal(i_g, i_o)
        assert np.array_equal(d_g, d_o)
        assert np.array_equal(d_g, g[tag + "live_tgt_dist"])
        orc.assert_tie_aware_equal(d_g, i_g, g[tag + "live_tgt_dist"], g[tag + "live_tgt_nn"], rtol=0, atol=0, gap_rtol=0)
        np.testing.assert_allclose(p_g, g[tag + "live_tgt_pred"], rtol=1e-12)
        d_o, i_o = orc.kneighbors(st, None, k=5)
        d_g, i_g, _ = ix.query(None, 5, exclude_self=True)
        np.testing.assert_array_equal(i_g, i_o)
        assert np.array_equal(d_g, d_o)
        assert np.array_equal(d_g, g[tag + "live_ref_dist"])


@pytest.mark.parametrize(("n_ref", "n_q", "T", "k", "n_codes", "wkind"), [
    (3000, 1000, 500, 7, 40, "decay"), (500, 300, 63, 5, 3, "random"), (1000, 257, 130, 1, 31743, "decay"),
    (2000, 400, 64, 12, 8, "zeros"), (2500, 300, 1000, 20, 6, "decay"), (700, 200, 33, 28, 4, "random"),
    (12, 50, 40, 5, 3, "random"), (1500, 300, 96, 5, 2, "two"),
])
def test_weighted_hamming_synthetic_bit_exact(n_ref, n_q, T, k, n_codes, wkind):
    """Unequal weights of several shapes (geometric decay like boosting stages, zeros, only two
    distinct values -> masses of exactly tied distances that the certificate must hand to the
    exhaustive kernel), k up to 28 (> 24: exhaustive only), fewer references than candidates."""
    from sknnr_b200 import _lib as L

    rng = np.random.default_rng(11)
    R = rng.integers(0, n_codes, size=(n_ref, T))
    Q = R[rng.integers(0, n_ref, size=n_q)].copy()
    flip = rng.random(Q.shape) < 0.4
    Q[flip] = rng.integers(0, n_codes, size=int(flip.sum()))
    if wkind == "decay":
        w = 0.97 ** np.arange(T) * (1.0 + 0.1 * rng.random(T))
    elif wkind == "random":
        w = rng.random(T) + 0.01
    elif wkind == "zeros":
        w = rng.random(T)
        w[::3] = 0.0
    else:
        w = np.where(np.arange(T) % 2 == 0, 1.0, 3.0)
    w = w / w.sum()
    st = orc.FittedState("hamming", fit_Z=R, y=np.zeros((n_ref, 1)), hamming_w=w)
    d_o, i_o = orc.kneighbors(st, Q, k=k)
    ix = _ham_index(R.astype(np.uint16), w)
    d_g, i_g, _ = ix.query(Q.astype(np.uint16), k)
    stats = ix.stats()
    assert stats["engine"] == (L.ENGINE_SIMT if k <= 24 else L.ENGINE_EXACT)
    np.testing.assert_array_equal(i_g, i_o)
    assert np.array_equal(d_g, d_o)
    if wkind in ("decay", "random") and n_ref > 32 and k <= 24:
        assert stats["n_fallback"] <= n_q // 20         # the filter certifies nearly every row
    L.set_option("engine", L.ENGINE_EXACT)
    try:
        d_e, i_e, _ = ix.query(Q.astype(np.uint16), k)
    finally:
        L.set_option("engine", L.ENGINE_AUTO)
    np.testing.assert_array_equal(i_e, i_g)
    assert np.array_equal(d_e, d_g)


def test_gb_forest_apply_and_fused_gbnn_query():
    """GBNodeTransformer.transform on the device == scikit-learn's apply with the reference's
    class-major column order (ref:src/sknnr/transformers/_tree_node_transformer.py:190-200), and
    GBNNRegressor on raw features (forest walk + weighted Hamming filter fused) == the oracle on
    scikit-learn's node IDs."""
    import warnings

    import sknnr_b200 as S

    rng = np.random.default_rng(12)
    X = rng.standard_normal((800, 7))
    cls = np.where(X[:, 0] + 0.3 * rng.standard_normal(800) > 0.5, "a", np.where(X[:, 1] > 0, "b", "c"))
    y = np.column_stack([X[:, 0] * 2 + rng.standard_normal(800), X[:, 1] - X[:, 2]])
    import pandas as pd
    y_fit = pd.DataFrame({"t0": y[:, 0], "kind": cls})
    Q = rng.standard_normal((300, 7))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", FutureWarning)
        est = S.GBNNRegressor(n_estimators=40, n_neighbors=4, random_state=0, weights="distance").fit(X, y, y_fit=y_fit)
    tr = est.transformer_
    assert tr.n_trees_per_iteration_ == [1, 3]

    def sk_apply(A):
        cols = []
        for e in tr.estimators_:
            a = e.apply(A)
            if a.ndim == 3:
                a = np.swapaxes(a, 1, 2).reshape(a.shape[0], -1)
            cols.append(a)
        return np.hstack(cols).astype(np.int64)

    ids_ref, ids_q = sk_apply(X), sk_apply(Q)
    np.testing.assert_array_equal(tr.transform(X), ids_ref)
    np.testing.assert_array_equal(tr.transform(Q.astype(np.float32)), sk_apply(Q.astype(np.float32)))
    w = est.hamming_weights_
    assert w.shape == (160,) and len(np.unique(w)) > 20
    st = orc.FittedState("hamming", fit_Z=ids_ref, y=y, hamming_w=w)
    d_o, i_o = orc.kneighbors(st, ids_q, k=4, transformed=True)
    d, i = est.kneighbors(Q)
    np.testing.assert_array_equal(i, i_o)
    np.testing.assert_array_equal(d, d_o)
    d2, i2 = est.regressor_.kneighbors(ids_q)
    np.testing.assert_array_equal(i2, i)
    np.testing.assert_array_equal(d2, d)
    p_o = orc.weighted_average(y, i_o, orc.get_weights(d_o, "distance"))
    np.testing.assert_allclose(est.predict(Q), p_o, rtol=RTOL, atol=1e-10)
    d_o, i_o = orc.kneighbors(st, None, k=4)
    d, i = est.kneighbors()
    np.testing.assert_array_equal(i, i_o)
    np.testing.assert_array_equal(d, d_o)


# ---- raster front end (scope row f4) ---------------------------------------------------------
@pytest.mark.parametrize(("hw", "dtype", "nodata", "chunk"), [
    ((97, 131), np.float64, None, 4096), ((64, 200), np.float32, -9999.0, 4096),
    ((33, 1000), np.float64, -1.0, 1 << 20), ((5, 7), np.float32, None, 4096),
])
def test_raster_kneighbors_equals_row_query_and_oracle(hw, dtype, nodata, chunk):
    """Band-major image in, band-major layers out == the oracle's flatten / mask / query / scatter
    loop, and bit-equal to this library's own row query on the unmasked pixels.  Covers several
    pixel blocks per call (chunk_rows 4096), a block with no valid pixel, NaN / inf / nodata masks
    and band-strided float32 input."""
    from sknnr_b200 import _lib as L

    d, k = 9, 5
    R, _, y = _synthetic(3000, 10, d)
    mean, scale = R.mean(0), R.std(0, ddof=1)
    st = orc.FittedState("euclidean", fit_Z=(R - mean) / scale, y=y, center=mean, scale=scale)
    ix = _index(st)
    rng = np.random.default_rng(21)
    n_pix = hw[0] * hw[1]
    big = np.zeros((d, n_pix + 13), dtype=dtype)          # bands strided by more than n_pix
    img = big[:, :n_pix]
    img[...] = rng.standard_normal((d, n_pix)).astype(dtype)
    drop = rng.random(n_pix) < 0.3
    img[rng.integers(0, d, size=n_pix)[drop], np.flatnonzero(drop)] = np.nan
    img[2, ::17] = np.inf
    if nodata is not None:
        img[rng.integers(0, d), ::11] = nodata
    if n_pix > 3 * 4096:
        img[0, 4096:8192] = np.nan                         # a whole block without a valid pixel
    image = img.reshape(d, *hw)
    L.set_option("chunk_rows", chunk)
    try:
        dist, idx, pred, n_valid = ix.query_raster(img, k, nodata=nodata, weights="distance", with_pred=True)
    finally:
        L.set_option("chunk_rows", 1 << 20)
    X = img.T.astype(np.float64)
    valid = np.isfinite(X).all(1)
    if nodata is not None:
        valid &= ~(img.T == nodata).any(1)
    assert n_valid == int(valid.sum()) and 0 < n_valid < n_pix
    # masked pixels: fill values
    assert np.isnan(dist[:, ~valid]).all() and (idx[:, ~valid] == -1).all() and np.isnan(pred[:, ~valid]).all()
    # unmasked pixels: bit-equal to the row query of the same library ...
    d_r, i_r, p_r = ix.query(np.ascontiguousarray(img.T[valid]), k, weights="distance", with_pred=True)
    np.testing.assert_array_equal(idx[:, valid].T, i_r)
    np.testing.assert_array_equal(dist[:, valid].T, d_r)
    np.testing.assert_array_equal(pred[:, valid].T, p_r)
    # ... and equal to the oracle's raster loop
    d_o, i_o, p_o = orc.raster_query(st, image, k=k, nodata=nodata, weights="distance")
    orc.assert_tie_aware_equal(dist[:, valid].T, idx[:, valid].T, d_o.reshape(k, -1)[:, valid].T,
                               i_o.reshape(k, -1)[:, valid].T, rtol=RTOL, atol=1e-7)
    same = (idx == i_o.reshape(k, -1)).all(axis=0) & valid
    np.testing.assert_allclose(pred[:, same], p_o.reshape(y.shape[1], -1)[:, same], rtol=RTOL, atol=1e-8)


def test_raster_estimator_helpers():
    """predict_raster / kneighbors_raster on fitted estimators: == predict / kneighbors on the
    flattened valid pixels (uniform, distance and callable weights), fills, and input errors."""
    import sknnr_b200 as S

    g = load_golden("moscow_split.npz")
    Xtr, ytr, Xte = g["X_train"], g["y_train"], g["X_test"]
    rng = np.random.default_rng(3)
    pix = np.vstack([Xte, Xtr[:27]])                        # 60 pixels -> 6 x 10 image
    image = np.ascontiguousarray(pix.T).reshape(Xtr.shape[1], 6, 10).copy()
    image[3, 2, 5] = np.nan
    image[0, 0, 0] = -9999.0
    valid = np.ones(60, dtype=bool)
    valid[[25, 0]] = False
    for cls, kw in ((S.MSNRegressor, {}), (S.EuclideanKNNRegressor, {"weights": "distance"}),
                    (S.GNNRegressor, {"weights": lambda dd: 1.0 / (1.0 + dd)}), (S.RawKNNRegressor, {})):
        est = cls(n_neighbors=5, **kw).fit(Xtr, ytr)
        pr = S.predict_raster(est, image, nodata=-9999.0, fill_value=-1.0)
        assert pr.shape == (ytr.shape[1], 6, 10)
        flat = pr.reshape(ytr.shape[1], -1)
        assert (flat[:, ~valid] == -1.0).all()
        np.testing.assert_allclose(flat[:, valid].T, est.predict(pix[valid]), rtol=1e-12, atol=1e-12)
        dist, idx = S.kneighbors_raster(est, image, nodata=-9999.0)
        d_r, i_r = est.kneighbors(pix[valid])
        np.testing.assert_array_equal(idx.reshape(5, -1)[:, valid].T, i_r)
        np.testing.assert_array_equal(dist.reshape(5, -1)[:, valid].T, d_r)
        assert (idx.reshape(5, -1)[:, ~valid] == -1).all()
        only = S.kneighbors_raster(est, image.astype(np.float32), n_neighbors=3, nodata=-9999.0, return_distance=False)
        assert only.shape == (3, 6, 10) and only.dtype == np.int64
    with pytest.raises(ValueError, match="features"):
        S.predict_raster(est, image[:-1])
    with pytest.raises(ValueError, match="bands, height, width"):
        S.predict_raster(est, pix)
    # tree-node estimators: forest walk + Hamming search behind the same front end
    import warnings

    for cls, kw in ((S.RFNNRegressor, {"n_estimators": 7}), (S.GBNNRegressor, {"n_estimators": 9, "weights": "distance"})):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", FutureWarning)
            est = cls(n_neighbors=4, random_state=0, **kw).fit(Xtr, ytr[:, :3])
        pr = S.predict_raster(est, image, nodata=-9999.0).reshape(3, -1)
        assert np.isnan(pr[:, ~valid]).all()
        np.testing.assert_allclose(pr[:, valid].T, est.predict(pix[valid]), rtol=1e-12, atol=1e-12)
        dist, idx = S.kneighbors_raster(est, image.astype(np.float32), nodata=-9999.0)
        d_r, i_r = est.kneighbors(pix[valid].astype(np.float32))
        np.testing.assert_array_equal(idx.reshape(4, -1)[:, valid].T, i_r)
        np.testing.assert_array_equal(dist.reshape(4, -1)[:, valid].T, d_r)
    with pytest.raises(NotImplementedError):
        S.predict_raster(S.RawKNNRegressor(n_neighbors=2, metric="hamming").fit(np.arange(40).reshape(10, 4) % 3, ytr[:10]), image[:4])


# ---- BASELINE.json's full C3 size, through size-independent properties ----------------------
def test_full_size_c3_properties():
    """10M queries x 50k plots x 32 features, k = 7 (the configuration the metric is quoted on).  The
    oracle cannot run this in seconds, so the result is checked through properties that do not
    depend on size: ordering, index validity, distances re-derived from the returned indices,
    exact agreement with the oracle on a random sample of rows, invariance under sharding /
    re-chunking (checksum of checksums), and the prediction identity."""
    from sknnr_b200 import _lib as L

    n_ref, n_q, d, k = 50_000, 10_000_000, 32, 7
    R = np.random.default_rng(0).standard_normal((n_ref, d))
    y = np.random.default_rng(1).standard_normal((n_ref, 8))
    mean, scale = R.mean(0), R.std(0, ddof=1)
    st = orc.FittedState("euclidean", fit_Z=(R - mean) / scale, y=y, center=mean, scale=scale)
    ix = _index(st)
    Q = np.empty((n_q, d))
    for b, ss in enumerate(np.random.SeedSequence(2).spawn(10)):
        Q[b * 1_000_000:(b + 1) * 1_000_000] = np.random.default_rng(ss).standard_normal((1_000_000, d))
    dist, idx, pred = ix.query(Q, k, weights="uniform", with_pred=True, deterministic=False)
    stats = ix.stats()
    assert stats["engine"] == L.ENGINE_TENSOR and stats["n_queries"] == n_q
    assert stats["n_fallback"] < n_q // 50                      # the filter certifies nearly every row
    # ordering and validity
    assert np.all(np.diff(dist, axis=1) >= 0) and np.all(dist > 0) and np.all(np.isfinite(dist))
    assert idx.min() >= 0 and idx.max() < n_ref
    srt = np.sort(idx, axis=1)
    assert np.all(srt[:, 1:] != srt[:, :-1])                   # no plot twice in a row's list
    # distances belong to the returned indices (float64 recomputation on a sample)
    rng = np.random.default_rng(5)
    rows = rng.choice(n_q, size=20_000, replace=False)
    Zs = (Q[rows] - mean) / scale
    recomputed = np.sqrt(((Zs[:, None, :] - st.fit_Z[idx[rows]]) ** 2).sum(-1))
    np.testing.assert_allclose(dist[rows], recomputed, rtol=1e-12, atol=1e-12)
    # exact agreement with the oracle on a sample of rows
    sub = rows[:3000]
    d_o, i_o = orc.kneighbors(st, Q[sub], k=k, deterministic=False)
    orc.assert_tie_aware_equal(dist[sub], idx[sub], d_o, i_o, rtol=RTOL, atol=1e-7)
    assert (idx[sub] == i_o).mean() > 0.9999
    # prediction identity: uniform weights = mean of the neighbours' targets
    np.testing.assert_allclose(pred[rows], y[idx[rows]].mean(axis=1), rtol=1e-12, atol=1e-12)
    # sharding / re-chunking invariance: two half calls with row offsets, another chunk size
    h = n_q // 2
    L.set_option("chunk_rows", 1 << 19)
    try:
        d_a, i_a, _ = ix.query(Q[:h], k, deterministic=False)
        d_b, i_b, _ = ix.query(Q[h:], k, deterministic=False, row_offset=h)
    finally:
        L.set_option("chunk_rows", 1 << 20)
    w = np.arange(1, k + 1, dtype=np.int64)
    assert int((i_a * w).sum() + (i_b * w).sum()) == int((idx * w).sum())     # checksum of checksums
    assert np.array_equal(i_a, idx[:h]) and np.array_equal(d_b, dist[h:])


def test_c4_shape_hamming_properties():
    """C4 shape (20k plots x 500 trees, k = 7) at 500k queries - a twentieth of BASELINE.json's 10M,
    which would need 10 GB of node codes on the host - through the same size-independent properties:
    ordering by (distance, index), distances re-derived from the returned indices, oracle agreement
    on a sample, sharding invariance.  Equal weights (RFNN) and boosting-like unequal weights (GBNN)."""
    n_ref, n_q, T, k = 20_000, 500_000, 500, 7
    rng = np.random.default_rng(0)
    Rc = rng.integers(0, 60, size=(n_ref, T)).astype(np.uint16)
    Qc = Rc[rng.integers(0, n_ref, size=n_q)].copy()
    flip = rng.random(Qc.shape) < 0.5
    Qc[flip] = rng.integers(0, 60, size=int(flip.sum())).astype(np.uint16)
    w_eq = np.full(T, 1.0 / T)
    w_gb = np.tile(0.97 ** np.arange(100), 5) * (1 + 0.1 * rng.random(T))
    w_gb /= w_gb.sum()
    rows = rng.choice(n_q, size=400, replace=False)
    for w in (w_eq, w_gb):
        ix = _ham_index(Rc, w)
        dist, idx, _ = ix.query(Qc, k, deterministic=False)   # plain (distance, index) order
        assert ix.stats()["n_fallback"] <= n_q // 100
        assert np.all(np.diff(dist, axis=1) >= 0)
        tie = np.diff(dist, axis=1) == 0
        assert np.all(np.diff(idx, axis=1)[tie] > 0)            # the lowest index wins every tie
        assert idx.min() >= 0 and idx.max() < n_ref
        # distances belong to the returned indices: SciPy's left-to-right float64 sums, bit for bit
        mism = Qc[rows][:, None, :] != Rc[idx[rows]]
        want = np.empty((len(rows), k))
        for a in range(len(rows)):
            for b in range(k):
                acc = 0.0
                for t in np.flatnonzero(mism[a, b]):
                    acc += w[t]
                want[a, b] = acc
        den = 0.0
        for t in range(T):
            den += w[t]
        assert np.array_equal(dist[rows], want / den)
        st = orc.FittedState("hamming", fit_Z=Rc.astype(np.int64), y=np.zeros((n_ref, 1)), hamming_w=w)
        d_o, i_o = orc.kneighbors(st, Qc[rows].astype(np.int64), k=k, deterministic=False)
        np.testing.assert_array_equal(idx[rows], i_o)
        assert np.array_equal(dist[rows], d_o)
        h = n_q // 2
        d_b, i_b, _ = ix.query(Qc[h:], k, row_offset=h, deterministic=False)
        assert np.array_equal(i_b, idx[h:]) and np.array_equal(d_b, dist[h:])
        ix.close()


# ---- round 2: host staging, device-side finite check, large shapes, non-integer node IDs -----
from sknnr_b200 import _lib as L  # noqa: E402


def test_pageable_and_page_locked_buffers_give_identical_results():
    """Ordinary NumPy arrays are staged through page-locked slot buffers by the library's host
    threads (csrc/api.cu); many small staged chunks, strided rows and caller-supplied result
    arrays must reproduce the page-locked path bit for bit."""
    from sknnr_b200._engine import KNNIndex, pinned_empty

    rng = np.random.default_rng(5)
    R = rng.standard_normal((700, 9))
    y = rng.standard_normal((700, 2))
    n_q = 20_000
    X = rng.standard_normal((n_q, 9))
    Xs = np.ascontiguousarray(np.hstack([X, rng.standard_normal((n_q, 3))]))[:, :9]   # row stride 12
    Xp = pinned_empty((n_q, 9))
    Xp[:] = X
    ix = KNNIndex(R, None, None, None, y)
    L.set_option("stage_rows", 1024)
    L.set_option("chunk_rows", 4096)
    try:
        ref = ix.query(Xp, 5, transformed=True, weights="distance", with_pred=True,
                       out=(pinned_empty((n_q, 5)), pinned_empty((n_q, 5), np.int64), pinned_empty((n_q, 2))))
        for Xin in (X, Xs, X.astype(np.float32).astype(np.float64)):
            got = ix.query(Xin, 5, transformed=True, weights="distance", with_pred=True)
            own = (np.empty((n_q, 5)), np.empty((n_q, 5), dtype=np.int64), np.empty((n_q, 2)))
            got2 = ix.query(Xin, 5, transformed=True, weights="distance", with_pred=True, out=own)
            if Xin is not X and Xin is not Xs:
                continue   # (the float32 round trip changes the values: only exercised, not compared)
            for a, b, c in zip(ref, got, got2):
                assert np.array_equal(a, b) and np.array_equal(a, c)
        with pytest.raises(ValueError, match="out"):
            ix.query(X, 5, transformed=True, out=(np.empty((n_q, 4)), np.empty((n_q, 5), dtype=np.int64), None))
    finally:
        L.set_option("stage_rows", 1 << 19)
        L.set_option("chunk_rows", 1 << 20)


def test_device_side_finite_check_raises_like_the_reference():
    from sknnr_b200 import EuclideanKNNRegressor, MSNRegressor, RawKNNRegressor
    from sknnr_b200._engine import KNNIndex

    rng = np.random.default_rng(6)
    R = rng.standard_normal((300, 6))
    y = rng.standard_normal((300, 3))
    X = rng.standard_normal((5000, 6))
    ix = KNNIndex(R, None, None, None, y)
    ok = ix.query(X, 3, transformed=True, check_finite=True)
    assert np.isfinite(ok[0]).all()
    for bad, where in ((np.nan, (4321, 2)), (np.inf, (0, 0)), (-np.inf, (4999, 5))):
        Xb = X.copy()
        Xb[where] = bad
        with pytest.raises(L.NonFiniteInput):
            ix.query(Xb, 3, transformed=True, check_finite=True)
        ix.query(Xb, 3, transformed=True)                 # without the flag the call does not judge
        for est in (EuclideanKNNRegressor(n_neighbors=3).fit(R, y), MSNRegressor(n_neighbors=3).fit(R, y),
                    RawKNNRegressor(n_neighbors=3).fit(R, y)):
            with pytest.raises(ValueError, match="NaN|infinity"):
                est.predict(Xb)
            with pytest.raises(ValueError, match="NaN|infinity"):
                est.kneighbors(Xb)
        assert np.isfinite(EuclideanKNNRegressor(n_neighbors=3).fit(R, y).predict(X)).all()


@pytest.mark.parametrize(("d_in", "d_out"), [(300, 20), (200, 200), (230, 230)])
def test_projection_of_shapes_beyond_shared_memory(d_in, d_out):
    """More raw features than a 128-row tile can stage (d_in > 225) and projectors beyond 227 KB
    (ADVICE round 1): the projection falls back to global-memory operands, same numbers."""
    from sknnr_b200._engine import KNNIndex

    rng = np.random.default_rng(d_in)
    n_ref = 400
    Xr = rng.standard_normal((n_ref, d_in)) * 3.0 + 10.0
    center, scale = Xr.mean(0), Xr.std(0, ddof=1)
    proj = rng.standard_normal((d_in, d_out)) / np.sqrt(d_in)
    Z = ((Xr - center) / scale) @ proj
    y = rng.standard_normal((n_ref, 2))
    ix = KNNIndex(Z, center, scale, proj, y)
    Q = rng.standard_normal((333, d_in)) * 3.0 + 10.0
    np.testing.assert_allclose(ix.transform(Q), ((Q - center) / scale) @ proj, rtol=1e-11, atol=1e-11)
    st = orc.FittedState("euclidean", fit_Z=Z, y=y, center=center, scale=scale, proj=proj)
    d_o, i_o = orc.kneighbors(st, Q, k=4)
    d_g, i_g, _ = ix.query(Q, 4)
    orc.assert_tie_aware_equal(d_g, i_g, d_o, i_o, rtol=1e-5, atol=1e-7 * float(np.sqrt((Z ** 2).sum(1).max())))
    Qb = Q.copy()
    Qb[17, d_in - 1] = np.nan
    with pytest.raises(L.NonFiniteInput):
        ix.query(Qb, 4, check_finite=True)


def test_hamming_non_integer_query_values_match_nothing():
    """scipy's hamming compares values ($SP/scipy/spatial/distance.py:1718-1723): a query value such as
    3.5 equals no node ID (ADVICE round 1: the int64 cast used to truncate it onto node 3)."""
    from sklearn.neighbors import KNeighborsRegressor

    from sknnr_b200 import RawKNNRegressor

    rng = np.random.default_rng(8)
    Rc = rng.integers(0, 6, size=(200, 12)).astype(np.float64)
    y = rng.standard_normal((200, 2))
    Q = Rc[rng.integers(0, 200, 50)].copy()
    Q[rng.random(Q.shape) < 0.25] += 0.5
    w = np.full(12, 1.0 / 12)            # (as RFNN passes them, ref:src/sknnr/_weighted_trees.py:139-140)
    ours = RawKNNRegressor(n_neighbors=4, metric="hamming", algorithm="brute", metric_params={"w": w}).fit(Rc, y)
    d_g, i_g = ours.kneighbors(Q, use_deterministic_ordering=False)
    ref = KNeighborsRegressor(n_neighbors=200, metric="hamming", algorithm="brute", metric_params={"w": w}).fit(Rc, y)
    d_all, i_all = ref.kneighbors(Q)
    full = np.empty_like(d_all)
    np.put_along_axis(full, i_all, d_all, axis=1)          # full[q, j] = scipy distance of plot j
    assert np.array_equal(d_g, np.take_along_axis(full, i_g, axis=1))
    order = np.lexsort((np.broadcast_to(np.arange(200), full.shape), full), axis=1)[:, :4]
    assert np.array_equal(i_g, order)


def test_raster_nodata_is_compared_in_the_band_dtype():
    """A float32 raster whose nodata literal is not representable in float32 (ADVICE round 1)."""
    from sknnr_b200._engine import KNNIndex

    rng = np.random.default_rng(9)
    R = rng.standard_normal((300, 4))
    y = rng.standard_normal((300, 2))
    ix = KNNIndex(R, None, None, None, y)
    img = rng.standard_normal((4, 1000)).astype(np.float32)
    nodata = -9999.9
    img[2, ::7] = nodata                       # stored as float32(-9999.9) != -9999.9
    _, idx, _, n_valid = ix.query_raster(img, 3, nodata=nodata)
    masked = (img == np.float32(nodata)).any(axis=0)
    assert n_valid == int((~masked).sum()) and masked.sum() > 0
    assert (idx[:, masked] == -1).all() and (idx[:, ~masked] >= 0).all()


@pytest.mark.parametrize(("k", "n_ref"), [(7, 20_000), (10, 20_000), (7, 2_000), (7, 5_000), (7, 9_000)])
def test_tensor_engine_certifies_nearly_every_row_and_stays_selected(k, n_ref):
    """Both stream layouts of the tensor engine (k <= 7: two streams, larger k: one) must certify
    all but a few per cent of the rows of an ordinary workload - otherwise the library demotes the
    index to the 10x slower FP32 engine - and a self-query (k + 1) must not spoil later calls."""
    from sknnr_b200._engine import KNNIndex

    rng = np.random.default_rng(12)
    R = rng.standard_normal((n_ref, 32))
    y = rng.standard_normal((n_ref, 2))
    Q = rng.standard_normal((40_000, 32))
    ix = KNNIndex(R, None, None, None, y)
    ix.query(None, k, exclude_self=True)
    st = ix.stats()
    assert st["engine"] == L.ENGINE_TENSOR and st["n_fallback"] < 0.05 * st["n_queries"], st
    for _ in range(2):
        ix.query(Q, k, transformed=True, weights="distance", with_pred=True)
        st = ix.stats()
        assert st["engine"] == L.ENGINE_TENSOR and st["n_fallback"] < 0.03 * st["n_queries"], st


@pytest.mark.parametrize(("k", "n_ref", "exclude_self"), [(5, 30_000, False), (7, 30_000, False), (12, 30_000, False),
                                                           (6, 8_000, True)])
def test_tensor_second_pass_equals_exact_engine_and_takes_most_of_its_rows(k, n_ref, exclude_self):
    """Stage 1b of the cascade (the tensor engine once more over its uncertified rows, each from the
    threshold the first pass proved sufficient) must change nothing but who certifies a row: results
    are bit-equal with the exhaustive float64 engine's, and it leaves the FP32 engine fewer rows than
    the first pass did."""
    from sknnr_b200._engine import KNNIndex

    rng = np.random.default_rng(31)
    R = rng.standard_normal((n_ref, 32))
    y = rng.standard_normal((n_ref, 3))
    Q = None if exclude_self else rng.standard_normal((150_000, 32))
    ix = KNNIndex(R, None, None, None, y)
    kw = dict(exclude_self=True) if exclude_self else dict(transformed=True)
    d1, i1, p1 = ix.query(Q, k, weights="distance", with_pred=True, **kw)
    c1 = ix.cascade_counts()
    assert ix.stats()["engine"] == L.ENGINE_TENSOR
    L.set_option("engine", L.ENGINE_EXACT)
    try:
        d0, i0, p0 = ix.query(Q, k, weights="distance", with_pred=True, **kw)
        assert ix.stats()["engine"] == L.ENGINE_EXACT
    finally:
        L.set_option("engine", L.ENGINE_AUTO)
    assert np.array_equal(i0, i1) and np.array_equal(d0, d1) and np.array_equal(p0, p1)
    assert c1["to_fp32"] <= c1["after_tensor"]
    if k + int(exclude_self) > 7:
        # one stream of 16 in the first pass already: a second pass would meet the same list, so there is none
        assert c1["to_fp32"] == c1["after_tensor"], c1
    elif c1["after_tensor"] >= 50:
        assert c1["to_fp32"] < 0.2 * c1["after_tensor"], c1


def test_joint_threshold_rank_adapts_to_crowded_neighbourhoods():
    """Few features and many plots put more references inside the FP16 error margin of the k-th
    neighbour than rank 10 of the two-stream layout's joint threshold allows for: after one call
    that saw > 4 % first-pass failures the index moves to rank 12.  Results do not depend on it."""
    from sknnr_b200._engine import KNNIndex

    rng = np.random.default_rng(5)
    R = rng.standard_normal((50_000, 8))
    Q = rng.standard_normal((60_000, 8))
    ix = KNNIndex(R, None, None, None, rng.standard_normal((50_000, 2)))
    d0, i0, _ = ix.query(Q, 7, transformed=True)
    c0 = ix.cascade_counts()
    d1, i1, _ = ix.query(Q, 7, transformed=True)
    c1 = ix.cascade_counts()
    assert ix.stats()["engine"] == L.ENGINE_TENSOR
    assert np.array_equal(i0, i1) and np.array_equal(d0, d1)
    assert c0["after_tensor"] > 0.04 * len(Q), c0
    assert c1["after_tensor"] < 0.6 * c0["after_tensor"], (c0, c1)


@pytest.mark.parametrize("pinned", [True, False])
def test_host_call_many_chunks_equal_one_chunk(pinned):
    """Host-buffer calls run as a three-stage pipeline (in-order H2D stream, compute stream, D2H
    stream; csrc/api.cu).  Many ramped chunks, more chunks than slots, a ragged last chunk, tensor
    and FP32 engines, a NaN row under the device-side finite check: all bit-equal with the same query
    made as a single chunk, and a second call on the same index reuses the slots cleanly."""
    from sknnr_b200._engine import KNNIndex, pinned_empty

    rng = np.random.default_rng(77)
    for n_ref, d in ((3000, 32), (600, 5)):          # tensor engine / FP32 engine
        R = rng.standard_normal((n_ref, d))
        y = rng.standard_normal((n_ref, 3))
        n_q = 70_001
        X = rng.standard_normal((n_q, d))
        if pinned:
            Xp = pinned_empty((n_q, d))
            Xp[:] = X
            X = Xp
        ix = KNNIndex(R, None, None, None, y)

        def run():
            out = None
            if pinned:
                out = (pinned_empty((n_q, 6)), pinned_empty((n_q, 6), np.int64), pinned_empty((n_q, 3)))
            got = ix.query(X, 6, transformed=True, weights="distance", with_pred=True, out=out)
            return [np.array(g) for g in got]

        one = run()                                  # default chunk_rows / stage_rows: a single chunk
        L.set_option("chunk_rows", 4096)
        L.set_option("stage_rows", 2048)
        try:
            many = run()
            for a, b in zip(one, many):
                assert np.array_equal(a, b)
            for a, b in zip(many, run()):
                assert np.array_equal(a, b)
            Xb = np.array(X)
            Xb[n_q - 3, 1] = np.nan
            with pytest.raises(L.NonFiniteInput):
                ix.query(Xb, 6, transformed=True, check_finite=True)
            again = ix.query(X, 6, transformed=True, weights="distance", with_pred=True)
            for a, b in zip(many, again):
                assert np.array_equal(a, b)
        finally:
            L.set_option("chunk_rows", 1 << 20)
            L.set_option("stage_rows", 1 << 19)
