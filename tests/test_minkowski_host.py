"""CPU tests of the Manhattan / Chebyshev searches: which metric arguments select them, which still
raise before any device call, and the C-ABI entry point that creates such an index."""

import ctypes

import numpy as np
import pytest
from sklearn.metrics import DistanceMetric
from sklearn.neighbors import KNeighborsRegressor


def _data(n=40, d=3, seed=0):
    rng = np.random.default_rng(seed)
    return rng.standard_normal((n, d)), rng.standard_normal((n, 2))


@pytest.mark.parametrize(("kw", "kind"), [
    ({}, "euclidean"),
    ({"metric": "euclidean"}, "euclidean"),
    ({"p": 1}, "manhattan"),
    ({"metric_params": {"p": 1}}, "manhattan"),
    ({"metric": "manhattan"}, "manhattan"),
    ({"metric": "cityblock"}, "manhattan"),
    ({"metric": "l1"}, "manhattan"),
    ({"p": np.inf}, "chebyshev"),
    ({"metric_params": {"p": np.inf}}, "chebyshev"),
    ({"metric": "chebyshev"}, "chebyshev"),
    ({"metric": "infinity"}, "chebyshev"),
    ({"metric": "hamming"}, "hamming"),
])
def test_effective_metric_selects_the_search(kw, kind):
    from sknnr_b200 import RawKNNRegressor

    X, y = _data()
    est = RawKNNRegressor(n_neighbors=3, **kw)
    KNeighborsRegressor.fit(est, X, y)   # scikit-learn's own metric resolution, no device involved
    assert est._metric_kind() == kind


@pytest.mark.parametrize("kw", [
    {"p": 3},
    {"p": 1, "metric_params": {"w": np.linspace(0.5, 1.5, 3)}},
    {"p": np.inf, "metric_params": {"w": np.linspace(0.5, 1.5, 3)}},
    {"metric": "cosine"},
    {"metric": "l2"},
    {"metric": lambda a, b: float(np.abs(a - b).sum())},
])
def test_uncovered_metrics_raise_from_fit_before_any_device_call(kw):
    """The index is built lazily by the self-query at the end of fit; NotImplementedError comes
    from the metric check in front of it (a device call without a GPU would raise SknnrError)."""
    from sknnr_b200 import RawKNNRegressor

    X, y = _data()
    with pytest.raises(NotImplementedError, match="Manhattan, Chebyshev"):
        RawKNNRegressor(n_neighbors=3, algorithm="brute", **kw).fit(X, y)


def test_create_metric_export_rejects_an_unknown_metric():
    from sknnr_b200 import _lib as L

    lib = L.load()
    assert hasattr(lib, "sknnr_index_create_metric")
    assert L.METRICS == {"euclidean": 0, "manhattan": 1, "chebyshev": 2}
    fit = np.zeros((4, 2))
    h = ctypes.c_void_p(None)
    for code in (-1, 3, 99):
        rc = lib.sknnr_index_create_metric(fit.ctypes.data_as(ctypes.c_void_p), 4, 2, None, None, None, 2,
                                           None, 0, code, 0, ctypes.byref(h))
        assert rc == -1   # SKNNR_EINVAL, before any device is looked at
        assert "metric" in lib.sknnr_last_error().decode()
        assert not h.value


def test_knn_index_rejects_an_unknown_metric_name():
    from sknnr_b200._engine import KNNIndex

    with pytest.raises(ValueError, match="metric must be one of"):
        KNNIndex(np.zeros((4, 2)), metric="cosine")


@pytest.mark.parametrize("metric", ["manhattan", "chebyshev"])
def test_sequential_float64_distance_is_what_scikit_learn_computes(metric):
    """The device kernels restate ManhattanDistance64 / ChebyshevDistance64 as a left-to-right
    float64 sum (max) of |x_j - y_j|.  That loop, written out here, is bit-equal to scikit-learn's
    DistanceMetric (which its brute ArgKmin search runs); NumPy's pairwise `abs(...).sum()` is not."""
    rng = np.random.default_rng(3)
    Q = rng.standard_normal((50, 37)) * rng.uniform(1e-3, 1e5, 37) + 5e5
    R = rng.standard_normal((60, 37)) * rng.uniform(1e-3, 1e5, 37) + 5e5
    ref = DistanceMetric.get_metric(metric).pairwise(Q, R)
    mine = np.zeros((50, 60))
    for j in range(37):
        t = np.abs(Q[:, None, j] - R[None, :, j])
        mine = mine + t if metric == "manhattan" else np.fmax(mine, t)
    np.testing.assert_array_equal(mine, ref)
