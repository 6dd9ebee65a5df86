"""CPU tests of the host side: the C-ABI library loads and exports every declared symbol,
fit-side transformer math reproduces the reference's fitted state, node-code mapping, and the
estimator surface's error behaviour that must not need a device."""

import ctypes
import inspect
import os
import re

import numpy as np
import pytest
from sklearn.exceptions import NotFittedError

from tests.conftest import ROOT, load_golden


def test_library_exports_every_declared_symbol():
    import __graft_entry__ as ge

    ge.build()
    from sknnr_b200 import _lib as L

    header = open(os.path.join(ROOT, "include", "sknnr_b200.h")).read()
    declared = set(re.findall(r"\b(sknnr_[a-z0-9_]+)\s*\(", header))
    declared -= {"sknnr_index", "sknnr_stats", "sknnr_hamming_index"}
    assert declared == set(L.EXPORTS)
    lib = ctypes.CDLL(L.lib_path())
    for name in declared:
        assert hasattr(lib, name), name
    assert L.load().sknnr_abi_version() == L.ABI_VERSION
    assert ctypes.sizeof(L.Stats) == 56


def test_no_cpu_fallback_without_device():
    """On a box without a GPU every compute entry point fails loudly."""
    from sknnr_b200 import _lib as L
    from sknnr_b200._engine import HammingIndex, KNNIndex

    if L.device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(L.SknnrError, match="no CUDA device"):
        KNNIndex(np.zeros((4, 2)))
    with pytest.raises(L.SknnrError, match="no CUDA device"):
        HammingIndex(np.zeros((4, 2), dtype=np.uint16), np.ones(2))


def test_product_never_imports_the_oracle():
    import sknnr_b200

    pkg = os.path.dirname(sknnr_b200.__file__)
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("sknnr_oracle", "oracle") or f == "__never__", (dirpath, f)


@pytest.mark.parametrize(("name", "cls_name", "kw"), [
    ("euclidean", "StandardScalerWithDOF", {"ddof": 1}),
    ("mahalanobis", "MahalanobisTransformer", {}),
    ("msn", "CCorATransformer", {}),
    ("gnn", "CCATransformer", {}),
])
@pytest.mark.parametrize("comp", ["full", "reduced"])
def test_fit_side_state_matches_reference(name, cls_name, kw, comp):
    """Fit math (NumPy, cold path) must hand the device the same (centre, scale, projector) the
    reference's transformers hold (ref:src/sknnr/transformers/*.py fit methods)."""
    import sknnr_b200.transformers as T

    if comp == "reduced":
        if name not in ("msn", "gnn"):
            pytest.skip("no n_components")
        kw = dict(kw, n_components=3)
    g = load_golden(f"moscow_{name}_{comp}.npz")
    sp = load_golden("moscow_split.npz")
    t = getattr(T, cls_name)(**kw).fit(sp["X_train"], sp["y_train"])
    center, scale, proj, d_out = t._affine()
    for key, arr in (("state_center", center), ("state_scale", scale), ("state_proj", proj)):
        if arr is None:
            assert key not in g
        else:
            np.testing.assert_allclose(arr, g[key], rtol=1e-10, atol=1e-12)
    assert d_out == g["state_fit_Z"].shape[1]


def test_n_components_validation():
    from sknnr_b200.transformers import CCATransformer, CCorATransformer

    sp = load_golden("moscow_split.npz")
    for cls in (CCATransformer, CCorATransformer):
        with pytest.raises(ValueError, match="n_components=99 must be between"):
            cls(n_components=99).fit(sp["X_train"], sp["y_train"])
        t = cls(n_components=2).fit(sp["X_train"], sp["y_train"])
        assert t.n_components_ == 2 and len(t.get_feature_names_out()) == 2


def test_node_code_mapping():
    from sknnr_b200._base import _encode_nodes, _node_code_tables

    ref = np.array([[3, 100000], [7, 5], [3, 70000]])
    tables = _node_code_tables(ref)
    assert tables is not None
    enc = _encode_nodes(ref, tables)
    assert enc.dtype == np.uint16 and enc[0, 0] == enc[2, 0] != enc[1, 0]
    q = _encode_nodes(np.array([[7, 123456], [4, 5]]), tables)
    assert q[0, 0] == enc[1, 0] and q[0, 1] == 31743 and q[1, 0] == 31743 and q[1, 1] == enc[1, 1]
    small = np.array([[0, 5], [9, 2]])
    assert _node_code_tables(small) is None
    assert _encode_nodes(np.array([[40000, -1]]), None).tolist() == [[31743, 31743]]


def test_signatures_match_reference_surface():
    """Constructor signatures of ref:src/sknnr/_base.py:196-218,385-408 and _rfnn.py:154-214."""
    import sknnr_b200 as S

    base = ["n_neighbors", "weights", "algorithm", "leaf_size", "p", "metric", "metric_params", "n_jobs"]
    for cls in (S.EuclideanKNNRegressor, S.MahalanobisKNNRegressor):
        assert list(inspect.signature(cls).parameters) == base
    for cls in (S.MSNRegressor, S.GNNRegressor):
        assert list(inspect.signature(cls).parameters) == ["n_neighbors", "n_components"] + base[1:]
    rf = list(inspect.signature(S.RFNNRegressor).parameters)
    assert rf[0] == "n_estimators" and rf[-3:] == ["forest_weights", "n_neighbors", "weights"] and len(rf) == 24
    gb = list(inspect.signature(S.GBNNRegressor).parameters)   # ref:src/sknnr/_gbnn.py:160-193
    assert gb[:3] == ["loss_reg", "loss_clf", "learning_rate"] and len(gb) == 27
    assert gb[-5:] == ["forest_weights", "tree_weighting_method", "n_neighbors", "weights", "n_jobs"]
    kn = list(inspect.signature(S.RawKNNRegressor.kneighbors).parameters)
    assert kn == ["self", "X", "n_neighbors", "return_distance", "return_dataframe_index",
                  "use_deterministic_ordering"]
    assert S.RawKNNRegressor.DISTANCE_PRECISION_DECIMALS == 10
    for cls in (S.EuclideanKNNRegressor, S.MSNRegressor, S.RFNNRegressor, S.GBNNRegressor, S.RawKNNRegressor):
        est = cls()
        assert type(est)(**est.get_params()).get_params().keys() == est.get_params().keys()


@pytest.mark.parametrize("name", ["RawKNNRegressor", "EuclideanKNNRegressor", "MahalanobisKNNRegressor",
                                  "MSNRegressor", "GNNRegressor", "RFNNRegressor", "GBNNRegressor"])
def test_unfitted_estimators_raise(name):
    import sknnr_b200 as S

    X = np.zeros((3, 4))
    with pytest.raises(NotFittedError):
        getattr(S, name)().kneighbors(X)
    with pytest.raises(NotFittedError):
        getattr(S, name)().predict(X)


def test_gbnode_transformer_fit_side_matches_reference():
    """Fit side of GBNN (cold path, scikit-learn trains the boosted models): tree weights, trees per
    iteration, Hamming weights and the column order of ``transform`` equal the live reference's
    (ref:src/sknnr/transformers/_gbnode_transformer.py:20-56,288-310; _weighted_trees.py:65-98).
    The node IDs are checked with scikit-learn's own ``Tree.apply`` on the trees in ``_trees()``
    order - the device walk of the same arrays is a GPU test."""
    import pandas as pd
    import warnings

    from sknnr_b200._estimators import GBNNRegressor
    from sknnr_b200.transformers import GBNodeTransformer

    g = load_golden("moscow_gbnn.npz")
    sp = load_golden("moscow_split.npz")
    Xtr, ytr = sp["X_train"], sp["y_train"]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", FutureWarning)
        tr = GBNodeTransformer(random_state=42).fit(Xtr, ytr)
    assert tr.n_forests_ == ytr.shape[1] and tr.n_trees_per_iteration_ == [1] * ytr.shape[1]
    trees = tr._trees()
    ids = np.stack([t.apply(Xtr.astype(np.float32)) for t in trees], axis=1)
    if not np.array_equal(ids, g["ids_train"].astype(np.int64)):
        pytest.skip("scikit-learn grew different boosted trees than the golden generator's")
    np.testing.assert_allclose(np.hstack(tr.tree_weights_), g["tree_weights"], rtol=1e-12)
    assert list(tr.get_feature_names_out()[:2]) == ["gb0_tree0", "gb0_tree1"]

    # hamming_weights_ = tree weights x forest weights / trees per iteration, without a device
    est = GBNNRegressor(random_state=42)
    est.transformer_ = tr
    np.testing.assert_allclose(est._get_hamming_weights(), g["hamming_w"], rtol=1e-12)

    # mixed targets: one regression model + one 3-class classifier (3 trees per stage, class-major)
    y_fit = pd.DataFrame({"Total_BA": g["mixed_yfit_total_ba"], "MAX_SPECIES": g["mixed_yfit_max_species"]})
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", FutureWarning)
        trm = GBNodeTransformer(random_state=42).fit(Xtr, y_fit)
    assert trm.n_trees_per_iteration_ == [1, 3]
    assert trm.estimator_type_dict_ == {"Total_BA": "regression", "MAX_SPECIES": "classification"}
    ids = np.stack([t.apply(Xtr.astype(np.float32)) for t in trm._trees()], axis=1)
    if np.array_equal(ids, g["mixed_ids_train"].astype(np.int64)):
        np.testing.assert_allclose(np.hstack(trm.tree_weights_), g["mixed_tree_weights"], rtol=1e-12)
        est.transformer_ = trm
        np.testing.assert_allclose(est._get_hamming_weights(), g["mixed_hamming_w"], rtol=1e-12)
    assert trm.get_feature_names_out()[100] == "gb1_cls0_tree0"
    with pytest.raises(ValueError, match="tree_weighting_method"):
        GBNodeTransformer(tree_weighting_method="nope", n_estimators=2).fit(Xtr, ytr[:, :1])
    tu = GBNodeTransformer(tree_weighting_method="uniform", n_estimators=4).fit(Xtr, ytr[:, :2])
    assert all(np.array_equal(w, np.full(4, 0.25)) for w in tu.tree_weights_)



def test_device_cache_is_outside_the_estimator_and_dies_with_it():
    """Device handles are cached in a weakly keyed side table (sknnr_b200/_cache.py): nothing is
    added to the estimator's __dict__, clones and pickles never see the cache, entries vanish with
    their owner and can be dropped on refit."""
    import gc
    import pickle

    from sklearn.base import clone

    from sknnr_b200 import _cache
    from sknnr_b200.transformers import StandardScalerWithDOF

    t = StandardScalerWithDOF().fit(np.arange(12.0).reshape(4, 3))
    before = dict(t.__dict__)
    _cache.put(t, "projector", object())
    assert t.__dict__.keys() == before.keys()
    assert _cache.get(t, "projector") is not None
    assert _cache.get(clone(t), "projector") is None
    assert _cache.get(pickle.loads(pickle.dumps(t)), "projector") is None
    _cache.drop(t, "projector")
    assert _cache.get(t, "projector") is None
    _cache.put(t, "projector", object())
    n = len(_cache._CACHE)
    del t
    gc.collect()
    assert len(_cache._CACHE) == n - 1


def test_host_chunk_schedule_ramps_and_covers_every_row():
    """The chunk schedule of a host-buffer call (csrc/api.cu, next_chunk_rows): every row exactly once,
    no chunk above the chunk size, a 1/4 - 1/2 ramp at both ends from four chunks' worth of rows up, and
    no sliver chunk in the middle of a large call."""
    from sknnr_b200 import _lib as L

    for chunk in (1024, 4096, 1 << 19, 1 << 20):
        for n_q in (0, 1, 255, 256, 1000, chunk - 1, chunk, chunk + 1, 4 * chunk - 1, 4 * chunk, 4 * chunk + 1,
                    5 * chunk + 37, 10_000_000, 9 * chunk + 3 * chunk // 4 + 5, 70_001, 12_345_678):
            plan = L.host_chunk_plan(n_q, chunk)
            assert sum(plan) == n_q, (n_q, chunk, plan)
            assert all(0 < r <= chunk for r in plan), (n_q, chunk, plan)
            if n_q >= 4 * chunk:
                assert plan[0] == chunk // 4 and plan[1] == chunk // 2, (n_q, chunk, plan[:3])
                assert plan[-1] <= chunk // 4 and plan[-2] <= chunk // 2 + chunk // 4, (n_q, chunk, plan[-3:])
                assert min(plan[:-1]) >= chunk // 4, (n_q, chunk, plan)
                assert all(r == chunk for r in plan[2:-3]), (n_q, chunk, plan)
            elif n_q > 0:
                assert plan == [min(chunk, n_q - i) for i in range(0, n_q, chunk)], (n_q, chunk, plan)
    assert L.host_chunk_plan(10_000_000, 1 << 20) == [262144, 524288] + [1 << 20] * 8 + [562816, 262144]
    with pytest.raises(ValueError):
        L.host_chunk_plan(-1, 1 << 20)


def test_set_option_accepts_the_kept_names_and_rejects_the_retired_ones():
    """The options that only chose between a measured winner and a measured loser are gone from
    sknnr_set_option: their names are unknown options now.  The kept ones still take a value."""
    from sknnr_b200 import _lib as L

    for name in ("host_pipeline", "tail_priority", "tc_retry", "tail_spread", "host_nt", "simt_min_rows",
                 "host_threads"):
        with pytest.raises(ValueError, match="unknown option"):
            L.set_option(name, 1)
    # (a value other than the default, then the default again)
    kept = {"engine": (3, 0), "chunk_rows": (4096, 1 << 20), "timing": (1, 0), "kc": (8, 16), "tc_streams": (1, 0),
            "tc_seed_stride": (2, 4), "tc_debug": (1, 0), "host_slots": (2, 8), "stage_rows": (2048, 1 << 19)}
    try:
        for name, (value, _) in kept.items():
            L.set_option(name, value)
    finally:
        for name, (_, default) in kept.items():
            L.set_option(name, default)
