"""Estimator surface of the drop-in: the same classes, constructor signatures, fitted
attributes and ``kneighbors`` keywords as ref:src/sknnr/_base.py, with the three seams

    S1  ref:src/sknnr/_base.py:162-175  (sklearn kneighbors + deterministic re-ordering)
    S2  ref:src/sknnr/_base.py:236-239  (_transform_X)
    S3  ref:src/sknnr/_base.py:346-352  (predict / score)

routed to the CUDA library through ``_engine`` (one fused device call when X is given).
Validation, NotFitted / ValueError behaviour and feature-name warnings stay in Python and use
scikit-learn's own helpers.  There is no CPU fallback: a search always runs on the device.
"""

from __future__ import annotations

import numbers
from abc import ABC, abstractmethod

import numpy as np
import scipy.sparse as sp
from sklearn.base import BaseEstimator
from sklearn.metrics import r2_score
from sklearn.neighbors import KNeighborsRegressor
from sklearn.utils import assert_all_finite
from sklearn.utils.validation import _is_arraylike, check_is_fitted, validate_data

from . import _lib as L
from ._engine import HammingIndex, KNNIndex
from ._sharding import MultiDeviceIndex, devices_from_env


class DFIndexCrosswalkMixin:
    """Crosswalk array indices to dataframe indexes (ref:src/sknnr/_base.py:23-30)."""

    def _set_dataframe_index_in(self, X) -> None:
        index = getattr(X, "index", None)
        if _is_arraylike(index):
            self.dataframe_index_in_ = np.asarray(index)


class IndependentPredictorMixin:
    """Leave-self-out prediction and score on the training plots
    (ref:src/sknnr/_base.py:33-40).  The reference runs the n_ref x n_ref self-query twice
    (predict(None), then score(None)); here it runs once and R^2 is derived from it."""

    def _set_independent_prediction_attributes(self, y) -> None:
        self.independent_prediction_ = self.predict(X=None)
        self.independent_score_ = float(r2_score(y, self.independent_prediction_))


class WideCodes:
    """Code tables of a wide Hamming index (a tree with more than ``L.MAX_CODE`` distinct node IDs):
    exact 32-bit codes, ``L.WIDE_NONE`` for a value that matches nothing.  ``tables`` None: every
    node ID is its own code (a forest's node IDs, which the device walk emits as they are); else,
    per tree, the sorted node IDs that map to codes 0, 1, ..."""

    def __init__(self, tables):
        self.tables = tables


def _node_code_tables(ref_ids: np.ndarray, ids_are_codes: bool = False):
    """Map each tree's node IDs to dense 16-bit codes (only equality matters): None when the IDs
    already fit, else the per-tree tables of sorted IDs.  When a tree has more distinct IDs than
    16-bit codes reach, a :class:`WideCodes` (``ids_are_codes``: the IDs are a forest's node IDs
    and serve as their own codes)."""
    if ref_ids.min() >= 0 and ref_ids.max() < L.MAX_CODE:
        return None  # IDs already fit: identity mapping
    tables = [np.unique(ref_ids[:, t]) for t in range(ref_ids.shape[1])]
    if max(len(u) for u in tables) <= L.MAX_CODE:
        return tables
    if ids_are_codes and ref_ids.min() >= 0 and ref_ids.max() < L.WIDE_NONE:
        return WideCodes(None)
    return WideCodes(tables)


def _forest_tables(tables):
    """The code tables a device forest needs for an index coded by ``tables``: none for a wide
    index, whose forest queries carry the node IDs themselves."""
    return None if isinstance(tables, WideCodes) else tables


def _encode_nodes(ids: np.ndarray, tables) -> np.ndarray:
    ids = np.asarray(ids)
    if isinstance(tables, WideCodes):
        return _encode_wide(ids, tables.tables)
    if tables is None:
        bad = (ids < 0) | (ids >= L.MAX_CODE)
        out = ids.astype(np.uint16)
        out[bad] = L.MAX_CODE  # unseen value: matches nothing
        return out
    out = np.empty(ids.shape, dtype=np.uint16)
    for t, u in enumerate(tables):
        pos = np.searchsorted(u, ids[:, t])
        pos_c = np.minimum(pos, len(u) - 1)
        hit = u[pos_c] == ids[:, t]
        out[:, t] = np.where(hit, pos_c, L.MAX_CODE)
    return out


def _encode_wide(ids: np.ndarray, tables) -> np.ndarray:
    """Exact u32 codes of a wide index (``WideCodes.tables``); unseen values match nothing."""
    if tables is None:
        out = np.full(ids.shape, L.WIDE_NONE, dtype=np.uint32)
        ok = (ids >= 0) & (ids < L.WIDE_NONE)
        out[ok] = ids[ok]
        return out
    out = np.empty(ids.shape, dtype=np.uint32)
    for t, u in enumerate(tables):
        pos = np.searchsorted(u, ids[:, t])
        pos_c = np.minimum(pos, len(u) - 1)
        hit = u[pos_c] == ids[:, t]
        out[:, t] = np.where(hit, pos_c, L.WIDE_NONE)
    return out


class RawKNNRegressor(DFIndexCrosswalkMixin, IndependentPredictorMixin, KNeighborsRegressor):
    """``KNeighborsRegressor`` with independent prediction / score, dataframe-index crosswalk
    and deterministic neighbour ordering (mirrors ref:src/sknnr/_base.py:43-182), searching on
    the B200.  Supported searches: brute Euclidean (``metric='minkowski', p=2`` or
    ``'euclidean'``), Manhattan (``p=1``, ``'manhattan'``, ``'cityblock'``, ``'l1'``), Chebyshev
    (``p=np.inf``, ``'chebyshev'``, ``'infinity'``) and weighted Hamming (``metric='hamming'``);
    ``algorithm`` is accepted for signature compatibility and the search is always exhaustive.
    """

    DISTANCE_PRECISION_DECIMALS = 10

    # -- device state (a cache: never pickled, rebuilt from the NumPy attributes) ----------
    def _drop_device_index(self):
        self.__dict__.pop("_device_index", None)
        self.__dict__.pop("_node_tables", None)

    def __getstate__(self):
        state = super().__getstate__()
        state.pop("_device_index", None)
        return state

    # effective_metric_ -> search: scikit-learn maps minkowski p=1 / p=inf without weights to
    # "manhattan" / "chebyshev", and its brute search runs the same distance for the aliases
    _KINDS = {"euclidean": "euclidean", "manhattan": "manhattan", "cityblock": "manhattan",
              "l1": "manhattan", "chebyshev": "chebyshev", "infinity": "chebyshev", "hamming": "hamming"}

    def _metric_kind(self) -> str:
        m = self.effective_metric_
        kind = self._KINDS.get(m) if isinstance(m, str) else None
        if kind in ("manhattan", "chebyshev") and self.effective_metric_params_:
            kind = None   # (a parametrised variant of the distance)
        if kind is None:
            raise NotImplementedError(
                f"sknnr_b200 covers the brute Euclidean, Manhattan, Chebyshev and Hamming searches; "
                f"metric={self.metric!r} (effective {m!r}) has no CUDA path and there is no CPU fallback")
        return kind

    def _get_index(self):
        ix = self.__dict__.get("_device_index")
        if ix is not None:
            return ix
        y = self._y
        devices = devices_from_env()    # SKNNR_B200_DEVICES: the same fitted state on several GPUs
        kind = self._metric_kind()
        if kind != "hamming":
            center, scale, proj = self.__dict__.get("_projection", (None, None, None))
            make = lambda dev: KNNIndex(self._fit_X, center, scale, proj, y, device=dev, metric=kind)  # noqa: E731
            ix = MultiDeviceIndex(make, devices) if devices else make(None)
        else:
            ref_ids = np.asarray(self._fit_X)
            if not np.all(ref_ids == np.floor(ref_ids)):
                raise NotImplementedError("the Hamming path expects integer node IDs")
            ref_ids = ref_ids.astype(np.int64)
            tables = _node_code_tables(ref_ids, ids_are_codes=self.__dict__.get("_forest_node_ids", False))
            self.__dict__["_node_tables"] = tables
            w = (self.effective_metric_params_ or {}).get("w")
            if w is None:
                w = np.full(ref_ids.shape[1], 1.0 / ref_ids.shape[1])
            codes = _encode_nodes(ref_ids, tables)
            make = lambda dev: HammingIndex(codes, w, y, device=dev)  # noqa: E731
            ix = MultiDeviceIndex(make, devices) if devices else make(None)
        self.__dict__["_device_index"] = ix
        return ix

    # -- fit ---------------------------------------------------------------------------
    def fit(self, X, y):
        if sp.issparse(X):   # dense searches only (input tag sparse = False), scikit-learn's wording
            raise TypeError("Sparse data was passed for X, but dense data is required. "
                            "Use '.toarray()' to convert to a dense numpy array.")
        self._set_dataframe_index_in(X)
        self._drop_device_index()
        super().fit(X, y)
        self._set_independent_prediction_attributes(y)
        return self

    # -- search ------------------------------------------------------------------------
    def _check_k(self, n_neighbors, query_is_train, n_queries):
        if n_neighbors is None:
            n_neighbors = self.n_neighbors
        elif not isinstance(n_neighbors, numbers.Integral):
            raise TypeError("n_neighbors does not take %s value, enter integer value" % type(n_neighbors))
        elif n_neighbors <= 0:
            raise ValueError("Expected n_neighbors > 0. Got %d" % n_neighbors)
        n_fit = self.n_samples_fit_
        if n_neighbors + (1 if query_is_train else 0) > n_fit:
            ineq = "n_neighbors < n_samples_fit" if query_is_train else "n_neighbors <= n_samples_fit"
            raise ValueError(
                f"Expected {ineq}, but n_neighbors = {n_neighbors}, n_samples_fit = {n_fit}, "
                f"n_samples = {n_queries}")
        return int(n_neighbors)

    def _search(self, X, n_neighbors, deterministic, *, raw=False, weights=None, with_pred=False,
                return_distance=True, forest=None, on_nonfinite=None):
        """One device call.  ``raw=True``: X holds untransformed features and the projection is
        fused in front (S2+S1[+S3]); ``forest`` (a fitted tree-node transformer): X holds validated
        raw features and the forest walk is fused in front of the Hamming search; otherwise X is
        already in the estimator's space."""
        check_is_fitted(self)
        ix = self._get_index()
        query_is_train = X is None
        kw = dict(deterministic=deterministic, decimals=self.DISTANCE_PRECISION_DECIMALS,
                  weights=weights, with_pred=with_pred, return_distance=return_distance)
        if query_is_train:
            k = self._check_k(n_neighbors, True, self.n_samples_fit_)
            return ix.query(None, k, exclude_self=True, **kw)
        if forest is not None:
            k = self._check_k(n_neighbors, False, X.shape[0])
            fx = forest._forest_index(_forest_tables(self.__dict__.get("_node_tables")),
                                      devices=getattr(ix, "devices", None))
            return ix.query_forest(fx, X, k, **kw)
        hamming = hasattr(ix, "n_trees")
        if not raw:
            # (Euclidean searches: the finite check runs on the device, see below)
            X = validate_data(self, X, ensure_all_finite=hamming, accept_sparse=False, reset=False, order="C")
        k = self._check_k(n_neighbors, False, X.shape[0])
        if hamming:
            Xa = np.asarray(X)
            codes = _encode_nodes(Xa.astype(np.int64), self._node_tables)
            if Xa.dtype.kind == "f":
                # scipy's hamming compares values, not truncated integers: a non-integer query
                # value equals no node ID ($SP/scipy/spatial/distance.py:1718-1723)
                codes[Xa != np.floor(Xa)] = L.WIDE_NONE if codes.dtype == np.uint32 else L.MAX_CODE
            return ix.query(codes, k, **kw)
        # The reference rejects non-finite values when the regressor validates the (transformed)
        # array ($SP/sklearn/neighbors/_base.py:831-838).  The projection kernel reads every query
        # value anyway and an affine map keeps NaN / inf, so the device does the check and the host
        # pass over the array only happens to word the error.
        try:
            return ix.query(X, k, transformed=not raw, check_finite=True, **kw)
        except L.NonFiniteInput:
            if on_nonfinite is not None:
                on_nonfinite()
            if not raw:
                validate_data(self, X, ensure_all_finite=True, accept_sparse=False, reset=False, order="C")
            assert_all_finite(X)
            raise

    def kneighbors(self, X=None, n_neighbors=None, return_distance=True,
                   return_dataframe_index=False, use_deterministic_ordering=True):
        """Same contract as ref:src/sknnr/_base.py:111-182."""
        dist, idx, _ = self._search(X, n_neighbors, use_deterministic_ordering,
                                    return_distance=return_distance)
        return self._finish_kneighbors(dist, idx, return_distance, return_dataframe_index)

    def _finish_kneighbors(self, dist, idx, return_distance, return_dataframe_index):
        if return_dataframe_index:
            msg = "Dataframe indexes can only be returned when fitted with a dataframe."
            check_is_fitted(self, "dataframe_index_in_", msg=msg)
            idx = self.dataframe_index_in_[idx]
        return (dist, idx) if return_distance else idx

    # -- predict -----------------------------------------------------------------------
    def _predict_impl(self, X, raw, forest=None, on_nonfinite=None):
        w = self.weights
        if w in (None, "uniform", "distance"):
            _, _, pred = self._search(X, None, True, raw=raw, weights=w, with_pred=True,
                                      return_distance=False, forest=forest, on_nonfinite=on_nonfinite)
        else:  # callable: evaluated by Python on the distances, averaged on the device
            dist, idx, _ = self._search(X, None, True, raw=raw, forest=forest, on_nonfinite=on_nonfinite)
            pred = self._get_index().weighted_average(idx, np.asarray(w(dist), dtype=np.float64))
        if self._y.ndim == 1:
            pred = pred.ravel()
        return pred

    def predict(self, X):
        """$SP/sklearn/neighbors/_regression.py:229-273 on the device."""
        return self._predict_impl(X, raw=False)

    def __sklearn_tags__(self):
        tags = super().__sklearn_tags__()
        tags.input_tags.sparse = False
        return tags


class TransformedKNeighborsRegressor(BaseEstimator, ABC):
    """kNN regressors that search in a transformed feature space
    (mirrors ref:src/sknnr/_base.py:185-358).  Not instantiated directly."""

    def __init__(self, n_neighbors=5, *, weights="uniform", algorithm="auto", leaf_size=30, p=2,
                 metric="minkowski", metric_params=None, n_jobs=None):
        self.n_neighbors = n_neighbors
        self.weights = weights
        self.algorithm = algorithm
        self.leaf_size = leaf_size
        self.p = p
        self.metric = metric
        self.metric_params = metric_params
        self.n_jobs = n_jobs

    @abstractmethod
    def _get_transformer(self): ...

    def _set_fitted_transformer(self, X, y) -> None:
        self.transformer_ = self._get_transformer().fit(X, y)

    def _get_additional_regressor_init_kwargs(self) -> dict:
        return {}

    def _transform_X(self, X):
        check_is_fitted(self, "transformer_")
        return self.transformer_.transform(X) if X is not None else X

    def _fusable(self) -> bool:
        """True when the transformer is an affine map the device fuses in front of the search."""
        return hasattr(self.transformer_, "_affine")

    def _forest_fusable(self) -> bool:
        """True when the transformer is a fitted forest the device walks in front of the Hamming
        search (raw features -> node codes -> neighbours in one call)."""
        return hasattr(self.transformer_, "_forest_index") and self.regressor_._metric_kind() == "hamming"

    def fit(self, X, y):
        validate_data(self, X=X, y=y, ensure_all_finite=True, multi_output=True)
        self._set_fitted_transformer(X, y)
        X_transformed = self.transformer_.transform(X)

        kwargs = dict(n_neighbors=self.n_neighbors, weights=self.weights, algorithm=self.algorithm,
                      leaf_size=self.leaf_size, p=self.p, metric=self.metric,
                      metric_params=self.metric_params, n_jobs=self.n_jobs)
        kwargs.update(self._get_additional_regressor_init_kwargs())
        self.regressor_ = RawKNNRegressor(**kwargs)
        if self._fusable():
            center, scale, proj, _ = self.transformer_._affine()
            self.regressor_._projection = (center, scale, proj)
        if hasattr(self.transformer_, "_forest_index"):
            # (node IDs the device forest walk reproduces: a wide index keeps them as its codes)
            self.regressor_._forest_node_ids = True
        self.regressor_.fit(X_transformed, y)
        self.regressor_._set_dataframe_index_in(X)

        self.n_features_in_ = self.regressor_.n_features_in_
        self.independent_prediction_ = self.regressor_.independent_prediction_
        self.independent_score_ = self.regressor_.independent_score_
        if hasattr(self.regressor_, "dataframe_index_in_"):
            self.dataframe_index_in_ = self.regressor_.dataframe_index_in_
        return self

    def _validated_raw(self, X, finite=True):
        """Run the transformer's own input validation (feature-name warnings, dtype, NaN and
        shape errors exactly as ``transform`` would raise them) and hand back the raw array.
        ``finite=False`` leaves the scan for NaN / inf to the device (fused affine path); when the
        device reports one, the full validation is repeated to raise the transformer's own error."""
        check_is_fitted(self, "transformer_")
        if finite:
            return self.transformer_._validate_query(X)
        return self.transformer_._validate_query(X, finite=False)

    def kneighbors(self, X=None, n_neighbors=None, return_distance=True,
                   return_dataframe_index=False, use_deterministic_ordering=True):
        """Same contract as ref:src/sknnr/_base.py:285-344."""
        check_is_fitted(self, "transformer_")
        reg = self.regressor_
        if X is not None and self._forest_fusable():
            dist, idx, _ = reg._search(self._validated_raw(X), n_neighbors, use_deterministic_ordering,
                                       forest=self.transformer_, return_distance=return_distance)
            return reg._finish_kneighbors(dist, idx, return_distance, return_dataframe_index)
        if X is None or not self._fusable():
            return reg.kneighbors(
                X=self._transform_X(X), n_neighbors=n_neighbors, return_distance=return_distance,
                return_dataframe_index=return_dataframe_index,
                use_deterministic_ordering=use_deterministic_ordering)
        dist, idx, _ = reg._search(self._validated_raw(X, finite=False), n_neighbors, use_deterministic_ordering,
                                   raw=True, return_distance=return_distance,
                                   on_nonfinite=lambda: self._validated_raw(X))
        return reg._finish_kneighbors(dist, idx, return_distance, return_dataframe_index)

    def predict(self, X):
        check_is_fitted(self, "transformer_")
        if X is not None and self._forest_fusable():
            return self.regressor_._predict_impl(self._validated_raw(X), raw=False, forest=self.transformer_)
        if X is None or not self._fusable():
            return self.regressor_.predict(self._transform_X(X))
        return self.regressor_._predict_impl(self._validated_raw(X, finite=False), raw=True,
                                             on_nonfinite=lambda: self._validated_raw(X))

    def score(self, X, y):
        return float(r2_score(y, self.predict(X)))

    def __sklearn_tags__(self):
        tags = super().__sklearn_tags__()
        tags.input_tags.sparse = False
        return tags


class YFitMixin(TransformedKNeighborsRegressor):
    """Optional ``y_fit`` used to fit the transformer (ref:src/sknnr/_base.py:361-374)."""

    def _set_fitted_transformer(self, X, y) -> None:
        y_fit = self.y_fit_ if self.y_fit_ is not None else y
        self.transformer_ = self._get_transformer().fit(X, y_fit)

    def fit(self, X, y, y_fit=None):
        self.y_fit_ = y_fit
        return super().fit(X, y)


class OrdinationKNeighborsRegressor(TransformedKNeighborsRegressor, ABC):
    """Transformed regressors with dimensionality reduction (ref:src/sknnr/_base.py:377-408)."""

    def __init__(self, n_neighbors=5, *, n_components=None, weights="uniform", algorithm="auto",
                 leaf_size=30, p=2, metric="minkowski", metric_params=None, n_jobs=None):
        super().__init__(n_neighbors=n_neighbors, weights=weights, algorithm=algorithm,
                         leaf_size=leaf_size, p=p, metric=metric, metric_params=metric_params,
                         n_jobs=n_jobs)
        self.n_components = n_components
