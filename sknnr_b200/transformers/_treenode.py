"""Tree-node transformers: one forest per target, ``transform`` returns the terminal-node ID of
every tree (mirrors ref:src/sknnr/transformers/_tree_node_transformer.py).  Forest TRAINING is
scikit-learn's (out of the hot-path scope); ``transform`` walks the fitted trees on the GPU
(``ForestIndex``: scikit-learn's ``tree_`` arrays flattened, ``Tree._apply_dense`` semantics
replicated bit for bit - scope row f1), and the RFNN / GBNN regressors query raw features ->
forest walk -> Hamming search without the node IDs ever leaving the device.
"""

from __future__ import annotations

from abc import ABC, abstractmethod
from collections import Counter

import numpy as np
from sklearn.base import BaseEstimator, TransformerMixin
from sklearn.utils.validation import check_array, check_is_fitted, validate_data

from .. import _cache
from .._lib import x_dtype_code


def _is_nan_like(v) -> bool:
    return v is None or (isinstance(v, float) and np.isnan(v)) or type(v).__name__ == "NAType"


def _target_names(y) -> list:
    if hasattr(y, "columns") and hasattr(y, "dtypes"):
        return list(y.columns)
    if hasattr(y, "name") and hasattr(y, "dtype") and not isinstance(y, np.ndarray):
        return ["0"] if y.name is None else [y.name]
    arr = np.asarray(y, dtype=object)
    return [str(i) for i in range(1 if arr.ndim == 1 else arr.shape[1])]


def _target_dtypes(y) -> list:
    """Smallest NumPy dtype holding each target column; pandas categoricals keep their tag."""
    arr = np.asarray(y, dtype=object)
    if arr.ndim == 1:
        arr = arr.reshape(-1, 1)
    promoted = [np.asarray(arr[:, i].tolist()).dtype for i in range(arr.shape[1])]
    native = None
    if hasattr(y, "columns") and hasattr(y, "dtypes"):
        native = list(getattr(y.dtypes, "values", y.dtypes))
    elif hasattr(y, "name") and hasattr(y, "dtype") and not isinstance(y, np.ndarray):
        native = [y.dtype]
    if native is None:
        return promoted
    return [n if str(n) == "category" else p for p, n in zip(promoted, native)]


def _is_numeric(dt) -> bool:
    try:
        return bool(np.issubdtype(np.dtype(dt), np.number))
    except TypeError:
        kind = getattr(dt, "kind", None)
        if kind:
            return kind in "iuf"
        raise TypeError(f"Unsupported type {dt}") from None


class TreeNodeTransformer(TransformerMixin, BaseEstimator, ABC):
    """Shared fit / transform of the tree-node transformers
    (ref:src/sknnr/transformers/_tree_node_transformer.py:38-211)."""

    # -- fit (cold path) ----------------------------------------------------------------
    def _prepare_targets(self, y, info):
        arr = np.asarray(y, dtype=object)
        if arr.ndim == 1:
            arr = arr.reshape(-1, 1)
        out = []
        for i, (name, dt) in enumerate(info.items()):
            col = arr[:, i]
            if any(_is_nan_like(v) for v in col):
                raise ValueError(f"Target {name} has NaN-like elements.")
            if str(dt) == "category":
                col = np.asarray(col.tolist())
            else:
                try:
                    npdt = np.dtype(dt)
                except TypeError:
                    npdt = None
                if npdt is not None:
                    if np.issubdtype(npdt, np.str_):
                        odd = {type(v) for v in col if not np.issubdtype(type(v), np.str_)}
                        if odd:
                            raise ValueError(
                                f"Target {name} has non-string types ({odd}) that cannot be "
                                f"safely converted to a string dtype ({npdt}).")
                    col = col.astype(npdt)
            out.append(check_array(col, ensure_all_finite=True, dtype=None, ensure_2d=False, estimator=self))
        return out

    def _fit(self, X, y, make_regressor, make_classifier):
        _cache.drop(self)        # device copies of a previous fit's trees
        X_arr = validate_data(self, X=X, reset=True)
        if y is None:
            raise ValueError(f"{type(self).__name__} requires y to be passed, but the target y is None.")
        names = _target_names(y)
        if len(set(names)) != len(names):
            dup = [n for n, c in Counter(names).items() if c > 1]
            raise ValueError(f"Duplicate feature names found: {dup}.")
        info = dict(zip(names, _target_dtypes(y)))
        targets = self._prepare_targets(y, info)
        self.estimator_type_dict_ = {
            n: ("regression" if _is_numeric(dt) else "classification") for n, dt in info.items()}
        kinds = list(self.estimator_type_dict_.values())
        self.estimators_ = [
            (make_regressor() if kind == "regression" else make_classifier()).fit(X_arr, target)
            for kind, target in zip(kinds, targets)]
        self.n_forests_ = len(self.estimators_)
        self.n_trees_per_iteration_ = self._set_n_trees_per_iteration()
        self.tree_weights_ = self._set_tree_weights(X_arr, targets)
        return self

    @abstractmethod
    def _set_n_trees_per_iteration(self): ...

    @abstractmethod
    def _set_tree_weights(self, X, y): ...

    @abstractmethod
    def _trees(self):
        """Fitted scikit-learn ``Tree`` objects in ``transform``'s column order."""

    @abstractmethod
    def fit(self, X, y): ...

    # -- transform ----------------------------------------------------------------------
    def _forest_index(self, node_code_tables=None, devices=None):
        """Device copy of the trees (a cache outside ``__dict__``: never pickled, rebuilt on demand).
        A copy made with ``node_code_tables`` also serves the fused Hamming query of the estimator
        that owns them.  ``devices``: one copy per listed GPU (for a multi-device index)."""
        from .._engine import ForestIndex

        if devices is not None:
            from .._sharding import _PerDevice

            return _PerDevice(self._forest_index_on(node_code_tables, d) for d in devices)
        return self._forest_index_on(node_code_tables, None)

    def _forest_index_on(self, node_code_tables, device):
        from .._engine import ForestIndex

        key = ("forest_coded" if node_code_tables is not None else "forest_plain") + ("" if device is None else f"@{device}")
        coded = node_code_tables is not None
        fx = _cache.get(self, key)
        if fx is not None and coded and _cache.get(self, "tables_id") != id(node_code_tables):
            fx = None   # the owning estimator rebuilt its code tables (refit)
        if fx is None:
            fx = _cache.put(self, key, ForestIndex(self._trees(), self.n_features_in_, node_code_tables, device=device))
            if coded:
                _cache.put(self, "tables_id", id(node_code_tables))
        return fx

    def _validate_query(self, X):
        """Input validation of ``transform`` (feature names, shape, NaN) plus scikit-learn's own
        float32 check of ``est.apply`` ($SP/sklearn/tree/_classes.py _validate_X_predict)."""
        check_is_fitted(self)
        X_arr = validate_data(self, X=X, reset=False, ensure_min_features=1, ensure_min_samples=1)
        if X_arr.dtype.kind in "iu" and x_dtype_code(X_arr) is not None:
            return X_arr   # uint8 ... int64: no NaN / inf to find, the device reads the array as it is
        with np.errstate(over="ignore"):
            X32 = np.asarray(X_arr, dtype=np.float32)
        check_array(X32, ensure_all_finite=True, estimator=self)
        return X_arr

    def transform(self, X):
        X_arr = self._validate_query(X)
        return self._forest_index().apply(X_arr)

    def fit_transform(self, X, y):
        return self.fit(X, y).transform(X)

    def __sklearn_tags__(self):
        tags = super().__sklearn_tags__()
        tags.target_tags.required = True
        tags.transformer_tags.preserves_dtype = ["int64"]
        return tags
