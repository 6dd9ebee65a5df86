"""Transformer building blocks: the ddof-aware scaler, the n_components mixin and the device
projection shared by the four float transformers."""

from __future__ import annotations

import numpy as np
from sklearn.preprocessing import StandardScaler
from sklearn.utils.validation import FLOAT_DTYPES, check_is_fitted, validate_data

from .. import _cache
from .._lib import NATIVE_INT_DTYPES

# dtypes a query keeps through validation: the floats scikit-learn keeps, plus the integer types the
# device reads as they are (any other dtype becomes float64, the first entry, as before)
QUERY_DTYPES = FLOAT_DTYPES + NATIVE_INT_DTYPES


class DeviceProjectionMixin:
    """``transform`` of every float transformer is one affine map
    ``Z = ((X - center) / scale) @ proj`` evaluated by the CUDA projection kernel
    (csrc/project.cu, C-ABI ``sknnr_transform``).  Subclasses return the three arrays."""

    def _affine(self):  # -> (center | None, scale | None, proj | None, d_out)
        raise NotImplementedError

    def _projector_handle(self):
        h = _cache.get(self, "projector")
        if h is None:
            from .._engine import KNNIndex

            center, scale, proj, d_out = self._affine()
            h = _cache.put(self, "projector", KNNIndex(np.zeros((1, d_out)), center, scale, proj))
        return h

    def _device_transform(self, X_arr):
        if self._affine()[3] == 0:   # n_components=0: nothing to compute (the reference returns [n, 0] too)
            return np.empty((np.asarray(X_arr).shape[0], 0), dtype=np.float64)
        return self._projector_handle().transform(X_arr)

    def _drop_device_state(self):
        _cache.drop(self)


class StandardScalerWithDOF(DeviceProjectionMixin, StandardScaler):
    """``StandardScaler`` whose ``scale_`` is the standard deviation with ``ddof`` degrees of
    freedom (mirrors ref:src/sknnr/transformers/_base.py:23-67; a constant feature yields
    ``scale_ == 0`` and is not guarded, exactly like the reference)."""

    def __init__(self, ddof: int = 0):
        super().__init__()
        self.ddof = ddof

    def fit(self, X, y=None):
        self._drop_device_state()
        super().fit(X, y)
        X_arr = validate_data(
            self, X=X, accept_sparse=False, dtype=FLOAT_DTYPES, ensure_all_finite="allow-nan",
            reset=False, ensure_min_samples=self.ddof + 1,
        )
        self.scale_ = np.std(X_arr, axis=0, ddof=self.ddof)
        return self

    def _validate_query(self, X, finite=True):
        check_is_fitted(self)
        return validate_data(
            self, X, reset=False, accept_sparse=False, copy=False, dtype=QUERY_DTYPES,
            force_writeable=False, ensure_all_finite="allow-nan" if finite else False,
        )

    def _affine(self):
        return self.mean_, self.scale_, None, self.n_features_in_

    def transform(self, X, copy=None):
        X_arr = self._validate_query(X)
        Z = self._device_transform(X_arr)
        # StandardScaler preserves float32 / float64 inputs (its tag says so); the device computes in
        # float64 and the result is rounded once
        return Z.astype(np.float32) if X_arr.dtype == np.float32 else Z


class ComponentReducerMixin:
    """Transformers whose projector can be truncated to ``n_components`` axes
    (mirrors ref:src/sknnr/transformers/_base.py:70-101)."""

    def __init__(self, n_components: int | None = None):
        self.n_components = n_components

    def get_feature_names_out(self, input_features=None):
        check_is_fitted(self, "n_components_")
        prefix = type(self.ordination_).__name__.lower().replace("result", "")
        return np.asarray([f"{prefix}{i}" for i in range(self.n_components_)], dtype=object)

    def set_n_components(self) -> None:
        limit = self.ordination_.max_components
        n = limit if self.n_components is None else self.n_components
        if not 0 <= n <= limit:
            raise ValueError(f"n_components={n} must be between 0 and {limit}")
        self.n_components_ = n
