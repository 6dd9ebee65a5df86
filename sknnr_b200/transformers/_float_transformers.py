"""Mahalanobis, CCA (GNN) and CCorA (MSN) transformers: NumPy fit, CUDA transform."""

from __future__ import annotations

import numpy as np
from sklearn.base import BaseEstimator, OneToOneFeatureMixin, TransformerMixin
from sklearn.utils.validation import FLOAT_DTYPES, check_is_fitted, validate_data

from ._base import QUERY_DTYPES, ComponentReducerMixin, DeviceProjectionMixin, StandardScalerWithDOF
from ._ordination import fit_cca, fit_ccora


class MahalanobisTransformer(DeviceProjectionMixin, OneToOneFeatureMixin, TransformerMixin, BaseEstimator):
    """Standardise (N-1 dof) then whiten with the inverse Cholesky factor of the covariance
    (mirrors ref:src/sknnr/transformers/_mahalanobis_transformer.py:20-64)."""

    def fit(self, X, y=None):
        self._drop_device_state()
        X_arr = validate_data(self, X=X, ensure_all_finite="allow-nan", reset=True, ensure_min_features=2)
        self.scaler_ = StandardScalerWithDOF(ddof=1).fit(X)
        Xs = (np.asarray(X_arr, dtype=np.float64) - self.scaler_.mean_) / self.scaler_.scale_
        chol = np.linalg.cholesky(np.cov(Xs, rowvar=False))
        self.transform_ = np.linalg.inv(chol.T)
        return self

    def _validate_query(self, X, finite=True):
        check_is_fitted(self)
        return validate_data(self, X=X, ensure_all_finite="allow-nan" if finite else False, reset=False)

    def _affine(self):
        return self.scaler_.mean_, self.scaler_.scale_, self.transform_, self.transform_.shape[1]

    def transform(self, X, y=None):
        return self._device_transform(self._validate_query(X))

    def fit_transform(self, X, y=None):
        return self.fit(X, y).transform(X)

    def __sklearn_tags__(self):
        tags = super().__sklearn_tags__()
        tags.input_tags.allow_nan = True
        return tags


class CCATransformer(DeviceProjectionMixin, ComponentReducerMixin, TransformerMixin, BaseEstimator):
    """Canonical correspondence analysis projector (GNN); transform is
    ``(X - env_center_) @ projector_`` with no scaling
    (mirrors ref:src/sknnr/transformers/_cca_transformer.py:21-97)."""

    def _checked(self, X, reset, finite=True):
        # (a query keeps its integer dtype for the device; fit works in floats)
        return validate_data(self, X=X, reset=reset, dtype=FLOAT_DTYPES if reset else QUERY_DTYPES,
                             ensure_all_finite=finite, ensure_min_features=2, ensure_min_samples=1)

    def fit(self, X, y):
        self._drop_device_state()
        X_arr = self._checked(X, reset=True)
        y = np.asarray(y)
        if y.ndim < 2:
            raise ValueError("`y` must be a 2D array.")
        self.ordination_ = fit_cca(X_arr, y)
        self.set_n_components()
        self.env_center_ = self.ordination_.env_center
        self.projector_ = self.ordination_.projector(self.n_components_)
        return self

    def get_feature_names_out(self, input_features=None):
        check_is_fitted(self, "n_components_")
        return np.asarray([f"cca{i}" for i in range(self.n_components_)], dtype=object)

    def _validate_query(self, X, finite=True):
        check_is_fitted(self)
        return self._checked(X, reset=False, finite=finite)

    def _affine(self):
        return self.env_center_, None, self.projector_, self.projector_.shape[1]

    def transform(self, X, y=None):
        return self._device_transform(self._validate_query(X))

    def fit_transform(self, X, y):
        return self.fit(X, y).transform(X)

    def __sklearn_tags__(self):
        tags = super().__sklearn_tags__()
        tags.target_tags.required = True
        tags.target_tags.positive_only = True
        return tags


class CCorATransformer(DeviceProjectionMixin, ComponentReducerMixin, TransformerMixin, BaseEstimator):
    """Canonical correlation analysis projector (MSN); transform is
    ``scaler_.transform(X) @ projector_``
    (mirrors ref:src/sknnr/transformers/_ccora_transformer.py:21-79)."""

    def fit(self, X, y):
        self._drop_device_state()
        X_arr, y_arr = validate_data(self, X=X, y=y, reset=True, multi_output=True)
        self.scaler_ = StandardScalerWithDOF(ddof=1).fit(X)
        if y_arr.ndim == 1:
            y_arr = y_arr.reshape(-1, 1)
        y_arr = np.asarray(y_arr, dtype=np.float64)
        y_std = (y_arr - y_arr.mean(axis=0)) / np.std(y_arr, axis=0, ddof=1)
        Xs = (np.asarray(X_arr, dtype=np.float64) - self.scaler_.mean_) / self.scaler_.scale_
        self.ordination_ = fit_ccora(Xs, y_std)
        self.set_n_components()
        self.projector_ = self.ordination_.projector(self.n_components_)
        return self

    def get_feature_names_out(self, input_features=None):
        check_is_fitted(self, "n_components_")
        return np.asarray([f"ccora{i}" for i in range(self.n_components_)], dtype=object)

    def _validate_query(self, X, finite=True):
        check_is_fitted(self)
        return validate_data(self, X=X, reset=False, ensure_all_finite=finite)

    def _affine(self):
        return self.scaler_.mean_, self.scaler_.scale_, self.projector_, self.projector_.shape[1]

    def transform(self, X, y=None):
        return self._device_transform(self._validate_query(X))

    def fit_transform(self, X, y):
        return self.fit(X, y).transform(X)

    def __sklearn_tags__(self):
        tags = super().__sklearn_tags__()
        tags.target_tags.required = True
        return tags
