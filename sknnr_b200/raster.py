"""Raster front end (SURVEY.md §8 f4): run a fitted estimator over every pixel of a band-major
image - the loop a "sknnr-spatial"-style caller writes around ``est.kneighbors`` / ``est.predict``
(ref:src/sknnr/_base.py:285-352): flatten ``[bands, H, W]`` to ``[H*W, bands]``, drop the pixels
with missing data, query, and put the results back as ``[k, H, W]`` / ``[n_targets, H, W]`` layers.

Here the image goes to the device as it is (float64, float32, or uint8 / int16 / uint16 / int32 /
int64 without a float copy); transpose, mask, compaction and the scatter back run there, next to the
search (``sknnr_raster_kneighbors``), pipelined block by block.  The unmasked
pixels, in row-major pixel order, are numbered like the rows of one ``kneighbors(X[valid])`` call.
"""

from __future__ import annotations

import numpy as np
from sklearn.utils.validation import check_is_fitted

from . import _lib as L
from ._base import _forest_tables

__all__ = ["kneighbors_raster", "predict_raster"]


def _regressor_and_image(est, image):
    """(regressor, query function (bands, k, **kw) -> (dist, idx, pred, n_valid), bands, (H, W))."""
    check_is_fitted(est)
    reg = getattr(est, "regressor_", est)
    kind = reg._metric_kind()
    image = np.asarray(image)
    if image.ndim != 3:
        raise ValueError(f"expected an image of shape [bands, height, width], got {image.shape}")
    if L.x_dtype_code(image) is None:   # (uint8 / int16 / uint16 / int32 / int64 bands go as they are)
        image = np.asarray(image, dtype=np.float64)
    # (a transformed estimator's own n_features_in_ counts the transformed axes, as in the reference)
    n_bands = est.transformer_.n_features_in_ if hasattr(est, "transformer_") else reg.n_features_in_
    if image.shape[0] != n_bands:
        raise ValueError(f"X has {image.shape[0]} features, but {type(est).__name__} is expecting "
                         f"{n_bands} features as input.")
    ix = reg._get_index()
    if kind != "hamming":
        if hasattr(est, "transformer_") and not est._fusable():
            raise NotImplementedError("the estimator's transformer is not an affine map")
        query = ix.query_raster
    elif hasattr(est, "transformer_") and est._forest_fusable():
        forest = est.transformer_._forest_index(_forest_tables(reg.__dict__.get("_node_tables")))
        query = lambda bands, k, **kw: ix.query_raster_forest(forest, bands, k, **kw)  # noqa: E731
    else:
        raise NotImplementedError(
            "a raster needs raw feature bands: Hamming searches are covered through a fitted "
            "tree-node transformer (RFNNRegressor / GBNNRegressor), not on bare node IDs")
    bands = image.reshape(image.shape[0], -1)      # a view for C-ordered (and band-strided) images
    return reg, ix, query, bands, image.shape[1:]


def kneighbors_raster(est, image, n_neighbors=None, *, nodata=None, return_distance=True,
                      use_deterministic_ordering=True, fill_distance=np.nan, fill_index=-1):
    """Neighbours of every pixel.  Returns ``(dist [k, H, W] float64, idx [k, H, W] int64)`` (or
    ``idx`` alone); masked pixels (any band NaN / inf / ``nodata``) hold the fill values.  ``idx``
    are row numbers of the training set, as ``kneighbors(return_dataframe_index=False)`` gives."""
    reg, _, query, bands, hw = _regressor_and_image(est, image)
    k = reg._check_k(n_neighbors, False, bands.shape[1])
    dist, idx, _, _ = query(
        bands, k, nodata=nodata, deterministic=use_deterministic_ordering,
        decimals=reg.DISTANCE_PRECISION_DECIMALS, return_distance=return_distance,
        fill_dist=fill_distance, fill_idx=fill_index)
    idx = idx.reshape(k, *hw)
    return (dist.reshape(k, *hw), idx) if return_distance else idx


def predict_raster(est, image, *, nodata=None, fill_value=np.nan):
    """``est.predict`` for every pixel: ``[n_targets, H, W]`` float64, ``fill_value`` where masked."""
    reg, ix, query, bands, hw = _regressor_and_image(est, image)
    w = reg.weights
    k = reg._check_k(None, False, bands.shape[1])
    if w in (None, "uniform", "distance"):
        _, _, pred, _ = query(bands, k, nodata=nodata, weights=w, with_pred=True,
                              decimals=reg.DISTANCE_PRECISION_DECIMALS,
                              return_distance=False, return_index=False, fill_pred=fill_value)
        return pred.reshape(pred.shape[0], *hw)
    # callable weights: evaluated by Python on the valid pixels' distances, averaged on the device
    dist, idx, _, _ = query(bands, k, nodata=nodata, decimals=reg.DISTANCE_PRECISION_DECIMALS)
    valid = idx[0] >= 0
    out = np.full((ix.n_out, bands.shape[1]), fill_value, dtype=np.float64)
    if valid.any():
        dv = np.ascontiguousarray(dist[:, valid].T)
        iv = np.ascontiguousarray(idx[:, valid].T)
        out[:, valid] = ix.weighted_average(iv, np.asarray(w(dv), dtype=np.float64)).T
    return out.reshape(ix.n_out, *hw)
