"""Device-resident fitted state: thin Python owners of the C-ABI index handles.

``KNNIndex`` serves the float estimators (Raw / Euclidean / Mahalanobis / MSN / GNN) with a
Euclidean, Manhattan or Chebyshev search, ``HammingIndex`` serves RFNN.  Handles are caches: they are rebuilt from the NumPy
fitted attributes on demand and never pickled.
"""

from __future__ import annotations

import ctypes as C
import os
import threading

import numpy as np

from . import _lib as L


def default_device() -> int:
    """Device ordinal for new indexes: SKNNR_B200_DEVICE, else LOCAL_RANK, else 0."""
    for var in ("SKNNR_B200_DEVICE", "LOCAL_RANK"):
        v = os.environ.get(var)
        if v not in (None, ""):
            return int(v)
    return 0


# Page-locked blocks are pooled: cudaHostAlloc of a gigabyte takes a large fraction of a second and a
# freshly allocated ndarray costs a page fault per 4 KiB when the results land in it, so result
# arrays of large queries come from blocks that earlier (dead) result arrays gave back.
_POOL_CAP = int(os.environ.get("SKNNR_B200_PINNED_POOL_MB", "4096")) << 20
_pool: dict[int, list] = {}
_pool_bytes = 0
_pool_lock = threading.Lock()


def _pool_take(nbytes):
    global _pool_bytes
    with _pool_lock:
        lst = _pool.get(nbytes)
        if lst:
            _pool_bytes -= nbytes
            return lst.pop()
    return None


def _pool_give(ptr, nbytes, lib):
    global _pool_bytes
    with _pool_lock:
        if _pool_bytes + nbytes <= _POOL_CAP:
            _pool.setdefault(nbytes, []).append(ptr)
            _pool_bytes += nbytes
            return
    lib.sknnr_host_free(ptr)


class _PinnedBlock:
    """Owner of one cudaHostAlloc block; handed back to the pool with the last NumPy view of it."""

    def __init__(self, nbytes, pooled=False):
        self._lib = L.load()
        self.nbytes = int(max(nbytes, 1))
        self.pooled = pooled
        self.ptr = _pool_take(self.nbytes) if pooled else None
        if self.ptr is None:
            self.ptr = C.c_void_p(None)
            L.check(self._lib.sknnr_host_alloc(C.byref(self.ptr), self.nbytes))

    def __del__(self):
        try:
            if self.ptr and self.ptr.value:
                if self.pooled:
                    _pool_give(self.ptr, self.nbytes, self._lib)
                else:
                    self._lib.sknnr_host_free(self.ptr)
        except Exception:
            pass


def pinned_empty(shape, dtype=np.float64, pooled=False) -> np.ndarray:
    """``np.empty`` in page-locked host memory: raster callers that fill / read such buffers get
    full-rate asynchronous copies (pageable arrays are staged by the library's host threads)."""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) if np.ndim(shape) else int(shape)
    nbytes = n * dtype.itemsize
    if pooled:
        nbytes = -(-max(nbytes, 1) // (1 << 20)) << 20       # size classes of 1 MiB
    block = _PinnedBlock(nbytes, pooled)
    buf = (C.c_char * max(nbytes, 1)).from_address(block.ptr.value)
    buf._owner = block                      # keeps the block alive as long as the array's base
    return np.frombuffer(buf, dtype=dtype, count=n).reshape(shape)


def _result_empty(shape, dtype):
    """Result array of a query: pooled page-locked memory once it is large enough to matter."""
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    if n >= (8 << 20) and _POOL_CAP > 0:
        return pinned_empty(shape, dtype, pooled=True)
    return np.empty(shape, dtype=dtype)


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _native(X):
    """``X`` as an array the library reads as it is (float64, float32, uint8, int16, uint16, int32,
    int64) and its ``x_dtype`` code; any other dtype is converted to float64 (exact for every integer
    below 2^53, so the results equal those of ``X.astype(np.float64)`` either way)."""
    X = np.asarray(X)
    code = L.x_dtype_code(X)
    if code is None:
        X = np.asarray(X, dtype=np.float64)
        code = L.F64
    return X, code


def _raster_nodata(nodata, dtype):
    """The float64 that the device compares every band value with.  A float band's nodata is first
    rounded to the band's own type, as an ``image == nodata`` test on the host would do; an integer
    band's stays the float64 given (``dtype.type(nodata)`` would truncate or overflow it), so a
    nodata that is no value of the band type masks nothing."""
    if nodata is None:
        return None
    if np.dtype(dtype).kind == "f":
        return float(np.dtype(dtype).type(nodata))
    return float(nodata)


def _f64(a, ndim=None):
    if a is None:
        return None
    a = np.ascontiguousarray(a, dtype=np.float64)
    if ndim == 2 and a.ndim == 1:
        a = a.reshape(-1, 1)
    return a


def _outputs(out, n_q, k, n_out, return_distance, return_index, mode):
    """Result arrays of a query: fresh ones, or the caller's (``out = (dist, idx, pred)``, C-contiguous
    row blocks of the right dtype - a multi-device query hands every device a slice of shared arrays)."""
    if out is None:
        return (_result_empty((n_q, k), np.float64) if return_distance else None,
                _result_empty((n_q, k), np.int64) if return_index else None,
                _result_empty((n_q, n_out), np.float64) if mode != L.W_NONE else None)
    dist, idx, pred = out
    for a, want, width, dt in ((dist, return_distance, k, np.float64), (idx, return_index, k, np.int64),
                               (pred, mode != L.W_NONE, n_out, np.float64)):
        if want and (a is None or a.shape != (n_q, width) or a.dtype != dt or not a.flags.c_contiguous):
            raise ValueError("`out` arrays must be C-contiguous, of the result's shape and dtype")
    return (dist if return_distance else None, idx if return_index else None, pred if mode != L.W_NONE else None)


def _weights_mode(weights, with_pred):
    if not with_pred:
        return L.W_NONE
    if weights in (None, "uniform"):
        return L.W_UNIFORM
    if isinstance(weights, str) and weights == "distance":
        return L.W_DISTANCE
    raise ValueError(f"unsupported device weights mode {weights!r}")


class _IndexBase:
    _destroy = None
    _stats = None

    def __init__(self):
        self._h = C.c_void_p(None)
        self._lib = L.load()

    def close(self):
        h, self._h = self._h, C.c_void_p(None)
        if h and h.value:
            getattr(self._lib, self._destroy)(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def stats(self) -> dict:
        st = L.Stats()
        L.check(getattr(self._lib, self._stats)(self._h, C.byref(st)))
        return st.as_dict()

    def _flags(self, exclude_self, deterministic, transformed=False):
        f = 0
        if exclude_self:
            f |= L.EXCLUDE_SELF
        if deterministic:
            f |= L.DETERMINISTIC
        if transformed:
            f |= L.TRANSFORMED
        return f


def _raster_call(index, fn, handles, n_bands, bands, k, *, nodata=None, deterministic=True, decimals=10,
                 weights=None, with_pred=False, return_distance=True, return_index=True, fill_dist=np.nan,
                 fill_idx=-1, fill_pred=np.nan, out_dist=None, out_idx=None, out_pred=None):
    """Shared body of the raster entry points (sknnr_raster_kneighbors and its Hamming + forest twin)."""
    bands, dt = _native(bands)
    if bands.ndim != 2 or bands.shape[0] != n_bands:
        raise ValueError(f"the image has {bands.shape[0] if bands.ndim == 2 else '?'} bands, "
                         f"but {n_bands} are expected")
    n_pix = bands.shape[1]
    if n_pix and (bands.strides[1] != bands.itemsize or bands.strides[0] % bands.itemsize
                  or bands.strides[0] < n_pix * bands.itemsize):
        bands = np.ascontiguousarray(bands)
    stride = bands.strides[0] // bands.itemsize if bands.shape[0] > 1 and n_pix else max(n_pix, 1)
    mode = _weights_mode(weights, with_pred)

    def _out(given, shape, dt):
        if given is None:
            return np.empty(shape, dtype=dt)
        if given.shape != shape or given.dtype != dt or not given.flags.c_contiguous:
            raise ValueError(f"preallocated output must be C-contiguous {dt} of shape {shape}")
        return given

    dist = _out(out_dist, (k, n_pix), np.float64) if return_distance else None
    idx = _out(out_idx, (k, n_pix), np.int64) if return_index else None
    pred = _out(out_pred, (index.n_out, n_pix), np.float64) if mode != L.W_NONE else None
    n_valid = C.c_int64(0)
    nodata = _raster_nodata(nodata, bands.dtype)
    L.check(fn(*handles, _ptr(bands), dt, n_pix, stride,
               0 if nodata is None else 1, 0.0 if nodata is None else float(nodata), int(k),
               index._flags(False, deterministic), int(decimals), _ptr(dist), _ptr(idx), mode, _ptr(pred),
               float(fill_dist), int(fill_idx), float(fill_pred), C.byref(n_valid)))
    return dist, idx, pred, n_valid.value


class KNNIndex(_IndexBase):
    """Fitted state of one float estimator on the device.

    ``fit_z``: transformed reference plots (``regressor_._fit_X``); ``center/scale/proj``:
    the affine projection ``Z = ((X - center) / scale) @ proj`` (any may be None);
    ``y``: targets (``regressor_._y``); ``metric``: ``"euclidean"``, ``"manhattan"`` or
    ``"chebyshev"``, the distance searched in the projected space.
    """

    _destroy = "sknnr_index_destroy"
    _stats = "sknnr_index_stats"

    def cascade_counts(self) -> dict:
        """Rows of the last call left uncertified by the tensor engine's first pass, rows that reached the
        FP32 engine and rows that reached the exhaustive float64 kernel."""
        out = (C.c_int64 * 3)()
        L.check(self._lib.sknnr_index_cascade_counts(self._h, out))
        return {"after_tensor": out[0], "to_fp32": out[1], "to_exact": out[2]}

    def __init__(self, fit_z, center=None, scale=None, proj=None, y=None, device=None, metric="euclidean"):
        super().__init__()
        if metric not in L.METRICS:
            raise ValueError(f"metric must be one of {sorted(L.METRICS)}, got {metric!r}")
        self.metric = metric
        fit_z = _f64(fit_z)
        if fit_z.ndim != 2:
            raise ValueError("fit_z must be 2-D")
        self.n_ref, self.d_out = fit_z.shape
        center, scale, proj, y = _f64(center), _f64(scale), _f64(proj), _f64(y, 2)
        if proj is not None:
            self.d_in = proj.shape[0]
            if proj.shape[1] != self.d_out:
                raise ValueError("proj has the wrong number of columns")
        elif center is not None:
            self.d_in = center.shape[0]
        elif scale is not None:
            self.d_in = scale.shape[0]
        else:
            self.d_in = self.d_out
        self.n_out = 0 if y is None else y.shape[1]
        self.device = default_device() if device is None else int(device)
        L.check(self._lib.sknnr_index_create_metric(
            _ptr(fit_z), self.n_ref, self.d_out, _ptr(center), _ptr(scale), _ptr(proj),
            self.d_in, _ptr(y), self.n_out, L.METRICS[metric], self.device, C.byref(self._h)))

    # -- host-buffer query (the drop-in call) ------------------------------------------
    def query(self, X, k, *, exclude_self=False, deterministic=True, decimals=10,
              row_offset=0, transformed=False, weights=None, with_pred=False,
              return_distance=True, return_index=True, check_finite=False, out=None):
        """kneighbors (+ optional predict) on host arrays.  ``X=None`` with
        ``exclude_self`` searches the reference set against itself.  ``check_finite``: the device
        looks for NaN / inf among the query values while it projects them and the call raises
        :class:`NonFiniteInput` (a ``ValueError``) instead of returning results."""
        if exclude_self:
            n_q, Xp, dt, ldx = self.n_ref, None, L.F64, 0
        else:
            X, dt = _native(X)
            if X.ndim != 2:
                raise ValueError("X must be 2-D")
            if X.strides[1] != X.itemsize or X.strides[0] % X.itemsize or X.strides[0] < X.shape[1] * X.itemsize:
                X = np.ascontiguousarray(X)
            n_q = X.shape[0]
            ldx = X.strides[0] // X.itemsize if n_q > 1 else X.shape[1]
            want = self.d_out if transformed else self.d_in
            if X.shape[1] != want:
                raise ValueError(f"X has {X.shape[1]} features, but {want} are expected")
            Xp = _ptr(X)
        mode = _weights_mode(weights, with_pred)
        dist, idx, pred = _outputs(out, n_q, k, self.n_out, return_distance, return_index, mode)
        flags = self._flags(exclude_self, deterministic, transformed)
        if check_finite and not exclude_self:
            flags |= L.CHECK_FINITE
        L.check(self._lib.sknnr_kneighbors(
            self._h, Xp, dt, n_q, ldx, int(row_offset), int(k), flags, int(decimals),
            _ptr(dist), _ptr(idx), mode, _ptr(pred), None))
        return dist, idx, pred

    # -- raster query: band-major image in, band-major layers out (scope row f4) -------
    def query_raster(self, bands, k, **kw):
        """``bands``: ``[d_in, n_pix]`` float64, float32, uint8, int16, uint16, int32 or int64 (any other
        dtype is converted to float64), pixels contiguous within a band (bands may be strided).  A pixel
        with a NaN / inf band, or a band equal to ``nodata``, is masked and
        receives the fill values; the others are queried in pixel order.  Returns
        ``(dist [k, n_pix], idx [k, n_pix], pred [n_out, n_pix], n_valid)``; ``out_*`` are optional
        preallocated C-contiguous result arrays (e.g. from :func:`pinned_empty`)."""
        return _raster_call(self, self._lib.sknnr_raster_kneighbors, (self._h,), self.d_in, bands, k, **kw)

    # -- device-pointer query (benchmarks, multi-GPU pipelines) -------------------------
    def query_device(self, x_ptr, x_is_f32, n_q, ldx, k, *, dist_ptr=0, idx_ptr=0, pred_ptr=0,
                     weights=None, deterministic=True, decimals=10, row_offset=0,
                     transformed=False, stream=0, x_dtype=None):
        """``x_dtype``: NumPy dtype of the rows at ``x_ptr`` (one :func:`_lib.x_dtype_code` maps);
        when given it takes the place of ``x_is_f32``."""
        mode = _weights_mode(weights, bool(pred_ptr))
        flags = self._flags(False, deterministic, transformed) | L.DEVICE_PTRS
        if x_dtype is not None:
            dt = L.x_dtype_code(np.dtype(x_dtype))
            if dt is None:
                raise ValueError(f"the device reads no {np.dtype(x_dtype)} rows")
        else:
            dt = L.F32 if x_is_f32 else L.F64
        L.check(self._lib.sknnr_kneighbors(
            self._h, C.c_void_p(x_ptr), dt, int(n_q), int(ldx),
            int(row_offset), int(k), flags, int(decimals), C.c_void_p(dist_ptr or None),
            C.c_void_p(idx_ptr or None), mode, C.c_void_p(pred_ptr or None),
            C.c_void_p(stream or None)))

    def transform(self, X):
        X, dt = _native(X)
        X = np.ascontiguousarray(X)
        out = np.empty((X.shape[0], self.d_out), dtype=np.float64)
        L.check(self._lib.sknnr_transform(self._h, _ptr(X), dt, X.shape[0], X.shape[1], _ptr(out)))
        return out

    def weighted_average(self, idx, w):
        idx = np.ascontiguousarray(idx, dtype=np.int64)
        w = np.ascontiguousarray(w, dtype=np.float64)
        out = np.empty((idx.shape[0], self.n_out), dtype=np.float64)
        L.check(self._lib.sknnr_weighted_average(self._h, _ptr(idx), _ptr(w), idx.shape[0],
                                                 idx.shape[1], _ptr(out)))
        return out


class HammingIndex(_IndexBase):
    """Fitted state of an RFNN-style estimator: node codes + Hamming weights.  ``ref_codes`` of
    dtype uint32 make a wide index (exact 32-bit codes, ``L.WIDE_NONE`` matches nothing, for trees
    with more than ``L.MAX_CODE`` distinct node IDs); any other dtype holds 16-bit codes."""

    _destroy = "sknnr_hamming_index_destroy"
    _stats = "sknnr_hamming_index_stats"

    def __init__(self, ref_codes, w, y=None, device=None):
        super().__init__()
        self.wide = np.asarray(ref_codes).dtype == np.uint32
        self._code_dtype = np.uint32 if self.wide else np.uint16
        ref_codes = np.ascontiguousarray(ref_codes, dtype=self._code_dtype)
        self.n_ref, self.n_trees = ref_codes.shape
        w = _f64(w)
        y = _f64(y, 2)
        self.n_out = 0 if y is None else y.shape[1]
        self.device = default_device() if device is None else int(device)
        create = self._lib.sknnr_hamming_index_create_wide if self.wide else self._lib.sknnr_hamming_index_create
        L.check(create(_ptr(ref_codes), self.n_ref, self.n_trees, _ptr(w), _ptr(y), self.n_out, self.device,
                       C.byref(self._h)))
        self._kneighbors = self._lib.sknnr_hamming_kneighbors_wide if self.wide else self._lib.sknnr_hamming_kneighbors

    def cascade_counts(self) -> dict:
        """Rows of the last call the filter left uncertified, and rows that reached the exhaustive
        float64 kernel (those, plus every row of a call the filter does not serve)."""
        out = (C.c_int64 * 3)()
        L.check(self._lib.sknnr_hamming_index_cascade_counts(self._h, out))
        return {"uncertified": out[0], "to_exact": out[2]}

    def query(self, codes, k, *, exclude_self=False, deterministic=True, decimals=10,
              row_offset=0, weights=None, with_pred=False, return_distance=True,
              return_index=True, out=None):
        if exclude_self:
            n_q, cp, ldq = self.n_ref, None, 0
        else:
            codes = np.ascontiguousarray(codes, dtype=self._code_dtype)
            n_q, ldq = codes.shape[0], codes.shape[1]
            if ldq != self.n_trees:
                raise ValueError(f"X has {ldq} features, but {self.n_trees} are expected")
            cp = _ptr(codes)
        mode = _weights_mode(weights, with_pred)
        dist, idx, pred = _outputs(out, n_q, k, self.n_out, return_distance, return_index, mode)
        L.check(self._kneighbors(
            self._h, cp, n_q, ldq, int(row_offset), int(k),
            self._flags(exclude_self, deterministic), int(decimals), _ptr(dist), _ptr(idx), mode,
            _ptr(pred), None))
        return dist, idx, pred

    def query_forest(self, forest, X, k, *, deterministic=True, decimals=10, row_offset=0,
                     weights=None, with_pred=False, return_distance=True, return_index=True, out=None):
        """kneighbors (+ predict) on RAW feature rows: forest walk -> node codes -> Hamming
        search in one device call (sknnr_hamming_kneighbors_forest)."""
        X, dt = _native(X)
        X = np.ascontiguousarray(X)
        if X.ndim != 2 or X.shape[1] != forest.n_features:
            raise ValueError(f"X has {X.shape[1] if X.ndim == 2 else '?'} features, but "
                             f"{forest.n_features} are expected")
        n_q = X.shape[0]
        mode = _weights_mode(weights, with_pred)
        dist, idx, pred = _outputs(out, n_q, k, self.n_out, return_distance, return_index, mode)
        L.check(self._lib.sknnr_hamming_kneighbors_forest(
            self._h, forest._h, _ptr(X), dt, n_q, X.shape[1],
            int(row_offset), int(k), self._flags(False, deterministic), int(decimals), _ptr(dist),
            _ptr(idx), mode, _ptr(pred), None))
        return dist, idx, pred

    def query_raster_forest(self, forest, bands, k, **kw):
        """:meth:`KNNIndex.query_raster` for the tree-node estimators: the unmasked pixels' feature
        rows are walked through ``forest`` and searched here without leaving the device."""
        return _raster_call(self, self._lib.sknnr_hamming_raster_kneighbors_forest, (self._h, forest._h),
                            forest.n_features, bands, k, **kw)

    def query_device(self, q_ptr, n_q, ldq, k, *, dist_ptr=0, idx_ptr=0, pred_ptr=0, weights=None,
                     deterministic=True, decimals=10, row_offset=0, stream=0):
        mode = _weights_mode(weights, bool(pred_ptr))
        flags = self._flags(False, deterministic) | L.DEVICE_PTRS
        L.check(self._kneighbors(
            self._h, C.c_void_p(q_ptr), int(n_q), int(ldq), int(row_offset), int(k), flags,
            int(decimals), C.c_void_p(dist_ptr or None), C.c_void_p(idx_ptr or None), mode,
            C.c_void_p(pred_ptr or None), C.c_void_p(stream or None)))

    def weighted_average(self, idx, w):
        idx = np.ascontiguousarray(idx, dtype=np.int64)
        w = np.ascontiguousarray(w, dtype=np.float64)
        out = np.empty((idx.shape[0], self.n_out), dtype=np.float64)
        L.check(self._lib.sknnr_hamming_weighted_average(self._h, _ptr(idx), _ptr(w), idx.shape[0],
                                                         idx.shape[1], _ptr(out)))
        return out


class ForestIndex:
    """Device copy of the fitted trees of an ``RFNodeTransformer`` (all forests, concatenated in
    ``transform``'s column order): scikit-learn's ``tree_`` arrays flattened, plus the 16-bit
    node code the Hamming index uses for every node.  Serves ``transform`` (node IDs) and the
    fused raw-features -> neighbours call of :class:`HammingIndex`."""

    def __init__(self, trees, n_features, node_code_tables=None, device=None):
        """``trees``: scikit-learn ``Tree`` objects (``est.tree_``) in column order;
        ``node_code_tables``: per tree, the sorted node IDs that map to codes 0, 1, ... (None =
        the node ID is its own code)."""
        self._h = C.c_void_p(None)
        self._lib = L.load()
        self.n_trees = len(trees)
        self.n_features = int(n_features)
        offs = np.zeros(self.n_trees + 1, dtype=np.int32)
        offs[1:] = np.cumsum([t.node_count for t in trees])
        cat = lambda name, dt: np.ascontiguousarray(np.concatenate([np.asarray(getattr(t, name)) for t in trees]), dtype=dt)
        left, right = cat("children_left", np.int32), cat("children_right", np.int32)
        feat = np.maximum(cat("feature", np.int32), 0)         # leaves carry -2
        thr = cat("threshold", np.float64)
        if all(hasattr(t, "missing_go_to_left") for t in trees):
            mgl = cat("missing_go_to_left", np.uint8)
        else:
            mgl = None
        code = np.empty(int(offs[-1]), dtype=np.uint16)
        for t in range(self.n_trees):
            ids = np.arange(trees[t].node_count, dtype=np.int64)
            if node_code_tables is None:
                c = np.where(ids < L.MAX_CODE, ids, L.MAX_CODE)
            else:
                u = node_code_tables[t]
                pos = np.searchsorted(u, ids)
                posc = np.minimum(pos, len(u) - 1)
                c = np.where(u[posc] == ids, pos, L.MAX_CODE)
            code[offs[t]:offs[t + 1]] = c.astype(np.uint16)
        self.device = default_device() if device is None else int(device)
        L.check(self._lib.sknnr_forest_create(
            _ptr(offs), _ptr(left), _ptr(right), _ptr(feat), _ptr(thr), _ptr(mgl), _ptr(code),
            self.n_trees, self.n_features, self.device, C.byref(self._h)))

    def apply(self, X) -> np.ndarray:
        """Node ID of every tree for every row, int64 ``[n, n_trees]`` (== hstack of est.apply)."""
        X, dt = _native(X)
        X = np.ascontiguousarray(X)
        out = np.empty((X.shape[0], self.n_trees), dtype=np.int32)
        L.check(self._lib.sknnr_forest_apply(self._h, _ptr(X), dt, X.shape[0], X.shape[1], _ptr(out)))
        return out.astype(np.int64)

    def close(self):
        h, self._h = self._h, C.c_void_p(None)
        if h and h.value:
            self._lib.sknnr_forest_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
