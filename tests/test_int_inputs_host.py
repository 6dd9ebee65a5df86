"""CPU tests of the integer query inputs (uint8, int16, uint16, int32, int64): the dtype codes of the C
ABI, the query validation that keeps such arrays as they are, and the nodata value of integer bands."""

import os
import re

import numpy as np
import pytest

from tests.conftest import ROOT

NATIVE = [(np.uint8, "U8", 2), (np.int16, "I16", 3), (np.uint16, "U16", 4), (np.int32, "I32", 5),
          (np.int64, "I64", 6)]
CONVERTED = [np.int8, np.uint32, np.uint64, np.bool_, np.float16, object, np.dtype(">i2"), np.complex128]


def _cca_data(n=60, d=4, seed=0):
    rng = np.random.default_rng(seed)
    X = rng.integers(-500, 500, size=(n, d)).astype(np.int16)
    y = rng.random((n, 3)) + 0.1
    return X, y


@pytest.mark.parametrize(("dt", "name", "code"), NATIVE)
def test_x_dtype_code_maps_the_native_integer_types(dt, name, code):
    from sknnr_b200 import _lib as L

    assert getattr(L, name) == code
    assert L.x_dtype_code(np.zeros((2, 3), dtype=dt)) == code
    assert L.x_dtype_code(np.dtype(dt)) == code


@pytest.mark.parametrize("dt", CONVERTED, ids=str)
def test_x_dtype_code_is_none_for_every_other_dtype(dt):
    from sknnr_b200 import _lib as L

    assert L.x_dtype_code(np.zeros((2, 3), dtype=dt)) is None


def test_x_dtype_code_keeps_the_float_codes():
    from sknnr_b200 import _lib as L

    assert L.x_dtype_code(np.zeros(2, np.float64)) == L.F64 == 0
    assert L.x_dtype_code(np.zeros(2, np.float32)) == L.F32 == 1


def test_header_declares_the_codes_the_binding_uses():
    from sknnr_b200 import _lib as L

    with open(os.path.join(ROOT, "include", "sknnr_b200.h")) as f:
        header = f.read()
    declared = {m.group(1): int(m.group(2)) for m in re.finditer(r"#define SKNNR_(\w+) (-?\d+)\b", header)}
    for name in ("F64", "F32", "U8", "I16", "U16", "I32", "I64"):
        assert declared[name] == getattr(L, name), name
    assert declared["ABI_VERSION"] == L.ABI_VERSION == 1


@pytest.mark.parametrize("finite", [False, True])
def test_scaler_query_validation_keeps_an_int16_array(finite):
    from sknnr_b200.transformers import StandardScalerWithDOF

    X, _ = _cca_data()
    sc = StandardScalerWithDOF(ddof=1).fit(X)
    assert sc.mean_.dtype == np.float64 and sc.scale_.dtype == np.float64
    Q = np.ascontiguousarray(X[:7])
    got = sc._validate_query(Q, finite=finite)
    assert got.dtype == np.int16
    assert np.shares_memory(got, Q)


@pytest.mark.parametrize("finite", [False, True])
def test_cca_query_validation_keeps_an_int16_array(finite):
    from sknnr_b200.transformers import CCATransformer

    X, y = _cca_data()
    t = CCATransformer().fit(X, y)
    assert t.env_center_.dtype == np.float64 and t.projector_.dtype == np.float64
    Q = np.ascontiguousarray(X[:7])
    got = t._validate_query(Q, finite=finite)
    assert got.dtype == np.int16
    assert np.shares_memory(got, Q)


@pytest.mark.parametrize("dt", [np.uint8, np.uint16, np.int32, np.int64])
def test_query_validation_keeps_every_native_integer_type(dt):
    from sknnr_b200.transformers import CCATransformer, StandardScalerWithDOF

    X, y = _cca_data()
    X = np.abs(X).astype(dt)
    for t in (StandardScalerWithDOF(ddof=1).fit(X), CCATransformer().fit(X, y)):
        assert t._validate_query(X, finite=False).dtype == dt


@pytest.mark.parametrize("dt", [np.int8, np.uint32, np.bool_])
def test_query_validation_still_converts_other_types_to_float64(dt):
    from sknnr_b200.transformers import CCATransformer, StandardScalerWithDOF

    X, y = _cca_data()
    X = (np.abs(X) % 100).astype(dt)
    y = y[: X.shape[0]]
    for t in (StandardScalerWithDOF(ddof=1).fit(X), CCATransformer().fit(X.astype(np.float64), y)):
        assert t._validate_query(X, finite=False).dtype == np.float64


def test_fit_on_int16_keeps_float64_state():
    from sknnr_b200.transformers import CCATransformer, StandardScalerWithDOF

    X, y = _cca_data()
    Xf = X.astype(np.float64)
    a, b = StandardScalerWithDOF(ddof=1).fit(X), StandardScalerWithDOF(ddof=1).fit(Xf)
    np.testing.assert_array_equal(a.mean_, b.mean_)
    np.testing.assert_array_equal(a.scale_, b.scale_)
    c, e = CCATransformer().fit(X, y), CCATransformer().fit(Xf, y)
    assert c.projector_.dtype == np.float64
    np.testing.assert_array_equal(c.env_center_, e.env_center_)
    np.testing.assert_array_equal(c.projector_, e.projector_)


def test_mixed_int16_float_dataframe_still_comes_back_float64():
    pd = pytest.importorskip("pandas")
    from sknnr_b200.transformers import CCATransformer, StandardScalerWithDOF

    X, y = _cca_data()
    df = pd.DataFrame({f"b{i}": X[:, i] for i in range(X.shape[1])})
    df["b1"] = df["b1"].astype(np.float64)
    for t in (StandardScalerWithDOF(ddof=1).fit(df), CCATransformer().fit(df, y)):
        got = t._validate_query(df, finite=False)
        assert got.dtype == np.float64
        np.testing.assert_array_equal(got, X.astype(np.float64))
    all_int = pd.DataFrame({f"b{i}": X[:, i] for i in range(X.shape[1])})
    assert StandardScalerWithDOF(ddof=1).fit(all_int)._validate_query(all_int, finite=False).dtype == np.int16


def test_tree_node_query_validation_keeps_an_int16_array():
    from sknnr_b200.transformers import RFNodeTransformer

    X, y = _cca_data()
    t = RFNodeTransformer(n_estimators=3, random_state=0).fit(X, y[:, 0])
    Q = np.ascontiguousarray(X[:5])
    got = t._validate_query(Q)
    assert got.dtype == np.int16 and np.shares_memory(got, Q)


def test_raster_nodata_of_integer_bands_stays_float64():
    from sknnr_b200._engine import _raster_nodata

    v = _raster_nodata(-9999.5, np.int16)
    assert type(v) is float and v == -9999.5
    assert _raster_nodata(-9999, np.uint16) == -9999.0       # no value of uint16: masks nothing, no error
    assert _raster_nodata(70000, np.int16) == 70000.0
    assert _raster_nodata(None, np.uint8) is None
    # float bands: rounded to the band's own type first, as before
    assert _raster_nodata(0.1, np.float32) == float(np.float32(0.1))
    assert _raster_nodata(0.1, np.float64) == 0.1
