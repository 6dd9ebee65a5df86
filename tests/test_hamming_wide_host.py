"""Host side of the wide Hamming mode: when a tree has more than 31,743 distinct node IDs the index
keeps exact 32-bit codes instead of 16-bit ones.  No device needed."""

import numpy as np

from sknnr_b200 import _lib as L
from sknnr_b200._base import WideCodes, _encode_nodes, _forest_tables, _node_code_tables


def _narrow_parent(ref_ids, ids):
    """The 16-bit coding as it stands for trees that fit (dense codes from sorted tables)."""
    out = np.empty(ids.shape, dtype=np.uint16)
    for t in range(ref_ids.shape[1]):
        u = np.unique(ref_ids[:, t])
        pos = np.searchsorted(u, ids[:, t])
        pos_c = np.minimum(pos, len(u) - 1)
        out[:, t] = np.where(u[pos_c] == ids[:, t], pos_c, L.MAX_CODE)
    return out


def test_reserved_codes():
    assert L.MAX_CODE == 31743 and L.WIDE_NONE == 0xFFFFFFFF


def test_wide_mode_exactly_when_a_tree_exceeds_16_bit_codes():
    rng = np.random.default_rng(0)
    fits = np.column_stack([rng.permutation(L.MAX_CODE) + 50000, rng.integers(0, 9, L.MAX_CODE)])
    tables = _node_code_tables(fits)
    assert isinstance(tables, list) and len(tables[0]) == L.MAX_CODE
    over = np.vstack([fits, [[123, 4]]])                    # 31744 distinct IDs in tree 0
    wide = _node_code_tables(over)
    assert isinstance(wide, WideCodes) and wide.tables is not None
    # a forest's node IDs are their own codes; the device forest then needs no code tables
    forest = _node_code_tables(over, ids_are_codes=True)
    assert isinstance(forest, WideCodes) and forest.tables is None
    assert _forest_tables(forest) is None and _forest_tables(wide) is None and _forest_tables(tables) is tables
    # IDs that cannot be codes themselves fall back to tables
    neg = over.copy()
    neg[0, 1] = -3
    assert _node_code_tables(neg, ids_are_codes=True).tables is not None
    assert _node_code_tables(np.array([[0, 5], [9, 2]]), ids_are_codes=True) is None


def test_narrow_mapping_unchanged_for_trees_that_fit():
    rng = np.random.default_rng(1)
    ref = rng.integers(-10**6, 10**12, size=(5000, 6))
    q = np.vstack([ref[rng.integers(0, 5000, 300)], rng.integers(-10**6, 10**12, size=(50, 6))])
    tables = _node_code_tables(ref)
    assert isinstance(tables, list)
    for ids in (ref, q):
        enc = _encode_nodes(ids, tables)
        assert enc.dtype == np.uint16
        np.testing.assert_array_equal(enc, _narrow_parent(ref, ids))


def test_dense_wide_codes_and_ids_beyond_int32():
    rng = np.random.default_rng(2)
    base = rng.permutation(40000).astype(np.int64)
    ref = np.column_stack([base * 3 + (1 << 40), base % 7 - 2])
    tables = _node_code_tables(ref)
    assert isinstance(tables, WideCodes) and tables.tables is not None
    enc = _encode_nodes(ref, tables)
    assert enc.dtype == np.uint32
    # dense per-tree codes: the rank of the ID among the tree's sorted IDs
    np.testing.assert_array_equal(enc[:, 0], np.argsort(np.argsort(ref[:, 0])))
    assert enc[:, 1].max() == 6 and enc[:, 0].max() == 39999
    assert not (enc == L.WIDE_NONE).any()
    q = np.array([[ref[5, 0], ref[9, 1]], [(1 << 40) + 1, 99], [-5, -2]])
    eq = _encode_nodes(q, tables)
    assert eq[0, 0] == enc[5, 0] and eq[0, 1] == enc[9, 1]
    assert eq[1].tolist() == [L.WIDE_NONE, L.WIDE_NONE]    # unseen IDs match nothing
    assert eq[2, 0] == L.WIDE_NONE and eq[2, 1] == enc[ref[:, 1] == -2][0, 1]


def test_identity_wide_codes():
    ids = np.array([[0, 70000], [5, 2**31 - 1], [-1, 2**33]])
    enc = _encode_nodes(ids, WideCodes(None))
    assert enc.dtype == np.uint32
    assert enc.tolist() == [[0, 70000], [5, 2**31 - 1], [L.WIDE_NONE, L.WIDE_NONE]]


def test_wide_entry_points_are_exported():
    lib = L.load()
    for name in ("sknnr_hamming_index_create_wide", "sknnr_hamming_kneighbors_wide",
                 "sknnr_hamming_index_cascade_counts"):
        assert name in L.EXPORTS
        assert hasattr(lib, name)
