"""CPU tests of the filtered-search facade: the faiss ID selectors' argument handling and membership rules
(convdr_b200/selectors.py), as faiss defines them.  The GPU evaluation of the same descriptions is checked in
tests/test_selector.py."""
import numpy as np
import pytest

import convdr_b200.faiss_compat as faiss
from convdr_b200 import selectors


def members(sel, n):
    return np.nonzero(sel._mask(np.arange(n)))[0].tolist()


def test_range_bounds_are_half_open():
    sel = faiss.IDSelectorRange(3, 7)
    assert members(sel, 10) == [3, 4, 5, 6]
    assert not sel.is_member(7) and sel.is_member(3) and not sel.is_member(-1)
    assert members(faiss.IDSelectorRange(5, 5), 10) == []
    assert members(faiss.IDSelectorRange(8, 2), 10) == []
    assert sel._describe()[:4] == (selectors.SEL_RANGE, 0, 3, 7)


def test_batch_accepts_unsorted_ids_with_duplicates_and_the_n_form():
    sel = faiss.IDSelectorBatch(np.array([9, 2, 2, 5, 9, 0]))
    assert members(sel, 12) == [0, 2, 5, 9]
    assert sel._describe()[4].tolist() == [0, 2, 5, 9]          # sorted and unique for the device binary search
    assert members(faiss.IDSelectorBatch(3, np.array([9, 2, 2, 5])), 12) == [2, 9]   # the first n ids only
    assert members(faiss.IDSelectorBatch([]), 5) == []
    assert not sel.is_member(-2) and not sel.is_member(1 << 40)
    with pytest.raises(ValueError):
        faiss.IDSelectorBatch(5, np.array([1, 2]))


def test_array_has_the_membership_of_batch():
    assert members(faiss.IDSelectorArray(np.array([4, 1, 4])), 6) == [1, 4]
    assert members(faiss.IDSelectorArray(2, [7, 3, 5]), 9) == [3, 7]


def test_bitmap_bit_order_is_lsb_first_within_each_byte():
    bm = np.array([0b00000101, 0b10000000], dtype=np.uint8)    # ids 0, 2 and 15
    sel = faiss.IDSelectorBitmap(bm)
    assert members(sel, 40) == [0, 2, 15]
    assert sel._describe()[5].tolist() == [5, 128]


def test_bitmap_n_counts_bytes_and_ids_beyond_8n_are_not_selected():
    bm = np.array([0xFF, 0xFF, 0xFF], dtype=np.uint8)
    assert members(faiss.IDSelectorBitmap(2, bm), 40) == list(range(16))    # n = 2 bytes: ids 0..15
    assert members(faiss.IDSelectorBitmap(bm), 40) == list(range(24))
    assert not faiss.IDSelectorBitmap(bm).is_member(-1)
    assert members(faiss.IDSelectorBitmap(np.zeros(0, dtype=np.uint8)), 8) == []
    with pytest.raises(ValueError):
        faiss.IDSelectorBitmap(4, bm)
    with pytest.raises(TypeError):
        faiss.IDSelectorBitmap(np.array([1, 2], dtype=np.int32))


def test_bitmap_copies_its_bytes():
    bm = np.array([1], dtype=np.uint8)
    sel = faiss.IDSelectorBitmap(bm)
    bm[0] = 2
    assert members(sel, 8) == [0]


def test_not_inverts_and_double_negation_collapses():
    base = faiss.IDSelectorRange(2, 5)
    n1 = faiss.IDSelectorNot(base)
    assert members(n1, 7) == [0, 1, 5, 6]
    assert n1._describe()[1] == 1
    n2 = faiss.IDSelectorNot(n1)
    assert n2._describe() == base._describe()
    assert members(n2, 7) == [2, 3, 4]
    inv_bm = faiss.IDSelectorNot(faiss.IDSelectorBitmap(np.array([0b11], dtype=np.uint8)))
    assert members(inv_bm, 12) == list(range(2, 12))    # beyond the bitmap: not in it, so in its complement
    with pytest.raises(TypeError):
        faiss.IDSelectorNot(lambda i: True)


@pytest.mark.parametrize("name", ["IDSelectorAnd", "IDSelectorOr", "IDSelectorXOr"])
def test_combinations_raise_not_implemented_with_a_clear_message(name):
    a, b = faiss.IDSelectorRange(0, 3), faiss.IDSelectorRange(2, 5)
    with pytest.raises(NotImplementedError, match="not supported.*IDSelectorBitmap or IDSelectorBatch"):
        getattr(faiss, name)(a, b)


def test_search_parameters_holds_a_selector_or_none():
    assert faiss.SearchParameters().sel is None
    sel = faiss.IDSelectorRange(0, 1)
    assert faiss.SearchParameters(sel=sel).sel is sel
    with pytest.raises(TypeError):
        faiss.SearchParameters(sel=[1, 2, 3])


def test_the_shim_exposes_the_selectors():
    import importlib.util
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("faiss_shim_probe", os.path.join(root, "convdr_b200", "shim", "faiss.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    for name in ("SearchParameters", "IDSelectorRange", "IDSelectorBatch", "IDSelectorArray", "IDSelectorBitmap",
                 "IDSelectorNot", "IDSelectorAnd", "IDSelectorOr", "IDSelectorXOr"):
        assert hasattr(mod, name), name
