"""faiss ID selectors for filtered search: `index.search(x, k, params=SearchParameters(sel=...))`.

A selector decides, from the label search would return (explicit ids or implicit positions), whether a row may
appear in the results.  The classes only describe the selection; the engine evaluates it on the GPU once per
index (b2f_selector_create) and the scoring kernels then stream only the row tiles that hold selected rows.
`is_member` restates faiss's rule on the host, for inspection and tests; search never calls it.
"""
from __future__ import annotations

import numpy as np

SEL_RANGE, SEL_BATCH, SEL_BITMAP = 1, 2, 3


class IDSelector:
    """Base of the selectors the engine can evaluate."""

    def _describe(self) -> tuple:
        """(kind, invert, imin, imax, ids int64 array or None, bitmap uint8 array or None)."""
        raise NotImplementedError

    def is_member(self, i: int) -> bool:
        return bool(self._mask(np.asarray([i], dtype=np.int64))[0])

    def _mask(self, ids: np.ndarray) -> np.ndarray:
        kind, invert, imin, imax, sel_ids, bitmap = self._describe()
        ids = np.asarray(ids, dtype=np.int64)
        if kind == SEL_RANGE:
            m = (ids >= imin) & (ids < imax)
        elif kind == SEL_BATCH:
            m = np.isin(ids, sel_ids)
        else:
            u = ids.astype(np.uint64)                   # negative ids wrap to huge values: never selected
            inside = (u >> np.uint64(3)) < np.uint64(bitmap.size)
            byte = bitmap[np.where(inside, u >> np.uint64(3), 0).astype(np.int64)] if bitmap.size else np.zeros_like(ids)
            m = inside & (((byte.astype(np.uint64) >> (u & np.uint64(7))) & np.uint64(1)) == 1)
        return m != bool(invert)


def _int64_array(ids, n=None, what="ids") -> np.ndarray:
    a = np.ascontiguousarray(np.asarray(ids).reshape(-1), dtype=np.int64)
    if n is not None:
        n = int(n)
        if n < 0 or n > a.size:
            raise ValueError(f"{what}: n = {n} but only {a.size} values given")
        a = a[:n]
    return a


class IDSelectorRange(IDSelector):
    """faiss.IDSelectorRange(imin, imax): ids with imin <= id < imax."""

    def __init__(self, imin: int, imax: int, assume_sorted: bool = False):
        self.imin, self.imax = int(imin), int(imax)
        self.assume_sorted = bool(assume_sorted)   # accepted for faiss compatibility; no effect on a flat index

    def _describe(self):
        return (SEL_RANGE, 0, self.imin, self.imax, None, None)


class IDSelectorBatch(IDSelector):
    """faiss.IDSelectorBatch(ids) or IDSelectorBatch(n, ids): the listed ids, in any order, duplicates allowed."""

    def __init__(self, *args):
        if len(args) == 1:
            self.ids = _int64_array(args[0])
        elif len(args) == 2:
            self.ids = _int64_array(args[1], args[0])
        else:
            raise TypeError("IDSelectorBatch(ids) or IDSelectorBatch(n, ids)")
        self.ids = np.unique(self.ids)

    def _describe(self):
        return (SEL_BATCH, 0, 0, 0, self.ids, None)


class IDSelectorArray(IDSelectorBatch):
    """faiss.IDSelectorArray(ids) or IDSelectorArray(n, ids): the same membership as IDSelectorBatch."""


class IDSelectorBitmap(IDSelector):
    """faiss.IDSelectorBitmap(bitmap) or IDSelectorBitmap(n, bitmap): `n` bytes; id is selected when
    (bitmap[id >> 3] >> (id & 7)) & 1, ids at or beyond 8 n are not."""

    def __init__(self, *args):
        if len(args) == 1:
            bm, n = args[0], None
        elif len(args) == 2:
            n, bm = args
        else:
            raise TypeError("IDSelectorBitmap(bitmap) or IDSelectorBitmap(n, bitmap)")
        bm = np.asarray(bm)
        if bm.dtype != np.uint8:
            raise TypeError(f"IDSelectorBitmap needs a uint8 array of bytes, got {bm.dtype}")
        bm = np.ascontiguousarray(bm.reshape(-1))
        if n is not None:
            n = int(n)
            if n < 0 or n > bm.size:
                raise ValueError(f"IDSelectorBitmap: n = {n} bytes but the bitmap has {bm.size}")
            bm = bm[:n]
        self.bitmap = bm.copy()

    def _describe(self):
        return (SEL_BITMAP, 0, 0, 0, None, self.bitmap)


class IDSelectorNot(IDSelector):
    """faiss.IDSelectorNot(sel): the complement.  Not(Not(s)) describes s itself."""

    def __init__(self, sel: IDSelector):
        if not isinstance(sel, IDSelector):
            raise TypeError("IDSelectorNot takes one of this module's selectors")
        self.sel = sel

    def _describe(self):
        kind, invert, imin, imax, ids, bitmap = self.sel._describe()
        return (kind, 1 - invert, imin, imax, ids, bitmap)


class _Unsupported(IDSelector):
    def __init__(self, *args, **kwargs):
        raise NotImplementedError(
            f"{type(self).__name__} is not supported by this engine: a filtered search takes one range, batch or "
            "bitmap selector, optionally negated with IDSelectorNot.  Combine the selections into one "
            "IDSelectorBitmap or IDSelectorBatch instead.")


class IDSelectorAnd(_Unsupported):
    """faiss.IDSelectorAnd: not supported (raises NotImplementedError)."""


class IDSelectorOr(_Unsupported):
    """faiss.IDSelectorOr: not supported (raises NotImplementedError)."""


class IDSelectorXOr(_Unsupported):
    """faiss.IDSelectorXOr: not supported (raises NotImplementedError)."""


class SearchParameters:
    """faiss.SearchParameters(sel=...): the selector of a filtered search (None: no filter)."""

    def __init__(self, sel: IDSelector | None = None):
        if sel is not None and not isinstance(sel, IDSelector):
            raise TypeError("SearchParameters(sel=...) takes an IDSelector")
        self.sel = sel
