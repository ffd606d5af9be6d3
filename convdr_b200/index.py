"""Host-side index object over the C ABI (include/b2f.h).

Mirrors the slice of `faiss.IndexFlatIP` that ConvDR's inference driver uses
(reference drivers/run_convdr_inference.py:180 `add`, :182 `search`, :202 `reset`, :353 ctor),
with the same argument meaning and error behaviour: float32 row-major inputs, results as fresh
numpy arrays `D float32 [nq,k]` (descending) and `I int64 [nq,k]`, `-1` / `-FLT_MAX` padding,
`RuntimeError` for engine failures, `AssertionError` for shape mismatches.

All arithmetic happens in libb2f.so on the GPU.  There is no CPU path in this module.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np

from . import _lib

PATHS = {"auto": 0, "scan_f32": 1, "scan_exact": 2, "umma_bf16": 3}
_SELECTOR_CACHE = 8   # compiled selectors kept per index (each holds a row bitmap per shard)
DIM = 768
MAX_K = 2048


def get_num_gpus() -> int:
    """faiss.get_num_gpus() (reference :327)."""
    return int(_lib.load().b2f_device_count())


class FlatIPIndex:
    """Exact inner-product index resident on one or more B200s."""

    def __init__(self, d: int = DIM, devices: Optional[Sequence[int]] = None):
        self.d = int(d)
        self.is_trained = True
        self.metric_type = 0  # faiss.METRIC_INNER_PRODUCT
        self._devices = None if devices is None else [int(x) for x in devices]
        self._h = None
        self._options: dict[str, int] = {}
        self._selectors: dict[int, tuple] = {}   # id(selector) -> (selector, index generation, b2f_selector handle)
        self._ext = None   # the first shard's index stream, as a torch stream
        if self.d != DIM:
            raise RuntimeError(f"b2f supports d = {DIM} only (ConvDR hard-codes IndexFlatIP(768)), got {d}")

    # -- lifetime -------------------------------------------------------------------------------
    def _ensure(self):
        if self._h is None:
            lib = _lib.load()
            h = C.c_void_p()
            if self._devices:
                arr = (C.c_int * len(self._devices))(*self._devices)
                _lib.check(lib.b2f_create(self.d, arr, len(self._devices), C.byref(h)))
            else:
                _lib.check(lib.b2f_create(self.d, None, 0, C.byref(h)))
            self._h = h
            for k, v in self._options.items():
                _lib.check(lib.b2f_set_option(self._h, k.encode(), int(v)))
        return self._h

    def close(self) -> None:
        if self._h is not None:
            for _, _, hs in self._selectors.values():   # a selector goes before its index
                _lib.load().b2f_selector_destroy(hs)
            self._selectors.clear()
            _lib.load().b2f_destroy(self._h)
            self._h = None
            self._ext = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- faiss surface --------------------------------------------------------------------------
    @property
    def ntotal(self) -> int:
        if self._h is None:
            return 0
        return int(_lib.load().b2f_ntotal(self._h))

    def _as_rows(self, x, what: str) -> np.ndarray:
        x = np.ascontiguousarray(x, dtype=np.float32)
        assert x.ndim == 2, f"{what} must be a 2-d array, got shape {x.shape}"
        assert x.shape[1] == self.d, f"{what} has dimension {x.shape[1]}, index has {self.d}"
        return x

    def add(self, x) -> None:
        """index.add(x): append rows; ids are implicit, continuing from ntotal.  Copies x."""
        x = self._as_rows(x, "x")
        h = self._ensure()
        _lib.check(_lib.load().b2f_add(h, x.ctypes.data, x.shape[0]))

    def add_with_ids(self, x, ids) -> None:
        """Append rows with explicit int64 labels (folds reference :190 `embedding2id[I]`)."""
        x = self._as_rows(x, "x")
        ids = np.ascontiguousarray(ids, dtype=np.int64)
        assert ids.shape == (x.shape[0],), "ids must have one label per row"
        h = self._ensure()
        _lib.check(_lib.load().b2f_add_with_ids(h, x.ctypes.data, ids.ctypes.data, x.shape[0]))

    def search(self, x, k: int, params=None):
        """D, I = index.search(x, k, params=None): exact top-k by inner product, sorted descending.  With
        `params=SearchParameters(sel=...)` only rows whose label the selector accepts can be returned; fewer than
        k such rows pad with -FLT_MAX / -1, as faiss does."""
        x = self._as_rows(x, "x")
        k = int(k)
        assert k > 0, "k must be positive"
        nq = x.shape[0]
        D = np.empty((nq, k), dtype=np.float32)
        I = np.empty((nq, k), dtype=np.int64)
        h = self._ensure()
        sel = self._selector(params)
        if sel is None:
            _lib.check(_lib.load().b2f_search(h, x.ctypes.data, nq, k, D.ctypes.data, I.ctypes.data))
        else:
            _lib.check(_lib.load().b2f_search_sel(h, sel, x.ctypes.data, nq, k, D.ctypes.data, I.ctypes.data))
        return D, I

    # -- filtered search ---------------------------------------------------------------------------
    def _selector(self, params):
        """The compiled selector of `params` (None: no filter).  Built on the GPU the first time a selector object
        is used with this index, and again after rows were added or the index was reset."""
        sel = getattr(params, "sel", None) if params is not None else None
        if sel is None:
            return None
        from .selectors import IDSelector
        if not isinstance(sel, IDSelector):
            raise TypeError("params.sel must be an IDSelector of convdr_b200.faiss_compat")
        lib = _lib.load()
        h = self._ensure()
        gen = int(self.stat("generation"))
        hit = self._selectors.get(id(sel))
        if hit is not None and hit[0] is sel and hit[1] == gen:
            return hit[2]
        for key in [key for key, (s, g, _) in self._selectors.items() if g != gen or key == id(sel)]:
            lib.b2f_selector_destroy(self._selectors.pop(key)[2])
        while len(self._selectors) >= _SELECTOR_CACHE:
            lib.b2f_selector_destroy(self._selectors.pop(next(iter(self._selectors)))[2])
        kind, invert, imin, imax, ids, bitmap = sel._describe()
        out = C.c_void_p()
        _lib.check(lib.b2f_selector_create(
            h, kind, int(invert), int(imin), int(imax), None if ids is None or ids.size == 0 else ids.ctypes.data,
            0 if ids is None else ids.size, None if bitmap is None or bitmap.size == 0 else bitmap.ctypes.data,
            0 if bitmap is None else bitmap.size, C.byref(out)))
        self._selectors[id(sel)] = (sel, gen, out)
        return out

    def selected_count(self, sel) -> int:
        """How many rows of the index the selector accepts (b2f_selector_count)."""
        from .selectors import SearchParameters
        out = C.c_int64()
        _lib.check(_lib.load().b2f_selector_count(self._selector(SearchParameters(sel=sel)), C.byref(out)))
        return int(out.value)

    def reconstruct_n(self, i0: int, ni: int, shard: int = 0) -> np.ndarray:
        """IndexFlat.reconstruct_n: stored rows [i0, i0+ni) of one shard, as float32 [ni, d]."""
        out = np.empty((int(ni), self.d), dtype=np.float32)
        _lib.check(_lib.load().b2f_reconstruct_n(self._ensure(), int(shard), int(i0), int(ni), out.ctypes.data))
        return out

    def reconstruct(self, key: int) -> np.ndarray:
        """index.reconstruct(key): the stored row of the label `key` (what `search` returns), float32 [d]."""
        return self.reconstruct_batch(np.array([key], dtype=np.int64))[0]

    def reconstruct_batch(self, keys) -> np.ndarray:
        """index.reconstruct_batch(keys): the stored rows of the labels `keys` (any order, repeats allowed), float32
        [n, d], gathered on the GPU.  RuntimeError naming the label when one is not in the index, is negative, or is
        held by more than one row."""
        keys = np.ascontiguousarray(keys, dtype=np.int64).reshape(-1)
        out = np.empty((keys.size, self.d), dtype=np.float32)
        _lib.check(_lib.load().b2f_reconstruct_batch(self._ensure(), keys.ctypes.data, keys.size, out.ctypes.data))
        return out

    def search_and_reconstruct(self, x, k: int, params=None):
        """D, I, R = index.search_and_reconstruct(x, k, params=None): `search`, plus R float32 [nq, k, d], the stored
        row of every result label; a -1 label (padding) gets a row of 0xFF bytes (NaN), as in faiss."""
        x = self._as_rows(x, "x")
        k = int(k)
        assert k > 0, "k must be positive"
        nq = x.shape[0]
        D = np.empty((nq, k), dtype=np.float32)
        I = np.empty((nq, k), dtype=np.int64)
        R = np.empty((nq, k, self.d), dtype=np.float32)
        h = self._ensure()
        _lib.check(_lib.load().b2f_search_and_reconstruct_sel(h, self._selector(params), x.ctypes.data, nq, k,
                                                              D.ctypes.data, I.ctypes.data, R.ctypes.data))
        return D, I, R

    def reset(self) -> None:
        """index.reset(): drop all rows (device buffers are kept for the next block by default)."""
        if self._h is not None:
            _lib.check(_lib.load().b2f_reset(self._h))

    # -- device-resident extensions ("next" rows of SURVEY §8f) ----------------------------------
    def reserve(self, n_per_shard: int) -> None:
        _lib.check(_lib.load().b2f_reserve(self._ensure(), int(n_per_shard)))

    def add_flat_file(self, path: str, shard: int = 0, threads: int = 0):
        """Stream one flat shard file (blocks.py format) into shard `shard` through pinned staging buffers
        (b2f_add_flat_file; threads = 0: the host's cores shared out over the shards); the stored passage
        offsets become the labels.  Returns (seconds, gigabytes).
        Thread-safe across different shards: ctypes releases the GIL, one host thread per GPU keeps every
        PCIe link busy."""
        secs, gb = C.c_double(), C.c_double()
        _lib.check(_lib.load().b2f_add_flat_file(self._ensure(), int(shard), str(path).encode(), int(threads),
                                                 C.byref(secs), C.byref(gb)))
        return float(secs.value), float(gb.value)

    def write_flat_file(self, path: str, shard: int = 0) -> None:
        """Dump one device-resident shard (rows + labels) to a flat shard file (b2f_write_flat_file) that
        `add_flat_file` / `blocks.open_flat_shard` read back — the writer side of the block format for a
        generator that hands its embeddings over on the device (`add_device`)."""
        _lib.check(_lib.load().b2f_write_flat_file(self._ensure(), int(shard), str(path).encode()))

    def rank_dedup(self, I, D, topN: int, offset2pid):
        """EvalDevQuery's id handling on device (reference drivers/run_convdr_inference.py:43-69): I [nq, >=topN]
        int64 offsets (best first), D float32/float64 scores, offset2pid int64 [n] — all CUDA tensors on the
        index's device.  Returns (pids int64 [nq, topN], scores float64 [nq, topN], counts int32 [nq]): the
        first topN entries translated to pids with repeated pids dropped, survivors first, tail (0, 0.0)."""
        import torch
        assert I.is_cuda and D.is_cuda and offset2pid.is_cuda and I.dtype == torch.int64 and offset2pid.dtype == torch.int64
        assert I.dim() == 2 and D.shape == I.shape and I.shape[1] >= topN and I.stride(1) == 1 and D.stride(1) == 1
        assert D.dtype in (torch.float32, torch.float64) and I.stride(0) == D.stride(0)
        nq = I.shape[0]
        pid = torch.empty((nq, topN), dtype=torch.int64, device=I.device)
        sc = torch.empty((nq, topN), dtype=torch.float64, device=I.device)
        cnt = torch.empty((nq,), dtype=torch.int32, device=I.device)
        d32 = D.data_ptr() if D.dtype == torch.float32 else None
        d64 = D.data_ptr() if D.dtype == torch.float64 else None
        torch.cuda.current_stream(I.device).synchronize()
        _lib.check(_lib.load().b2f_rank_dedup_device(self._ensure(), I.data_ptr(), d32, d64, nq, I.stride(0), int(topN),
                                                     offset2pid.data_ptr(), offset2pid.numel(), pid.data_ptr(),
                                                     sc.data_ptr(), cnt.data_ptr()))
        return pid, sc, cnt

    def add_device(self, x, shard: int = 0) -> None:
        """Append a CUDA float32 torch tensor [n, d] living on the shard's device (no host copy)."""
        assert x.is_cuda and x.dtype.is_floating_point and x.dim() == 2 and x.shape[1] == self.d
        import torch
        x = x.contiguous().to(torch.float32)
        _lib.check(_lib.load().b2f_add_device(self._ensure(), int(shard), x.data_ptr(), x.shape[0]))

    def add_synthetic(self, n: int, *, first_row: int = 0, seed: int = 0, stream: int = 0, norm: float = 1.0,
                      shard: int = 0, id_base: Optional[int] = None) -> None:
        """Append rows [first_row, first_row+n) of the synthetic stream (seed, stream); see synth.py."""
        if id_base is None:
            id_base = first_row
        _lib.check(_lib.load().b2f_add_synthetic(self._ensure(), int(shard), int(first_row), int(n), int(seed),
                                                 int(stream), float(norm), int(id_base)))

    def _first_device(self) -> int:
        """The device of the first shard: device-resident queries and results live there."""
        return self._devices[0] if self._devices else 0

    def _device_call(self, q, *out):
        """Checks that q and the outputs live on the first shard's device (outputs may also be page-locked host
        tensors, which the last kernel writes directly), then orders the index stream after the caller's current
        stream there: q may have just been produced by work queued on it (an encoder)."""
        import torch
        dev = self._first_device()
        for t in (q,) + out:
            assert (t.is_cuda and t.device.index == dev) or (t is not q and not t.is_cuda and t.is_pinned()), \
                f"device search tensors must be on cuda:{dev}, the first shard's device; got {t.device}"
        h = self._ensure()
        if self._ext is None:
            self._ext = torch.cuda.ExternalStream(self.stream_ptr(0), device=q.device)
        self._ext.wait_stream(torch.cuda.current_stream(q.device))
        return h

    def search_device(self, q, k: int, params=None):
        """Search with a CUDA torch tensor of queries on the first shard's device (any number of shards); returns
        CUDA tensors (D, I) on that device.  `params` as in `search`."""
        import torch
        assert q.is_cuda and q.dim() == 2 and q.shape[1] == self.d
        q = q.contiguous().to(torch.float32)
        nq = q.shape[0]
        D = torch.empty((nq, int(k)), dtype=torch.float32, device=q.device)
        I = torch.empty((nq, int(k)), dtype=torch.int64, device=q.device)
        if self._selector(params) is None:
            _lib.check(_lib.load().b2f_search_device(self._device_call(q, D, I), q.data_ptr(), nq, int(k),
                                                     D.data_ptr(), I.data_ptr()))
        else:
            self.search_device_async(q, k, D, I, params=params)
            self.finish()
        return D, I

    def search_and_reconstruct_device(self, q, k: int, params=None):
        """`search_and_reconstruct` with a CUDA torch tensor of queries on the first shard's device (any number of
        shards): returns CUDA tensors (D, I, R) there, R float32 [nq, k, d].  The rows are gathered on the GPUs that
        hold them, next to the resident index."""
        import torch
        assert q.is_cuda and q.dim() == 2 and q.shape[1] == self.d
        q = q.contiguous().to(torch.float32)
        nq, k = q.shape[0], int(k)
        D = torch.empty((nq, k), dtype=torch.float32, device=q.device)
        I = torch.empty((nq, k), dtype=torch.int64, device=q.device)
        R = torch.empty((nq, k, self.d), dtype=torch.float32, device=q.device)
        sel = self._selector(params)
        _lib.check(_lib.load().b2f_search_and_reconstruct_device_sel(self._device_call(q, D, I, R), sel, q.data_ptr(),
                                                                     nq, k, D.data_ptr(), I.data_ptr(), R.data_ptr()))
        return D, I, R

    def search_device_into(self, q, k: int, D, I) -> None:
        """Same, into caller-provided CUDA tensors (no allocation inside a timed loop)."""
        _lib.check(_lib.load().b2f_search_device(self._device_call(q, D, I), q.data_ptr(), q.shape[0], int(k),
                                                 D.data_ptr(), I.data_ptr()))

    def search_device_async(self, q, k: int, D, I, params=None) -> None:
        """Enqueue only (b2f_search_device_async): q, D, I are CUDA tensors on the first shard's device that must
        stay alive until `finish()`; later work on the index stream (`stream_ptr(0)`) may consume D / I without a
        host round trip.  Until then, a row whose candidate list overflowed carries id -2 in its first slot.
        `params` as in `search`; searches with different selectors may be in flight together."""
        sel = self._selector(params)
        h = self._device_call(q, D, I)
        if sel is None:
            _lib.check(_lib.load().b2f_search_device_async(h, q.data_ptr(), q.shape[0], int(k), D.data_ptr(),
                                                           I.data_ptr()))
        else:
            _lib.check(_lib.load().b2f_search_device_async_sel(h, sel, q.data_ptr(), q.shape[0], int(k), D.data_ptr(),
                                                               I.data_ptr()))

    def finish(self) -> None:
        """Wait for every search enqueued with `search_device_async` (re-running overflowed queries)."""
        if self._h is not None:
            _lib.check(_lib.load().b2f_search_finish(self._h))

    def merge_packed_device_async(self, parts, n_parts: int, part_bytes: int, i_offset: int, nq: int, k: int, D, I):
        """Merge packed [D | I] parts (one all-gather's receive buffer, uint8) on the index stream."""
        _lib.check(_lib.load().b2f_merge_packed_device_async(self._ensure(), parts.data_ptr(), int(n_parts),
                                                             int(part_bytes), int(i_offset), int(nq), int(k),
                                                             D.data_ptr(), I.data_ptr()))

    # -- peer-memory exchange (one process per GPU) ------------------------------------------------
    def xchg_create(self, rank: int, world: int, max_nq: int, max_k: int) -> bytes:
        """Allocate this rank's exchange buffer; returns its 64-byte CUDA IPC handle."""
        buf = C.create_string_buffer(64)
        _lib.check(_lib.load().b2f_xchg_create(self._ensure(), int(rank), int(world), int(max_nq), int(max_k), buf))
        return buf.raw

    def xchg_connect(self, handles) -> None:
        """handles: the 64-byte handles of all ranks, in rank order."""
        blob = b"".join(handles)
        _lib.check(_lib.load().b2f_xchg_connect(self._ensure(), blob))

    def search_xchg_async(self, q, k: int, D, I, repush_only: bool = False, params=None) -> None:
        """Collective: local search -> NVLink push of the packed part to every rank -> wait + merge.  With
        `params`, every rank filters its own rows with the same selector description."""
        _lib.check(_lib.load().b2f_search_xchg_async_sel(self._ensure(), self._selector(params), q.data_ptr(),
                                                         q.shape[0], int(k), D.data_ptr(), I.data_ptr(),
                                                         1 if repush_only else 0))

    def search_xchg_host(self, x, k: int, D=None, I=None):
        """Collective end-to-end search with host buffers (b2f_search_xchg_host): numpy in, numpy out; pass
        page-locked arrays (e.g. views of torch pinned tensors) to skip the staging copies."""
        x = self._as_rows(x, "x")
        nq = x.shape[0]
        if D is None:
            D = np.empty((nq, int(k)), dtype=np.float32)
            I = np.empty((nq, int(k)), dtype=np.int64)
        _lib.check(_lib.load().b2f_search_xchg_host(self._ensure(), x.ctypes.data, nq, int(k), D.ctypes.data, I.ctypes.data))
        return D, I

    def xchg_flush(self) -> None:
        """Enqueue the exchange merge that is still owed (deferred by one search), without waiting."""
        _lib.check(_lib.load().b2f_xchg_flush(self._ensure()))

    def reset_stats(self) -> None:
        self.set_option("reset_stats", 1)

    def merge_device(self, D_parts, I_parts):
        """Merge per-shard results [G, nq, k] (CUDA tensors on this index's device) into [nq, k]."""
        import torch
        G, nq, k = D_parts.shape
        D = torch.empty((nq, k), dtype=torch.float32, device=D_parts.device)
        I = torch.empty((nq, k), dtype=torch.int64, device=D_parts.device)
        _lib.check(_lib.load().b2f_merge_device(self._ensure(), D_parts.data_ptr(), I_parts.data_ptr(), int(G),
                                                int(nq), int(k), D.data_ptr(), I.data_ptr()))
        return D, I

    # -- knobs / introspection --------------------------------------------------------------------
    def set_option(self, key: str, value) -> None:
        """Engine knob (include/b2f.h b2f_set_option), e.g. "shadow": 0 none, 1 bf16, 2 int8, 3 AUTO (default:
        int8 or bf16 per shard, chosen from its first rows; stat "shadow_format" tells which)."""
        if key == "path" and isinstance(value, str):
            value = PATHS[value]
        self._options[key] = int(value)
        if self._h is not None:
            _lib.check(_lib.load().b2f_set_option(self._h, key.encode(), int(value)))

    def stat(self, key: str) -> float:
        out = C.c_double()
        _lib.check(_lib.load().b2f_get_stat(self._ensure(), key.encode(), C.byref(out)))
        return float(out.value)

    def stream_ptr(self, shard: int = 0) -> int:
        return int(_lib.load().b2f_stream(self._ensure(), int(shard)) or 0)

    @property
    def num_shards(self) -> int:
        return int(_lib.load().b2f_num_shards(self._ensure()))

    def shard_rows(self, shard: int) -> int:
        return int(_lib.load().b2f_shard_rows(self._ensure(), int(shard)))
