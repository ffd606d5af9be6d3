"""`faiss`-compatible facade: exactly the names ConvDR's inference driver touches.

Reference call sites (drivers/run_convdr_inference.py):
    faiss.get_num_gpus()                      :327
    faiss.StandardGpuResources() .setTempMemory  :332-334
    faiss.IndexFlatIP(768)                    :353
    faiss.GpuMultipleClonerOptions() .shard .usePrecomputed   :356-358
    faiss.GpuResourcesVector() / faiss.Int32Vector() .push_back  :360-364
    faiss.index_cpu_to_gpu_multiple(vres, vdev, cpu_index, co)   :365-367
    index.add / index.search / index.reset    :180, :182, :202
Beyond the driver: filtered search, `index.search(x, k, params=SearchParameters(sel=IDSelector...(...)))`
(selectors.py).

Use it either as `import convdr_b200.faiss_compat as faiss` or by putting `convdr_b200/shim`
on PYTHONPATH, which makes a plain `import faiss` resolve to this module (INTEGRATION.md).
Both the `--use_gpu` and the plain path of the driver end up on the same B200 engine; there is no
CPU index behind `IndexFlatIP`.
"""
from __future__ import annotations

from .index import FlatIPIndex, get_num_gpus  # noqa: F401  (get_num_gpus is part of the surface)
from .selectors import (IDSelector, IDSelectorAnd, IDSelectorArray, IDSelectorBatch, IDSelectorBitmap,  # noqa: F401
                        IDSelectorNot, IDSelectorOr, IDSelectorRange, IDSelectorXOr, SearchParameters)

METRIC_INNER_PRODUCT = 0
METRIC_L2 = 1


class IndexFlatIP(FlatIPIndex):
    """faiss.IndexFlatIP(d).  Binds lazily to GPU 0 on first add/search unless cloned to more GPUs."""

    def __init__(self, d: int):
        super().__init__(d, devices=None)


class StandardGpuResources:
    """faiss.StandardGpuResources(): the engine owns its streams and scratch; nothing to configure."""

    def __init__(self):
        self.temp_memory = None

    def setTempMemory(self, nbytes: int) -> None:  # reference :334 (dead code there: tempmem = -1)
        self.temp_memory = int(nbytes)

    def noTempMemory(self) -> None:
        self.temp_memory = 0


class GpuMultipleClonerOptions:
    """faiss.GpuMultipleClonerOptions(): `shard` is honoured (the collection is always row-sharded;
    a replicated flat index would only multiply HBM traffic), `usePrecomputed` is irrelevant to flat
    indexes."""

    def __init__(self):
        self.shard = False
        self.usePrecomputed = False
        self.useFloat16 = False
        self.indicesOptions = 0
        self.verbose = False


class GpuClonerOptions(GpuMultipleClonerOptions):
    pass


class _Vector:
    def __init__(self):
        self._items = []

    def push_back(self, x) -> None:
        self._items.append(x)

    def size(self) -> int:
        return len(self._items)

    def at(self, i: int):
        return self._items[i]

    def __len__(self) -> int:
        return len(self._items)

    def __iter__(self):
        return iter(self._items)


class GpuResourcesVector(_Vector):
    """faiss.GpuResourcesVector()"""


class Int32Vector(_Vector):
    """faiss.Int32Vector()"""


IntVector = Int32Vector


def _clone_to(devices, cpu_index) -> FlatIPIndex:
    if not isinstance(cpu_index, FlatIPIndex):
        raise TypeError("only IndexFlatIP can be moved to the GPUs")
    if cpu_index.ntotal != 0:
        raise RuntimeError("cloning a non-empty index is not supported: add after index_cpu_to_gpu*")
    idx = FlatIPIndex(cpu_index.d, devices=list(devices))
    idx._options = dict(cpu_index._options)
    return idx


def index_cpu_to_gpu_multiple(vres, vdev, cpu_index, co=None) -> FlatIPIndex:
    """faiss.index_cpu_to_gpu_multiple (reference :365-367): one shard per listed device."""
    devices = [int(d) for d in vdev]
    if len(devices) == 0:
        raise RuntimeError("index_cpu_to_gpu_multiple: empty device list")
    if len(vres) != len(devices):
        raise RuntimeError("index_cpu_to_gpu_multiple: resources and devices differ in length")
    return _clone_to(devices, cpu_index)


def index_cpu_to_gpu(res, device: int, cpu_index, co=None) -> FlatIPIndex:
    return _clone_to([int(device)], cpu_index)


def index_cpu_to_all_gpus(cpu_index, co=None, ngpu: int = -1) -> FlatIPIndex:
    n = get_num_gpus() if ngpu < 0 else ngpu
    return _clone_to(list(range(max(n, 1))), cpu_index)


def omp_set_num_threads(n: int) -> None:  # appears only in a comment in the reference (:352)
    return None
