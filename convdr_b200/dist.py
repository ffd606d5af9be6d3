"""One-process-per-GPU layout of the sharded index (SURVEY.md §8e).

The collection is row-sharded across the ranks of a `torch.distributed` group (NCCL over
NVLink/NVSwitch on the GPU box, gloo in the CPU tests); the queries are replicated; every rank
computes its local top-k with global ids; ONE all-gather of the tiny packed `[nq, k]` (score, id)
lists follows, and a device k-way merge kernel produces the global top-k on every rank.

This replaces FAISS's `IndexShards` (host threads + PCIe + CPU merge) that the reference builds with
`index_cpu_to_gpu_multiple(..., shard=True)` (drivers/run_convdr_inference.py:355-368).
`torch.distributed` is plumbing only: the local search and the merge are libb2f kernels.
"""
from __future__ import annotations

from typing import Callable, Optional

import torch
import torch.distributed as dist


def shard_range(n_total: int, rank: int, world: int, weights=None) -> tuple[int, int]:
    """Contiguous split, identical to b2f_add's per-device split (FAISS shard=True, successive ids).
    `weights` (one positive number per rank, same on every rank) makes the split proportional to them:
    every search waits for the slowest GPU, and the B200s of one box differ by several percent under
    the power cap, so a rank's share can follow its measured speed (`balance_weights`)."""
    if weights is None:
        return n_total * rank // world, n_total * (rank + 1) // world
    assert len(weights) == world and all(w > 0 for w in weights)
    total = float(sum(weights))
    cuts = [0]
    acc = 0.0
    for w in weights:
        acc += w
        cuts.append(int(round(n_total * acc / total)))
    cuts[-1] = n_total
    return cuts[rank], cuts[rank + 1]


def balance_weights(times, clamp: float = 0.15):
    """Shares proportional to 1/time, limited to +-clamp around the equal share (a noisy calibration
    must not unbalance the shards)."""
    inv = [1.0 / max(t, 1e-9) for t in times]
    mean = sum(inv) / len(inv)
    return [min(max(v / mean, 1.0 - clamp), 1.0 + clamp) for v in inv]


class ShardedFlatIP:
    """Rank-local view of a collection sharded over the process group.

    `local_search(q, k) -> (D [nq,k] float32, I [nq,k] int64 global ids)` and
    `merge(D_parts [W,nq,k], I_parts [W,nq,k]) -> (D, I)` default to the rank's FlatIPIndex; the CPU
    (gloo) tests inject stand-ins to exercise the partitioning and the collective plumbing.
    """

    def __init__(self, index=None, group=None, local_search: Optional[Callable] = None,
                 merge: Optional[Callable] = None):
        self.group = group
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.index = index
        self._local_search = local_search or (lambda q, k: self.index.search_device(q, k))
        self._merge = merge or (lambda Dp, Ip: self.index.merge_device(Dp, Ip))
        self.ntotal = 0

    # -- building -------------------------------------------------------------------------------
    def add_synthetic(self, n_total: int, seed: int = 0, stream: int = 0, norm: float = 1.0, chunk: int = 1 << 22,
                      weights=None):
        """Every rank generates its own slice of the synthetic stream on its GPU; ids are global rows."""
        lo, hi = shard_range(n_total, self.rank, self.world, weights)
        self.index.reserve(hi - lo)
        for a in range(lo, hi, chunk):
            b = min(hi, a + chunk)
            self.index.add_synthetic(b - a, first_row=a, seed=seed, stream=stream, norm=norm, id_base=a)
        self.ntotal += n_total
        return lo, hi

    def reset(self):
        self.index.reset()
        self.ntotal = 0

    def local_seconds_per_search(self, q: torch.Tensor, k: int, reps: int = 8) -> float:
        """Device time of this rank's LOCAL search (no exchange), for speed-weighted sharding."""
        D = torch.empty((q.shape[0], k), dtype=torch.float32, device=q.device)
        I = torch.empty((q.shape[0], k), dtype=torch.int64, device=q.device)
        ext = torch.cuda.ExternalStream(self.index.stream_ptr(0), device=q.device)
        for _ in range(2):
            self.index.search_device_async(q, k, D, I)
        self.index.finish()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(ext)
        for _ in range(reps):
            self.index.search_device_async(q, k, D, I)
        self.index.finish()
        e1.record(ext)
        torch.cuda.synchronize(q.device)
        return e0.elapsed_time(e1) * 1e-3 / reps

    def gather_floats(self, value: float):
        """The same scalar from every rank, in rank order (small control-plane exchange)."""
        if self.world == 1:
            return [float(value)]
        out = [None] * self.world
        dist.all_gather_object(out, float(value), group=self.group)
        return out

    def add(self, x_global):
        """Every rank holds the same host array and keeps its slice (labels = global positions)."""
        import numpy as np
        n = x_global.shape[0]
        lo, hi = shard_range(n, self.rank, self.world)
        ids = np.arange(self.ntotal + lo, self.ntotal + hi, dtype=np.int64)
        self.index.add_with_ids(x_global[lo:hi], ids)
        self.ntotal += n
        return lo, hi

    # -- exchange --------------------------------------------------------------------------------
    def enable_peer_exchange(self, max_nq: int, max_k: int) -> bool:
        """Switch the result exchange from ncclAllGather + merge to the engine's own peer-memory
        kernels (CUDA IPC over NVLink/NVSwitch; include/b2f.h b2f_xchg_*).  torch.distributed only
        carries the 64-byte IPC handles, once.  Returns False (and keeps NCCL) if every rank cannot
        map every other rank's buffer — the decision is collective."""
        if self.world == 1 or self.index is None:
            return False
        ok, handle = 1, b"\0" * 64
        try:
            handle = self.index.xchg_create(self.rank, self.world, max_nq, max_k)
        except RuntimeError:
            ok = 0
        gathered = [None] * self.world
        dist.all_gather_object(gathered, (ok, handle), group=self.group)
        if all(g[0] for g in gathered):
            try:
                self.index.xchg_connect([g[1] for g in gathered])
            except RuntimeError:
                ok = 0
        else:
            ok = 0
        flags = [None] * self.world
        dist.all_gather_object(flags, ok, group=self.group)
        self._peer = all(flags)
        self._peer_cap = (max_nq, max_k)
        return self._peer

    # -- searching ------------------------------------------------------------------------------
    def _buffers(self, nq: int, k: int, device):
        """Packed exchange buffers: one part = [D float32 [nq,k] | pad to 16 B | I int64 [nq,k]]."""
        key = (nq, k, str(device))
        if getattr(self, "_key", None) != key:
            i_off = (nq * k * 4 + 15) // 16 * 16
            part = i_off + nq * k * 8
            send = torch.empty(part, dtype=torch.uint8, device=device)
            recv = torch.empty((self.world, part), dtype=torch.uint8, device=device)
            self._send, self._recv, self._i_off, self._part = send, recv, i_off, part
            self._Dl = send[:nq * k * 4].view(torch.float32).view(nq, k)
            self._Il = send[i_off:].view(torch.int64).view(nq, k)
            self._key = key
        return self._send, self._recv

    def search(self, q: torch.Tensor, k: int, params=None):
        """q: [nq, 768] float32 on this rank's device (replicated).  Returns the global (D, I).
        `params=SearchParameters(sel=...)` filters: every rank builds the selector on its own rows from the same
        description (the labels are global), so the merged result is the filtered global top-k.

        GPU ranks: local search, ONE all-gather of the packed (score, id) lists and the merge kernel
        are queued on the engine's stream without a host round trip in between; the host waits once,
        at the end (where the overflow flags of the local search are checked)."""
        nq = q.shape[0]
        if self.index is not None and q.is_cuda:
            return self._search_cuda(q, k, params)
        if params is not None:
            if self.index is None:
                raise NotImplementedError("filtered search needs a rank that owns a FlatIPIndex")
            D, I = self.index.search_device(q, k, params=params)
        else:
            D, I = self._local_search(q, k)
        if self.world == 1:
            return D, I
        send, recv = self._buffers(nq, k, D.device)
        self._Dl.copy_(D)
        self._Il.copy_(I)
        dist.all_gather_into_tensor(recv.view(-1), send, group=self.group)
        Dg = torch.stack([recv[w, :nq * k * 4].view(torch.float32).view(nq, k) for w in range(self.world)])
        Ig = torch.stack([recv[w, self._i_off:].view(torch.int64).view(nq, k) for w in range(self.world)])
        return self._merge(Dg, Ig)

    def search_async(self, q: torch.Tensor, k: int, D: torch.Tensor, I: torch.Tensor, params=None) -> None:
        """Queue local search -> all-gather -> merge on the engine's stream and return; `finish()`
        settles.  q, D, I (CUDA tensors) must stay alive; consecutive calls reuse the exchange buffers
        in stream order."""
        nq = q.shape[0]
        idx = self.index
        if getattr(self, "_ext", None) is None:
            self._ext = torch.cuda.ExternalStream(idx.stream_ptr(0), device=q.device)
        self._ext.wait_stream(torch.cuda.current_stream(q.device))     # q may have been produced there
        if self.world == 1:
            idx.search_device_async(q, k, D, I, params=params)
            return
        if getattr(self, "_peer", False) and nq * k <= self._peer_cap[0] * self._peer_cap[1] and nq <= self._peer_cap[0] \
                and k <= self._peer_cap[1]:
            idx.search_xchg_async(q, k, D, I, params=params)   # search -> NVLink push -> wait + merge, all engine kernels
            self._last_peer = True
            return
        self._last_peer = False
        send, recv = self._buffers(nq, k, q.device)
        with torch.cuda.stream(self._ext):
            idx.search_device_async(q, k, self._Dl, self._Il, params=params)   # local top-k with global ids
            dist.all_gather_into_tensor(recv.view(-1), send, group=self.group)  # the only exchange (NCCL)
            idx.merge_packed_device_async(recv, self.world, self._part, self._i_off, nq, k, D, I)
        self._last = (q, k, D, I)

    def finish(self) -> bool:
        """Wait for the queued searches.  Returns False if a candidate list overflowed on some rank
        (every rank sees the same answer): the caller must repeat those searches synchronously."""
        self.index.finish()
        return not (self.world > 1 and self.index.stat("merge_saw_overflow") > 0)

    def _search_cuda(self, q: torch.Tensor, k: int, params=None):
        nq = q.shape[0]
        idx = self.index
        D = torch.empty((nq, k), dtype=torch.float32, device=q.device)
        I = torch.empty((nq, k), dtype=torch.int64, device=q.device)
        q = q.contiguous()
        self.search_async(q, k, D, I, params)
        if self.world == 1:
            idx.finish()
            return D, I
        # One host wait.  A local query whose candidate list overflowed (adversarial data) is re-run by
        # finish(); its rows travelled with the id -2 marker, which the merge kernel reports on EVERY
        # rank (they all merge the same gathered bytes), so the decision to repeat the exchange is
        # collective without an extra collective.
        idx.finish()
        if idx.stat("xchg_timeout") > 0:
            raise RuntimeError("peer exchange timed out: a rank's part never arrived")
        redo = idx.stat("merge_saw_overflow") > 0      # read-and-clear; identical on every rank
        if redo and self._last_peer:
            idx.search_xchg_async(q, k, D, I, repush_only=True)
            idx.finish()
        elif redo:
            send, recv = self._send, self._recv
            with torch.cuda.stream(self._ext):
                dist.all_gather_into_tensor(recv.view(-1), send, group=self.group)
                idx.merge_packed_device_async(recv, self.world, self._part, self._i_off, nq, k, D, I)
            self._ext.synchronize()
        return D, I

    def search_host(self, q_host, k: int, device=None):
        """End-to-end call with host buffers: pinned H2D of the queries, search, results in host memory.
        GPU ranks: upload, search, exchange and merge are all queued on the engine's stream; the merge kernel
        (the LAST kernel of the call) stores the [nq, k] results straight into pinned host memory over PCIe,
        so no device-to-host copy is queued and the host waits exactly once."""
        if device is None or self.index is None:
            D, I = self.search(torch.from_numpy(q_host), k)
            return D.cpu().numpy(), I.cpu().numpy()
        nq = q_host.shape[0]
        if self.world > 1 and getattr(self, "_peer", False) and nq <= self._peer_cap[0] and k <= self._peer_cap[1] \
                and nq * k <= self._peer_cap[0] * self._peer_cap[1]:
            # peer-memory exchange: the whole call is ONE entry point of the engine (upload, search, NVLink
            # push, merge into page-locked host memory, one wait, overflow protocol)
            return self.index.search_xchg_host(q_host, k)
        key = (nq, k, str(device))
        if getattr(self, "_hkey", None) != key:
            self._hq = torch.empty((nq, q_host.shape[1]), dtype=torch.float32).pin_memory()
            self._hD = torch.empty((nq, k), dtype=torch.float32).pin_memory()
            self._hI = torch.empty((nq, k), dtype=torch.int64).pin_memory()
            self._dq = torch.empty((nq, q_host.shape[1]), dtype=torch.float32, device=device)
            self._hkey = key
        if getattr(self, "_ext", None) is None:
            self._ext = torch.cuda.ExternalStream(self.index.stream_ptr(0), device=device)
        # The pinned query tensor only ever meets torch's own stream (its host allocator records the streams a
        # pinned block was used on); the engine stream is ordered behind the upload by search_async.  The
        # pinned result tensors are only ever written by engine kernels and read after the wait below.
        if q_host.ctypes.data != self._hq.data_ptr():
            self._hq.numpy()[...] = q_host
        self._dq.copy_(self._hq, non_blocking=True)

        def settle():
            if self.world > 1 and getattr(self, "_last_peer", False):
                self.index.xchg_flush()              # the deferred merge joins the engine stream now, no wait
            self._ext.synchronize()                  # the one host wait: upload, search, exchange, merge
            self.index.finish()                      # stream already idle: settles the overflow flags

        self.search_async(self._dq, k, self._hD, self._hI)   # waits (on device) for the upload; writes host memory
        settle()
        # Rare: a candidate list overflowed; finish() re-ran those queries locally.  With several ranks the
        # decision to repeat the exchange must be the same everywhere, so it only looks at the in-band marker
        # every rank's merge saw (never at a rank-local counter).
        if self.world > 1:
            if self.index.stat("merge_saw_overflow") > 0:
                D, I = self._search_cuda(self._dq, k)
                self._hD.copy_(D)
                self._hI.copy_(I)
                torch.cuda.current_stream(device).synchronize()
        else:
            fb = self.index.stat("fallback_queries")      # cumulative over asynchronous searches
            if fb != getattr(self, "_fb_seen", 0.0):
                self._fb_seen = fb                        # finish() rewrote the affected rows in place
        return self._hD.numpy().copy(), self._hI.numpy().copy()
