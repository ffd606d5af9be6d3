"""Rows by label on one GPU: the cost of `search_and_reconstruct_device` over `search_device`, the gather's own rate,
and the first lookup on a shard whose labels need a sorted copy.

    python tools/reconstruct_bench.py [--rows 4830815] [--nq 173] [--ks 100,1000] [--rounds 5] [--calls 20] [--out FILE]

The rows are the synthetic stream of bench.py (seed 0, stream 0, unit norm; AUTO shadow) with their positions as labels
(segment labels), the queries its query stream (seed 0, stream 1).  Per k:
  search / search_and_reconstruct  `search_device(q, k)` and `search_and_reconstruct_device(q, k)`, `--calls` calls
      each, alternating in `--rounds` rounds; host clock around calls that end in a device synchronise; median ms;
  gather  device time of `gather_rows_kernel` from torch.profiler over `--calls` calls (a run of its own), and its
      rate 2 * nq * k * 3072 bytes (rows read + written) per second, next to the device-to-device `copy_` rate of a
      4 GB tensor timed with CUDA events on the same GPU.
Sorted label copy: a second index of `--rows` rows with shuffled explicit labels (added from host memory in 1 M-row
pieces that repeat one block of rows); the first `reconstruct_batch` of nq * 100 labels builds the copy (the sort),
the later ones reuse it.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

N_SHARD = 4_830_815   # one of the eight shards of the headline collection (38,636,520 rows)


def gpu_info() -> list[str]:
    """Name and power limit of the GPU (read-only query)."""
    try:
        return subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    except Exception as e:   # informational only
        return [f"unavailable: {e}"]


def copy_rate(torch) -> float:
    """Device-to-device copy_ of a 4 GB float32 tensor: bytes read + written per second."""
    a = torch.empty(1 << 30, dtype=torch.float32, device="cuda")
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    return 2 * a.numel() * 4 * 10 / (e0.elapsed_time(e1) * 1e-3)


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--rows", type=int, default=N_SHARD)
    ap.add_argument("--nq", type=int, default=173)
    ap.add_argument("--ks", default="100,1000")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from convdr_b200 import FlatIPIndex, synth

    if torch.cuda.device_count() < 1:
        raise SystemExit("reconstruct_bench: no CUDA device")
    idx = FlatIPIndex(768)
    idx.reserve(args.rows)
    for a in range(0, args.rows, 1 << 22):
        idx.add_synthetic(min(1 << 22, args.rows - a), first_row=a, seed=0, stream=0)
    nq = args.nq
    q = torch.from_numpy(synth.block(0, nq, seed=0, stream=1)).cuda()
    res = {"gpu": gpu_info(), "rows": args.rows, "nq": nq, "shadow_format": idx.stat("shadow_format"),
           "copy_GBps": copy_rate(torch) / 1e9, "k": {}}

    for k in (int(x) for x in args.ks.split(",")):
        forms = {"search": lambda: idx.search_device(q, k), "search_and_reconstruct": lambda: idx.search_and_reconstruct_device(q, k)}
        for f in forms.values():
            f()
        ms = {name: [] for name in forms}
        for _ in range(args.rounds):
            for name, f in forms.items():
                t0 = time.perf_counter()
                for _ in range(args.calls):
                    out = f()
                ms[name].append((time.perf_counter() - t0) * 1e3 / args.calls)
        D, I = idx.search_device(q, k)
        Dr, Ir, R = idx.search_and_reconstruct_device(q, k)
        identical = torch.equal(I, Ir) and torch.equal(D.view(torch.int32), Dr.view(torch.int32))
        rows_ok = torch.equal(R[7, :5].cpu(), torch.from_numpy(idx.reconstruct_batch(I[7, :5].cpu().numpy())))
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(args.calls):
                idx.search_and_reconstruct_device(q, k)
        gather_us = sum(e.device_time_total for e in prof.key_averages()
                        if "gather_rows_kernel" in e.key) / args.calls
        gbytes = 2 * nq * k * 3072 / 1e9
        res["k"][k] = {
            "search_ms": float(np.median(ms["search"])), "search_and_reconstruct_ms": float(np.median(ms["search_and_reconstruct"])),
            "ms_rounds": ms, "gather_us": gather_us, "gather_GBps": gbytes / (gather_us * 1e-6) if gather_us else None,
            "gather_GB": gbytes, "D_I_identical_to_search": bool(identical), "rows_match_reconstruct_batch": bool(rows_ok),
            "fallback_queries": idx.stat("fallback_queries")}
        del out
    idx.close()

    # sorted label copy: shuffled explicit labels
    rng = np.random.default_rng(0)
    labels = rng.permutation(args.rows).astype(np.int64)
    piece = min(1 << 20, args.rows)
    block = synth.block(0, piece, seed=0, stream=0)
    sh = FlatIPIndex(768)
    sh.reserve(args.rows)
    for a in range(0, args.rows, piece):
        b = min(args.rows, a + piece)
        sh.add_with_ids(block[:b - a], labels[a:b])
    keys = rng.choice(labels, nq * 100)
    times = []
    for _ in range(6):
        t0 = time.perf_counter()
        sh.reconstruct_batch(keys)
        times.append((time.perf_counter() - t0) * 1e3)
    res["shuffled"] = {"labels": int(keys.size), "first_lookup_ms": times[0], "later_lookup_ms": times[1:],
                       "label_index_bytes": sh.stat("label_index_bytes")}
    sh.close()

    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
