"""One index sharded over the GPUs of this process: time per search of the three call forms on the same queries.

    python tools/sharded_device_bench.py [--devices 0,1,...] [--rows 38636520] [--nq 173] [--k 100]
                                         [--queue 20] [--rounds 5] [--out FILE]

--devices defaults to every GPU; `--devices 0,0` puts two shards on one GPU.  The rows are the synthetic stream of
bench.py (seed 0, stream 0, unit norm) cut into contiguous per-shard ranges with their global ids, the queries its
query stream (seed 0, stream 1).  The call forms, each warmed up first:
  host    `index.search(q_host, k)`: numpy in, numpy out (page-locked staging inside the engine);
  sync    `index.search_device(q_dev, k)`: CUDA tensor in, CUDA tensors out, one host wait per call;
  queued  `--queue` back-to-back `index.search_device_async(q_dev, k, D, I)` calls and one `finish()`.
Time: host clock from before the first call to the return of the call that waits (every form ends in a device
synchronise), per search, median over `--rounds` rounds in which the three forms alternate.  The outputs of the
three forms are compared bit for bit and the exact-fallback queries of every timed search are reported.
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

N_CAST = 38_636_520   # the headline collection (bench.py)


def gpu_info() -> list[str]:
    """Name and power limit of every GPU (read-only query)."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out
    except Exception as e:   # informational only
        return [f"unavailable: {e}"]


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--devices", default=None, help="comma-separated CUDA devices of the shards (default: every GPU)")
    ap.add_argument("--rows", type=int, default=N_CAST)
    ap.add_argument("--nq", type=int, default=173)
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--queue", type=int, default=20, help="searches queued before one finish()")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from convdr_b200 import FlatIPIndex, synth

    if torch.cuda.device_count() < 1:
        raise SystemExit("sharded_device_bench: no CUDA device")
    devices = ([int(d) for d in args.devices.split(",")] if args.devices
               else list(range(torch.cuda.device_count())))
    G = len(devices)
    idx = FlatIPIndex(768, devices=devices)
    cuts = [args.rows * g // G for g in range(G + 1)]
    t0 = time.perf_counter()
    idx.reserve(max(cuts[g + 1] - cuts[g] for g in range(G)))
    for g in range(G):
        for a in range(cuts[g], cuts[g + 1], 1 << 22):
            idx.add_synthetic(min(1 << 22, cuts[g + 1] - a), first_row=a, seed=0, stream=0, shard=g, id_base=a)
    build_s = time.perf_counter() - t0

    nq, k = args.nq, args.k
    q_host = synth.block(0, nq, seed=0, stream=1)
    q_dev = torch.from_numpy(q_host).to(f"cuda:{devices[0]}")
    Dq = [torch.empty((nq, k), dtype=torch.float32, device=q_dev.device) for _ in range(args.queue)]
    Iq = [torch.empty((nq, k), dtype=torch.int64, device=q_dev.device) for _ in range(args.queue)]

    # each form runs `queue` searches and returns the last result and the exact-fallback queries of all of them
    # (a synchronous search restarts the counters, queued searches accumulate until finish())
    def host():
        fb = 0.0
        for _ in range(args.queue):
            out = idx.search(q_host, k)
            fb += idx.stat("fallback_queries")
        return out, fb

    def sync():
        fb = 0.0
        for _ in range(args.queue):
            out = idx.search_device(q_dev, k)
            fb += idx.stat("fallback_queries")
        return out, fb

    def queued():
        idx.reset_stats()
        for D, I in zip(Dq, Iq):
            idx.search_device_async(q_dev, k, D, I)
        idx.finish()
        return (Dq[-1], Iq[-1]), idx.stat("fallback_queries")

    forms = {"host": host, "sync": sync, "queued": queued}
    for f in forms.values():      # warm-up: modules, workspaces, parts areas
        f()
    torch.cuda.synchronize(q_dev.device)
    ms = {name: [] for name in forms}
    fallbacks = {name: 0.0 for name in forms}
    outs = {}
    for _ in range(args.rounds):
        for name, f in forms.items():
            t0 = time.perf_counter()
            outs[name], fb = f()
            ms[name].append((time.perf_counter() - t0) * 1e3 / args.queue)
            fallbacks[name] += fb
    to_np = lambda t: t.cpu().numpy() if hasattr(t, "cpu") else t
    D0, I0 = (to_np(x) for x in outs["host"])
    identical = all(np.array_equal(to_np(outs[n][1]), I0) and to_np(outs[n][0]).tobytes() == D0.tobytes()
                    for n in ("sync", "queued"))
    identical = identical and all(D.cpu().numpy().tobytes() == D0.tobytes() and np.array_equal(I.cpu().numpy(), I0)
                                  for D, I in zip(Dq, Iq))
    res = {}
    for name in forms:
        med = float(np.median(ms[name]))
        res[name] = {"ms_per_search": med, "queries_per_s": nq / med * 1e3, "ms_rounds": ms[name],
                     "fallback_queries": fallbacks[name]}
    out = {"devices": devices, "rows": args.rows, "nq": nq, "k": k, "queue": args.queue, "rounds": args.rounds,
           "build_s": build_s, "shadow_format": idx.stat("shadow_format"), "gpus": gpu_info(),
           "outputs_bit_identical": bool(identical), "forms": res}
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    idx.close()


if __name__ == "__main__":
    main()
