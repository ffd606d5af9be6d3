"""Filtered search on one GPU: time per search, streamed shadow bytes and exact-fallback queries for no selector and
four selectors, as one A/B on one box (DESIGN.md section 7: the cases alternate round by round, so drift of the
shared machine hits every case alike).

    python tools/selector_bench.py [--rows 4830000] [--nq 173] [--k 100] [--rounds 5] [--reps 20] [--out FILE]

The shard is synthetic (seed 0, AUTO shadow format).  Time: host clock around `reps` back-to-back
`search_device_async` calls and the `finish()` that waits for them (and re-runs overflowed queries), median over
the rounds.  Bytes: the rows of the listed tiles
(stat score_rows of one profiled search) times the shadow bytes per row.  `fallback_queries`: queries whose k-th
selected score fell outside the tightening window or whose lists overflowed, re-run on the exact engine.
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


def gpu_info() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return {"nvidia_smi": out[0] if out else ""}
    except Exception as e:   # informational only
        return {"nvidia_smi": f"unavailable: {e}"}


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--rows", type=int, default=4830000)
    ap.add_argument("--nq", type=int, default=173)
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import convdr_b200.faiss_compat as faiss
    from convdr_b200 import FlatIPIndex

    n = args.rows
    rng = np.random.default_rng(0)
    cases = {
        "none": None,
        "all_rows": faiss.IDSelectorRange(0, n),
        "range_10pct": faiss.IDSelectorRange(n // 3, n // 3 + n // 10),
        "batch_1pct_scattered": faiss.IDSelectorBatch(rng.choice(n, n // 100, replace=False)),
        "bitmap_50pct_scattered": faiss.IDSelectorBitmap(np.packbits(rng.random(n) < 0.5, bitorder="little")),
    }
    idx = FlatIPIndex(768)
    idx.add_synthetic(n, seed=0)
    bytes_per_row = {1: 1536, 2: 768}[int(idx.stat("shadow_format"))]
    q = torch.from_numpy(np.random.default_rng(1).standard_normal((args.nq, 768)).astype(np.float32)).cuda()
    q = torch.nn.functional.normalize(q, dim=1)
    D = torch.empty((args.nq, args.k), dtype=torch.float32, device="cuda")
    I = torch.empty((args.nq, args.k), dtype=torch.int64, device="cuda")
    params = {name: (None if s is None else faiss.SearchParameters(sel=s)) for name, s in cases.items()}
    res = {name: {"ms": [], "selected": (n if s is None else idx.selected_count(s))} for name, s in cases.items()}

    for name in cases:   # warm-up, profiled search: streamed rows and fallbacks of one search
        idx.set_option("profile", 1)
        idx.reset_stats()
        idx.search_device_async(q, args.k, D, I, params=params[name])
        idx.finish()
        res[name]["score_rows"] = idx.stat("score_rows")
        res[name]["streamed_bytes"] = idx.stat("score_rows") * bytes_per_row
        res[name]["fallback_queries"] = idx.stat("fallback_queries")
        idx.set_option("profile", 0)
    for _ in range(args.rounds):
        for name in cases:
            idx.reset_stats()
            t0 = time.perf_counter()
            for _ in range(args.reps):
                idx.search_device_async(q, args.k, D, I, params=params[name])
            idx.finish()                   # waits for the stream and runs any exact re-run: both are timed
            res[name]["ms"].append((time.perf_counter() - t0) * 1e3 / args.reps)
            res[name].setdefault("fallback_queries_timed", 0.0)
            res[name]["fallback_queries_timed"] += idx.stat("fallback_queries")
    for name, r in res.items():
        r["ms_median"] = float(np.median(r["ms"]))
        r["fallback_queries_timed_per_search"] = r.pop("fallback_queries_timed") / (args.rounds * args.reps)
    out = {"rows": n, "nq": args.nq, "k": args.k, "shadow_bytes_per_row": bytes_per_row,
           "device": torch.cuda.get_device_name(0), **gpu_info(), "cases": res}
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    idx.close()


if __name__ == "__main__":
    main()
