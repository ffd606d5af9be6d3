#!/usr/bin/env python
"""Benchmark of the dense-retrieval hot path: exact top-100 queries/sec over a CAsT-sized
38.6M x 768 synthetic collection (BASELINE.json `metric`), one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # our arm
    torchrun ... bench.py --gpus N --steps K --warmup W            # N > 1 (driver launches this)
    python bench.py --impl reference [...]                         # CPU reference arm
    python bench.py [...] --dump-outputs DIR                       # also write the last step's results

A "step" is one search of the 173-query CAsT-19 batch over the whole collection.  The collection
(fixed total size, so scaling is "strong") is row-sharded over the N ranks and resident in HBM;
each rank searches its shard with the fused tcgen05 score+select kernel, the [nq,k] (score,id) lists
are all-gathered over NCCL and merged on device.  `value` times the device-resident call (queries
and results in HBM, CUDA events on the engine's stream, max over ranks); `e2e` times the public
host-buffer API (pinned H2D of the queries, D2H of the result inside the timed region).
One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_CAST = 38_636_520          # MS MARCO 8,841,823 + TREC-CAR 29,794,697 passages (preprocess_cast19.py)
NQ = 173                     # CAsT-19 judged query batch (BASELINE.json configs)
TOPK = 100                   # reference default --top_n (run_convdr_inference.py:316-319)
D = 768
METRIC = "exact top-100 queries/sec over 38M x 768"
UNIT = "queries/s"
BYTES_STREAMED_PER_ROW = D * 2      # bf16 shadow row read by the scoring kernel
BYTES_ALGO_FP32_PER_ROW = D * 4     # SURVEY §8(d) B_algo = 3072 * N (fp32 collection read once)


# BASELINE.json `configs` (SURVEY.md §8: C1..C5).  c4 is the headline metric and the default.
CONFIGS = {
    "c1": dict(rows=100_000, nq=173, k=100, name="configs[0]: 100k x 768, 173 queries, top-100"),
    "c2": dict(rows=8_841_823, nq=173, k=1000, name="configs[1]: MS MARCO-sized 8.8M x 768, 173 queries, top-1000"),
    "c3": dict(rows=11_100_000, nq=5571, k=100, name="configs[2]: OR-QuAC-sized 11.1M x 768, 5,571 queries, top-100"),
    "c4": dict(rows=N_CAST, nq=NQ, k=TOPK, name="configs[3]: CAsT-sized 38.6M x 768, 173 queries, top-100"),
    "c5": dict(rows=N_CAST, nq=16384, k=1000, name="configs[4]: batch sweep 1..16,384 queries x 38.6M x 768, top-1000"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="c4", choices=sorted(CONFIGS),
                    help="BASELINE.json config: sets --rows/--nq/--k (c5 runs the batch-size sweep)")
    ap.add_argument("--sweep-nq", default="1,2,4,8,16,32,64,128,173,256,512,1024,2048,4096,8192,16384")
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b2f", choices=["b2f", "reference"])
    ap.add_argument("--rows", type=int, default=N_CAST, help="total collection rows (default: CAsT size)")
    ap.add_argument("--nq", type=int, default=NQ)
    ap.add_argument("--k", type=int, default=TOPK)
    ap.add_argument("--path", default="auto")
    ap.add_argument("--growth", type=int, default=0, help="phase growth factor override (0 = engine default)")
    ap.add_argument("--variant", type=int, default=0,
                    help="tensor engine variant: 0 auto (QS up to 208 queries per pass, TS above), 1 QS with resident "
                         "queries, 2 TS, 3 QS")
    ap.add_argument("--data", default="iso", choices=["iso", "aniso"],
                    help="synthetic rows: iso = isotropic unit-norm (BASELINE.json), aniso = norm 28 with a common "
                         "mean component, cos(p,p') ~ 0.9 (LayerNorm-like ANCE embeddings)")
    ap.add_argument("--tighten", type=int, default=-1, help="-1 engine default, 0 off, >0 refresher pause in ns")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"],
                    help="N > 1: result exchange through the engine's peer-memory kernels (default) or ncclAllGather")
    ap.add_argument("--balance", type=int, default=0,
                    help="N > 1: 1 = size each rank's shard by its measured local search speed (calibrated before "
                         "the timed region), 0 = equal shards")
    ap.add_argument("--opt", action="append", default=[], help="engine option key=value (A/B experiments)")
    ap.add_argument("--cpu-sample-rows", type=int, default=2_000_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-check", action="store_true")
    ap.add_argument("--no-oracle-check", action="store_true",
                    help="skip the two oracle legs of the untimed check (full-size fp64 truth, overflow protocol)")
    ap.add_argument("--inproc", type=int, default=1,
                    help="N > 1: 1 = rank 0 also measures the single-process layout (one index over all GPUs, "
                         "host buffers) after the main run and reports it under `inproc`")
    ap.add_argument("--sustain-seconds", type=float, default=2.0,
                    help="length of the extra back-to-back run reported under `sustained` (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the results of the last one to DIR/scores.npy (float32) and "
                         "DIR/ids.npy (float64), for output-for-output comparison of two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.config != "c4":
        c = CONFIGS[args.config]
        args.rows, args.nq, args.k = c["rows"], c["nq"], c["k"]
    return args


def metric_name(args):
    if args.config == "c4" and args.rows == N_CAST and args.k == TOPK:
        return METRIC
    return f"exact top-{args.k} queries/sec over {args.rows / 1e6:.1f}M x 768"


def measured_peaks():
    """(HBM GB/s, bf16 TFLOP/s sustained, source).  MEASURED_PEAKS.json is driver-written per pod."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            with open(path) as f:
                j = json.load(f)
            return float(j["hbm_gbs"]), float(j.get("bf16_tflops_sustained") or j.get("bf16_tflops") or 0.0), \
                "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, 1500.0, "fallback (B200_PROFILING.md)"


def ncu_traffic_per_launch(rows_per_launch: float, kernel: str = "umma_score_select_kernel"):
    """DRAM bytes (read + write) per launch of the dominant kernel, from the committed
    `ncu --set full` capture (profiles/ncu_summary.json: bytes per row of the captured launch) scaled
    to the rows one average launch of this run streams."""
    path = os.path.join(ROOT, "profiles", "ncu_summary.json")
    try:
        with open(path) as f:
            j = json.load(f)
            per_row = (j.get(kernel) or j["umma_score_select_kernel"])["dram_bytes_per_row"]
        return per_row * rows_per_launch
    except Exception:
        return None


DUMP_MAX_BYTES = 64_000_000


def dump_outputs(out_dir: str, D, I) -> None:
    """Write what a caller of the timed path receives, (D [nq,k] scores, I [nq,k] ids), as DIR/scores.npy
    (float32) and DIR/ids.npy (float64: exact for every id below 2**53).  When the files would exceed
    64 MB in all, only a fixed sample of query rows (seed 0, ascending) is written, and their indices go to
    DIR/query_rows.npy (float64)."""
    D = np.asarray(D, dtype=np.float32)
    I = np.asarray(I).astype(np.float64)
    nq, k = D.shape
    os.makedirs(out_dir, exist_ok=True)
    budget = DUMP_MAX_BYTES - 4096          # room for the .npy headers
    if nq * k * (4 + 8) > budget:
        max_rows = budget // (k * (4 + 8) + 8)
        rows = np.sort(np.random.default_rng(0).choice(nq, size=max_rows, replace=False))
        D, I = D[rows], I[rows]
        np.save(os.path.join(out_dir, "query_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "scores.npy"), D)
    np.save(os.path.join(out_dir, "ids.npy"), I)


class ClockSampler:
    """SM clock / power / throttle reasons of this rank's GPU, sampled through NVML from a thread
    every ~2 ms (the timed region of a multi-GPU run lasts tens of milliseconds: a 20 ms nvidia-smi loop
    cannot see it).  `mark()` brackets the timed region; only samples inside it are reported.  Falls back
    to an `nvidia-smi -lms` subprocess when pynvml is unavailable."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown"}
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index: int = 0):
        import threading
        self.device_index = device_index
        self.samples = []            # (t, sm_mhz, watts, reasons bitmask)
        self.t0 = self.t1 = None
        self._stop = threading.Event()
        self._thread = None
        self.sm_max = None
        self.proc = None
        self.tmp = None

    def _run(self, nv, h):
        while not self._stop.is_set():
            try:
                clk = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                mw = nv.nvmlDeviceGetPowerUsage(h)
                rs = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                self.samples.append((time.perf_counter(), float(clk), mw / 1000.0, int(rs)))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        import threading
        try:
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = self.device_index
            if vis:
                ids = [x for x in vis.split(",") if x.strip() != ""]
                if self.device_index < len(ids) and ids[self.device_index].strip().isdigit():
                    phys = int(ids[self.device_index])
            h = nv.nvmlDeviceGetHandleByIndex(phys)
            self.sm_max = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self._thread = threading.Thread(target=self._run, args=(nv, h), daemon=True)
            self._thread.start()
            return
        except Exception:
            self._thread = None
        try:
            self.tmp = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=self.tmp, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def mark(self):
        """Call right before and right after the timed region."""
        if self.t0 is None:
            self.t0 = time.perf_counter()
        else:
            self.t1 = time.perf_counter()

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self._thread is not None:
            self._stop.set()
            self._thread.join(timeout=2)
            sel = [x for x in self.samples if self.t0 is not None and self.t1 is not None and self.t0 <= x[0] <= self.t1]
            out["source"] = "nvml, 2 ms period, samples inside the timed region"
            if not sel:              # region shorter than one period: take the samples closest to it
                sel = sorted(self.samples, key=lambda x: abs(x[0] - (self.t0 or 0)))[:3]
                out["source"] = "nvml, nearest samples (timed region shorter than the sampling period)"
            if sel:
                mask = 0
                for x in sel:
                    mask |= x[3]
                out.update({"sm_mhz": statistics.median(x[1] for x in sel), "sm_mhz_min": min(x[1] for x in sel),
                            "sm_max_mhz": self.sm_max, "power_w_median": statistics.median(x[2] for x in sel),
                            "reasons": sorted(name for bit, name in self.REASONS.items() if mask & bit),
                            "samples": len(sel)})
            return out
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.tmp.flush()
        sm, mx, pw, reasons = [], [], [], set()
        with open(self.tmp.name) as f:
            for line in f:
                p = [x.strip() for x in line.split(",")]
                if len(p) < 9:
                    continue
                try:
                    clk, cmax, watts = float(p[1]), float(p[2]), float(p[3])
                except ValueError:
                    continue
                if watts < 250.0:      # idle sample (before / after the load): not "under load"
                    continue
                sm.append(clk); mx.append(cmax); pw.append(watts)
                for name, val in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], p[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        os.unlink(self.tmp.name)
        out["source"] = "nvidia-smi -lms 20, samples above 250 W"
        if sm:
            out["sm_mhz"] = statistics.median(sm)
            out["sm_mhz_min"] = min(sm)
            out["sm_max_mhz"] = max(mx)
            out["power_w_median"] = statistics.median(pw)
            out["reasons"] = sorted(reasons)
            out["samples"] = len(sm)
        return out


# ---------------------------------------------------------------------------------------------
# CPU legs (the only place bench.py touches oracle/)
# ---------------------------------------------------------------------------------------------
def cpu_reference_search(sample_rows: int, nq: int, k: int, steps: int, warmup: int, total_rows: int):
    """Times the FAISS-equivalent CPU restatement (oracle port: MKL/OpenBLAS sgemm + top-k) with all
    host threads on a bounded row sample of the same synthetic workload; q/s scaled to total_rows
    (exhaustive search is linear in N)."""
    from oracle import c_oracle, flat_ip
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    P = c_oracle.synth_block(0, sample_rows, seed=0, stream=0)
    Q = c_oracle.synth_block(0, nq, seed=0, stream=1)
    idx = flat_ip.IndexFlatIP(D, backend="torch", db_block=65536)
    idx.add(P)
    for _ in range(max(warmup, 1)):
        Dc, Ic = idx.search(Q, k)
    times = []
    for _ in range(max(steps, 1)):
        t0 = time.perf_counter()
        Dc, Ic = idx.search(Q, k)
        times.append(time.perf_counter() - t0)
    t = statistics.median(times)
    qps_sample = nq / t
    qps_full = qps_sample * sample_rows / total_rows
    return dict(value=qps_full, unit=UNIT, cores=cores, kind="port",
                sample=f"{nq} queries x {sample_rows} of {total_rows} rows (seed 0), median of {len(times)} "
                       f"searches, torch/MKL sgemm + top-k restatement of faiss.IndexFlatIP; q/s scaled by rows",
                ms_per_search_on_sample=t * 1e3), (P, Q, Dc, Ic)


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # A step = one search of the bounded row sample, ~1.3 s on 16 cores; exactly --steps of them are timed.
    # `ms_per_step` is what a step really took; `value` is the metric of the full workload (q/s scaled by rows:
    # exhaustive search is linear in N) and `ms_per_step_scaled_to_full_rows` the corresponding time of one
    # full-size search.
    steps = args.steps
    warmup = max(1, min(args.warmup, 10))
    sample_rows = min(args.cpu_sample_rows, args.rows)
    cb, (_, _, Dc, Ic) = cpu_reference_search(sample_rows, args.nq, args.k, steps, warmup, args.rows)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, Dc, Ic)
    line = {
        "impl": "reference", "metric": metric_name(args), "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup,
        "ms_per_step": cb["ms_per_search_on_sample"],
        "ms_per_step_scaled_to_full_rows": cb["ms_per_search_on_sample"] * args.rows / sample_rows,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"BASELINE.json {CONFIGS[args.config]['name']}: {args.rows}x768 fp32 collection, "
                               f"{args.nq} queries, top-{args.k}; CPU arm: each step searches a {sample_rows}-row "
                               f"sample, q/s scaled by rows"},
        "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------
def run_b2f_arm(args):
    import torch
    import torch.distributed as dist
    from convdr_b200 import FlatIPIndex, synth
    from convdr_b200.dist import ShardedFlatIP, shard_range

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the b2f engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL prints its version banner on stdout when the communicator comes up; stdout carries ONE
        # JSON line, so the banner goes to stderr (fd-level redirect, NCCL writes from C).
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", init_method="env://", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize(dev)
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    n_gpus = world

    index = FlatIPIndex(D, devices=[local_rank])
    index.set_option("path", args.path)
    index.set_option("profile", 1)
    if args.growth:
        index.set_option("growth", args.growth)
    index.set_option("umma_variant", args.variant)
    if args.tighten >= 0:
        index.set_option("tighten", args.tighten)
    for kv in args.opt:
        key, val = kv.split("=")
        index.set_option(key, int(val))
    data_norm, data_shift = (28.0, 443) if args.data == "aniso" else (1.0, 0)
    index.set_option("synth_mean_shift", data_shift)
    sharded = ShardedFlatIP(index=index)
    exchange = "none"
    if world > 1:
        exchange = "peer-memory kernels (CUDA IPC over NVLink)" if (args.exchange == "peer" and
                   sharded.enable_peer_exchange(args.nq, args.k)) else "ncclAllGather + merge kernel"
    t0 = time.perf_counter()
    lo, hi = sharded.add_synthetic(args.rows, seed=0, stream=0, norm=data_norm)
    build_s = time.perf_counter() - t0
    n_local = hi - lo

    q_host = synth.block(0, args.nq, seed=0, stream=1, norm=data_norm, mean_shift=data_shift)
    q_pin = torch.from_numpy(q_host).pin_memory()
    q_dev = q_pin.to(dev)
    nq, k = args.nq, args.k
    balance = None
    if world > 1 and args.balance:
        # Speed-weighted sharding: every search waits for the slowest GPU, and the GPUs of one box differ
        # by several percent under the power cap.  Calibrate (local search only, equal shards), then
        # rebuild the shards with shares proportional to the measured speeds.  Setup, not timed.
        from convdr_b200.dist import balance_weights
        times = sharded.gather_floats(sharded.local_seconds_per_search(q_dev, k))
        weights = balance_weights(times)
        sharded.reset()
        lo, hi = sharded.add_synthetic(args.rows, seed=0, stream=0, norm=data_norm, weights=weights)
        n_local = hi - lo
        balance = {"calibration_ms_equal_shards": [round(t * 1e3, 4) for t in times],
                   "shares": [round(w / sum(weights), 5) for w in weights]}
    stream = torch.cuda.ExternalStream(index.stream_ptr(0), device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    if args.config == "c5":
        run_sweep(args, index, sharded, stream, barrier, dev, world, rank, n_local, data_norm, data_shift, exchange)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    Dd = torch.empty((nq, k), dtype=torch.float32, device=dev)
    Id = torch.empty((nq, k), dtype=torch.int64, device=dev)

    def step_device():
        # The device-resident call is asynchronous: local search (b2f_search_device_async), and for N > 1
        # ONE NCCL all-gather of the packed lists + the merge kernel, all queued on the engine's stream.
        # The K searches of the timed region are queued back to back and settled once, inside the
        # region, by finish() (stream wait + overflow flags of every queued search).
        sharded.search_async(q_dev, k, Dd, Id)
        return Dd, Id

    # ---- device-resident timing ----
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()          # nvidia-smi needs ~100 ms to start: begin before the warm-up
    for _ in range(max(args.warmup, 3)):
        Dd, Id = step_device()
    sharded.finish()
    engine_path = int(index.stat("path"))
    barrier()
    index.reset_stats()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = score_ms = score_launches = score_rows = select_ms = 0.0
    sampler.mark()
    ev0.record(stream)
    for _ in range(args.steps):
        Dd, Id = step_device()
    clean = sharded.finish()     # waits for the stream and checks the overflow flags of every queued search
    if not clean:                # a list overflowed on some rank (never on this data): repeat synchronously, timed
        for _ in range(args.steps):
            Dd, Id = sharded.search(q_dev, k)
    ev1.record(stream)
    barrier()
    sampler.mark()
    dev_ms = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0:      # every rank holds the same merged result
        dump_outputs(args.dump_outputs, Dd.cpu().numpy(), Id.cpu().numpy())
    launches, score_ms, score_launches = index.stat("launches"), index.stat("score_ms"), index.stat("score_launches")
    score_rows, select_ms = index.stat("score_rows"), index.stat("select_ms")
    passes_per_search, qs_passes = index.stat("passes") / max(args.steps, 1), index.stat("qs_passes") / max(args.steps, 1)
    fallbacks_timed = index.stat("fallback_queries")
    per_rank = None
    if world > 1:   # where every rank spent the step: local scoring, selection, waiting for + merging the parts
        per_rank = {"score_ms_per_step": [round(v / args.steps, 4) for v in sharded.gather_floats(score_ms)],
                    "select_ms_per_step": [round(v / args.steps, 4) for v in sharded.gather_floats(select_ms)],
                    "exchange_wait_merge_ms_per_step": [round(v / args.steps, 4)
                                                        for v in sharded.gather_floats(index.stat("xchg_ms"))]}
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms_max = float(t.item())

    # ---- sustained: the same step queued back to back for >= --sustain-seconds, so that the board's power
    # governor is in steady state (the headline region at N = 8 lasts ~30 ms: a burst) ----
    sustained = None
    if args.sustain_seconds > 0:
        n_iter = int(min(max(args.sustain_seconds / max(dev_ms_max / args.steps * 1e-3, 1e-6), args.steps), 20000))
        samp2 = ClockSampler(local_rank)
        if rank == 0:
            samp2.start()
        barrier()
        samp2.mark()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record(stream)
        for _ in range(n_iter):
            step_device()
        sharded.finish()
        s1.record(stream)
        barrier()
        samp2.mark()
        ts = torch.tensor([s0.elapsed_time(s1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ts, op=dist.ReduceOp.MAX)
        sus_ms = float(ts.item())
        sustained = {"seconds": round(sus_ms * 1e-3, 3), "steps": n_iter, "value": nq * n_iter / (sus_ms * 1e-3),
                     "unit": UNIT, "ms_per_step": sus_ms / n_iter,
                     "streamed_gbs_per_gpu": n_local * BYTES_STREAMED_PER_ROW * n_iter / (sus_ms * 1e-3) / 1e9,
                     "clocks": samp2.stop() if rank == 0 else None}

    # ---- end-to-end timing through the public host-buffer API ----
    index.set_option("profile", 0)   # the per-launch CUDA events served the device-timed region; the e2e call runs bare
    q_pin_np = q_pin.numpy()       # the step's inputs live in pinned host memory (bench contract): uploaded from there
    def step_e2e():
        if world == 1:
            return index.search(q_pin_np, k)               # faiss-style call: numpy in, numpy out
        return sharded.search_host(q_pin_np, k, device=dev)
    for _ in range(2):
        De, Ie = step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        De, Ie = step_e2e()
    barrier()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t.item())

    # ---- correctness check of the timed configuration (not timed) ----
    check = None
    if not args.no_check:
        check = self_check(index, sharded, q_host, q_dev, Dd, Id, De, Ie, args, lo, hi, world, rank, dev)
        check["fallback_queries"] = fallbacks_timed      # of the timed searches (0: no list overflowed)

    stats_local = torch.tensor([score_ms, score_launches, score_rows, launches, select_ms], dtype=torch.float64, device=dev)
    if world > 1:
        stats_sum = stats_local.clone()
        dist.all_reduce(stats_sum, op=dist.ReduceOp.SUM)
    else:
        stats_sum = stats_local
    if rank == 0:
        peak, tensor_peak, peak_src = measured_peaks()
        sl = stats_local.tolist()
        # dominant kernel: umma_score_select_kernel.  Per launch: rows streamed * 1536 B (bf16 shadow).
        ms_per_launch = sl[0] / max(sl[1], 1.0)
        rows_per_launch = sl[2] / max(sl[1], 1.0)
        # which scoring kernel ran, and the MMA lanes it issues per passage row: QS puts the queries on the N side
        # (batch rounded up to 16), TS always issues M = 256 query lanes
        all_qs = qs_passes > 0 and qs_passes >= passes_per_search
        kernel_name = "umma_qs_score_select_kernel" if all_qs else (
            "umma_score_select_kernel" if qs_passes == 0 else "umma_score_select_kernel + umma_qs_score_select_kernel")
        lanes_issued = (-(-min(nq, 256) // 16) * 16) if all_qs else 256
        achieved = rows_per_launch * BYTES_STREAMED_PER_ROW / (ms_per_launch * 1e-3) / 1e9 if ms_per_launch > 0 else 0.0
        line = {
            "metric": metric_name(args), "value": nq * args.steps / (dev_ms_max * 1e-3), "unit": UNIT, "n_gpus": n_gpus,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": dev_ms_max / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "bf16 prefilter + f64-accumulated exact rescoring (fp32 out)", "data": "synthetic",
            "config": {
                "workload": f"BASELINE.json {CONFIGS[args.config]['name']}: {args.rows}x768 collection, {nq} queries, "
                            f"top-{k}, row-sharded over {n_gpus} GPU(s), {n_local} rows on rank 0",
                "l2_policy": "inputs larger than L2 (>= 7 GB streamed per GPU per step vs 126 MB L2); no flush needed",
                "engine_path": engine_path, "tensor_variant": args.variant, "data": args.data,
                "passes_per_search": passes_per_search, "qs_passes_per_search": qs_passes,
                "build_seconds": round(build_s, 2),
                "parallelism": f"shard{n_gpus}", "exchange": exchange, "balance": balance,
            },
            "roofline": {
                "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak if peak else None, "traffic": ncu_traffic_per_launch(rows_per_launch, kernel_name),
                "algorithmic_bytes_per_launch": rows_per_launch * BYTES_STREAMED_PER_ROW,
                "peak_source": peak_src, "kernel": kernel_name,
                "bytes_per_row_streamed": BYTES_STREAMED_PER_ROW,
                "achieved_fp32_equivalent": achieved * BYTES_ALGO_FP32_PER_ROW / BYTES_STREAMED_PER_ROW,
                "rows_per_launch": rows_per_launch, "ms_per_launch": ms_per_launch,
                "score_kernel_share_of_step": sl[0] / dev_ms_max if dev_ms_max else None,
                "select_kernels_ms_per_step": sl[4] / args.steps,
                "whole_step_streamed_gbs_per_gpu": n_local * BYTES_STREAMED_PER_ROW * args.steps / (dev_ms_max * 1e-3) / 1e9,
                # the same kernel against the tensor roofline: lanes issued per passage row (TS: always 256,
                # the cta_group::2 M granularity; QS: the batch rounded up to 16) vs the queries actually served
                "tensor": (lambda rps, passes: {
                    "lanes_issued_per_row": lanes_issued,
                    "issued_tflops": rps * 2 * lanes_issued * D / 1e12,
                    "useful_tflops": rps * 2 * (nq / passes) * D / 1e12,
                    "peak_bf16_sustained_tflops": tensor_peak,
                    "frac_issued": (rps * 2 * lanes_issued * D / 1e12) / tensor_peak if tensor_peak else None,
                })(rows_per_launch / (ms_per_launch * 1e-3) if ms_per_launch > 0 else 0.0, max(-(-nq // 256), 1)),
            },
            "e2e": {"value": nq * args.steps / e2e_s, "unit": UNIT,
                    "h2d_bytes_per_step": int(q_host.nbytes) * n_gpus,
                    "d2h_bytes_per_step": int(nq * k * 12) * n_gpus, "ms_per_step": e2e_s / args.steps * 1e3},
            "sustained": sustained,
            "per_rank": per_rank,
            "gpu_launches": int(stats_sum.tolist()[3]),
            "clocks": clocks,
            "check": check,
        }
        if n_gpus == 1 and not args.no_cpu_baseline:
            cb, _ = cpu_reference_search(min(args.cpu_sample_rows, args.rows), nq, k, 3, 1, args.rows)
            line["cpu_baseline"] = {kk: cb[kk] for kk in ("value", "unit", "cores", "kind", "sample")}
    if world > 1 and args.inproc:
        # The layout ConvDR's single-process driver actually uses (reference run_convdr_inference.py:324,
        # :355-368): ONE process, one index object over all GPUs (faiss.index_cpu_to_gpu_multiple with
        # shard=True), host buffers in and out.  Measured by rank 0 after the other ranks released their
        # shards; they wait on a gloo barrier (a host wait: an NCCL barrier would spin a kernel on their GPUs).
        ctl = dist.new_group(backend="gloo")
        index.set_option("keep_on_reset", 0)
        sharded.reset()
        torch.cuda.synchronize(dev)
        dist.barrier(group=ctl)
        if rank == 0:
            try:
                line["inproc"] = inproc_measure(args, world, q_host, De, Ie)
            except Exception as e:      # never lose the headline line to the extra measurement
                line["inproc"] = {"error": repr(e)[:300]}
        dist.barrier(group=ctl)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_sweep(args, index, sharded, stream, barrier, dev, world, rank, n_local, data_norm, data_shift, exchange):
    """BASELINE.json configs[4]: 1..16,384 queries against the resident 38.6M-row collection, top-1000 (what
    data/gen_ranking_data.py:541-567 consumes after --top_n 1000): the memory- to compute-bound crossover.
    Device-resident calls, CUDA events on the engine's stream, max over ranks, ~1 s per point."""
    import torch
    import torch.distributed as dist
    from convdr_b200 import synth
    peak, tensor_peak, peak_src = measured_peaks()
    nqs = [int(x) for x in args.sweep_nq.split(",")]
    k = args.k
    q_all = torch.from_numpy(synth.block(0, max(nqs), seed=0, stream=1, norm=data_norm, mean_shift=data_shift)).to(dev)
    points = []
    for nq in nqs:
        q = q_all[:nq].contiguous()
        Dd = torch.empty((nq, k), dtype=torch.float32, device=dev)
        Id = torch.empty((nq, k), dtype=torch.int64, device=dev)

        def timed(reps):
            barrier()
            index.reset_stats()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(reps):
                sharded.search_async(q, k, Dd, Id)
            clean = sharded.finish()
            e1.record(stream)
            barrier()
            t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item()) / reps, clean

        est, _ = timed(2)                                   # also the warm-up (workspace growth)
        reps = int(min(max(1000.0 / max(est, 1e-3), 3), 200))   # ~1 s per point, the same on every rank
        ms, clean = timed(reps)
        passes = index.stat("passes") / reps
        fb = sum(sharded.gather_floats(index.stat("fallback_queries")))
        streamed = n_local * BYTES_STREAMED_PER_ROW * passes / (ms * 1e-3) / 1e9
        useful_tf = 2.0 * nq * args.rows * D / (ms * 1e-3) / 1e12
        points.append({"nq": nq, "ms_per_search": ms, "queries_per_s": nq / (ms * 1e-3), "passes": passes,
                       "qs_passes": index.stat("qs_passes") / reps, "streamed_gbs_per_gpu": streamed,
                       "hbm_frac": streamed / peak, "useful_tflops_all_gpus": useful_tf,
                       "tensor_frac": useful_tf / (world * tensor_peak) if tensor_peak else None,
                       "bound": "hbm" if streamed / peak >= useful_tf / (world * tensor_peak) else "tensor",
                       "fallback_queries": fb, "clean": bool(clean), "reps": reps,
                       "sorted_desc": bool((Dd[:, 1:] <= Dd[:, :-1]).all().item())})
        if rank == 0:
            print(json.dumps(points[-1]), file=sys.stderr, flush=True)
    if args.dump_outputs and rank == 0:      # the last search of the last batch size
        dump_outputs(args.dump_outputs, Dd.cpu().numpy(), Id.cpu().numpy())
    if rank == 0:
        best = max(points, key=lambda p: p["queries_per_s"])
        cross = next((p["nq"] for p in points if p["bound"] == "tensor"), None)
        print(json.dumps({
            "metric": metric_name(args) + " (batch-size sweep)", "value": best["queries_per_s"], "unit": UNIT,
            "n_gpus": world, "steps": sum(p["reps"] for p in points), "warmup": 2 * len(points),
            "ms_per_step": best["ms_per_search"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "bf16 prefilter + f64-accumulated exact rescoring (fp32 out)", "data": "synthetic",
            "config": {"workload": CONFIGS["c5"]["name"] + f", row-sharded over {world} GPU(s)", "data": args.data,
                       "exchange": exchange, "peak_source": peak_src, "hbm_peak_gbs": peak,
                       "tensor_peak_tflops_sustained": tensor_peak,
                       "first_batch_size_where_the_tensor_fraction_exceeds_the_hbm_fraction": cross},
            "sweep": points}), flush=True)


def inproc_measure(args, n_dev, q_host, D_ref, I_ref):
    """index.search(queries, k) with host buffers on ONE FlatIPIndex sharded over n_dev devices of this process."""
    from convdr_b200 import FlatIPIndex
    data_norm, data_shift = (28.0, 443) if args.data == "aniso" else (1.0, 0)
    idx = FlatIPIndex(D, devices=list(range(n_dev)))
    idx.set_option("path", args.path)
    idx.set_option("umma_variant", args.variant)
    idx.set_option("synth_mean_shift", data_shift)
    cuts = [args.rows * i // n_dev for i in range(n_dev + 1)]
    idx.reserve(max(cuts[i + 1] - cuts[i] for i in range(n_dev)))
    for g in range(n_dev):
        for a in range(cuts[g], cuts[g + 1], 1 << 22):
            idx.add_synthetic(min(1 << 22, cuts[g + 1] - a), first_row=a, seed=0, stream=0, norm=data_norm,
                              shard=g, id_base=a)
    for _ in range(3):
        Di, Ii = idx.search(q_host, args.k)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        Di, Ii = idx.search(q_host, args.k)
    dt = (time.perf_counter() - t0) / args.steps
    out = {"layout": f"one process, one index, {n_dev} shards, host buffers (index.search)", "value": args.nq / dt,
           "unit": UNIT, "ms_per_step": dt * 1e3, "launches_per_search": idx.stat("launches"),
           "equals_one_process_per_gpu_result": bool(np.array_equal(Ii, I_ref) and np.array_equal(Di, D_ref))}
    idx.close()
    return out


def self_check(index, sharded, q_host, q_dev, Dd, Id, De, Ie, args, lo, hi, world, rank, dev):
    """Size-independent properties at the full benchmark size (no CPU pass over 38.6M rows):
    sortedness, device == host-API results, scores re-derived on the host from regenerated rows
    (fp64), and agreement of the tensor engine with the independent SIMT engine on a query subset."""
    import torch
    from convdr_b200 import synth
    out = {}
    Dn, In = Dd.cpu().numpy(), Id.cpu().numpy()
    out["sorted_desc"] = bool((np.diff(Dn, axis=1) <= 0).all())
    out["ids_in_range"] = bool(((In >= 0) & (In < args.rows)).all())
    out["host_api_equals_device_api"] = bool(np.array_equal(In, Ie) and np.array_equal(Dn, De))
    sel = [0, args.nq // 2, args.nq - 1]
    data_norm, data_shift = (28.0, 443) if args.data == "aniso" else (1.0, 0)
    rows = synth.rows(In[sel].reshape(-1).astype(np.uint64), seed=0, stream=0, norm=data_norm,
                      mean_shift=data_shift).reshape(len(sel), args.k, D)
    s64 = np.einsum("qd,qkd->qk", q_host[sel].astype(np.float64), rows.astype(np.float64))
    rel = np.abs(Dn[sel] - s64) / np.maximum(np.abs(s64), 1e-30)
    out["max_rel_err_vs_host_fp64_rescoring"] = float(rel.max())
    # independent engine on 4 queries (SIMT fp32 scan, no tensor cores, no bf16)
    index.set_option("path", "scan_f32")
    qsub = q_dev[:4].contiguous()
    Ds, Is = sharded.search(qsub, args.k)
    index.set_option("path", args.path)
    out["tensor_engine_equals_simt_engine_4q"] = bool(torch.equal(Is, Id[:4]) and torch.equal(Ds, Dd[:4]))
    if not args.no_oracle_check:
        out.update(oracle_check_full_size(args, q_host, Dn, In, rank))
        out.update(overflow_redo_check(args, world, rank, dev))
    return out


def oracle_check_full_size(args, q_host, Dn, In, rank, n_queries: int = 16):
    """Oracle parity AT THE BENCHMARK SIZE (VERDICT r1 next #3): the float64 ground truth of a query subset over
    the WHOLE collection, regenerated on the host block by block (oracle/flat_ip_c.c `oracle_topk_synth_f64`,
    all host threads; ~10-25 s for 38.6M rows), compared with the engine's (merged) answer by the parity
    comparator of BASELINE.json (ids identical except at ties within 1e-5 relative; scores within 1e-5).
    Unlike re-deriving the scores of the RETURNED rows, this detects a missed row.  Rank 0 computes it; every
    rank holds the same merged (D, I).  Not timed."""
    if rank != 0:
        return {}
    from oracle import c_oracle, flat_ip
    from convdr_b200 import synth
    data_norm, data_shift = (28.0, 443) if args.data == "aniso" else (1.0, 0)
    sel = sorted(set(np.linspace(0, args.nq - 1, min(n_queries, args.nq)).astype(int).tolist()))
    c_oracle.set_threads(os.cpu_count() or 1)      # torchrun exports OMP_NUM_THREADS=1; the other ranks are idle here
    t0 = time.perf_counter()
    Dt, It = c_oracle.topk_synth_f64(q_host[sel], args.k, 0, args.rows, seed=0, stream=0, norm=data_norm,
                                     mean_shift=data_shift)
    secs = time.perf_counter() - t0

    def score_of(qi, ids):
        r = synth.rows(np.asarray(ids).astype(np.uint64), seed=0, stream=0, norm=data_norm, mean_shift=data_shift)
        return r.astype(np.float64) @ q_host[sel[qi]].astype(np.float64)

    r = flat_ip.compare(Dn[sel], In[sel], Dt, It, score_of, rtol=1e-5)
    return {"oracle_queries": len(sel), "oracle_rows": args.rows, "oracle_violations": r["violations"],
            "oracle_exact_rows": r["exact_rows"], "oracle_tie_excused": r["tie_excused"],
            "oracle_max_rel_score_err": r["max_rel_score_err"], "oracle_seconds": round(secs, 1),
            "oracle_host_threads": os.cpu_count()}


def overflow_redo_check(args, world, rank, dev):
    """The overflow protocol at THIS world size (VERDICT r1 next #1): a small second collection whose last
    5000 rows are identical (more than a candidate list holds) is sharded over the ranks; a 173-query
    batch with two planted queries that rank those rows first makes the owning rank's lists overflow, the rows
    travel with the in-band marker, every rank repeats the exchange after the owner's exact re-run
    (convdr_b200/dist.py search_host's redo branch).  The result must equal the oracle's float64 truth."""
    from convdr_b200 import FlatIPIndex
    from convdr_b200.dist import ShardedFlatIP
    from oracle import c_oracle, flat_ip
    n = 60000
    P = c_oracle.synth_block(0, n, seed=41)
    P[55000:60000] = P[55000]
    qh = c_oracle.synth_block(0, 173, seed=3, stream=1)
    qh[7], qh[150] = P[55000], P[55000] * np.float32(0.5)
    idx2 = FlatIPIndex(D, devices=[dev.index])
    sh2 = ShardedFlatIP(index=idx2)
    if world > 1 and args.exchange == "peer":
        sh2.enable_peer_exchange(173, 100)
    sh2.add(P)
    idx2.reset_stats()
    if world > 1:
        Dh, Ih = sh2.search_host(qh, 100, device=dev)
    else:
        Dh, Ih = idx2.search(qh, 100)
    reran = sum(sh2.gather_floats(idx2.stat("fallback_queries")))
    ok = True
    if rank == 0:
        Dt, It = flat_ip.truth_fp64(qh, P, 100)
        score_of = lambda qi, ids: qh[qi].astype(np.float64) @ P[ids].astype(np.float64).T
        r = flat_ip.compare(Dh, Ih, Dt, It, score_of, rtol=1e-5)
        ok = r["violations"] == 0 and bool(np.array_equal(Ih[7], It[7]) and np.array_equal(Ih[150], It[150]))
    oks = sh2.gather_floats(1.0 if ok else 0.0)
    idx2.close()
    return {"overflow_redo_ok": bool(all(v > 0 for v in oks) and reran >= 2), "overflow_queries_rerun": reran}


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_b2f_arm(args)


if __name__ == "__main__":
    main()
