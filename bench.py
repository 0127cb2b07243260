#!/usr/bin/env python
"""bench.py — QPS @ 99% recall@10 of the diskann index-scan hot path on B200.

A "step" is one pass of the hot path (amrescan preparation -> StreamingDiskANN beam search over
SBQ codes -> exact f32 rerank window) over one batch of 4096 synthetic queries against a
50M x 768-d index resident in HBM (BASELINE.json configs[2], the configuration the metric is
quoted on; 176 GB of the 180).  `--n 1000000 --batch 1024` is configs[1]; a short configs[1] run is
also attached to the default line under "secondary".  Weak scaling: every rank holds a full
replica and its own batch; the only collective is the final gather of the top-k rows.

  python bench.py [--gpus N --steps K --warmup W]          our CUDA path (one JSON line)
  python bench.py --impl reference ...                     the CPU path (oracle port) on host cores
  python bench.py ... --dump-outputs DIR                    also the last timed step's outputs, DIR/<name>.npy

`value`  : whole-job queries/s with the query batch already in HBM (device-timed, max over ranks)
`e2e`    : the same metric through the host-buffer C-ABI call (dann_search_batch): pinned host
           queries in, (tid, dist) rows out, H2D/D2H inside the timed region
`roofline`: the beam-search kernel (dominant kernel) against the measured HBM peak
`cpu_baseline`: the CPU oracle timed on a bounded sample on this box's host cores
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the tree as it found it (it may be read-only)

import numpy as np  # noqa: E402


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=50_000_000)
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--batch", type=int, default=0, help="queries per GPU per step (0 = 4096 at >= 10M nodes, else 1024)")
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--data", default="lowrank", choices=["lowrank", "gaussian"])
    ap.add_argument("--bits", type=int, default=0, help="SBQ bits/dim (0 = reference default)")
    ap.add_argument("--L", type=int, default=0, help="fix search_list_size (0 = sweep for 99%% recall)")
    ap.add_argument("--rescore", type=int, default=0)
    ap.add_argument("--target-recall", type=float, default=0.99)
    ap.add_argument("--cpu-sample", type=int, default=0, help="queries in the CPU-baseline sample (0 = auto)")
    ap.add_argument("--sweep", action="store_true", help="print the whole recall/QPS sweep to stderr")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--parity-queries", type=int, default=256)
    ap.add_argument("--no-secondary", action="store_true", help="skip the attached configs[1] (1M x 768, batch 1024) run")
    ap.add_argument("--mode", default="batch", choices=["batch", "scan"],
                    help="scan: per-row latency of the operator surface (rescan + gettuple x k) instead of batch QPS")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path returned in its last step as DIR/<name>.npy (float32/float64)")
    a = ap.parse_args()
    if a.dump_outputs and a.mode == "scan":
        ap.error("--dump-outputs covers the batch path (--mode batch) and --impl reference")
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if not a.batch:
        a.batch = 4096 if a.n >= 10_000_000 else 1024
    return a


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# The contract is ONE JSON line on stdout.  Libraries print there too (NCCL's version banner, for one),
# so fd 1 is pointed at stderr for the whole run and only emit() writes to the real stdout.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(line: dict):
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, arrays: dict):
    """--dump-outputs: each array as out_dir/<name>.npy, integers as float64 (exact below 2**53; an empty tid slot,
    ~0 as int64, reads -1).  All arrays share their leading (query) axis; when they would exceed DUMP_LIMIT bytes in
    all, the same fixed, seeded sample of queries is kept in each and its indices are written as rows.npy."""
    arrays = {k: np.asarray(v).astype(np.float32 if np.asarray(v).dtype == np.float32 else np.float64)
              for k, v in arrays.items()}
    nq = next(iter(arrays.values())).shape[0]
    room = DUMP_LIMIT - 4096 * (len(arrays) + 1)                  # .npy headers
    if sum(a.nbytes for a in arrays.values()) > room:
        per_query = sum(a.nbytes for a in arrays.values()) // nq + 8
        rows = np.sort(np.random.default_rng(0).choice(nq, room // per_query, replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
        arrays["rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)
    log(f"[bench] outputs of the last timed step -> {out_dir}: " + ", ".join(f"{k}{list(a.shape)}" for k, a in arrays.items()))


# (search_list_size, rescore) in increasing cost (visits ~ L + rescore); recall is driven mostly by rescore
SWEEP = [(25, 50), (50, 50), (100, 50), (50, 100), (100, 100), (64, 150), (100, 150), (64, 200), (100, 200),
         (150, 200), (200, 200), (150, 250), (200, 250), (150, 300), (200, 300), (300, 300), (400, 400), (800, 400),
         (800, 800), (1000, 1000), (1600, 1000)]


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed regions (every ~5 ms through NVML;
    falls back to polling nvidia-smi when pynvml is unavailable)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.sm = []
        self.sm_max = None
        self.reasons = set()
        self._stop = threading.Event()
        self._t = None
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(gpu_index))
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
            self._nvml = pynvml
        except Exception:
            self._nvml = None

    @staticmethod
    def _physical_index(i):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[i])
            except Exception:
                return i
        return i

    def _sample_nvml(self):
        n = self._nvml
        self.sm.append(float(n.nvmlDeviceGetClockInfo(self._h, n.NVML_CLOCK_SM)))
        try:
            r = n.nvmlDeviceGetCurrentClocksEventReasons(self._h)
        except Exception:
            r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
        for name, bit in (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20),
                          ("hw_thermal_slowdown", 0x40), ("hw_power_brake_slowdown", 0x80)):
            if r & bit:
                self.reasons.add(name)

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout.strip()
        if out:
            f = [x.strip() for x in out.split(",")]
            self.sm.append(float(f[0]))
            self.sm_max = float(f[1])
            for i, name in enumerate(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]):
                if f[3 + i].lower().startswith("active"):
                    self.reasons.add(name)

    def _run(self):
        while not self._stop.is_set():
            try:
                if self._nvml:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            self._stop.wait(0.005)

    def __enter__(self):
        self._stop.clear()
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": ["no samples"], "samples": 0}
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2], "sm_min_mhz": sm[0], "sm_max_mhz": self.sm_max,
                "reasons": sorted(self.reasons), "samples": len(sm),
                "source": "nvml" if self._nvml else "nvidia-smi"}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# (search_list_size, rescore) in increasing cost (visits ~ L + rescore); recall is driven mostly by rescore, whose
# GUC maximum is 1000 (guc.rs:29-43).  The operating point is the first one whose recall@10 on the SELECTION SAMPLE
# (the first SEL queries of batch 0) reaches the target: both arms apply the same rule to the same queries, the
# CPU arm cannot afford whole 4096-query batches per point at 50M.
SWEEP_SMALL = [(25, 50), (50, 50), (100, 50), (50, 100), (100, 100), (64, 150), (100, 150), (64, 200), (100, 200),
               (150, 200), (200, 200), (150, 250), (200, 250), (150, 300), (200, 300), (300, 300), (400, 400), (800, 400),
               (800, 800), (1000, 1000), (1600, 1000)]
SWEEP_LARGE = [(200, 300), (300, 400), (400, 600), (600, 600), (600, 800), (800, 800), (800, 1000), (1000, 1000),
               (1500, 1000), (2000, 1000), (3000, 1000)]
SEL = 512


def sweep_points(args, n=None):
    if args.L:
        return [(args.L, args.rescore or 50)]
    return SWEEP_LARGE if (n or args.n) >= 10_000_000 else SWEEP_SMALL


def recall_at_k(tid, truth_nodes, k):
    """tid [B,k] uint64 -> fraction of the exact top-k found."""
    from tools.fixture import tid_to_node
    nodes = tid_to_node(tid)
    hits = 0
    for b in range(tid.shape[0]):
        hits += len(set(nodes[b].tolist()) & set(truth_nodes[b].tolist()))
    return hits / (tid.shape[0] * k)


def workload_name(n, dim, data, bits, batch, k):
    cfg = "configs[2]" if n >= 10_000_000 else "configs[1]"
    return (f"{cfg}: {n}x{dim}-d {data} ('Cohere-shape' synthetic) SBQ {bits}-bit diskann index in HBM, "
            f"batch={batch} queries/GPU/step, k={k}")


def metric_name(n, dim):
    return f"QPS @ 99% recall@10, {n // 1_000_000}Mx{dim}-d SBQ diskann scan, k=10"


def cpu_latency(oracle, snap, qs, L, rescore, k):
    """Single-thread per-query latency of the CPU path (= one Postgres backend, BASELINE.md §3): p50 / p95 in ms."""
    lat = []
    for i in range(qs.shape[0]):
        t0 = time.perf_counter()
        oracle.scan_batch(snap, qs[i:i + 1], None, None, L, rescore, k, threads=1)
        lat.append((time.perf_counter() - t0) * 1e3)
    lat.sort()
    return {"queries": len(lat), "p50_ms": round(lat[len(lat) // 2], 3), "p95_ms": round(lat[min(len(lat) - 1, int(len(lat) * 0.95))], 3),
            "qps_1thread": round(1e3 * len(lat) / sum(lat), 1)}


def native_arm(oracle, snap, qs, L, rescore, k, threads, seconds):
    """Optional CPU arm (BASELINE.md §3): the same oracle source built with -march=native on this box (AVX-512 VPOPCNTDQ
    where the CPU has it) - NOT the reference's build flags (.cargo/config.toml: +avx2,+fma), reported beside them."""
    try:
        oracle.scan_batch(snap, qs[:8], None, None, L, rescore, k, threads=threads, native=True)      # builds the library
        t1, reps = time.perf_counter(), 0
        while True:
            oracle.scan_batch(snap, qs, None, None, L, rescore, k, threads=threads, native=True)
            reps += 1
            if time.perf_counter() - t1 > seconds or reps >= 20:
                break
        return {"value": reps * qs.shape[0] / (time.perf_counter() - t1), "unit": "queries/s", "cores": threads,
                "flags": "-O2 -march=native (not the reference's build flags)"}
    except Exception as e:
        return {"error": repr(e)}


def run_reference(args):
    """--impl reference: the reference's own CPU algorithm for this path on the box's host cores.
    The Rust/pgrx extension cannot be built in this image (no rustc/cargo/Postgres), so this is the oracle port
    (oracle/oracle.cpp, the reference's AVX2+FMA flag family), one host thread per usable core, on the same index,
    queries, k and operating-point rule as our arm.  This process never loads libdiskann_b200.so: the index fixture
    (SBQ codes + Vamana graph; the reference's serial build would take days at 50M) comes from a child process
    (tools/make_fixture.py) through files; torch on the GPU is used here only for untimed setup - regenerating the
    deterministic dataset chunks for the exact-kNN ground truth and for the heap rows the sampled scans rerank."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from oracle import oracle
    from pgvectorscale_b200.snapshot import COSINE, Snapshot, make_heap_tids
    from tools import fixture as fx
    oracle.build_lib()
    device = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(device)
    n, dim, B, k = args.n, args.dim, args.batch, args.k
    cores = fx.host_cores()
    threads = cores["effective"]
    prefix = os.path.join("/dev/shm" if os.path.isdir("/dev/shm") else "/tmp", f"dann_fx_{os.getpid()}")
    t0 = time.time()
    try:
        subprocess.run([sys.executable, os.path.join(ROOT, "tools", "make_fixture.py"), "--n", str(n), "--dim", str(dim),
                        "--data", args.data, "--bits", str(args.bits), "--device", str(device.index or 0), "--out", prefix],
                       check=True, stdout=sys.stderr)
        codes = np.load(prefix + "_codes.npy")
        nbrs = np.load(prefix + "_nbrs.npy")
        meta = np.load(prefix + "_meta.npz")
    finally:
        for suf in ("_codes.npy", "_nbrs.npy", "_meta.npz"):
            try:
                os.remove(prefix + suf)
            except OSError:
                pass
    bits, words = int(meta["bits"]), int(meta["words"])
    log(f"[bench/reference] fixture from the child process in {time.time() - t0:.1f}s")
    rows = fx.SparseRows(n, dim)
    snap = Snapshot(n=n, dim=dim, dim_index=dim, bits=bits, words=words, R=int(meta["R"]), distance_type=COSINE,
                    has_labels=False, count=n, mean=meta["mean"], m2=meta["m2"], codes=codes, nbrs=nbrs,
                    heap_tid=make_heap_tids(n), vectors=rows.arr, start_default=0, start_labels=None,
                    start_label_nodes=None, label_off=None, labels=None)
    # queries: batch 0 of rank 0 (operating point), then the timed sample
    sel = min(SEL, B)
    q0 = fx.gen_queries(B, 1, dim, args.data, device)[:sel]
    topk = fx.RunningTopK(q0, k)
    for c, s, e in fx.chunks(n):
        topk.add(fx.gen_chunk(c, e - s, dim, args.data, device), s)
    truth = topk.result()
    q0h = q0.cpu().numpy()
    chosen = None
    for (L, rescore) in sweep_points(args):
        rows.fill_from_generator(fx.oracle_rerank_rows(oracle, snap, q0h, L, rescore, k, threads), dim, args.data, device)
        tid, _, _, _ = oracle.scan_batch(snap, q0h, None, None, L, rescore, k, threads=threads)
        rec = recall_at_k(tid, truth, k)
        log(f"[bench/reference] sweep L={L} rescore={rescore}: recall@{k}={rec:.4f} on {sel} queries")
        chosen = (L, rescore, rec)
        if rec >= args.target_recall:
            break
    L, rescore, recall = chosen
    # bounded sample per step: sized from a probe so that one step is about a second of CPU work
    t1 = time.perf_counter()
    oracle.scan_batch(snap, q0h[:64], None, None, L, rescore, k, threads=threads)
    rate = 64 / (time.perf_counter() - t1)
    sample = args.cpu_sample or int(min(B, max(32, 2 ** int(np.log2(max(rate * 1.0, 32))))))
    nb = args.warmup + args.steps
    qs = fx.gen_queries(sample, nb, dim, args.data, device, rank=1000).cpu().numpy()   # its own query stream
    rows.fill_from_generator(fx.oracle_rerank_rows(oracle, snap, qs, L, rescore, k, threads), dim, args.data, device)
    for w in range(args.warmup):
        oracle.scan_batch(snap, qs[w * sample:(w + 1) * sample], None, None, L, rescore, k, threads=threads)
    t0 = time.perf_counter()
    for s in range(args.warmup, nb):
        res = oracle.scan_batch(snap, qs[s * sample:(s + 1) * sample], None, None, L, rescore, k, threads=threads)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        tid, dist_, count, stats = res
        dump_outputs(args.dump_outputs, {"tid": tid.view(np.int64), "dist": dist_, "count": count,
                                         "stats": np.stack([stats[f] for f in stats.dtype.names], 1)})
    qps = args.steps * sample / dt
    lat = cpu_latency(oracle, snap, qs[:16], L, rescore, k)
    native = native_arm(oracle, snap, qs[:sample], L, rescore, k, threads, 3.0)
    line = {
        "impl": "reference", "metric": metric_name(n, dim),
        "value": qps, "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u64 popcount + f32", "data": "synthetic",
        "config": {"workload": workload_name(n, dim, args.data, bits, B, k), "search_list_size": L, "rescore": rescore,
                   "recall_at_10": round(recall, 4), "recall_queries": sel,
                   "operating_point_rule": f"first sweep point with recall@10 >= {args.target_recall} on the first {sel} queries of batch 0",
                   "note": f"CPU arm: each step scans a bounded sample of {sample} queries of the workload; index fixture "
                           "built by a child process, libdiskann_b200.so is never mapped here"},
        "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": threads, "kind": "port", "cores_detail": cores,
                         "single_thread": lat, "march_native": native,
                         "sample": f"{args.steps} steps x {sample} queries, {threads} host threads "
                                   "(oracle/oracle.cpp, -O2 -mavx2 -mfma -mpopcnt)"},
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def run_ours(args, n, B, steps, warmup, device, rank, world, full=True, dump=None):
    """One measurement of our CUDA path on an n x dim index with B queries per GPU per step -> result dict (rank 0).
    dump: directory for the outputs of the last timed step (dump_outputs)."""
    import torch
    import torch.distributed as dist
    from pgvectorscale_b200 import diskann
    from pgvectorscale_b200.group import QueryShardGroup
    from tools import fixture as fx

    k, dim = args.k, args.dim
    local_rank = device.index or 0
    need_oracle = rank == 0 and not args.no_parity
    t0 = time.time()
    snap, idx, bst = fx.codes_and_graph(n, dim, args.data, args.bits, device, log=log, download_nbrs=need_oracle)
    nb = warmup + steps
    q_all = fx.gen_queries(B, nb, dim, args.data, device, rank=rank)
    torch.cuda.empty_cache()
    X = torch.empty((n, dim), dtype=torch.float32, device=device)       # the heap rows, borrowed by the index
    topk = fx.RunningTopK(q_all[:B], k)
    fx.fill_rows(X, n, dim, args.data, device, topk)
    truth = topk.result()
    del topk
    def checksum():        # bit patterns, 256K rows at a time (the int64 upcast of the whole table would be 286 GiB)
        acc = 0
        for _, s_, e_ in fx.chunks(n):
            acc = (acc + int(X[s_:e_].view(torch.int32).sum(dtype=torch.int64).item())) & 0xFFFFFFFFFFFFFFFF
        return acc
    chk0 = checksum()
    idx.set_vectors_device(X.data_ptr())
    rows_unchanged = chk0 == checksum()
    torch.cuda.empty_cache()
    t_fixture = time.time() - t0
    log(f"[bench] rank {rank}: n={n} fixture {t_fixture:.1f}s (build {bst['total_ms'] / 1e3:.1f}s), index in HBM "
        f"{idx.hbm_bytes / 1e9:.2f} GB, rows untouched by the load-time normalisation: {rows_unchanged}")

    stream = torch.cuda.Stream(device)       # search, rerank and the collective all run in this stream's order
    d_tid = torch.empty((B, k), dtype=torch.int64, device=device)
    d_dist = torch.empty((B, k), dtype=torch.float32, device=device)
    d_cnt = torch.empty(B, dtype=torch.int32, device=device)
    d_stats = torch.empty((B, 6), dtype=torch.int32, device=device)

    def run_device(qb, L, rescore):
        idx.search_batch_device(qb, k, L, rescore, d_tid, d_dist, d_cnt, d_stats, stream=stream.cuda_stream)

    # ---- operating point: first (L, rescore) of the sweep reaching the target recall on the selection sample
    sel = min(SEL, B)
    chosen = None
    sweep_log = []
    for (L, rescore) in sweep_points(args, n):
        run_device(q_all[:B], L, rescore)          # first run of a plan pays for workspace (re)allocation
        run_device(q_all[:B], L, rescore)
        torch.cuda.synchronize(device)
        tids = d_tid.cpu().numpy().view(np.uint64)
        rec, rec_sel = recall_at_k(tids, truth, k), recall_at_k(tids[:sel], truth[:sel], k)
        t = idx.last_batch_timing()
        sweep_log.append({"L": L, "rescore": rescore, "recall": round(rec, 4), "recall_selection_sample": round(rec_sel, 4),
                          "device_ms": round(t["total_ms"], 3), "qps_1gpu": round(B / t["total_ms"] * 1e3)})
        if args.sweep or rank == 0:
            log(f"[bench] sweep L={L} rescore={rescore}: recall@{k}={rec:.4f} ({rec_sel:.4f} on the first {sel}) device "
                f"{t['total_ms']:.2f} ms (search {t['search_ms']:.2f}, rerank {t['rerank_ms']:.2f}, retries {t['retries']})")
        if rec_sel >= args.target_recall and chosen is None:
            chosen = (L, rescore, rec, rec_sel)
            if not args.sweep:
                break
    if chosen is None:
        L, rescore = sweep_points(args, n)[-1]
        chosen = (L, rescore, sweep_log[-1]["recall"], sweep_log[-1]["recall_selection_sample"])
        log(f"[bench] WARNING: target recall {args.target_recall} not reached; reporting at L={L}")
    L, rescore, recall, recall_sel = chosen

    # ---- parity gate (BASELINE.md §3): identical TIDs vs the CPU oracle before any timing
    parity = None
    rows = None
    cores = fx.host_cores()
    threads = cores["effective"]
    if need_oracle:
        from oracle import oracle
        oracle.build_lib()
        ns = min(args.parity_queries, B)
        rows = fx.SparseRows(n, dim)
        snap.vectors = rows.arr
        qh = q_all[:ns].cpu().numpy()
        rows.fill_from_device(fx.oracle_rerank_rows(oracle, snap, qh, L, rescore, k, threads), X)
        run_device(q_all[:B], L, rescore)
        torch.cuda.synchronize(device)
        g_tid = d_tid[:ns].cpu().numpy().view(np.uint64)
        g_dist = d_dist[:ns].cpu().numpy()
        g_st = d_stats[:ns].cpu().numpy()
        otid, odist, _, ostats = oracle.scan_batch(snap, qh, None, None, L, rescore, k, threads=threads)
        same_ids = bool(np.array_equal(g_tid, otid))
        same_dist = bool(np.array_equal(g_dist.view(np.uint32), odist.view(np.uint32)))
        same_cnt = bool(np.array_equal(g_st[:, 0].astype(np.uint64), ostats["visits"].astype(np.uint64)) and
                        np.array_equal(g_st[:, 1].astype(np.uint64), ostats["d_quantized"].astype(np.uint64)))
        parity = {"queries": ns, "tids_identical": same_ids, "dist_bits_identical": same_dist, "counters_identical": same_cnt}
        log(f"[bench] parity vs oracle on {ns} queries: ids {same_ids}, dist bits {same_dist}, counters {same_cnt}")
        if not same_ids:
            raise SystemExit("parity FAILED: returned row ids differ from the CPU oracle; refusing to report a number")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    shard = QueryShardGroup(None, k, device)

    # ---- device-resident timed region: CUDA events on the stream the kernels run on --------------
    with torch.cuda.stream(stream):
        for w in range(warmup):
            run_device(q_all[w * B:(w + 1) * B], L, rescore)
            shard.gather_packed(d_tid, d_dist, B)
        launches0 = idx.kernel_launches
        search_ms = rerank_ms = prepare_ms = 0.0
        step_search_ms, step_retries = [], 0
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        clocks = ClockSampler(local_rank)
        gathered = None
        with clocks:
            ev0.record(stream)
            for s in range(warmup, nb):
                run_device(q_all[s * B:(s + 1) * B], L, rescore)
                gathered = shard.gather_packed(d_tid, d_dist, B)
                t = idx.last_batch_timing()
                search_ms += t["search_ms"]
                step_search_ms.append(round(t["search_ms"], 3))
                step_retries += int(t["retries"])
                rerank_ms += t["rerank_ms"]
                prepare_ms += t["prepare_ms"]
            ev1.record(stream)
            barrier()
        dev_ms = ev0.elapsed_time(ev1)
        launches = idx.kernel_launches - launches0
    # the gathered rows of the last step: rank r's block must be rank r's own result (checked on every rank)
    gather_ok = None
    if world > 1:
        gt, gd = gathered
        gather_ok = bool(torch.equal(gt[rank * B:(rank + 1) * B], d_tid) and
                         torch.equal(gd[rank * B:(rank + 1) * B].view(torch.int32), d_dist.view(torch.int32)))
    # counters of the last batch -> algorithmic bytes (SURVEY §8d): taken after timing
    st = d_stats.cpu().numpy().astype(np.float64)
    visits_q, dq_q = st[:, 0].mean(), st[:, 1].mean()

    # ---- end-to-end through the host-buffer C ABI ---------------------------------------------
    h_q = torch.empty((nb * B, dim), dtype=torch.float32).pin_memory()
    h_q.copy_(q_all)
    h_tid = torch.empty((B, k), dtype=torch.int64).pin_memory()
    h_dist = torch.empty((B, k), dtype=torch.float32).pin_memory()
    for w in range(warmup):
        idx.search_batch_ptrs(h_q[w * B:(w + 1) * B].data_ptr(), B, k, L, rescore, h_tid.data_ptr(), h_dist.data_ptr())
    barrier()
    with clocks:
        t0 = time.perf_counter()
        for s in range(warmup, nb):
            idx.search_batch_ptrs(h_q[s * B:(s + 1) * B].data_ptr(), B, k, L, rescore, h_tid.data_ptr(), h_dist.data_ptr())
            if world > 1:
                shard.gather_packed(h_tid.to(device, non_blocking=True), h_dist.to(device, non_blocking=True), B)
        barrier()
        e2e_s = time.perf_counter() - t0
    if dump and rank == 0:
        gt, gd = gathered
        out = {"tid": gt.cpu().numpy(), "dist": gd.cpu().numpy()}
        if world == 1:      # the per-query counters, and the host-buffer call's rows for the same last-step queries
            out.update(count=d_cnt.cpu().numpy(), stats=d_stats.cpu().numpy(), e2e_tid=h_tid.numpy(), e2e_dist=h_dist.numpy())
        dump_outputs(dump, out)

    # ---- max over ranks ---------------------------------------------------------------------
    tm = torch.tensor([dev_ms, e2e_s * 1e3, search_ms, rerank_ms], dtype=torch.float64, device=device)
    ok = torch.tensor([1 if gather_ok in (None, True) else 0], dtype=torch.int32, device=device)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    dev_ms, e2e_ms, search_ms_max, rerank_ms_max = tm.tolist()
    if world > 1 and int(ok.item()) != 1:
        raise SystemExit("gather check FAILED: a rank's block of the gathered rows differs from its own result")
    total_q = steps * B * world
    value = total_q / (dev_ms / 1e3)
    e2e_value = total_q / (e2e_ms / 1e3)

    if rank != 0:
        idx.close()
        return None

    # ---- roofline of the dominant kernel (beam search) ----------------------------------------
    peak, peak_src = measured_peak()
    code_bytes = idx.code_stride * 8
    nbr_bytes = 50 * 4                                                 # R = 50 ids per list (rows hold 64 slots)
    alg_bytes_q = dq_q * code_bytes + visits_q * nbr_bytes             # SURVEY §8d per-query search bytes
    alg_bytes_launch = alg_bytes_q * B
    search_avg_ms = search_ms / steps
    achieved = alg_bytes_launch / (search_avg_ms / 1e3) / 1e9
    rerank_bytes_launch = B * (rescore + k - 1 if rescore else 0) * dim * 4
    rerank_avg_ms = rerank_ms / steps
    # DRAM traffic of one search-kernel launch from the committed `ncu --set full` capture of the same operating
    # point (profiles/r02_traffic.json); null when the capture is for another configuration
    traffic = None
    try:
        for tj in json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json"))):
            if (tj.get("L"), tj.get("rescore"), tj.get("n"), tj.get("batch")) == (L, rescore, n, B):
                traffic = tj["dram_bytes_per_launch"]
    except Exception:
        pass
    tinfo = idx.last_batch_timing()
    roofline = {"kernel": "dann_search3_kernel (lean warp-per-query beam search)", "bound": "hbm", "achieved": round(achieved, 1),
                "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4), "traffic": traffic, "peak_source": peak_src,
                "alg_bytes_per_launch": int(alg_bytes_launch), "avg_launch_ms": round(search_avg_ms, 4),
                "timing": "CUDA events around the kernel on its launch stream (dann_last_batch_timing.search_ms), averaged over the timed steps",
                "launch_ms_per_step": step_search_ms, "growth_retries_in_timed_steps": step_retries,
                "per_query": {"visits": round(visits_q, 1), "d_quantized": round(dq_q, 1), "code_bytes": code_bytes,
                              "nbr_bytes_per_visit": nbr_bytes}}
    others = {"dann_rerank_kernel": {"alg_bytes_per_launch": int(rerank_bytes_launch),
                                     "avg_launch_ms": round(rerank_avg_ms, 4),
                                     "achieved_gbs": round(rerank_bytes_launch / max(rerank_avg_ms, 1e-9) / 1e6, 1),
                                     "frac": round(rerank_bytes_launch / max(rerank_avg_ms, 1e-9) / 1e6 / peak, 4)},
              "dann_prepare_kernel": {"avg_launch_ms": round(prepare_ms / steps, 4)}}

    # ---- stand-alone SBQ-distance kernel (the metric's named kernel) ---------------------------
    if full:
        try:
            npairs = 64 * 1024 * 1024 if n >= 500_000 else 4 * 1024 * 1024
            g = torch.Generator(device=device)
            g.manual_seed(1)
            with torch.cuda.stream(stream):
                pn = torch.randint(0, n, (npairs,), generator=g, device=device, dtype=torch.int32)
                pq = torch.randint(0, B, (npairs,), generator=g, device=device, dtype=torch.int32)
                qc = torch.empty((B, idx.code_stride), dtype=torch.int64, device=device)
                idx.prepare_queries(q_all[:B].contiguous(), None, qc)
                out = torch.empty(npairs, dtype=torch.int32, device=device)
                for _ in range(3):
                    idx.sbq_distance(qc, pq, pn, out, stream=stream.cuda_stream)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize(device)
                reps = 5
                a.record(stream)
                for _ in range(reps):
                    idx.sbq_distance(qc, pq, pn, out, stream=stream.cuda_stream)
                b.record(stream)
                torch.cuda.synchronize(device)
            ms = a.elapsed_time(b) / reps
            sb = npairs * (code_bytes + 12)
            others["dann_sbq_distance_kernel"] = {"npairs": npairs, "alg_bytes_per_launch": sb, "avg_launch_ms": round(ms, 4),
                                                  "achieved_gbs": round(sb / ms / 1e6, 1), "frac": round(sb / ms / 1e6 / peak, 4)}
            del pn, pq, out
        except Exception as e:  # the headline must not die on the side measurement
            others["dann_sbq_distance_kernel"] = {"error": str(e)}

    # ---- CPU baseline: the oracle port on this box's cores, bounded sample ------------------------
    cpu = None
    if need_oracle and world == 1:
        from oracle import oracle
        probe = q_all[:64].cpu().numpy()
        t1 = time.perf_counter()
        oracle.scan_batch(snap, probe, None, None, L, rescore, k, threads=threads)       # rows are resident: parity sample
        rate = 64 / (time.perf_counter() - t1)
        sample = args.cpu_sample or int(min(B, max(64, 2 ** int(np.log2(max(rate * 4.0, 64))))))
        qs = fx.gen_queries(sample, 1, dim, args.data, device, rank=2000).cpu().numpy()
        rows.fill_from_device(fx.oracle_rerank_rows(oracle, snap, qs, L, rescore, k, threads), X)
        t1 = time.perf_counter()
        reps = 0
        while True:
            oracle.scan_batch(snap, qs, None, None, L, rescore, k, threads=threads)
            reps += 1
            if time.perf_counter() - t1 > (12.0 if full else 5.0) or reps >= 20:
                break
        cpu_qps = reps * sample / (time.perf_counter() - t1)
        lat = cpu_latency(oracle, snap, qs[:16 if full else 8], L, rescore, k)
        cpu = {"value": cpu_qps, "unit": "queries/s", "cores": threads, "kind": "port", "cores_detail": cores,
               "single_thread": lat, "march_native": native_arm(oracle, snap, qs, L, rescore, k, threads, 4.0 if full else 2.0),
               "sample": f"{reps} x {sample} queries of the same workload, {threads} host threads "
                         f"(oracle/oracle.cpp, -O2 -mavx2 -mfma -mpopcnt)"}

    # ---- the operator surface north_star keeps (scan.rs:336-405): amrescan + k x amgettuple, one scan at a time -----
    operator = None
    if need_oracle and world == 1:
        try:
            from oracle import oracle
            from tools import scan_latency
            nsc = min(40 if full else 24, ns)       # the parity sample's queries: their rerank rows are resident
            operator = scan_latency.measure(idx, snap, oracle, q_all[:nsc].cpu().numpy(), L, rescore, k, warm=8, both=False)
            log(f"[bench] operator surface: scan of {k} rows p50 {operator['gettuple']['scan_of_k_rows_ms']['p50']} ms "
                f"(CPU oracle, one thread: {operator['cpu_oracle_single_thread_ms']['p50']} ms), rows identical: "
                f"{operator['parity']['rows_identical']}")
        except Exception as e:  # the headline must not die on the side measurement
            operator = {"error": repr(e)}

    plan = idx.last_search_plan() if hasattr(idx, "last_search_plan") else None
    line = {
        "metric": metric_name(n, dim),
        "value": value, "unit": "queries/s", "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": dev_ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u64 popcount + f32", "data": "synthetic",
        "config": {"workload": workload_name(n, dim, args.data, snap.bits, B, k),
                   "search_list_size": L, "rescore": rescore, "recall_at_10": round(recall, 4),
                   "recall_at_10_selection_sample": round(recall_sel, 4),
                   "operating_point_rule": f"first sweep point with recall@10 >= {args.target_recall} on the first {sel} queries of batch 0",
                   "parallelism": f"query-shard x{world} (replicated index, one packed gather of the top-k rows on the search stream)",
                   "l2_policy": f"index {idx.hbm_bytes / 1e9:.2f} GB >> 126 MB L2, random gathers, distinct queries every step",
                   "search_kernel": "dann_search3_kernel (lean warp-per-query; DANN_SEARCH_KERNEL=2 selects the round-1 two-warp kernel)",
                   "search_plan": plan,
                   "index_fixture": "dann_build_graph: GPU batch Vamana over SBQ codes (R=50, L_build=100, alpha=1.2), "
                                    "the reference's build algorithm with batched insertion",
                   "fixture_seconds": round(t_fixture, 1)},
        "recall_sweep": sweep_log,
        "parity": parity,
        "gather_check": gather_ok,
        "e2e": {"value": e2e_value, "unit": "queries/s", "h2d_bytes_per_step": B * dim * 4,
                "d2h_bytes_per_step": B * k * 12, "ms_per_step": e2e_ms / steps},
        "gpu_launches": int(launches),
        "roofline": roofline,
        "kernels": others,
        "cpu_baseline": cpu,
        "operator": operator,
        "clocks": clocks.summary(),
    }
    idx.close()
    del X
    torch.cuda.empty_cache()
    return line


def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)

    if args.mode == "scan":
        from tools import scan_latency
        line = scan_latency.run(args, device, log)
        if rank == 0:
            emit(line)
        return

    secondary = None
    if world == 1 and args.n >= 10_000_000 and not args.no_secondary:
        # configs[1] (1M x 768-d, batch 1024) first, while HBM is empty; a shorter run, attached as a secondary key
        try:
            s = run_ours(args, 1_000_000, 1024, min(args.steps, 10), min(args.warmup, 3), device, rank, world, full=False)
            secondary = {kk: s[kk] for kk in ("metric", "value", "unit", "ms_per_step", "e2e", "roofline", "parity", "cpu_baseline", "operator")}
            secondary["config"] = {kk: s["config"][kk] for kk in ("workload", "search_list_size", "rescore", "recall_at_10")}
        except SystemExit:
            raise
        except Exception as e:
            secondary = {"error": repr(e)}
    line = run_ours(args, args.n, args.batch, args.steps, args.warmup, device, rank, world, dump=args.dump_outputs)
    if rank == 0:
        if secondary is not None:
            line["secondary"] = secondary
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
