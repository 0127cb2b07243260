"""bench.py --mode scan: latency of the OPERATOR SURFACE the reference exposes - one backend, one scan at a time:
amrescan + k x amgettuple (scan.rs:336-405) through dann_scan_rescan / dann_scan_gettuple - next to the CPU oracle
doing the same single-threaded (BASELINE.md §3 "CPU-1: p50/p95").  The default amgettuple makes one host
synchronisation per row; the step-by-step flavour (DANN_SCAN_FUSED=0) is timed beside it.  bench.py's default run
calls measure() on the loaded 50M index and attaches the result as "operator".

The index is the bench fixture (default here: configs[1], 1M x 768; pass --n for larger).  One JSON line."""
from __future__ import annotations

import os
import time

import numpy as np


def _pct(v, p):
    v = sorted(v)
    return round(v[min(len(v) - 1, int(len(v) * p))], 4)


def measure(idx, snap, oracle, q, L, rescore, k, warm=20, both=True):
    """amrescan + k x amgettuple, one scan at a time, for every row of q (host array; the heap rows the oracle reranks for
    these queries must already be resident in snap.vectors) -> dict.  `both`: also time DANN_SCAN_FUSED=0 (one launch
    and one synchronisation per step instead of one synchronisation per row)."""
    nq = q.shape[0]

    def one_pass(fused):
        os.environ["DANN_SCAN_FUSED"] = "1" if fused else "0"
        sc = idx.begin_scan()
        first, per_row, whole, got = [], [], [], []
        for i in range(nq):
            t0 = time.perf_counter()
            sc.rescan(q[i], None, L, rescore)
            r = sc.gettuple()
            t1 = time.perf_counter()
            out = [r]
            for _ in range(k - 1):
                out.append(sc.gettuple())
            t2 = time.perf_counter()
            if i >= warm:      # warm-up scans excluded
                first.append((t1 - t0) * 1e3)
                per_row.append((t2 - t1) * 1e3 / (k - 1))
                whole.append((t2 - t0) * 1e3)
            got.append([(x[0] << 16) | x[1] if x else 0xFFFFFFFFFFFFFFFF for x in out])
        sc.end()
        os.environ.pop("DANN_SCAN_FUSED", None)
        return {"rescan_plus_first_row_ms": {"p50": _pct(first, 0.5), "p95": _pct(first, 0.95)},
                "next_row_ms": {"p50": _pct(per_row, 0.5), "p95": _pct(per_row, 0.95)},
                "scan_of_k_rows_ms": {"p50": _pct(whole, 0.5), "p95": _pct(whole, 0.95)},
                "scans_per_s_one_backend": round(1e3 / (sum(whole) / len(whole)), 1)}, np.array(got, dtype=np.uint64)

    res_fused, tids_f = one_pass(True)
    res_steps, tids_s = one_pass(False) if both else (None, None)
    # CPU: the oracle, one query at a time on one thread (= one Postgres backend)
    lat = []
    otid = np.zeros((nq, k), np.uint64)
    for i in range(nq):
        t0 = time.perf_counter()
        t, _, _, _ = oracle.scan_batch(snap, q[i:i + 1], None, None, L, rescore, k, threads=1)
        if i >= warm:
            lat.append((time.perf_counter() - t0) * 1e3)
        otid[i] = t[0]
    out = {"scans": nq - warm, "search_list_size": L, "rescore": rescore, "k": k,
           "gettuple": res_fused,
           "cpu_oracle_single_thread_ms": {"p50": _pct(lat, 0.5), "p95": _pct(lat, 0.95),
                                           "scans_per_s_one_backend": round(1e3 / (sum(lat) / len(lat)), 1)},
           "parity": {"rows_identical": bool(np.array_equal(tids_f, otid))}}
    if both:
        out["gettuple_step_by_step (DANN_SCAN_FUSED=0)"] = res_steps
        out["parity"]["step_by_step_rows_identical"] = bool(np.array_equal(tids_s, otid))
    return out


def run(args, device, log):
    import torch
    from oracle import oracle
    from pgvectorscale_b200 import diskann  # noqa: F401
    from tools import fixture as fx
    oracle.build_lib()
    n = args.n if args.n < 10_000_000 or os.environ.get("DANN_SCAN_BENCH_FULL") else 1_000_000
    dim, k = args.dim, args.k
    L, rescore = (args.L or 150), (args.rescore or 250)
    snap, idx, _ = fx.codes_and_graph(n, dim, args.data, args.bits, device, log=log, download_nbrs=True)
    X = torch.empty((n, dim), dtype=torch.float32, device=device)
    fx.fill_rows(X, n, dim, args.data, device)
    idx.set_vectors_device(X.data_ptr())
    nq = args.warmup + args.steps          # one step = one scan
    q = fx.gen_queries(nq, 1, dim, args.data, device).cpu().numpy()
    rows = fx.SparseRows(n, dim)
    snap.vectors = rows.arr
    rows.fill_from_device(fx.oracle_rerank_rows(oracle, snap, q, L, rescore, k, fx.host_cores()["effective"]), X)
    m = measure(idx, snap, oracle, q, L, rescore, k, warm=args.warmup)
    line = {"metric": f"index-scan operator latency (amrescan + {k} x amgettuple), {n}x{dim}-d SBQ diskann index",
            "mode": "scan", "unit": "ms", "higher_is_better": False, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
            "value": m["gettuple"]["scan_of_k_rows_ms"]["p50"],
            "config": {"workload": f"{n}x{dim}-d, one scan at a time, search_list_size={L}, rescore={rescore}, k={k}, {args.steps} timed scans"}}
    line.update({kk: v for kk, v in m.items() if kk not in ("scans", "search_list_size", "rescore", "k")})
    idx.close()
    return line
