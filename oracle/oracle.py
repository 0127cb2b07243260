"""ctypes binding of the CPU oracle (oracle/liboracle.so).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  The product package never imports this module.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

INVALID_NODE = 0xFFFFFFFF
COSINE, L2, IP = 0, 1, 2


class _Snapshot(C.Structure):
    _fields_ = [
        ("n", C.c_uint32), ("dim", C.c_uint32), ("dim_index", C.c_uint32), ("bits", C.c_uint32),
        ("words", C.c_uint32), ("R", C.c_uint32), ("distance_type", C.c_int32),
        ("has_labels", C.c_int32), ("count", C.c_uint64),
        ("mean", C.c_void_p), ("m2", C.c_void_p), ("codes", C.c_void_p), ("nbrs", C.c_void_p),
        ("heap_tid", C.c_void_p), ("vectors", C.c_void_p),
        ("start_default", C.c_uint32), ("n_start_labels", C.c_uint32),
        ("start_labels", C.c_void_p), ("start_label_nodes", C.c_void_p),
        ("label_off", C.c_void_p), ("labels", C.c_void_p),
        ("storage_type", C.c_int32), ("index_vectors", C.c_void_p),
    ]


class _Stats(C.Structure):
    _fields_ = [("visits", C.c_uint64), ("d_quantized", C.c_uint64), ("candidates", C.c_uint64),
                ("d_full", C.c_uint64), ("stream_len", C.c_uint64)]


STATS_DTYPE = np.dtype([("visits", "<u8"), ("d_quantized", "<u8"), ("candidates", "<u8"),
                        ("d_full", "<u8"), ("stream_len", "<u8")])


def build_lib(force: bool = False) -> str:
    """Compile oracle/liboracle.so with the committed Makefile (gcc only)."""
    so = os.path.join(_HERE, "liboracle.so")
    src = [os.path.join(_HERE, f) for f in ("oracle.cpp", "oracle.h", "Makefile")]
    if force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in src):
        subprocess.run(["make", "-C", _HERE, "-B" if force else "-s"], check=True,
                       stdout=subprocess.DEVNULL)
    return so


def lib():
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(build_lib())
        _LIB.orc_hamming.restype = C.c_uint64
        _LIB.orc_distance.restype = C.c_float
        _LIB.orc_distance_avx2.restype = C.c_float
        _LIB.orc_distance_unoptimized.restype = C.c_float
        _LIB.orc_code_words.restype = C.c_uint32
        _LIB.orc_labels_normalize.restype = C.c_uint32
        _LIB.orc_binary_heap_script.restype = C.c_uint32
        _LIB.orc_scan.restype = C.c_uint32
        _LIB.orc_build.argtypes = [C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32,
                                   C.c_double, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32]
        _LIB.orc_build.restype = None
    return _LIB


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def hamming(a, b) -> int:
    a = np.ascontiguousarray(a, dtype=np.uint64)
    b = np.ascontiguousarray(b, dtype=np.uint64)
    return int(lib().orc_hamming(_p(a), _p(b), C.c_uint32(a.size)))


def distance(kind: int, x, y, impl: str = "emu") -> float:
    x, y = _f32(x), _f32(y)
    fn = {"emu": lib().orc_distance, "avx2": lib().orc_distance_avx2,
          "unoptimized": lib().orc_distance_unoptimized}[impl]
    return float(fn(C.c_int(kind), _p(x), _p(y), C.c_uint32(x.size)))


def preprocess_cosine(v):
    v = _f32(v).copy()
    lib().orc_preprocess_cosine(_p(v), C.c_uint32(v.size))
    return v


def code_words(dim: int, bits: int) -> int:
    return int(lib().orc_code_words(C.c_uint32(dim), C.c_uint32(bits)))


def train(vectors, bits: int):
    """vectors: [n, dim_index] already truncated / cosine-normalised. -> mean, m2, count"""
    v = _f32(vectors)
    n, dim = v.shape
    mean = np.zeros(dim, np.float32)
    m2 = np.zeros(dim, np.float32)
    cnt = C.c_uint64(0)
    lib().orc_train(_p(v), C.c_uint32(n), C.c_uint32(dim), C.c_uint32(bits), _p(mean), _p(m2),
                    C.byref(cnt))
    return mean, m2, int(cnt.value)


def quantize(v, bits: int, mean, m2, count: int):
    v = _f32(v)
    out = np.zeros(code_words(v.size, bits), np.uint64)
    mean, m2 = _f32(mean), _f32(m2)
    lib().orc_quantize(_p(v), C.c_uint32(v.size), C.c_uint32(bits), _p(mean), _p(m2),
                       C.c_uint64(count), _p(out))
    return out


def quantize_all(vectors, bits: int, mean, m2, count: int):
    v = _f32(vectors)
    out = np.zeros((v.shape[0], code_words(v.shape[1], bits)), np.uint64)
    mean, m2 = _f32(mean), _f32(m2)
    fn = lib().orc_quantize
    for i in range(v.shape[0]):
        fn(C.c_void_p(v[i].ctypes.data), C.c_uint32(v.shape[1]), C.c_uint32(bits), _p(mean),
           _p(m2), C.c_uint64(count), C.c_void_p(out[i].ctypes.data))
    return out


def labels_overlap(a, b) -> bool:
    a = np.ascontiguousarray(a, dtype=np.int16)
    b = np.ascontiguousarray(b, dtype=np.int16)
    return bool(lib().orc_labels_overlap(_p(a), C.c_uint32(a.size), _p(b), C.c_uint32(b.size)))


def labels_contains_intersection(self_, a, b) -> bool:
    s = np.ascontiguousarray(self_, dtype=np.int16)
    a = np.ascontiguousarray(a, dtype=np.int16)
    b = np.ascontiguousarray(b, dtype=np.int16)
    return bool(lib().orc_labels_contains_intersection(_p(s), C.c_uint32(s.size), _p(a),
                                                       C.c_uint32(a.size), _p(b), C.c_uint32(b.size)))


def labels_normalize(labels):
    a = np.ascontiguousarray(labels, dtype=np.int16).copy()
    n = lib().orc_labels_normalize(_p(a), C.c_uint32(a.size))
    return a[:n]


def binary_heap_script(ops):
    ops = np.ascontiguousarray(ops, dtype=np.int64)
    out = np.zeros(max(1, ops.size), np.int64)
    n = lib().orc_binary_heap_script(_p(ops), C.c_uint32(ops.size), _p(out))
    return out[:n]


def build_graph(codes, R: int, search_list_size: int = 100, max_alpha: float = 1.2,
                label_off=None, labels=None):
    """Serial Vamana build over SBQ codes. -> nbrs[n,R], start_default, start_labels, start_nodes"""
    codes = np.ascontiguousarray(codes, dtype=np.uint64)
    n, words = codes.shape
    has_labels = label_off is not None
    nbrs = np.full((n, R), INVALID_NODE, np.uint32)
    cap = 65536
    sl = np.zeros(cap, np.int16)
    sn = np.zeros(cap, np.uint32)
    sd = C.c_uint32(INVALID_NODE)
    ns = C.c_uint32(0)
    if has_labels:
        label_off = np.ascontiguousarray(label_off, dtype=np.uint32)
        labels = np.ascontiguousarray(labels, dtype=np.int16)
    lib().orc_build(n, words, _p(codes), R, search_list_size, max_alpha, int(has_labels),
                    _p(label_off) if has_labels else None, _p(labels) if has_labels else None,
                    _p(nbrs), C.addressof(sd), _p(sl), _p(sn), C.addressof(ns), cap)
    k = int(ns.value)
    return nbrs, int(sd.value), sl[:k].copy(), sn[:k].copy()


@dataclass
class _Keep:
    arrays: list


def _snapshot_struct(s):
    """s: any object with the attribute names of pgvectorscale_b200.snapshot.Snapshot."""
    keep = []

    def arr(a, dt):
        if a is None:
            return None
        a = np.ascontiguousarray(a, dtype=dt)
        keep.append(a)
        return C.c_void_p(a.ctypes.data)

    st = _Snapshot()
    st.n, st.dim, st.dim_index, st.bits = s.n, s.dim, s.dim_index, s.bits
    st.words, st.R = s.words, s.R
    st.distance_type = s.distance_type
    st.has_labels = int(s.has_labels)
    st.count = s.count
    st.mean = arr(s.mean, np.float32)
    st.m2 = arr(s.m2 if s.m2 is not None else np.zeros(s.dim_index, np.float32), np.float32)
    st.codes = arr(s.codes, np.uint64)
    st.nbrs = arr(s.nbrs, np.uint32)
    st.heap_tid = arr(s.heap_tid, np.uint64)
    st.vectors = arr(s.vectors, np.float32)
    st.start_default = s.start_default
    st.n_start_labels = 0 if s.start_labels is None else len(s.start_labels)
    st.start_labels = arr(s.start_labels, np.int16)
    st.start_label_nodes = arr(s.start_label_nodes, np.uint32)
    st.label_off = arr(s.label_off, np.uint32)
    st.labels = arr(s.labels, np.int16)
    st.storage_type = int(getattr(s, "storage_type", 0) or 0)
    st.index_vectors = arr(getattr(s, "index_vectors", None), np.float32)
    return st, _Keep(keep)


def scan(s, query, labels=None, search_list_size: int = 100, rescore: int = 50,
         max_rows: int = 10, stream_cap: int = 4096):
    """amrescan + amgettuple*max_rows. labels=None => no scan key; [] => empty key.
    Returns dict(tid, node, dist, stream, stats)."""
    st, keep = _snapshot_struct(s)
    q = None if query is None else _f32(query)
    if labels is None:
        lab, nl = None, -1
    else:
        lab = np.ascontiguousarray(labels, dtype=np.int16)
        nl = lab.size
    tid = np.zeros(max_rows, np.uint64)
    node = np.zeros(max_rows, np.uint32)
    dist = np.zeros(max_rows, np.float32)
    stream = np.full(stream_cap, INVALID_NODE, np.uint32)
    stats = _Stats()
    rows = lib().orc_scan(C.byref(st), _p(q), _p(lab) if lab is not None and lab.size else None,
                          C.c_int32(nl), C.c_uint32(search_list_size), C.c_uint32(rescore),
                          C.c_uint32(max_rows), _p(tid), _p(node), _p(dist), _p(stream),
                          C.c_uint32(stream_cap), C.byref(stats))
    sl = min(int(stats.stream_len), stream_cap)
    return dict(tid=tid[:rows], node=node[:rows], dist=dist[:rows], stream=stream[:sl],
                stats={k: int(getattr(stats, k)) for k, _ in _Stats._fields_})


_NATIVE = None


def native_lib():
    """liboracle_native.so: the same oracle.cpp compiled with -march=native (optional CPU-baseline arm, BASELINE.md §3:
    "not the reference's build flags").  Only scan_batch(native=True) uses it; parity always runs on the reference-flag build."""
    global _NATIVE
    if _NATIVE is None:
        # -march=native code must never run on another machine, and the tree may be read-only: built per process in a
        # temporary directory, removed at exit
        import atexit
        import shutil
        import tempfile
        tmp = tempfile.mkdtemp(prefix="dann_oracle_native_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "liboracle_native.so")
        subprocess.run(["make", "-C", _HERE, "-s", "native", f"NATIVE_SO={so}"], check=True, stdout=subprocess.DEVNULL)
        _NATIVE = C.CDLL(so)
    return _NATIVE


def scan_batch(s, queries, labels=None, label_off=None, search_list_size: int = 100,
               rescore: int = 50, k: int = 10, threads: int = 0, native: bool = False):
    """One independent scan per query row. Returns tid[B,k] (~0 = none), dist[B,k], count[B], stats[B]."""
    st, keep = _snapshot_struct(s)
    q = _f32(queries)
    B = q.shape[0]
    tid = np.zeros((B, k), np.uint64)
    dist = np.zeros((B, k), np.float32)
    count = np.zeros(B, np.uint32)
    stats = np.zeros(B, STATS_DTYPE)
    lab = lo = None
    if label_off is not None:
        lab = np.ascontiguousarray(labels, dtype=np.int16)
        lo = np.ascontiguousarray(label_off, dtype=np.int32)
    (native_lib() if native else lib()).orc_scan_batch(C.byref(st), _p(q), _p(lab), _p(lo), C.c_uint32(B),
                         C.c_uint32(search_list_size), C.c_uint32(rescore), C.c_uint32(k),
                         _p(tid), _p(dist), _p(count), _p(stats), C.c_uint32(threads))
    return tid, dist, count, stats
