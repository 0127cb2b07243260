"""Second, independent restatement of the scan path in plain Python (small cases only).

Written from the reference sources, not from oracle.cpp, so that a slip in one restatement
shows up as a disagreement between the two (tests/test_oracle_kats.py).  Reference paths are
relative to /root/reference/pgvectorscale/src/access_method/."""
import math

import numpy as np

INVALID = 0xFFFFFFFF


class RustBinaryHeap:
    """alloc::collections::BinaryHeap (max-heap on `le`), Rust 1.7x-1.8x sift rules."""

    def __init__(self, le):
        self.data = []
        self.le = le          # le(a, b) == (a <= b)

    def __len__(self):
        return len(self.data)

    def peek(self):
        return self.data[0]

    def push(self, x):
        old = len(self.data)
        self.data.append(x)
        self._sift_up(0, old)

    def pop(self):
        item = self.data.pop()
        if self.data:
            item, self.data[0] = self.data[0], item
            self._sift_down_to_bottom(0)
        return item

    def _sift_up(self, start, pos):
        d = self.data
        elem = d[pos]
        while pos > start:
            parent = (pos - 1) // 2
            if self.le(elem, d[parent]):
                break
            d[pos] = d[parent]
            pos = parent
        d[pos] = elem

    def _sift_down_to_bottom(self, pos):
        d = self.data
        end = len(d)
        start = pos
        elem = d[pos]
        child = 2 * pos + 1
        while child <= max(end - 2, 0) and end >= 2:
            if self.le(d[child], d[child + 1]):
                child += 1
            d[pos] = d[child]
            pos = child
            child = 2 * pos + 1
        if child == end - 1:
            d[pos] = d[child]
            pos = child
        d[pos] = elem
        self._sift_up(start, pos)


def total_key(f):
    b = int(np.float32(f).view(np.int32))
    b ^= ((b >> 31) & 0xFFFFFFFF) >> 1
    return b


def hamming(a, b):
    return sum(bin(int(x) ^ int(y)).count("1") for x, y in zip(a, b))


def preprocess_cosine(v):
    """distance/mod.rs:225-253"""
    v = np.array(v, np.float32)
    norm = np.float32(0)
    for x in v:
        norm = np.float32(norm + np.float32(x * x))
    eps = np.float32(1.1920929e-07)
    if norm < eps:
        return v
    adj = np.float32(eps * np.float32(len(v)))
    if np.float32(1.0) - adj <= norm <= np.float32(1.0) + adj:
        return v
    s = np.float32(math.sqrt(float(norm)))   # f32 sqrt of an f32 is correctly rounded via f64
    return (v / s).astype(np.float32)


def quantize(v, bits, mean, m2, count, words):
    """sbq/quantize.rs:52-102"""
    out = [0] * words
    for i, x in enumerate(np.asarray(v, np.float32)):
        if bits == 1:
            ones = 1 if x > mean[i] else 0
        else:
            with np.errstate(all="ignore"):
                var = np.float32(m2[i]) / np.float32(count)
                std = np.sqrt(var, dtype=np.float32)
                z = np.float32(np.float32(x - mean[i]) / std)
                idx = np.float32(np.float32(z + np.float32(2.0)) / np.float32(np.float32(4.0) / np.float32(bits + 1)))
            if idx < 1.0:
                ones = 0
            elif np.isnan(idx):
                ones = 0
            elif np.isinf(idx):     # constant dimension (m2 = 0), query above its value: `inf as usize` saturates
                ones = bits
            else:
                ones = min(int(math.floor(float(idx))), bits)
        for j in range(ones):
            p = i * bits + j
            out[p // 64] |= 1 << (p % 64)
    return out


def hadd8(a):
    f = np.float32
    return f(f(f(a[0] + a[4]) + f(a[1] + a[5])) + f(f(a[2] + a[6]) + f(a[3] + a[7])))


def distance(kind, x, y):
    """distance/mod.rs:325-434 with 8-lane accumulators; kind 0 cosine, 1 l2, 2 ip"""
    f = np.float32
    x = np.asarray(x, f)
    y = np.asarray(y, f)
    acc = np.zeros((4, 8), f)
    n = len(x)
    i = 0
    while n - i >= 32:
        for k in range(4):
            for j in range(8):
                a, b = x[i + 8 * k + j], y[i + 8 * k + j]
                if kind == 1:
                    d = f(a - b)
                    acc[k, j] = f(acc[k, j] + f(d * d))
                else:
                    acc[k, j] = f(np.float64(a) * np.float64(b) + np.float64(acc[k, j]))   # exact product, one rounding
        i += 32
    dist = f(f(f(hadd8(acc[0]) + hadd8(acc[1])) + hadd8(acc[2])) + hadd8(acc[3]))
    while i < n:
        if kind == 1:
            d = f(x[i] - y[i])
            dist = f(dist + f(d * d))
        else:
            dist = f(dist + f(x[i] * y[i]))
        i += 1
    if kind == 1:
        return dist
    if kind == 2:
        return f(-dist)
    r = f(f(1.0) - dist)
    return r if r > 0 else f(0.0)


def overlaps(a, b):
    i = j = 0
    while i < len(a) and j < len(b):
        if a[i] == b[j]:
            return True
        if a[i] < b[j]:
            i += 1
        else:
            j += 1
    return False


def scan(s, query, labels, L, rescore, max_rows):
    """amrescan + amgettuple*max_rows (scan.rs:176-305, graph/mod.rs:97-185,331-385,
    sbq/storage.rs:125-190,365-414). Returns (tids, nodes, dists, stats)."""
    f = np.float32
    if query is None:
        q_full = np.zeros(s.dim, f)
        q_index = np.zeros(s.dim_index, f)
        labels = None
    else:
        q_full = np.array(query, f)
        q_index = np.array(query[:s.dim_index], f)
        if s.distance_type == 0:
            q_full = preprocess_cosine(q_full)
            q_index = preprocess_cosine(q_index)
    if labels is not None:
        labels = sorted(set(int(x) for x in labels))
    has_filter = labels is not None and len(labels) > 0
    stats = dict(visits=0, d_quantized=0, candidates=0, d_full=0, stream_len=0)
    cand = RustBinaryHeap(lambda a, b: b[0] <= a[0])      # Reverse<Lsn>: a <= b  <=>  b.dist <= a.dist
    visited = []
    inserted = set()
    qcode = None

    def node_labels(n):
        if not s.has_labels:
            return []
        return list(s.labels[s.label_off[n]:s.label_off[n + 1]])

    plain = int(getattr(s, "storage_type", 0) or 0) == 1
    if plain:                                   # plain/storage.rs:260 asserts no_filter
        labels = None
        has_filter = False

    def add(n):
        if plain:                               # plain/mod.rs:22-32, plain/storage.rs:223-299
            stats["d_full"] += 1
            d = float(distance(s.distance_type, q_index, np.array(s.index_vectors[n], f)))
        else:
            stats["d_quantized"] += 1
            d = float(hamming(s.codes[n], qcode))
        stats["candidates"] += 1
        cand.push((d, n))

    if s.start_default != INVALID:
        if not plain:
            qcode = quantize(q_index, s.bits, s.mean, s.m2, s.count, s.words)
        if labels is None:
            starts = [s.start_default]
        else:
            m = dict(zip([int(x) for x in s.start_labels], [int(x) for x in s.start_label_nodes])) \
                if s.start_labels is not None else {}
            starts = [m[l] for l in labels if l in m]
        for n in starts:
            if n in inserted:
                continue
            inserted.add(n)
            add(n)

    def visit_closest():
        if len(cand) == 0:
            return None
        if len(visited) > L:
            if cand.peek()[0] >= visited[L - 1][0]:
                return None
        head = cand.pop()
        lo, hi = 0, len(visited)
        while lo < hi:                      # partition_point(|x| x < head)
            mid = (lo + hi) // 2
            if visited[mid][0] < head[0]:
                lo = mid + 1
            else:
                hi = mid
        visited.insert(lo, head)
        return lo

    def iterate():
        while True:
            idx = visit_closest()
            if idx is None:
                return
            stats["visits"] += 1
            v = visited[idx][1]
            for n in s.nbrs[v]:
                n = int(n)
                if n == INVALID:
                    break
                if n in inserted:
                    continue
                inserted.add(n)
                if labels is not None and has_filter and not overlaps(labels, node_labels(n)):
                    continue
                add(n)

    def nxt():
        while True:
            iterate()
            if not visited:
                return None
            d, n = visited.pop(0)
            tid = int(s.heap_tid[n])
            if tid & 0xFFFF == 0:
                continue
            stats["stream_len"] += 1
            return tid, n

    resort = RustBinaryHeap(lambda a, b: total_key(b[0]) <= total_key(a[0]))
    rows = []
    while len(rows) < max_rows:
        if rescore == 0 or (plain and s.dim == s.dim_index):    # scan.rs:392-403
            r = nxt()
            if r is None:
                break
            rows.append((r[0], r[1], float("nan")))
            continue
        while len(resort) < rescore:
            r = nxt()
            if r is None:
                break
            stats["d_full"] += 1
            x = np.array(s.vectors[r[1]], f)
            if s.distance_type == 0:
                x = preprocess_cosine(x)
            resort.push((distance(s.distance_type, x, q_full), r[0], r[1]))
        if len(resort) == 0:
            break
        d, tid, n = resort.pop()
        rows.append((tid, n, float(d)))
    return rows, stats
