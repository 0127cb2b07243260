"""Wide SBQ codes against the oracle: up to 16000 dimensions at 1 bit per dimension (the reference's MAX_DIMENSION,
build.rs:192) and up to 32 bits per dimension (options.rs:253-260), and the shared-memory limits they run into.

The kernels take their shape from the code width: the 16-byte chunk mapping (G lanes x NCH chunks, pick_code_mapping in
dann_plan.h), the NCH template instances of the three search kernels and of dann_sbq_distance_kernel, the heap entry
layout, the lean kernel's width limit (192 words) and the launches above 48 KB of dynamic shared memory.  Every case
below is bit-exact parity with the oracle: row ids, distance bits and all five scan counters.  Small indexes (300 rows)
keep the oracle's serial build cheap at 16000 dimensions."""
import numpy as np
import pytest

from conftest import buffer_device, build_case, dptr, emulating

pytestmark = pytest.mark.gpu

COSINE, L2, IP = 0, 1, 2
N = 300
EMU_SMEM_OPTIN = 232448          # what the emulated runtime reports (tests/simt/shim/fake_cuda.h)

# id -> (dim, bits, distance, dim_index, G, NCH): the code mapping dann_plan.h picks for the code width
CASES = {
    "3072x1": (3072, 1, COSINE, None, 8, 3),           # 48 words: round-1 kernels' default entry is Ent32x16
    "8000x1": (8000, 1, L2, None, 32, 2),              # 125 words: 63 chunks, not a whole number of lane groups
    "12288x1": (12288, 1, IP, None, 32, 3),            # 192 words: the widest code the lean kernel serves
    "12289x1": (12289, 1, COSINE, None, 32, 4),        # 193 words: NCH=4
    "16000x1": (16000, 1, L2, None, 32, 4),            # 250 words: NCH=4, the reference's largest dimension
    "16000i12289x1": (16000, 1, COSINE, 12289, 32, 4),  # dim_index < dim: the truncated copy is quantized
    "768x3": (768, 3, IP, None, 8, 3),                 # 36 words: a dimension's bits straddle a 64-bit word
    "768x5": (768, 5, COSINE, None, 16, 2),            # 60 words
    "768x7": (768, 7, L2, None, 16, 3),                # 84 words
    "930x20": (930, 20, IP, None, 32, 8),              # 291 words: NCH=8
    "930x32": (930, 32, COSINE, None, 32, 8),          # 465 words: NCH=8
}
_FIXTURES = {}


def _case(cid, **kw):
    key = (cid, tuple(sorted(kw.items())))
    if key not in _FIXTURES:
        dim, bits, dist, dim_index, _, _ = CASES[cid]
        args = dict(R=16, L_build=32)
        args.update(kw)
        _FIXTURES[key] = build_case(N, dim, dist, bits=bits, seed=dim + bits, kind="normal", dim_index=dim_index, **args)
    return _FIXTURES[key]


def _queries(s, B, seed, kind="normal"):
    from oracle import fixtures
    return fixtures.gen_vectors(B, s.dim, seed, kind)


def _code_mapping(cw):
    """pick_code_mapping (dann_plan.h) for a code stride of cw words -> (G, NCH)."""
    chunks = cw // 2
    g = 1
    while g < (chunks + 2) // 3:
        g <<= 1
    g = min(g, 32)
    n = (chunks + g - 1) // g
    return g, (n if n <= 4 else 8)


def _compare_batch(s, idx, q, k, L, rescore, labels=None):
    """Counts, row ids, distance bits, the five counters and a zero status, against the oracle."""
    from oracle import oracle
    lab = off = None
    if labels is not None:
        off = np.zeros(len(labels) + 1, np.int32)
        vals = []
        for i, ls in enumerate(labels):
            vals.extend(ls)
            off[i + 1] = len(vals)
        lab = np.asarray(vals, np.int16)
    otid, odist, ocount, ostats = oracle.scan_batch(s, q, lab, off, L, rescore, k, threads=0)
    g = idx.search_batch(q, labels=labels, k=k, search_list_size=L, rescore=rescore)
    assert np.array_equal(g["count"], ocount)
    assert np.array_equal(g["tid"], otid), "row ids differ from the oracle"
    if rescore > 0:
        assert np.array_equal(g["dist"].view(np.uint32), odist.view(np.uint32))
    for f in ("visits", "d_quantized", "candidates", "d_full", "stream_len"):
        assert np.array_equal(g["stats"][f].astype(np.uint64), ostats[f]), f
    assert not g["stats"]["status"].any()
    return g


@pytest.fixture(scope="module")
def lib(lib_built):
    from pgvectorscale_b200 import diskann
    if diskann.device_count() < 1:
        pytest.fail("no CUDA device visible: -m gpu tests need the B200 box")
    return diskann


def test_cases_cover_every_wide_code_mapping():
    """The parametrization reaches NCH 2, 3, 4 and 8 at G=32, the lean kernel's last width and G=8 / G=16."""
    from pgvectorscale_b200.snapshot import code_words
    for cid, (dim, bits, _, dim_index, G, NCH) in CASES.items():
        words = code_words(dim_index or dim, bits)
        assert _code_mapping((words + 1) & ~1) == (G, NCH), cid
    shapes = {(c[4], c[5]) for c in CASES.values()}
    assert {(32, 2), (32, 3), (32, 4), (32, 8), (8, 3), (16, 2), (16, 3)} <= shapes


# -- 1. query preparation ---------------------------------------------------------------------------------------------

def _check_prepare(lib, s, q):
    import torch
    import pyref
    from oracle import oracle
    B = q.shape[0]
    with lib.DiskAnnIndex(s) as idx:
        dev = buffer_device()
        d_q = torch.from_numpy(q).to(dev)
        d_full = torch.empty((B, s.dim), dtype=torch.float32, device=dev)
        d_codes = torch.full((B, idx.code_stride), -1, dtype=torch.int64, device=dev)   # padding must be written
        idx.prepare_queries(dptr(d_q), dptr(d_full), dptr(d_codes))
        full = d_full.cpu().numpy()
        codes = d_codes.cpu().numpy().view(np.uint64)
    for b in range(B):
        qf = oracle.preprocess_cosine(q[b]) if s.distance_type == COSINE else q[b]
        qi = q[b, :s.dim_index].copy()
        if s.distance_type == COSINE:
            qi = oracle.preprocess_cosine(qi)
        assert np.array_equal(full[b].view(np.uint32), qf.view(np.uint32)), b
        ref = oracle.quantize(qi, s.bits, s.mean, s.m2, s.count)
        assert np.array_equal(codes[b, :s.words], ref), b
        assert np.array_equal(ref, np.array(pyref.quantize(qi, s.bits, s.mean, s.m2, s.count, s.words), np.uint64)), b
        assert not codes[b, s.words:].any(), b


@pytest.mark.parametrize("cid", list(CASES))
def test_prepare_queries_wide_codes(lib, cid):
    s = _case(cid)
    q = _queries(s, 5, 14, "uniform") * 3.0
    q[0] = 0.0
    _check_prepare(lib, s, q)


@pytest.mark.parametrize("bits", [3, 7])
def test_prepare_queries_constant_dimension(lib, bits):
    """m2 = 0 with count > 0: the z-score of a constant dimension is +inf above it, -inf below and NaN on it."""
    from oracle import fixtures
    v = fixtures.gen_vectors(N, 768, 40 + bits, "uniform")
    v[:, 5] = 0.5
    v[:, 700] = -0.25
    s = fixtures.make_index(v, L2, bits=bits, R=16, L_build=32)
    assert s.count > 0 and s.m2[5] == 0.0 and s.m2[700] == 0.0
    q = _queries(s, 6, 15, "uniform")
    q[:, 5] = [0.5, 0.75, 0.25, 0.5, 1e30, -1e30]
    q[:, 700] = [-0.25, -0.25, 0.0, -1.0, -0.25, 3.0]
    _check_prepare(lib, s, q)
    with lib.DiskAnnIndex(s) as idx:
        _compare_batch(s, idx, q, 10, 40, 20)


# -- 2. Hamming kernel ------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("cid", ["8000x1", "12288x1", "16000x1", "930x32"])   # NCH 2, 3 (G=32), 4, 8
def test_sbq_distance_wide_codes(lib, cid):
    import torch
    s = _case(cid)
    with lib.DiskAnnIndex(s) as idx:
        dev = buffer_device()
        Q, npairs = 5, 2053                      # prime: not a multiple of any lane-group count
        rng = np.random.default_rng(len(cid))
        qcodes = rng.integers(0, 2**63, size=(Q, idx.code_stride), dtype=np.uint64) * np.uint64(2) + np.uint64(1)
        qcodes[:, s.words:] = 0
        pq = rng.integers(0, Q, size=npairs, dtype=np.uint32)
        pn = rng.integers(0, s.n, size=npairs, dtype=np.uint32)
        d_q = torch.from_numpy(qcodes.view(np.int64)).to(dev)
        d_pq = torch.from_numpy(pq.view(np.int32)).to(dev)
        d_pn = torch.from_numpy(pn.view(np.int32)).to(dev)
        d_out = torch.empty(npairs, dtype=torch.int32, device=dev)
        idx.sbq_distance(dptr(d_q), dptr(d_pq), dptr(d_pn), dptr(d_out))
        x = s.codes[pn] ^ qcodes[pq][:, :s.words]
        ref = np.unpackbits(x.view(np.uint8), axis=1).sum(1).astype(np.int32)
        assert np.array_equal(d_out.cpu().numpy(), ref)


# -- 3. exact distance ------------------------------------------------------------------------------------------------

def _f64_distance_and_bound(kind, x, y):
    """float64 distance of the same f32 inputs, and a bound on the f32 result's error: the AVX2 body keeps 32 partial
    sums of dim/32 terms, then adds them in 5 levels and the tail (< 32 terms) one by one, so no term passes through
    more than dim/32 + 40 roundings of relative size 2^-24 (plus the subtraction / product of an L2 term)."""
    x, y = x.astype(np.float64), y.astype(np.float64)
    terms = (x - y) ** 2 if kind == L2 else x * y
    s = terms.sum()
    d = s if kind == L2 else -s if kind == IP else max(1.0 - s, 0.0)
    bound = (x.size / 32 + 48) * 2.0**-24 * np.abs(terms).sum() + 2.0**-24 * (1.0 if kind == COSINE else 0.0)
    return d, bound


@pytest.mark.parametrize("cid", ["12288x1", "12289x1", "16000x1"])
def test_full_distance_long_rows(lib, cid):
    """12289 is not a multiple of 4: scalar tail and the plain-load staging of the query row instead of TMA."""
    import torch
    from oracle import oracle
    s = _case(cid)
    with lib.DiskAnnIndex(s) as idx:
        dev = buffer_device()
        B, m = 3, 13
        q = _queries(s, B, 16)
        d_q = torch.from_numpy(q).to(dev)
        d_full = torch.empty((B, s.dim), dtype=torch.float32, device=dev)
        d_codes = torch.empty((B, idx.code_stride), dtype=torch.int64, device=dev)
        idx.prepare_queries(dptr(d_q), dptr(d_full), dptr(d_codes))
        full = d_full.cpu().numpy()
        nodes = np.random.default_rng(2).integers(0, s.n, size=(B, m), dtype=np.uint32)
        d_nodes = torch.from_numpy(nodes.view(np.int32)).to(dev)
        d_out = torch.empty((B, m), dtype=torch.float32, device=dev)
        idx.full_distance(dptr(d_full), dptr(d_nodes), dptr(d_out))
        out = d_out.cpu().numpy()
    for b in range(B):
        for i in range(m):
            x = s.vectors[nodes[b, i]]
            if s.distance_type == COSINE:
                x = oracle.preprocess_cosine(x)
            ref = np.float32(oracle.distance(s.distance_type, x, full[b], "avx2"))
            assert out[b, i].view(np.uint32) == ref.view(np.uint32), (b, i)
            d64, bound = _f64_distance_and_bound(s.distance_type, x, full[b])
            assert abs(float(out[b, i]) - d64) <= bound, (b, i, float(out[b, i]), d64, bound)


# -- 4. batch parity on every kernel ----------------------------------------------------------------------------------

def _set(monkeypatch, name, value):
    if value is None:
        monkeypatch.delenv(name, raising=False)
    else:
        monkeypatch.setenv(name, value)


@pytest.mark.parametrize("cid", list(CASES))
def test_batch_parity_every_kernel_and_entry(lib, monkeypatch, cid):
    s = _case(cid)
    lean_ok = ((s.words + 1) & ~1) <= 192
    assert s.words * 64 >= 2048            # Ent32x21 (11-bit distance keys) cannot hold these distances
    q = _queries(s, 6, 21)
    with lib.DiskAnnIndex(s) as idx:
        monkeypatch.delenv("DANN_SEARCH_ENTRY", raising=False)
        for kernel in (None, "1", "2", "3"):
            _set(monkeypatch, "DANN_SEARCH_KERNEL", kernel)
            for rescore in (20, 0):
                _compare_batch(s, idx, q, 10, 40, rescore)
                p = idx.last_search_plan()
                # a batch this small stays on the two-warp kernel; the lean kernel serves codes of at most 192 words
                assert p["kernel"] == {None: 2, "1": 1, "2": 2, "3": 3 if lean_ok else 2}[kernel], (kernel, p)
                # default entries: the lean kernel's 8-byte key32|node32, Ent32x16 for the round-1 kernels
                assert p["entry_bytes"] == (8 if p["kernel"] == 3 else 4), p
        for entry in ("1", "2"):
            monkeypatch.setenv("DANN_SEARCH_ENTRY", entry)
            for kernel in ("1", "2", "3"):
                monkeypatch.setenv("DANN_SEARCH_KERNEL", kernel)
                _compare_batch(s, idx, q, 10, 40, 20)
                p = idx.last_search_plan()
                assert p["entry_bytes"] == (8 if entry == "2" or p["kernel"] == 3 else 4), (entry, kernel, p)


@pytest.mark.parametrize("cid", ["12289x1", "930x20"])       # NCH=4 and NCH=8
def test_labeled_deleted_and_regrown_wide_codes(lib, monkeypatch, cid):
    s = _case(cid, labels=True, deleted_every=4)
    B = 6
    q = _queries(s, B, 22)
    keys = [[1 + (i % 16)] for i in range(B)]
    with lib.DiskAnnIndex(s) as idx:
        for shrink in (None, "16"):            # second pass: every query outgrows its workspace and is rerun
            _set(monkeypatch, "DANN_DEBUG_SHRINK", shrink)
            for kernel in ("1", "2"):
                monkeypatch.setenv("DANN_SEARCH_KERNEL", kernel)
                g = _compare_batch(s, idx, q, 10, 40, 20, labels=keys)
                assert ((g["tid"][g["tid"] != lib.INVALID_TID] & np.uint64(0xFFFF)) != 0).all()
                if shrink:
                    assert idx.last_batch_timing()["retries"] >= 1
                _compare_batch(s, idx, q, 10, 40, 0, labels=keys)
                _compare_batch(s, idx, q, 10, 40, 20)            # unkeyed scan over a labeled index


# -- 5. streaming scan at 16000 dimensions ----------------------------------------------------------------------------

@pytest.mark.parametrize("fused", ["1", "0"])
def test_streaming_scan_16000_dimensions(lib, monkeypatch, fused):
    """One-synchronisation amgettuple (dann_scan_distance_kernel) and the step-by-step one (dann_full_distance_kernel),
    both with a 64 KB query row in shared memory; 270 rows cross the 16 -> 64 -> 256 refetch points."""
    from oracle import oracle
    monkeypatch.setenv("DANN_SCAN_FUSED", fused)
    s = _case("16000x1")
    q = _queries(s, 2, 23)
    rows_max, L, rescore = 270, 40, 10
    with lib.DiskAnnIndex(s) as idx:
        sc = idx.begin_scan()
        for qi in range(2):
            ref = oracle.scan(s, q[qi], None, L, rescore, rows_max)
            assert len(ref["tid"]) > 256
            sc.rescan(q[qi], search_list_size=L, rescore=rescore)
            for i in range(1, rows_max + 1):
                row = sc.gettuple()
                if i > len(ref["tid"]):
                    assert row is None
                    break
                assert ((row[0] << 16) | row[1]) == int(ref["tid"][i - 1]) and row[2] == int(ref["node"][i - 1]), i
                assert np.float32(row[3]).view(np.uint32) == ref["dist"][i - 1].view(np.uint32), i
                if i in (1, 15, 16, 17, 63, 64, 65, 255, 256, 257) or i % 37 == 0:
                    ref_i = oracle.scan(s, q[qi], None, L, rescore, i)["stats"]
                    st = sc.stats()
                    for f in ("visits", "d_quantized", "candidates", "d_full", "stream_len"):
                        assert st[f] == ref_i[f], (f, i)
        sc.end()


# -- 6. rerank shared-memory boundary ---------------------------------------------------------------------------------

def _rerank_smem(dim, k, rescore):
    """dann_rerank_kernel's dynamic shared memory for one request (rerank_smem_bytes in diskann_b200.cu)."""
    c_target = k if rescore == 0 else rescore + k - 1
    return ((dim + 3) & ~3) * 4 + ((c_target + 1) & ~1) * 4 + rescore * 8 + 16 + 128


def _smem_optin():
    if emulating():
        return EMU_SMEM_OPTIN
    import torch
    return int(torch.cuda.get_device_properties(0).shared_memory_per_block_optin)


@pytest.mark.parametrize("rescore", [0, 10, 1000])
@pytest.mark.parametrize("dim", [64, 16000])
def test_rerank_shared_memory_boundary(lib, dim, rescore):
    """The largest k the rerank kernel's shared memory allows returns the oracle's rows; one more is refused as an
    invalid argument, and the handle keeps working (no CUDA error, no poisoned index)."""
    limit = _smem_optin()
    k_max = (limit - _rerank_smem(dim, 0, rescore)) // 4
    while _rerank_smem(dim, k_max, rescore) > limit:
        k_max -= 1
    while _rerank_smem(dim, k_max + 1, rescore) <= limit:
        k_max += 1
    assert k_max > N
    s = _case("16000x1") if dim == 16000 else build_case(N, 64, L2, seed=71, kind="uniform", R=12, L_build=24)
    q = _queries(s, 1, 3, "uniform")
    with lib.DiskAnnIndex(s) as idx:
        g = _compare_batch(s, idx, q, k_max, 50, rescore)
        assert 0 < g["count"][0] <= N and (g["tid"][0, g["count"][0]:] == lib.INVALID_TID).all()
        with pytest.raises(lib.DiskAnnError) as e:
            idx.search_batch(q, k=k_max + 1, search_list_size=50, rescore=rescore)
        assert e.value.code == -1          # DANN_ERR_INVALID_ARG, not a CUDA error
        _compare_batch(s, idx, q, 10, 50, 20)


# -- 7. builder at wide codes -----------------------------------------------------------------------------------------

def _prune_warps(words, smem_optin):
    """Prune warps per CTA of dann_build_graph: 128 staged candidate codes of (cw | 1) words per warp."""
    cws = ((words + 1) & ~1) | 1
    pw = (128 * 8 + 128 * cws * 8 + 128 * 4 + 64 * 4 + 64 * 2 + 15) & ~15
    return min(8, (smem_optin - 1024) // pw)


def _empty_build_slots(s):
    from pgvectorscale_b200.snapshot import INVALID_NODE
    s.R = 64
    s.nbrs = np.full((s.n, 64), INVALID_NODE, np.uint32)
    s.start_default = 0
    return s


def test_builder_at_12000_dimensions(lib):
    from oracle import oracle
    s = _empty_build_slots(build_case(N, 12000, L2, bits=1, seed=12000, kind="normal", R=8, L_build=16))
    assert _prune_warps(s.words, _smem_optin()) == 1
    R = 24
    with lib.DiskAnnIndex(s) as idx:
        idx.build_graph(R, 48, 1.2, 64)
        s.nbrs = idx.download_nbrs()
        nb = s.nbrs
        valid = nb != 0xFFFFFFFF
        deg = valid.sum(1)
        assert deg.max() <= R and deg[1:].min() >= 1
        assert (valid[:, :-1] >= valid[:, 1:]).all()                      # INVALID-terminated prefixes
        assert (nb[valid] < s.n).all()
        assert not (nb == np.arange(s.n, dtype=np.uint32)[:, None]).any()
        for i in range(s.n):
            row = nb[i][valid[i]]
            assert len(set(row.tolist())) == len(row)
        q = _queries(s, 6, 24)
        _compare_batch(s, idx, q, 10, 40, 20)
        sc = idx.begin_scan()
        sc.rescan(q[0], search_list_size=40, rescore=20)
        rows = [sc.gettuple() for _ in range(30)]
        sc.end()
        ref = oracle.scan(s, q[0], None, 40, 20, 30)
        assert [(b << 16) | o for b, o, _, _ in rows[:len(ref["tid"])]] == ref["tid"].tolist()


@pytest.mark.parametrize("cid", ["16000x1", "930x32"])
def test_builder_refuses_too_wide_codes_and_keeps_the_graph(lib, cid):
    s = _case(cid, R=64, L_build=32)       # an oracle-built graph in 64 slots, start node 0
    assert s.start_default == 0
    assert _prune_warps(s.words, _smem_optin()) < 1
    q = _queries(s, 6, 25)
    with lib.DiskAnnIndex(s) as idx:
        with pytest.raises(lib.DiskAnnError) as e:
            idx.build_graph(24, 48, 1.2, 64)
        assert e.value.code == -5          # DANN_ERR_CAPACITY
        assert np.array_equal(idx.download_nbrs(), s.nbrs)
        _compare_batch(s, idx, q, 10, 40, 20)
