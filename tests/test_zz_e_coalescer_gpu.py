"""Query coalescer (SURVEY.md §8f row 4) through the C ABI.  Written after this round's GPU minutes were spent: it
passes on the CPU against the emulated ABI (tests/test_emulated_abi.py); the file name sorts it after the tests that
have already been on hardware."""
import numpy as np
import pytest

from conftest import build_case
from test_gpu_parity import _queries

pytestmark = pytest.mark.gpu

COSINE = 0


@pytest.fixture(scope="module")
def lib(lib_built):
    from pgvectorscale_b200 import diskann
    if diskann.device_count() < 1:
        pytest.fail("no CUDA device visible: -m gpu tests need the B200 box")
    return diskann


@pytest.fixture
def sock_dir():
    """A short directory for the sidecar's Unix-domain socket: a socket path holds at most 107 bytes, which a deep
    tmp_path (a long TMPDIR, xdist's per-worker directories) can exceed."""
    import os
    import shutil
    import tempfile
    d = tempfile.mkdtemp(prefix="dann", dir="/tmp" if os.path.isdir("/tmp") else None)
    yield d
    shutil.rmtree(d, ignore_errors=True)


def test_coalescer_concurrent_single_query_callers_get_private_scan_results(lib):
    """SURVEY §8f row 4: many blocking single-query callers (backends) -> few batch calls; every caller gets exactly
    what the oracle's private scan of its query returns, whatever it was batched with."""
    import threading
    from oracle import oracle
    s = build_case(2000, 96, COSINE, seed=44, labels=True, R=24, L_build=50, deleted_every=9)
    q = _queries(s, 48, 7)
    params = [(10, 60, 25, None), (10, 60, 25, [3, 9]), (7, 30, 0, None)]      # (k, L, rescore, labels) per caller class
    results, errors = {}, []
    with lib.DiskAnnIndex(s) as idx, lib.Coalescer(idx, max_batch=16, max_wait_us=20000) as co:
        start = threading.Barrier(12)

        def backend(t):
            try:
                start.wait()
                for j in range(4):
                    i = t * 4 + j
                    k, L, rescore, lab = params[i % 3]
                    results[i] = co.search(q[i], labels=lab, k=k, search_list_size=L, rescore=rescore)
            except Exception as e:      # noqa: BLE001
                errors.append(e)

        th = [threading.Thread(target=backend, args=(t,)) for t in range(12)]
        for x in th:
            x.start()
        for x in th:
            x.join()
        st = co.stats()
    assert not errors, errors
    assert st["queries"] == 48 and st["batches"] < 48 and st["largest_batch"] > 1, st
    for i in range(48):
        k, L, rescore, lab = params[i % 3]
        r = oracle.scan(s, q[i], lab, L, rescore, k)
        g = results[i]
        n = len(r["tid"])
        assert g["count"] == n and g["tid"][:n].tolist() == r["tid"].tolist(), i
        if rescore:
            assert g["dist"][:n].view(np.uint32).tolist() == r["dist"].view(np.uint32).tolist()
        for f in ("visits", "d_quantized", "candidates", "d_full"):
            assert g["stats"][f] == r["stats"][f], (i, f)


def test_c_load_generator_through_the_coalescer(lib, lib_built, tmp_path):
    """harness/coalescer_load.c: pthread clients over the C ABI, index from the raw snapshot file (harness/snapshot_raw.h);
    the checksum of every returned TID equals the oracle's private scans."""
    import json
    import os
    import shutil
    import subprocess
    from oracle import fixtures, oracle
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "coalescer_load")
    libdir = os.path.dirname(lib_built)
    subprocess.run([gcc, "-std=c99", "-O2", "-Wall", "-Wextra", "-Werror", "-I" + os.path.join(root, "include"),
                    "-I" + os.path.join(root, "harness"), os.path.join(root, "harness", "coalescer_load.c"), "-L" + libdir,
                    "-l:" + os.path.basename(lib_built), "-Wl,-rpath," + libdir, "-lpthread", "-o", exe], check=True)
    s = build_case(1500, 64, COSINE, seed=4, kind="normal", R=24, L_build=48)
    s.save_raw(str(tmp_path / "snap.raw"))
    q = fixtures.gen_vectors(64, 64, 8, "normal")
    q.astype(np.float32).tofile(str(tmp_path / "q.f32"))
    T, per, L, rescore, k = 8, 8, 40, 20, 10
    r = subprocess.run([exe, str(tmp_path / "snap.raw"), str(tmp_path / "q.f32"), str(T), str(per), str(L), str(rescore), str(k),
                        "16", "20000"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    d = json.loads(r.stdout)
    assert d["queries"] == T * per and d["batches"] < T * per
    chk = 0
    for t in range(T):
        for i in range(per):
            o = oracle.scan(s, q[(t * per + i) % 64], None, L, rescore, k)
            for x in list(o["tid"]) + [0xFFFFFFFFFFFFFFFF] * (k - len(o["tid"])):
                chk = (chk * 1099511628211 + int(x)) % (1 << 64)
    assert chk == d["tid_checksum"]


def test_sidecar_process_serves_concurrent_backends(lib, lib_built, tmp_path, sock_dir):
    """sidecar/dann_sidecar.c: one process owns the index, every connection is a backend; concurrent clients get
    exactly the oracle's private scans (rows, distance bits, counters), keyed and unkeyed."""
    import os
    import shutil
    import signal
    import subprocess
    import threading
    import time
    from oracle import fixtures, oracle
    from pgvectorscale_b200.sidecar_client import SidecarClient
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "dann_sidecar")
    libdir = os.path.dirname(lib_built)
    subprocess.run([gcc, "-std=c99", "-O2", "-Wall", "-Wextra", "-Werror", "-I" + os.path.join(root, "include"),
                    os.path.join(root, "sidecar", "dann_sidecar.c"), "-L" + libdir, "-l:" + os.path.basename(lib_built),
                    "-Wl,-rpath," + libdir, "-lpthread", "-o", exe], check=True)
    s = build_case(1200, 48, COSINE, seed=12, kind="normal", R=24, L_build=48, labels=True, deleted_every=10)
    s.save_raw(str(tmp_path / "snap.raw"))
    sock = os.path.join(sock_dir, "dann.sock")
    proc = subprocess.Popen([exe, str(tmp_path / "snap.raw"), sock, "32", "20000"], stderr=subprocess.PIPE, text=True)
    try:
        for _ in range(600):
            if os.path.exists(sock) or proc.poll() is not None:
                break
            time.sleep(0.05)
        if proc.poll() is not None:
            err = proc.stderr.read()
            if "unavailable" in err or "exclusive" in err.lower():      # GPU in exclusive-process mode: one context only
                pytest.skip("a second process cannot open the GPU on this box: " + err.strip()[-120:])
            pytest.fail("sidecar exited: " + err)
        assert os.path.exists(sock), "no socket"
        q = fixtures.gen_vectors(24, 48, 31, "normal")
        out, errors = {}, []

        def backend(t):
            try:
                with SidecarClient(sock) as c:
                    assert (c.dim, c.n) == (48, 1200)
                    for j in range(4):
                        i = t * 4 + j
                        key = [3, 9] if i % 2 else None
                        out[i] = c.scan(q[i], labels=key, k=10, search_list_size=40, rescore=15)
            except Exception as e:      # noqa: BLE001
                errors.append(e)

        th = [threading.Thread(target=backend, args=(t,)) for t in range(6)]
        for x in th:
            x.start()
        for x in th:
            x.join()
        assert not errors, errors
        for i in range(24):
            r = oracle.scan(s, q[i], [3, 9] if i % 2 else None, 40, 15, 10)
            n = len(r["tid"])
            assert out[i]["count"] == n and out[i]["tid"][:n].tolist() == r["tid"].tolist()
            assert out[i]["dist"][:n].view(np.uint32).tolist() == r["dist"].view(np.uint32).tolist()
            assert out[i]["stats"]["visits"] == r["stats"]["visits"]
        # the socket belongs to the sidecar's account alone, and a malformed header is answered before the connection drops
        import socket
        import stat
        import struct
        assert stat.S_IMODE(os.stat(sock).st_mode) & 0o077 == 0
        c = socket.socket(socket.AF_UNIX, socket.SOCK_STREAM)
        c.settimeout(20)
        c.connect(sock)
        assert len(c.recv(12, socket.MSG_WAITALL)) == 12                       # hello
        c.sendall(struct.pack("<Iiiii", 0x12345678, 10, 40, 15, -1))            # wrong magic
        status, count = struct.unpack("<iI", c.recv(8, socket.MSG_WAITALL))
        (ln,) = struct.unpack("<I", c.recv(4, socket.MSG_WAITALL))
        msg = c.recv(ln, socket.MSG_WAITALL).decode()
        assert status == -1 and count == 0 and "malformed request header" in msg
        assert c.recv(1) == b""                                                 # then the server closes
        c.close()
    finally:
        proc.send_signal(signal.SIGTERM)
        try:
            proc.wait(timeout=20)
        except subprocess.TimeoutExpired:
            proc.kill()
    assert "queries in" in proc.stderr.read()


def test_sidecar_cold_start_from_relation_files_and_staleness_signal(lib, lib_built, tmp_path, sock_dir):
    """dann_sidecar --relation: index pages (dann_pg_extract_sbq) + the table's vector column from its heap and TOAST
    files (dann_pg_heap_fetch_vectors) -> the served index; scans equal the oracle's on the snapshot the files were
    written from.  SIGHUP re-reads the page headers: unchanged -> keeps serving; a page LSN moved -> exits with status 5."""
    import os
    import shutil
    import signal
    import struct
    import subprocess
    import time
    import pgpages
    from oracle import fixtures, oracle
    from pgvectorscale_b200.sidecar_client import SidecarClient
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "dann_sidecar")
    libdir = os.path.dirname(lib_built)
    subprocess.run([gcc, "-std=c99", "-O2", "-Wall", "-Wextra", "-Werror", "-I" + os.path.join(root, "include"),
                    os.path.join(root, "sidecar", "dann_sidecar.c"), "-L" + libdir, "-l:" + os.path.basename(lib_built),
                    "-Wl,-rpath," + libdir, "-lpthread", "-o", exe], check=True)
    s = build_case(500, 768, COSINE, seed=17, kind="normal", R=16, L_build=32, deleted_every=9)
    ipath, hpath, tpath = str(tmp_path / "idx"), str(tmp_path / "heap"), str(tmp_path / "toast")
    pre = [[struct.pack("<q", i)] for i in range(s.n)]
    htids = pgpages.write_table(s.vectors, hpath, tpath, prefix_values=pre, prefix_atts=[(8, "d")])
    dead = (s.heap_tid & np.uint64(0xFFFF)) == 0               # vacuumed nodes keep their invalid heap pointer
    s.heap_tid = np.where(dead, htids & np.uint64(0xFFFFFFFFFFFF0000), htids)
    meta, _, _ = pgpages.write_index(s, ipath)
    sock = os.path.join(sock_dir, "pg.sock")
    args = [exe, "--relation", ipath, hpath, tpath, sock, "dim=768", f"R={s.R}", "bits=%d" % s.bits, "distance=0",
            "start=%d:%d" % meta["start"], "means=%d:%d" % meta["means"], "atts=8d", "max_batch=16", "max_wait_us=2000"]
    proc = subprocess.Popen(args, stderr=subprocess.PIPE, text=True)
    try:
        for _ in range(600):
            if os.path.exists(sock) or proc.poll() is not None:
                break
            time.sleep(0.05)
        if proc.poll() is not None:
            err = proc.stderr.read()
            if "unavailable" in err or "exclusive" in err.lower():
                pytest.skip("a second process cannot open the GPU on this box: " + err.strip()[-120:])
            pytest.fail("sidecar exited: " + err)
        q = fixtures.gen_vectors(6, 768, 23, "normal")
        with SidecarClient(sock) as c:
            assert (c.dim, c.n) == (768, s.n)
            for i in range(6):
                got = c.scan(q[i], k=10, search_list_size=40, rescore=20)
                r = oracle.scan(s, q[i], None, 40, 20, 10)
                n = len(r["tid"])
                assert got["count"] == n and got["tid"][:n].tolist() == r["tid"].tolist()
                assert got["dist"][:n].view(np.uint32).tolist() == r["dist"].view(np.uint32).tolist()
        proc.send_signal(signal.SIGHUP)                          # nothing changed: keeps serving
        time.sleep(0.5)
        assert proc.poll() is None
        with SidecarClient(sock) as c:
            assert c.scan(q[0], k=5, search_list_size=20, rescore=10)["count"] == 5
        blob = bytearray(open(ipath, "rb").read())               # an insert rewrote a neighbour list: the page's LSN moved
        lo = struct.unpack_from("<I", blob, 2 * 8192 + 4)[0]
        struct.pack_into("<I", blob, 2 * 8192 + 4, lo + 0x58)
        open(ipath, "wb").write(blob)
        proc.send_signal(signal.SIGHUP)
        assert proc.wait(timeout=30) == 5
        assert "reload needed" in proc.stderr.read()
    finally:
        if proc.poll() is None:
            proc.kill()
