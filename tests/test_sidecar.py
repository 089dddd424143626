"""pgemb_sidecar + libpgemb_client.so: the forked-backend deployment of the drop-in boundary (DESIGN.md section 12).

Backends are separate processes; each calls the reference-shaped `hnsw_search` / `hnsw_bind_point` (embedding.h:46-47)
of libpgemb_client.so, which forwards to the one GPU-owning sidecar over shared memory; the sidecar gathers concurrent
searches into batched launches.  What must hold: results identical to the oracle's whatever the interleaving, the
reference's ownership / failure behaviour at the boundary, and no hang when either side dies.

CPU suite: the sidecar dlopen()s the host-emulated build of the C-ABI library (tests/emu) -- the protocol, batching and
host logic are what is under test here.  `-m gpu`: the same through the real libpgemb_b200.so on a B200."""
import json
import os
import signal
import subprocess
import sys
import time

import numpy as np
import pytest

pytestmark = pytest.mark.timeout(900, method="thread")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "kat_regress.json")))["cases"]


def _start(lib, name, **kw):
    from pg_embedding_b200 import build, sidecar
    build.build_sidecar()
    srv = sidecar.SidecarProcess(name, lib=lib, env={"PGEMB_EMU_SMS": "2", "PGEMB_EMU_TMA": "late"}, **kw)
    srv.wait_ready()
    return srv


@pytest.fixture(scope="module")
def emulated_lib(tmp_path_factory):
    from emu_build import build_emulated
    return build_emulated(tmp_path_factory.mktemp("emu_sidecar"))


@pytest.fixture()
def served(emulated_lib):
    """A sidecar over the emulated library, and this process connected to it."""
    from pg_embedding_b200 import sidecar
    name = f"/pgemb_test_{os.getpid()}_{int(time.time() * 1e3) % 100000}"
    srv = _start(emulated_lib, name, slots=16, max_dim=64, max_ef=64, bulk_mb=1, linger_us=20000)
    yield sidecar
    sidecar.client().pgemb_client_disconnect()
    assert srv.stop() == 0, srv.proc.stderr.read()[-2000:]


def _graph(oracle_mod, rng, n, dims, m, efc, metric, labels=None):
    x = rng.standard_normal((n, dims)).astype(np.float32) + (1.0 if metric == "cosine" else 0.0)
    orc = oracle_mod.FlatIndex("port", dims, m, efc, 64, metric, capacity=n)
    orc.build(x, labels)
    return x, orc


def _run_backends(shm, rel_key, cfg, q, ef, P, tmp_path):
    """P backend processes (tests/sidecar_backend.py), each with its own slice of the queries, all running at once."""
    per = q.shape[0] // P
    procs = []
    for p in range(P):
        qf, of = str(tmp_path / f"q{p}.npy"), str(tmp_path / f"out{p}.json")
        np.save(qf, q[p * per:(p + 1) * per])
        cmd = [sys.executable, os.path.join(ROOT, "tests", "sidecar_backend.py"), shm, str(rel_key)] + [str(c) for c in cfg] + [str(ef), qf, of]
        procs.append((subprocess.Popen(cmd, stderr=subprocess.PIPE, text=True), of))
    deadline = time.time() + 300
    while not all(os.path.exists(of + ".ready") or pr.poll() is not None for pr, of in procs) and time.time() < deadline:
        time.sleep(0.01)
    open(str(tmp_path / "go"), "w").close()
    got = []
    for pr, of in procs:
        _, err = pr.communicate(timeout=600)
        assert pr.returncode == 0, err[-2000:]
        got += json.load(open(of))
    return got


@pytest.mark.parametrize("metric", ["l2", "cosine", "manhattan"])
def test_concurrent_backends_get_the_oracle_results(served, oracle_mod, metric, tmp_path):
    rng = np.random.default_rng(5)
    n, dims, m, efc, ef = 400, 24, 6, 24, 12
    labels = (rng.permutation(n).astype(np.uint64) << np.uint64(16)) | np.uint64(7)
    x, orc = _graph(oracle_mod, rng, n, dims, m, efc, metric, labels)
    for i in range(0, n, 9):
        orc.mark_deleted(i)
    idx = served.RemoteIndex(42, dims, m, efc, 64, metric, capacity=n)
    idx.append_records(orc.records())                     # mirror the relation's pages (reference record layout)
    assert len(idx) == n
    P, per = 4, 6
    q = rng.standard_normal((P * per, dims)).astype(np.float32) + (1.0 if metric == "cosine" else 0.0)
    want = orc.search_many(q, ef)
    got = _run_backends(idx_shm(served), 42, (dims, m, efc, 64, metric), q, ef, P, tmp_path)
    for k in range(P * per):
        assert got[k] == want["labels"][k, : want["n"][k]].tolist(), (metric, k)
    st = served.stats()
    assert st["searches"] == P * per
    assert st["batches"] < st["searches"] and st["max_batch"] >= 2, st   # concurrent callers were gathered into shared launches
    # this process is a backend too; efSearch is re-read on every call (the scan doubles it, embedding.c:334)
    for ef2 in (1, 5, 64):
        assert idx.search(q[0], ef2).tolist() == orc.search(q[0], ef2).tolist()
    idx.drop()


def idx_shm(sidecar_mod):
    return sidecar_mod.client().pgemb_client_segment_name().decode()


def _tid_label(blk, pos, flags=0):
    return (blk >> 16) | ((blk & 0xFFFF) << 16) | (pos << 32) | (flags << 48)     # ItemPointerData + flags (embedding.c:44-56)


def _add_point(idx, vec, label):
    """hnsw_add_point as the glue does it (embedding.c:606-701): store the record with zeroed links (:619-621), ship it to
    the mirror, then hnsw_bind_point(meta, coord, cur_c) (:695)."""
    m, dims, rs = int(idx.h.meta.M), idx.dims, idx.record_bytes
    cur = len(idx)
    rec = np.zeros((1, rs), np.uint8)
    rec[0, (2 * m + 1) * 4:(2 * m + 1) * 4 + dims * 4] = np.frombuffer(np.asarray(vec, np.float32).tobytes(), np.uint8)
    rec[0, rs - 8:] = np.frombuffer(np.uint64(label).tobytes(), np.uint8)
    idx.append_records(rec)
    idx.bind_point(cur)


@pytest.mark.parametrize("case", GOLD, ids=[c["name"] for c in GOLD])
def test_regress_kats_and_insert_path_through_the_sidecar(served, oracle_mod, case):
    """The reference's regress suite (knn.out, gh-2, gh-3, README smoke) with every insert and search going through the
    reference-shaped calls of the client library; the mirror's link lists equal the oracle's after the same inserts."""
    o = case["options"]
    for mi, metric in enumerate(case.get("expected", case.get("expected_tids")).keys()):
        idx = served.RemoteIndex(5000 + mi, o["dims"], o["m"], o["efconstruction"], o["efsearch"], metric, capacity=64)
        orc = oracle_mod.FlatIndex("port", o["dims"], o["m"], o["efconstruction"], o["efsearch"], metric, capacity=64)
        by_label = {}
        for r in case.get("rows_before_truncate", []):
            _add_point(idx, r["val"], _tid_label(*r["tid"]))
        if "rows_before_truncate" in case:
            idx.truncate()
        for r in case["rows"]:
            lab = _tid_label(*r["tid"])
            _add_point(idx, r["val"], lab)
            orc.add(np.array(r["val"], np.float32), lab)
            by_label[lab] = r
        if "delete_all_then_insert" in case:
            n0 = len(idx)
            idx.set_labels(0, orc.labels() | np.uint64(1 << 48))          # vacuum: DELETED_FLAG (embedding.c:912-922)
            for i in range(n0):
                orc.mark_deleted(i)
            by_label = {}
            for r in case["delete_all_then_insert"]:
                lab = _tid_label(*r["tid"])
                _add_point(idx, r["val"], lab)
                orc.add(np.array(r["val"], np.float32), lab)
                by_label[lab] = r
        if len(idx):
            assert idx.links().tobytes() == orc.links().tobytes(), (case["name"], metric)
            assert idx.export_records(0, len(idx)).tobytes() == orc.records().tobytes()
        labels = idx.search(np.array(case["query"], np.float32))          # hnsw_search
        rows = [by_label[int(l)] for l in labels]
        if "expected" in case:
            assert [r["val"] for r in rows] == case["expected"][metric], metric
        if "expected_tids" in case:
            assert [r["tid"] for r in rows] == case["expected_tids"][metric], metric
        idx.drop()
        orc.close()


def test_scan_iteration_with_ef_doubling_through_the_sidecar(served, oracle_mod):
    """`SELECT ... ORDER BY val <-> q LIMIT n` with n > efSearch: the scan doubles efSearch and de-duplicates (embedding.c:322-366)."""
    rng = np.random.default_rng(14)
    n, dims, m, efc = 300, 10, 5, 20
    x, orc = _graph(oracle_mod, rng, n, dims, m, efc, "l2")
    idx = served.RemoteIndex(61, dims, m, efc, 4, "l2", capacity=n)            # efSearch = 4
    idx.append_records(orc.records())
    q = rng.standard_normal(dims).astype(np.float32)
    got = list(idx.scan(q, limit=50))
    # the same iteration over the oracle's hnsw_search
    want, ef = orc.search(q, 4).tolist(), 4
    while len(want) < 50:
        ef *= 2
        new = orc.search(q, ef).tolist()
        if len(new) <= len(want):
            break
        seen = set(want)
        want += [l for l in new if l not in seen]
        if len(new) < ef:
            break
    assert got == want[:50] and len(set(got)) == len(got)
    assert int(idx.h.meta.efSearch) == 4                                         # restored: the handle is per scan
    assert list(idx.scan(q, limit=3)) == want[:3]


@pytest.mark.parametrize("metric", ["l2", "cosine", "manhattan"])
def test_c_backend_linked_against_the_client_library(served, metric, tmp_path):
    """examples/backend_demo.c: a C program with the reference's call sites (hnsw_bind_point, hnsw_search, free) linked
    against libpgemb_client.so replays test/sql/knn.sql and prints test/expected/knn.out's order."""
    from pg_embedding_b200 import sidecar
    exe = str(tmp_path / "backend_demo")
    res = subprocess.run(["gcc", "-std=gnu11", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "examples", "backend_demo.c"),
                          "-L", os.path.dirname(sidecar.CLIENT_PATH), "-lpgemb_client", "-Wl,-rpath," + os.path.dirname(sidecar.CLIENT_PATH), "-o", exe],
                         capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    env = dict(os.environ, PGEMB_SIDECAR_SHM=idx_shm(served))
    out = subprocess.run([exe, metric], capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0, out.stderr
    knn = [c for c in GOLD if c["name"] == "knn"][0]
    want = ["{%g,%g,%g}" % tuple(v) for v in knn["expected"][metric]]
    assert out.stdout.split() == want
    # a second backend finds the relation's mirror (nothing to insert) and gets the same answer
    out2 = subprocess.run([exe, metric], capture_output=True, text=True, env=env, timeout=300)
    assert out2.returncode == 0 and out2.stdout == out.stdout


def test_failure_behaviour_at_the_boundary(served, oracle_mod):
    import ctypes as C
    rng = np.random.default_rng(1)
    x, orc = _graph(oracle_mod, rng, 60, 8, 3, 8, "l2")
    idx = served.RemoteIndex(7, 8, 3, 8, 16, "l2", capacity=60)
    idx.append_records(orc.records())
    # the reference's {dims, maxM} check of an existing index (embedding.c:594-602)
    with pytest.raises(served.SidecarError, match="differ from the attached index"):
        served.RemoteIndex(7, 9, 3, 8, 16, "l2", capacity=60)
    # unknown relation: hnsw_search returns false, nothing is allocated (embedding.c:318 then raises)
    ghost = served.RemoteIndex.__new__(served.RemoteIndex)
    ghost.h = served.PgembClientIndex()
    C.memmove(C.byref(ghost.h), C.byref(idx.h), C.sizeof(idx.h))
    ghost.h.rel_key, ghost.dims = 999, 8
    with pytest.raises(served.SidecarError, match="HNSW index search failed.*no device index attached"):
        ghost.search(x[0])
    # efSearch beyond the sidecar's --max-ef
    with pytest.raises(served.SidecarError, match="outside the sidecar's limits"):
        idx.search(x[0], 65)
    # binding a node that was never stored
    with pytest.raises(served.SidecarError, match="HNSW index insert failed"):
        idx.bind_point(60)
    # one-pair distance (the SQL operators' path, embedding.c:1037), bit-exact
    for metric in ("l2", "cosine", "manhattan"):
        assert served.dist(metric, x[1] + 1, x[2] + 1).tobytes() == oracle_mod.dist("port", metric, x[1] + 1, x[2] + 1).tobytes()
    assert served.client().hnsw_is_deleted(1 << 48) and not served.client().hnsw_is_deleted(1 << 47)
    # vacuum marks labels deleted in the mirror (embedding.c:912-922): filtered after the traversal (hnswalg.cpp:245)
    lab = orc.labels().copy()
    lab[::2] |= np.uint64(1 << 48)
    idx.set_labels(0, lab)
    for i in range(0, 60, 2):
        orc.mark_deleted(i)
    assert idx.search(x[3], 16).tolist() == orc.search(x[3], 16).tolist()
    idx.truncate()
    assert len(idx) == 0 and idx.search(x[3], 16).size == 0      # gh-3: TRUNCATE, then no rows


def test_bulk_transfers_larger_than_the_bulk_area_and_exact_build(served, oracle_mod):
    rng = np.random.default_rng(2)
    n, dims, m, efc = 5000, 48, 4, 8          # 5000 records x 236 B = 1.2 MB > the 1 MB bulk area: chunked
    x = rng.standard_normal((n, dims)).astype(np.float32)
    idx = served.RemoteIndex(77, dims, m, efc, 16, "l2", capacity=n)
    rs = idx.record_bytes
    rec = np.zeros((n, rs), np.uint8)
    rec[:, (2 * m + 1) * 4:(2 * m + 1) * 4 + dims * 4] = x.view(np.uint8)
    rec[:, rs - 8:] = np.arange(n, dtype=np.uint64).view(np.uint8).reshape(n, 8)
    idx.append_records(rec)
    assert len(idx) == n
    back = idx.export_records(0, n)
    assert back.tobytes() == rec.tobytes()
    # CREATE INDEX through the sidecar: exact parallel build of the first 160 nodes == 160 sequential reference inserts
    idx.truncate()
    idx.append_records(rec[:160])
    idx.build(0, 160, batch_max=64, exact=True)
    orc = oracle_mod.FlatIndex("port", dims, m, efc, 16, "l2", capacity=160)
    orc.build(x[:160], np.arange(160, dtype=np.uint64))
    assert idx.links().tobytes() == orc.links().tobytes()


def test_mirror_grows_with_the_relation(served, oracle_mod):
    """The glue attaches with the relation's current size; rows keep arriving (embedding.c:636-691 extends the relation page by
    page): the sidecar grows the mirror in place, ids and link lists stay what sequential inserts give."""
    rng = np.random.default_rng(41)
    n, dims, m, efc = 90, 6, 3, 8
    x = rng.standard_normal((n, dims)).astype(np.float32)
    orc = oracle_mod.FlatIndex("port", dims, m, efc, 16, "l2", capacity=n)
    idx = served.RemoteIndex(88, dims, m, efc, 16, "l2", capacity=4)              # room for 4 nodes only
    assert idx.capacity == 4
    for i in range(n):
        orc.add(x[i], 500 + i)
        _add_point(idx, x[i], 500 + i)
    assert len(idx) == n and idx.links().tobytes() == orc.links().tobytes()
    again = served.RemoteIndex(88, dims, m, efc, 16, "l2", capacity=4 * n)        # a later attach may ask for more room up front
    assert again.capacity >= 4 * n and len(again) == n
    assert idx.search(x[7], 16).tolist() == orc.search(x[7], 16).tolist()


def test_groups_larger_than_max_batch_are_split(emulated_lib, oracle_mod, tmp_path):
    """--max-batch 2 with five concurrent backends: a group of pending searches is served in several launches, every caller
    still gets its own answer."""
    from pg_embedding_b200 import sidecar
    name = f"/pgemb_test_mb_{os.getpid()}"
    srv = _start(emulated_lib, name, slots=16, max_dim=32, max_ef=32, bulk_mb=1, linger_us=20000, max_batch=2)
    try:
        sidecar.client().pgemb_client_disconnect()
        sidecar.connect(name)
        rng = np.random.default_rng(15)
        n, dims, m, efc, ef = 200, 10, 4, 16, 8
        x, orc = _graph(oracle_mod, rng, n, dims, m, efc, "l2")
        idx = sidecar.RemoteIndex(21, dims, m, efc, 64, "l2", capacity=n)
        idx.append_records(orc.records())
        P, per = 5, 5
        q = rng.standard_normal((P * per, dims)).astype(np.float32)
        want = orc.search_many(q, ef)
        got = _run_backends(name, 21, (dims, m, efc, 64, "l2"), q, ef, P, tmp_path)
        for k in range(P * per):
            assert got[k] == want["labels"][k, : want["n"][k]].tolist(), k
        st = sidecar.stats()
        assert st["searches"] == P * per and st["max_batch"] <= 2, st
    finally:
        sidecar.client().pgemb_client_disconnect()
        assert srv.stop() == 0


def test_client_does_not_hang_when_the_sidecar_dies(emulated_lib, oracle_mod):
    from pg_embedding_b200 import sidecar
    name = f"/pgemb_test_die_{os.getpid()}"
    srv = _start(emulated_lib, name, slots=4, max_dim=16, max_ef=16, bulk_mb=1)
    rng = np.random.default_rng(3)
    x, orc = _graph(oracle_mod, rng, 50, 8, 3, 8, "l2")
    idx = sidecar.RemoteIndex(5, 8, 3, 8, 16, "l2", capacity=50)
    idx.append_records(orc.records())
    assert idx.search(x[0]).tolist() == orc.search(x[0], 16).tolist()
    srv.proc.send_signal(signal.SIGKILL)
    srv.proc.wait()
    t0 = time.time()
    with pytest.raises(sidecar.SidecarError, match="HNSW index search failed"):
        idx.search(x[0])
    assert time.time() - t0 < 5.0
    # a restarted sidecar is found again under the same name; the mirror has to be rebuilt (INTEGRATION.md section 2)
    srv2 = _start(emulated_lib, name, slots=4, max_dim=16, max_ef=16, bulk_mb=1)
    idx2 = sidecar.RemoteIndex(5, 8, 3, 8, 16, "l2", capacity=50)
    assert len(idx2) == 0
    idx2.append_records(orc.records())
    assert idx2.search(x[0]).tolist() == orc.search(x[0], 16).tolist()
    sidecar.client().pgemb_client_disconnect()
    assert srv2.stop() == 0


def test_resources_of_a_dead_backend_are_reclaimed(served, oracle_mod):
    """A backend that dies while it owns the bulk area and a claimed request slot must not block the others for ever."""
    import struct
    name = idx_shm(served)
    code = (
        "import mmap, os, struct, sys\n"
        "f = open('/dev/shm' + sys.argv[1], 'r+b'); m = mmap.mmap(f.fileno(), 0)\n"
        "slots_off = struct.unpack_from('<Q', m, 24)[0]\n"
        "struct.pack_into('<I', m, 64, os.getpid())            # PgembIpcHeader.bulk_lock\n"
        "struct.pack_into('<IIii', m, slots_off, 1, 0, 0, os.getpid())   # slot 0: CLAIMED, owner = me\n"
        "m.flush()\n")
    subprocess.run([sys.executable, "-c", code, name], check=True)
    hdr = open("/dev/shm" + name, "rb").read(72)
    assert struct.unpack_from("<I", hdr, 64)[0] != 0                      # the dead process still owns the bulk area
    rng = np.random.default_rng(4)
    x, orc = _graph(oracle_mod, rng, 40, 8, 3, 8, "l2")
    idx = served.RemoteIndex(9, 8, 3, 8, 16, "l2", capacity=40)
    t0 = time.time()
    idx.append_records(orc.records())                                     # needs the bulk area: waits for the sidecar's reclaim pass
    assert time.time() - t0 < 20.0
    assert idx.search(x[0]).tolist() == orc.search(x[0], 16).tolist()
    time.sleep(1.2)
    raw = open("/dev/shm" + name, "rb").read()
    slots_off = struct.unpack_from("<Q", raw, 24)[0]
    assert struct.unpack_from("<I", raw, slots_off)[0] == 0 and struct.unpack_from("<I", raw, 64)[0] == 0   # slot FREE again, bulk area free


def test_cancelled_call_returns_and_the_sidecar_cleans_up(served, oracle_mod):
    """Query cancel: the glue's interrupt check makes a pending call give up (embedding.c then runs CHECK_FOR_INTERRUPTS);
    the sidecar finishes the abandoned request, frees its slot and -- for a bulk request -- the bulk area."""
    import ctypes as C
    rng = np.random.default_rng(12)
    n, dims, m, efc = 220, 8, 3, 10
    x, orc = _graph(oracle_mod, rng, 50, dims, m, efc, "l2")
    idx = served.RemoteIndex(31, dims, m, efc, 16, "l2", capacity=n)
    rs = idx.record_bytes
    big = rng.standard_normal((n, dims)).astype(np.float32)
    rec = np.zeros((n, rs), np.uint8)
    rec[:, (2 * m + 1) * 4:(2 * m + 1) * 4 + dims * 4] = big.view(np.uint8)
    rec[:, rs - 8:] = np.arange(n, dtype=np.uint64).view(np.uint8).reshape(n, 8)
    idx.append_records(rec)
    pending = C.c_int(0)
    CB = C.CFUNCTYPE(C.c_int)
    cb = CB(lambda: pending.value)
    served.client().pgemb_client_set_interrupt_check(C.cast(cb, C.c_void_p))
    try:
        pending.value = 1
        t0 = time.time()
        with pytest.raises(served.SidecarError, match="interrupted"):
            idx.build(0, n, batch_max=32, exact=True)            # seconds of work on the emulated library
        assert time.time() - t0 < 2.0
        pending.value = 0
        # the next call queues behind the abandoned build and then works; the index is fully bound by then
        assert len(idx) == n
        lk = idx.links()
        assert (lk[1:, 0] > 0).all()
        q = big[5]
        assert idx.search(q, 8).size == 8
    finally:
        served.client().pgemb_client_set_interrupt_check(None)
    raw = open("/dev/shm" + idx_shm(served), "rb").read()
    import struct
    slots_off, stride, nslots = struct.unpack_from("<Q", raw, 24)[0], struct.unpack_from("<I", raw, 20)[0], struct.unpack_from("<I", raw, 8)[0]
    assert all(struct.unpack_from("<I", raw, slots_off + i * stride)[0] == 0 for i in range(nslots)), "a slot was leaked"
    assert struct.unpack_from("<I", raw, 64)[0] == 0


def test_two_replicas_stay_identical_and_share_the_searches(emulated_lib, oracle_mod, monkeypatch):
    """One sidecar per GPU: every change goes to all replicas (same sequence of deterministic binds -> bit-identical
    graphs), a backend's searches go to one of them."""
    from pg_embedding_b200 import sidecar
    names = [f"/pgemb_test_rep{i}_{os.getpid()}" for i in range(2)]
    srvs = [_start(emulated_lib, nm, slots=8, max_dim=32, max_ef=32, bulk_mb=1) for nm in names]
    try:
        sidecar.client().pgemb_client_disconnect()
        sidecar.connect(",".join(names))
        assert sidecar.client().pgemb_client_replicas() == 2
        rng = np.random.default_rng(8)
        n, dims, m, efc = 40, 6, 3, 8
        x = rng.integers(0, 3, (n, dims)).astype(np.float32)
        orc = oracle_mod.FlatIndex("port", dims, m, efc, 16, "l2", capacity=n)
        idx = sidecar.RemoteIndex(3, dims, m, efc, 16, "l2", capacity=n)
        for i in range(n):
            orc.add(x[i], 100 + i)
            _add_point(idx, x[i], 100 + i)                      # record + hnsw_bind_point: both replicas
        assert idx.links().tobytes() == orc.links().tobytes()
        q = rng.integers(0, 3, (6, dims)).astype(np.float32)
        for rep in ("0", "1"):                                   # the same answers from either replica
            monkeypatch.setenv("PGEMB_CLIENT_REPLICA", rep)
            for v in q:
                assert idx.search(v, 8).tolist() == orc.search(v, 8).tolist()
        monkeypatch.delenv("PGEMB_CLIENT_REPLICA")
        assert sidecar.stats()["searches"] == 12
        # each replica on its own holds the whole graph
        for nm in names:
            sidecar.client().pgemb_client_disconnect()
            sidecar.connect(nm)
            one = sidecar.RemoteIndex(3, dims, m, efc, 16, "l2", capacity=n)
            assert len(one) == n and one.links().tobytes() == orc.links().tobytes()
            assert sidecar.stats()["searches"] == 6
    finally:
        sidecar.client().pgemb_client_disconnect()
        for s in srvs:
            assert s.stop() == 0


def test_sidecar_refuses_to_start_without_a_device(tmp_path):
    """No CPU fallback anywhere: with the product library and no CUDA device the sidecar exits instead of serving.  The
    sidecar is started with CUDA_VISIBLE_DEVICES empty, so it sees no device on a machine with a GPU either."""
    import subprocess
    from pg_embedding_b200 import build, sidecar
    build.build()
    res = subprocess.run([sidecar.SERVER_PATH, "--shm", f"/pgemb_test_nodev_{os.getpid()}"], capture_output=True, text=True, timeout=120,
                         env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert res.returncode == 4 and "no CPU fallback" in res.stderr


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_sidecar_on_gpu_matches_oracle(oracle_mod, tmp_path):
    from pg_embedding_b200 import build, sidecar
    build.build()
    name = f"/pgemb_gpu_{os.getpid()}"
    srv = sidecar.SidecarProcess(name, slots=128, bulk_mb=8)
    srv.wait_ready(120)
    try:
        rng = np.random.default_rng(8)
        n, dims, m, efc, ef = 20000, 128, 16, 64, 64
        x = rng.standard_normal((n, dims)).astype(np.float32)
        idx = sidecar.RemoteIndex(1, dims, m, efc, ef, "l2", capacity=n)
        rs = idx.record_bytes
        rec = np.zeros((n, rs), np.uint8)
        rec[:, (2 * m + 1) * 4:(2 * m + 1) * 4 + dims * 4] = x.view(np.uint8)
        rec[:, rs - 8:] = np.arange(n, dtype=np.uint64).view(np.uint8).reshape(n, 8)
        idx.append_records(rec)
        idx.build(0, n, batch_max=1024, exact=False)
        orc = oracle_mod.FlatIndex("port", dims, m, efc, ef, "l2", capacity=n)
        orc.load_graph(x, idx.links())
        P, per = 16, 40
        q = rng.standard_normal((P * per, dims)).astype(np.float32)
        want = orc.search_many(q, ef)
        got = _run_backends(name, 1, (dims, m, efc, ef, "l2"), q, ef, P, tmp_path)
        for k in range(P * per):
            assert got[k] == want["labels"][k, : want["n"][k]].tolist(), k
        st = sidecar.stats()
        assert st["searches"] == P * per and st["max_batch"] >= 2, st
    finally:
        sidecar.client().pgemb_client_disconnect()
        srv.stop()


# (kept in this file because it sorts last: a first-time failure here must not stop the `-x` GPU run before the parity tests)
@pytest.mark.gpu
@pytest.mark.parametrize("metric", ["l2", "cosine", "manhattan"])
def test_c_program_replays_the_knn_regress_test(metric, tmp_path):
    """examples/inprocess_demo.c linked against libpgemb_b200.so (in-process variant of the drop-in boundary)."""
    from test_abi import _build_inprocess_demo
    out = subprocess.run([_build_inprocess_demo(tmp_path), metric], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    knn = [c for c in GOLD if c["name"] == "knn"][0]
    assert out.stdout.split() == ["{%g,%g,%g}" % tuple(v) for v in knn["expected"][metric]]


@pytest.mark.gpu
def test_index_grows_in_place_on_gpu(oracle_mod):
    """pgemb_index_reserve on the device (new entry point; body shared with the emulated test)."""
    import pg_embedding_b200 as pg
    import test_gpu_parity as G
    G.check_reserve_keeps_contents_and_ids(pg, oracle_mod)

