"""The WHOLE library on the host: capi.cu (the C ABI: workspaces, staging, build orchestration, error paths) compiled by
g++ against tests/emu's stand-in CUDA runtime, its kernels run by the SIMT emulator.  The bodies of the GPU parity tests
(tests/test_gpu_parity.py) are reused on their small configurations, so the same assertions that gate the B200 run
also exercise the host logic here -- bit-exact against the oracle -- without a GPU.

This is test infrastructure, not a fallback: the emulated library is built into a temporary directory by this module's
fixture and is the only thing that ever loads it; `pg_embedding_b200._lib.load()` knows nothing about it."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.timeout(1800, method="thread")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def emu_lib(tmp_path_factory):
    """capi.cu as the product library compiles it."""
    from emu_build import build_emulated
    from pg_embedding_b200 import _lib
    return _lib._bind(C.CDLL(build_emulated(tmp_path_factory.mktemp("emu"))))


def _swap(lib, monkeypatch):
    import pg_embedding_b200 as pkg
    from pg_embedding_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", lib)
    monkeypatch.setenv("PGEMB_EMU_SMS", "2")
    # bulk copies land only when their mbarrier is polled (the schedule that exposes a missing / wrong wait);
    # tests/test_search_emulated.py runs the kernels under both schedules
    monkeypatch.setenv("PGEMB_EMU_TMA", "late")
    assert pkg.device_count() == 1
    return pkg


@pytest.fixture()
def pg(emu_lib, monkeypatch):
    """pg_embedding_b200 with its library handle swapped for the emulated build (restored after each test)."""
    return _swap(emu_lib, monkeypatch)


@pytest.fixture()
def pg_proto(pg):
    """Round 1's -DPGEMB_PROTO variants were measured in round 2 and are product code now (or deleted): same library."""
    return pg


@pytest.fixture(scope="module")
def P():
    import test_gpu_variants as p     # GPU tests of the variants measured in round 2: bodies reused below
    return p


@pytest.fixture(scope="module")
def G():
    import test_gpu_parity as g     # the GPU parity tests: bodies reused below
    return g


def test_kats(pg, G):
    for case in G.GOLD:
        G.test_kat_regress(pg, case)


@pytest.mark.parametrize("metric", ["l2", "cosine", "manhattan"])
def test_distance_entry_points(pg, G, oracle_mod, metric):
    rng = np.random.default_rng(1)
    for dim in (1, 3, 16, 33, 129):
        a = rng.standard_normal((7, dim)).astype(np.float32)
        b = rng.standard_normal((7, dim)).astype(np.float32)
        assert pg.dist_batch(metric, a, b).tobytes() == oracle_mod.dist_many("port", metric, a, b).tobytes()
        assert pg.dist_batch(metric, a[0], b).tobytes() == oracle_mod.dist_many("port", metric, a[0], b).tobytes()
    G.test_sql_distance_functions(pg, oracle_mod)


@pytest.mark.parametrize("metric", ["l2", "cosine", "manhattan"])
@pytest.mark.parametrize("ci", [0, 1, 3], ids=["ties", "duplicates", "padded"])
def test_search_through_the_abi(pg, G, oracle_mod, metric, ci):
    G.test_search_identical_to_oracle(pg, oracle_mod, metric, G.SEARCH_CFGS[ci])


def test_empty_and_tiny(pg, G, oracle_mod):
    G.test_search_empty_and_tiny(pg, oracle_mod)


@pytest.mark.parametrize("metric,ci", [("l2", 0), ("cosine", 0), ("manhattan", 1)], ids=["ties-l2", "ties-cosine", "duplicates-manhattan"])
def test_inserts_through_the_abi(pg, G, oracle_mod, metric, ci):
    G.test_bind_links_identical_to_oracle(pg, oracle_mod, metric, G.BIND_CFGS[ci])


def test_record_layout(pg, G, oracle_mod):
    G.test_record_layout_roundtrip(pg, oracle_mod, 3, 3)
    G.test_record_layout_roundtrip(pg, oracle_mod, 33, 5)


def test_exact_parallel_build_orchestration(pg, oracle_mod):
    """pgemb_build_exact: speculative batches, stamp/validate kernels, prefix acceptance, restart -- must equal n sequential inserts."""
    rng = np.random.default_rng(5)
    for metric, dims, m, efc, n, levels in (("l2", 4, 3, 10, 120, 3), ("cosine", 12, 4, 16, 130, 0)):
        x = rng.integers(0, levels, (n, dims)).astype(np.float32) if levels else rng.standard_normal((n, dims)).astype(np.float32)
        if metric == "cosine":
            x = x + 1.0
        orc = oracle_mod.FlatIndex("port", dims, m, efc, 64, metric, capacity=n)
        orc.build(x)
        idx = pg.HnswIndex(dims, m, efc, 64, metric, capacity=n)
        idx.append(x)
        _, st = idx.build_exact(0, n, 64)
        assert idx.links().tobytes() == orc.links().tobytes(), metric
        assert st["batches"] < n - 1, "no batch ever accepted more than one insert"
        idx.close()


def test_bulk_build_orchestration(pg, oracle_mod):
    """pgemb_build_bulk: batch_max = 1 is the sequential build; larger batches give a valid graph (sorted back-link pairs,
    per-target serialisation) that the traversal searches with the reference's results on that same graph."""
    rng = np.random.default_rng(6)
    dims, m, efc, n = 8, 4, 16, 400
    x = rng.standard_normal((n, dims)).astype(np.float32)
    orc = oracle_mod.FlatIndex("port", dims, m, efc, 64, "l2", capacity=n)
    orc.build(x)
    a = pg.HnswIndex(dims, m, efc, 64, "l2", capacity=n)
    a.build(x, batch_max=1)
    assert a.links().tobytes() == orc.links().tobytes()
    a.close()
    b = pg.HnswIndex(dims, m, efc, 64, "l2", capacity=n)
    b.build(x, batch_max=32)
    links = b.links()
    cnt = links[:, 0]
    assert cnt.max() <= 2 * m and (cnt[1:] > 0).all()
    for i in range(n):
        ids = links[i, 1:1 + cnt[i]]
        assert (ids < n).all() and (ids != i).all() and len(set(ids.tolist())) == len(ids)
    chk = oracle_mod.FlatIndex("port", dims, m, efc, 64, "l2", capacity=n)
    chk.load_graph(x, links, b.labels())
    q = rng.standard_normal((20, dims)).astype(np.float32)
    assert b.search_batch(q, 10)["labels"].tobytes() == chk.search_many(q, 10)["labels"].tobytes()
    b.close()


def test_index_grows_in_place(pg, G, oracle_mod):
    G.check_reserve_keeps_contents_and_ids(pg, oracle_mod)


def test_scan_and_merge(pg, G, oracle_mod):
    G.test_scan_topk_regress_seqscan(pg)
    for cfg in G.SCAN_ITER_CFGS[1:]:
        G.test_index_scan_iteration_equals_reference_loop(pg, oracle_mod, cfg)


def test_error_paths(pg):
    from pg_embedding_b200._lib import PgembError
    idx = pg.HnswIndex(4, 2, 4, 4, "l2", capacity=3)
    idx.append(np.zeros((3, 4), np.float32))
    with pytest.raises(PgembError):
        idx.append(np.zeros((1, 4), np.float32))          # capacity exceeded
    with pytest.raises(PgembError):
        idx.links(2, 5)                                   # range beyond the index
    with pytest.raises(Exception):
        pg.HnswIndex(0, 2, 4, 4, "l2", capacity=3)        # dims must be given (embedding.c:219-221)
    idx.close()


@pytest.mark.parametrize("env", [{"PGEMB_STREAM_QUERIES": "0"}, {"CUDA_LAUNCH_BLOCKING": "1"}, {"PGEMB_STREAM_QUERIES": "1"}],
                         ids=["copy-then-launch", "launch-blocking", "streamed"])
def test_host_pointer_search_both_copy_orders(pg, G, oracle_mod, env, monkeypatch):
    """pgemb_search_batch copies the batch before the launch under serialising tools and streams it in otherwise; a batch
    larger than one 4096-query chunk takes several chunks either way.  Same results."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    rng = np.random.default_rng(12)
    dims, m, efc, n = 5, 3, 8, 120
    x = rng.standard_normal((n, dims)).astype(np.float32)
    q = rng.standard_normal((4200, dims)).astype(np.float32)
    orc = oracle_mod.FlatIndex("port", dims, m, efc, 64, "l2", capacity=n)
    orc.build(x)
    idx = pg.HnswIndex(dims, m, efc, 64, "l2", capacity=n)
    idx.append(x, orc.labels(), orc.links())
    out = idx.search_batch(q, 4)
    want = orc.search_many(q, 4, nthreads=4)
    assert out["labels"].tobytes() == want["labels"].tobytes() and out["n"].tolist() == want["n"].tolist()
    idx.close()


# ---- the variants measured in round 2 (flags now default on; every flag value must give the oracle's result) ----------------
def test_flags_off_give_the_same_results(pg, G, oracle_mod, monkeypatch):
    for k, v in {"PGEMB_VISITED_PAIRS": "0", "PGEMB_SMEM_VISITED": "0", "PGEMB_L2_TPR8": "0", "PGEMB_SCAN_TILED": "0", "PGEMB_FAST_SMALL": "0",
                 "PGEMB_EXACT_CLAMP_SMS": "0", "PGEMB_SCAN_TC": "0"}.items():
        monkeypatch.setenv(k, v)
    G.test_search_identical_to_oracle(pg, oracle_mod, "l2", G.SEARCH_CFGS[3])
    G.test_scan_topk_regress_seqscan(pg)


@pytest.mark.parametrize("flags", [{"PGEMB_VISITED_PAIRS": "1"}, {"PGEMB_VISITED_PAIRS": "1", "PGEMB_SMEM_VISITED": "2048"}],
                         ids=["pairs", "both"])     # the shared-memory set alone: tests/test_search_emulated.py
def test_prototype_traversal_flags(pg_proto, G, P, oracle_mod, flags, monkeypatch):
    pg = pg_proto
    P.test_visited_pairs_mode(pg, oracle_mod, G.SEARCH_CFGS[0], flags, monkeypatch)       # incl. the repeated-id fallback
    for k, v in flags.items():
        monkeypatch.setenv(k, v)
    G.test_search_identical_to_oracle(pg, oracle_mod, "cosine", G.SEARCH_CFGS[3])
    G.test_bind_links_identical_to_oracle(pg, oracle_mod, "l2", G.BIND_CFGS[0])


@pytest.mark.parametrize("metric", ["l2", "cosine", "manhattan"])
def test_tiled_scan(pg_proto, G, oracle_mod, metric, monkeypatch):
    pg = pg_proto
    monkeypatch.setenv("PGEMB_SCAN_TC", "0")
    G.test_scan_topk_regress_seqscan(pg)
    rng = np.random.default_rng(3)
    for dims, n, k in ((33, 700, 20), (100, 300, 5)):
        x = rng.standard_normal((n, dims)).astype(np.float32) + (1.0 if metric == "cosine" else 0.0)
        q = rng.standard_normal((37, dims)).astype(np.float32) + (1.0 if metric == "cosine" else 0.0)
        labels = rng.permutation(n).astype(np.uint64) + np.uint64(9)
        idx = pg.HnswIndex(dims, 4, 8, 16, metric, capacity=n)
        idx.append(x, labels)
        out = idx.scan_topk(q, k)
        for i in range(q.shape[0]):
            d = oracle_mod.dist_many("port", metric, q[i], x)
            order = sorted((float(d[j]), int(labels[j])) for j in range(n))[:k]
            assert out["labels"][i].tolist() == [o[1] for o in order], (metric, dims, i)
            assert out["dists"][i].tobytes() == np.array([o[0] for o in order], np.float32).tobytes()
        idx.close()


def test_prototype_exact_build_batch_clamp(pg_proto, oracle_mod, monkeypatch):
    """PGEMB_EXACT_CLAMP_SMS=1 only changes batch sizes of the exact parallel build: still the sequential graph."""
    monkeypatch.setenv("PGEMB_EXACT_CLAMP_SMS", "1")
    rng = np.random.default_rng(6)
    n, dims, m, efc = 150, 6, 3, 10
    x = rng.integers(0, 3, (n, dims)).astype(np.float32)          # ties and duplicates
    orc = oracle_mod.FlatIndex("port", dims, m, efc, 16, "l2", capacity=n)
    orc.build(x)
    idx = pg_proto.HnswIndex(dims, m, efc, 16, "l2", capacity=n)
    idx.append(x)
    idx.build_exact(0, n, 64)
    assert idx.links().tobytes() == orc.links().tobytes()
    idx.close()


def test_prototype_fast_small_batches(pg_proto, G, oracle_mod, monkeypatch):
    """PGEMB_FAST_SMALL=1: <= 64 queries go copy -> launch -> copy back on one stream (no streaming protocol), repeated
    launches skip the attribute / occupancy / L2-window driver calls.  Same results as the default host path."""
    monkeypatch.setenv("PGEMB_FAST_SMALL", "1")
    pg = pg_proto
    for case in G.GOLD:
        G.test_kat_regress(pg, case)
    G.test_search_empty_and_tiny(pg, oracle_mod)
    rng = np.random.default_rng(21)
    n, dims, m, efc = 500, 20, 5, 24
    x = rng.standard_normal((n, dims)).astype(np.float32) + 1.0
    q = rng.standard_normal((70, dims)).astype(np.float32) + 1.0
    for metric in ("cosine", "l2"):
        orc = oracle_mod.FlatIndex("port", dims, m, efc, 64, metric, capacity=n)
        orc.build(x)
        idx = pg.HnswIndex(dims, m, efc, 64, metric, capacity=n)
        idx.append(x, orc.labels(), orc.links())
        for nq, ef in ((1, 10), (1, 10), (64, 16), (70, 16), (3, 40), (1, 10)):     # 70 > 64: the streamed path in between
            out = idx.search_batch(q[:nq], ef, want_stats=True)
            want = orc.search_many(q[:nq], ef, want_counters=True)
            assert out["labels"].tobytes() == want["labels"].tobytes() and out["n"].tolist() == want["n"].tolist(), (metric, nq, ef)
            assert out["stats"][:, :3].tolist() == want["counters"][:, :3].tolist()
        assert idx.search(q[0], 12).tolist() == orc.search(q[0], 12).tolist()         # hnsw_search
        idx.close()


@pytest.fixture(scope="module")
def U():
    import test_gpu_scan_umma as u     # GPU tests of the tensor-core scan path: bodies reused below
    return u


@pytest.mark.parametrize("metric", ["l2", "cosine"])
def test_tensor_core_filter_scan(pg, G, U, oracle_mod, metric, monkeypatch):
    """K6 on the host: the filter predicate, the chunk orchestration, candidate lists and the re-scoring kernel run as compiled;
    only the tcgen05 product itself is replaced by a TF32-truncated host product that is additionally pushed by +-90 % of the
    error bound the filter assumes (adversarial but legal).  A product 4x outside the bound must trip the tripwire and the exact
    kernels must take over."""
    for case in ((33, 900, 20, 9), (100, 400, 5, 9), (16, 300, 64, 7), (3, 40, 64, 5)):
        U.check_scan_equals_exact(pg, oracle_mod, metric, case, monkeypatch)
    U.check_scan_overflow_and_chunks(pg, oracle_mod, metric, monkeypatch, n=700, dims=10)
    dims, n, k = 33, 900, 20
    rng = np.random.default_rng(17)
    c = rng.standard_normal((12, dims)).astype(np.float32)
    shift = 1.0 if metric == "cosine" else 0.0
    x = (c[rng.integers(0, 12, n)] + 0.15 * rng.standard_normal((n, dims))).astype(np.float32) + shift
    q = (c[rng.integers(0, 12, 9)] + 0.15 * rng.standard_normal((9, dims))).astype(np.float32) + shift
    idx = pg.HnswIndex(dims, 4, 8, 16, metric, capacity=n)
    idx.append(x)
    monkeypatch.setenv("PGEMB_SCAN_TC", "0")
    want = idx.scan_topk(q, k)
    monkeypatch.setenv("PGEMB_SCAN_TC", "2")
    bound_ppm = U.rel_bound(dims) / 1.5 * 1e6
    c0 = U.counters()
    # the stand-in's operand truncation uses up to 2 * 2^-10 of the assumed bound itself: push by 90 % of what is left
    monkeypatch.setenv("PGEMB_EMU_GEMM_ERR_PPM", str(0.9 * (U.rel_bound(dims) - 2.0 / 1024.0) * 1e6))
    got = idx.scan_topk(q, k)
    assert got["labels"].tobytes() == want["labels"].tobytes() and got["dists"].tobytes() == want["dists"].tobytes()
    c1 = U.counters()
    assert c1["tc"] == c0["tc"] + 1 and c1["fallbacks"] == c0["fallbacks"]
    assert (c1["rescored"] - c0["rescored"]) < 0.5 * (c1["pairs"] - c0["pairs"]), "the filter discarded almost nothing"
    monkeypatch.setenv("PGEMB_EMU_GEMM_ERR_PPM", str(4.0 * 1.5 * bound_ppm))
    got = idx.scan_topk(q, k)
    assert got["labels"].tobytes() == want["labels"].tobytes() and got["dists"].tobytes() == want["dists"].tobytes()
    assert U.counters()["fallbacks"] == c1["fallbacks"] + 1
    monkeypatch.setenv("PGEMB_EMU_GEMM_ERR_PPM", "0")
    idx.close()
    if metric == "l2":
        U.test_scan_umma_l2_norm_cache_follows_appends(pg, oracle_mod, monkeypatch)
        U.test_scan_umma_default_policy(pg, monkeypatch)


def test_prototype_l2_eight_lanes(pg_proto, G, oracle_mod, monkeypatch):
    pg = pg_proto
    monkeypatch.setenv("PGEMB_L2_TPR8", "1")
    monkeypatch.setenv("PGEMB_L2_TPR8_MIN_BYTES", "0")     # the small test rows too
    G.test_search_identical_to_oracle(pg, oracle_mod, "l2", G.SEARCH_CFGS[3])
    G.test_bind_links_identical_to_oracle(pg, oracle_mod, "l2", G.BIND_CFGS[0])


def test_peer_memory_exchange_two_shards(pg, oracle_mod):
    """K5 without a collective (pgemb_exchange_*): two id-range shards in one process (same_process attach), three steps so that both
    result parities and the flag sequence are used.  Every rank's merged answer == the reference per shard + a (dist,label)
    merge on the CPU (SURVEY.md 8(e)); the packed single-buffer merge (what ONE all-gather delivers) gives the same bytes."""
    from pg_embedding_b200 import _lib, sharded
    lib = _lib.load()
    rng = np.random.default_rng(12)
    n, dims, m, efc, ef, nq, world = 600, 12, 5, 20, 16, 23, 2
    x = rng.integers(0, 4, (n, dims)).astype(np.float32)            # ties across shards: the merge order is (dist,label)
    bounds = sharded.shard_bounds(n, world)
    idxs, orcs, exs = [], [], []
    for r, (lo, hi) in enumerate(bounds):
        labels = np.arange(lo, hi, dtype=np.uint64)
        orc = oracle_mod.FlatIndex("port", dims, m, efc, ef, "l2", capacity=hi - lo)
        orc.build(x[lo:hi], labels)
        idx = pg.HnswIndex(dims, m, efc, ef, "l2", capacity=hi - lo)
        idx.append(x[lo:hi], labels, orc.links())
        ex = C.c_void_p()
        _lib.check(lib.pgemb_exchange_create(0, r, world, 64, ef, C.byref(ex)))
        idxs.append(idx); orcs.append(orc); exs.append(ex)
    handles = (C.c_char * (64 * world))()
    for r in range(world):
        C.memmove(C.addressof(handles) + 64 * r, C.byref(C.c_void_p(lib.pgemb_exchange_buffer(exs[r]))), 8)
    for r in range(world):
        _lib.check(lib.pgemb_exchange_attach(exs[r], handles, 1))
    for step in range(3):
        q = rng.integers(0, 4, (nq - step, dims)).astype(np.float32)
        nqs = q.shape[0]
        for r in range(world):
            _lib.check(lib.pgemb_sharded_search_device(idxs[r].dev, exs[r], nqs, q.ctypes.data_as(C.c_void_p), ef, None))
        want = []
        for i in range(nqs):
            pairs = []
            for r in range(world):
                res = orcs[r].search(q[i], ef)
                d = oracle_mod.dist_many("port", "l2", q[i], x[res.astype(np.int64)])
                pairs += list(zip(d.tolist(), res.tolist()))
            want.append(sorted(pairs)[:ef])
        outs = []
        for r in range(world):
            ol = np.zeros((nqs, ef), np.uint64); od = np.zeros((nqs, ef), np.float32); on = np.zeros(nqs, np.int32)
            _lib.check(lib.pgemb_sharded_merge_device(exs[r], nqs, ol.ctypes.data_as(C.c_void_p), od.ctypes.data_as(C.c_void_p), on.ctypes.data_as(C.c_void_p), None))
            assert lib.pgemb_exchange_error(exs[r]) == 0
            for i in range(nqs):
                assert on[i] == len(want[i]) and ol[i, :on[i]].tolist() == [w[1] for w in want[i]], (step, r, i)
                assert od[i, :on[i]].tobytes() == np.array([w[0] for w in want[i]], np.float32).tobytes()
            outs.append((ol, od, on))
        assert outs[0][0].tobytes() == outs[1][0].tobytes()
        # the packed layout of ONE all-gather: [shard][labels | dists | counts]
        nbytes = int(lib.pgemb_packed_topk_bytes(nqs, ef))
        stride = (nbytes + 7) & ~7                 # every shard's block starts 8-byte aligned (u64 labels first)
        packed = np.zeros(world * stride, np.uint8)
        for r in range(world):
            o = idxs[r].search_batch(q, ef)
            lab, dd = o["labels"].copy(), o["dists"].copy()
            for i in range(nqs):                       # the device search pads with ~0 / +inf beyond n: same as the exchange area
                lab[i, o["n"][i]:] = np.uint64(0xFFFFFFFFFFFFFFFF); dd[i, o["n"][i]:] = np.inf
            packed[r * stride:r * stride + nbytes] = np.concatenate([lab.view(np.uint8).ravel(), dd.view(np.uint8).ravel(), o["n"].astype(np.int32).view(np.uint8).ravel()])
        ol = np.zeros((nqs, ef), np.uint64); od = np.zeros((nqs, ef), np.float32); on = np.zeros(nqs, np.int32)
        _lib.check(lib.pgemb_merge_topk_packed_device(nqs, world, ef, packed.ctypes.data_as(C.c_void_p), stride, od.ctypes.data_as(C.c_void_p),
                                                      ol.ctypes.data_as(C.c_void_p), on.ctypes.data_as(C.c_void_p), None))
        assert ol.tobytes() == outs[0][0].tobytes() and od.tobytes() == outs[0][1].tobytes() and on.tolist() == outs[0][2].tolist()
    # a merge whose peer never searched must give up and flag it, not hang
    _lib.check(lib.pgemb_sharded_search_device(idxs[0].dev, exs[0], nq, q.ctypes.data_as(C.c_void_p) if nq <= q.shape[0] else rng.integers(0, 4, (nq, dims)).astype(np.float32).ctypes.data_as(C.c_void_p), ef, None))
    for r in range(world):
        lib.pgemb_exchange_destroy(exs[r]); idxs[r].close(); orcs[r].close()


@pytest.mark.parametrize("metric,tc", [("cosine", "2"), ("l2", "2"), ("manhattan", "0")])
def test_sharded_scan_two_shards(pg, oracle_mod, monkeypatch, metric, tc):
    """BASELINE configs[4]'s step on two id-range shards in one process: pgemb_scan_topk_device == pgemb_scan_topk byte for byte, and
    pgemb_sharded_scan_device + the wait+merge kernel == the oracle's distances over the WHOLE table sorted by (dist,label)."""
    from pg_embedding_b200 import _lib, sharded
    lib = _lib.load()
    monkeypatch.setenv("PGEMB_SCAN_TC", tc)
    rng = np.random.default_rng(31)
    n, dims, k, nq, world = 900, 20, 12, 9, 2
    x = rng.integers(0, 3, (n, dims)).astype(np.float32) + (1.0 if metric == "cosine" else 0.0)   # ties across the shards
    labels_all = rng.permutation(n).astype(np.uint64) + np.uint64(5)
    labels_all[::13] |= np.uint64(1 << 48)                                                         # deleted rows
    bounds = sharded.shard_bounds(n, world)
    idxs, exs = [], []
    for r, (lo, hi) in enumerate(bounds):
        idx = pg.HnswIndex(dims, 4, 8, 16, metric, capacity=hi - lo)
        idx.append(x[lo:hi], labels_all[lo:hi])
        ex = C.c_void_p()
        _lib.check(lib.pgemb_exchange_create(0, r, world, 32, k, C.byref(ex)))
        idxs.append(idx); exs.append(ex)
    handles = (C.c_char * (64 * world))()
    for r in range(world):
        C.memmove(C.addressof(handles) + 64 * r, C.byref(C.c_void_p(lib.pgemb_exchange_buffer(exs[r]))), 8)
    for r in range(world):
        _lib.check(lib.pgemb_exchange_attach(exs[r], handles, 1))
    live = [j for j in range(n) if not (int(labels_all[j]) >> 48) & 1]
    for step in range(2):
        q = rng.integers(0, 3, (nq - step, dims)).astype(np.float32) + (1.0 if metric == "cosine" else 0.0)
        nqs = q.shape[0]
        for r in range(world):
            host = idxs[r].scan_topk(q, k)
            ol = np.zeros((nqs, k), np.uint64); od = np.zeros((nqs, k), np.float32); on = np.zeros(nqs, np.int32)
            _lib.check(lib.pgemb_scan_topk_device(idxs[r].dev, nqs, q.ctypes.data_as(C.c_void_p), k, ol.ctypes.data_as(C.c_void_p), od.ctypes.data_as(C.c_void_p),
                                                  on.ctypes.data_as(C.c_void_p), None))
            assert ol.tobytes() == host["labels"].tobytes() and od.tobytes() == host["dists"].tobytes() and on.tolist() == host["n"].tolist()
            _lib.check(lib.pgemb_sharded_scan_device(idxs[r].dev, exs[r], nqs, q.ctypes.data_as(C.c_void_p), k, None))
        for r in range(world):
            ol = np.zeros((nqs, k), np.uint64); od = np.zeros((nqs, k), np.float32); on = np.zeros(nqs, np.int32)
            _lib.check(lib.pgemb_sharded_merge_device(exs[r], nqs, ol.ctypes.data_as(C.c_void_p), od.ctypes.data_as(C.c_void_p), on.ctypes.data_as(C.c_void_p), None))
            assert lib.pgemb_exchange_error(exs[r]) == 0
            for i in range(nqs):
                d = oracle_mod.dist_many("port", metric, q[i], x)
                want = sorted((float(d[j]), int(labels_all[j])) for j in live)[:k]
                assert on[i] == len(want) and ol[i, :on[i]].tolist() == [w[1] for w in want], (metric, step, r, i)
                assert od[i, :on[i]].tobytes() == np.array([w[0] for w in want], np.float32).tobytes()
    assert lib.pgemb_sharded_scan_device(idxs[0].dev, exs[0], nq, q.ctypes.data_as(C.c_void_p), k + 1, None) == 2     # k differs from the exchange's
    for r in range(world):
        lib.pgemb_exchange_destroy(exs[r]); idxs[r].close()


def test_device_scan_edge_cases(pg, oracle_mod):
    import test_gpu_scan_umma as U
    U.check_device_scan_edge_cases(pg, oracle_mod, device_memory=False)


def test_ef_beyond_shared_memory(pg, G, oracle_mod, monkeypatch):
    """ef = 20000 through the library on the host: launch_search must fall back to the global-memory result queues by itself;
    PGEMB_RES_GLOBAL=1 forces that variant for ordinary searches too."""
    G.check_ef_beyond_shared_memory(pg, oracle_mod, 12, 300, (20000, 64))
    monkeypatch.setenv("PGEMB_RES_GLOBAL", "1")
    G.test_search_identical_to_oracle(pg, oracle_mod, "manhattan", G.SEARCH_CFGS[3])


def test_new_entry_points_argument_checks(pg):
    """Round-2 entry points fail loudly on bad arguments (status + message), never crash."""
    from pg_embedding_b200 import _lib
    lib = _lib.load()
    idx = pg.HnswIndex(4, 3, 8, 4, "l2", capacity=16)
    idx.append(np.eye(4, dtype=np.float32))
    assert lib.pgemb_index_poll_error(idx.dev, None) == 0                       # nothing raised
    assert lib.pgemb_index_poll_error(None, None) == 2
    sc = C.c_void_p()
    q = np.ones(4, np.float32)
    assert lib.pgemb_index_scan_begin(idx.dev, q.ctypes.data_as(C.POINTER(C.c_float)), 0, C.byref(sc)) == 2   # efsearch >= 1
    assert lib.pgemb_index_scan_begin(None, q.ctypes.data_as(C.POINTER(C.c_float)), 4, C.byref(sc)) == 2
    t = C.c_uint64(0)
    assert lib.pgemb_index_scan_next(None, C.byref(t)) == -2
    ex = C.c_void_p()
    assert lib.pgemb_exchange_create(0, 3, 2, 8, 4, C.byref(ex)) == 2           # rank >= world
    assert lib.pgemb_exchange_create(0, 0, 17, 8, 4, C.byref(ex)) == 2          # more than 16 shards
    _lib.check(lib.pgemb_exchange_create(0, 0, 2, 8, 4, C.byref(ex)))
    dq = np.ones((2, 4), np.float32)
    assert lib.pgemb_sharded_search_device(idx.dev, ex, 2, dq.ctypes.data_as(C.c_void_p), 4, None) == 4      # not attached yet
    assert b"attach" in lib.pgemb_last_error()
    handles = (C.c_char * 128)()
    assert lib.pgemb_exchange_attach(ex, handles, 1) == 2                        # null peer buffer
    lib.pgemb_exchange_destroy(ex)
    # one rank is its own world: search + merge degenerate to the local result
    _lib.check(lib.pgemb_exchange_create(0, 0, 1, 8, 4, C.byref(ex)))
    assert lib.pgemb_sharded_search_device(idx.dev, ex, 2, dq.ctypes.data_as(C.c_void_p), 5, None) == 2      # ef != k
    _lib.check(lib.pgemb_sharded_search_device(idx.dev, ex, 2, dq.ctypes.data_as(C.c_void_p), 4, None))
    ol = np.zeros((2, 4), np.uint64); od = np.zeros((2, 4), np.float32); on = np.zeros(2, np.int32)
    _lib.check(lib.pgemb_sharded_merge_device(ex, 2, ol.ctypes.data_as(C.c_void_p), od.ctypes.data_as(C.c_void_p), on.ctypes.data_as(C.c_void_p), None))
    want = idx.search_batch(dq, 4)
    assert ol.tobytes() == want["labels"].tobytes() and on.tolist() == want["n"].tolist()
    # the scan as the local step: same degenerate world, equals the host-pointer scan; argument errors
    assert lib.pgemb_sharded_scan_device(idx.dev, ex, 2, dq.ctypes.data_as(C.c_void_p), 3, None) == 2        # k != the exchange's
    assert lib.pgemb_sharded_scan_device(idx.dev, ex, 9, dq.ctypes.data_as(C.c_void_p), 4, None) == 2        # nq > max_nq
    assert lib.pgemb_sharded_scan_device(None, ex, 2, dq.ctypes.data_as(C.c_void_p), 4, None) == 2
    _lib.check(lib.pgemb_sharded_scan_device(idx.dev, ex, 2, dq.ctypes.data_as(C.c_void_p), 4, None))
    _lib.check(lib.pgemb_sharded_merge_device(ex, 2, ol.ctypes.data_as(C.c_void_p), od.ctypes.data_as(C.c_void_p), on.ctypes.data_as(C.c_void_p), None))
    want = idx.scan_topk(dq, 4)
    assert ol.tobytes() == want["labels"].tobytes() and od.tobytes() == want["dists"].tobytes() and on.tolist() == want["n"].tolist()
    assert lib.pgemb_scan_topk_device(idx.dev, 2, None, 4, ol.ctypes.data_as(C.c_void_p), None, on.ctypes.data_as(C.c_void_p), None) == 2   # null queries
    assert lib.pgemb_scan_topk_device(idx.dev, 2, dq.ctypes.data_as(C.c_void_p), 0, ol.ctypes.data_as(C.c_void_p), None, on.ctypes.data_as(C.c_void_p), None) == 2   # k = 0
    _lib.check(lib.pgemb_scan_topk_device(idx.dev, 2, dq.ctypes.data_as(C.c_void_p), 4, ol.ctypes.data_as(C.c_void_p), None, on.ctypes.data_as(C.c_void_p), None))    # distances optional
    assert ol.tobytes() == want["labels"].tobytes()
    lib.pgemb_exchange_destroy(ex)
    idx.close()
