"""GPU tests of K6, the tensor-core path of the brute-force operator scan (csrc/scan_umma_kernel.cuh; SURVEY.md 8(f3)):

* the raw tcgen05 products (TMA swizzled tiles -> UMMA descriptors -> TMEM -> tcgen05.ld) against a float64 product,
  inside the TF32 error bound the filter assumes, over tile-edge shapes;
* pgemb_scan_topk through the filter == the exact kernels, bit for bit (labels, order, distances), == the oracle's
  distances sorted by (dist,label): ties, duplicates, deleted labels, k > N, ragged dims, several chunks, candidate-list
  overflow, several query tiles.

tests/test_capi_emulated.py reuses the bodies on the emulated library (the filter predicate, the chunk orchestration, the
re-scoring kernel; the tcgen05 kernel itself only runs here)."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pg():
    import pg_embedding_b200 as pg
    from pg_embedding_b200 import build
    build.build()
    if pg.device_count() < 1:
        pytest.fail("no CUDA device: the product path has no CPU fallback")
    return pg


def counters():
    from pg_embedding_b200 import _lib
    out = (C.c_uint64 * 6)()
    _lib.load().pgemb_scan_counters(out)
    return dict(tc=out[0], pairs=out[1], rescored=out[2], fallbacks=out[3], overflow=out[4], exact=out[5])


def rel_bound(dims):
    return 1.5 * (2.0 / 1024.0 + dims / 2097152.0)


def umma_product(pg, idx, q, r0, nr):
    from pg_embedding_b200 import _lib
    q = np.ascontiguousarray(q, np.float32)
    out = np.empty((q.shape[0], nr), np.float32)
    _lib.check(_lib.load().pgemb_debug_umma_product(idx.dev, q.shape[0], q.ctypes.data_as(C.POINTER(C.c_float)), r0, nr,
                                                    out.ctypes.data_as(C.POINTER(C.c_float))))
    return out


PRODUCT_SHAPES = [  # dims, rows, nq, r0, nr
    (3, 5, 1, 0, 5), (32, 256, 128, 0, 256), (33, 700, 129, 7, 600), (100, 1000, 37, 256, 511), (768, 3000, 260, 1, 2999), (1536, 900, 130, 300, 600),
    (2000, 300, 5, 0, 300),
]


@pytest.mark.parametrize("shape", PRODUCT_SHAPES, ids=[f"d{s[0]}n{s[1]}q{s[2]}" for s in PRODUCT_SHAPES])
def test_umma_product_within_tf32_bound(pg, shape):
    dims, n, nq, r0, nr = shape
    rng = np.random.default_rng(dims * 31 + n)
    x = rng.standard_normal((n, dims)).astype(np.float32)
    q = rng.standard_normal((nq, dims)).astype(np.float32)
    x[n // 2] *= 37.0                      # rows of very different norms
    q[0] *= 0.01
    idx = pg.HnswIndex(dims, 4, 8, 16, "l2", capacity=n)
    idx.append(x)
    got = umma_product(pg, idx, q, r0, nr)
    want = q.astype(np.float64) @ x[r0:r0 + nr].astype(np.float64).T
    bound = rel_bound(dims) / 1.5 * np.outer(np.linalg.norm(q.astype(np.float64), axis=1), np.linalg.norm(x[r0:r0 + nr].astype(np.float64), axis=1))
    err = np.abs(got - want)
    assert np.isfinite(got).all()
    assert (err <= bound + 1e-30).all(), f"max err/bound {np.max(err / (bound + 1e-30)):.3f} at {np.unravel_index(np.argmax(err / (bound + 1e-30)), err.shape)}"
    # and it really is a reduced-precision product, not an fp32 one, once the dimension is long enough to tell
    if dims >= 768:
        assert np.max(err / (bound + 1e-30)) > 1e-3
    idx.close()


def _clusters(rng, n, dims, nc=12, noise=0.15, shift=0.0):
    c = rng.standard_normal((nc, dims)).astype(np.float32)
    return (c[rng.integers(0, nc, n)] + noise * rng.standard_normal((n, dims))).astype(np.float32) + np.float32(shift), c


SCAN_CASES = [  # dims, n, k, nq
    (3, 40, 64, 5), (33, 3000, 64, 40), (128, 30000, 10, 70), (100, 5000, 300, 130), (768, 40000, 10, 300), (1536, 6000, 64, 17),
]


def check_scan_equals_exact(pg, oracle_mod, metric, case, monkeypatch, full_oracle=True):
    dims, n, k, nq = case
    rng = np.random.default_rng(23 + dims)
    shift = 1.0 if metric == "cosine" else 0.0
    x, c = _clusters(rng, n, dims, shift=shift)
    q = (c[rng.integers(0, len(c), nq)] + 0.15 * rng.standard_normal((nq, dims))).astype(np.float32) + np.float32(shift)
    if n > 10:
        x[n // 2] = x[n // 3]              # an exact tie: ordered by label
        x[n // 5] = q[0]                   # distance exactly 0 (L2) for one pair
    labels = rng.permutation(n).astype(np.uint64) + np.uint64(3)
    labels[::11] |= np.uint64(1 << 48)     # deleted rows are skipped
    idx = pg.HnswIndex(dims, 4, 8, 16, metric, capacity=n)
    idx.append(x, labels)
    monkeypatch.setenv("PGEMB_SCAN_TC", "0")
    want = idx.scan_topk(q, k)
    c0 = counters()
    monkeypatch.setenv("PGEMB_SCAN_TC", "2")
    got = idx.scan_topk(q, k)
    c1 = counters()
    assert got["n"].tolist() == want["n"].tolist()
    assert got["labels"].tobytes() == want["labels"].tobytes(), (metric, case)
    assert got["dists"].tobytes() == want["dists"].tobytes()
    assert c1["tc"] == c0["tc"] + 1 and c1["fallbacks"] == c0["fallbacks"], "the TF32 error bound was exceeded (tripwire)"
    frac = (c1["rescored"] - c0["rescored"]) / max(1, c1["pairs"] - c0["pairs"])
    print(f"K6 {metric} dims={dims} n={n} k={k} nq={nq}: {frac:.4f} of the pairs re-scored exactly, overflowed queries {c1['overflow'] - c0['overflow']}")
    if n >= 30000:
        assert frac < 0.2, "the filter discarded almost nothing"
    if full_oracle:
        live = [j for j in range(n) if not (int(labels[j]) >> 48) & 1]
        for i in range(0, nq, max(1, nq // 8)):
            d = oracle_mod.dist_many("port", metric, q[i], x)
            order = sorted((float(d[j]), int(labels[j])) for j in live)[:k]
            assert got["labels"][i, :len(order)].tolist() == [o[1] for o in order], (metric, case, i)
            assert got["dists"][i, :len(order)].tobytes() == np.array([o[0] for o in order], np.float32).tobytes()
    idx.close()


@pytest.mark.parametrize("metric", ["l2", "cosine"])
@pytest.mark.parametrize("case", SCAN_CASES, ids=[f"d{c[0]}n{c[1]}k{c[2]}" for c in SCAN_CASES])
def test_scan_umma_equals_exact_path(pg, oracle_mod, metric, case, monkeypatch):
    check_scan_equals_exact(pg, oracle_mod, metric, case, monkeypatch)


def check_scan_overflow_and_chunks(pg, oracle_mod, metric, monkeypatch, n=5000, dims=24):
    """Tiny candidate lists (every query overflows -> whole-chunk exact re-scoring) and tiny first chunks (many chunks,
    the threshold is handed from chunk to chunk): still the exact path's result."""
    rng = np.random.default_rng(5)
    x = (rng.integers(0, 3, (n, dims))).astype(np.float32) + (1.0 if metric == "cosine" else 0.0)   # heavy ties / duplicates
    q = (rng.integers(0, 3, (50, dims))).astype(np.float32) + (1.0 if metric == "cosine" else 0.0)
    idx = pg.HnswIndex(dims, 4, 8, 16, metric, capacity=n)
    idx.append(x)
    monkeypatch.setenv("PGEMB_SCAN_TC", "0")
    want = idx.scan_topk(q, 20)
    monkeypatch.setenv("PGEMB_SCAN_TC", "2")
    for env in ({"PGEMB_SCAN_TC_CAP": "16"}, {"PGEMB_SCAN_TC_CHUNK0_LOG2": "5"}, {"PGEMB_SCAN_TC_CAP": "64", "PGEMB_SCAN_TC_CHUNK0_LOG2": "6"}):
        for kk, vv in env.items():
            monkeypatch.setenv(kk, vv)
        c0 = counters()
        got = idx.scan_topk(q, 20)
        c1 = counters()
        assert got["labels"].tobytes() == want["labels"].tobytes() and got["dists"].tobytes() == want["dists"].tobytes(), env
        if env.get("PGEMB_SCAN_TC_CAP") == "16":      # smaller than the first chunk: every query overflows there
            assert c1["overflow"] > c0["overflow"]
        for kk in env:
            monkeypatch.delenv(kk)
    idx.close()


@pytest.mark.parametrize("metric", ["l2", "cosine"])
def test_scan_umma_overflow_and_chunks(pg, oracle_mod, metric, monkeypatch):
    check_scan_overflow_and_chunks(pg, oracle_mod, metric, monkeypatch)


def test_scan_umma_l2_norm_cache_follows_appends(pg, oracle_mod, monkeypatch):
    """L2 indexes compute row norms lazily for the filter: rows appended after a scan must get theirs."""
    rng = np.random.default_rng(8)
    dims, n = 40, 6000
    x, c = _clusters(rng, n, dims)
    q = x[rng.integers(0, n, 30)] + 0.01
    idx = pg.HnswIndex(dims, 4, 8, 16, "l2", capacity=n)
    idx.append(x[:4000])
    monkeypatch.setenv("PGEMB_SCAN_TC", "2")
    a = idx.scan_topk(q, 10)
    idx.append(x[4000:])
    b = idx.scan_topk(q, 10)
    monkeypatch.setenv("PGEMB_SCAN_TC", "0")
    want = idx.scan_topk(q, 10)
    assert b["labels"].tobytes() == want["labels"].tobytes() and b["dists"].tobytes() == want["dists"].tobytes()
    assert a["labels"].max() < 4000
    idx.close()


def test_scan_umma_default_policy(pg, monkeypatch):
    """PGEMB_SCAN_TC unset: tables of >= 4096 rows take the tensor-core path for L2 / cosine, manhattan never does."""
    monkeypatch.delenv("PGEMB_SCAN_TC", raising=False)
    rng = np.random.default_rng(2)
    for metric, n, expect_tc in (("l2", 5000, True), ("cosine", 1000, False), ("manhattan", 5000, False)):
        x = rng.standard_normal((n, 16)).astype(np.float32)
        idx = pg.HnswIndex(16, 4, 8, 16, metric, capacity=n)
        idx.append(x)
        c0 = counters()
        idx.scan_topk(x[:3], 5)
        c1 = counters()
        assert (c1["tc"] - c0["tc"] == 1) == expect_tc and (c1["exact"] - c0["exact"] == 1) == (not expect_tc), (metric, n)
        idx.close()


def check_device_scan_edge_cases(pg, oracle_mod, device_memory=True):
    """pgemb_scan_topk_device on tables smaller than k, on an empty table and with every row deleted: counts, fill values
    (~0 / +inf) and the host-pointer call's bytes.  device_memory=False for the host-emulated library, whose "device"
    pointers are host pointers (a machine with a GPU runs that test too, so torch seeing a device does not decide it)."""
    from pg_embedding_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(3)
    k, nq, dims = 6, 4, 5
    q = rng.standard_normal((nq, dims)).astype(np.float32)
    for n, deleted in ((0, False), (3, False), (3, True), (40, False)):
        idx = pg.HnswIndex(dims, 3, 8, 4, "l2", capacity=max(n, 1))
        x = rng.standard_normal((n, dims)).astype(np.float32)
        if n:
            labels = np.arange(n, dtype=np.uint64) + np.uint64(7)
            if deleted:
                labels |= np.uint64(1 << 48)
            idx.append(x, labels)
        ol = np.full((nq, k), 123, np.uint64); od = np.full((nq, k), 5.0, np.float32); on = np.full(nq, -1, np.int32)
        if device_memory:                  # a real device: the entry point takes device pointers
            import torch
            tq = torch.from_numpy(q).cuda(); tl = torch.from_numpy(ol.view(np.int64)).cuda(); td = torch.from_numpy(od).cuda(); tn = torch.from_numpy(on).cuda()
            _lib.check(lib.pgemb_scan_topk_device(idx.dev, nq, tq.data_ptr(), k, tl.data_ptr(), td.data_ptr(), tn.data_ptr(), None))
            torch.cuda.synchronize()
            ol, od, on = tl.cpu().numpy().view(np.uint64), td.cpu().numpy(), tn.cpu().numpy()
        else:                              # the host-emulated library (tests/test_capi_emulated.py): all memory is host memory
            _lib.check(lib.pgemb_scan_topk_device(idx.dev, nq, q.ctypes.data_as(C.c_void_p), k, ol.ctypes.data_as(C.c_void_p), od.ctypes.data_as(C.c_void_p),
                                                  on.ctypes.data_as(C.c_void_p), None))
        live = 0 if deleted else n
        assert on.tolist() == [min(k, live)] * nq, (n, deleted)
        assert (ol[:, min(k, live):] == np.uint64(0xFFFFFFFFFFFFFFFF)).all() and np.isinf(od[:, min(k, live):]).all()
        host = idx.scan_topk(q, k)
        assert ol.tobytes() == host["labels"].tobytes() and od.tobytes() == host["dists"].tobytes() and on.tolist() == host["n"].tolist()
        if live:
            for i in range(nq):
                d = oracle_mod.dist_many("port", "l2", q[i], x)
                want = sorted((float(d[j]), j + 7) for j in range(n))[:k]
                assert ol[i, :len(want)].tolist() == [w[1] for w in want]
        idx.close()


def test_device_scan_edge_cases(pg, oracle_mod):
    check_device_scan_edge_cases(pg, oracle_mod)
