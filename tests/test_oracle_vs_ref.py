"""Pins the C restatement (oracle/hnsw_oracle.c, `port`) to the UNMODIFIED compiled reference
(oracle/_ref, `ref`) bit for bit: distances for every dim / metric, link lists after sequential
builds, and search results -- including duplicate vectors (exact distance ties).

What the reference returns on these seeded inputs is stored as SHA-256 digests of the raw bytes in
tests/golden/ref_outputs.json (written from oracle/_ref by tests/golden/gen_ref_outputs.py), so the
comparison runs without the reference tree.  Where oracle/_ref is built, the port is also compared with
it directly."""
import hashlib
import json
import os

import numpy as np
import pytest

METRICS = ["l2", "cosine", "manhattan"]
GOLD = os.path.join(os.path.dirname(__file__), "golden", "ref_outputs.json")


def digest(a) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def check_against_reference(oracle_mod, section, outputs):
    """outputs(which) -> {key: array}: the port's arrays must be the reference's, byte for byte."""
    want = json.load(open(GOLD))[section]
    got = outputs("port")
    assert sorted(got) == sorted(want)
    for key, a in got.items():
        assert digest(a) == want[key], f"{key}: differs from the compiled reference's stored output"
    if oracle_mod.available("ref"):
        for key, r in outputs("ref").items():
            a = got[key]
            assert r.tobytes() == a.tobytes(), (key, np.flatnonzero(r.ravel() != a.ravel())[:5])


def distance_outputs(oracle_mod, metric):
    def outputs(which):
        rng = np.random.default_rng(7)
        dims = list(range(1, 70)) + [96, 100, 127, 128, 129, 255, 256, 300, 768, 769, 1000, 1536, 2000]
        out = {}
        for dim in dims:
            a = rng.standard_normal((64, dim)).astype(np.float32)
            b = rng.standard_normal((64, dim)).astype(np.float32)
            # mix magnitudes so that rounding order matters
            a *= rng.choice([1e-3, 1.0, 37.0], size=(64, 1)).astype(np.float32)
            out[f"d{dim}"] = oracle_mod.dist_many(which, metric, a, b)
            out[f"d{dim}/broadcast"] = oracle_mod.dist_many(which, metric, a[0], b)  # broadcast query form
        return out
    return outputs


@pytest.mark.parametrize("metric", METRICS)
def test_distance_bits_all_dims(oracle_mod, metric):
    check_against_reference(oracle_mod, f"distance_bits/{metric}", distance_outputs(oracle_mod, metric))


def cosine_parts_outputs(oracle_mod):
    """|b|^2 cached per node + dot (port) against the reference's hnsw_dist_func (ref) on the same pairs."""
    import ctypes as C

    def outputs(which):
        rng = np.random.default_rng(3)
        out = {}
        for dim in [1, 3, 4, 5, 17, 128, 768, 1001]:
            d = np.empty(20, np.float32)
            for i in range(20):
                a = rng.standard_normal(dim).astype(np.float32)
                b = rng.standard_normal(dim).astype(np.float32)
                if which == "port":
                    d[i] = oracle_mod.load("port").oracle_cosine_from_parts(a.ctypes.data_as(C.POINTER(C.c_float)),
                                                                            b.ctypes.data_as(C.POINTER(C.c_float)), dim)
                else:
                    d[i] = oracle_mod.dist("ref", "cosine", a, b)
            out[f"d{dim}"] = d
        return out
    return outputs


def test_cosine_parts_recompose(oracle_mod):
    """|b|^2 cached per node + dot recomposes to the exact reference cosine distance."""
    check_against_reference(oracle_mod, "cosine_parts", cosine_parts_outputs(oracle_mod))


def _data(rng, n, dim, dup_frac=0.0, clustered=False):
    if clustered:
        c = rng.standard_normal((max(4, int(np.sqrt(n))), dim)).astype(np.float32)
        x = c[rng.integers(0, len(c), n)] + 0.3 * rng.standard_normal((n, dim)).astype(np.float32)
    else:
        x = rng.standard_normal((n, dim)).astype(np.float32)
    if dup_frac > 0:
        k = int(n * dup_frac)
        src = rng.integers(0, n, k)
        dst = rng.integers(0, n, k)
        x[dst] = x[src]
    return np.ascontiguousarray(x, dtype=np.float32)


CONFIGS = [
    # dims, m, efC, efS, n, dup_frac, clustered
    (3, 3, 16, 64, 200, 0.3, False),
    (8, 4, 10, 16, 600, 0.2, False),
    (16, 8, 40, 32, 1500, 0.0, True),
    (33, 5, 20, 64, 800, 0.1, True),
    (128, 16, 64, 64, 1200, 0.0, True),
]
CONFIG_IDS = [f"d{c[0]}m{c[1]}n{c[4]}" for c in CONFIGS]


def build_and_search_outputs(oracle_mod, metric, cfg):
    dims, m, efc, efs, n, dup, clustered = cfg

    def outputs(which):
        rng = np.random.default_rng(hash((dims, m, n)) % (2**32))
        x = _data(rng, n, dims, dup, clustered)
        if metric == "cosine":
            x += 0.01  # avoid exact zero vectors (NaN distance in the reference, distfunc.c:144)
        q = _data(rng, 50, dims, 0.0, clustered)
        q[:10] = x[:10]  # exact hits
        idx = oracle_mod.FlatIndex(which, dims, m, efc, efs, metric, capacity=n)
        idx.build(x)
        out = {"links": idx.links()}
        for ef in (1, 5, efs):
            r = idx.search_many(q, ef, nthreads=2 if which == "ref" else 1, want_counters=True)
            out[f"ef{ef}/n"], out[f"ef{ef}/labels"] = r["n"], r["labels"]
            out[f"ef{ef}/counters"] = r["counters"]  # identical traversal work
        # deleted labels are post-filtered identically
        for i in range(0, n, 3):
            idx.mark_deleted(i)
        r = idx.search_many(q, efs)
        out["deleted/n"], out["deleted/labels"] = r["n"], r["labels"]
        idx.close()
        return out
    return outputs


@pytest.mark.parametrize("metric", METRICS)
@pytest.mark.parametrize("cfg", CONFIGS, ids=CONFIG_IDS)
def test_build_and_search_identical(oracle_mod, metric, cfg):
    check_against_reference(oracle_mod, f"build_and_search/{metric}/{CONFIG_IDS[CONFIGS.index(cfg)]}",
                            build_and_search_outputs(oracle_mod, metric, cfg))
