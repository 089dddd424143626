"""Known-answer tests: both CPU checkers (compiled reference `ref`, C restatement `port`) against the
results the reference's own pg_regress suite pins (tests/golden/kat_regress.json, transcribed from the
reference's test/expected/*.out)."""
import json
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(__file__), "golden", "kat_regress.json")
CASES = json.load(open(GOLD))["cases"]
REF = os.path.join(os.path.dirname(__file__), "golden", "ref_outputs.json")


def tid_label(blk: int, pos: int, flags: int = 0) -> int:
    """HnswLabel (embedding.c:50-56): {BlockIdData{bi_hi,bi_lo}, ip_posid, flags} as a little-endian u64."""
    return (blk >> 16) | ((blk & 0xFFFF) << 16) | (pos << 32) | (flags << 48)


def run_case(oracle_mod, which, case, metric):
    """The case's inserts, TRUNCATE and deletes through checker `which`; the labels hnsw_search returns for its query."""
    o = case["options"]
    idx = oracle_mod.FlatIndex(which, o["dims"], o["m"], o["efconstruction"], o["efsearch"], metric, capacity=64)
    for r in case.get("rows_before_truncate", []):
        idx.add(np.array(r["val"], np.float32), tid_label(*r["tid"]))
    if "rows_before_truncate" in case:
        idx.truncate()  # TRUNCATE gives the index a fresh, empty relation (gh-3)
    for r in case["rows"]:
        idx.add(np.array(r["val"], np.float32), tid_label(*r["tid"]))
    if "delete_all_then_insert" in case:
        for i in range(len(idx)):
            idx.mark_deleted(i)  # ambulkdelete after `delete from t; vacuum t`
        for r in case["delete_all_then_insert"]:
            idx.add(np.array(r["val"], np.float32), tid_label(*r["tid"]))
    return [int(l) for l in idx.search(np.array(case["query"], np.float32))]


def rows_by_label(case):
    """The rows a search can return (those inserted after the last delete-all), by label."""
    return {tid_label(*r["tid"]): r for r in case.get("delete_all_then_insert", case["rows"])}


def metrics(case):
    return list(case.get("expected", case.get("expected_tids")).keys())


def kat_answer(oracle_mod, which, case, metric):
    """What checker `which` answers: the labels and the fp32 bits of their distances (hnsw_dist_func) to the query."""
    labels = run_case(oracle_mod, which, case, metric)
    by_label = rows_by_label(case)
    q = np.array(case["query"], np.float32)
    bits = [int(oracle_mod.dist(which, metric, q, np.array(by_label[l]["val"], np.float32)).view(np.uint32)) for l in labels]
    return {"labels": labels, "dist_bits": bits}


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
@pytest.mark.parametrize("which", ["port", "ref"])
def test_kat(oracle_mod, which, case):
    """The regress results, per checker.  `port`: the C restatement runs here; its answer must be the regress suite's and,
    bit for bit, the compiled reference's as stored in tests/golden/ref_outputs.json.  `ref`: where oracle/_ref is built,
    the compiled reference runs here and its answer must be the regress suite's and the stored one.  Where it is NOT
    built, nothing of the reference runs: this case then only checks the stored reference answers against the regress
    results, i.e. the two golden files against each other."""
    stored = json.load(open(REF))["kat"][case["name"]]
    by_label = rows_by_label(case)
    for metric in metrics(case):
        if which == "port" or oracle_mod.available("ref"):
            ans = kat_answer(oracle_mod, which, case, metric)
            assert ans == stored[metric], (which, metric)
        else:                   # no compiled reference here: the golden-file consistency check described above
            ans = stored[metric]
        rows = [by_label[l] for l in ans["labels"]]
        if "expected" in case:
            assert [r["val"] for r in rows] == case["expected"][metric], (which, metric)
        if "expected_tids" in case:
            assert [r["tid"] for r in rows] == case["expected_tids"][metric], (which, metric)
        if "expected_distances" in case:
            got = np.array(ans["dist_bits"], np.uint32).view(np.float32)
            np.testing.assert_allclose(got, case["expected_distances"][metric], rtol=0, atol=5e-7)


def test_kat_seqscan_equals_index(oracle_mod):
    """knn.out:63-91: the seq-scan (exact) order equals the index order on the KAT data, all 3 metrics."""
    case = CASES[0]
    q = np.array(case["query"], np.float32)
    for metric in ("l2", "cosine", "manhattan"):
        vals = [np.array(r["val"], np.float32) for r in case["rows"]]
        labs = [tid_label(*r["tid"]) for r in case["rows"]]
        d = [float(oracle_mod.dist("port", metric, q, v)) for v in vals]
        order = sorted(range(len(vals)), key=lambda i: (d[i], labs[i]))
        assert [case["rows"][i]["val"] for i in order] == case["expected"][metric]
