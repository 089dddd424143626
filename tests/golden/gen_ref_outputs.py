#!/usr/bin/env python
"""Generate tests/golden/ref_outputs.json from the UNMODIFIED compiled reference (oracle/_ref/libpgemb_ref.so, built in place
from the reference's hnswalg.cpp + distfunc.c by oracle/Makefile; PGEMB_REFERENCE_DIR names the reference tree):

    python tests/golden/gen_ref_outputs.py

It holds what the reference returns on the seeded inputs of tests/test_oracle_vs_ref.py (SHA-256 digests of the raw output
bytes: distances, link lists, search labels, counts and traversal counters) and on the regress cases of
tests/test_oracle_kat.py (labels and distance bits), and the field names of HnswMetadata in its embedding.h
(tests/test_abi.py), so that those tests compare with the reference without the reference tree."""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
from oracle import oracle  # noqa: E402
import test_abi  # noqa: E402
import test_oracle_kat as kat  # noqa: E402
import test_oracle_vs_ref as vs  # noqa: E402

oracle.build("ref")
assert oracle.available("ref"), "needs the reference tree to build oracle/_ref"


def digests(outputs):
    return {k: vs.digest(a) for k, a in outputs("ref").items()}


out = {}
for metric in vs.METRICS:
    out[f"distance_bits/{metric}"] = digests(vs.distance_outputs(oracle, metric))
out["cosine_parts"] = digests(vs.cosine_parts_outputs(oracle))
for cfg, cid in zip(vs.CONFIGS, vs.CONFIG_IDS):
    for metric in vs.METRICS:
        out[f"build_and_search/{metric}/{cid}"] = digests(vs.build_and_search_outputs(oracle, metric, cfg))
out["metadata_fields"] = test_abi.reference_metadata_fields(os.path.join(oracle.REF_SRC, "embedding.h"))
out["kat"] = {c["name"]: {m: kat.kat_answer(oracle, "ref", c, m) for m in kat.metrics(c)} for c in kat.CASES}
with open(os.path.join(HERE, "ref_outputs.json"), "w") as f:
    json.dump(out, f, indent=1, sort_keys=True)
    f.write("\n")
print("wrote ref_outputs.json with", len(out), "sections")
