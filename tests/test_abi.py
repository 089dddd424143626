"""CPU-side checks of the drop-in boundary: the C-ABI library loads, exports every symbol
include/pgemb_b200.h declares, HnswMetadata has the reference's layout, and the product path fails
loudly (no fallback) when no CUDA device is usable."""
import ctypes as C
import json
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from pg_embedding_b200 import build
    build.build()
    from pg_embedding_b200 import _lib
    return _lib.load()


def test_exports_every_declared_symbol(lib):
    from pg_embedding_b200 import _lib
    header = open(os.path.join(ROOT, "include", "pgemb_b200.h")).read()
    declared = set(re.findall(r"\b((?:pgemb|hnsw)_[a-z_0-9]+)\s*\(", header))
    declared -= {"pgemb_status", "pgemb_index"}
    assert declared, "no prototypes parsed"
    assert declared == set(_lib.ABI_SYMBOLS), declared ^ set(_lib.ABI_SYMBOLS)
    for name in declared:
        assert hasattr(lib, name), f"{name} not exported by libpgemb_b200.so"


def test_metadata_layout_matches_reference(lib):
    from pg_embedding_b200._lib import HnswMetadata
    # embedding.h:28-42: 10 size_t + idx_t + enum
    assert C.sizeof(HnswMetadata) == 10 * 8 + 4 + 4
    assert HnswMetadata.enterpoint_node.offset == 80 and HnswMetadata.dist_func.offset == 84
    fields = [f[0] for f in HnswMetadata._fields_]
    # the reference's field names, as stored from its embedding.h by tests/golden/gen_ref_outputs.py
    assert fields == json.load(open(os.path.join(ROOT, "tests", "golden", "ref_outputs.json")))["metadata_fields"]
    ref_dir = os.environ.get("PGEMB_REFERENCE_DIR")
    if ref_dir and os.path.isfile(os.path.join(ref_dir, "embedding.h")):   # and the reference tree itself where it is present
        assert reference_metadata_fields(os.path.join(ref_dir, "embedding.h")) == fields


def reference_metadata_fields(embedding_h):
    """HnswMetadata's field names in the reference's embedding.h, in declaration order."""
    return re.findall(r"^\s*(?:size_t|idx_t|dist_func_t)\s+(\w+);", open(embedding_h).read(), re.M)


def test_meta_init_follows_hnsw_get_index(lib):
    from pg_embedding_b200._lib import HnswMetadata
    m = HnswMetadata()
    assert lib.pgemb_meta_init(C.byref(m), 768, 32, 200, 64, 1) == 0
    assert (m.dim, m.M, m.maxM, m.efConstruction, m.efSearch, m.dist_func) == (768, 32, 64, 200, 64, 1)
    assert m.offset_data == 65 * 4 and m.offset_label == 260 + 3072 and m.size_data_per_element == 3340
    assert m.elems_per_page == 2  # SURVEY.md section 8: d=768/m=32 -> 3340 B, 2 per page
    assert lib.pgemb_meta_init(C.byref(m), 3, 3, 16, 64, 0) == 0
    assert m.size_data_per_element == 48 and m.elems_per_page == 157
    assert lib.pgemb_meta_init(C.byref(m), 0, 3, 16, 64, 0) != 0          # dims required (embedding.c:219)
    assert b"dims" in lib.pgemb_last_error()
    assert lib.pgemb_meta_init(C.byref(m), 4000, 32, 16, 64, 0) != 0      # record does not fit a page (:229)


def test_is_deleted_flag(lib):
    assert lib.hnsw_is_deleted(1 << 48) and not lib.hnsw_is_deleted((1 << 48) - 1)
    assert not lib.hnsw_is_deleted(2 << 48)


def test_no_silent_cpu_fallback(lib):
    """Without a CUDA device every compute entry point must FAIL, never compute on the CPU."""
    if lib.pgemb_device_count() > 0:
        pytest.skip("CUDA device present")
    from pg_embedding_b200._lib import HnswMetadata
    m = HnswMetadata()
    assert lib.pgemb_meta_init(C.byref(m), 3, 3, 16, 64, 0) == 0
    h = C.c_void_p()
    assert lib.pgemb_index_create(C.byref(m), 16, 0, C.byref(h)) != 0
    a = np.ones(3, np.float32)
    out = np.zeros(1, np.float32)
    fp = C.POINTER(C.c_float)
    assert lib.pgemb_dist_batch(0, 3, 1, a.ctypes.data_as(fp), 0, a.ctypes.data_as(fp), out.ctypes.data_as(fp)) != 0
    assert np.isnan(lib.hnsw_dist_func(0, a.ctypes.data_as(fp), a.ctypes.data_as(fp), 3))


def test_product_does_not_import_oracle():
    """The product package must not reference oracle/ (rule: oracle is test infrastructure only)."""
    pkg = os.path.join(ROOT, "pg_embedding_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f), errors="replace").read()
                assert "import oracle" not in src and "from oracle" not in src and "libpgemb_port" not in src \
                    and "libpgemb_ref" not in src, f


def test_product_library_is_blackwell_native(lib):
    """SASS evidence (B200_PROFILING.md "What proves a Blackwell-native kernel"): the traversal gathers rows with the bulk-copy
    engine (UBLKCP + mbarrier SYNCS), the brute-force scan's dense contraction runs on the 5th-gen tensor cores
    (tcgen05.mma -> UTC*MMA, TMEM read-back LDTM, 2-D TMA tensor-map loads UTMALDG) -- and nothing is a legacy mma.sync/wgmma
    path or a library GEMM (no cuBLAS symbol, no HMMA)."""
    import shutil
    import subprocess
    from pg_embedding_b200 import build
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.isfile(cuobjdump):
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([cuobjdump, "-sass", build.OUT], capture_output=True, text=True).stdout
    ops = {}
    fn = None
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            fn = m.group(1)
            continue
        m = re.search(r"\s(UTC[A-Z0-9]*MMA|LDTM|UTMALDG|UBLKCP|HMMA|HGMMA|UTCBAR)\b", line)
        if m and fn:
            ops.setdefault(fn, {}).setdefault(m.group(1), 0)
            ops[fn][m.group(1)] += 1
    umma = [f for f in ops if "scan_filter_umma_kernel" in f]
    assert len(umma) == 2, umma                                   # L2 and cosine
    for f in umma:
        assert any(k.startswith("UTC") and k.endswith("MMA") for k in ops[f]), (f, ops[f])
        assert ops[f].get("LDTM", 0) >= 1 and ops[f].get("UTMALDG", 0) >= 2 and ops[f].get("UTCBAR", 0) >= 2, (f, ops[f])
    search = [f for f in ops if "search_kernel" in f]
    assert len(search) == 11                                      # 3 metrics x 2 modes + the 8-lanes-per-row L2 pair + 3 huge-ef variants
    for f in search:
        assert ops[f].get("UBLKCP", 0) >= 2, (f, ops[f])
    assert not any("HMMA" in v or "HGMMA" in v for v in ops.values())
    needed = subprocess.run(["ldd", build.OUT], capture_output=True, text=True).stdout
    assert "cublas" not in needed.lower()
    assert "cublas" not in open(os.path.join(ROOT, "pg_embedding_b200", "csrc", "capi.cu")).read().lower()


def test_client_library_exports_the_reference_symbols_and_no_cuda():
    """libpgemb_client.so (what a forked backend links instead of hnswalg.o distfunc.o when a sidecar owns the GPU) exports
    the algorithm-side symbols of embedding.h:44-56 plus everything include/pgemb_client.h declares, and has no CUDA in it."""
    import subprocess
    from pg_embedding_b200 import build
    _, client_path = build.build_sidecar()
    lib = C.CDLL(client_path)
    header = open(os.path.join(ROOT, "include", "pgemb_client.h")).read()
    declared = set(re.findall(r"\b(pgemb_client_[a-z_0-9]+)\s*\(", header))
    assert len(declared) >= 12
    for name in declared | {"hnsw_search", "hnsw_bind_point", "hnsw_dist_func", "hnsw_init_dist_func", "hnsw_is_deleted"}:
        assert hasattr(lib, name), f"{name} not exported by libpgemb_client.so"
    needed = subprocess.run(["ldd", client_path], capture_output=True, text=True).stdout
    assert "cuda" not in needed.lower() and "pgemb_b200" not in needed
    # without a sidecar every call fails -- there is nothing to fall back to
    import numpy as np
    lib.hnsw_dist_func.restype = C.c_float
    a = np.ones(4, np.float32)
    os.environ.pop("PGEMB_SIDECAR_SHM", None)
    d = lib.hnsw_dist_func(0, a.ctypes.data_as(C.POINTER(C.c_float)), a.ctypes.data_as(C.POINTER(C.c_float)), C.c_size_t(4))
    assert np.isnan(d)


def _build_inprocess_demo(tmp_path):
    import subprocess
    from pg_embedding_b200 import build
    build.build()
    exe = str(tmp_path / "inprocess_demo")
    d = os.path.dirname(build.OUT)
    res = subprocess.run(["gcc", "-std=gnu11", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "examples", "inprocess_demo.c"),
                          "-L", d, "-lpgemb_b200", "-Wl,-rpath," + d, "-o", exe], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    return exe


def test_c_program_links_against_the_library_and_fails_loudly_without_a_device(lib, tmp_path):
    """examples/inprocess_demo.c: the reference's call sites in C with libpgemb_b200.so where the reference links
    hnswalg.o distfunc.o.  On a machine without a CUDA device it must refuse to run -- not compute on the CPU.  The demo is
    started with CUDA_VISIBLE_DEVICES empty, so it sees no device on a machine with a GPU either."""
    import subprocess
    out = subprocess.run([_build_inprocess_demo(tmp_path)], capture_output=True, text=True, timeout=120,
                         env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert out.returncode == 3 and "no CPU fallback" in out.stderr and out.stdout == ""


def test_product_kernels_are_the_measured_ones(lib):
    """The kernels of libpgemb_b200.so must be, instruction for instruction, the ones the numbers in profiles/ and DESIGN.md
    section 9 were measured with (tests/golden/product_sass.json; refresh it with tools/sass_hash.py --write together with the
    numbers when a kernel changes on purpose).  Only meaningful with the toolchain that recorded the hashes."""
    import json
    import shutil
    import subprocess
    import sys
    if not shutil.which("cuobjdump") or not shutil.which("nvcc"):
        pytest.skip("CUDA toolchain not available")
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "product_sass.json")))
    if subprocess.run(["nvcc", "--version"], capture_output=True, text=True).stdout.strip().splitlines()[-2] != gold["nvcc"]:
        pytest.skip("other nvcc than the one that recorded the hashes")
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from sass_hash import sass_hashes
    from pg_embedding_b200 import build
    got = sass_hashes(build.OUT)
    assert set(got) == set(gold["kernels"]), set(got) ^ set(gold["kernels"])
    changed = sorted(k for k in got if got[k] != gold["kernels"][k])
    assert not changed, f"kernels differ from the measured build: {changed}"

