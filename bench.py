#!/usr/bin/env python
"""bench.py -- QPS of the HNSW candidate-scoring path on B200 (BASELINE.json metric).

Workload (BASELINE.json configs[2], the configuration the metric is quoted on):
    dims=768, N=1M synthetic fp32 vectors (clustered mixture, L2-normalised), cosine `<=>`,
    hnsw(m=32, efconstruction=200, efsearch=64); a *step* = one batch of `--batch` k-NN queries
    (k = efsearch = 64) through the search path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Our arm     : the CUDA path.  `value` = queries/s with the query batch already resident in HBM
              (pgemb_search_batch_device on torch's stream, CUDA-event timed, max over ranks);
              `e2e`   = the same through the host-pointer C-ABI call pgemb_search_batch with pinned HOST
              buffers (H2D of the queries and D2H of labels+counts inside the timed region).
Reference arm (`--impl reference`): the reference's own CPU implementation (oracle/_ref = unmodified
              hnswalg.cpp + distfunc.c on a flat-memory host; falls back to the oracle port if the
              prebuilt .so is absent) on all host threads, timed on a bounded sample of the same queries
              against the SAME graph.

The graph: a sequential reference-exact build of 1M x 768 takes hours on any hardware (SURVEY.md
section 6), so both arms search the graph produced by the GPU bulk builder (pgemb_build_bulk: the
reference's search + heuristics applied in batches, DESIGN.md section 8).  The build is setup, not
timed.  Search parity on that graph is checked in-run: the CPU reference and the GPU must return
identical labels for the sampled queries (`parity` in the JSON line).

N>1 (`torchrun`): the index (3.3 GB) fits one GPU, so ranks hold replicas and split the queries
(SURVEY.md section 8(e)): no data-path collective, "scaling": "weak" (per-GPU batch fixed).

Besides the headline, the ONE JSON line carries legs for the other BASELINE configurations, each with its own in-run parity
check against the compiled reference (untimed) -- so that the driver's records hold evidence for them too:
  "configs1"   (N=1)  configs[1]: dims 128, N 100K, L2, m 16 -- a 51 MB working set that lives in L2 (bound stated as such);
  "scan_topk"  (N=1)  the brute-force operator path (SURVEY.md 8(f3) / K6): 1024 queries x the 1M x 768 table through the
                      tcgen05 tensor-core filter + exact re-scoring, TF/s against the TF32 roof, parity against the exact kernels;
  "sharded"    (N>1)  configs[3] shape: dims 1536, L2, m 32, id-range shards of PGEMB_BENCH_SHARD_ROWS (1.25M) rows per GPU
                      (10M rows at 8 GPUs), every query searched on every shard, exchange + merge INSIDE the timed region --
                      peers' lists read over NVLink by the wait+merge kernel (no collective) and, for comparison, ONE NCCL
                      all-gather + merge; parity of a 1024-query sample against "compiled reference per shard + CPU merge".
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DIMS, M, EFC, EFS = 768, 32, 200, 64
JSON_OUT = sys.stdout
METRIC = "cosine"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30, help="timed steps of the headline search (and of its e2e loop); the legs "
                    "for the other configurations use their own step counts, which each reports in its JSON")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", dest="n", type=int, default=int(os.environ.get("PGEMB_BENCH_N", 1_000_000)),
                    help="index size (default 1M = the BASELINE config; smaller values are for development only)")
    ap.add_argument("--batch", type=int, default=int(os.environ.get("PGEMB_BENCH_BATCH", 32768)), help="queries per step per GPU")
    ap.add_argument("--build-batch", type=int, default=int(os.environ.get("PGEMB_BENCH_BUILD_BATCH", 4096)))
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target CPU time of the cpu_baseline sample")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (development)")
    ap.add_argument("--no-legs", action="store_true", help="headline only: skip the configs1 / scan_topk / sharded legs (development)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned (labels, counts, counters) "
                    "as DIR/<name>.npy, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the CUDA path's results; the reference arm has none to write")
    return args


DUMP_LIMIT = 64 << 20     # bytes --dump-outputs writes at most


def dump_outputs(out_dir, labels, n, stats):
    """The last timed step's results as float64 .npy files: labels [B, k] (unused tail -1), n [B], stats [B, 4], and the
    queries they belong to (query_index [B]).  A batch too large for DUMP_LIMIT is cut to a fixed, seeded sample of queries."""
    arrays = {"labels": labels, "n": n, "stats": stats}
    B = labels.shape[0]
    per_query = 8 * (sum(a[0].size for a in arrays.values()) + 1)
    rows = np.arange(B)
    if B * per_query > DUMP_LIMIT - 4096:          # room for the four .npy headers
        rows = np.sort(np.random.default_rng(0).choice(B, (DUMP_LIMIT - 4096) // per_query, replace=False))
    arrays = {name: a[rows] for name, a in arrays.items()}
    arrays["query_index"] = rows
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a.astype(np.float64))


# ---------------------------------------------------------------------------------------------------
# synthetic data (SURVEY.md section 8(d)): mixture of ~sqrt(N) Gaussian centres, noise norm = 0.3 x the
# typical inter-centre distance, L2-normalised for cosine; fixed seeds 1234 (base) / 5678 (queries).
# ---------------------------------------------------------------------------------------------------
def gen_points(torch, n, seed, centres, chunk=1 << 16):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    dims = centres.shape[1]
    spacing = float((2.0 * dims) ** 0.5)          # E|c_i - c_j| for N(0,I) centres
    sigma = 0.3 * spacing / float(dims ** 0.5)    # per-coordinate noise
    out = torch.empty((n, dims), dtype=torch.float32, device="cuda")
    for s in range(0, n, chunk):
        e = min(n, s + chunk)
        a = torch.randint(0, centres.shape[0], (e - s,), generator=g, device="cuda")
        x = centres[a] + sigma * torch.randn((e - s, dims), generator=g, device="cuda")
        out[s:e] = x / x.norm(dim=1, keepdim=True)
    return out


def make_data(torch, n, nq):
    g = torch.Generator(device="cuda")
    g.manual_seed(99)
    centres = torch.randn((max(4, int(round(n ** 0.5))), DIMS), generator=g, device="cuda")
    return gen_points(torch, n, 1234, centres), gen_points(torch, nq, 5678, centres)


def gen_points_raw(torch, n, seed, centres, chunk=1 << 16):
    """Same mixture, NOT normalised (the L2 legs)."""
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    dims = centres.shape[1]
    sigma = 0.3 * float((2.0 * dims) ** 0.5) / float(dims ** 0.5)
    out = torch.empty((n, dims), dtype=torch.float32, device="cuda")
    for s in range(0, n, chunk):
        e = min(n, s + chunk)
        a = torch.randint(0, centres.shape[0], (e - s,), generator=g, device="cuda")
        out[s:e] = centres[a] + sigma * torch.randn((e - s, dims), generator=g, device="cuda")
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={gpu_index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def ncu_traffic_bytes(batch):
    """DRAM read+write bytes of one traversal launch from the committed ncu --set full capture (profiles/; the newest round's),
    valid for the default 32768-query launch of this workload only; (None, None) otherwise."""
    if batch != 32768:
        return None, None
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    for name in ("r2_search_kernel_cosine768_metrics.csv", "r1_search_kernel_cosine768_metrics.csv"):
        p = os.path.join(ROOT, "profiles", name)
        if not os.path.isfile(p):
            continue
        tot = 0.0
        try:
            for line in open(p):
                f = line.strip().split(",")
                if len(f) >= 4 and f[-3] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    tot += float(f[-1]) * scale.get(f[-2], 1.0)
        except Exception:
            continue
        if tot > 0:
            return int(tot), name
    return None, None


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def protect_stdout():
    """The contract is ONE JSON line on stdout.  Libraries (NCCL prints its version banner) write to fd 1 too, so fd 1 is
    pointed at stderr for the whole run and the JSON line goes to a private duplicate of the original stdout."""
    sys.stdout.flush()
    keep = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(keep, "w")


def main():
    args = parse()
    global JSON_OUT
    JSON_OUT = protect_stdout()
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference" and rank != 0:
        return 0  # the reference arm is a single-process CPU run
    if world > 1 and args.impl == "ours":
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)

    import pg_embedding_b200 as pg
    from pg_embedding_b200 import _lib
    lib = _lib.load()
    if pg.device_count() < 1:
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback)")

    n, B, K, W = args.n, args.batch, args.steps, max(args.warmup, 3 if args.impl == "ours" else 0)
    workload = f"dims={DIMS} N={n} cosine m={M} efC={EFC} efS={EFS} (BASELINE configs[2])" + ("" if n == 1_000_000 else " [REDUCED N: development run]")
    t0 = time.time()
    nq_total = B * (K + W)
    X, Q = make_data(torch, n, nq_total if args.impl == "ours" else max(B, 4096))
    torch.cuda.synchronize()
    log(f"[rank {rank}] data generated in {time.time() - t0:.1f}s")

    # ---- the device index + bulk build (setup, untimed) --------------------------------------------
    idx = pg.HnswIndex(DIMS, M, EFC, EFS, METRIC, capacity=n, device=local)
    stream = torch.cuda.current_stream().cuda_stream
    _lib.check(lib.pgemb_index_append_device(idx.dev, n, X.data_ptr(), None, None, stream))
    torch.cuda.synchronize()
    t0 = time.time()
    build_s = idx.build_appended(0, n, args.build_batch)
    log(f"[rank {rank}] bulk build of {n} nodes: {build_s:.1f}s device ({time.time() - t0:.1f}s wall)")

    ef = EFS
    if args.impl == "reference":
        return reference_arm(args, torch, pg, idx, X, Q, n, K, W)

    # ---- device-resident outputs ---------------------------------------------------------------------
    d_lab = torch.empty((B, ef), dtype=torch.int64, device="cuda")
    d_n = torch.empty((B,), dtype=torch.int32, device="cuda")
    # the traversal's own per-query counters, written by the TIMED launches themselves (16 bytes per query next to the ~3.8 MB
    # it reads): the roofline below is "algorithmic bytes of the timed launches / their device time", nothing re-run
    d_stats = torch.empty((K, B, 4), dtype=torch.int32, device="cuda")
    d_nres = torch.empty((K, B), dtype=torch.int32, device="cuda")
    d_stats_w = torch.empty((B, 4), dtype=torch.int32, device="cuda")

    def step_device(s, k_timed=None):
        q = Q[s * B:(s + 1) * B]
        st_ptr = d_stats[k_timed].data_ptr() if k_timed is not None else d_stats_w.data_ptr()
        n_ptr = d_nres[k_timed].data_ptr() if k_timed is not None else d_n.data_ptr()
        _lib.check(lib.pgemb_search_batch_device(idx.dev, B, q.data_ptr(), ef, d_lab.data_ptr(), None, None, n_ptr, st_ptr, stream))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for s in range(W):
        step_device(s)
    barrier()
    log(f"[rank {rank}] warm-up done, timing {K} steps of {B} queries")
    if os.environ.get("PGEMB_PROFILE"):   # ncu --profile-from-start off: capture exactly the timed region
        torch.cuda.profiler.start()
    launches0 = int(lib.pgemb_launch_count())
    sampler = ClockSampler(local)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for s in range(W, W + K):
        step_device(s, s - W)
    ev1.record()
    torch.cuda.synchronize()
    if os.environ.get("PGEMB_PROFILE"):
        torch.cuda.profiler.stop()
    ms = ev0.elapsed_time(ev1)
    launches = int(lib.pgemb_launch_count()) - launches0
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, d_lab.cpu().numpy(), d_nres[K - 1].cpu().numpy(), d_stats[K - 1].cpu().numpy())
    tms = torch.tensor([ms], device="cuda")
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms_max = float(tms.item())
    value = world * B * K / (ms_max * 1e-3)
    log(f"[rank {rank}] timed region: {ms_max:.1f} ms (max over ranks)")

    # ---- roofline of the dominant kernel (the traversal = gather+score; ONE launch per step, so the timed region IS K launches) ----
    st = d_stats.cpu().numpy().astype(np.int64).reshape(K * B, 4)
    nres = d_nres.cpu().numpy().astype(np.int64).reshape(K * B)
    alg_bytes = int((st[:, 0] * DIMS * 4 + st[:, 2] * 4 + nres * 8).sum()) // K       # per launch, mean over the timed launches
    kms = ms / K                                                                       # this rank's launches (CUDA events on the launching stream)
    peak, peak_src = measured_peak_gbs()
    achieved = alg_bytes / (kms * 1e-3) / 1e9
    traffic, traffic_file = ncu_traffic_bytes(B) if n == 1_000_000 else (None, None)
    roofline = {"bound": "hbm", "kernel": "search_kernel<cosine> (K3: TMA row gather + exact distance + queue update)",
                "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                "peak_source": peak_src, "traffic": traffic,
                "traffic_source": f"static: profiles/{traffic_file} (ncu --set full capture of this launch shape; not re-measured in this run)" if traffic else None,
                "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": round(kms, 3), "kernel_ms_source": "timed region / steps (one launch per step)",
                "per_query": {"dist_evals": float(st[:, 0].mean()), "expansions": float(st[:, 1].mean()),
                              "bytes": float(alg_bytes / B)}}

    # ---- e2e through the host-pointer C ABI with pinned host buffers ------------------------------------
    NB = min(K + W, 4)                                   # distinct pinned query batches, cycled
    hq = torch.empty((NB, B, DIMS), dtype=torch.float32).pin_memory()
    hq.copy_(Q[: NB * B].view(NB, B, DIMS).cpu())
    hl = torch.empty((B, ef), dtype=torch.int64).pin_memory()
    hn = torch.empty((B,), dtype=torch.int32).pin_memory()
    fp, u64p, i32p = C.POINTER(C.c_float), C.POINTER(C.c_uint64), C.POINTER(C.c_int32)

    def step_host(s):
        # the call a host application makes: host pointers in, host pointers out
        _lib.check(lib.pgemb_search_batch(idx.dev, B, C.cast(hq[s % NB].data_ptr(), fp), ef, C.cast(hl.data_ptr(), u64p), None, None,
                                          C.cast(hn.data_ptr(), i32p), None))

    for s in range(2):
        step_host(s)
    barrier()
    t0 = time.perf_counter()
    for s in range(K):
        step_host(s)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], device="cuda")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    log(f"[rank {rank}] e2e region: {float(te.item()):.3f} s")
    e2e = {"value": round(world * B * K / float(te.item()), 1), "unit": "queries/s",
           "h2d_bytes_per_step": B * DIMS * 4, "d2h_bytes_per_step": B * ef * 8 + B * 4}

    # ---- recall@10 vs exact brute force (rank 0; reported, not tuned) -----------------------------------
    out = None
    recall = cpu_baseline = parity = None
    if rank == 0:
        ns = min(1000, B)
        qs = Q[W * B: W * B + ns]
        truth = torch.topk(qs @ X.T, 10, dim=1).indices.cpu().numpy()
        step_device(W)
        torch.cuda.synchronize()
        got = d_lab[:ns, :10].cpu().numpy()
        recall = float(np.mean([len(set(truth[i].tolist()) & set(got[i].tolist())) / 10.0 for i in range(ns)]))
        if not args.no_cpu and world == 1:
            cpu_baseline, parity = cpu_leg(args, idx, Q[W * B:(W + 1) * B], d_lab.cpu().numpy(), d_n.cpu().numpy(), n)

    # ---- the other BASELINE configurations (legs; each frees what it allocates) --------------------------
    legs = {}
    if not args.no_legs:
        if world == 1:
            try:
                legs["scan_topk"] = leg_scan_topk(args, torch, lib, _lib, idx, X, Q, n)
            except Exception as e:                                   # a leg must never take the headline down with it
                legs["scan_topk"] = {"error": repr(e)[:300]}
        del X, Q, d_stats, d_nres, hq
        idx.close()
        torch.cuda.empty_cache()
        if world == 1:
            try:
                legs["configs1"] = leg_configs1(args, torch, pg, lib, _lib, local)
            except Exception as e:
                legs["configs1"] = {"error": repr(e)[:300]}
        else:
            try:
                legs["sharded"] = leg_sharded(args, torch, dist, pg, lib, _lib, rank, world, local)
            except Exception as e:
                legs["sharded"] = {"error": repr(e)[:300]}
                log(f"[rank {rank}] sharded leg failed: {e!r}")
        if world > 1 or os.environ.get("PGEMB_BENCH_C4", "1") != "0":
            try:
                legs["configs4"] = leg_configs4(args, torch, dist, pg, lib, _lib, rank, world, local)
            except Exception as e:
                legs["configs4"] = {"error": repr(e)[:300]}
                log(f"[rank {rank}] configs4 leg failed: {e!r}")
    if rank == 0:
        out = {
            "metric": "QPS @ recall@10, dims=768 N=1M efSearch=64", "value": round(value, 1), "unit": "queries/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": round(ms_max / K, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload, "queries_per_step": B, "queries_per_step_per_gpu": B, "k": ef, "parallelism": f"replicas x{world}, queries split",
                       "l2": "inputs larger than L2 (3.3 GB index vs 126 MB L2); distinct queries every step",
                       "graph": f"GPU bulk build (batch<={args.build_batch}), {build_s:.1f}s, shared by both arms",
                       "distribution": "mixture of sqrt(N) Gaussians, noise 0.3x inter-centre spacing, L2-normalised; seeds 1234/5678"},
            "recall_at_10": round(recall, 4),
            "e2e": e2e, "gpu_launches": launches, "clocks": clocks, "roofline": roofline,
            "cpu_baseline": cpu_baseline, "parity": parity,
        }
        out.update(legs)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if out is not None:
        JSON_OUT.write(json.dumps(out) + "\n")
        JSON_OUT.flush()
    return 0


# ---------------------------------------------------------------------------------------------------------------------
# leg: the brute-force operator path (K6) on the headline table
# ---------------------------------------------------------------------------------------------------------------------
def scan_counters(lib):
    out = (C.c_uint64 * 6)()
    lib.pgemb_scan_counters(out)
    return dict(tc=out[0], pairs=out[1], rescored=out[2], fallbacks=out[3], overflow=out[4], exact=out[5])


def leg_scan_topk(args, torch, lib, _lib, idx, X, Q, n):
    nq, k = int(os.environ.get("PGEMB_BENCH_SCAN_QUERIES", 1024)), 64
    q = Q[:nq].cpu().numpy()
    fp, u64p, i32p = C.POINTER(C.c_float), C.POINTER(C.c_uint64), C.POINTER(C.c_int32)
    lab = np.empty((nq, k), np.uint64); dd = np.empty((nq, k), np.float32); nn = np.zeros(nq, np.int32)

    def run(qq, L, D, Nn):
        _lib.check(lib.pgemb_scan_topk(idx.dev, qq.shape[0], qq.ctypes.data_as(fp), k, L.ctypes.data_as(u64p), D.ctypes.data_as(fp), Nn.ctypes.data_as(i32p)))

    os.environ.pop("PGEMB_SCAN_TC", None)
    run(q, lab, dd, nn)                                            # warm-up: staging buffers, norms
    c0 = scan_counters(lib)
    reps, times = 3, []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        run(q, lab, dd, nn)                                        # host pointers in / out: H2D of the queries and D2H of the results inside
        times.append(time.perf_counter() - t0)
    c1 = scan_counters(lib)
    t = sorted(times)[len(times) // 2]
    # parity: the exact kernels (no filter) on a sample of the same queries -- labels, order and distance bits
    ns = min(32, nq)
    os.environ["PGEMB_SCAN_TC"] = "0"
    l2 = np.empty((ns, k), np.uint64); d2 = np.empty((ns, k), np.float32); n2 = np.zeros(ns, np.int32)
    t0 = time.perf_counter()
    run(q[:ns], l2, d2, n2)
    t_exact = time.perf_counter() - t0
    os.environ.pop("PGEMB_SCAN_TC", None)
    same = bool(lab[:ns].tobytes() == l2.tobytes() and dd[:ns].tobytes() == d2.tobytes() and nn[:ns].tolist() == n2.tolist())
    flops = 2.0 * nq * n * DIMS
    try:
        bf16 = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops"])
    except Exception:
        bf16 = 1590.0
    peak_tf32 = bf16 / 2.0
    hbm, _ = measured_peak_gbs()
    table_bytes = n * DIMS * 4
    qtiles = (nq + 127) // 128
    return {"workload": f"pgemb_scan_topk: {nq} queries x {n} rows x {DIMS} dims, cosine, k={k} (exact brute-force k-NN, SURVEY.md 8(f3))",
            "seconds": round(t, 5), "pairs_per_s": round(nq * n / t, 0), "queries_per_s": round(nq / t, 1),
            "tensor": {"bound": "tensor", "achieved": round(flops / t / 1e12, 1), "peak": round(peak_tf32, 1), "unit": "TFLOP/s",
                       "frac": round(flops / t / 1e12 / peak_tf32, 4), "peak_source": "MEASURED_PEAKS.json bf16_tflops / 2 (TF32 runs at half the bf16 rate)"},
            "hbm_bound_one_table_pass_per_query_tile_s": round(qtiles * table_bytes / (hbm * 1e9), 5),
            "x_of_that_bound": round(t / (qtiles * table_bytes / (hbm * 1e9)), 2),
            "rescored_fraction": round((c1["rescored"] - c0["rescored"]) / max(1, c1["pairs"] - c0["pairs"]), 6),
            "tripwire_fallbacks": int(c1["fallbacks"] - c0["fallbacks"]), "overflowed_queries": int(c1["overflow"] - c0["overflow"]),
            "through_tensor_path": bool(c1["tc"] - c0["tc"] == reps),
            "exact_kernels_same_sample": {"queries": ns, "seconds": round(t_exact, 4), "pairs_per_s": round(ns * n / t_exact, 0)},
            "parity": {"queries": ns, "identical_to_exact_kernels_labels_order_bits": same},
            "timing": "host wall clock around the C-ABI call (host buffers), median of 3"}


# ---------------------------------------------------------------------------------------------------------------------
# leg: BASELINE configs[1] (dims 128, N 100K, L2, m 16) on one GPU
# ---------------------------------------------------------------------------------------------------------------------
def leg_configs1(args, torch, pg, lib, _lib, local):
    dims, n, m, efc, efs, B, K, W = 128, 100_000, 16, 200, 64, 32768, 10, 3
    g = torch.Generator(device="cuda"); g.manual_seed(99)
    centres = torch.randn((max(4, int(round(n ** 0.5))), dims), generator=g, device="cuda")
    X, Q = gen_points_raw(torch, n, 1234, centres), gen_points_raw(torch, B * (K + W), 5678, centres)
    idx = pg.HnswIndex(dims, m, efc, efs, "l2", capacity=n, device=local)
    stream = torch.cuda.current_stream().cuda_stream
    _lib.check(lib.pgemb_index_append_device(idx.dev, n, X.data_ptr(), None, None, stream)); torch.cuda.synchronize()
    build_s = idx.build_appended(0, n, 4096)
    d_lab = torch.empty((B, efs), dtype=torch.int64, device="cuda"); d_n = torch.empty((K, B), dtype=torch.int32, device="cuda")
    d_st = torch.empty((K, B, 4), dtype=torch.int32, device="cuda")

    def step(s, kt):
        _lib.check(lib.pgemb_search_batch_device(idx.dev, B, Q[s * B:(s + 1) * B].data_ptr(), efs, d_lab.data_ptr(), None, None, d_n[kt].data_ptr(),
                                                  d_st[kt].data_ptr(), stream))
    for s in range(W):
        step(s, 0)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(W, W + K):
        step(s, s - W)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / K
    st = d_st.cpu().numpy().astype(np.int64).reshape(K * B, 4); nres = d_n.cpu().numpy().astype(np.int64).reshape(K * B)
    alg = int((st[:, 0] * dims * 4 + st[:, 2] * 4 + nres * 8).sum()) // K
    hbm, _ = measured_peak_gbs()
    # parity: the compiled reference on the same graph, the whole last batch (100K x 128 is small enough for the CPU)
    par, cpu = None, None
    if not args.no_cpu:
        from oracle import oracle
        which, kind = pick_checker()
        orc = oracle.FlatIndex(which, dims, m, efc, efs, "l2", capacity=n)
        orc.load_records(idx.export_records(0, n))
        qh = Q[(W + K - 1) * B:(W + K) * B].cpu().numpy()
        cores = os.cpu_count() or 1
        ns = 8192
        ref = orc.search_many(qh[:ns], efs, nthreads=cores)
        step(W + K - 1, 0); torch.cuda.synchronize()
        got = d_lab.cpu().numpy()[:ns].view(np.uint64)
        par = {"queries": ns, "labels_identical_to_cpu_reference": bool((ref["labels"] == got).all() and (ref["n"] == d_n[0].cpu().numpy()[:ns]).all())}
        cpu = {"value": round(ns / ref["seconds"], 1), "unit": "queries/s", "cores": cores, "kind": kind, "sample": f"{ns} queries, one pass, same graph"}
        orc.close()
    truth = torch.cat([torch.topk(torch.cdist(Q[W * B + i: W * B + i + 250], X), 10, dim=1, largest=False).indices for i in range(0, 1000, 250)]).cpu().numpy()
    step(W, 0); torch.cuda.synchronize()
    got10 = d_lab[:1000, :10].cpu().numpy()
    recall = float(np.mean([len(set(truth[i].tolist()) & set(got10[i].tolist())) / 10.0 for i in range(1000)]))
    idx.close()
    return {"workload": f"dims={dims} N={n} L2 m={m} efC={efc} efS={efs} (BASELINE configs[1]), {B} queries per step, bulk build {build_s:.1f}s",
            "value": round(B / (ms * 1e-3), 1), "unit": "queries/s", "ms_per_step": round(ms, 3), "steps": K, "warmup": W, "recall_at_10": round(recall, 4),
            "roofline": {"bound": "instruction issue / hop latency (working set L2-resident)", "achieved": round(alg / (ms * 1e-3) / 1e9, 1), "unit": "GB/s", "algorithmic_bytes_per_launch": alg,
                         "hbm_peak": hbm, "frac_of_hbm_peak": round(alg / (ms * 1e-3) / 1e9 / hbm, 4),
                         "note": "working set 51 MB vectors + 13 MB links < 126 MB L2: the HBM roof is NOT the binding one here (ncu: DRAM 12 % of peak). "
                                 "The kernel is bound by instruction issue and the dependent hop chain: 64 % of the issue slots busy with 30 warps per SM, "
                                 "about 1400 warp instructions of queue / visited / prefetch bookkeeping per hop around 7.5 rows x 512 B of scoring "
                                 "(profiles/r2_configs1_metrics.csv, profiles/README.md)",
                         "per_query": {"dist_evals": float(st[:, 0].mean()), "expansions": float(st[:, 1].mean())}},
            "cpu_baseline": cpu, "parity": par}


# ---------------------------------------------------------------------------------------------------------------------
# leg: BASELINE configs[3] shape, id-range shards across the ranks (N > 1)
# ---------------------------------------------------------------------------------------------------------------------
def leg_sharded(args, torch, dist, pg, lib, _lib, rank, world, local):
    from pg_embedding_b200 import sharded
    dims, m, efc, efs = 1536, 32, 200, 64
    rows = int(os.environ.get("PGEMB_BENCH_SHARD_ROWS", 1_250_000))
    B = int(os.environ.get("PGEMB_BENCH_SHARD_BATCH", 16384))
    K, W = min(args.steps, 10), 2
    n_total = rows * world
    lo, hi = sharded.shard_bounds(n_total, world)[rank]
    g = torch.Generator(device="cuda"); g.manual_seed(99)
    centres = torch.randn((max(4, int(round(n_total ** 0.5))), dims), generator=g, device="cuda")
    X = gen_points_raw(torch, hi - lo, 1234 + rank, centres)           # this rank's id range
    Q = gen_points_raw(torch, B * (K + W), 5678, centres)              # the same queries on every rank
    idx = pg.HnswIndex(dims, m, efc, efs, "l2", capacity=hi - lo, device=local)
    labels = torch.arange(lo, hi, dtype=torch.int64, device="cuda")   # labels = global ids
    stream = torch.cuda.current_stream().cuda_stream
    _lib.check(lib.pgemb_index_append_device(idx.dev, hi - lo, X.data_ptr(), labels.data_ptr(), None, stream)); torch.cuda.synchronize()
    build_s = idx.build_appended(0, hi - lo, 4096)
    log(f"[rank {rank}] sharded leg: shard [{lo},{hi}) built in {build_s:.1f}s")
    peer = sharded.PeerExchange(idx, B, efs)
    nccl = sharded.ShardedSearch(sharded.gpu_local_search_packed(idx), sharded.gpu_merge_packed())

    def timed(run):
        for s in range(W):
            run(Q[s * B:(s + 1) * B])
        dist.barrier(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = int(lib.pgemb_launch_count())
        e0.record()
        for s in range(W, W + K):
            out = run(Q[s * B:(s + 1) * B])
        e1.record(); torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / K, out, (int(lib.pgemb_launch_count()) - l0) / K

    ms_peer, out_peer, launches_peer = timed(lambda q: peer.search(q, efs))
    merge_ms = peer.merge_ms()
    c0 = nccl.collectives
    ms_nccl, out_nccl, launches_nccl = timed(lambda q: nccl.search(q, efs))
    coll_per_step = (nccl.collectives - c0) / (K + W)
    same_exchanges = bool(torch.equal(out_peer[1], out_nccl[1]) and torch.equal(out_peer[0], out_nccl[0]) and torch.equal(out_peer[2], out_nccl[2]))
    # ---- parity of a query sample: compiled reference per shard + (dist,label) merge on the CPU (SURVEY.md 8(e)) ----
    parity = parity_ok = None
    if not args.no_cpu:
        ns = 1024
        qs = Q[(W + K - 1) * B:(W + K - 1) * B + ns]
        from oracle import oracle
        which, kind = pick_checker()
        orc = oracle.FlatIndex(which, dims, m, efc, efs, "l2", capacity=hi - lo)
        chunk = 1 << 15
        for s0 in range(0, hi - lo, chunk):
            orc.load_records(idx.export_records(s0, min(chunk, hi - lo - s0)))
        qh = qs.cpu().numpy()
        ref = orc.search_many(qh, efs, nthreads=max(1, (os.cpu_count() or 1) // world))
        orc.close()
        lab = torch.from_numpy(ref["labels"].view(np.int64).copy()).cuda()
        cnt = torch.from_numpy(ref["n"].astype(np.int32)).cuda()
        # the reference returns no distances: score its labels with its own distance function (rows fetched from this shard)
        dd = np.full((ns, efs), np.inf, np.float32)
        for i in range(ns):
            c = int(ref["n"][i])
            if c:
                rowsel = X[(lab[i, :c] - lo)].cpu().numpy()
                dd[i, :c] = oracle.dist_many(which, "l2", qh[i], rowsel)
        dref = torch.from_numpy(dd).cuda()
        gl = [torch.empty_like(lab) for _ in range(world)]; gd = [torch.empty_like(dref) for _ in range(world)]; gn = [torch.empty_like(cnt) for _ in range(world)]
        dist.all_gather(gl, lab); dist.all_gather(gd, dref); dist.all_gather(gn, cnt)      # parity plumbing, untimed
        if rank == 0:
            L = torch.stack(gl).cpu().numpy(); D = torch.stack(gd).cpu().numpy(); Nn = torch.stack(gn).cpu().numpy()
            gpu_l = out_peer[1][:ns].cpu().numpy(); gpu_d = out_peer[0][:ns].cpu().numpy(); gpu_n = out_peer[2][:ns].cpu().numpy()
            ok = True
            for i in range(ns):
                pairs = sorted((float(D[s, i, j]), int(L[s, i, j])) for s in range(world) for j in range(int(Nn[s, i])))[:efs]
                if gpu_n[i] != len(pairs) or gpu_l[i, :len(pairs)].tolist() != [p_[1] for p_ in pairs] or \
                        gpu_d[i, :len(pairs)].tobytes() != np.array([p_[0] for p_ in pairs], np.float32).tobytes():
                    ok = False
                    break
            parity = {"queries": ns, "identical_to_reference_per_shard_plus_cpu_merge": ok, "checker": kind}
            parity_ok = ok
    err = peer.error()
    peer.close()
    idx.close()
    del X, Q
    torch.cuda.empty_cache()
    bytes_rank = sharded.packed_bytes(B, efs)
    return {"workload": f"dims={dims} N={n_total} ({rows} per shard) L2 m={m} efC={efc} efS={efs} (BASELINE configs[3] shape), index sharded by id range over {world} GPUs, "
                        f"{B} queries per step searched on EVERY shard, bulk build {build_s:.1f}s per shard",
            "value": round(B / (ms_peer * 1e-3), 1), "unit": "queries/s", "ms_per_step": round(ms_peer, 3), "steps": K, "warmup": W, "scaling": "weak (shard size fixed, index grows with N)",
            "exchange": "peer memory: per-shard top-k read over NVLink by the wait+merge kernel (CUDA IPC), flags published by 4-byte copies; no collective",
            "launches_per_step": launches_peer, "collectives_per_step": 0, "merge_kernel_ms_incl_peer_wait": round(merge_ms, 3),
            "exchange_bytes_read_per_rank_per_step": bytes_rank * (world - 1), "peer_error": err,
            "nccl_allgather": {"value": round(B / (ms_nccl * 1e-3), 1), "ms_per_step": round(ms_nccl, 3), "collectives_per_step": coll_per_step,
                               "launches_per_step": launches_nccl, "bytes_per_rank": bytes_rank, "same_results_as_peer_exchange": same_exchanges},
            "parity": parity_ok, "parity_detail": parity}


# ---------------------------------------------------------------------------------------------------------------------
# leg: BASELINE configs[4] shape -- dims 768, cosine, 1024-query batches against a table sharded by id range, every rank scans
# its rows on the tensor-core path (K6), per-shard top-k exchanged and merged (K5).  12.5M rows per GPU: 100M at 8 GPUs.
# ---------------------------------------------------------------------------------------------------------------------
def leg_configs4(args, torch, dist, pg, lib, _lib, rank, world, local):
    from pg_embedding_b200 import sharded
    dims, k, nq = 768, 10, 1024
    rows = int(os.environ.get("PGEMB_BENCH_C4_ROWS", 12_500_000))
    K, W = min(args.steps, 5), 2
    n_total = rows * world
    lo, hi = sharded.shard_bounds(n_total, world)[rank]
    g = torch.Generator(device="cuda"); g.manual_seed(99)
    centres = torch.randn((max(4, int(round(n_total ** 0.5))), dims), generator=g, device="cuda")
    idx = pg.HnswIndex(dims, 2, 4, 16, "cosine", capacity=hi - lo, device=local)   # no graph is built: the operator path scans the table
    stream = torch.cuda.current_stream().cuda_stream
    t0 = time.time()
    chunk = 1 << 20
    for s0 in range(lo, hi, chunk):                                                 # generated and appended chunk by chunk (38 GB per shard)
        e = min(hi, s0 + chunk)
        x = gen_points(torch, e - s0, 1234 + 7919 * (s0 // chunk), centres)
        labels = torch.arange(s0, e, dtype=torch.int64, device="cuda")              # labels = global ids
        _lib.check(lib.pgemb_index_append_device(idx.dev, e - s0, x.data_ptr(), labels.data_ptr(), None, stream)); torch.cuda.synchronize()
        del x, labels
    Q = gen_points(torch, nq * (K + W), 5678, centres)                              # the same queries on every rank
    log(f"[rank {rank}] configs4 leg: shard [{lo},{hi}) generated in {time.time() - t0:.1f}s")
    os.environ.pop("PGEMB_SCAN_TC", None)
    peer = nccl = None
    if world > 1:
        peer = sharded.PeerExchange(idx, nq, k)
        nccl = sharded.ShardedSearch(sharded.gpu_local_scan_packed(idx), sharded.gpu_merge_packed())

    def scan_local(q):
        od = torch.empty((q.shape[0], k), dtype=torch.float32, device="cuda"); ol = torch.empty((q.shape[0], k), dtype=torch.int64, device="cuda")
        on = torch.empty((q.shape[0],), dtype=torch.int32, device="cuda")
        _lib.check(lib.pgemb_scan_topk_device(idx.dev, q.shape[0], q.data_ptr(), k, ol.data_ptr(), od.data_ptr(), on.data_ptr(), stream))
        return od, ol, on

    def timed(run):
        for s in range(W):
            run(Q[s * nq:(s + 1) * nq])
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = int(lib.pgemb_launch_count())
        e0.record()
        for s in range(W, W + K):
            out = run(Q[s * nq:(s + 1) * nq])
        e1.record(); torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / K, out, (int(lib.pgemb_launch_count()) - l0) / K

    c0 = scan_counters(lib)
    ms, out, launches = timed((lambda q: peer.scan(q, k)) if world > 1 else scan_local)
    c1 = scan_counters(lib)
    nccl_part = None
    if world > 1:
        ms_n, out_n, launches_n = timed(lambda q: nccl.search(q, k))
        nccl_part = {"value": round(nq / (ms_n * 1e-3), 1), "ms_per_step": round(ms_n, 3), "collectives_per_step": 1, "launches_per_step": launches_n,
                     "bytes_per_rank": sharded.packed_bytes(nq, k),
                     "same_results_as_peer_exchange": bool(torch.equal(out[1], out_n[1]) and torch.equal(out[0], out_n[0]) and torch.equal(out[2], out_n[2]))}
    # ---- parity of a query sample: the exact kernels (no filter; themselves pinned to the oracle by the tests) per shard,
    #      merged on the CPU by (dist,label)
    ns = 16
    qs = Q[(W + K - 1) * nq:(W + K - 1) * nq + ns].contiguous()
    os.environ["PGEMB_SCAN_TC"] = "0"
    t0 = time.perf_counter()
    ed, el, en = scan_local(qs)
    torch.cuda.synchronize()
    t_exact = time.perf_counter() - t0
    os.environ.pop("PGEMB_SCAN_TC", None)
    if world > 1:
        gl = [torch.empty_like(el) for _ in range(world)]; gd = [torch.empty_like(ed) for _ in range(world)]; gn = [torch.empty_like(en) for _ in range(world)]
        dist.all_gather(gl, el); dist.all_gather(gd, ed); dist.all_gather(gn, en)      # parity plumbing, untimed
    else:
        gl, gd, gn = [el], [ed], [en]
    parity_ok = None
    if rank == 0:
        L = torch.stack(gl).cpu().numpy(); D = torch.stack(gd).cpu().numpy(); Nn = torch.stack(gn).cpu().numpy()
        gpu_l = out[1][:ns].cpu().numpy(); gpu_d = out[0][:ns].cpu().numpy(); gpu_n = out[2][:ns].cpu().numpy()
        parity_ok = True
        for i in range(ns):
            pairs = sorted((float(D[s, i, j]), int(L[s, i, j])) for s in range(world) for j in range(int(Nn[s, i])))[:k]
            if gpu_n[i] != len(pairs) or gpu_l[i, :len(pairs)].tolist() != [p_[1] for p_ in pairs] or \
                    gpu_d[i, :len(pairs)].tobytes() != np.array([p_[0] for p_ in pairs], np.float32).tobytes():
                parity_ok = False
                break
    err = peer.error() if peer else 0
    merge_ms = peer.merge_ms() if peer else 0.0
    if peer:
        peer.close()
    idx.close()
    del Q
    torch.cuda.empty_cache()
    try:
        bf16 = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops"])
    except Exception:
        bf16 = 1590.0
    hbm, _ = measured_peak_gbs()
    t = ms * 1e-3
    flops_gpu = 2.0 * nq * rows * dims
    qtiles = (nq + 127) // 128
    return {"workload": f"dims={dims} N={n_total} ({rows} rows per shard) cosine, {nq}-query batches, k={k} (BASELINE configs[4] shape: {world} of its 8 shards), "
                        f"every rank scans its id range on the tensor-core path (K6), per-shard top-k exchanged and merged (K5); no graph",
            "value": round(nq / t, 1), "unit": "queries/s", "ms_per_step": round(ms, 3), "steps": K, "warmup": W, "scaling": "weak (shard size fixed, table grows with N)",
            "pairs_per_s": round(nq * n_total / t, 0),
            "tensor": {"bound": "tensor", "achieved_per_gpu": round(flops_gpu / t / 1e12, 1), "peak": round(bf16 / 2.0, 1), "unit": "TFLOP/s",
                       "frac": round(flops_gpu / t / 1e12 / (bf16 / 2.0), 4), "peak_source": "MEASURED_PEAKS.json bf16_tflops / 2 (TF32 runs at half the bf16 rate)"},
            "hbm_bound_one_table_pass_per_query_tile_s": round(qtiles * rows * dims * 4 / (hbm * 1e9), 5),
            "x_of_that_bound": round(t / (qtiles * rows * dims * 4 / (hbm * 1e9)), 2),
            "rescored_fraction": round((c1["rescored"] - c0["rescored"]) / max(1, c1["pairs"] - c0["pairs"]), 8),
            "tripwire_fallbacks": int(c1["fallbacks"] - c0["fallbacks"]), "overflowed_queries": int(c1["overflow"] - c0["overflow"]),
            "through_tensor_path": bool(c1["tc"] - c0["tc"] == K + W),
            "exchange": ("peer memory: per-shard top-k read over NVLink by the wait+merge kernel (CUDA IPC); no collective" if world > 1 else "none (one shard)"),
            "launches_per_step": launches, "collectives_per_step": 0, "merge_kernel_ms_incl_peer_wait": round(merge_ms, 3),
            "exchange_bytes_read_per_rank_per_step": sharded.packed_bytes(nq, k) * (world - 1), "peer_error": err,
            "nccl_allgather": nccl_part,
            "exact_kernels_same_sample": {"queries": ns, "seconds": round(t_exact, 4), "pairs_per_s": round(ns * rows / t_exact, 0)},
            "parity": parity_ok, "parity_detail": {"queries": ns, "identical_to_exact_kernels_per_shard_plus_cpu_merge_labels_order_bits": parity_ok}}


def host_graph(idx, n, which):
    """Copy the GPU index (reference record layout) into the CPU checker's flat host."""
    from oracle import oracle
    orc = oracle.FlatIndex(which, DIMS, M, EFC, EFS, METRIC, capacity=n)
    chunk = 1 << 16
    for s in range(0, n, chunk):
        orc.load_records(idx.export_records(s, min(chunk, n - s)))
    return orc


def pick_checker():
    from oracle import oracle
    if oracle.available("ref"):
        return "ref", "reference"
    oracle.build("port")
    return "port", "port"


def cpu_leg(args, idx, q_dev, gpu_labels, gpu_n, n):
    which, kind = pick_checker()
    orc = host_graph(idx, n, which)
    cores = os.cpu_count() or 1
    q = q_dev.cpu().numpy()
    cal = orc.search_many(q[:cores * 2], EFS, nthreads=cores, want_labels=False)
    qps_est = max(1.0, cores * 2 / max(cal["seconds"], 1e-6))
    reps = 3                                                          # SURVEY.md 8(d): warm cache, >= 3 repetitions, median
    ns = int(min(q.shape[0], max(cores * 4, qps_est * args.cpu_seconds / reps)))
    # untimed pass over the WHOLE step: warms the 3.3 GB graph (page faults, caches) and is the parity check
    full = orc.search_many(q, EFS, nthreads=cores)
    same = bool((full["labels"] == gpu_labels[:q.shape[0]].view(np.uint64)).all() and (full["n"] == gpu_n[:q.shape[0]]).all())
    secs = sorted(orc.search_many(q[:ns], EFS, nthreads=cores, want_labels=False)["seconds"] for _ in range(reps))
    med = secs[len(secs) // 2]
    base = {"value": round(ns / med, 1), "unit": "queries/s", "cores": cores, "kind": kind,
            "sample": f"{ns} of the step's queries, one reader thread per host core, median of {reps} warm passes "
                      f"({secs[0]:.1f}/{med:.1f}/{secs[-1]:.1f}s), same graph"}
    par = {"queries": int(q.shape[0]), "labels_identical_to_cpu_reference": same}
    orc.close()
    return base, par


def reference_arm(args, torch, pg, idx, X, Q, n, K, W):
    which, kind = pick_checker()
    orc = host_graph(idx, n, which)
    cores = os.cpu_count() or 1
    q = Q.cpu().numpy()
    cal = orc.search_many(q[:cores * 2], EFS, nthreads=cores, want_labels=False)
    qps_est = max(1.0, cores * 2 / max(cal["seconds"], 1e-6))
    per_step = int(min(q.shape[0], max(cores * 2, qps_est * max(2.0, 60.0 / max(1, K + W)))))
    for s in range(W):
        orc.search_many(q[:per_step], EFS, nthreads=cores, want_labels=False)
    t = 0.0
    for s in range(K):
        off = (s * per_step) % max(1, q.shape[0] - per_step + 1)
        t += orc.search_many(q[off:off + per_step], EFS, nthreads=cores, want_labels=False)["seconds"]
    v = round(per_step * K / t, 1)
    sample = f"{per_step} queries per step, one reader thread per host core ({cores}), same GPU-built graph"
    out = {"impl": "reference", "metric": "QPS @ recall@10, dims=768 N=1M efSearch=64", "value": v, "unit": "queries/s",
           "n_gpus": args.gpus, "steps": K, "warmup": W, "ms_per_step": round(1e3 * t / K, 3), "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": f"dims={DIMS} N={n} cosine m={M} efC={EFC} efS={EFS} (BASELINE configs[2])", "k": EFS,
                      "queries_per_step": per_step, "graph": "GPU bulk build, shared by both arms"},
           "cpu_baseline": {"value": v, "unit": "queries/s", "cores": cores, "kind": kind, "sample": sample},
           "e2e": {"value": v, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    JSON_OUT.write(json.dumps(out) + "\n")
    JSON_OUT.flush()
    return 0


if __name__ == "__main__":
    sys.exit(main())
