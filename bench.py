#!/usr/bin/env python
"""Benchmark of the recommendation scoring hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--rows R] [--dump-outputs DIR]

Workload (BASELINE.json `metric`): single-query cosine top-10 with a 133-row seen-movie exclusion over a
10M x 1536 bf16 synthetic catalog.  One step = one query through the whole hot path.
  N = 1 : the whole catalog on one B200 (30.7 GB).
  N > 1 : the same 10M catalog row-sharded over N ranks (strong scaling); local fast + exact pass, NVLink exchange + merge
          inside the same kernel launch.
`value`  : queries/s with the query already resident in HBM (ONE kernel launch per query).
`e2e`    : queries/s through CatalogStore.recommend / ShardedCatalog.recommend with HOST buffers in and out (the request is
           read from pinned memory by the first kernel, the result written there by the last, stream sync) inside the timed region.
`result_digest` : sha1 over the k returned row ids and fp64 score bits of the fixed workload (catalog seed 0, query seed 1,
           exclusion seed 1).  It must be the SAME at every N — one global order, lib.py:55,63 — and is asserted against
           tests/golden/bench_digests.json; an independent dense-score kernel + host fp64 re-score checks it in every run.
`configs`: every BASELINE.json config measured in this run (C1 CPU-sized catalog with the reference's CPU path beside it,
           C2 1M fp32 / bf16, C3 4096 x 1M batched top-100, C4 = the headline + the batched 10M leg, C5 CSR profiles +
           genre/year-filtered top-50 at N > 1), plus a profile request (85 liked + 133 rated rows, the reference's real
           route, lib.py:43-55) and the int8-prefilter variant of the headline.  Secondary: never instead of the headline.
`--impl reference` times the reference's own CPU path (oracle/, pandas + scikit-learn, float64, all host threads) on
a bounded row sample of the same workload and scales to the full catalog.
`--dump-outputs DIR` writes what the last timed step returned as float64 .npy files, so that two builds can be compared
           output for output on the same seeded inputs: rows.npy / scores.npy of the device-resident step (`value`) and
           e2e_rows.npy / e2e_scores.npy of the host-buffer request (`e2e`); row ids are exact in float64.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

N_ROWS, DIM, DTYPE, K, N_EXCL = 10_000_000, 1536, "bf16", 10, 133
METRIC = "queries/s top-k cosine retrieval (10M x 1536 bf16)"
DIGESTS = os.path.join(REPO, "tests", "golden", "bench_digests.json")


def workload_name(rows):
    return f"single-query cosine top-{K} + {N_EXCL}-row exclusion over {rows} x {DIM} {DTYPE} synthetic catalog"


def digest(rows, scores=None):
    h = hashlib.sha1(np.ascontiguousarray(rows, dtype=np.int64).tobytes())
    if scores is not None:
        h.update(np.ascontiguousarray(scores, dtype=np.float64).tobytes())
    return h.hexdigest()[:16]


def expected_digest(key):
    try:
        return json.load(open(DIGESTS)).get(key)
    except Exception:
        return None


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def __exit__(self, *a):
        if self.proc is not None:
            time.sleep(0.25)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()
            self.t.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0]))
                mx.append(float(p[1]))
            except ValueError:
                continue
            for nm, v in zip(names, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    out = {"hbm": 6650.0, "hbm_src": "fallback (B200_PROFILING.md)", "bf16": 1590.0, "bf16_sustained": None}
    if os.path.exists(path):
        try:
            mp = json.load(open(path))
            out.update(hbm=float(mp["hbm_gbs"]), hbm_src="measured (MEASURED_PEAKS.json hbm_gbs)", bf16=float(mp["bf16_tflops"]),
                       bf16_sustained=float(mp.get("bf16_tflops_sustained") or 0) or None)
        except Exception:
            pass
    return out


def ncu_traffic(key):
    """dram bytes of one launch from the committed ncu capture (profiles/roofline_traffic.json) — NOT measured in this run."""
    path = os.path.join(REPO, "profiles", "roofline_traffic.json")
    try:
        return json.load(open(path)).get(key)
    except Exception:
        return None


def cpu_model():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


# ------------------------------------------------------------------------------------------------ CPU legs (oracle/)
def cpu_reference_leg(rows_full: int, steps: int, warmup: int, sample_rows: int, budget_s: float = 60.0):
    """The reference's own CPU path (restated lib.py:51-55, L=1) on a bounded row sample; returns (q/s scaled to
    rows_full, description, seconds per sample query, cores).  The sample is sized from a short calibration so that
    the whole (warmup + steps) run stays near `budget_s` seconds whatever K the caller asks for."""
    from oracle import reference_scoring as ora
    from robot_ebert_b200 import synth

    def build(nrows):
        m = np.empty((nrows, DIM), dtype=np.float64)
        for s in range(0, nrows, 8192):
            e = min(nrows, s + 8192)
            m[s:e] = synth.quantise(synth.catalog_rows_f32(0, s, e - s, DIM), DTYPE)
        emb = ora.catalog_frame(synth.row_ids(nrows), m)               # float64 frame, string index (constants.py:56)
        excl_rows = np.random.default_rng(1).choice(nrows, size=min(N_EXCL, nrows // 2), replace=False)
        return emb, [emb.index[r] for r in excl_rows]

    q = synth.query_f32(1, DIM).astype(np.float64)
    cal_rows = min(8192, rows_full)
    emb, excl_ids = build(cal_rows)
    ora.single_query(emb, q, excl_ids, K)
    t0 = time.perf_counter()
    ora.single_query(emb, q, excl_ids, K)
    per_row = (time.perf_counter() - t0) / cal_rows
    fit = int(budget_s / max(1, steps + warmup) / per_row)
    sample_rows = int(max(4096, min(sample_rows, rows_full, fit)))
    emb, excl_ids = build(sample_rows)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        ora.single_query(emb, q, excl_ids, K)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    t = sum(times) / len(times)
    qps = 1.0 / (t * rows_full / sample_rows)
    desc = (f"{len(times)} queries over the first {sample_rows} of {rows_full} rows x {DIM} (float64 DataFrame, pandas + "
            f"sklearn cosine_similarity + sort, as lib.py:51-55); per-query time scaled by {rows_full / sample_rows:.0f}x")
    return qps, desc, t, os.cpu_count()


def config_c1(dev):
    """BASELINE config 1, MEASURED (not scaled): 10k x 1536 fp32 catalog, (i) the reference's user-recs request
    (lib.py:42-55, ~85 liked of ~133 rated) and (ii) a single query, on the host cores with pandas + sklearn in float64,
    and the GPU path end to end on the very same inputs with the parity assertion."""
    import pandas as pd
    from oracle import reference_scoring as ora
    from robot_ebert_b200 import CatalogStore, synth
    n, d, k = 10_000, 1536, 10
    m32 = synth.catalog_rows_f32(0, 0, n, d)
    ids = synth.row_ids(n)
    emb = ora.catalog_frame(ids, m32.astype(np.float64))
    rated, rts = None, None
    for cand_rated, cand_rts in synth.user_ratings(2, n, 64):                      # the synthetic user closest to 85 liked / 133 rated
        if rated is None or abs(int((cand_rts >= 3.5).sum()) - 85) + abs(len(cand_rated) - 133) < abs(int((rts >= 3.5).sum()) - 85) + abs(len(rated) - 133):
            rated, rts = cand_rated, cand_rts
    liked = rated[rts >= 3.5]
    ratings = pd.DataFrame({"tmdb_id": [ids[r] for r in rated], "rating": rts})
    q = synth.query_f32(1, d)
    excl_ids = [ids[r] for r in rated]

    def best_median(fn, runs=5):
        fn()
        ts = []
        for _ in range(runs):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        return min(ts) * 1e3, statistics.median(ts) * 1e3

    cpu_user = best_median(lambda: ora.user_recs_ranked(emb, ratings, k))
    cpu_query = best_median(lambda: ora.single_query(emb, q.astype(np.float64), excl_ids, k))
    want_user = ora.user_recs_ranked(emb, ratings, k)
    want_query = ora.single_query(emb, q.astype(np.float64), excl_ids, k)

    store = CatalogStore.from_host(ids, m32, "fp32", device=dev)
    got_u = store.recommend(liked_rows=liked, exclude_rows=rated, k=k)
    got_q = store.recommend(query=q, exclude_rows=rated, k=k)
    for (rows, scores), want in ((got_u, want_user), (got_q, want_query)):
        assert [ids[r] for r in rows] == [w[0] for w in want], "C1: ids differ from the reference arithmetic"
        assert np.allclose(scores, [w[1] for w in want], rtol=1e-9, atol=0), "C1: scores differ from the reference arithmetic"
    gpu_user = best_median(lambda: store.recommend(liked_rows=liked, exclude_rows=rated, k=k), 200)
    gpu_query = best_median(lambda: store.recommend(query=q, exclude_rows=rated, k=k), 200)
    threads = None
    try:
        from threadpoolctl import threadpool_info
        threads = [{"api": t.get("internal_api"), "threads": t.get("num_threads")} for t in threadpool_info()]
    except Exception:
        pass
    return {"workload": f"{n} x {d} fp32 values (float64 frame on the CPU), k={k}, user with {len(liked)} liked of {len(rated)} rated movies",
            "cpu": {"impl": "oracle/reference_scoring.py = lib.py:42-55 (pandas + sklearn cosine_similarity), float64, measured at this size (not scaled)",
                    "user_recs_ms_best_median": cpu_user, "single_query_ms_best_median": cpu_query, "cores": os.cpu_count(),
                    "cpu_model": cpu_model(), "blas": threads},
            "gpu_e2e": {"impl": "CatalogStore.recommend, host buffers in and out", "user_recs_ms_best_median": gpu_user,
                        "single_query_ms_best_median": gpu_query},
            "speedup_user_recs": cpu_user[1] / gpu_user[1], "speedup_single_query": cpu_query[1] / gpu_query[1],
            "parity": "ids identical, scores within 1e-9 of the reference arithmetic (asserted in this run)"}


# ------------------------------------------------------------------------------------------------ GPU helpers
def independent_topk(store, dist_mod, world, q, excl, k, dtype, seed=0):
    """The answer by a route that shares nothing with the fused path: the plain dense-score kernel over every shard,
    torch.topk, all-gather of the shard winners, fp64 re-score of the union on the HOST from regenerated rows, one global
    (score desc, row asc) order (lib.py:55,63)."""
    import torch
    from robot_ebert_b200 import synth
    d = store.d
    qn = q.astype(np.float64) / np.linalg.norm(q.astype(np.float64))
    q32 = torch.zeros((1, store.ld), dtype=torch.float32, device=store.device)
    q32[0, :d] = torch.from_numpy(qn.astype(np.float32)).to(store.device)
    dense = store.scores_dense(q32)[0]
    loc = excl[(excl >= store.row_base) & (excl < store.row_base + store.n)] - store.row_base
    if len(loc):
        dense[torch.from_numpy(loc).to(store.device)] = -float("inf")
    top = torch.topk(dense, min(k + 8, store.n))
    cand = top.indices + store.row_base
    if world > 1:
        allc = torch.empty(world * cand.numel(), dtype=cand.dtype, device=store.device)
        dist_mod.all_gather_into_tensor(allc, cand.contiguous())
        cand = allc
    cand = np.unique(cand.cpu().numpy())
    exact = np.empty(len(cand))
    for i, r in enumerate(cand):
        row = synth.quantise(synth.catalog_rows_f32(seed, int(r), 1, d), dtype)[0]
        exact[i] = float(row @ qn / np.linalg.norm(row))
    order = np.lexsort((cand, -exact))[:k]
    return cand[order], exact[order]


def time_device(fn, steps, warmup, barrier, world, dist_mod, dev):
    """CUDA-event time of `steps` calls (ms per step, max over ranks), barrier + synchronize on both sides."""
    import torch
    for _ in range(warmup):
        fn()
    barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        fn()
    t1.record()
    barrier()
    ms = t0.elapsed_time(t1) / steps
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist_mod.all_reduce(t, op=dist_mod.ReduceOp.MAX)
        ms = float(t.item())
    return ms


def time_wall(fn, steps, warmup, barrier, world, dist_mod, dev):
    import torch
    for _ in range(warmup):
        fn()
    barrier()
    w0 = time.perf_counter()
    for _ in range(steps):
        fn()
    torch.cuda.synchronize()
    s = (time.perf_counter() - w0) / steps
    if world > 1:
        t = torch.tensor([s], dtype=torch.float64, device=dev)
        dist_mod.all_reduce(t, op=dist_mod.ReduceOp.MAX)
        s = float(t.item())
    return s


def batched_leg(store, sharded, world, rows_total, dev, barrier, B=4096, KB=100, steps=3, warmup=2, int8=False):
    """BASELINE configs 3/4: B users x catalog, top-KB, on the tcgen05 path; sharded when N>1.  One step = the whole batch
    INCLUDING the re-run of every query the batched pass could not prove (sync + single-query route inside the timed region)."""
    import ctypes as C
    import torch
    import torch.distributed as dist
    from robot_ebert_b200 import synth
    from robot_ebert_b200 import _native as nat
    lib = nat.load()
    q = synth.catalog_rows_f32(11, 0, B, DIM)
    qn32, qn64, qbf = store.prepare_queries(q)
    rng = np.random.default_rng(2)
    ep = np.zeros(B + 1, dtype=np.int64)
    ec = []
    for u in range(B):
        c = np.unique(rng.integers(0, rows_total, size=N_EXCL))
        ec.append(c)
        ep[u + 1] = ep[u] + len(c)
    ec = np.concatenate(ec).astype(np.int32)
    reruns = [0]
    if int8 and not store.batch_shadow_ok:
        raise RuntimeError("int8 operands need enable_prefilter() and rows of whole 128-byte k-blocks")
    if sharded is not None:
        ctx = sharded.batch_context(qbf, qn64, KB, ep, ec, qn32=qn32 if int8 else None)
        assert (ctx["shadow"] is not None) == int8
        plan = ctx["plan"]

        def step():
            sharded.batch_step(ctx)
            rows, scores, counts, status = sharded.batch_collect(ctx, q, ep, ec)
            reruns[0] = int((status != 0).sum())
            return rows, scores
    else:
        plan = store.gemm_plan(B, KB, shadow=int8)
        shadow = store.quantize_queries(qn32) if int8 else None
        ept, ect = torch.from_numpy(ep).to(dev), torch.from_numpy(ec).to(dev)
        ws = torch.empty(lib.rebert_gemm_workspace_bytes(C.byref(store._c), C.byref(plan)), dtype=torch.uint8, device=dev)
        o_rows = torch.empty((B, KB), dtype=torch.int64, device=dev)
        o_scores = torch.empty((B, KB), dtype=torch.float64, device=dev)
        o_count = torch.empty(B, dtype=torch.int32, device=dev)
        o_status = torch.empty(B, dtype=torch.int32, device=dev)
        scratch = store._scratch()

        def step():
            store.enqueue_batch(plan, qbf, qn64, ept, ect, ws, o_rows, o_scores, o_count, o_status, shadow=shadow)
            status = o_status.cpu().numpy()                                  # the sync a caller needs to know what to re-run
            redo = np.nonzero(status)[0]
            reruns[0] = len(redo)
            fix = {}
            for u in redo:
                scratch.qn32.copy_(qn32[u])
                scratch.qn64.copy_(qn64[u])
                fix[int(u)] = store.topk_prepared(KB, ect.data_ptr() + 4 * int(ep[u]), int(ep[u + 1] - ep[u]))
            return fix
    ms = time_device(step, steps, warmup, barrier, world, dist, dev)
    # digest of the whole [B, k] answer (re-runs patched in), identical at every N
    if sharded is not None:
        rows, scores = step()
    else:
        fix = step()
        rows, scores = o_rows.cpu().numpy(), o_scores.cpu().numpy()
        for u, (r, sc) in fix.items():
            rows[u, :len(r)], scores[u, :len(r)] = r, sc
    pk = measured_peaks()
    flops = 2.0 * B * rows_total * DIM
    tf = flops / (ms * 1e-3) / 1e12
    return {"workload": f"{B} users x {rows_total} x {DIM} bf16, top-{KB}, {N_EXCL}-row exclusions per user",
            "operands": "int8 shadow (tcgen05 kind::i8), exact fp64 pass over the bf16 rows" if int8 else "bf16 (tcgen05 kind::f16)",
            "value": B / (ms * 1e-3), "unit": "queries/s", "ms_per_batch": ms, "tflops": tf,
            "tflops_note": "2*B*N*D / time: the work of the bf16 GEMM the path replaces, whatever the operand type",
            "frac_of_measured_bf16_peak": tf / (pk["bf16"] * world),
            "frac_of_sustained_bf16_peak": (tf / (pk["bf16_sustained"] * world)) if pk["bf16_sustained"] else None,
            "peak_note": "burst = cuBLAS best of 10; sustained = cuBLAS back to back for seconds (the regime a ~100 ms batch runs in)",
            "bound": "tensor",
            "includes": "threshold sample + fused GEMM filter + per-query select + fp64 exact pass + status read-back + re-run of unproven queries"
                        + (" + all-gather + merge" if world > 1 else ""),
            "queries_rerun_on_single_query_path": reruns[0], "reruns_inside_timed_region": True,
            "ids_digest": digest(rows), "result_digest": digest(rows, scores), "_rows": rows, "_scores": scores,
            "digest_note": "ids_digest (sha1 over the [B, k] row ids) is the same at every N and for either operand type; score bits may "
                           "differ in the last ulp for queries that were re-run (the single-query exact pass divides element-wise "
                           "first, the batched one once per row)",
            "plan": {f: getattr(plan, f) for f, _ in plan._fields_}}


# ------------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    rows = args.rows or N_ROWS
    steps, warmup = max(1, args.steps), max(1, args.warmup)
    qps, desc, t, cores = cpu_reference_leg(rows, steps, warmup, args.cpu_sample_rows, budget_s=90.0)
    line = {"impl": "reference", "metric": METRIC, "value": qps, "unit": "queries/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": warmup, "ms_per_step": 1e3 / qps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": {"workload": workload_name(rows), "rows": rows, "dim": DIM, "k": K},
            "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": cores, "cpu_model": cpu_model(), "kind": "port", "sample": desc},
            "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def run_b200(args):
    import torch
    import torch.distributed as dist

    from robot_ebert_b200 import CatalogStore, RowFilter, synth
    from robot_ebert_b200 import _native as nat
    from robot_ebert_b200.catalog import unpack_result
    from robot_ebert_b200.sharding import ShardedCatalog

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; there is no CPU fallback for the scoring path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    rows = args.rows or N_ROWS
    steps, warmup = args.steps, max(3, args.warmup)
    lib = nat.load()
    kc = lib.rebert_candidates_for_k(K)
    pk = measured_peaks()

    if world > 1:
        sharded = ShardedCatalog.synthetic(0, rows, DIM, DTYPE, device=dev)
        store = sharded.backend.store
    else:
        sharded = None
        store = CatalogStore.synthetic(0, rows, DIM, DTYPE, device=dev)
    api = sharded if sharded is not None else store
    q = synth.query_f32(1, DIM)
    excl = np.random.default_rng(1).choice(rows, size=N_EXCL, replace=False).astype(np.int64)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- correctness of this very configuration, before timing: the answer of an independent route (dense-score kernel
    # over every shard + host fp64 re-score + one global order), and the digest every N must share
    got_rows, got_scores, info = api.recommend(query=q, exclude_rows=excl, k=K, return_info=True)
    want_rows, want_scores = independent_topk(store, dist, world, q, excl, K, DTYPE)
    assert np.array_equal(got_rows, want_rows), ("top-k ids differ from the independent route", got_rows, want_rows)
    assert np.allclose(got_scores, want_scores, rtol=1e-9, atol=0), (got_scores, want_scores)
    assert info["proven_exact"] and len(got_rows) == K and not set(got_rows.tolist()) & set(excl.tolist())
    result_digest = digest(got_rows, got_scores)
    dkey = f"query:{rows}x{DIM}:{DTYPE}:k{K}:excl{N_EXCL}"
    want_digest = expected_digest(dkey)
    if want_digest is not None:
        assert result_digest == want_digest, f"result digest {result_digest} != the committed single-GPU digest {want_digest} ({dkey})"

    # ---- value: device-resident query, ONE launch per step (fast pass + exact pass + ranking [+ exchange + merge])
    excl_ptr, ne = store.stage_inputs(q, None, None, excl, K, kc)
    if sharded is not None:
        sharded.backend._excl = (excl_ptr, ne)
    torch.cuda.synchronize()

    if sharded is not None:
        step = lambda: sharded.enqueue(K, kc)
    else:
        step = lambda: store.enqueue_fused(K, kc, excl_ptr, ne)
    for _ in range(warmup):
        step()
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    with ClockSampler(local_rank) as clocks:
        t0.record()
        for i in range(steps):
            kev[i][0].record()
            packed = step()
            kev[i][1].record()
        t1.record()
        barrier()
    outputs = dict(zip(("rows", "scores"), unpack_result(packed.cpu().numpy(), K)[:2]))
    elapsed_ms = t0.elapsed_time(t1)
    kernel_ms = sum(a.elapsed_time(b) for a, b in kev) / steps
    if world > 1:
        t = torch.tensor([elapsed_ms, kernel_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms, kernel_ms = float(t[0].item()), float(t[1].item())
    value = steps / (elapsed_ms * 1e-3)

    # ---- e2e: host buffers in, host buffers out, through the public API
    def e2e_step():
        outputs["e2e_rows"], outputs["e2e_scores"] = api.recommend(query=q, exclude_rows=excl, k=K)
    e2e_s = time_wall(e2e_step, steps, warmup, barrier, world, dist, dev)
    e2e = 1.0 / e2e_s
    h2d, d2h = int(store.last_h2d_bytes), int(store.last_d2h_bytes)

    configs = {}

    def compare_batched(a, b_, what):
        """bf16 vs int8 operands: the ids must be identical, the scores equal to the last ulp or so (see digest_note)."""
        if "_rows" in a and "_rows" in b_:
            assert np.array_equal(a["_rows"], b_["_rows"]), f"{what}: int8 operands changed the ids"
            assert np.allclose(a["_scores"], b_["_scores"], rtol=1e-12, atol=0, equal_nan=True), f"{what}: int8 operands changed the scores"
            b_["same_ids_as_bf16_operands"] = True

    def guarded(name, fn):
        try:
            configs[name] = fn()
        except Exception as e:  # the headline line must survive a failure of a secondary measurement
            configs[name] = {"error": repr(e)[:300]}

    # ---- profile request: the reference's real route (lib.py:43-55): ~85 liked rows -> profile, ~133 rated rows masked
    def profile_leg():
        rated, rts = None, None
        for cr, ct in synth.user_ratings(2, rows, 64):
            if rated is None or abs(int((ct >= 3.5).sum()) - 85) + abs(len(cr) - 133) < abs(int((rts >= 3.5).sum()) - 85) + abs(len(rated) - 133):
                rated, rts = cr, ct
        liked = rated[rts >= 3.5]
        r, sc, inf = api.recommend(liked_rows=liked, exclude_rows=rated, k=K, return_info=True)
        assert inf["proven_exact"] and not set(r.tolist()) & set(rated.tolist())
        ikey = f"profile-ids:{rows}x{DIM}:{DTYPE}:k{K}"
        want = expected_digest(ikey)
        if want is not None:
            assert digest(r) == want, f"profile request: ids digest {digest(r)} != the committed single-GPU digest {want}"
        s = time_wall(lambda: api.recommend(liked_rows=liked, exclude_rows=rated, k=K), steps, warmup, barrier, world, dist, dev)
        return {"workload": f"user-profile request: {len(liked)} liked rows -> mean of unit rows, {len(rated)} rated rows excluded, top-{K} over {rows} x {DIM} {DTYPE}",
                "e2e": {"value": 1.0 / s, "unit": "queries/s", "ms_per_step": 1e3 * s}, "vs_query_request_e2e": (1.0 / s) / e2e,
                "ids_digest": digest(r), "result_digest": digest(r, sc),
                "note": "ids identical at every N (asserted against tests/golden/bench_digests.json); scores agree to 1e-12 — the fp64 "
                        "partial profiles of the shards are added in rank order, a different association than one GPU's row order"}
    guarded("profile_request", profile_leg)

    # ---- int8 prefilter shadow: same request, half the bytes in the fast pass, same ids and scores (proven per request)
    def prefilter_leg():
        eps = api.enable_prefilter()
        r, sc, inf = api.recommend(query=q, exclude_rows=excl, k=K, return_info=True)
        same = bool(np.array_equal(r, got_rows) and np.array_equal(sc, got_scores))
        # The int8 kernel is partly compute-bound (dp4a), so its speed follows the SM clock: a 20-step burst right after an idle
        # phase ran 8 % faster than the same launches in a longer loop (tools/latency_breakdown.py: back-to-back = one at a time
        # = end to end once the clocks have settled).  Both measurements therefore run >= 60 steps after >= 20 warm-up steps.
        pf_steps, pf_warm = max(min(steps, 100), 60), max(warmup, 20)
        if sharded is not None:
            dev_ms = None
        else:
            dev_ms = time_device(lambda: store.enqueue_fused(K, 256, excl_ptr, ne, None, prefilter=True), pf_steps, pf_warm, barrier, world, dist, dev)
        s = time_wall(lambda: api.recommend(query=q, exclude_rows=excl, k=K), pf_steps, pf_warm, barrier, world, dist, dev)
        shadow_bytes = store.n * store._c8.ld
        out = {"workload": f"same request, fast pass over an int8 shadow of the catalog ({shadow_bytes / 1e9:.2f} GB per GPU), 256 candidates, "
                           f"exact fp64 pass over the bf16 rows in the same launch",
               "e2e": {"value": 1.0 / s, "unit": "queries/s", "ms_per_step": 1e3 * s},
               "error_bound": eps, "margin": inf.get("margin"), "proven_on_shadow_candidates": bool(inf.get("prefilter")),
               "same_ids_and_scores_as_plain_path": same, "result_digest": digest(r, sc), "rows": rows}
        if dev_ms is not None:
            out.update(value=1e3 / dev_ms, unit="queries/s", ms_per_step=dev_ms, shadow_gbs=shadow_bytes / (dev_ms * 1e-3) / 1e9,
                       frac_of_measured_hbm_peak=shadow_bytes / (dev_ms * 1e-3) / 1e9 / pk["hbm"],
                       e2e_vs_device_resident=(1.0 / s) / (1e3 / dev_ms))
        return out
    if not args.no_prefilter:
        guarded("prefilter_int8", prefilter_leg)

    # ---- C4 batched: 4096 users x the 10M catalog, top-100 (tcgen05), sharded when N > 1; bf16 operands, then int8
    if not args.no_batched:
        guarded("C4_batched_10M", lambda: batched_leg(store, sharded, world, rows, dev, barrier))
        if store.batch_shadow_ok:
            guarded("C4_batched_10M_int8", lambda: batched_leg(store, sharded, world, rows, dev, barrier, int8=True))
            compare_batched(configs.get("C4_batched_10M", {}), configs.get("C4_batched_10M_int8", {}), "C4")
        for name in ("C4_batched_10M", "C4_batched_10M_int8"):
            want = expected_digest(f"batched-ids:{rows}x{DIM}:B4096:k100")
            if want is not None and isinstance(configs.get(name), dict) and "ids_digest" in configs[name]:
                assert configs[name]["ids_digest"] == want, f"{name}: ids digest {configs[name]['ids_digest']} != committed {want}"

    # ---- C5 (N > 1): ragged-CSR profile build + genre/year-filtered top-50 over the sharded catalog
    def c5_leg():
        B, K5 = 4096, 50
        g, y = synth.movie_metadata(3, store.row_base, store.n)
        store.set_metadata(g, y)
        rf = RowFilter(genre_any=0b1011, year_lo=1960, year_hi=2000)
        rng = np.random.default_rng(2)
        lp = np.zeros(B + 1, dtype=np.int64)
        ep = np.zeros(B + 1, dtype=np.int64)
        lc, ec = [], []
        for u in range(B):                                   # ~133 rated / ~85 liked per user (create-embeddings.ipynb:961-975)
            rated = np.unique(rng.integers(0, rows, size=max(2, int(rng.lognormal(np.log(133) - 0.4, 0.9)))))
            liked = rated[rng.random(len(rated)) < 0.637]
            if len(liked) == 0:
                liked = rated[:1]
            lc.append(liked); ec.append(rated); lp[u + 1] = lp[u] + len(liked); ep[u + 1] = ep[u] + len(rated)
        lc = np.concatenate(lc).astype(np.int32)
        ec = np.concatenate(ec).astype(np.int32)
        red = (lambda t: dist.all_reduce(t, op=dist.ReduceOp.SUM)) if world > 1 else None
        build = lambda: store.build_profiles(lp, lc, None, reduce_fn=red)
        qn32, qn64, qbf = build()
        t_prof = time_device(build, 3, 1, barrier, world, dist, dev)
        if sharded is not None:
            ctx = sharded.batch_context(qbf, qn64, K5, ep, ec, rf)
            t_step = time_device(lambda: sharded.batch_step(ctx), 3, 1, barrier, world, dist, dev)
            status = ctx["gathered"][:, 2 * B * K5 + ctx["hb"]:].contiguous().view(torch.int32)[:, :B].max(dim=0).values
            nrerun = int((status != 0).sum().item())
            plan = ctx["plan"]
        else:
            import ctypes as C
            plan = store.gemm_plan(B, K5)
            ept, ect = torch.from_numpy(ep).to(dev), torch.from_numpy(ec).to(dev)
            ws = torch.empty(lib.rebert_gemm_workspace_bytes(C.byref(store._c), C.byref(plan)), dtype=torch.uint8, device=dev)
            o = (torch.empty((B, K5), dtype=torch.int64, device=dev), torch.empty((B, K5), dtype=torch.float64, device=dev),
                 torch.empty(B, dtype=torch.int32, device=dev), torch.empty(B, dtype=torch.int32, device=dev))
            t_step = time_device(lambda: store.enqueue_batch(plan, qbf, qn64, ept, ect, ws, *o, rf), 3, 1, barrier, world, dist, dev)
            nrerun = int((o[3] != 0).sum().item())
        flops = 2.0 * B * rows * DIM
        out = {"workload": f"C5: {world} x B200, {B} users (CSR, nnz_liked={len(lc)}), profile build + genre/year-filtered top-{K5} over {rows} x {DIM} bf16",
               "profile_build_ms": t_prof, "score_filter_topk_ms": t_step, "users_per_s": B / ((t_prof + t_step) * 1e-3),
               "tflops_scoring": flops / (t_step * 1e-3) / 1e12, "frac_of_measured_bf16_peak": flops / (t_step * 1e-3) / 1e12 / (pk["bf16"] * world),
               "queries_flagged_for_rerun": nrerun, "plan": {f: getattr(plan, f) for f, _ in plan._fields_}}
        if store.batch_shadow_ok:
            # the same step on int8 operands (the prefilter shadow, tcgen05 kind::i8): the ids of every user both passes prove must agree
            if sharded is not None:
                bf_rows, bf_status = ctx["m_rows"].clone(), status.clone()
                ctx8 = sharded.batch_context(qbf, qn64, K5, ep, ec, rf, qn32=qn32)
                t8 = time_device(lambda: sharded.batch_step(ctx8), 3, 1, barrier, world, dist, dev)
                st8 = ctx8["gathered"][:, 2 * B * K5 + ctx8["hb"]:].contiguous().view(torch.int32)[:, :B].max(dim=0).values
                rows8 = ctx8["m_rows"]
            else:
                bf_rows, bf_status = o[0].clone(), o[3].clone()
                plan8 = store.gemm_plan(B, K5, shadow=True)
                sh = store.quantize_queries(qn32)
                ws8 = torch.empty(lib.rebert_gemm_workspace_bytes(C.byref(store._c), C.byref(plan8)), dtype=torch.uint8, device=dev)
                t8 = time_device(lambda: store.enqueue_batch(plan8, qbf, qn64, ept, ect, ws8, *o, rf, shadow=sh), 3, 1, barrier, world, dist, dev)
                st8, rows8 = o[3], o[0]
            both = (bf_status == 0) & (st8 == 0)
            assert bool((rows8[both] == bf_rows[both]).all().item()), "C5: int8 and bf16 operands disagree on a proven user"
            out["int8_operands"] = {"score_filter_topk_ms": t8, "users_per_s": B / ((t_prof + t8) * 1e-3), "tflops_scoring": flops / (t8 * 1e-3) / 1e12,
                                    "queries_flagged_for_rerun": int((st8 != 0).sum().item()), "users_proven_by_both_with_equal_ids": int(both.sum().item())}
        return out
    if not args.no_batched:
        guarded("C5_csr_profiles_genre_year_top50", c5_leg)
    store._c8 = None                                     # free the shadow
    store._q8_rows = store._q8_factor = None
    if sharded is not None:
        sharded.q8_eps = None
    torch.cuda.empty_cache()

    # ---- single-GPU configs measured on rank 0's GPU only at N = 1 (they do not shard: C1-C3 are one-GPU configs)
    if world == 1 and not args.no_configs:
        del store
        if sharded is None:
            api = None
        torch.cuda.empty_cache()

        def c2_leg():
            out = {}
            for dt in ("fp32", "bf16"):
                n2 = 1_000_000
                st2 = CatalogStore.synthetic(0, n2, DIM, dt, device=dev)
                ex2 = np.random.default_rng(1).choice(n2, size=N_EXCL, replace=False).astype(np.int64)
                r, sc, inf = st2.recommend(query=q, exclude_rows=ex2, k=K, return_info=True)
                wr, ws_ = independent_topk(st2, dist, 1, q, ex2, K, dt)
                assert np.array_equal(r, wr) and np.allclose(sc, ws_, rtol=1e-9, atol=0) and inf["proven_exact"], f"C2 {dt}: parity"
                p2, n2e = st2.stage_inputs(q, None, None, ex2, K, kc)
                ms = time_device(lambda: st2.enqueue_fused(K, kc, p2, n2e), max(steps, 50), warmup, barrier, 1, dist, dev)
                s = time_wall(lambda: st2.recommend(query=q, exclude_rows=ex2, k=K), max(steps, 50), warmup, barrier, 1, dist, dev)
                nbytes = n2 * DIM * (4 if dt == "fp32" else 2)
                out[dt] = {"ms_per_query": ms, "queries_per_s": 1e3 / ms, "gbs": nbytes / (ms * 1e-3) / 1e9,
                           "frac_of_measured_hbm_peak": nbytes / (ms * 1e-3) / 1e9 / pk["hbm"],
                           "e2e_queries_per_s": 1.0 / s, "result_digest": digest(r, sc),
                           "parity": "ids == independent dense-kernel route, scores within 1e-9 (asserted)"}
                if dt == "bf16":
                    out["_bf16_store"] = st2
                else:
                    del st2
                    torch.cuda.empty_cache()
            return out
        guarded("C2_1M_single_query", c2_leg)
        st_1m = None
        if isinstance(configs.get("C2_1M_single_query"), dict):
            st_1m = configs["C2_1M_single_query"].pop("_bf16_store", None)
            configs["C2_1M_single_query"]["workload"] = f"1M x {DIM}, single-query top-{K} + {N_EXCL}-row exclusion, one launch per query"
        if st_1m is not None and not args.no_batched:
            guarded("C3_batched_4096x1M_top100", lambda: batched_leg(st_1m, None, 1, 1_000_000, dev, barrier, steps=5))
            if not args.no_prefilter:
                def c3_int8():
                    st_1m.enable_prefilter()
                    return batched_leg(st_1m, None, 1, 1_000_000, dev, barrier, steps=5, int8=True)
                guarded("C3_batched_4096x1M_top100_int8", c3_int8)
                compare_batched(configs.get("C3_batched_4096x1M_top100", {}), configs.get("C3_batched_4096x1M_top100_int8", {}), "C3")
        del st_1m
        torch.cuda.empty_cache()
        guarded("C1_cpu_sized_catalog", lambda: config_c1(dev))
        # the reference's production catalog shape (movies-collab: 2269 x 32, create-embeddings.ipynb:1241)
        def prod_leg():
            n3, d3 = 2269, 32
            st3 = CatalogStore.synthetic(0, n3, d3, "fp32", device=dev)
            (rated, rts), = synth.user_ratings(2, n3, 1)
            liked = rated[rts >= 3.5]
            r, sc, inf = st3.recommend(liked_rows=liked, exclude_rows=rated, k=K, return_info=True)
            s1 = time_wall(lambda: st3.recommend(liked_rows=liked, exclude_rows=rated, k=K), 2000, 50, barrier, 1, dist, dev)
            q3 = synth.query_f32(1, d3)
            s2 = time_wall(lambda: st3.recommend(query=q3, exclude_rows=rated, k=K), 2000, 50, barrier, 1, dist, dev)
            return {"workload": f"{n3} x {d3} fp32 (the reference's production collab catalog), user with {len(liked)} liked / {len(rated)} rated",
                    "e2e_user_recs_us": s1 * 1e6, "e2e_single_query_us": s2 * 1e6, "kernels_per_request": 3,
                    "route": "general (staging kernel -> streaming kernel -> exact-pass cluster kernel)"}
        guarded("production_shape_2269x32", prod_leg)

    for v in configs.values():                               # arrays kept only for the comparisons above
        if isinstance(v, dict):
            v.pop("_rows", None)
            v.pop("_scores", None)
    if rank == 0:
        shard_rows = (rows * 1) // world if world > 1 else rows
        alg_bytes = shard_rows * DIM * 2                                  # catalog bytes one launch must read
        achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
        traffic = ncu_traffic(f"gemv_topk_bf16_{shard_rows}") if world == 1 else None
        line = {
            "metric": METRIC, "value": value, "unit": "queries/s", "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": elapsed_ms / steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": workload_name(rows), "rows": rows, "dim": DIM, "k": K, "exclusions": N_EXCL,
                       "arithmetic": "bf16 catalog, fp32 accumulate in the streaming kernel, fp64 exact pass over the candidates",
                       "parallelism": f"row-shard x{world}" if world > 1 else "single GPU",
                       "exchange": (("NVLink peer-memory stores + flags + merge in the tail of the scoring launch" if sharded.backend.exchange == "p2p"
                                     else "NCCL all-gather + merge kernel") if world > 1 else None),
                       "l2": f"inputs larger than L2 ({alg_bytes / 1e9:.2f} GB read per step per GPU)"},
            "result_digest": result_digest, "result_digest_expected": want_digest,
            "result_check": "ids == independent dense-score-kernel route over all shards + host fp64 re-score; digest == committed single-GPU digest",
            "roofline": {"bound": "hbm", "kernel": "gemv_topk_kernel<bf16,6,32,1> (scores + mask + top-k, publishes pruned keys) with the exact-pass "
                                                   "cluster kernel behind it (selection + fp64 re-score + ranking"
                                                   + (" + NVLink exchange + merge" if world > 1 else "") + "): the time is the pair's, per request; "
                                                   "the bytes are the streaming kernel's",
                         "achieved": achieved, "peak": pk["hbm"], "peak_source": pk["hbm_src"], "unit": "GB/s", "frac": achieved / pk["hbm"],
                         "note": "the measured peak is a read+write copy; this kernel only reads, which HBM serves faster, so frac can exceed 1",
                         "kernel_ms": kernel_ms, "algorithmic_bytes": alg_bytes, "traffic": traffic,
                         "traffic_source": "profiles/roofline_traffic.json (ncu --set full capture of this kernel, not measured in this run)" if traffic else None},
            "e2e": {"value": e2e, "unit": "queries/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": 1e3 * e2e_s, "kernels_per_request": 3,
                    "kernels": "stage_query_kernel (zero-copy from the pinned request) -> gemv_topk_kernel -> finalize_published_kernel (cluster of 8)"},
            "gpu_launches": 2 * steps,
            "gpu_launches_note": "timed device-resident step = gemv_topk_kernel + finalize_published_kernel per request",
            "clocks": clocks.summary(),
            "configs": configs,
            "batched": configs.get("C4_batched_10M"),
            "prefilter_int8": configs.get("prefilter_int8"),
        }
        if world == 1 and not args.no_cpu_baseline:
            qps, desc, _, cores = cpu_reference_leg(rows, 5, 1, args.cpu_sample_rows, budget_s=20.0)
            line["cpu_baseline"] = {"value": qps, "unit": "queries/s", "cores": cores, "cpu_model": cpu_model(), "kind": "port", "sample": desc}
        if args.dump_outputs:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in outputs.items():
                np.save(os.path.join(args.dump_outputs, f"{name}.npy"), np.asarray(a, dtype=np.float64))
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rows", type=int, default=0, help="override catalog rows (default 10M)")
    ap.add_argument("--cpu-sample-rows", type=int, default=200_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-prefilter", action="store_true", help="skip the int8-prefilter measurement")
    ap.add_argument("--no-batched", action="store_true", help="skip the batched (tcgen05) measurements")
    ap.add_argument("--no-configs", action="store_true", help="skip the single-GPU BASELINE configs C1-C3 and the production shape")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
