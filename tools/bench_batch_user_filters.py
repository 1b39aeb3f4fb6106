#!/usr/bin/env python
"""Batched top-50 with a genre / year filter per user: 4096 users (liked-rows CSR profiles, per-user exclusion CSR) x 1M and
10M rows x 1536 bf16, metadata from synth.movie_metadata(3, ...), bf16 and int8 operands.

Legs of the device-resident batched step (CatalogStore.enqueue_batch):
  a  no filter
  b  the shared C5 filter RowFilter(0b1011, 1960, 2000)
  c  a random genre set (1-6 of 19 bits) and year window (10-60 years) per user
  d  like c, with 1 % of users narrowed to one genre bit and one year, which leaves fewer than sample_rank allowed rows in the
     threshold sample for most of them (tau = -inf: every allowed row survives, the epilogue takes its rare path per chunk)
  e  per-user filters all equal to b's
For each leg: step time (CUDA events over --steps steps after --warmup), users/s, queries flagged for re-run, queries whose
threshold came out -inf, and the wall time of the per-query re-run of the flagged queries (host clock around a synchronised
call).  Asserts that e equals b bit for bit and that 64 sampled proven users of c equal their single-query results.
Records the GPU name and power limit in the same run.  Writes <out>.json.  Needs a GPU; nothing here falls back to the CPU.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from robot_ebert_b200 import CatalogStore, QueryFilters, RowFilter, _native as nat, synth  # noqa: E402
from robot_ebert_b200.catalog import sorted_csr  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--rows", type=str, default="1000000,10000000")
ap.add_argument("--batch", type=int, default=4096)
ap.add_argument("--dim", type=int, default=1536)
ap.add_argument("--k", type=int, default=50)
ap.add_argument("--steps", type=int, default=5)
ap.add_argument("--warmup", type=int, default=2)
ap.add_argument("--out", type=str, required=True, help="output path prefix (writes <out>.json)")
args = ap.parse_args()
assert torch.cuda.is_available(), "needs a CUDA device"

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True).stdout.strip()
dev = torch.device("cuda:0")
lib = nat.load()
B, K = args.batch, args.k
C5 = (0b1011, 1960, 2000)


def users(rows):
    """~133 rated / ~85 liked per user, as bench.py's C5 leg."""
    rng = np.random.default_rng(2)
    lp, ep = np.zeros(B + 1, dtype=np.int64), np.zeros(B + 1, dtype=np.int64)
    lc, ec = [], []
    for u in range(B):
        rated = np.unique(rng.integers(0, rows, size=max(2, int(rng.lognormal(np.log(133) - 0.4, 0.9)))))
        liked = rated[rng.random(len(rated)) < 0.637]
        if len(liked) == 0:
            liked = rated[:1]
        lc.append(liked); ec.append(rated); lp[u + 1] = lp[u] + len(liked); ep[u + 1] = ep[u] + len(rated)
    return lp, np.concatenate(lc).astype(np.int32), ep, np.concatenate(ec).astype(np.int32)


def random_filters(seed, narrow_frac):
    rng = np.random.default_rng(seed)
    ga = np.zeros(B, dtype=np.uint32)
    for u in range(B):
        ga[u] = np.bitwise_or.reduce(np.uint32(1) << rng.choice(19, size=int(rng.integers(1, 7)), replace=False).astype(np.uint32))
    width = rng.integers(10, 61, size=B)
    lo = rng.integers(1920, 2024 - width)
    hi = lo + width - 1
    narrow = rng.random(B) < narrow_frac
    ga[narrow] = np.uint32(1) << rng.integers(0, 19, size=int(narrow.sum())).astype(np.uint32)
    hi[narrow] = lo[narrow]
    return QueryFilters(ga, lo, hi), narrow


def tau_of(ws, plan):
    """The thresholds of the last step: the workspace starts with the sample [b, sample_rows] fp32, then tau [b] (256-byte
    aligned pieces, gemm_topk.cu carve())."""
    off = (plan.b * plan.sample_rows * 4 + 255) // 256 * 256
    return ws[off:off + 4 * plan.b].view(torch.float32).cpu().numpy()


results = []
for rows in [int(x) for x in args.rows.split(",")]:
    store = CatalogStore.synthetic(0, rows, args.dim, "bf16", device=dev)
    store.enable_prefilter()
    store.set_metadata(*synth.movie_metadata(3, 0, rows))
    lp, lc, ep, ec = users(rows)
    qn32, qn64, qbf = store.build_profiles(lp, lc)
    ep_s, ec_s = sorted_csr(ep, ec)
    ept, ect = torch.from_numpy(ep_s).to(dev), torch.from_numpy(ec_s).to(dev)
    qf_c, _ = random_filters(5, 0.0)
    qf_d, narrow = random_filters(5, 0.01)
    legs = {"a": (None, None), "b": (RowFilter(*C5), None), "c": (None, qf_c), "d": (None, qf_d),
            "e": (None, QueryFilters(np.full(B, C5[0]), np.full(B, C5[1]), np.full(B, C5[2])))}
    for op, int8 in (("bf16", False), ("int8", True)):
        plan = store.gemm_plan(B, K, shadow=int8)
        shadow = store.quantize_queries(qn32) if int8 else None
        ws = torch.empty(lib.rebert_gemm_workspace_bytes(C.byref(store._c), C.byref(plan)), dtype=torch.uint8, device=dev)
        out = {}
        for leg, (rf, qf) in legs.items():
            o = (torch.empty((B, K), dtype=torch.int64, device=dev), torch.empty((B, K), dtype=torch.float64, device=dev),
                 torch.empty(B, dtype=torch.int32, device=dev), torch.empty(B, dtype=torch.int32, device=dev))
            step = lambda: store.enqueue_batch(plan, qbf, qn64, ept, ect, ws, *o, rf, shadow=shadow, query_filters=qf)  # noqa: E731
            for _ in range(args.warmup):
                step()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                step()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / args.steps
            tau = tau_of(ws, plan)
            r_rows, r_scores, r_count, r_status = (t.cpu().numpy() for t in o)
            redo = np.nonzero(r_status)[0]
            t0 = time.perf_counter()
            store._rerun_prepared(redo, qn32, qn64, ep_s, ect, K, rf, r_rows.copy(), r_scores.copy(), r_count.copy(), qf)
            torch.cuda.synchronize()
            rerun_s = time.perf_counter() - t0
            out[leg] = dict(rows=r_rows, scores=r_scores, status=r_status)
            r = {"rows": rows, "operands": op, "leg": leg, "step_ms": ms, "users_per_s": B / (ms * 1e-3),
                 "queries_flagged_for_rerun": int(len(redo)), "rerun_wall_s": rerun_s,
                 "tau_minus_inf": int(np.isneginf(tau).sum()),
                 "status_hist": {int(a): int(c) for a, c in zip(*np.unique(r_status, return_counts=True))}}
            if leg == "d":
                r["narrow_users"] = int(narrow.sum())
                r["narrow_users_tau_minus_inf"] = int(np.isneginf(tau[narrow]).sum())
            results.append(r)
            print(json.dumps(r), flush=True)
        # e is the shared C5 filter expressed per user: same thresholds, same survivors, same bits
        assert np.array_equal(out["e"]["rows"], out["b"]["rows"]), f"{rows} {op}: per-user C5 filters differ from the shared one"
        assert np.array_equal(out["e"]["scores"].view(np.int64), out["b"]["scores"].view(np.int64))
        assert np.array_equal(out["e"]["status"], out["b"]["status"])
        # 64 sampled proven users of c against the single-query path with their own RowFilter
        proven = np.nonzero(out["c"]["status"] == 0)[0]
        for u in np.random.default_rng(rows).choice(proven, size=min(64, len(proven)), replace=False):
            r_, s_ = store.recommend(liked_rows=lc[lp[u]:lp[u + 1]], exclude_rows=ec[ep[u]:ep[u + 1]], k=K, row_filter=qf_c.row_filter(u))
            got = out["c"]["rows"][u]
            assert np.array_equal(got[:len(r_)], r_) and (got[len(r_):] == -1).all(), f"{rows} {op}: user {u} differs from recommend()"
        del ws, shadow
    del store, qn32, qn64, qbf
    torch.cuda.empty_cache()

summary = {}
for r in results:
    summary.setdefault(f"{r['rows']} {r['operands']}", {})[r["leg"]] = round(r["step_ms"], 3)
for key, legs in summary.items():
    legs["c_over_b"] = round(legs["c"] / legs["b"], 3)
    legs["d_over_b"] = round(legs["d"] / legs["b"], 3)
res = {"gpu": gpu, "workload": f"{B} users (liked-rows CSR profiles, exclusion CSR) x {args.dim} bf16, top-{K}, metadata synth.movie_metadata(3)",
       "steps": args.steps, "warmup": args.warmup, "step_ms_by_leg": summary, "results": results}
os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
with open(args.out + ".json", "w") as f:
    json.dump(res, f, indent=1)
print(gpu)
print(json.dumps(summary, indent=1))
