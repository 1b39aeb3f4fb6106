#!/usr/bin/env python
"""Batched recommendations with long lists: 4096 users x 1M x 1536 bf16 with per-user exclusion CSR, k from 100 to 2048.

In one process, for k in --ks and both operand types (bf16, int8 over the prefilter shadow):
  * device step time of the batched pass (CUDA events around --steps steps after --warmup), users/s, the plan, its workspace
    bytes and the fraction of queries with status != 0;
  * end-to-end CatalogStore.recommend_batch (host clock around a synchronised call: staging, the pass, the widened retry of
    long lists and the per-query route for what is still unproven);
  * per-kernel device times from a separate torch.profiler pass (one step per configuration);
  * recommend() one user at a time at k = 1000 for 16 users, which is what long lists cost before they had a batched path;
  * the GPU name and power limit (nvidia-smi), which belong beside every number.
Writes <out>.json (everything) and prints a summary.  Needs a GPU; nothing here falls back to the CPU.
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

from robot_ebert_b200 import CatalogStore, _native as nat, synth  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--rows", type=int, default=1_000_000)
ap.add_argument("--batch", type=int, default=4096)
ap.add_argument("--dim", type=int, default=1536)
ap.add_argument("--ks", type=str, default="100,241,500,1000,2048")
ap.add_argument("--steps", type=int, default=5)
ap.add_argument("--warmup", type=int, default=2)
ap.add_argument("--single-users", type=int, default=16)
ap.add_argument("--out", type=str, required=True, help="output path prefix (writes <out>.json)")
args = ap.parse_args()
assert torch.cuda.is_available(), "needs a CUDA device"

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True).stdout.strip()
dev = torch.device("cuda:0")
lib = nat.load()
store = CatalogStore.synthetic(0, args.rows, args.dim, "bf16", device=dev)
store.enable_prefilter()
q = synth.catalog_rows_f32(11, 0, args.batch, args.dim)
qn32, qn64, qbf = store.prepare_queries(q)
users = synth.user_ratings(2, args.rows, args.batch)
ep = np.zeros(args.batch + 1, dtype=np.int64)
ec = []
for u, (rated, _) in enumerate(users):
    ec.append(np.sort(rated))
    ep[u + 1] = ep[u] + len(rated)
ec = np.concatenate(ec).astype(np.int32)
ept, ect = torch.from_numpy(ep).to(dev), torch.from_numpy(ec).to(dev)
ks = [int(x) for x in args.ks.split(",")]
ops = [("bf16", False), ("int8", True)]
shadow = store.quantize_queries(qn32)


def setup(k, int8):
    plan = store.gemm_plan(args.batch, k, shadow=int8)
    wsb = lib.rebert_gemm_workspace_bytes(C.byref(store._c), C.byref(plan))
    t = dict(plan=plan, ws_bytes=wsb, ws=torch.empty(wsb, dtype=torch.uint8, device=dev),
             rows=torch.empty((args.batch, k), dtype=torch.int64, device=dev),
             scores=torch.empty((args.batch, k), dtype=torch.float64, device=dev),
             count=torch.empty(args.batch, dtype=torch.int32, device=dev),
             status=torch.empty(args.batch, dtype=torch.int32, device=dev))
    t["step"] = lambda: store.enqueue_batch(plan, qbf, qn64, ept, ect, t["ws"], t["rows"], t["scores"], t["count"], t["status"],
                                            shadow=shadow if int8 else None)
    return t


results = []
for k in ks:
    for name, int8 in ops:
        t = setup(k, int8)
        for _ in range(args.warmup):
            t["step"]()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            t["step"]()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / args.steps
        status = t["status"].cpu().numpy()
        plan = t["plan"]
        r = {"k": k, "operands": name, "step_ms": ms, "users_per_s": args.batch / (ms * 1e-3),
             "plan": {f: getattr(plan, f) for f, _ in plan._fields_}, "workspace_bytes": t["ws_bytes"],
             "status_nonzero_fraction": float((status != 0).mean()),
             "status_hist": {int(a): int(c) for a, c in zip(*np.unique(status, return_counts=True))}}
        del t
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        _, _, _, info = store.recommend_batch(queries=q, excl_ptr=ep, excl_col=ec, k=k, return_info=True, prefilter=int8)
        torch.cuda.synchronize()
        r["e2e_recommend_batch_s"] = time.perf_counter() - t0
        r["e2e_per_query_route"] = int(info["per_query"])
        results.append(r)
        print(json.dumps({x: r[x] for x in ("k", "operands", "step_ms", "users_per_s", "status_nonzero_fraction", "workspace_bytes",
                                            "e2e_recommend_batch_s", "e2e_per_query_route")}), flush=True)

# per-kernel times: one profiled step per configuration, in a pass of its own
from torch.profiler import ProfilerActivity, profile  # noqa: E402
kernels = {}
for k in ks:
    for name, int8 in ops:
        t = setup(k, int8)
        t["step"]()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            t["step"]()
            torch.cuda.synchronize()
        per = {}
        for ev in prof.events():
            if ev.device_type == torch.autograd.DeviceType.CUDA:
                key = ev.name.split("(")[0][:90]
                per[key] = per.get(key, 0.0) + ev.device_time_total / 1e3
        kernels[f"{name} k={k}"] = dict(sorted(per.items(), key=lambda kv: -kv[1]))
        del t

# what a long list cost before: recommend() one user at a time
single = []
for u in range(args.single_users):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    store.recommend(query=q[u], exclude_rows=ec[ep[u]:ep[u + 1]], k=1000)
    torch.cuda.synchronize()
    single.append(time.perf_counter() - t0)

out = {"gpu": gpu, "workload": f"{args.batch} users x {args.rows} rows x {args.dim} bf16, per-user exclusion CSR "
                               f"({len(ec)} rows in all)", "steps": args.steps, "warmup": args.warmup,
       "results": results, "kernel_ms_per_step": kernels,
       "recommend_k1000_single_user_s": {"median": float(np.median(single)), "min": float(np.min(single)),
                                         "max": float(np.max(single)), "users": args.single_users}}
os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
with open(args.out + ".json", "w") as f:
    json.dump(out, f, indent=1)
print(gpu)
print(json.dumps(out["recommend_k1000_single_user_s"]))
for key, per in kernels.items():
    print(key, {a: round(b, 3) for a, b in list(per.items())[:6]})
