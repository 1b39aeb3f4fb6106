#!/usr/bin/env python
"""A/B of the int8-gated single-query fast pass against the plain one (DESIGN.md §4.5), in one process.

For each catalog the same store is timed through enqueue_fused (the device-resident request: streaming kernel + exact-pass
cluster kernel) with its gate and with the gate removed — the gate-free store runs the plain kernel path.  The two
alternate ROUNDS times, STEPS steps each, timed by CUDA events; the packed results of both must be equal bit for bit.
Reports per-variant median / min / max step time, rows fetched from the catalog of record per query (the gate's pass
rate) and the gated kernel's int8 GB/s.  Prints the GPU's name, power limit and max SM clock first.
    python tools/bench_gate.py [--cases headline,c2,small,realistic] [--rounds 5] [--steps 200]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from robot_ebert_b200 import CatalogStore, synth  # noqa: E402
from robot_ebert_b200 import _native as nat  # noqa: E402

K, N_EXCL = 10, 133
CASES = {
    "headline": [(10_000_000, 1536, "bf16")],
    "c2": [(1_000_000, 1536, "fp32"), (1_000_000, 1536, "bf16")],
    "small": [(30_000, 1536, "bf16"), (100_000, 1536, "bf16"), (300_000, 1536, "bf16"), (10_000, 1536, "fp32"),
              (100_000, 1536, "fp32")],
    "realistic": [(1_000_000, 1536, "bf16"), (10_000_000, 1536, "bf16")],
}


def fetches(store):
    return store.gate_fetches()


def shared_mean_rows(store, seed, cos=0.7):
    """Overwrite the rows with a shared unit direction + isotropic noise (pairwise cosine ~cos, like ada-002 embeddings)."""
    g = torch.Generator(device=store.device).manual_seed(seed)
    d = store.d
    m = torch.randn(d, generator=g, device=store.device, dtype=torch.float32)
    m /= m.norm()
    for s in range(0, store.n, 1 << 18):
        e = min(store.n, s + (1 << 18))
        noise = torch.randn((e - s, d), generator=g, device=store.device, dtype=torch.float32) / np.sqrt(d)
        store.rows[s:e, :d] = (np.sqrt(cos) * m + np.sqrt(1 - cos) * noise).to(store.rows.dtype)
    lib = nat.load()
    nat.check(lib.rebert_catalog_norms(store.rows.data_ptr(), store.n, store.ld, nat.DTYPES[store.dtype], store.inv_norm.data_ptr(),
                                       store.norm64.data_ptr(), torch.cuda.current_stream().cuda_stream))
    q = (np.sqrt(cos) * m + np.sqrt(1 - cos) * torch.randn(d, generator=g, device=store.device) / np.sqrt(d)).cpu().numpy()
    return q.astype(np.float32)


def time_steps(step, steps):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    torch.cuda.synchronize()
    ev[0].record()
    for _ in range(steps):
        out = step()
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / steps, out


def ab(n, d, dtype, rounds, steps, realistic=False):
    st = CatalogStore.synthetic(0, n, d, dtype, device="cuda:0")
    q = synth.query_f32(1, d)
    if realistic:
        q = shared_mean_rows(st, 7)
    kept = st.has_gate                                 # the constructor's rule (for the realistic rows: before they were written)
    if realistic:
        st.drop_gate()
        st.build_gate()
        kept = st._gate_pays()
    if not st.build_gate():
        return {"catalog": f"{n} x {d} {dtype}", "gate": "not available for this layout"}
    kc = nat.load().rebert_candidates_for_k(K)
    excl = np.random.default_rng(1).choice(n, size=N_EXCL, replace=False).astype(np.int64)
    excl_ptr, ne = st.stage_inputs(q, None, None, excl, K, kc)
    step = lambda: st.enqueue_fused(K, kc, excl_ptr, ne)
    res = {"gated": [], "plain": []}
    outs = {}
    fetched = []
    for _ in range(3):
        step()
    for r in range(rounds):
        for variant in ("gated", "plain"):
            if variant == "gated":
                st.build_gate()
            else:
                st.drop_gate()
            step()
            f0 = fetches(st)
            ms, out = time_steps(step, steps)
            if variant == "gated":
                fetched.append((fetches(st) - f0) / steps)
            res[variant].append(ms)
            outs.setdefault(variant, out.cpu().numpy().copy())
            assert np.array_equal(out.cpu().numpy(), outs[variant]), "result changed between rounds"
    assert np.array_equal(outs["gated"], outs["plain"]), "gated and plain results differ"
    rows = outs["plain"][:K]
    ld8 = st.layout(n, d, "i8")[0]
    med = {v: float(np.median(t)) for v, t in res.items()}
    out = {"catalog": f"{n} x {d} {dtype}" + (" shared-mean rows (pairwise cosine ~0.7)" if realistic else " synthetic"),
           "rounds": rounds, "steps_per_round": steps, "top_rows": rows.tolist(), "bit_equal": True,
           "row_err": st.q8_row_err, "constructor_keeps_gate": kept, "probe_fetches": getattr(st, "last_probe_fetches", None)}
    for v in ("gated", "plain"):
        out[v] = {"median_ms": med[v], "min_ms": min(res[v]), "max_ms": max(res[v]), "qps": 1e3 / med[v], "all_ms": res[v]}
    out["speedup"] = med["plain"] / med["gated"]
    out["fetched_rows_per_query"] = float(np.median(fetched))
    out["fetched_fraction"] = float(np.median(fetched)) / n
    out["gated_int8_gbs"] = n * ld8 / (med["gated"] * 1e-3) / 1e9
    out["plain_gbs"] = n * st.ld * st.rows.element_size() / (med["plain"] * 1e-3) / 1e9
    del st
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="headline,c2,small,realistic")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_gate.py needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print(json.dumps({"gpu": smi}), flush=True)
    for case in args.cases.split(","):
        for n, d, dtype in CASES[case]:
            r = ab(n, d, dtype, args.rounds, args.steps, realistic=(case == "realistic"))
            r["case"] = case
            print(json.dumps(r), flush=True)


if __name__ == "__main__":
    main()
