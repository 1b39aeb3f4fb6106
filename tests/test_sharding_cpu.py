"""Sharding layer host logic on CPU: ShardPlan arithmetic and a world_size-2 gloo run of ShardedCatalog with an
oracle-backed shard backend (tests only) — results must equal the unsharded oracle on every rank."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from robot_ebert_b200 import synth
from robot_ebert_b200.catalog import close_proof, unpack_result, widen_until_proven
from robot_ebert_b200.sharding import ShardedCatalog, ShardPlan


def test_shard_plan_partitions_rows():
    for n, w in [(10, 3), (10_000_000, 8), (7, 8), (0, 2), (1_000_003, 4)]:
        plan = ShardPlan(n, w)
        ranges = [plan.range(g) for g in range(w)]
        assert ranges[0][0] == 0 and sum(c for _, c in ranges) == n
        for g in range(w - 1):
            assert ranges[g][0] + ranges[g][1] == ranges[g + 1][0]
        assert max(c for _, c in ranges) - min(c for _, c in ranges) <= 1
        for row in ([0, n - 1, n // 2, n // 3] if n else []):
            g = plan.owner(row)
            assert ranges[g][0] <= row < ranges[g][0] + ranges[g][1]
    with pytest.raises(ValueError):
        ShardPlan(10, 0)


class OracleShardBackend:
    """Test double with the CudaShardBackend interface; arithmetic by the oracle on CPU tensors."""

    def __init__(self, m_local, row0):
        from oracle.reference_scoring import _normalize_rows
        self.unit = _normalize_rows(m_local)
        self.row0, self.n, self.d = row0, m_local.shape[0], m_local.shape[1]
        self.device = torch.device("cpu")

    def stage(self, query, liked_rows, weights, exclude_rows, k, kc):
        self.excl = None if exclude_rows is None else np.asarray(exclude_rows, dtype=np.int64)
        if liked_rows is None:
            q = np.asarray(query, dtype=np.float64)
            nrm = np.linalg.norm(q)
            self.vec = q / (nrm if nrm else 1.0)
            return None
        liked = np.asarray(liked_rows, dtype=np.int64)
        w = np.ones(len(liked)) if weights is None else np.asarray(weights, dtype=np.float64)
        mine = (liked >= self.row0) & (liked < self.row0 + self.n)
        part = (self.unit[liked[mine] - self.row0] * w[mine, None]).sum(axis=0)
        return torch.from_numpy(np.concatenate([part, [w.sum()]]))

    def set_profile(self, summed):
        s = summed.numpy()
        self.vec = s[:self.d] / (s[self.d] / self._world)

    def _allowed_scores(self):
        scores = self.unit @ self.vec
        ok = np.ones(self.n, dtype=bool)
        if self.excl is not None:
            ok[self.excl[(self.excl >= self.row0) & (self.excl < self.row0 + self.n)] - self.row0] = False
        return scores, ok

    def count_local(self, threshold, row_filter):
        scores, ok = self._allowed_scores()
        return int(np.count_nonzero(ok & (scores >= threshold)))

    def sweep_local(self, threshold, row_filter):
        scores, ok = self._allowed_scores()
        rows = np.nonzero(ok & (scores >= threshold))[0]
        return rows.astype(np.int64) + self.row0, scores[rows]

    def local_topk(self, k, kc, row_filter):
        from oracle.reference_scoring import topk_rows
        scores = self.unit @ self.vec
        excl = None
        if self.excl is not None:
            excl = self.excl[(self.excl >= self.row0) & (self.excl < self.row0 + self.n)] - self.row0
        rows, sc = topk_rows(scores, k, excl)
        words = np.zeros(2 * k + 2, dtype=np.int64)
        words[:len(rows)] = rows + self.row0
        words[len(rows):k] = -1
        words[k:k + len(rows)] = sc.view(np.int64)
        words[2 * k:2 * k + 1].view(np.int32)[0] = len(rows)
        words[2 * k + 1:].view(np.float64)[0] = np.inf
        return torch.from_numpy(words)

    def merge(self, gathered, k):
        g = gathered.numpy()
        rows, scores = [], []
        for l in range(g.shape[0]):
            r, s, _ = unpack_result(g[l], k)
            rows.append(r)
            scores.append(s)
        rows, scores = np.concatenate(rows), np.concatenate(scores)
        order = np.lexsort((rows, -scores))[:k]
        words = np.zeros(2 * k + 2, dtype=np.int64)
        words[:len(order)] = rows[order]
        words[k:k + len(order)] = scores[order].view(np.int64)
        words[2 * k:2 * k + 1].view(np.int32)[0] = len(order)
        words[2 * k + 1:].view(np.float64)[0] = np.inf
        return torch.from_numpy(words)

    def fetch(self, packed, k):
        return unpack_result(packed.numpy(), k)


class UnprovenShardBackend(OracleShardBackend):
    """The merged result reports margin 0, so no candidate list proves itself and the fail-closed route must answer."""

    def merge(self, gathered, k):
        words = super().merge(gathered, k)
        words.numpy()[2 * k + 1:].view(np.float64)[0] = 0.0
        return words


class OverflowShardBackend(UnprovenShardBackend):
    """... and every sweep overflows, so neither exhaustive route can answer either."""

    def sweep_local(self, threshold, row_filter):
        return None


def _batch_inputs(n, d, b):
    """b queries, a weighted liked CSR over both shards, and a per-user exclusion CSR (seeded)."""
    rng = np.random.default_rng(5)
    queries = synth.catalog_rows_f32(11, 0, b, d)
    liked = [rng.choice(n, size=int(rng.integers(1, 9)), replace=False) for _ in range(b)]
    excl = [np.sort(rng.choice(n, size=int(rng.integers(0, 30)), replace=False)) for _ in range(b)]
    ptr = lambda segs: np.concatenate([[0], np.cumsum([len(x) for x in segs])]).astype(np.int64)
    lw = rng.uniform(0.5, 2.0, size=sum(len(x) for x in liked)).astype(np.float32)
    return queries, ptr(liked), np.concatenate(liked).astype(np.int32), lw, ptr(excl), np.concatenate(excl).astype(np.int32)


def _worker(rank, world, port, n, d, out_q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        plan = ShardPlan(n, world)
        row0, cnt = plan.range(rank)
        m_local = synth.catalog_rows_f32(0, row0, cnt, d, scale_rows=True).astype(np.float64)
        sc = ShardedCatalog(OracleShardBackend(m_local, row0), n)
        q = synth.query_f32(1, d)
        excl = np.random.default_rng(3).choice(n, size=40, replace=False)
        out = {"rank": rank}
        out["r1"] = sc.recommend(query=q, exclude_rows=excl, k=10)
        (rated, rts), = synth.user_ratings(2, n, 1, mean_rated=60)
        liked = rated[rts >= 3.5]
        out["r2"] = sc.recommend(liked_rows=liked, exclude_rows=rated, k=25)
        # k beyond the register-list kernel: sharded threshold bisection + sweep (query form, then profile form with
        # fewer allowed rows than k)
        out["r3"] = sc.recommend(query=q, exclude_rows=excl, k=300)
        out["r4"] = sc.recommend(liked_rows=liked, exclude_rows=np.setdiff1d(np.arange(n), np.arange(0, n, 11)), k=400)
        # fail closed: an unproven merged result is answered by the exhaustive sweep, or raises when that cannot decide
        out["r5"] = ShardedCatalog(UnprovenShardBackend(m_local, row0), n).recommend(query=q, exclude_rows=excl, k=10,
                                                                                      return_info=True)
        out["r6"] = ShardedCatalog(UnprovenShardBackend(m_local, row0), n).recommend(liked_rows=liked, exclude_rows=rated,
                                                                                      k=25, return_info=True)
        try:
            ShardedCatalog(OverflowShardBackend(m_local, row0), n).recommend(query=q, exclude_rows=excl, k=10)
            out["err"] = None
        except RuntimeError as e:
            out["err"] = str(e)
        # per-query re-run of a batch (what batch_collect and the small-shard loop use), for queries and a weighted liked
        # CSR, with exclusions; users 1 and 3 are left alone
        b, k = 5, 12
        queries, lp, lc, lw, ep, ec = _batch_inputs(n, d, b)
        for name, src in (("rq", (queries, None, None, None)), ("rp", (None, lp, lc, lw))):
            rows, scores, counts = np.full((b, k), -7, dtype=np.int64), np.zeros((b, k)), np.zeros(b, dtype=np.int32)
            sc._rerun([0, 2, 4], *src, ep, ec, k, None, False, rows, scores, counts)
            out[name] = (rows, scores, counts)
        out_q.put(out)
    finally:
        dist.destroy_process_group()


def test_two_rank_gloo_matches_unsharded_oracle():
    from oracle import reference_scoring as ora
    n, d, world = 3001, 48, 2
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    out_q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, n, d, out_q)) for r in range(world)]
    for p in procs:
        p.start()
    results = [out_q.get(timeout=120) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    m = synth.catalog_rows_f32(0, 0, n, d, scale_rows=True).astype(np.float64)
    q = synth.query_f32(1, d).astype(np.float64)
    excl = np.random.default_rng(3).choice(n, size=40, replace=False)
    want1 = ora.query_rows(m, q, excl, 10)
    (rated, rts), = synth.user_ratings(2, n, 1, mean_rated=60)
    want2 = ora.recommend_rows(m, rated[rts >= 3.5], rated, 25)
    want3 = ora.query_rows(m, q, excl, 300)
    allowed4 = np.arange(0, n, 11)
    want4 = ora.recommend_rows(m, rated[rts >= 3.5], np.setdiff1d(np.arange(n), allowed4), 400)
    assert len(want3[0]) == 300 and len(want4[0]) == len(allowed4) < 400
    for res in results:
        rank = res["rank"]
        for key, want in (("r1", want1), ("r2", want2), ("r3", want3), ("r4", want4)):
            assert res[key][0].tolist() == want[0].tolist(), (rank, key)
            np.testing.assert_allclose(res[key][1], want[1], rtol=1e-12)
        for key, want in (("r5", want1), ("r6", want2)):
            rows, scores, info = res[key]
            assert rows.tolist() == want[0].tolist(), (rank, key)
            np.testing.assert_allclose(scores, want[1], rtol=1e-12)
            assert info["kc"] == 256 and info["proven_exact"] and info["exact_sweep"], (rank, key, info)
        assert res["err"] is not None and "cannot be proven exact" in res["err"] and "overflow" in res["err"], (rank, res["err"])
        b, k = 5, 12
        queries, lp, lc, lw, ep, ec = _batch_inputs(n, d, b)
        for key in ("rq", "rp"):
            rows, scores, counts = res[key]
            for u in range(b):
                if u in (1, 3):
                    assert (rows[u] == -7).all() and counts[u] == 0, (rank, key, u)
                    continue
                ex = ec[ep[u]:ep[u + 1]]
                if key == "rq":
                    want = ora.query_rows(m, queries[u].astype(np.float64), ex, k)
                else:
                    want = ora.recommend_rows(m, lc[lp[u]:lp[u + 1]], ex, k, weights=lw[lp[u]:lp[u + 1]])
                assert counts[u] == k and rows[u].tolist() == want[0].tolist(), (rank, key, u)
                np.testing.assert_allclose(scores[u], want[1], rtol=1e-12)


def _fast_exact(n, noise, seed, ties=False):
    """Exact scores and a simulated fast pass within `noise` of them (test_large_k_search.py), as numpy count / sweep."""
    rng = np.random.default_rng(seed)
    exact = rng.uniform(-1.0, 1.0, size=n)
    if ties:
        exact = np.round(exact, 2)
    fast = exact + rng.uniform(-noise, noise, size=n)
    rows = np.arange(n, dtype=np.int64)
    calls = {"count": 0, "sweep": []}

    def count(thr):
        calls["count"] += 1
        return int(np.count_nonzero(fast >= thr))

    def sweep(thr):
        calls["sweep"].append(thr)
        sel = fast >= thr
        return rows[sel], exact[sel]

    return exact, fast, rows, count, sweep, calls


def test_close_proof_routes():
    eps = 2e-4
    exact, fast, rows, count, sweep, calls = _fast_exact(4000, eps / 2, seed=7, ties=True)
    k = 50
    cand = np.argsort(-fast, kind="stable")[:k]                            # an unproven candidate list of the fast pass
    cand = cand[np.lexsort((cand, -exact[cand]))]
    order = np.lexsort((rows, -exact))[:k]
    # the sweep at the k-th exact score - 2 eps answers: no bisection
    got = close_proof(rows[cand], exact[cand], k, eps, 0.0, count, sweep)
    np.testing.assert_array_equal(got[0], rows[order])
    np.testing.assert_array_equal(got[1], exact[order])
    assert calls["count"] == 0 and calls["sweep"] == [exact[cand[-1]] - 2 * eps]
    # that sweep overflows: the bisection answers
    first = [True]

    def sweep_once_overflowing(thr):
        if first[0]:
            first[0] = False
            return None
        return sweep(thr)

    got = close_proof(rows[cand], exact[cand], k, eps, 0.0, count, sweep_once_overflowing)
    np.testing.assert_array_equal(got[0], rows[order])
    np.testing.assert_array_equal(got[1], exact[order])
    assert calls["count"] > 0
    # every sweep overflows: RuntimeError, with the cause
    with pytest.raises(RuntimeError, match="cannot be proven exact") as ei:
        close_proof(rows[cand], exact[cand], k, eps, 0.0, count, lambda thr: None)
    assert "overflow" in str(ei.value) and isinstance(ei.value.__cause__, RuntimeError)
    # fewer rows than k (fewer allowed rows than k): straight to the bisection route, which returns every row
    exact, fast, rows, count, sweep, calls = _fast_exact(300, eps / 2, seed=8)
    k = 500
    cand = np.lexsort((rows, -exact))[:290]
    got = close_proof(rows[cand], exact[cand], k, eps, 0.0, count, sweep)
    order = np.lexsort((rows, -exact))
    np.testing.assert_array_equal(got[0], rows[order])
    np.testing.assert_array_equal(got[1], exact[order])
    assert calls["count"] == 1 and calls["sweep"] == [-2.0]


def test_widen_until_proven():
    def run(margins):
        seen = []

        def attempt(kc):
            seen.append(kc)
            return np.arange(3), np.zeros(3), margins[len(seen) - 1]

        return widen_until_proven(attempt, 32, 1e-6)[2:], seen

    assert run([1.0]) == ((1.0, 32), [32])
    assert run([0.0, 1e-6, 1.0]) == ((1.0, 256), [32, 128, 256])
    assert run([0.0, 0.0, 0.0]) == ((0.0, 256), [32, 128, 256])          # 256 candidates: the caller takes over
