"""The batched tensor-core path for long lists (241 <= k <= 2048) against float64 on the host.

Same comparison as tests/test_gpu_batched_edges.py (its oracle helpers are reused): ids exact save the oracle's own
float64 noise on mathematically tied rows, scores to 1e-9.  Every batched case asserts that a plan was made and bounds
the fraction of queries the batched pass could not prove (status != 0), since the widened retry and the per-query route
behind it would hide a kernel bug.
"""
import numpy as np
import pytest
import torch

from oracle import reference_scoring as ora
from robot_ebert_b200 import CatalogStore, RowFilter, synth
from robot_ebert_b200.batcher import RatingsBatcher, recommend_all
from tests.test_gpu_batched_edges import (KX, _assert_matches_oracle, _check_against, _excl_csr, _liked_csr, _oracle_profile_topk,
                                          _oracle_query_topk, _queries, _status_fraction, _stored_f64)

pytestmark = pytest.mark.gpu

# status != 0 bounds, set from a B200 run (NVIDIA B200, 1000 W power limit); see the module docstring
STATUS_MAX_BF16 = 0.02
STATUS_MAX_INT8 = 0.03

# (k, b, n): n above both plans' minimum (64 x max(3 kc, 3200): bf16 204,800 up to k = 1000 at kc <= 1066, 245,760 at
# k = 1000, 491,520 at k = 2048; int8 204,800 up to k = 500, 387,072 at k = 1000, 786,432 at k = 2048), not a multiple of 256.
# d = 128 keeps the host oracle at n * d * b <= 1.4e10.
GRID = [
    (241, 129, 250_001),
    (500, 128, 250_001),
    (1000, 129, 400_003),
    (2048, 130, 800_011),
]
D = 128


@pytest.fixture(scope="module")
def stores():
    cache = {}

    def get(n):
        if n not in cache:
            cache.clear()
            store = CatalogStore.synthetic(0, n, D, "bf16", scale_rows=True)
            store.enable_prefilter()
            assert store.batch_shadow_ok and store.batch_gemm_ok
            cache[n] = (store, ora._normalize_rows(_stored_f64(store)))
        return cache[n]
    return get


@pytest.mark.parametrize("k,b,n", GRID)
def test_recommend_batch_long_lists_vs_oracle(stores, k, b, n):
    store, unit = stores(n)
    rng = np.random.default_rng(k + b)
    ep, ec, excl = _excl_csr(rng, n, b, max_len=200)
    q = _queries(b, D, seed=k)
    lp, lc, lw, liked, ws = _liked_csr(rng, n, b)
    runs = [("queries", dict(queries=q), _oracle_query_topk(unit, q, k, excl)),
            ("profiles", dict(liked_ptr=lp, liked_col=lc, liked_w=lw),
             _oracle_profile_topk(unit, liked, [w.astype(np.float64) for w in ws], k, excl))]
    for what, src, want in runs:
        rb, sb, cb, ib = store.recommend_batch(**src, excl_ptr=ep, excl_col=ec, k=k, return_info=True, prefilter=False)
        assert ib["plan"] is not None and ib["plan"]["sample_rank"] == 64 and not ib["int8_operands"]
        assert _status_fraction(ib, f"bf16 {what} b={b} k={k} n={n}") < STATUS_MAX_BF16
        _check_against(want, rb, sb, cb, ib, k, f"bf16 {what} k={k}")
        r8, s8, c8, i8 = store.recommend_batch(**src, excl_ptr=ep, excl_col=ec, k=k, return_info=True, prefilter=True)
        assert i8["plan"] is not None and i8["int8_operands"]
        assert _status_fraction(i8, f"int8 {what} b={b} k={k} n={n}") < STATUS_MAX_INT8
        np.testing.assert_array_equal(r8, rb)
        np.testing.assert_array_equal(s8, sb)                     # same exact pass on the same rows: same bits
        np.testing.assert_array_equal(c8, cb)


def test_k241_extends_the_k240_path(stores):
    """The first 240 entries of a k = 241 call (long-list kernels) equal the k = 240 call (the k <= 240 kernels)."""
    n, b = 250_001, 129
    store, _ = stores(n)
    rng = np.random.default_rng(5)
    ep, ec, _ = _excl_csr(rng, n, b, max_len=200)
    q = _queries(b, D, seed=5)
    r0, s0, c0, i0 = store.recommend_batch(queries=q, excl_ptr=ep, excl_col=ec, k=240, return_info=True, prefilter=False)
    r1, s1, c1, i1 = store.recommend_batch(queries=q, excl_ptr=ep, excl_col=ec, k=241, return_info=True, prefilter=False)
    assert i0["plan"]["sample_rank"] == 16 and i1["plan"]["sample_rank"] == 64
    np.testing.assert_array_equal(r1[:, :240], r0)
    both = (np.asarray(i0["status"]) == 0) & (np.asarray(i1["status"]) == 0)
    assert both.mean() > 0.9
    np.testing.assert_array_equal(s1[both, :240], s0[both])
    np.testing.assert_array_equal(np.minimum(c1, 240), c0)


def test_exact_duplicates_at_k1000_come_back_in_row_order():
    """Five rows, each copied 150 times over the catalog, near the queries: the copies tie exactly and must come back in
    ascending row order from the long-list exact pass."""
    n, d, b, k = 250_003, 64, 40, 1000
    rng = np.random.default_rng(11)
    m = rng.standard_normal((n, d)).astype(np.float32)
    srcs = rng.choice(n, size=5, replace=False)
    for s in srcs:
        m[rng.choice(n, size=150, replace=False)] = m[s]
    store = CatalogStore.from_host(None, m, "bf16")
    ms = _stored_f64(store)
    q = (ms[srcs[np.arange(b) % 5]] + 0.3 * rng.standard_normal((b, d))).astype(np.float32)
    ep, ec, excl = _excl_csr(rng, n, b, max_len=50)
    rows, scores, counts, info = store.recommend_batch(queries=q, excl_ptr=ep, excl_col=ec, k=k, return_info=True)
    assert info["plan"] is not None
    assert _status_fraction(info, "duplicates k=1000") < STATUS_MAX_BF16 * 3
    unit = ora._normalize_rows(ms)
    want = _oracle_query_topk(unit, q, k, excl)
    _check_against(want, rows, scores, counts, info, k, "duplicates")
    for u in range(b):
        sc = scores[u, :counts[u]]
        tied = np.nonzero(np.diff(sc) == 0)[0]
        assert len(tied) > 100, u                                  # the copies did reach the top-k
        assert (np.diff(rows[u, :counts[u]])[tied] > 0).all(), u


def test_row_filter_leaving_fewer_than_k_rows(stores):
    n, b, k = 250_001, 129, 500
    store, unit = stores(n)
    year = np.full(n, 1950, dtype=np.uint16)
    allowed = np.random.default_rng(2).choice(n, size=300, replace=False)
    year[allowed] = 2001
    store.set_metadata(np.ones(n, dtype=np.uint32), year)
    try:
        q = _queries(b, D, seed=9)
        ep, ec, excl = _excl_csr(np.random.default_rng(3), n, b, max_len=40)
        rows, scores, counts, info = store.recommend_batch(queries=q, excl_ptr=ep, excl_col=ec, k=k, return_info=True,
                                                           row_filter=RowFilter(year_lo=2000, year_hi=2010), prefilter=False)
        assert info["plan"] is not None
        keep = np.zeros(n, dtype=bool)
        keep[allowed] = True
        qn = q.astype(np.float64) / np.linalg.norm(q.astype(np.float64), axis=1, keepdims=True)
        sc = qn @ unit.T
        for u in range(b):
            n_ok = int(keep.sum() - np.isin(excl[u], allowed).sum())
            assert counts[u] == n_ok
            assert (rows[u, n_ok:] == -1).all() and np.isneginf(scores[u, n_ok:]).all()
            wr, ws = ora.topk_rows(sc[u], k + KX, excl[u], keep_mask=keep)
            _assert_matches_oracle(rows[u, :n_ok], scores[u, :n_ok], wr, ws, k, f"filter query {u}")
    finally:
        store.genre_bits = store.year = None


def test_catalog_below_the_plan_minimum_is_served_by_the_loop():
    n, b, k = 150_001, 6, 500
    store = CatalogStore.synthetic(0, n, D, "bf16", scale_rows=True)
    unit = ora._normalize_rows(_stored_f64(store))
    rng = np.random.default_rng(4)
    ep, ec, excl = _excl_csr(rng, n, b, max_len=100)
    q = _queries(b, D, seed=4)
    rows, scores, counts, info = store.recommend_batch(queries=q, excl_ptr=ep, excl_col=ec, k=k, return_info=True)
    assert info["plan"] is None and info["per_query"] == b
    _check_against(_oracle_query_topk(unit, q, k, excl), rows, scores, counts, info, k, "loop k=500")


def test_k3000_goes_through_the_per_query_route(stores):
    n, b, k = 250_001, 3, 3000
    store, unit = stores(n)
    rng = np.random.default_rng(6)
    ep, ec, excl = _excl_csr(rng, n, b, max_len=100)
    q = _queries(b, D, seed=6)
    rows, scores, counts, info = store.recommend_batch(queries=q, excl_ptr=ep, excl_col=ec, k=k, return_info=True)
    assert info["plan"] is None and info["per_query"] == b
    _check_against(_oracle_query_topk(unit, q, k, excl), rows, scores, counts, info, k, "k=3000")
    with pytest.raises(ValueError, match="too large"):
        store.recommend_batch(queries=q, k=40_000)


def test_recommend_all_k500_vs_oracle():
    n, k = 250_001, 500
    m = synth.catalog_rows_f32(0, 0, n, D, scale_rows=True)
    store = CatalogStore.from_host(synth.row_ids(n), m, "bf16")
    ms = _stored_f64(store)
    batcher = RatingsBatcher(store)
    users = synth.user_ratings(4, n, 160)
    for i, (rated, rts) in enumerate(users):
        batcher.add_user(f"u{i}", [(store.id_of(int(r)), float(x)) for r, x in zip(rated, rts)])
    assert len(batcher) > 129
    recs = recommend_all(store, batcher, k=k)
    unit = ora._normalize_rows(ms)
    for i, (rated, rts) in enumerate(users):
        if f"u{i}" not in batcher.users:
            continue
        liked = rated[rts >= 3.5]
        wr, ws = ora.topk_rows((unit[liked] @ unit.T).mean(axis=0), k + KX, rated)
        got = np.array([store.row_of(t) for t, _ in recs[f"u{i}"]])
        _assert_matches_oracle(got, np.array([x for _, x in recs[f"u{i}"]]), wr, ws, k, f"user {i}")
