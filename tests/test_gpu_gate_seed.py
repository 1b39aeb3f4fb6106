"""The gate's seed kernel (DESIGN.md §4.5) writes a lower bound of the final kc-th best fast score into the grid-wide hint
before the gated kernel starts.  For every case the bound it wrote (workspace control word 21) must not exceed the plain
pass's kc-th candidate key, and the packed request result and the candidate keys must equal the plain pass bit for bit.
"""
import numpy as np
import pytest
import torch

from robot_ebert_b200 import CatalogStore, RowFilter, synth
from robot_ebert_b200 import _native as nat

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
CTL_SEED_BOUND = 21


def seed_rows(n):
    """Rows i * (n // m), i < m, are sampled (gemv_topk.cu: seed_rows)."""
    m = min(max(n // 64, 16384), 131072)
    m = min(m, n)
    return np.arange(m, dtype=np.int64) * (n // m)


def seed_word(store):
    ws = store._scratch().ws
    off = (-ws.data_ptr()) % 128
    return int(ws[off:off + 128].cpu().numpy().view(np.uint32)[CTL_SEED_BOUND])


def run(store, k, query=None, liked=None, excl=None, row_filter=None, q_scale=None):
    """(packed request result, candidate keys, seed word of each launch) for one request."""
    kc = nat.load().rebert_candidates_for_k(k)
    excl_ptr, ne = store.stage_inputs(query, liked, None, excl, k, kc)
    s = store._scratch()
    if q_scale is not None:
        s.qn32.mul_(q_scale)
    packed = store.enqueue_fused(k, kc, excl_ptr, ne, row_filter).cpu().numpy().copy()
    w_fused = seed_word(store)
    store.enqueue_topk(k, kc, excl_ptr, ne, row_filter)
    keys = s.cand.cpu().numpy().copy().view(np.uint64)
    return packed, keys, (w_fused, seed_word(store))


def check(store, k, expect_bound=True, **kw):
    """Gated vs plain, bit for bit; the seed's bound <= the plain kc-th key.  expect_bound: whether a bound must (True) or
    must not (False) have been written, None = either.  Returns the bound's score (None: no bound)."""
    kc = nat.load().rebert_candidates_for_k(k)
    run(store, k, **kw)                                  # sizes the scratch
    assert store.build_gate()
    a = run(store, k, **kw)
    store.drop_gate()
    b = run(store, k, **kw)
    assert store.build_gate()
    assert np.array_equal(a[0], b[0]), ("packed result differs", a[0], b[0])
    assert np.array_equal(a[1], b[1]), "candidate keys differ"
    assert a[2][0] == a[2][1], "the two entry points seeded different bounds"
    w = a[2][0]
    kth = int(b[1][kc - 1])                               # 0 when the plain list is not full
    if expect_bound is not None:
        assert (w != 0) == expect_bound, ("bound seeded" if w else "no bound seeded", expect_bound)
    if w:
        assert kth != 0 and w <= kth >> 32, (w, kth >> 32)
        return float(np.array([w ^ (0x80000000 if w & 0x80000000 else 0xFFFFFFFF)], dtype=np.uint32).view(np.float32)[0])
    return None


_STORES = {}


def store_for(dtype, d, n=40_000):
    key = (dtype, d, n)
    if key not in _STORES:
        _STORES.clear()
        torch.cuda.empty_cache()
        _STORES[key] = CatalogStore.synthetic(0, n, d, dtype, scale_rows=True, device=DEV)
    return _STORES[key]


@pytest.mark.parametrize("k", [1, 10, 240])
@pytest.mark.parametrize("d,dtype", [(1536, "bf16"), (700, "fp32"), (3000, "bf16")])
def test_seeded_request_is_the_plain_request(dtype, d, k):
    st = store_for(dtype, d)
    excl = np.random.default_rng(1).choice(st.n, size=133, replace=False)
    check(st, k, query=synth.query_f32(1, d), excl=excl)


def test_exclusion_list_covers_most_sampled_rows():
    st = store_for("bf16", 1536)
    s = seed_rows(st.n)
    keep = np.random.default_rng(2).choice(s.size, size=300, replace=False)
    excl = np.setdiff1d(s, s[keep])                       # 16k of the sampled rows excluded, 300 left
    for k in (10, 100):
        check(st, k, query=synth.query_f32(3, 1536), excl=excl)


def test_filters_reject_most_sampled_rows():
    st = store_for("bf16", 1536)
    g, y = synth.movie_metadata(3, 0, st.n)
    g = g.copy()
    y = y.copy()
    s = seed_rows(st.n)
    g[s] = 0                                              # no genre on any sampled row ...
    g[s[::50]] = 0b1                                      # ... but a fiftieth of them
    st.set_metadata(g, y)
    bits = np.zeros((st.n + 31) // 32, dtype=np.uint32)
    bits[::4] = 0x55555555                                # excludes a quarter of the words' even rows
    bm = torch.from_numpy(bits.view(np.int32)).to(DEV)
    rf = RowFilter(genre_any=0b1011, year_lo=1950, year_hi=2010, exclude_bitmap=bm)
    for k in (10, 100):
        check(st, k, expect_bound=None, query=synth.query_f32(4, 1536), excl=np.arange(0, st.n, 7), row_filter=rf)


def test_fewer_than_kc_allowed_sampled_rows_write_no_bound():
    """Sample i goes to warp i % (8 warps x grid), so samples 8 j (j < 148) go to warp 0 of CTA j: one allowed row per
    CTA, which every CTA publishes."""
    st = store_for("bf16", 1536)
    s = seed_rows(st.n)
    for k, kc in ((10, 32), (100, 128)):
        excl = np.setdiff1d(s, s[8 * np.arange(kc - 1)])   # kc - 1 sampled rows stay allowed: no bound
        check(st, k, expect_bound=False, query=synth.query_f32(5, 1536), excl=excl)
        excl = np.setdiff1d(s, s[8 * np.arange(kc)])       # kc rows: a bound
        check(st, k, query=synth.query_f32(5, 1536), excl=excl)


@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
def test_integer_catalog_ties_at_the_kth_score(dtype):
    """Small-integer rows and query: every fp32 dot is exact, and 40 copies of each of the best rows sit on sampled rows,
    so the seed's kc-th score ties exactly with the final kc-th score."""
    rng = np.random.default_rng(5)
    d, n = 700, 40_000
    base = rng.integers(-8, 9, size=(500, d)).astype(np.float32)
    m = base[rng.integers(0, 500, size=n)]
    q = rng.integers(-4, 5, size=d).astype(np.float32)
    top = np.argsort(-(base @ q) / np.linalg.norm(base, axis=1))[:8]
    s = seed_rows(n)
    m[s[:320]] = base[np.repeat(top, 40)]
    st = CatalogStore.from_host(None, m, dtype, device=DEV)
    for k in (10, 100, 240):
        check(st, k, query=q, excl=np.arange(1, n, 11))


@pytest.mark.parametrize("q_scale", [7.5, 1e-3])
def test_non_unit_queries(q_scale):
    st = store_for("bf16", 1536)
    check(st, 10, query=synth.query_f32(2, 1536), q_scale=q_scale)


def test_profile_request():
    st = store_for("fp32", 1536)
    (rated, rts), = synth.user_ratings(2, st.n, 1)
    check(st, 10, liked=rated[rts >= 3.5], excl=rated)
