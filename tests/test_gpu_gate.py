"""The int8 gate of the single-query fast pass (DESIGN.md §4.5) changes which rows are read, never the result.

For every case the packed output of the request path (enqueue_fused: rows, scores, count, margin) and the candidate keys
of rebert_gemv_topk are compared between the same store with its gate and without it, bit for bit, and the fetch
counter shows that the gated kernel ran.
"""
import numpy as np
import pytest
import torch

from robot_ebert_b200 import CatalogStore, RowFilter, synth
from robot_ebert_b200 import _native as nat

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
# d of every gated int8 layout: 32 lanes x 1, 2, 3, 4, 6 chunks per lane
GATED_D = (300, 700, 1536, 2000, 3000)


def fetches(store):
    return store.gate_fetches()


def run(store, k, query=None, liked=None, excl=None, row_filter=None, q_scale=None):
    """(packed request result, rebert_gemv_topk keys) for one request."""
    kc = nat.load().rebert_candidates_for_k(k)
    excl_ptr, ne = store.stage_inputs(query, liked, None, excl, k, kc)
    s = store._scratch()
    if q_scale is not None:                             # a non-unit query straight into the kernels
        s.qn32.mul_(q_scale)
    packed = store.enqueue_fused(k, kc, excl_ptr, ne, row_filter).cpu().numpy().copy()
    store.enqueue_topk(k, kc, excl_ptr, ne, row_filter)
    keys = s.cand.cpu().numpy().copy()
    return packed, keys


def gated_equals_plain(store, k, expect_fetch=True, **kw):
    store._scratch().ensure_out(k, nat.load().rebert_candidates_for_k(k))   # the counter lives in this workspace
    assert store.build_gate()
    f0 = fetches(store)
    a = run(store, k, **kw)
    nf = fetches(store) - f0
    store.drop_gate()
    b = run(store, k, **kw)
    assert store.build_gate()
    assert np.array_equal(a[0], b[0]), ("packed result differs", a[0], b[0])
    assert np.array_equal(a[1], b[1]), "candidate keys differ"
    if expect_fetch:
        assert nf > 0, "the gated kernel did not run"
    return a[0], nf


_STORES = {}


def store_for(dtype, d, n=40_000):
    key = (dtype, d, n)
    if key not in _STORES:
        _STORES.clear()
        torch.cuda.empty_cache()
        _STORES[key] = CatalogStore.synthetic(0, n, d, dtype, scale_rows=True, device=DEV)
    return _STORES[key]


@pytest.mark.parametrize("k", [1, 10, 100, 240])
@pytest.mark.parametrize("d", GATED_D)
@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
def test_gated_request_is_the_plain_request_bit_for_bit(dtype, d, k):
    st = store_for(dtype, d)
    assert st.gate_layout_ok
    excl = np.random.default_rng(1).choice(st.n, size=133, replace=False)
    run(st, k, query=synth.query_f32(1, d))            # sizes the scratch, so the fetch counter can be read before
    gated_equals_plain(st, k, query=synth.query_f32(1, d), excl=excl)


@pytest.mark.parametrize("q_scale", [7.5, 1e-3])
def test_non_unit_queries(q_scale):
    st = store_for("bf16", 1536)
    run(st, 10, query=synth.query_f32(2, 1536))
    gated_equals_plain(st, 10, query=synth.query_f32(2, 1536), q_scale=q_scale)


def test_bitmap_and_genre_year_filters():
    st = store_for("bf16", 1536)
    g, y = synth.movie_metadata(3, 0, st.n)
    st.set_metadata(g, y)
    bits = np.zeros((st.n + 31) // 32, dtype=np.uint32)
    bits[::3] = 0xF0F0F0F0
    bm = torch.from_numpy(bits.view(np.int32)).to(DEV)
    rf = RowFilter(genre_any=0b1011, year_lo=1960, year_hi=2000, exclude_bitmap=bm)
    q = synth.query_f32(4, 1536)
    run(st, 100, query=q)
    for k in (10, 100):
        gated_equals_plain(st, k, query=q, excl=np.arange(0, st.n, 7), row_filter=rf)


def test_profile_request():
    st = store_for("fp32", 1536)
    (rated, rts), = synth.user_ratings(2, st.n, 1)
    run(st, 10, query=synth.query_f32(1, 1536))
    gated_equals_plain(st, 10, liked=rated[rts >= 3.5], excl=rated)


@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
def test_integer_catalog_with_exact_ties(dtype):
    """Small-integer rows and query: every fp32 dot is exact, duplicates and power-of-two copies tie exactly."""
    rng = np.random.default_rng(5)
    d, n = 700, 30_000
    base = rng.integers(-8, 9, size=(500, d)).astype(np.float32)
    m = base[rng.integers(0, 500, size=n)] * (2.0 ** rng.integers(-2, 3, size=(n, 1))).astype(np.float32)
    st = CatalogStore.from_host(None, m, dtype, device=DEV)
    q = rng.integers(-4, 5, size=d).astype(np.float32)
    run(st, 240, query=q)
    for k in (10, 100, 240):
        gated_equals_plain(st, k, query=q, excl=np.arange(0, n, 11))


def test_dominant_column_passes_most_rows():
    """One column dominates every row: the int8 rows lose the rest, delta is large and most rows are fetched."""
    rng = np.random.default_rng(6)
    d, n = 1536, 20_000
    m = rng.standard_normal((n, d)).astype(np.float32)
    m[:, 0] += 80.0
    st = CatalogStore.from_host(None, m, "bf16", device=DEV)
    q = rng.standard_normal(d).astype(np.float32)
    run(st, 10, query=q)
    _, nf = gated_equals_plain(st, 10, query=q)
    assert nf > n // 2


def test_under_full_list():
    """Fewer allowed rows than candidates: the lists never fill, the bound stays -inf, every allowed row is fetched."""
    st = CatalogStore.synthetic(1, 300, 1536, "bf16", device=DEV)
    q = synth.query_f32(1, 1536)
    run(st, 100, query=q)
    packed, nf = gated_equals_plain(st, 100, query=q, excl=np.arange(0, 300, 2))
    assert int(packed[200:201].view(np.int32)[0]) == 100
    empty, _ = gated_equals_plain(st, 10, query=q, excl=np.arange(300), expect_fetch=False)
    assert int(empty[20:21].view(np.int32)[0]) == 0


def test_in_place_row_write_rebuilds_the_gate():
    """A row written after the first request (the planted-row pattern of test_gpu_fullsize) must be found: the store
    re-quantizes its gate when rows / inv_norm / norm64 changed."""
    st = CatalogStore.synthetic(2, 50_000, 1536, "bf16", device=DEV)
    assert st.build_gate()
    q = synth.query_f32(3, 1536)
    r0, _ = st.recommend(query=q, k=10)
    plant = 31_337
    assert plant not in r0
    st.rows[plant, :1536] = torch.from_numpy(q).to(DEV, torch.bfloat16)
    lib = nat.load()
    nat.check(lib.rebert_catalog_norms(st.rows.data_ptr(), st.n, st.ld, nat.DTYPES["bf16"], st.inv_norm.data_ptr(),
                                       st.norm64.data_ptr(), torch.cuda.current_stream().cuda_stream))
    r1, _ = st.recommend(query=q, k=10)
    assert r1[0] == plant
    gated_equals_plain(st, 10, query=q)


def test_fetches_stay_below_one_percent_at_10M():
    st = CatalogStore.synthetic(0, 10_000_000, 1536, "bf16", device=DEV)
    assert st.has_gate                                  # built by the constructor: its probe request fetched few rows
    q = synth.query_f32(1, 1536)
    excl = np.random.default_rng(1).choice(st.n, size=133, replace=False)
    st._scratch().ensure_out(10, 32)
    f0 = fetches(st)
    run(st, 10, query=q, excl=excl)
    nf = fetches(st) - f0
    assert 0 < nf < 2 * st.n // 100                     # two launches: enqueue_fused + enqueue_topk


def test_crowded_catalog_keeps_the_plain_pass():
    """Rows around a shared mean direction (pairwise cosine ~0.7): a quarter of the rows pass the gate, which would make
    requests slower, so the constructor's probe leaves the catalog without one."""
    rng = np.random.default_rng(8)
    n, d = 1_500_000, 1536
    m = rng.standard_normal(d).astype(np.float32)
    m /= np.linalg.norm(m)
    rows = torch.empty((n, d), dtype=torch.float32, device=DEV)
    g = torch.Generator(device=DEV).manual_seed(8)
    for s in range(0, n, 1 << 18):
        e = min(n, s + (1 << 18))
        rows[s:e] = np.sqrt(0.7) * torch.from_numpy(m).to(DEV) + np.sqrt(0.3) * torch.randn((e - s, d), generator=g, device=DEV) / np.sqrt(d)
    ld, _ = CatalogStore.layout(n, d, "fp32")
    inv = torch.empty(n, dtype=torch.float32, device=DEV)
    n64 = torch.empty(n, dtype=torch.float64, device=DEV)
    lib = nat.load()
    nat.check(lib.rebert_catalog_norms(rows.data_ptr(), n, ld, nat.DTYPES["fp32"], inv.data_ptr(), n64.data_ptr(),
                                       torch.cuda.current_stream().cuda_stream))
    st = CatalogStore(rows, inv, n64, n, d, ld, "fp32")
    assert not st.has_gate and st.last_probe_fetches > n // 20
