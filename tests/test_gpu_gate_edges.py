"""The int8 gate of the single-query fast pass (DESIGN.md §4.5) at its edges: the seed's bound where it meets the final
kc-th score exactly, row shards (row_base != 0), the public request path (recommend(): proof loop, exact sweep, prefilter,
CPython side door and ctypes), back-to-back requests of different kc on one workspace, concurrent threads, and Python's
gate decision against the library's.

Gated requests are compared with the same store after drop_gate(): packed result (rows, fp64 score bits, count, margin)
and candidate keys bit for bit; and, where the request path is the public one, with the float64 oracle.
"""
import ctypes as C
import threading

import numpy as np
import pytest
import torch

from oracle import reference_scoring as ora
from robot_ebert_b200 import CatalogStore, RowFilter, synth
from robot_ebert_b200 import _native as nat
from robot_ebert_b200.catalog import unpack_result

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
CTL_SEED_BOUND = 21
SCORE_RTOL = 1e-9
GATED_D = (300, 700, 1536, 2000, 3000)          # int8 rows of 1, 2, 3, 4, 6 chunks per lane: every gated kernel


# ------------------------------------------------------------------ helpers ---------------------------------------------
def seed_rows(n):
    """Rows i * (n // m), i < m, are sampled (gemv_topk.cu: seed_rows)."""
    m = min(max(n // 64, 16384), 131072)
    m = min(m, n)
    return np.arange(m, dtype=np.int64) * (n // m)


def seed_cta(i, sms):
    """The CTA of gate_seed_kernel that scores sample i: warp w of CTA c takes samples c * 8 + w + t * (8 * grid)."""
    w = sms * 8
    return (np.asarray(i) % w) // 8


def num_sms():
    return torch.cuda.get_device_properties(DEV).multi_processor_count


def seed_word(ws):
    off = (-ws.data_ptr()) % 128
    return int(ws[off:off + 128].cpu().numpy().view(np.uint32)[CTL_SEED_BOUND])


def fetch_count(ws):
    """The gate-fetch control word of a workspace (a request scratch's, or the device block of a host scratch)."""
    out = C.c_uint32(0)
    nat.check(nat.load().rebert_gate_fetches(ws.data_ptr(), ws.numel(), C.byref(out), torch.cuda.current_stream().cuda_stream))
    return out.value


def host_fetches(store):
    """Fetch count of the calling thread's rebert_recommend_host scratch.  The gemv workspace is the first region of that
    scratch's device block (csrc/host_api.cu, host_layout: off_ws = 0, placed first so its control words are the ones
    zero-filled once); the library exports no offset for it, so a change of that layout has to be mirrored here."""
    s = store._scratch()
    return fetch_count(s.hdev) if hasattr(s, "hdev") else 0


def key_rows(keys):
    return (0xFFFFFFFF - (keys.astype(np.uint64) & np.uint64(0xFFFFFFFF))).astype(np.int64)


def run(store, k, query=None, liked=None, excl=None, row_filter=None, q_scale=None, q_raw=None):
    """(packed request result, candidate keys, seed word of each launch) for one request.  q_raw: the fast pass gets this
    fp32 query as it is (not normalised; the exact pass keeps the normalised one)."""
    kc = nat.load().rebert_candidates_for_k(k)
    excl_ptr, ne = store.stage_inputs(query, liked, None, excl, k, kc)
    s = store._scratch()
    if q_scale is not None:
        s.qn32.mul_(q_scale)
    if q_raw is not None:
        s.qn32.zero_()
        s.qn32[:len(q_raw)] = torch.from_numpy(np.asarray(q_raw, dtype=np.float32)).to(s.qn32.device)
    packed = store.enqueue_fused(k, kc, excl_ptr, ne, row_filter).cpu().numpy().copy()
    w_fused = seed_word(s.ws)
    store.enqueue_topk(k, kc, excl_ptr, ne, row_filter)
    keys = s.cand.cpu().numpy().copy().view(np.uint64)
    return packed, keys, (w_fused, seed_word(s.ws))


def check(store, k, **kw):
    """Gated vs plain, bit for bit.  Returns (seed word, plain candidate keys, packed result)."""
    run(store, k, **kw)                                   # sizes the scratch
    assert store.build_gate()
    a = run(store, k, **kw)
    store.drop_gate()
    b = run(store, k, **kw)
    assert store.build_gate()
    assert np.array_equal(a[0], b[0]), ("packed result differs", a[0], b[0])
    assert np.array_equal(a[1], b[1]), "candidate keys differ"
    assert a[2][0] == a[2][1], "the two entry points seeded different bounds"
    return a[2][0], b[1], b[0]


def write_rows(store, dst, src=None, values=None):
    """Overwrite rows dst (local) with rows src of the store, or with fp32 values, and recompute the norms."""
    idx = torch.as_tensor(np.asarray(dst, dtype=np.int64), device=DEV)
    if src is not None:
        store.rows[idx] = store.rows[torch.as_tensor(np.asarray(src, dtype=np.int64), device=DEV)]
    else:
        store.rows[idx, :store.d] = torch.from_numpy(np.asarray(values, dtype=np.float32)).to(DEV, store.rows.dtype)
    lib = nat.load()
    nat.check(lib.rebert_catalog_norms(store.rows.data_ptr(), store.n, store.ld, nat.DTYPES[store.dtype], store.inv_norm.data_ptr(),
                                       store.norm64.data_ptr(), torch.cuda.current_stream().cuda_stream))
    torch.cuda.current_stream().synchronize()


def plant(store, rows, q, seed):
    """Rows q + 0.5 * noise (cosine ~0.89 to q, distinct, non-integer) on the given local rows."""
    noise = np.random.default_rng(seed).standard_normal((len(rows), store.d)).astype(np.float32)
    write_rows(store, rows, values=q[None, :] + 0.5 * np.linalg.norm(q) / np.sqrt(store.d) * noise)


def stored(store):
    """The catalog's stored values (exact in fp32 for bf16 and fp32 rows); the oracle upcasts them chunk by chunk."""
    return store.rows[:store.n, :store.d].float().cpu().numpy()


def oracle_check(store, packed, k, q=None, liked=None, excl=None, keep=None):
    """A packed result of a (possibly row-shard) store against the float64 oracle on the shard's rows: ids exact, scores
    to 1e-9 relative.  excl: global ids; liked: local rows."""
    base = store.row_base
    ex = None
    if excl is not None:
        ex = np.asarray(excl, dtype=np.int64)
        ex = ex[(ex >= base) & (ex < base + store.n)] - base
    m = stored(store)
    if q is not None:
        want_rows, want_scores = ora.query_rows(m, np.asarray(q, dtype=np.float64), ex, k, keep)
    else:
        want_rows, want_scores = ora.recommend_rows(m, liked, ex, k, keep)
    rows, scores, _ = unpack_result(packed, k)
    np.testing.assert_array_equal(rows, want_rows + base)
    np.testing.assert_allclose(scores, want_scores, rtol=SCORE_RTOL, atol=1e-300)


# ------------------------------------------------------------------ a. the seed's bound, bit for bit --------------------
N_SEED = 40_000


def seed_p(kc):
    """Keys each seed warp and CTA publishes (gemv_topk.cu: seed_P)."""
    return min(2 * -(-kc // num_sms()), 32)


def planted_store(dtype, d, kc, seed=0):
    """Gaussian catalog whose best kc rows are planted on samples s[8 j], j = 1..kc: each seed CTA holds at most
    seed_P of them, and they are far above every other row in int8 too, so the seed's selection is exactly the planted
    rows and its bound the smallest of their fast scores: the final kc-th fast score."""
    st = CatalogStore.synthetic(seed, N_SEED, d, dtype, scale_rows=True, device=DEV)
    j = np.arange(1, kc + 1)
    assert np.bincount(seed_cta(8 * j, num_sms())).max() <= seed_p(kc)
    rows = seed_rows(N_SEED)[8 * j]
    q = synth.query_f32(1, d)
    plant(st, rows, q, seed=d + kc)
    return st, rows, q


@pytest.mark.parametrize("d", GATED_D)
@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
def test_seed_bound_is_the_final_kth_fast_score(dtype, d):
    for k in (10, 40, 100, 240):
        kc = nat.load().rebert_candidates_for_k(k)
        st, planted, q = planted_store(dtype, d, kc)
        others = np.setdiff1d(np.arange(N_SEED), planted)
        excl = np.random.default_rng(1).choice(others, size=133, replace=False)
        for q_scale in (None, 7.5, 1e-3):
            w, keys, _ = check(st, k, query=q, excl=excl, q_scale=q_scale)
            assert np.array_equal(np.sort(key_rows(keys)), np.sort(planted)), "the planted rows are not the plain pass's candidates"
            assert w == int(keys[kc - 1]) >> 32, (k, q_scale, w, int(keys[kc - 1]) >> 32)
        del st
        torch.cuda.empty_cache()


@pytest.mark.parametrize("d,dtype", [(1536, "bf16"), (700, "fp32"), (3000, "bf16")])
def test_unsampled_ties_at_the_bound_are_kept(dtype, d):
    """Copies of the kc-th planted row on unsampled rows with lower ids: the final kc-th key is a copy the seed never saw,
    tied with its bound, and the gated kernel must keep it (sc >= hint)."""
    for k in (10, 40, 100, 240):
        kc = nat.load().rebert_candidates_for_k(k)
        st, planted, q = planted_store(dtype, d, kc)
        _, keys, _ = check(st, k, query=q)
        rk = int(key_rows(keys[kc - 1:kc])[0])
        copies = np.arange(1, rk, 2)[:3]                     # odd rows: the sample stride is 2, so none is sampled
        assert len(copies) and not np.isin(copies, seed_rows(N_SEED)).any()
        write_rows(st, copies, src=np.full(len(copies), rk))
        w, keys, packed = check(st, k, query=q)
        assert key_rows(keys[kc - 1:kc])[0] == copies[0], "the kc-th key is not the lowest copy"
        assert w == int(keys[kc - 1]) >> 32
        oracle_check(st, packed, k, q=q)
        del st
        torch.cuda.empty_cache()


@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
def test_all_winners_in_one_seed_cta_lose_the_bound_not_the_result(dtype):
    """All kc planted rows among the samples of seed CTA 0: it publishes only seed_P of them, so the bound comes from
    other rows and is strictly below the kc-th key (the documented seed_P loss); results stay the plain pass's."""
    d = 1536
    s = seed_rows(N_SEED)
    sms = num_sms()
    cta0 = s[np.nonzero(seed_cta(np.arange(len(s)), sms) == 0)[0]]
    for k in (10, 40):
        kc = nat.load().rebert_candidates_for_k(k)
        assert len(cta0) >= kc
        st = CatalogStore.synthetic(3, N_SEED, d, dtype, scale_rows=True, device=DEV)
        q = synth.query_f32(2, d)
        plant(st, cta0[:kc], q, seed=k)
        w, keys, packed = check(st, k, query=q)
        assert np.isin(key_rows(keys), cta0[:kc]).all()
        assert 0 < w < int(keys[kc - 1]) >> 32, (w, int(keys[kc - 1]) >> 32)
        oracle_check(st, packed, k, q=q)


# ------------------------------------------------------------------ b. row shards ---------------------------------------
R0 = 1_000_003          # first global row of the shard: above n, so no local row id equals a global id inside the shard


def shard_with_planted(dtype, kc, n=N_SEED, d=1536):
    """A shard of rows [R0, R0 + n) whose best 2 kc rows are planted on samples s[8 j], j = 1..2 kc.  The odd j are the
    ones the tests leave allowed: kc rows, at most seed_P per seed CTA."""
    st = CatalogStore.synthetic(11, n, d, dtype, scale_rows=True, device=DEV, row0=R0)
    assert st.row_base == R0
    j = np.arange(1, 2 * kc + 1)
    assert np.bincount(seed_cta(8 * j[::2], num_sms())).max() <= seed_p(kc)
    planted = seed_rows(n)[8 * j]
    q = synth.query_f32(4, d)
    plant(st, planted, q, seed=5 + kc)
    return st, planted, q


def shard_case(st, k, q, excl=None, rf=None, keep=None, planted_allowed=None):
    w, keys, packed = check(st, k, query=q, excl=excl, row_filter=rf)
    oracle_check(st, packed, k, q=q, excl=excl, keep=keep)
    if planted_allowed is not None:
        # exactly kc allowed planted rows, the shard's best: the seed's bound is the final kc-th key
        kc = nat.load().rebert_candidates_for_k(k)
        assert np.array_equal(np.sort(key_rows(keys)), np.sort(planted_allowed))
        assert w == int(keys[kc - 1]) >> 32, (k, w, int(keys[kc - 1]) >> 32)
    return packed


@pytest.mark.parametrize("long_list", [False, True], ids=["smem_list", "global_list"])
@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
def test_shard_exclusions_of_global_ids(dtype, long_list):
    """Exclusion lists of global ids below, inside and above the shard, staged in shared memory (<= 4096 ids) or searched
    in global memory (> 4096).  Half the planted best rows are excluded by global id: a seed or gated kernel that tested
    local ids would take their scores into its bound and lose the allowed winners."""
    for k in (10, 40, 100, 240):
        kc = nat.load().rebert_candidates_for_k(k)
        st, planted, q = shard_with_planted(dtype, kc)
        n = st.n
        others = np.setdiff1d(np.arange(n), planted)
        inside = R0 + np.random.default_rng(7).choice(others, size=6000 if long_list else 1500, replace=False)
        excl = np.concatenate([[0, 5, 77, R0 - 1], R0 + planted[1::2], inside, [R0 + n, R0 + n + 7, 2**31 - 2]])
        assert (len(np.unique(excl)) > 4096) == long_list
        shard_case(st, k, q, excl=excl, planted_allowed=planted[0::2])
        del st
        torch.cuda.empty_cache()


@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
def test_shard_bitmap_and_genre_year_columns(dtype):
    """A local-row bitmap and genre / year columns sliced to the shard (as a ShardedCatalog rank sets them); half the
    planted best rows are removed by the genre test, the year range or the bitmap."""
    for k in (10, 40, 100, 240):
        kc = nat.load().rebert_candidates_for_k(k)
        st, planted, q = shard_with_planted(dtype, kc)
        n = st.n
        ok, out = planted[0::2], planted[1::2]
        g, y = synth.movie_metadata(3, R0, n)
        g, y = g.copy(), y.copy()
        g[ok] |= 0b1
        y[ok] = 1980
        g[out[0::3]] = 0b10000                             # no genre of the filter
        y[out[1::3]] = 1900                                # outside the year range
        st.set_metadata(g, y)
        bits = np.zeros((n + 31) // 32, dtype=np.uint32)
        bits[::5] = 0x0F0F0F0F
        for r in ok:
            bits[r >> 5] &= ~np.uint32(1 << (r & 31))
        for r in out[2::3]:                                # the rest: excluded by the bitmap
            bits[r >> 5] |= np.uint32(1 << (r & 31))
        bm = torch.from_numpy(bits.view(np.int32)).to(DEV)
        rf = RowFilter(genre_any=0b1011, year_lo=1960, year_hi=2000, exclude_bitmap=bm)
        keep = ((g & 0b1011) != 0) & (y >= 1960) & (y <= 2000)
        keep &= ((bits[np.arange(n) >> 5] >> (np.arange(n) & 31).astype(np.uint32)) & 1) == 0
        assert keep[ok].all() and not keep[out].any()
        excl = R0 + np.setdiff1d(np.arange(0, n, 13), ok)
        shard_case(st, k, q, excl=excl, rf=rf, keep=keep, planted_allowed=ok)
        del st, bm
        torch.cuda.empty_cache()


@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
def test_under_full_and_empty_shards(dtype):
    """Fewer allowed rows than kc on a shard (150 rows, kc = 256 at k = 140 and 240), and a shard without rows: nothing
    to bound, every allowed row is fetched."""
    q = synth.query_f32(1, 1536)
    st = CatalogStore.synthetic(1, 300, 1536, dtype, scale_rows=True, device=DEV, row0=R0)
    excl = np.concatenate([[3, R0 - 1], R0 + np.arange(0, 300, 2), [R0 + 300, R0 + 301]])
    for k in (140, 240):
        assert nat.load().rebert_candidates_for_k(k) > 150
        packed = shard_case(st, k, q, excl=excl)
        assert int(packed[2 * k:2 * k + 1].view(np.int32)[0]) == min(k, 150)
    empty = CatalogStore.synthetic(1, 0, 1536, dtype, device=DEV, row0=R0)
    for k in (10, 240):
        packed = shard_case(empty, k, q, excl=excl)
        assert int(packed[2 * k:2 * k + 1].view(np.int32)[0]) == 0


def test_bench_sized_row_shards_build_their_gates():
    """The two row shards of a 2-GPU catalog just above the gate threshold (each saves GATE_MIN_SAVED_BYTES on its own),
    built on one device: each constructor must build its gate (size rule and probe request), each shard's gated requests
    must read rows of record, and the shards' results merged by (score desc, row asc) must equal the whole catalog's
    plain pass, ids exact and fp64 score bits equal.  The exchange between ranks is tests/test_multigpu_gate.py's."""
    from robot_ebert_b200.catalog import topk_order
    from robot_ebert_b200.sharding import ShardPlan
    d = 1536
    n = 2 * (CatalogStore.GATE_MIN_SAVED_BYTES // d + 8192)          # bf16 rows of 1536: d bytes saved per row
    plan = ShardPlan(n, 2)
    shards = [CatalogStore.synthetic(0, cnt, d, "bf16", scale_rows=True, device=DEV, row0=row0)
              for row0, cnt in (plan.range(0), plan.range(1))]
    for st in shards:
        assert st.n * st.ld >= CatalogStore.GATE_MIN_SAVED_BYTES
        assert st.has_gate, f"shard at row {st.row_base}: the constructor did not build the gate ({st.last_probe_fetches} probe fetches)"
    edge = plan.start(1)
    excl = np.unique(np.concatenate([np.random.default_rng(3).choice(n, size=400, replace=False), edge + np.arange(-3, 3)]))
    reqs = [dict(query=synth.query_f32(1, d), exclude_rows=excl, k=k) for k in (10, 100, 240)]
    got = []
    for r in reqs:
        parts = []
        for st in shards:
            st._scratch().ensure_host(1, 1, 256)
            f0 = host_fetches(st)
            parts.append(st.recommend(**r))
            assert host_fetches(st) - f0 > 0, f"shard at row {st.row_base}: the gated kernel did not run"
        got.append(topk_order(np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts]), r["k"]))
    del shards
    torch.cuda.empty_cache()
    whole = CatalogStore.synthetic(0, n, d, "bf16", scale_rows=True, device=DEV)
    whole.drop_gate()
    for r, (rows, scores) in zip(reqs, got):
        want = whole.recommend(**r)
        np.testing.assert_array_equal(rows, want[0])
        np.testing.assert_array_equal(scores, want[1])


# ------------------------------------------------------------------ c. the public request path -------------------------
@pytest.fixture(params=["pycall", "ctypes"])
def entry(request, monkeypatch):
    """Run recommend() through the CPython side door (csrc/pycall.c) or through ctypes."""
    if request.param == "pycall":
        if nat.fast_recommend_host() is None:
            pytest.skip("the CPython side door is not built")
    else:
        monkeypatch.setattr(nat, "_fast_call", None)
    return request.param


def recommend_both(st, **kw):
    """recommend() on the gated store (which must read rows of record) and after drop_gate(); both must agree bit for
    bit.  Returns the gated (rows, scores, info)."""
    assert st.build_gate()
    st._scratch().ensure_host(1, 1, 256)                  # sized before the count is read (lists of <= 4096 entries)
    f0 = host_fetches(st)
    g = st.recommend(return_info=True, **kw)
    nf = host_fetches(st) - f0
    st.drop_gate()
    p = st.recommend(return_info=True, **kw)
    assert st.build_gate()
    np.testing.assert_array_equal(g[0], p[0])
    np.testing.assert_array_equal(g[1], p[1])
    for key in ("kc", "margin", "proven_exact", "exact_sweep"):
        assert g[2][key] == p[2][key], (key, g[2], p[2])
    assert nf > 0, "the gated kernel did not run"
    return g


def assert_oracle(st, got, k, q=None, liked=None, excl=None):
    m = stored(st)
    if q is not None:
        want_rows, want_scores = ora.query_rows(m, np.asarray(q, dtype=np.float64), excl, k)
    else:
        want_rows, want_scores = ora.recommend_rows(m, liked, excl, k)
    np.testing.assert_array_equal(got[0], want_rows)
    np.testing.assert_allclose(got[1], want_scores, rtol=SCORE_RTOL, atol=1e-300)


@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
def test_recommend_queries_and_profiles(dtype, entry):
    st = CatalogStore.synthetic(0, N_SEED, 1536, dtype, scale_rows=True, device=DEV)
    q = synth.query_f32(1, 1536)
    excl = np.random.default_rng(1).choice(st.n, size=133, replace=False)
    users = synth.user_ratings(2, st.n, 3)
    for k in (1, 10, 100, 240):
        got = recommend_both(st, query=q, exclude_rows=excl, k=k)
        assert got[2]["proven_exact"]
        assert_oracle(st, got, k, q=q, excl=excl)
        for rated, rts in users:
            liked = rated[rts >= 3.5] if (rts >= 3.5).any() else rated[:1]
            got = recommend_both(st, liked_rows=liked, exclude_rows=rated, k=k)
            assert_oracle(st, got, k, liked=liked, excl=rated)


@pytest.mark.parametrize("copies,want_kc,sweep", [(40, 128, False), (300, 256, True)], ids=["widened", "exact_sweep"])
def test_recommend_near_ties_widen_the_proof(copies, want_kc, sweep, entry):
    """Exact duplicates of the best row, many more than k: with 40 of them the list of 32 cannot prove the top 10 and the
    proof loop widens to 128 candidates; with 300 no list can, and the exact sweep answers.  Ties order by row."""
    d, k = 1536, 10
    st = CatalogStore.synthetic(5, N_SEED, d, "bf16", scale_rows=True, device=DEV)
    best = 12_345
    q = st.rows[best, :d].float().cpu().numpy() + 0.05 * synth.query_f32(6, d)
    dups = np.random.default_rng(copies).choice(np.setdiff1d(np.arange(st.n), [best]), size=copies, replace=False)
    write_rows(st, dups, src=np.full(copies, best))
    excl = dups[::7]
    got = recommend_both(st, query=q, exclude_rows=excl, k=k)
    assert got[2]["kc"] == want_kc and got[2]["exact_sweep"] == sweep, got[2]
    assert_oracle(st, got, k, q=q, excl=excl)
    assert np.isin(got[0], np.append(dups, best)).all()


def test_recommend_prefilter_on_a_gated_store(entry):
    """enable_prefilter() on a gated store reuses the gate's int8 rows.  The shadow proves the top 10 of 200k gaussian rows
    (prefilter=True takes it); the plain pass without gate gives the same bits, and so does the oracle."""
    n, d, k = 200_003, 1536, 10
    st = CatalogStore.synthetic(0, n, d, "bf16", scale_rows=True, device=DEV)
    assert st.build_gate()
    st.enable_prefilter()
    assert st._q8_rows is st._gate[0]
    q = synth.query_f32(1, d)
    excl = np.random.default_rng(5).choice(n, size=133, replace=False)
    got = st.recommend(query=q, exclude_rows=excl, k=k, return_info=True, prefilter=True)
    assert got[2]["prefilter"] is True and got[2]["proven_exact"]
    st.drop_gate()
    plain = st.recommend(query=q, exclude_rows=excl, k=k, prefilter=False)
    np.testing.assert_array_equal(got[0], plain[0])
    np.testing.assert_array_equal(got[1], plain[1])
    assert_oracle(st, got, k, q=q, excl=excl)


def test_recommend_prefilter_falls_back_to_the_gated_pass(entry):
    """Rows dominated by one huge element: the shadow's bound cannot prove the result, and the request falls back to the
    standard path — which on this store is the gated pass."""
    n, d, k = 50_000, 1536, 10
    m = synth.catalog_rows_f32(0, 0, n, d)
    m[::3, 7] = 400.0
    st = CatalogStore.from_host(None, m, "bf16", device=DEV)
    assert st.build_gate()
    st.enable_prefilter()
    q = synth.query_f32(1, d)
    f0 = host_fetches(st)
    got = st.recommend(query=q, k=k, return_info=True, prefilter=True)
    assert not got[2]["prefilter"] and got[2]["proven_exact"]
    assert host_fetches(st) - f0 > 0, "the fallback did not take the gated pass"
    st.drop_gate()
    plain = st.recommend(query=q, k=k, prefilter=False)
    np.testing.assert_array_equal(got[0], plain[0])
    np.testing.assert_array_equal(got[1], plain[1])
    assert_oracle(st, got, k, q=q)


def test_row_write_between_drop_and_build_refreshes_the_shared_int8_rows(entry):
    """drop_gate() keeps the int8 rows while the prefilter shadow uses them; a row written before build_gate() must be in
    the rows the gate and the shadow share by the next request (_fresh_int8), or the gate would hide it."""
    n, d = 50_000, 1536
    st = CatalogStore.synthetic(2, n, d, "bf16", device=DEV)
    assert st.build_gate()
    st.enable_prefilter()
    q = synth.query_f32(3, d)
    r0 = st.recommend(query=q, k=10)[0]
    plant_row = 31_337
    assert plant_row not in r0
    st.drop_gate()
    write_rows(st, [plant_row], values=q[None, :])
    assert st.build_gate()
    assert st._gate[0] is st._q8_rows
    for prefilter in (False, True):
        got = st.recommend(query=q, k=10, return_info=True, prefilter=prefilter)
        assert got[0][0] == plant_row
        assert_oracle(st, got, 10, q=q)
    got = recommend_both(st, query=q, k=10, prefilter=False)    # the standard path: the gated kernel
    assert got[0][0] == plant_row


# ------------------------------------------------------------------ d. back to back, and threads -----------------------
def test_back_to_back_requests_of_different_kc_on_one_workspace():
    """Gated requests with different queries, exclusions and kc (32 -> 256 -> 64 -> 32 -> 128) enqueued on one stream and
    ONE workspace with no host sync between them: the seed ticket, the bound word, the fetch counter and the grid-wide hint
    are reused across kc.  Each result must equal the plain pass's for the same request."""
    lib = nat.load()
    d = 1536
    st = CatalogStore.synthetic(0, N_SEED, d, "bf16", scale_rows=True, device=DEV)
    ks = [10, 240, 40, 1, 100, 10, 240]
    qs, q64, _ = st.prepare_queries(np.stack([synth.query_f32(20 + i, d) for i in range(len(ks))]))
    rng = np.random.default_rng(9)
    excls = [torch.from_numpy(np.unique(rng.choice(st.n, size=50 + 900 * i, replace=False)).astype(np.int32)).to(DEV)
             for i in range(len(ks))]
    ws = torch.zeros(lib.rebert_gemv_workspace_bytes(st.n, 256), dtype=torch.uint8, device=DEV)

    def sequence():
        outs = [torch.zeros(2 * k + 2, dtype=torch.int64, device=DEV) for k in ks]
        stream = torch.cuda.current_stream().cuda_stream
        for i, k in enumerate(ks):
            f = nat.Filter()
            f.exclude_rows, f.n_exclude = excls[i].data_ptr(), excls[i].numel()
            nat.check(lib.rebert_recommend_device(C.byref(st._c), None, qs[i].data_ptr(), q64[i].data_ptr(), C.byref(f), k,
                                                  lib.rebert_candidates_for_k(k), ws.data_ptr(), ws.numel(), outs[i].data_ptr(),
                                                  0, None, None, stream))
        return [o.cpu().numpy() for o in outs]                # the first host sync

    assert st.build_gate()
    f0 = fetch_count(ws)
    gated = sequence()
    assert fetch_count(ws) - f0 > 0
    st.drop_gate()
    plain = sequence()
    for i, k in enumerate(ks):
        np.testing.assert_array_equal(gated[i], plain[i], err_msg=f"request {i} (k = {k})")
        assert int(plain[i][2 * k:2 * k + 1].view(np.int32)[0]) == k


def test_concurrent_threads_on_one_gated_store():
    """4 threads x 20 requests (queries and profiles, k from 1 to 240) on one gated store, each with its own scratch:
    every result equals the plain pass's for the same request."""
    d = 1536
    st = CatalogStore.synthetic(0, N_SEED, d, "bf16", scale_rows=True, device=DEV)
    users = synth.user_ratings(4, st.n, 80)
    reqs = []
    for i in range(80):
        k = (1, 10, 40, 100, 240)[i % 5]
        rated, rts = users[i]
        if i % 2:
            reqs.append(dict(query=synth.query_f32(100 + i, d), exclude_rows=rated, k=k))
        else:
            reqs.append(dict(liked_rows=rated[rts >= 3.5] if (rts >= 3.5).any() else rated[:1], exclude_rows=rated, k=k))
    plain = [st.recommend(**r) for r in reqs]
    assert st.build_gate()
    got = [None] * len(reqs)
    errors = []

    def worker(t):
        try:
            for i in range(t, len(reqs), 4):
                got[i] = st.recommend(**reqs[i])
        except BaseException as e:  # noqa: BLE001
            errors.append(e)

    threads = [threading.Thread(target=worker, args=(t,)) for t in range(4)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    for i, (a, b) in enumerate(zip(got, plain)):
        np.testing.assert_array_equal(a[0], b[0], err_msg=f"request {i}")
        np.testing.assert_array_equal(a[1], b[1], err_msg=f"request {i}")


# ------------------------------------------------------------------ e. Python's gate decision = the library's ----------
@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
def test_build_gate_agrees_with_the_library(dtype):
    """For d around every layout boundary: build_gate() returns True exactly when the library takes the gate.  The
    library's decision is read from a store whose int8 rows are handed to it regardless (fetches counted or not)."""
    lib = nat.load()
    for d in (256, 257, 511, 512, 513, 1024, 1025, 1536, 1537, 2048, 2049, 2560, 3072, 3073):
        st = CatalogStore.synthetic(0, 2048, d, dtype, scale_rows=True, device=DEV)
        q = synth.query_f32(1, d)
        kc = lib.rebert_candidates_for_k(10)

        def fetched():
            excl_ptr, ne = st.stage_inputs(q, None, None, None, 10, kc)
            f0 = st.gate_fetches()
            st.enqueue_fused(10, kc, excl_ptr, ne)
            return st.gate_fetches() - f0

        try:
            fetched()
        except nat.NativeError as e:                          # fp32 rows of d > 3072 exceed the streaming kernels' stage
            assert e.code == nat.ERR_UNSUPPORTED and dtype == "fp32" and d > 3072, (d, dtype, e)
            assert not st.gate_layout_ok and not st.build_gate() and not st.has_gate
            continue
        rows8, factor = st._int8_buffers()                    # handed to the library whatever Python decides
        st._c.gate_rows, st._c.gate_factor, st._c.gate_err = rows8.data_ptr(), factor.data_ptr(), st.q8_row_err
        library_gates = fetched() > 0
        st._c.gate_rows, st._c.gate_factor, st._c.gate_err = None, None, 0.0
        assert st.gate_layout_ok == library_gates, (d, dtype, st.gate_layout_ok, library_gates)
        built = st.build_gate()
        assert built == library_gates, (d, dtype)
        if built:
            assert fetched() > 0
        else:
            assert not st.has_gate and not st._c.gate_rows and not st._c.gate_factor
            assert fetched() == 0
        del st, rows8, factor
