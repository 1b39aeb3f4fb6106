"""recommend_batch with a genre / year filter per user (QueryFilters) on the tensor-core path, against float64 on the host.

Every batch mixes unrestricted users, broad (~50 % of rows), narrow (~1 %: fewer than sample_rank allowed rows in the
threshold sample, so tau = -inf and every allowed row survives), fewer-than-k and zero-row users, on top of a per-user
exclusion CSR and a shared exclude_bitmap.  Each user's ids must equal the float64 oracle restricted to that user's rows and
the single-query path with that user's RowFilter.  The per-query re-run would hide a kernel bug, so every test asserts that
a plan was made and bounds the re-run fraction on the unrestricted and broad users.
"""
import numpy as np
import pytest
import torch

from oracle import reference_scoring as ora
from robot_ebert_b200 import CatalogStore, QueryFilters, RowFilter, synth
from tests.test_gpu_batched_edges import KX, _assert_matches_oracle, _excl_csr, _liked_csr, _queries, _status_fraction, _stored_f64

pytestmark = pytest.mark.gpu

D = 128                   # bf16 rows of whole 64-element k-blocks, int8 shadow rows of whole 128-byte k-blocks
N_K50 = 70_001            # above both plans' minimum at k = 50 (bf16 49,152, int8 65,536 rows); 273 tiles + 113 rows
N_K500 = 205_003          # above the long-list minimum at k = 500 (204,800 rows)
# status != 0 bound on the unrestricted and broad users (the rest may legitimately need the re-run, e.g. an overflow).
STATUS_MAX_OPEN = 0.03
KINDS = ("open", "broad", "narrow", "fewer", "zero")


def _store(n):
    store = CatalogStore.synthetic(0, n, D, "bf16", scale_rows=True)
    store.enable_prefilter()
    assert store.batch_gemm_ok and store.batch_shadow_ok
    store.set_metadata(*synth.movie_metadata(3, 0, n))
    return store


def _bitmap(n, seed):
    """Shared exclude_bitmap (~3 % of rows) as the device words RowFilter takes, and its boolean mask."""
    mask = np.random.default_rng(seed).random(n) < 0.03
    words = np.packbits(np.concatenate([mask, np.zeros(-n % 32, bool)]), bitorder="little").view(np.uint32)   # bit r & 31 of word r >> 5
    return torch.from_numpy(words.view(np.int32).copy()).cuda(), mask


def _user_filters(store, b, k, seed, excl):
    """QueryFilters over the kinds in turn, and each user's kind.  'fewer' users get a narrow filter and exclusions (added to
    their CSR segment in place) that leave fewer than k of its rows."""
    g = store.genre_bits.cpu().numpy().view(np.uint32)
    y = store.year.cpu().numpy().view(np.uint16).astype(np.int64)
    rng = np.random.default_rng(seed)
    ga, lo, hi, kinds = [], [], [], []
    for u in range(b):
        kind = KINDS[u % len(KINDS)]
        if kind == "open":
            f = (0, 0, 65535)
        elif kind == "broad":                                      # ~50 %: half the years, or genres of ~half the rows
            y0 = int(rng.integers(1920, 1972))
            f = (0, y0, y0 + 51) if u % 2 else (int(rng.choice(1 << 19, 1)[0]) | 0x1F, 0, 65535)
        elif kind in ("narrow", "fewer"):                          # one genre bit (~13 %) x 8 years (~8 %)
            y0 = int(rng.integers(1920, 2016))
            f = (1 << int(rng.integers(0, 19)), y0, y0 + 7)
        else:                                                      # no allowed row: an empty window, or years nobody has
            f = (0, 2000, 1999) if u % 2 else (0b1, 0, 1900)
        ga.append(f[0]); lo.append(f[1]); hi.append(f[2]); kinds.append(kind)
        if kind == "fewer":
            allowed = np.nonzero(((g & f[0]) != 0) & (y >= f[1]) & (y <= f[2]))[0]
            excl[u] = np.union1d(excl[u], rng.choice(allowed, size=max(len(allowed) - k // 3, 0), replace=False)).astype(np.int32)
    return QueryFilters(ga, lo, hi), np.array(kinds)


def _csr(excl):
    ptr = np.zeros(len(excl) + 1, dtype=np.int64)
    np.cumsum([len(e) for e in excl], out=ptr[1:])
    return ptr, np.concatenate(excl).astype(np.int32)


def _scores(unit, src):
    """float64 score rows of every user: cosines of unit queries, or oracle.recommend_rows' weighted profile formula."""
    if "queries" in src:
        q = src["queries"].astype(np.float64)
        return (q / np.linalg.norm(q, axis=1, keepdims=True)) @ unit.T
    lp, lc, lw = src["liked_ptr"], src["liked_col"], src["liked_w"].astype(np.float64)
    out = np.empty((len(lp) - 1, unit.shape[0]))
    for u in range(len(lp) - 1):
        w = lw[lp[u]:lp[u + 1]]
        out[u] = (w @ (unit[lc[lp[u]:lp[u + 1]]] @ unit.T)) / w.sum()
    return out


def _assert_batched(info, kinds, k, what):
    """The tensor-core pass ran (a plan) and re-ran few of the unrestricted and broad users."""
    assert info["plan"] is not None and info["plan"]["k"] == k, what
    open_ = np.isin(kinds, ("open", "broad"))
    frac = _status_fraction({"status": np.asarray(info["status"])[open_]}, f"{what} (unrestricted + broad users)")
    assert frac <= STATUS_MAX_OPEN, (what, frac)


def _check_users(store, qf, kinds, bitmap_mask, excl, sc, res, k, what):
    rows, scores, counts, info = res
    g = store.genre_bits.cpu().numpy().view(np.uint32)
    y = store.year.cpu().numpy().view(np.uint16)
    for u in range(len(kinds)):
        keep = ~bitmap_mask & ((qf.genre_any[u] == 0) | ((g & qf.genre_any[u]) != 0)) & (y >= qf.year_lo[u]) & (y <= qf.year_hi[u])
        wr, ws = ora.topk_rows(sc[u], k + KX, excl[u], keep_mask=keep)
        msg = f"{what}: user {u} ({kinds[u]}) status {info['status'][u]}"
        if kinds[u] == "zero":
            assert len(wr) == 0, msg
        if kinds[u] == "fewer":
            assert 0 < len(wr) < k, msg
        _assert_matches_oracle(rows[u, :counts[u]], scores[u, :counts[u]], wr, ws, k, msg)
        assert (rows[u, counts[u]:] == -1).all() and np.isneginf(scores[u, counts[u]:]).all(), msg


def _single_query_equal(store, qf, bitmap, src, excl, res, k, users, what):
    rows, scores, counts, _ = res
    for u in users:
        kw = (dict(query=src["queries"][u]) if "queries" in src else
              dict(liked_rows=src["liked_col"][src["liked_ptr"][u]:src["liked_ptr"][u + 1]],
                   weights=src["liked_w"][src["liked_ptr"][u]:src["liked_ptr"][u + 1]]))
        r, s = store.recommend(**kw, exclude_rows=excl[u], k=k, row_filter=qf.row_filter(u, exclude_bitmap=bitmap))
        assert counts[u] == len(r), (what, u)
        np.testing.assert_array_equal(rows[u, :counts[u]], r, err_msg=f"{what}: user {u}")
        np.testing.assert_allclose(scores[u, :counts[u]], s, rtol=1e-9, err_msg=f"{what}: user {u}")


@pytest.mark.parametrize("b,k,n", [(100, 50, N_K50), (129, 50, N_K50), (300, 50, N_K50), (129, 500, N_K500)])
def test_per_user_filters_vs_float64_and_single_query(b, k, n):
    """b = 100: the 1-CTA kernel; b = 129 / 300: the cta_group::2 kernel (a partial second 256-query tile at 300).
    k = 500 takes the long-list stages and the widened retry.  bf16 and int8 operands; queries and CSR profiles."""
    store = _store(n)
    unit = ora._normalize_rows(_stored_f64(store))
    rng = np.random.default_rng(b + k)
    _, _, excl = _excl_csr(rng, n, b)
    qf, kinds = _user_filters(store, b, k, b * k, excl)
    ep, ec = _csr(excl)
    bitmap, bitmap_mask = _bitmap(n, b)
    shared = RowFilter(exclude_bitmap=bitmap)
    lp, lc, lw, _, _ = _liked_csr(rng, n, b)
    sample = [u for u in range(b) if u % 7 == 0 or kinds[u] in ("fewer", "zero")][:40]
    for what, src in [("queries", dict(queries=_queries(b, D, seed=k))), ("profiles", dict(liked_ptr=lp, liked_col=lc, liked_w=lw))]:
        sc = _scores(unit, src)
        runs = {}
        for prefilter in (False, True):
            tag = f"{what} {'int8' if prefilter else 'bf16'} b={b} k={k}"
            res = store.recommend_batch(**src, excl_ptr=ep, excl_col=ec, k=k, row_filter=shared, query_filters=qf,
                                        return_info=True, prefilter=prefilter)
            assert res[3]["int8_operands"] == prefilter
            _assert_batched(res[3], kinds, k, tag)
            _check_users(store, qf, kinds, bitmap_mask, excl, sc, res, k, tag)
            runs[prefilter] = res
        np.testing.assert_array_equal(runs[True][0], runs[False][0])           # same exact pass on the same rows: same bits
        np.testing.assert_array_equal(runs[True][1], runs[False][1])
        _single_query_equal(store, qf, bitmap, src, excl, runs[False], k, sample, f"{what} b={b} k={k}")


@pytest.mark.parametrize("prefilter", [False, True])
@pytest.mark.parametrize("b", [100, 129])
def test_identical_user_filters_equal_the_shared_filter(b, prefilter):
    """Per-user filters that all equal one shared RowFilter give the ids and score bits of recommend_batch(row_filter=...)."""
    n, k = N_K50, 50
    store = _store(n)
    rng = np.random.default_rng(b)
    ep, ec, _ = _excl_csr(rng, n, b)
    q = _queries(b, D, seed=b)
    want = store.recommend_batch(queries=q, excl_ptr=ep, excl_col=ec, k=k, row_filter=RowFilter(0b1011, 1960, 2000),
                                 return_info=True, prefilter=prefilter)
    qf = QueryFilters(np.full(b, 0b1011), np.full(b, 1960), np.full(b, 2000))
    got = store.recommend_batch(queries=q, excl_ptr=ep, excl_col=ec, k=k, query_filters=qf, return_info=True, prefilter=prefilter)
    assert got[3]["plan"] is not None and got[3]["int8_operands"] == prefilter
    assert _status_fraction(got[3], f"identical filters b={b} int8={prefilter}") <= STATUS_MAX_OPEN
    np.testing.assert_array_equal(got[0], want[0])
    np.testing.assert_array_equal(got[1].view(np.int64), want[1].view(np.int64))
    np.testing.assert_array_equal(got[2], want[2])


def test_small_catalog_loop_applies_each_users_filter():
    """Below the plan minimum the batch runs one query at a time: each with its own RowFilter."""
    n, b, k = 5_003, 10, 20
    store = _store(n)
    unit = ora._normalize_rows(_stored_f64(store))
    rng = np.random.default_rng(5)
    _, _, excl = _excl_csr(rng, n, b)
    qf, kinds = _user_filters(store, b, k, 5, excl)
    ep, ec = _csr(excl)
    q = _queries(b, D, seed=5)
    res = store.recommend_batch(queries=q, excl_ptr=ep, excl_col=ec, k=k, query_filters=qf, return_info=True)
    assert res[3]["plan"] is None and res[3]["per_query"] == b
    sc = _scores(unit, dict(queries=q))
    _check_users(store, qf, kinds, np.zeros(n, bool), excl, sc, res, k, "single-query loop")
