"""The batched many-user path at the shapes, widths and ties where kernels go wrong, against float64 on the host.

The reference is always float64 computed from the STORED values (bf16 / fp32 upcast), rankings by
oracle/reference_scoring.py: ids exact (save where the oracle itself orders mathematically tied rows by float64
rounding noise: _assert_matches_oracle), fp64 scores to 1e-9 relative.

recommend_batch hands a query to the single-query kernel when the catalog is below gemm_plan's minimum or when the
batched pass could not prove it (status != 0).  The fallback still returns the right answer, so a GEMM bug would hide
behind it: every batched test asserts that a plan was made and that the fraction of re-run queries stays below a
bound (STATUS_MAX_*).
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import reference_scoring as ora
from robot_ebert_b200 import CatalogStore, _native as nat, synth
from robot_ebert_b200.batcher import RatingsBatcher, recommend_all
from tests.test_prefilter_math import _quantize_rows

pytestmark = pytest.mark.gpu

U32 = 2.0 ** -24            # unit roundoff of fp32
U64 = 2.0 ** -53            # unit roundoff of fp64
N_RAGGED = 4099             # 16 whole 256-row GEMM tiles and a last tile of 3 rows


def _stored_f64(store):
    return store.rows[:store.n, :store.d].to(torch.float64).cpu().numpy()


def _queries(b, d, seed=11):
    return synth.catalog_rows_f32(seed, 0, b, d)


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _excl_csr(rng, n, b, row_base=0, max_len=60):
    """Per-user exclusion CSR of global rows, sorted within a user; some users exclude nothing."""
    ptr, cols = [0], []
    for _ in range(b):
        c = np.sort(rng.choice(n, size=int(rng.integers(0, max_len)), replace=False)) + row_base
        cols.append(c)
        ptr.append(ptr[-1] + len(c))
    return np.array(ptr), np.concatenate(cols).astype(np.int32), cols


def _liked_csr(rng, n, b, max_len=6):
    """Weighted liked-rows CSR: 1..max_len rows per user (duplicates allowed), weights k/8 (exact in fp32 and fp64)."""
    ptr, cols, ws = [0], [], []
    for _ in range(b):
        c = rng.integers(0, n, size=int(rng.integers(1, max_len + 1)))
        if len(c) > 2:
            c[-1] = c[0]                                  # a liked row listed twice
        cols.append(c)
        ws.append(rng.integers(1, 33, size=len(c)) / 8.0)
        ptr.append(ptr[-1] + len(c))
    return np.array(ptr), np.concatenate(cols).astype(np.int32), np.concatenate(ws).astype(np.float32), cols, ws


def _status_fraction(info, what):
    frac = float((np.asarray(info["status"]) != 0).mean())
    print(f"\nstatus!=0 fraction {what}: {frac:.4f}")
    return frac


# =====================================================================================================================
# 1. GEMM building blocks at padded widths (ld > d), whole matrix, ragged last row tile
# =====================================================================================================================
@pytest.mark.parametrize("b", [1, 127, 128, 129, 255, 256, 257])
@pytest.mark.parametrize("d", [40, 50, 100, 300, 1000])
def test_gemm_scores_whole_matrix_vs_float64(d, b):
    """b = 128 / 129 and 256 / 257 straddle the switch from the 1-CTA kernel to the cta_group::2 kernel and its query
    tiles; ld - d = 24, 14, 28, 212, 24 padded columns."""
    n = N_RAGGED
    store = CatalogStore.synthetic(0, n, d, "bf16", scale_rows=True)
    assert store.ld % 64 == 0 and store.ld > d
    _, _, qbf = store.prepare_queries(_queries(b, d))
    nrows = (n + 255) // 256 * 256
    got = store.gemm_scores(qbf, 0, nrows)[:, :n].to(torch.float64).cpu().numpy()
    row0 = nrows - 512                                    # a window over the last two tiles, the ragged one included
    win = store.gemm_scores(qbf, row0, 512)[:, :n - row0].to(torch.float64).cpu().numpy()
    m = _stored_f64(store)
    qh = qbf[:, :d].to(torch.float64).cpu().numpy()
    inv = store.inv_norm[:n].to(torch.float64).cpu().numpy()
    ref = (qh @ m.T) * inv                                # bf16 x bf16 products are exact; fp64 sum
    absdot = (np.abs(qh) @ np.abs(m).T) * inv
    # fp32 accumulation of d exact products, then one fp32 multiply by inv_norm
    gamma = d * U32 / (1.0 - d * U32)
    bound = gamma * absdot * (1.0 + U32) + U32 * np.abs(ref)
    err = np.abs(got - ref)
    bad = np.argwhere(err > bound)
    assert len(bad) == 0, (len(bad), bad[:5].tolist(), float((err / np.maximum(bound, 1e-300)).max()))
    np.testing.assert_array_equal(win, got[:, row0:])


@pytest.mark.parametrize("b", [1, 128, 129, 257])
@pytest.mark.parametrize("d", [100, 300, 1000])
def test_int8_gemm_scores_at_padded_widths_are_the_integer_dot_products(d, b):
    n = N_RAGGED
    lib = nat.load()
    store = CatalogStore.synthetic(0, n, d, "bf16", scale_rows=True)
    store.enable_prefilter()
    ld8 = store._c8.ld
    assert store.batch_shadow_ok and ld8 > d
    qn32, _, _ = store.prepare_queries(_queries(b, d))
    q8, qscale, _ = store.quantize_queries(qn32)
    nrows = (n + 255) // 256 * 256
    out = torch.empty((b, nrows), dtype=torch.float32, device=store.device)
    nat.check(lib.rebert_gemm_scores_i8(C.byref(store._c8), q8.data_ptr(), qscale.data_ptr(), b, 0, nrows, out.data_ptr(),
                                        _stream()))
    torch.cuda.synchronize()
    rows8 = store._q8_rows[:n].cpu().numpy().astype(np.int64)
    q8h = q8.cpu().numpy().astype(np.int64)
    assert not rows8[:, d:].any() and not q8h[:, d:].any()           # padding is zero on both operands
    factor = store._q8_factor[:n].cpu().numpy().astype(np.float64)
    acc = q8h @ rows8.T                                               # exact integer dot products
    want = acc.astype(np.float64) * factor[None, :] * qscale.cpu().numpy().astype(np.float64)[:, None]
    got = out[:, :n].cpu().numpy().astype(np.float64)
    np.testing.assert_allclose(got, want, rtol=3e-7, atol=1e-9)      # two fp32 multiplies on an exact integer


# =====================================================================================================================
# 2. Small kernels against numpy, bit-exact where the arithmetic allows
# =====================================================================================================================
def _awkward_rows(n, d, seed):
    """Gaussian rows, rows scaled by 1e-4 .. 1e4, spiky rows (one entry of 300) and an all-zero row."""
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n, d)).astype(np.float32)
    x[1::7] *= (10.0 ** rng.integers(-4, 5, size=(len(x[1::7]), 1))).astype(np.float32)
    x[2::5, rng.integers(0, d)] = 300.0
    x[5] = 0.0
    return x


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("d", [7, 50, 100, 300, 1536])
def test_catalog_quantize_i8_matches_the_numpy_restatement(d, dtype):
    n = 1000
    store = CatalogStore.from_host(None, _awkward_rows(n, d, d), dtype)
    store.enable_prefilter()
    x = store.rows[:n, :d].to(torch.float32).cpu().numpy()          # the stored values
    nrm = store.norm64[:n].cpu().numpy()                              # the store's own norms (a numpy norm may differ in the last bit)
    q8, factor, row_err = _quantize_rows(x, nrm)
    got8 = store._q8_rows[:n].cpu().numpy()
    assert store._c8.ld >= d
    np.testing.assert_array_equal(got8[:, :d].astype(np.int32), q8)
    assert not got8[:, d:].any()
    gf = store._q8_factor[:n].cpu().numpy()
    np.testing.assert_array_equal(gf.view(np.uint32), factor.astype(np.float32).view(np.uint32))
    assert store.q8_row_err == pytest.approx(row_err, rel=1e-12, abs=0)
    # the shadow's proven bound: |dequantised score - true cosine| <= max_err for any unit query (Cauchy-Schwarz), up to
    # the fp32 rounding of the stored factor
    rng = np.random.default_rng(d + 1)
    qs = rng.standard_normal((64, d))
    qs /= np.linalg.norm(qs, axis=1, keepdims=True)
    shadow = (got8[:, :d].astype(np.float64) @ qs.T) * gf.astype(np.float64)[:, None]
    true = (x.astype(np.float64) @ qs.T) / nrm[:, None]
    assert (np.abs(shadow - true) <= store.q8_row_err + 2 * U32 * np.abs(shadow)).all()


def test_query_quantize_i8_matches_the_numpy_restatement():
    """Unit queries, a zero query and CSR profiles (shorter than 1: the bound scales with the length) at three widths."""
    for d in (100, 300, 1536):
        n = 3000
        store = CatalogStore.synthetic(0, n, d, "bf16", scale_rows=True)
        store.enable_prefilter()
        ld8 = store._c8.ld
        q = _queries(40, d)
        q[3] = 0.0
        q[4, 7] = 500.0                                               # one dominant entry
        qn32, _, _ = store.prepare_queries(q)
        rng = np.random.default_rng(d)
        lp, lc, lw, liked, _ = _liked_csr(rng, n, 40, max_len=12)
        p32, _, _ = store.build_profiles(lp, lc, lw)
        for src, unit in ((qn32, True), (p32, False)):
            q8, qscale, qeps = store.quantize_queries(src)
            x = src[:, :d].cpu().numpy()
            mx = np.abs(x).max(axis=1)
            step = np.where(mx > 0, mx / np.float32(127), np.float32(1)).astype(np.float32)
            want8 = np.clip(np.rint(x / step[:, None]), -127, 127).astype(np.int32)
            got8 = q8.cpu().numpy()
            np.testing.assert_array_equal(got8[:, :d].astype(np.int32), want8)
            assert not got8[:, d:ld8].any()
            np.testing.assert_array_equal(qscale.cpu().numpy().view(np.uint32), step.view(np.uint32))
            x64 = x.astype(np.float64)
            e = x64 - want8 * step.astype(np.float64)[:, None]
            E, N = (e * e).sum(axis=1), (x64 * x64).sum(axis=1)
            with np.errstate(invalid="ignore", divide="ignore"):
                rho = np.where(N > 0, np.sqrt(E / N), 0.0)
            r = store.q8_row_err
            eps = 6.0 * np.sqrt(r * r + rho * rho) / np.sqrt(float(d)) * np.maximum(np.sqrt(N), 1e-30) + 64.0 * 5.96e-8
            np.testing.assert_allclose(qeps.cpu().numpy(), eps, rtol=1e-12, atol=0)
            if not unit:
                multi = np.array([len(np.unique(c)) > 1 for c in liked])
                assert multi.sum() > 20 and (np.sqrt(N[multi]) < 1.0).all()   # means of distinct unit rows are shorter than 1


@pytest.mark.parametrize("weighted", [True, False])
@pytest.mark.parametrize("b", [1, 8, 9, 64])
@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
def test_profile_build_on_a_row_shard_vs_float64(dtype, b, weighted):
    """rebert_profile_accumulate + rebert_profile_finalize on a shard holding global rows [7000, 12000): the CSR also names
    rows of other shards (they count in wsum, their rows are not added), duplicates and the shard's edge rows.
    b <= 8 divides element-wise (DIV), b > 8 multiplies by one reciprocal per row."""
    lib = nat.load()
    n, d, base, total = 5000, 300, 7000, 20_000
    store = CatalogStore.synthetic(0, n, d, dtype, scale_rows=True, row0=base)
    assert store.row_base == base
    rng = np.random.default_rng(b * 2 + weighted)
    edges = np.array([base - 1, base, base + n - 1, base + n])
    ptr, cols = [0], []
    for u in range(b):
        c = np.concatenate([rng.integers(0, total, size=int(rng.integers(0, 30))),
                            rng.integers(base, base + n, size=int(rng.integers(1, 30))), edges[rng.integers(0, 4, size=2)]])
        c[-1] = c[0]                                                  # a liked row listed twice
        cols.append(c)
        ptr.append(ptr[-1] + len(c))
    col = np.concatenate(cols).astype(np.int32)
    w = (rng.integers(1, 33, size=len(col)) / 8.0).astype(np.float32) if weighted else None
    dev, ld = store.device, store.ld
    rp = torch.from_numpy(np.array(ptr, dtype=np.int64)).to(dev)
    cl = torch.from_numpy(col).to(dev)
    wt = None if w is None else torch.from_numpy(w).to(dev)
    sum64 = torch.empty((b, ld), dtype=torch.float64, device=dev)
    wsum = torch.empty(b, dtype=torch.float64, device=dev)
    p32 = torch.empty((b, ld), dtype=torch.float32, device=dev)
    p64 = torch.empty((b, ld), dtype=torch.float64, device=dev)
    pbf = torch.empty((b, ld), dtype=torch.bfloat16, device=dev)
    nat.check(lib.rebert_profile_accumulate(C.byref(store._c), rp.data_ptr(), cl.data_ptr(), None if wt is None else wt.data_ptr(),
                                            b, sum64.data_ptr(), wsum.data_ptr(), _stream()))
    nat.check(lib.rebert_profile_finalize(sum64.data_ptr(), wsum.data_ptr(), b, ld, p32.data_ptr(), p64.data_ptr(), pbf.data_ptr(),
                                          _stream()))
    torch.cuda.synchronize()
    m = _stored_f64(store)
    unit = m / store.norm64[:n].cpu().numpy()[:, None]
    gp64, gws = p64.cpu().numpy(), wsum.cpu().numpy()
    w64 = np.ones(len(col)) if w is None else w.astype(np.float64)
    for u in range(b):
        c, wu = col[ptr[u]:ptr[u + 1]].astype(np.int64), w64[ptr[u]:ptr[u + 1]]
        W = wu.sum()                                                  # multiples of 1/8: exact in any order
        assert gws[u] == W, (u, gws[u], W)
        mine = (c >= base) & (c < base + n)
        ref = (wu[mine, None] * unit[c[mine] - base]).sum(axis=0) / W
        scale = (wu[mine, None] * np.abs(unit[c[mine] - base])).sum(axis=0) / W
        bound = 2 * (mine.sum() + 4) * U64 * scale                    # both fp64 sums of <= L terms, division / reciprocal
        err = np.abs(gp64[u, :d] - ref)
        assert (err <= bound).all(), (u, float(err.max()), float(bound[err.argmax()]))
        assert not gp64[u, d:].any()
    np.testing.assert_array_equal(p32.cpu().numpy(), gp64.astype(np.float32))
    np.testing.assert_array_equal(pbf.view(torch.int16).cpu().numpy().view(np.uint16),
                                  synth.f32_to_bf16_bits(gp64.astype(np.float32)))


@pytest.mark.parametrize("layout", ["dense", "packed"])
@pytest.mark.parametrize("lists,k", [(1, 10), (2, 1), (3, 16), (8, 64)])
def test_merge_topk_vs_lexsort(lists, k, layout):
    """Sorted per-list results with counts 0..k and exact score ties within and across lists, in the dense [lists, b, k]
    layout and in the packed per-rank buffers ShardedCatalog.batch_step all-gathers (rows | scores | counts | status)."""
    lib = nat.load()
    b = 37
    rng = np.random.default_rng(lists * 1000 + k)
    rows = np.full((lists, b, k), -7, dtype=np.int64)                # padding that would win if it were ever read
    scores = np.full((lists, b, k), 5.0)
    counts = np.zeros((lists, b), dtype=np.int32)
    for u in range(b):
        pool = rng.permutation(100_000)[:lists * k]                  # the lists of one query hold distinct rows
        for l in range(lists):
            c = int(rng.integers(0, k + 1)) if u % 5 else (k if u % 10 else 0)
            r = pool[l * k:l * k + c]
            s = rng.integers(-3, 4, size=c) / 4.0                    # few distinct values: exact ties everywhere
            o = np.lexsort((r, -s))
            rows[l, u, :c], scores[l, u, :c], counts[l, u] = r[o], s[o], c
    dev = torch.device("cuda:0")
    if layout == "dense":
        d_rows = torch.from_numpy(rows).to(dev)
        d_scores = torch.from_numpy(scores).to(dev)
        d_counts = torch.from_numpy(counts).to(dev)
        ptrs = (d_rows.data_ptr(), d_scores.data_ptr(), d_counts.data_ptr())
        strides = (b * k, b * k, b)
    else:
        hb = (b + 1) // 2
        words = 2 * b * k + 2 * hb
        buf = rng.integers(-(1 << 40), 1 << 40, size=(lists, words)).astype(np.int64)   # status words: junk
        for l in range(lists):
            buf[l, :b * k] = rows[l].ravel()
            buf[l, b * k:2 * b * k] = scores[l].ravel().view(np.int64)
            buf[l, 2 * b * k:2 * b * k + hb].view(np.int32)[:b] = counts[l]
        d_buf = torch.from_numpy(buf).to(dev)
        base = d_buf.data_ptr()
        ptrs = (base, base + 8 * b * k, base + 16 * b * k)
        strides = (words, words, 2 * words)
    out_rows = torch.empty((b, k), dtype=torch.int64, device=dev)
    out_scores = torch.empty((b, k), dtype=torch.float64, device=dev)
    out_count = torch.empty(b, dtype=torch.int32, device=dev)
    nat.check(lib.rebert_merge_topk(*ptrs, *strides, lists, b, k, out_rows.data_ptr(), out_scores.data_ptr(), out_count.data_ptr(),
                                    _stream()))
    got_r, got_s, got_c = out_rows.cpu().numpy(), out_scores.cpu().numpy(), out_count.cpu().numpy()
    for u in range(b):
        rr = np.concatenate([rows[l, u, :counts[l, u]] for l in range(lists)])
        ss = np.concatenate([scores[l, u, :counts[l, u]] for l in range(lists)])
        o = np.lexsort((rr, -ss))[:k]
        c = len(o)
        assert got_c[u] == c, u
        np.testing.assert_array_equal(got_r[u, :c], rr[o], err_msg=f"query {u}")
        np.testing.assert_array_equal(got_s[u, :c], ss[o])
        assert (got_r[u, c:] == -1).all() and (got_s[u, c:] == -np.inf).all()


def test_score_subset_vs_float64_and_nan_outside_the_shard():
    n, d, base = 6000, 300, 50_000
    rng = np.random.default_rng(4)
    for dtype in ("bf16", "fp32"):
        store = CatalogStore.synthetic(3, n, d, dtype, scale_rows=True, row0=base)
        _, qn64, _ = store.prepare_queries(_queries(5, d))
        sub = np.concatenate([rng.integers(base, base + n, size=300), [base, base + n - 1, base - 1, base + n, 0, 1_000_000]])
        got = store.score_subset(qn64, sub)
        inside = (sub >= base) & (sub < base + n)
        assert np.isnan(got[:, ~inside]).all() and not np.isnan(got[:, inside]).any()
        m = _stored_f64(store)[sub[inside] - base].astype(np.longdouble)
        nrm = store.norm64[:n].cpu().numpy()[sub[inside] - base].astype(np.longdouble)
        unit = m / nrm[:, None]
        q = qn64[:, :d].cpu().numpy().astype(np.longdouble)
        ref = (q @ unit.T).astype(np.float64)                          # extended precision: its own error is negligible here
        absd = (np.abs(q) @ np.abs(unit).T).astype(np.float64)
        # per element one fp64 division and one fma; lanes sum ld / 32 terms, then a 5-level shuffle tree
        bound = (store.ld // 32 + 8) * U64 * absd
        err = np.abs(got[:, inside] - ref)
        assert (err <= bound).all(), (dtype, float(err.max()))


# =====================================================================================================================
# 3. recommend_batch against the oracle, every query, across the grid the other tests skip
# =====================================================================================================================
def _oracle_query_topk(unit, queries, k, excl_cols):
    qn = queries.astype(np.float64)
    qn /= np.linalg.norm(qn, axis=1, keepdims=True)
    sc = qn @ unit.T
    return [ora.topk_rows(sc[u], k + KX, excl_cols[u]) for u in range(len(qn))]


def _oracle_profile_topk(unit, liked, weights, k, excl_cols):
    """oracle.recommend_rows' weighted formula, sum_i w_i cos_i / sum_i w_i, on a precomputed unit matrix (the cosines
    of 32 users' liked rows come from one pass over the matrix)."""
    out = []
    for s in range(0, len(liked), 32):
        grp = liked[s:s + 32]
        sims_all = unit[np.concatenate(grp)] @ unit.T
        o = 0
        for c, w, ex in zip(grp, weights[s:s + 32], excl_cols[s:s + 32]):
            sims = sims_all[o:o + len(c)]
            o += len(c)
            out.append(ora.topk_rows((w[:, None] * sims).sum(axis=0) / w.sum(), k + KX, ex))
    return out


KX = 8        # the oracle lists carry k + KX rows, so that ties straddling the k boundary are visible


def _assert_matches_oracle(rows, scores, want_rows, want_scores, k, msg):
    """Ids bit-exact against the oracle, scores to 1e-9, with the one allowance the suite makes on every path
    (tests/test_properties.py): where the oracle orders MATHEMATICALLY tied rows by float64 rounding noise, the GPU may
    order them differently.  Example: a profile of two liked rows of equal weight scores both (1 + cos) / 2, but the
    oracle evaluates x_hat . x_hat as 1 +- 1 ulp, so it puts one of them 1 ulp ahead.  Such a position must hold a row
    the oracle scores within 1e-12 of it, and the oracle's scores there must differ; exact oracle ties are NOT excused
    and must come back in ascending row order."""
    c = min(k, len(want_rows))
    assert len(rows) == c and len(np.unique(rows)) == c, msg
    np.testing.assert_allclose(scores, want_scores[:c], rtol=1e-9, atol=1e-15, err_msg=msg)
    for pos in np.nonzero(rows != want_rows[:c])[0]:
        close = np.abs(want_scores - want_scores[pos]) < 1e-12
        assert (want_scores[close] != want_scores[pos]).any(), (msg, int(pos), rows[:c], want_rows[:c])
        assert rows[pos] in want_rows[close], (msg, int(pos), rows[:c], want_rows[:c])


def _check_against(want, rows, scores, counts, info, k, what):
    for u, (wr, ws) in enumerate(want):
        _assert_matches_oracle(rows[u, :counts[u]], scores[u, :counts[u]], wr, ws, k, f"{what}: query {u} status {info['status'][u]}")
        assert (rows[u, counts[u]:] == -1).all()


# status != 0 bounds (fraction of queries re-run through the single-query kernel), set from a B200 run (NVIDIA B200,
# 1000 W power limit).  Observed: bf16 operands 0 on every grid case but the k = 240 profiles at d = 40, 1 of 257 (0.0039);
# int8 operands 0 on the grid, 1 of 129 (0.0078) for the profiles over an fp32 catalog of record.
STATUS_MAX_BF16 = 0.02
STATUS_MAX_INT8 = 0.03
# Profiles of plain rows in the tie test: two liked rows of equal weight tie mathematically (see _assert_matches_oracle),
# and the batched exact pass rightly sends such near-ties back.  Observed 5 of 100 (0.05).
STATUS_MAX_TIE_PROFILES = 0.10

# (d, b, k, n): n above gemm_plan's minimum for k (bf16 operands: 16,616 for k <= 16, 33,000 for k = 17, 164,072 for
# k = 240; int8 operands: 49,384 for k <= 64, 245,992 for k = 240).  n * d * b stays near 1e10 or below (host oracle).
GRID = [
    (40, 129, 16, 20_000),
    (40, 257, 240, 170_000),
    (100, 257, 17, 60_000),
    (100, 129, 240, 250_000),
    (300, 1, 1, 60_000),
    (300, 257, 1, 60_000),
    (300, 129, 16, 60_000),
    (1000, 129, 16, 60_000),
    (1000, 1, 240, 250_000),
]
I8_MIN_N = {1: 49_384, 16: 49_384, 17: 49_384, 240: 245_992}


@pytest.mark.parametrize("d,b,k,n", GRID)
def test_recommend_batch_bf16_grid_vs_oracle(d, b, k, n):
    store = CatalogStore.synthetic(0, n, d, "bf16", scale_rows=True)
    store.enable_prefilter()
    int8 = store.batch_shadow_ok and n >= I8_MIN_N[k]
    unit = ora._normalize_rows(_stored_f64(store))
    rng = np.random.default_rng(d * 7 + b + k)
    ep, ec, excl = _excl_csr(rng, n, b)
    q = _queries(b, d, seed=d + k)
    lp, lc, lw, liked, ws = _liked_csr(rng, n, b)
    runs = [("queries", dict(queries=q), _oracle_query_topk(unit, q, k, excl)),
            ("profiles", dict(liked_ptr=lp, liked_col=lc, liked_w=lw),
             _oracle_profile_topk(unit, liked, [w.astype(np.float64) for w in ws], k, excl))]
    for what, src, want in runs:
        rb, sb, cb, ib = store.recommend_batch(**src, excl_ptr=ep, excl_col=ec, k=k, return_info=True, prefilter=False)
        assert ib["plan"] is not None and not ib["int8_operands"]
        assert _status_fraction(ib, f"bf16 {what} d={d} b={b} k={k} n={n}") < STATUS_MAX_BF16
        _check_against(want, rb, sb, cb, ib, k, f"bf16 {what}")
        if int8:
            r8, s8, c8, i8 = store.recommend_batch(**src, excl_ptr=ep, excl_col=ec, k=k, return_info=True, prefilter=True)
            assert i8["plan"] is not None and i8["int8_operands"]
            assert _status_fraction(i8, f"int8 {what} d={d} b={b} k={k} n={n}") < STATUS_MAX_INT8
            np.testing.assert_array_equal(r8, rb)
            np.testing.assert_array_equal(s8, sb)                     # same exact pass on the same rows: same bits
            np.testing.assert_array_equal(c8, cb)


@pytest.mark.parametrize("d", [256, 1000])
def test_fp32_catalog_with_int8_operands_vs_oracle(d):
    """An fp32 catalog of record: the GEMM runs on its int8 shadow, the exact pass reads the fp32 rows."""
    n, b, k = 60_000, 129, 10
    store = CatalogStore.synthetic(0, n, d, "fp32", scale_rows=True)
    store.enable_prefilter()
    assert store.batch_shadow_ok and not store.batch_gemm_ok
    unit = ora._normalize_rows(_stored_f64(store))
    rng = np.random.default_rng(d)
    ep, ec, excl = _excl_csr(rng, n, b)
    q = _queries(b, d)
    lp, lc, lw, liked, ws = _liked_csr(rng, n, b)
    for what, src, want in [("queries", dict(queries=q), _oracle_query_topk(unit, q, k, excl)),
                            ("profiles", dict(liked_ptr=lp, liked_col=lc, liked_w=lw),
                             _oracle_profile_topk(unit, liked, [w.astype(np.float64) for w in ws], k, excl))]:
        rows, scores, counts, info = store.recommend_batch(**src, excl_ptr=ep, excl_col=ec, k=k, return_info=True)
        assert info["int8_operands"] and info["plan"] is not None
        assert _status_fraction(info, f"fp32/int8 {what} d={d}") < STATUS_MAX_INT8
        _check_against(want, rows, scores, counts, info, k, f"fp32 catalog, int8 operands, {what}")
    # without the int8 operands no GEMM takes an fp32 catalog: the single-query loop serves it, with the same answer
    rows, scores, counts, info = store.recommend_batch(queries=q[:9], excl_ptr=ep[:10], excl_col=ec[:ep[9]], k=k,
                                                       return_info=True, prefilter=False)
    assert info["plan"] is None
    _check_against(_oracle_query_topk(unit, q[:9], k, excl[:9]), rows, scores, counts, info, k,
                   "fp32 catalog, single-query loop")


def test_batched_exact_ties_come_back_in_row_order():
    """Scaled one-hot rows (each scores exactly +-q_hat[j] in the oracle, whose normalisation divides first) and exact
    duplicate rows.  The batched exact pass divides after the dot product, so one-hot ties may differ there in the last
    bit: its margin must send those queries back to the single-query route.  Exact duplicates tie on both sides and must
    come back in ascending row order from the batched pass itself."""
    n, d, b, k = 60_000, 64, 200, 20
    rng = np.random.default_rng(7)
    m = rng.standard_normal((n, d)).astype(np.float32)
    hot = rng.choice(n, size=3000, replace=False)                    # ~23 rows per (axis, sign)
    m[hot] = 0.0
    m[hot, rng.integers(0, d, size=len(hot))] = (rng.uniform(0.1, 9.0, size=len(hot)) * rng.choice([-1, 1], size=len(hot)))
    plain = np.setdiff1d(np.arange(n), hot)
    src = rng.choice(plain, size=4000, replace=False)
    m[rng.choice(plain, size=4000, replace=False)] = m[src]           # exact duplicates (some of them duplicated twice)
    store = CatalogStore.from_host(None, m, "bf16")
    assert store.batch_gemm_ok
    ms = _stored_f64(store)
    ep, ec, excl = _excl_csr(rng, n, b, max_len=30)
    # queries: even ones plain gaussian (duplicates reach their top-k), odd ones spiky on one axis (one-hot ties on top)
    q = _queries(b, d, seed=3)
    odd = np.arange(1, b, 2)
    q[odd, rng.integers(0, d, size=len(odd))] += 6.0 * rng.choice([-1, 1], size=len(odd)).astype(np.float32)
    rows, scores, counts, info = store.recommend_batch(queries=q, excl_ptr=ep, excl_col=ec, k=k, return_info=True)
    assert info["plan"] is not None
    st = np.asarray(info["status"]) != 0
    print(f"\nstatus!=0 fraction ties: plain queries {st[0::2].mean():.4f}, spiky queries {st[1::2].mean():.4f}")
    assert st[0::2].mean() < STATUS_MAX_BF16
    for u in range(b):
        wr, ws = ora.query_rows(ms, q[u].astype(np.float64), excl[u], k + KX)
        _assert_matches_oracle(rows[u, :counts[u]], scores[u, :counts[u]], wr, ws, k, f"query {u} status {info['status'][u]}")
    # profiles: odd users like a few one-hot rows of one axis and sign (profile = +-e_j), even users plain rows
    by_axis = {}
    for r in hot:
        j = int(np.flatnonzero(ms[r])[0])
        by_axis.setdefault((j, ms[r, j] > 0), []).append(int(r))
    groups = [g for g in by_axis.values() if len(g) >= 8]
    lp, lc, lw, lks, lws = [0], [], [], [], []
    for u in range(b):
        c = np.array(groups[u % len(groups)][:3]) if u % 2 else rng.choice(plain, size=int(rng.integers(1, 6)))
        w = (rng.integers(1, 33, size=len(c)) / 8.0).astype(np.float32)
        lks.append(c); lws.append(w); lc.append(c); lw.append(w); lp.append(lp[-1] + len(c))
    rows, scores, counts, info = store.recommend_batch(liked_ptr=np.array(lp), liked_col=np.concatenate(lc).astype(np.int32),
                                                       liked_w=np.concatenate(lw), excl_ptr=ep, excl_col=ec, k=k, return_info=True)
    assert info["plan"] is not None
    st = np.asarray(info["status"]) != 0
    print(f"status!=0 fraction ties: plain profiles {st[0::2].mean():.4f}, one-hot profiles {st[1::2].mean():.4f}")
    assert st[0::2].mean() < STATUS_MAX_TIE_PROFILES
    for u in range(b):
        wr, ws = ora.recommend_rows(ms, lks[u], excl[u], k + KX, weights=lws[u])
        _assert_matches_oracle(rows[u, :counts[u]], scores[u, :counts[u]], wr, ws, k, f"profile {u} status {info['status'][u]}")


# =====================================================================================================================
# 4. Routing: bf16 catalogs the GEMM cannot take (rows of 16 / 32 elements) go to the single-query loop
# =====================================================================================================================
@pytest.mark.parametrize("d", [8, 16, 24, 32])
def test_narrow_bf16_catalogs_are_served_by_the_single_query_loop(d):
    """bf16 rows of d <= 32 are stored 16 or 32 elements wide, less than one 64-element GEMM k-block.  The catalog is
    big enough for a gemm_plan, so only the width routes it; recommend_batch and the offline recommend_all job must
    still answer every user."""
    n, b, k = 40_000, 24, 10
    m = synth.catalog_rows_f32(0, 0, n, d, scale_rows=True)
    store = CatalogStore.from_host(synth.row_ids(n), m, "bf16")
    assert store.ld in (16, 32)
    store.gemm_plan(b, k)                                             # the size alone would admit the batched path
    ms = _stored_f64(store)
    rng = np.random.default_rng(d)
    ep, ec, excl = _excl_csr(rng, n, b)
    q = _queries(b, d)
    rows, scores, counts, info = store.recommend_batch(queries=q, excl_ptr=ep, excl_col=ec, k=k, return_info=True)
    assert info["plan"] is None and not store.batch_gemm_ok
    for u in range(b):
        wr, ws = ora.query_rows(ms, q[u].astype(np.float64), excl[u], k + KX)
        _assert_matches_oracle(rows[u, :counts[u]], scores[u, :counts[u]], wr, ws, k, f"query {u}")
    batcher = RatingsBatcher(store)
    users = synth.user_ratings(4, n, 16)
    for i, (rated, rts) in enumerate(users):
        batcher.add_user(f"u{i}", [(store.id_of(int(r)), float(x)) for r, x in zip(rated, rts)])
    recs = recommend_all(store, batcher, k=k)
    assert len(batcher) > 8
    for i, (rated, rts) in enumerate(users):
        if f"u{i}" not in batcher.users:
            continue
        wr, ws = ora.recommend_rows(ms, rated[rts >= 3.5], rated, k + KX)
        got = np.array([store.row_of(t) for t, _ in recs[f"u{i}"]])
        _assert_matches_oracle(got, np.array([x for _, x in recs[f"u{i}"]]), wr, ws, k, f"user {i}")
