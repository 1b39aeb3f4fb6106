"""GPU parity: the CUDA path (through the C ABI) against the oracle and the reference's golden outputs."""
import numpy as np
import pytest
import torch

from oracle import reference_scoring as ora
from robot_ebert_b200 import CatalogStore, RowFilter, synth
from tests.helpers import build_catalog_f32, build_catalog_f64

pytestmark = pytest.mark.gpu

SCORE_RTOL = 1e-9      # fp64 re-score vs the float64 oracle (north_star allows 1e-5 for fp32)


def _stored_f64(store: CatalogStore) -> np.ndarray:
    return store.rows[:store.n, :store.d].to(torch.float64).cpu().numpy()


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("d,scale", [(32, False), (50, True), (1536, True)])
def test_synth_generator_bit_identical(dtype, d, scale):
    n, row0 = 300, 12345
    store = CatalogStore.synthetic(7, n, d, dtype, scale_rows=scale, row0=row0)
    want = synth.quantise(synth.catalog_rows_f32(7, row0, n, d, scale), dtype)
    np.testing.assert_array_equal(_stored_f64(store), want)
    if store.ld > d:
        assert float(store.rows[:, d:].abs().max()) == 0.0


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_catalog_build_and_norms(dtype):
    m = synth.catalog_rows_f32(3, 0, 500, 96, scale_rows=True)
    m[17] = 0.0
    store = CatalogStore.from_host(synth.row_ids(500), m, dtype)
    want = synth.quantise(m, dtype)
    np.testing.assert_array_equal(_stored_f64(store), want)
    nrm = np.sqrt(np.einsum("ij,ij->i", want, want))
    nrm[nrm == 0] = 1.0
    np.testing.assert_allclose(store.norm64[:500].cpu().numpy(), nrm, rtol=1e-14)
    np.testing.assert_allclose(store.inv_norm[:500].cpu().numpy(), (1.0 / nrm).astype(np.float32), rtol=1e-6)
    assert store.norm64[17].item() == 1.0


def test_golden_user_recs(golden):
    """Every get_user_recs case the unmodified reference produced: ids exact, scores to 1e-9 relative."""
    stores = {}
    checked = 0
    for case in golden["user_recs"]:
        spec = golden["catalogs"][case["catalog"]]
        if case["catalog"] not in stores:
            m = build_catalog_f32(spec)
            stores[case["catalog"]] = CatalogStore.from_host(synth.row_ids(m.shape[0]), m, spec["dtype"])
        store = stores[case["catalog"]]
        rated = [(store.row_of(i), r) for i, r in case["ratings"] if store.row_of(i) is not None]   # lib.py:44
        if not case["ratings"]:
            continue                                                                                # lib.py:39-40
        liked = np.array([r for r, x in rated if x >= 3.5], dtype=np.int64)
        excl = np.array([r for r, _ in rated], dtype=np.int64)
        if case.get("raises"):
            with pytest.raises(ValueError):
                store.recommend(liked_rows=liked, exclude_rows=excl, k=case["k"])
            continue
        rows, scores, info = store.recommend(liked_rows=liked, exclude_rows=excl, k=case["k"], return_info=True)
        assert [store.id_of(r) for r in rows] == [e[0] for e in case["expect"]], case["user_id"]
        np.testing.assert_allclose(scores, [e[1] for e in case["expect"]], rtol=SCORE_RTOL, atol=1e-15)
        checked += 1
    assert checked >= 20


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("n,d,k", [(10_000, 1536, 10), (50_000, 1536, 100), (4099, 32, 10), (20_001, 50, 25),
                                   (3000, 1000, 10), (2500, 2200, 10), (70_000, 256, 50), (1, 1536, 10), (33, 8, 10)])
def test_single_query_vs_oracle(dtype, n, d, k):
    store = CatalogStore.synthetic(0, n, d, dtype, scale_rows=True)
    m = _stored_f64(store)
    q = synth.query_f32(1, d)
    rng = np.random.default_rng(5)
    excl = rng.choice(n, size=min(n // 2, 133), replace=False) if n > 1 else np.array([], dtype=np.int64)
    rows, scores, info = store.recommend(query=q, exclude_rows=excl, k=k, return_info=True)
    want_rows, want_scores = ora.query_rows(m, q.astype(np.float64), excl, k)
    assert info["proven_exact"]
    np.testing.assert_array_equal(rows, want_rows)
    np.testing.assert_allclose(scores, want_scores, rtol=SCORE_RTOL, atol=1e-15)


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_user_profile_vs_oracle(dtype):
    n, d = 30_000, 1536
    store = CatalogStore.synthetic(0, n, d, dtype, scale_rows=True)
    m = _stored_f64(store)
    for rows_u, rts in synth.user_ratings(2, n, 3):
        liked = rows_u[rts >= 3.5]
        got_rows, got_scores = store.recommend(liked_rows=liked, exclude_rows=rows_u, k=10)
        want_rows, want_scores = ora.recommend_rows(m, liked, rows_u, 10)
        np.testing.assert_array_equal(got_rows, want_rows)
        np.testing.assert_allclose(got_scores, want_scores, rtol=SCORE_RTOL, atol=1e-15)


def test_ties_zero_rows_and_short_lists():
    n, d = 5000, 64
    m = synth.catalog_rows_f32(9, 0, n, d)
    dups = [4000, 17, 2500, 900, 4999, 3]
    for r in dups:
        m[r] = m[100]                  # exact duplicates of row 100 -> exact score ties
    m[7] = 0.0                         # zero-norm row must score exactly 0
    store = CatalogStore.from_host(synth.row_ids(n), m, "fp32")
    q = m[100].copy()
    rows, scores = store.recommend(query=q, k=5)
    assert rows.tolist() == sorted(dups + [100])[:5]          # ties resolved by ascending row
    want_rows, want_scores = ora.query_rows(m.astype(np.float64), q.astype(np.float64), None, 5)
    np.testing.assert_array_equal(rows, want_rows)
    # all but 3 rows excluded -> fewer than k results, like lib.py:55 on a short `unrated`
    keep = [7, 100, 4321]
    excl = np.setdiff1d(np.arange(n), keep)
    rows, scores = store.recommend(query=q, exclude_rows=excl, k=10)
    want_rows, want_scores = ora.query_rows(m.astype(np.float64), q.astype(np.float64), excl, 10)
    np.testing.assert_array_equal(rows, want_rows)
    np.testing.assert_allclose(scores, want_scores, rtol=SCORE_RTOL, atol=1e-15)
    assert scores[rows.tolist().index(7)] == 0.0
    # everything excluded -> empty
    rows, scores = store.recommend(query=q, exclude_rows=np.arange(n), k=10)
    assert rows.shape == (0,) and scores.shape == (0,)


def test_predicate_filter_and_bitmap():
    n, d = 40_000, 128
    store = CatalogStore.synthetic(4, n, d, "bf16")
    g, y = synth.movie_metadata(3, 0, n)
    store.set_metadata(g, y)
    m = _stored_f64(store)
    q = synth.query_f32(1, d)
    keep = ((g & 0b1011) != 0) & (y >= 1960) & (y <= 2000)
    rows, scores = store.recommend(query=q, k=50, row_filter=RowFilter(genre_any=0b1011, year_lo=1960, year_hi=2000))
    want_rows, want_scores = ora.query_rows(m, q.astype(np.float64), None, 50, keep_mask=keep)
    np.testing.assert_array_equal(rows, want_rows)
    # same mask expressed as an exclusion bitmap
    bits = np.packbits(~keep, bitorder="little")
    bits = np.concatenate([bits, np.zeros((-len(bits)) % 4, np.uint8)]).view(np.int32)
    bm = torch.from_numpy(bits.copy()).to(store.device)
    rows2, _ = store.recommend(query=q, k=50, row_filter=RowFilter(exclude_bitmap=bm))
    np.testing.assert_array_equal(rows2, want_rows)


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_million_rows_against_dense_scores(dtype):
    """BASELINE config 2 size: the fused path against the independent dense-score kernel + torch.topk."""
    n, d, k = 1_000_000, 1536, 10
    store = CatalogStore.synthetic(0, n, d, dtype)
    q = synth.query_f32(1, d)
    excl = np.random.default_rng(1).choice(n, size=133, replace=False)
    rows, scores, info = store.recommend(query=q, exclude_rows=excl, k=k, return_info=True)
    assert info["proven_exact"]
    qn = (q.astype(np.float64) / np.linalg.norm(q.astype(np.float64)))
    q32 = torch.zeros((1, store.ld), dtype=torch.float32, device=store.device)
    q32[0, :d] = torch.from_numpy(qn.astype(np.float32)).to(store.device)
    dense = store.scores_dense(q32)[0]
    dense[torch.from_numpy(excl).to(store.device)] = -float("inf")
    top = torch.topk(dense, k + 8)
    cand = top.indices.cpu().numpy()
    # exact fp64 scores of the dense path's candidates, computed on the host from regenerated rows
    exact = []
    for r in cand:
        row = synth.quantise(synth.catalog_rows_f32(0, int(r), 1, d), dtype)[0]
        exact.append(float(row @ qn / np.linalg.norm(row)))
    order = np.lexsort((cand, -np.array(exact)))[:k]
    np.testing.assert_array_equal(rows, cand[order])
    np.testing.assert_allclose(scores, np.array(exact)[order], rtol=SCORE_RTOL)


def test_unsupported_and_invalid_arguments():
    store = CatalogStore.synthetic(0, 100, 32, "fp32")
    q = synth.query_f32(1, 32)
    with pytest.raises(ValueError):
        store.recommend(query=q, k=0)
    with pytest.raises(ValueError):
        store.recommend(query=q, k=10**6)
    with pytest.raises(ValueError):
        store.recommend(query=q[:5], k=3)
    with pytest.raises(ValueError):
        store.recommend(query=q, liked_rows=np.array([1]), k=3)


def test_concurrent_requests_from_threads():
    """FastAPI's threadpool pattern: many threads share one immutable catalog, each with its own scratch + stream."""
    import threading
    n, d = 60_000, 256
    store = CatalogStore.synthetic(0, n, d, "bf16", scale_rows=True)
    m = _stored_f64(store)
    users = synth.user_ratings(2, n, 8)
    want = [ora.recommend_rows(m, r[x >= 3.5], r, 10) for r, x in users]
    errors = []

    def worker(u):
        try:
            stream = torch.cuda.Stream()
            with torch.cuda.stream(stream):
                for _ in range(25):
                    r, x = users[u]
                    rows, scores = store.recommend(liked_rows=r[x >= 3.5], exclude_rows=r, k=10)
                    assert np.array_equal(rows, want[u][0])
                    assert np.allclose(scores, want[u][1], rtol=1e-9)
        except Exception as e:  # noqa: BLE001
            errors.append((u, repr(e)))

    threads = [threading.Thread(target=worker, args=(u,)) for u in range(8)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors


@pytest.mark.parametrize("n,d,k", [(624, 1, 1), (3000, 1, 10), (5000, 2, 25), (40_000, 2, 100)])
def test_mass_ties_are_resolved_by_the_exact_sweep(n, d, k):
    """Hundreds of rows tie EXACTLY in float64 (d = 1: every cosine is +-1; d = 2: rows on a few rays) but not in fp32.
    No candidate list can prove that; the exact sweep must, and the row-ascending tie-break must hold."""
    m = synth.catalog_rows_f32(0, 0, n, d, scale_rows=True)
    if d == 2:
        rays = np.array([[1.0, 1.0], [1.0, -1.0], [-1.0, 1.0], [3.0, 1.0]], dtype=np.float32)
        scale = np.exp2(np.random.default_rng(0).integers(-8, 8, size=n)).astype(np.float32)
        m = rays[np.arange(n) % 4] * scale[:, None]
    store = CatalogStore.from_host(synth.row_ids(n), m, "fp32")
    q = np.ones(d, dtype=np.float32)
    excl = np.arange(0, n, 7)
    with np.errstate(all="ignore"):
        rows, scores, info = store.recommend(query=q, exclude_rows=excl, k=k, return_info=True)
    want_rows, want_scores = ora.query_rows(m.astype(np.float64), q.astype(np.float64), excl, k)
    assert info["proven_exact"]
    np.testing.assert_array_equal(rows, want_rows)
    np.testing.assert_allclose(scores, want_scores, rtol=1e-12)


def test_exact_ties_follow_sklearn_operation_order():
    """Found by hypothesis: d = 1 profile mode, and scaled one-hot rows in any d, tie EXACTLY in the float64 reference
    (x/||x|| is exactly +-1).  The exact pass must divide element-wise first, like sklearn's normalize(), to keep the tie."""
    m = synth.catalog_rows_f32(0, 0, 17, 1, scale_rows=True)
    m[int(np.random.default_rng(0).integers(0, 17))] = 0.0
    store = CatalogStore.from_host(synth.row_ids(17), m, "fp32")
    liked = np.array([2, 5, 11])
    rows, scores = store.recommend(liked_rows=liked, k=1)
    want_rows, want_scores = ora.recommend_rows(m.astype(np.float64), liked, None, 1)
    np.testing.assert_array_equal(rows, want_rows)
    # scaled one-hot rows, d = 48: every row on axis j scores exactly q_hat[j] * sign
    rng = np.random.default_rng(1)
    n, d = 4000, 48
    m = np.zeros((n, d), dtype=np.float32)
    m[np.arange(n), rng.integers(0, d, size=n)] = rng.uniform(0.1, 9.0, size=n).astype(np.float32) * rng.choice([-1, 1], size=n)
    store = CatalogStore.from_host(synth.row_ids(n), m, "fp32")
    for liked in (rng.choice(n, size=7, replace=False), rng.choice(n, size=40, replace=False)):
        rows, scores = store.recommend(liked_rows=np.sort(liked), exclude_rows=liked, k=25)
        want_rows, want_scores = ora.recommend_rows(m.astype(np.float64), np.sort(liked), liked, 25)
        np.testing.assert_allclose(scores, want_scores, rtol=1e-12, atol=1e-15)
        np.testing.assert_array_equal(rows, want_rows)


@pytest.mark.parametrize("n,d,k", [(30_000, 64, 241), (50_000, 256, 1000), (300, 32, 500)])
def test_large_k_route(n, d, k):
    """k beyond the register-list kernel (the reference takes any k: api/users.py:151) — bisection + sweep, still exact."""
    store = CatalogStore.synthetic(0, n, d, "bf16", scale_rows=True)
    m = _stored_f64(store)
    q = synth.query_f32(1, d)
    excl = np.random.default_rng(2).choice(n, size=min(n // 3, 133), replace=False)
    rows, scores, info = store.recommend(query=q, exclude_rows=excl, k=k, return_info=True)
    want_rows, want_scores = ora.query_rows(m, q.astype(np.float64), excl, k)
    assert info["proven_exact"] and len(rows) == min(k, n - len(excl))
    np.testing.assert_array_equal(rows, want_rows)
    np.testing.assert_allclose(scores, want_scores, rtol=1e-9, atol=1e-15)
    (rated, rts), = synth.user_ratings(2, n, 1, mean_rated=min(60, n // 4))
    rows, scores = store.recommend(liked_rows=rated[rts >= 3.5] if (rts >= 3.5).any() else rated[:1], exclude_rows=rated, k=k)
    want_rows, want_scores = ora.recommend_rows(m, rated[rts >= 3.5] if (rts >= 3.5).any() else rated[:1], rated, k)
    np.testing.assert_array_equal(rows, want_rows)


def test_plain_c_program_serves_a_request(tmp_path):
    """examples/c_embed.c built with -DWITH_CUDA: a C program (no Python, no torch) builds a catalog with the library's
    kernels and serves one request with host buffers through rebert_recommend_host; same rows/scores as the Python path."""
    import os
    import shutil
    import subprocess
    from robot_ebert_b200 import _native as nat
    gcc, cuda = shutil.which("gcc"), "/usr/local/cuda"
    if gcc is None or not os.path.exists(os.path.join(cuda, "include", "cuda_runtime_api.h")):
        pytest.skip("gcc / CUDA headers not available")
    repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    libdir = os.path.dirname(nat.LIB_PATH)
    exe = str(tmp_path / "c_embed")
    cmd = [gcc, "-std=c99", "-Wall", "-DWITH_CUDA", "-I", os.path.join(repo, "include"), "-I", os.path.join(cuda, "include"),
           os.path.join(repo, "examples", "c_embed.c"), "-o", exe, "-L", libdir, "-lrebert_b200", "-L", os.path.join(cuda, "lib64"),
           "-lcudart", f"-Wl,-rpath,{libdir}", f"-Wl,-rpath,{os.path.join(cuda, 'lib64')}"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    n, d, k = 200_000, 1536, 10
    r = subprocess.run([exe, str(n), str(d), str(k)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, (r.stdout, r.stderr)
    got = [(int(l.split()[1]), float(l.split()[3])) for l in r.stdout.splitlines() if l.startswith("row ")]
    store = CatalogStore.synthetic(0, n, d, "bf16", scale_rows=True)
    rows, scores = store.recommend(query=synth.query_f32(1, d), exclude_rows=np.arange(0, 700, 7), k=k)
    assert [g[0] for g in got] == rows.tolist() and "margin_ok 1" in r.stdout
    np.testing.assert_allclose([g[1] for g in got], scores, rtol=1e-15)


@pytest.mark.parametrize("n,d,dtype,k", [(70_001, 1536, "bf16", 10), (70_001, 1536, "bf16", 100), (9_000, 1536, "fp32", 25),
                                         (40_000, 50, "fp32", 10), (70_001, 1536, "bf16", 200)])
def test_back_to_back_launches_and_both_request_forms_agree(n, d, dtype, k):
    """Every launch leaves the workspace's control words at zero, so back-to-back launches give identical candidate keys
    (a full list of kc) and identical packed results of the one-launch request path.  That path, whose winner selection
    runs in every CTA for kc < 128 and across the cluster for kc >= 128, equals the two-kernel form bit for bit."""
    import ctypes as C
    from robot_ebert_b200 import _native as nat
    lib = nat.load()
    store = CatalogStore.synthetic(0, n, d, dtype, scale_rows=True)
    q = synth.query_f32(1, d)
    excl = np.random.default_rng(1).choice(n, size=133, replace=False)
    kc = lib.rebert_candidates_for_k(k)
    ptr, ne = store.stage_inputs(q, None, None, excl, k, kc)
    s = store._scratch()
    f = nat.Filter()
    f.exclude_rows, f.n_exclude = ptr, ne
    keys = []
    for _ in range(3):
        nat.check(lib.rebert_gemv_topk(C.byref(store._c), s.qn32.data_ptr(), C.byref(f), kc, s.ws.data_ptr(), s.ws.numel(),
                                       s.cand.data_ptr(), torch.cuda.current_stream().cuda_stream))
        keys.append(s.cand.cpu().numpy().copy())
    fused = []
    for _ in range(2):
        store.enqueue_fused(k, kc, ptr, ne)
        fused.append(s.d_out.cpu().numpy().copy())
    store.enqueue_topk(k, kc, ptr, ne)                           # two-kernel form: gemv_topk -> finalize_topk
    two = s.d_out.cpu().numpy().copy()
    for other in keys[1:]:
        np.testing.assert_array_equal(other, keys[0])
    assert int((keys[0] != 0).sum()) == kc
    np.testing.assert_array_equal(fused[1], fused[0])
    np.testing.assert_array_equal(fused[0], two)


@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
@pytest.mark.parametrize("n,d,k", [(200_003, 1536, 10), (60_000, 1536, 100), (30_011, 50, 25), (9_001, 32, 10), (40_000, 768, 240)])
def test_int8_prefilter_same_results_as_the_plain_path_and_the_oracle(dtype, n, d, k):
    """The int8 shadow only chooses candidates; ids and fp64 scores must equal the plain path's and the oracle's."""
    store = CatalogStore.synthetic(0, n, d, dtype, scale_rows=True)
    eps = store.enable_prefilter()
    assert 0.0 < eps < 0.05                                     # gaussian rows: ~0.009 at any d (per-row scale)
    q = synth.query_f32(1, d)
    excl = np.random.default_rng(5).choice(n, size=133, replace=False)
    rows, scores, info = store.recommend(query=q, exclude_rows=excl, k=k, return_info=True, prefilter=True)
    plain_rows, plain_scores = store.recommend(query=q, exclude_rows=excl, k=k, prefilter=False)
    np.testing.assert_array_equal(rows, plain_rows)
    np.testing.assert_array_equal(scores, plain_scores)         # same exact-pass kernel on the same rows: same bits
    want_rows, want_scores = ora.query_rows(_stored_f64(store), q.astype(np.float64), excl, k)
    np.testing.assert_array_equal(rows, want_rows)
    np.testing.assert_allclose(scores, want_scores, rtol=SCORE_RTOL)
    if n >= 200_000 and k <= 10:
        assert info.get("prefilter") is True and info["margin"] > eps      # 10th and 256th best of 200k rows are ~0.02 apart
    # a profile request (mean of unit rows, norm < 1) through the same route
    (rated, rts), = synth.user_ratings(2, n, 1)
    liked = rated[rts >= 3.5] if (rts >= 3.5).any() else rated[:1]
    r2, s2 = store.recommend(liked_rows=liked, exclude_rows=rated, k=k, prefilter=True)
    w2, ws2 = ora.recommend_rows(_stored_f64(store), liked, rated, k)
    np.testing.assert_array_equal(r2, w2)
    np.testing.assert_allclose(s2, ws2, rtol=SCORE_RTOL)


def test_int8_prefilter_falls_back_when_its_bound_cannot_prove_the_result():
    """Rows dominated by one huge element quantise badly (bound ~ 0.09 at d = 1536): the proof fails and the request
    silently takes the plain path — results still equal the oracle's."""
    n, d, k = 50_000, 1536, 10
    m = synth.catalog_rows_f32(0, 0, n, d)
    m[::3, 7] = 400.0                                           # one dominant column in every third row
    store = CatalogStore.from_host(None, m, "bf16")
    eps = store.enable_prefilter()
    assert eps > 0.02
    q = synth.query_f32(1, d)
    rows, scores, info = store.recommend(query=q, k=k, return_info=True)
    assert not info.get("prefilter") and info["proven_exact"]
    want_rows, want_scores = ora.query_rows(_stored_f64(store), q.astype(np.float64), None, k)
    np.testing.assert_array_equal(rows, want_rows)
    np.testing.assert_allclose(scores, want_scores, rtol=SCORE_RTOL)


def test_one_workspace_serves_every_candidate_count():
    """A thread's host scratch is zero-filled ONCE and then reused for every kc (k = 10 -> 32 candidates, k = 100 -> 128,
    forced 256): the kernel's control words must not move with kc.  Regression test for stale candidates after a kc change:
    same query, DIFFERENT exclusions per call, every answer checked against the independent dense kernel."""
    n, d = 1_000_000, 1536
    store = CatalogStore.synthetic(0, n, d, "bf16")
    q = synth.query_f32(1, d)
    qn = (q.astype(np.float64) / np.linalg.norm(q.astype(np.float64)))
    q32 = torch.zeros((1, store.ld), dtype=torch.float32, device=store.device)
    q32[0, :d] = torch.from_numpy(qn.astype(np.float32)).to(store.device)
    dense = store.scores_dense(q32)[0]

    def expect(excl, k):
        sc = dense.clone()
        sc[torch.from_numpy(excl).to(store.device)] = -float("inf")
        cand = torch.topk(sc, k + 8).indices.cpu().numpy()
        exact = np.array([float(row @ qn / np.linalg.norm(row)) for row in
                          (synth.quantise(synth.catalog_rows_f32(0, int(r), 1, d), "bf16")[0] for r in cand)])
        order = np.lexsort((cand, -exact))[:k]
        return cand[order], exact[order]

    first_rows, _ = store.recommend(query=q, k=10)
    for i, (k, forced_kc) in enumerate([(10, None), (100, None), (10, None), (10, 256), (10, None), (50, None), (10, None)]):
        excl = np.unique(np.concatenate([first_rows[:i % 4], np.random.default_rng(i).choice(n, size=133, replace=False)]))
        if forced_kc:
            rows, scores, info = store._recommend_host(q, None, None, excl, k, forced_kc, None)
        else:
            rows, scores, info = store.recommend(query=q, exclude_rows=excl, k=k, return_info=True)
        want_rows, want_scores = expect(excl, k)
        np.testing.assert_array_equal(rows, want_rows)
        np.testing.assert_allclose(scores, want_scores, rtol=SCORE_RTOL)
        assert info["proven_exact"] and not set(rows.tolist()) & set(excl.tolist())
        assert info["attempts"] == 1 and info["kc"] == (forced_kc or (32 if k <= 16 else 128)), info     # never a silent widening


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("n,d", [(2269, 32), (2264, 50), (700, 150), (8000, 16), (85, 1536), (3, 32)])
def test_tiny_catalogs_vs_oracle(dtype, n, d):
    """The reference's production shape (movies-collab: 2269 x 32, create-embeddings.ipynb:1241) and other tiny catalogs:
    a handful of CTAs, lists that are never full, k up to the row count."""
    store = CatalogStore.synthetic(0, n, d, dtype, scale_rows=True)
    m = _stored_f64(store)
    q = synth.query_f32(1, d)
    excl = np.arange(0, n, 7)
    for k in (1, 10, 50, 240):
        rows, scores, info = store.recommend(query=q, exclude_rows=excl, k=k, return_info=True)
        want_rows, want_scores = ora.query_rows(m, q.astype(np.float64), excl, k)
        assert info["proven_exact"]
        np.testing.assert_array_equal(rows, want_rows)
        np.testing.assert_allclose(scores, want_scores, rtol=SCORE_RTOL, atol=1e-300)
    for rated, rts in synth.user_ratings(2, n, 4):
        liked = rated[rts >= 3.5] if (rts >= 3.5).any() else rated[:1]
        rows, scores = store.recommend(liked_rows=liked, exclude_rows=rated, k=10)
        want_rows, want_scores = ora.recommend_rows(m, liked, rated, 10)
        np.testing.assert_array_equal(rows, want_rows)
        np.testing.assert_allclose(scores, want_scores, rtol=SCORE_RTOL, atol=1e-300)


def test_unprovable_result_raises_when_every_sweep_overflows(monkeypatch):
    """Fail closed: when neither a candidate list nor the exhaustive routes can prove the ids, recommend() raises.  Every
    sweep reports an overflow, so the mass-tie sweep and the bisection route both fail for real."""
    n = 3000
    m = synth.catalog_rows_f32(0, 0, n, 1, scale_rows=True)      # d = 1: every cosine is +-1, thousands of exact ties
    store = CatalogStore.from_host(None, np.repeat(m, 64, axis=1), "fp32")        # 3000 x 64, every cosine exactly +-1
    monkeypatch.setattr(CatalogStore, "sweep_above", lambda self, *a, **k: None)   # every sweep overflows: both exhaustive routes fail
    with pytest.raises(RuntimeError, match="cannot be proven exact"):
        store.recommend(query=np.ones(64, dtype=np.float32), k=10)
