"""The single-query kernel's int8 score S, bit for bit, with both query planes live (csrc/gemv_topk.cu: quant_planes,
i8_dot4 / i8_dot4_32, i8_score; the exact model is tests/int8_score_model.py).

S is the one number every int8 path computes: the prefilter shadow, the gate, the gate's seed (standalone and folded).
The prefilter's proof bound q8_eps and the gate's delta are only sound for the S the kernel really forms, and an S that is
off by about the query's quantisation error changes no result: only the fetch counts, the seed's bound and the proof
margins see it.  So this file compares exactly those, on general rows and queries (row scales far from 1, so the low
plane l is not zero):

  A. the shadow's candidate keys at every int8 instantiation, against keys of the model's S;
  B. the seed's bound (control word 21) against the seed restated on the model's S and the exact fast scores of an
     integer catalog, at every gated width, folded and standalone;
  C. the gated loop's own S, through its fetch count: with the standalone seed every CTA streams from tile 0 against
     T = fl32(L0 - delta) with L0 the final kc-th fast score, so it fetches exactly kc + #{allowed rows with S >= T}.
"""
import ctypes as C
import types
import zlib

import numpy as np
import pytest
import torch

from robot_ebert_b200 import CatalogStore
from robot_ebert_b200 import _native as nat
from tests import int8_score_model as model
from tests.test_gate_math import quantize_rows
from tests.test_gate_seed_math import orderable, seed_bound
from tests.test_gpu_candidate_keys import (I8_WIDTHS, Exact, Filt, f32_keys, gated_seed_mode, kernel_class, num_sms,
                                           plan_gemv, qbuf, row_layout, template_scores, top_keys)
from tests.test_gpu_gate_edges import GATED_D, check, key_rows, seed_rows

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
ROW_KINDS = ("gauss", "scaled", "dominant_column", "shared_mean")
QUERY_KINDS = ("gauss", "scaled_up", "scaled_down", "spiky", "one_hot", "all_negative", "zero")
UNIT_QUERIES = ("gauss", "spiky", "one_hot", "all_negative")
N_ZERO_ROWS = 5


@pytest.fixture(scope="module")
def ws():
    return torch.zeros(nat.load().rebert_gemv_workspace_bytes(0, 256), dtype=torch.uint8, device=DEV)


def _stream():
    return torch.cuda.current_stream().cuda_stream


def f32_of(keys):
    """The fp32 score of candidate keys."""
    o = (np.asarray(keys, dtype=np.uint64) >> np.uint64(32)).astype(np.uint32)
    b = np.where(o & 0x80000000, o & 0x7FFFFFFF, ~o & 0xFFFFFFFF).astype(np.uint32)
    return b.view(np.float32)


# ------------------------------------------------------------------ A. the shadow's keys ---------------------------------
def catalog_rows(kind, rng, n, d):
    x = rng.standard_normal((n, d)).astype(np.float32)
    if kind == "scaled":                                  # per-row scales 1e-2 .. 1e2
        x *= (10.0 ** rng.uniform(-2, 2, size=(n, 1))).astype(np.float32)
    elif kind == "dominant_column":
        x[:, 0] = np.abs(x[:, 0]) + 60.0
    elif kind == "shared_mean":                           # rows ~0.7 cosine apart: many rows take the insert path
        m = rng.standard_normal(d)
        x = (np.sqrt(0.7) * m / np.linalg.norm(m) + np.sqrt(0.3) * x / np.sqrt(d)).astype(np.float32)
    x[rng.choice(n, size=N_ZERO_ROWS, replace=False)] = 0.0
    return x


def make_query(kind, rng, d, x):
    g = rng.standard_normal(d)
    if kind == "zero":
        return np.zeros(d, dtype=np.float32)
    if kind == "one_hot":
        q = np.zeros(d)
        q[rng.integers(d)] = 1.0
    elif kind == "spiky":
        q = 0.01 * g
        q[rng.integers(d)] = 3.0
    elif kind == "all_negative":                          # against the mean direction of the rows
        nrm = np.linalg.norm(x, axis=1, keepdims=True)
        q = -(x / np.where(nrm > 0, nrm, 1)).sum(axis=0).astype(np.float64)
    else:
        q = g
    q = q / np.linalg.norm(q)
    return (q * {"scaled_up": 7.5, "scaled_down": 1e-3}.get(kind, 1.0)).astype(np.float32)


def shadow_keys(store, q, ws, filt=None):
    lib = nat.load()
    qb = qbuf(q, max(store._c8.ld, store.ld))
    cand = torch.zeros(256, dtype=torch.int64, device=DEV)
    nat.check(lib.rebert_gemv_topk(C.byref(store._c8), qb.data_ptr(), C.byref(filt.f if filt else nat.Filter()), 256,
                                   ws.data_ptr(), ws.numel(), cand.data_ptr(), _stream()))
    return cand.cpu().numpy().view(np.uint64), qb.cpu().numpy()


def host_S(store, qb):
    """The model's S of every shadow row for the query buffer qb (the shadow rows are copied to the host once)."""
    if getattr(store, "_host_q8", None) is None:
        store._host_q8 = (store._q8_rows[:store.n].cpu().numpy(), store._q8_factor[:store.n].cpu().numpy())
    return model.int8_scores(*store._host_q8, qb, store.d)


def check_shadow(store, q, ws, what, filt=None, S=None):
    got, qb = shadow_keys(store, q, ws, filt)
    if S is None:
        S = host_S(store, qb)
    keys = f32_keys(S, np.arange(store.n))
    want = top_keys(keys if filt is None else keys[filt.allowed], 256)
    if not np.array_equal(got, want):
        bad = int(np.nonzero(got != want)[0][0])
        raise AssertionError(f"{what}: {int((got != want).sum())} of 256 keys differ, first at {bad}: got row "
                             f"{key_rows(got[bad:bad + 1])[0]} S={f32_of(got[bad:bad + 1])[0]!r}, want row "
                             f"{key_rows(want[bad:bad + 1])[0]} S={f32_of(want[bad:bad + 1])[0]!r}")
    return got, S, qb


def check_q8_eps(store, keys, qb, what):
    """|S - cos| <= q8_eps on the returned rows (a unit query): the prefilter proof's constant against the kernel's S."""
    rows = key_rows(keys[keys != 0])
    x = store.rows[torch.from_numpy(rows).to(DEV), :store.d].double().cpu().numpy()
    nrm = store.norm64[torch.from_numpy(rows).to(DEV)].cpu().numpy()
    cos = (x @ qb[:store.d].astype(np.float64)) / np.where(nrm > 0, nrm, 1.0)
    err = np.abs(f32_of(keys[keys != 0]).astype(np.float64) - cos).max()
    assert err <= store.q8_eps, (what, err, store.q8_eps)


@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
@pytest.mark.parametrize("d", I8_WIDTHS)
def test_shadow_keys_are_the_models(d, dtype, ws):
    """Every int8 instantiation (LANES 2/4/8/16, 32-lane CPL 1/2/3/4/6/12): rows of four kinds with all-zero rows among
    them, n = 1, 2, 3 (mod 4) with a partial last tile, seven queries."""
    for i, kind in enumerate(ROW_KINDS):
        rng = np.random.default_rng(zlib.crc32(f"{d}{dtype}{kind}".encode()))
        n = (3001, 3002, 3003, 2999)[i]
        p = plan_gemv(d, "i8", n, 256)
        assert n % 4 and n % p["tile_rows"], (n, p["tile_rows"])
        x = catalog_rows(kind, rng, n, d)
        st = CatalogStore.from_host(None, x, dtype, device=DEV)
        st.enable_prefilter()
        for qk in QUERY_KINDS:
            q = make_query(qk, rng, d, x)
            what = f"{dtype} d={d} {kernel_class(d, 'i8')} rows={kind} q={qk}"
            keys, S, qb = check_shadow(st, q, ws, what)
            if qk == "zero":                              # S == +0 everywhere: the keys are the first 256 rows
                assert np.array_equal(key_rows(keys), np.arange(256)) and not S.view(np.uint32).any()
            if qk == "all_negative" and kind in ("dominant_column", "shared_mean"):
                assert (S < 0).sum() == n - N_ZERO_ROWS, what
            if qk in UNIT_QUERIES:
                check_q8_eps(st, keys, qb, what)
            dh, dl, h, l = model.query_planes(qb, d)
            if qk not in ("zero", "one_hot"):             # the low plane is live
                assert np.count_nonzero(l[:d]) > d // 4, what
        del st
    torch.cuda.empty_cache()


def test_shadow_keys_with_filters_on_a_row_shard(ws):
    d, n, base = 1000, 20003, 5000
    rng = np.random.default_rng(31)
    x = catalog_rows("scaled", rng, n, d)
    st = CatalogStore.from_host(None, x, "bf16", device=DEV, row_base=base)
    st.enable_prefilter()
    sh = types.SimpleNamespace(store=st, n=n)
    q = make_query("gauss", rng, d, x)
    _, S, _ = check_shadow(st, q, ws, "no filter")
    best = np.argsort(-S, kind="stable")[:300]                       # the unfiltered winners and more
    outside = np.array([0, base - 1, base + n, base + n + 999])      # global ids outside the shard
    for length in (4096, 4097):                                      # staged in shared memory / searched in global memory
        fill = rng.choice(np.setdiff1d(np.arange(n), best), size=length - len(best) - len(outside), replace=False)
        f = Filt(sh, excl=np.concatenate([best + base, fill + base, outside]))
        assert f.f.n_exclude == length
        keys, _, _ = check_shadow(st, q, ws, f"exclusions {length}", f, S)
        assert not np.isin(key_rows(keys), best).any()
    f = Filt(sh, bitmap_rows=np.union1d(best[::2], rng.choice(n, size=n // 3, replace=False)))
    check_shadow(st, q, ws, "bitmap", f, S)


def test_shadow_keys_on_a_catalog_with_a_dynamic_tail(ws):
    """300k x 1536: the last tiles are claimed from the grid-wide counter."""
    d, n = 1536, 300_000
    p = plan_gemv(d, "i8", n, 256)
    assert p["grid"] == num_sms() and p["rounds"] - p["static_rounds"] >= 8
    st = CatalogStore.synthetic(3, n, d, "bf16", scale_rows=True, device=DEV)
    st.enable_prefilter()
    rng = np.random.default_rng(5)
    x = st.rows[:4096, :d].float().cpu().numpy()
    for qk in ("gauss", "scaled_up", "spiky", "all_negative"):
        q = make_query(qk, rng, d, x)
        keys, _, qb = check_shadow(st, q, ws, f"300k q={qk}")
        if qk in UNIT_QUERIES:
            check_q8_eps(st, keys, qb, qk)
    del st
    torch.cuda.empty_cache()


# ------------------------------------------------------------------ B. the seed's bound ----------------------------------
N_SEED = 40_000
SMALL_N = 1000                                            # a gated grid smaller than the SM count at every gated width
SEED_CASES = [(d, N_SEED) for d in GATED_D] + [(700, SMALL_N), (1536, SMALL_N)]


def integer_query(rng, d):
    """Entries in [-8, 8]: max |q| is not 127, so q / dh is not an integer and the low plane is live."""
    q = rng.integers(-8, 9, size=d)
    q[0] = 8
    return q


def raw_query(ex):
    return ex.q.astype(np.float32)


def gate_S(store, q, rows):
    """The model's S of the gate rows at the given local rows."""
    r8, fac = store._gate
    idx = torch.from_numpy(np.asarray(rows, dtype=np.int64)).to(DEV)
    return model.int8_scores(r8[idx].cpu().numpy(), fac[idx].cpu().numpy(), q, store.d)


def test_seed_cases_reach_the_folded_seed_and_the_seed_kernel():
    modes = set()
    for d, n in SEED_CASES:
        for kc in (32, 64, 128, 256):
            mode, grid = gated_seed_mode(d, "bf16", n, kc)
            modes.add((mode, row_layout(d, "i8")[1] <= 4, grid == num_sms()))
    assert {("fold", True, True), ("kernel", False, True), ("kernel", True, False)} <= modes, modes


@pytest.mark.parametrize("excl", [False, True])
@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
@pytest.mark.parametrize("d,n", SEED_CASES)
def test_seed_bound_is_the_restated_seed_on_the_models_S(d, n, dtype, excl):
    rng = np.random.default_rng(zlib.crc32(f"{d}{n}{dtype}{excl}".encode()))
    pool = rng.integers(-8, 9, size=(3000, d))
    q = integer_query(rng, d)
    ex = Exact(pool, rng.integers(0, len(pool), size=n), q, dtype)
    st = ex.store
    assert st.build_gate()
    s = seed_rows(n)
    S = np.full(n, -np.inf, dtype=np.float32)
    S[s] = gate_S(st, raw_query(ex), s)
    F = ex.dots().astype(np.float32) * ex.inv
    allowed = np.ones(n, dtype=bool)
    ex_rows = None
    if excl:                                              # the sample's best rows by S, and a third of the rest
        best = s[np.argsort(-S[s], kind="stable")[:40]]
        ex_rows = np.union1d(best, rng.choice(s, size=len(s) // 3, replace=False))
        allowed[ex_rows] = False
    for k in (10, 40, 100, 240):
        kc = nat.load().rebert_candidates_for_k(k)
        bound, _ = seed_bound(S, F, allowed, kc, grid=num_sms())
        want = 0 if bound is None else int(orderable(np.float32(bound)))
        w, keys, _ = check(st, k, query=raw_query(ex), excl=ex_rows, q_raw=raw_query(ex))
        assert np.array_equal(keys, ex.keys(kc, allowed)), "plain candidates"
        assert w == want, (k, gated_seed_mode(d, dtype, n, kc, 0 if ex_rows is None else len(ex_rows)), hex(w), hex(want))


# ------------------------------------------------------------------ C. the gated loop's S, through its fetch count -------
def band_catalog(rng, d, dtype, n, kc):
    """An integer catalog: kc winners on samples s[8 j] (at most seed_P per seed CTA), far above every other sampled row in
    int8, so the seed's bound L0 is the final kc-th fast score; a band of rows whose fast score lies just under L0, so that
    S straddles T = fl32(L0 - delta); gaussian-like integer rows everywhere else, far below."""
    q = integer_query(rng, d)
    P = q[None, :] + rng.integers(-8, 9, size=(min(30000, 20_000_000 // d), d))
    Fp = template_scores(P, q)
    _, first = np.unique(Fp, return_index=True)
    P, Fp = P[first], Fp[first]                           # distinct fast scores, ascending
    win = P[-kc:]
    L0 = Fp[-kc]
    bg = rng.integers(-8, 9, size=(500, d))
    # delta from the row error the gate will have (its largest rows are these templates; checked after the build)
    row_err = quantize_rows(np.concatenate([P, bg]).astype(np.float32))[2]
    epl = (row_layout(d, dtype)[1]) * (8 if dtype == "bf16" else 4)
    delta = float(model.gate_delta(q.astype(np.float32), d, row_err, epl))
    band = P[(Fp >= L0 - 1.6 * delta) & (Fp <= L0 - 0.4 * delta)]
    assert len(band) >= 10, len(band)
    s = seed_rows(n)
    win_rows = s[8 * np.arange(1, kc + 1)]
    free = np.setdiff1d(np.arange(n), win_rows)
    if n > len(s):                                        # sampling stride 2: the band sits on unsampled rows
        free = np.setdiff1d(free, s)
    band_rows = rng.choice(free, size=min(len(band) * 2, len(free) // 2), replace=False)
    T = np.concatenate([bg, win, band])
    idx = rng.integers(0, len(bg), size=n)
    idx[win_rows] = len(bg) + np.arange(kc)
    idx[band_rows] = len(bg) + kc + rng.integers(0, len(band), size=len(band_rows))
    return Exact(T, idx, q, dtype), win_rows, np.float32(L0), epl


FETCH_CASES = [(3000, N_SEED, 32), (3000, N_SEED, 256)] + [(d, SMALL_N, kc) for d in (300, 700, 1536, 2000) for kc in (32, 64)] + \
              [(d, N_SEED, 32) for d in (300, 1536)]


@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
@pytest.mark.parametrize("d,n,kc", FETCH_CASES)
def test_gated_fetch_count_is_the_models(d, n, kc, dtype):
    rng = np.random.default_rng(zlib.crc32(f"{d}{n}{kc}{dtype}".encode()))
    ex, win_rows, L0, epl = band_catalog(rng, d, dtype, n, kc)
    st = ex.store
    assert st.build_gate()
    q = raw_query(ex)
    F = ex.dots().astype(np.float32) * ex.inv
    S = gate_S(st, q, np.arange(n))
    delta = model.gate_delta(q, d, st.q8_row_err, epl)
    T = np.float32(L0 - delta)
    # rows whose S is within 1e-6 of T could go either way if the kernel's delta differs in its last bit: exclude them
    near = np.nonzero(np.abs(S.astype(np.float64) - T) <= 1e-6 * abs(float(T)))[0]
    assert not np.isin(near, win_rows).any()
    allowed = np.ones(n, dtype=bool)
    allowed[near] = False
    mode, grid = gated_seed_mode(d, dtype, n, kc, len(near))
    # preconditions: the winners are the final kc and the seed's selection; the band straddles T
    assert np.array_equal(np.sort(key_rows(ex.keys(kc, allowed))), np.sort(win_rows))
    bound, sel = seed_bound(S, F, allowed, kc, grid=num_sms())
    assert bound is not None and np.float32(bound) == L0 and np.array_equal(np.sort(sel), np.sort(win_rows))
    band = allowed & (F < L0) & (F >= L0 - 2 * delta)
    assert (S[band] >= T).sum() >= 3 and (S[band] < T).sum() >= 3, ((S[band] >= T).sum(), (S[band] < T).sum())
    predicted = kc + int((allowed & (S >= T)).sum())
    k = {32: 10, 64: 40, 128: 100, 256: 240}[kc]
    excl = near if len(near) else None
    excl_ptr, ne = st.stage_inputs(q, None, None, excl, k, kc)
    s = st._scratch()
    s.qn32.zero_()
    s.qn32[:d] = torch.from_numpy(q).to(DEV)
    before = st.gate_fetches()
    st.enqueue_topk(k, kc, excl_ptr, ne)
    got = (st.gate_fetches() - before) & 0xFFFFFFFF
    keys = s.cand.cpu().numpy().view(np.uint64)
    assert np.array_equal(keys, ex.keys(kc, allowed)), "gated candidates"
    print(f"fetches d={d} n={n} kc={kc} {dtype} seed={mode} grid={grid}: {got} observed, {predicted} predicted "
          f"(kc + {predicted - kc} rows with S >= T)")
    if mode == "kernel":
        assert got == predicted, (got, predicted)
    else:                                                 # a CTA that stopped waiting for the folded seed fetches more
        assert got >= predicted, (got, predicted)
