"""The single-query streaming kernel's candidate keys (gemv_topk_kernel + the winner selection of merge.cuh), bit for bit.

DESIGN §4.2 proves the ids from `margin > eps`, and that proof assumes the candidate list is exactly the kc best allowed rows
under (fast score desc, row asc).  Here rows and queries are small integers: every partial sum of a dot product stays below
2^24 (asserted), so every fp32 dot the kernel forms is exact whatever its summation order, and its score
fl32(dot * inv_norm[r]) is one correctly rounded multiply that numpy repeats.  The keys the kernel returns must then equal
the host's bit for bit — at every kernel instantiation, at exact ties (duplicates and power-of-two scaled copies, which tie
in fp32 and in fp64), in every winner-selection regime, and through the request path with k = kc, where the packed result
shows which candidates the cluster kernel selected.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import reference_scoring as ora
from robot_ebert_b200 import CatalogStore, RowFilter, synth
from robot_ebert_b200 import _native as nat
from tests.test_selection_math import _select

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
ESIZE = {"fp32": 4, "bf16": 2, "i8": 1}
REG_CPL = (1, 2, 3, 4, 6, 12)                     # register-query instantiations of launch_gemv / launch_gemv_i8
PLAIN_CLASSES = {("lanes", l) for l in (2, 4, 8, 16)} | {("cpl", c) for c in REG_CPL} | {("generic",)}
I8_CLASSES = PLAIN_CLASSES - {("generic",)}      # the int8 shadow has no generic kernel
# widths that reach every class: LANES 2, 4, 8, 16; LANES 32 with CPL 1, 2, 3, 4, 6, 12; generic (CPL 5)
PLAIN_WIDTHS = [("fp32", d) for d in (7, 13, 30, 50, 100, 200, 300, 500, 700, 1536, 600)] + \
               [("bf16", d) for d in (9, 24, 50, 100, 256, 384, 700, 1000, 1536, 3000, 1100)]
I8_WIDTHS = (20, 50, 100, 200, 400, 1000, 1500, 2000, 3000, 6000)
KCS = (32, 64, 128, 256)


# ------------------------------------------------------------------ restatements of the launch code -------------------
def row_layout(d, dtype):
    """csrc/catalog.cu row_layout: (lanes, chunks per lane, ld)."""
    esize = ESIZE[dtype]
    chunks = (d * esize + 15) // 16
    if chunks <= 16:
        lanes = 2
        while lanes < chunks:
            lanes <<= 1
        cpl = 1
    else:
        lanes, cpl = 32, (chunks + 31) // 32
    return lanes, cpl, lanes * cpl * (16 // esize)


def kernel_class(d, dtype):
    """The gemv_topk_kernel family launch_gemv / launch_gemv_i8 picks for rows of width d."""
    lanes, cpl, _ = row_layout(d, dtype)
    if lanes < 32:
        return ("lanes", lanes)
    return ("cpl", cpl) if cpl in REG_CPL else ("generic",)


def num_sms():
    return torch.cuda.get_device_properties(DEV).multi_processor_count


def seed_smem_bytes(kc):
    """csrc/gemv_topk.cu seed_smem_bytes: the folded seed's keys beside the gated kernel's pipeline."""
    p = min(2 * -(-kc // num_sms()), 32)
    return (8 * 32 + 32 + num_sms() * p) * 8 + 8


def plan_gemv(d, dtype, n, kc, n_excl=0, q_floats=None, seed_bytes=0):
    """csrc/gemv_topk.cu plan_gemv and gemv_launch's static / dynamic split.  q_floats: query floats staged in shared memory
    (default: ld for the generic kernel, else none; the gated kernel stages the record's ld); seed_bytes: seed_smem_bytes."""
    sms = num_sms()
    lanes, cpl, ld = row_layout(d, dtype)
    row_bytes = ld * ESIZE[dtype]
    rpw = 32 // lanes
    unit = 8 * rpw
    tr = 48 * 1024 // row_bytes
    if tr >= 2 * unit:
        tr = tr // (2 * unit) * (2 * unit)
    elif tr >= unit:
        tr = unit
    tr &= ~3
    tr = max(tr, 4)
    while tr >= 2 * unit and (n + tr - 1) // tr < sms and ((tr // 2) & 3) == 0:
        tr //= 2
    stage_stride = tr * row_bytes + ((tr * 4 + 127) & ~127)
    if q_floats is None:
        q_floats = ld if kernel_class(d, dtype) == ("generic",) else 0
    fixed = 2 * 4 * 8 + q_floats * 4 + (4 * n_excl if 0 < n_excl <= 4096 else 0) + 128 + seed_bytes
    stages = 4
    while stages > 1 and stages * stage_stride + fixed > 220 * 1024:
        stages -= 1
    smem = max(stages * stage_stride + fixed, 9 * kc * 8)
    cap = 2
    while cap < max(2 * kc, kc + sms):
        cap <<= 1
    while cap < 16384 and cap * 16 <= smem:
        cap <<= 1
    tiles = (n + tr - 1) // tr
    grid = min(sms, max(tiles, 1))
    rounds = (tiles + grid - 1) // grid
    sr = rounds - (rounds * 12 + 99) // 100
    if rounds - sr < 8:
        sr = rounds
    sr = max(sr, 1)
    return dict(tile_rows=tr, grid=grid, static_rounds=sr, rounds=rounds, tiles=tiles, merge_cap=cap, rpw=rpw, stages=stages)


def gated_seed_mode(d, dtype, n, kc, n_excl=0):
    """gemv_launch's choice for a gated request: "fold" (the seed as the gated kernel's prologue: grid of one CTA per SM,
    int8 rows of at most 4 chunks per lane, and the seed's keys fit without a shallower ring) or "kernel" (gate_seed_kernel
    ahead of it).  Also returns the gated grid."""
    x_ld = row_layout(d, dtype)[2]
    g = plan_gemv(d, "i8", n, kc, n_excl, q_floats=x_ld)
    fold = n > 0 and g["grid"] == num_sms() and row_layout(d, "i8")[1] <= 4 and \
        plan_gemv(d, "i8", n, kc, n_excl, q_floats=x_ld, seed_bytes=seed_smem_bytes(kc))["stages"] == g["stages"]
    return ("fold" if fold else "kernel"), g["grid"]


# ------------------------------------------------------------------ exact integer catalogs ----------------------------
def f32_keys(scores, local_rows):
    """The kernel's candidate keys: (orderable fp32 bits << 32) | (0xFFFFFFFF - local row)."""
    b = np.ascontiguousarray(scores, dtype=np.float32).view(np.uint32).astype(np.uint64)
    o = np.where(b & 0x80000000, ~b & 0xFFFFFFFF, b | 0x80000000)
    return (o << np.uint64(32)) | (np.uint64(0xFFFFFFFF) - np.asarray(local_rows, dtype=np.uint64))


def top_keys(keys, kc):
    out = np.zeros(kc, dtype=np.uint64)
    t = np.sort(keys)[::-1][:kc]
    out[:len(t)] = t
    return out


def template_scores(T, q):
    """Fast score of each integer row of T against q (what the kernel computes, host arithmetic)."""
    T = np.asarray(T, dtype=np.int64)
    nrm = np.sqrt((T * T).sum(axis=1).astype(np.float64))
    nrm[nrm == 0] = 1.0
    return (T @ q).astype(np.float32) * (1.0 / nrm).astype(np.float32)


def score_pool(rng, d, q, size, lo=-8, hi=9, sign=None):
    """Integer rows with pairwise distinct fast scores, ascending by score."""
    T = rng.integers(lo, hi, size=(size, d))
    s = template_scores(T, q)
    if sign is not None:
        keep = s < 0 if sign < 0 else s > 0
        T, s = T[keep], s[keep]
    _, first = np.unique(s, return_index=True)
    return T[first], s[first]


class Exact:
    """A catalog whose row r is templates[idx[r]] * 2**exps[r] (integers), built on the device through the same calls as
    CatalogStore.from_host, and the host model of its fast pass."""

    def __init__(self, templates, idx, q, dtype, exps=None, row_base=0):
        lib = nat.load()
        T = np.asarray(templates, dtype=np.int64)
        self.q = np.asarray(q, dtype=np.int64)
        self.idx = np.asarray(idx, dtype=np.int64)
        self.n, self.d = len(self.idx), T.shape[1]
        self.exps = np.zeros(self.n, dtype=np.int64) if exps is None else np.asarray(exps, dtype=np.int64)
        emax = int(self.exps.max()) if self.n else 0
        if len(T):
            # every partial sum of every dot product the kernel forms is an integer below 2^24: exact in fp32, any order
            assert float((np.abs(T) @ np.abs(self.q)).max()) * 2.0 ** emax < 2 ** 24
            assert float(np.abs(T).max()) * 2.0 ** emax <= (256 if dtype == "bf16" else 2 ** 24)   # stored exactly
        self.tdots = T @ self.q
        ld, rows, inv_norm, norm64 = CatalogStore._alloc(self.n, self.d, dtype, DEV)
        st = torch.cuda.current_stream().cuda_stream
        tdev = torch.from_numpy(T.astype(np.float32)).to(DEV)
        chunk = max(1, (64 << 20) // (4 * self.d))
        for s in range(0, self.n, chunk):
            e = min(self.n, s + chunk)
            src = tdev[torch.from_numpy(self.idx[s:e]).to(DEV)]
            src = (src * torch.from_numpy(np.exp2(self.exps[s:e]).astype(np.float32)).to(DEV)[:, None]).contiguous()
            nat.check(lib.rebert_catalog_store_rows(src.data_ptr(), e - s, self.d, nat.DTYPES[dtype],
                                                    rows.data_ptr() + s * ld * rows.element_size(), ld, st))
            torch.cuda.current_stream().synchronize()
        if self.n:
            nat.check(lib.rebert_catalog_norms(rows.data_ptr(), self.n, ld, nat.DTYPES[dtype], inv_norm.data_ptr(),
                                               norm64.data_ptr(), st))
        torch.cuda.current_stream().synchronize()
        self.store = CatalogStore(rows, inv_norm, norm64, self.n, self.d, ld, dtype, row_base, None)
        self.inv = inv_norm[:self.n].cpu().numpy()

    def dots(self, s=0, e=None):
        return self.tdots[self.idx[s:e]] << self.exps[s:e]

    def keys(self, kc, allowed=None, shadow=False):
        """The kc best keys of the allowed rows (descending, zero padded): what rebert_gemv_topk must return."""
        w = self.store._q8_factor[:self.n].cpu().numpy() if shadow else self.inv
        best = np.zeros(0, dtype=np.uint64)
        step = 1 << 21
        for s in range(0, self.n, step):                 # chunked: host memory stays small for large catalogs
            e = min(self.n, s + step)
            k = f32_keys(self.dots(s, e).astype(np.float32) * w[s:e], np.arange(s, e))
            if allowed is not None:
                k = k[allowed[s:e]]
            best = np.concatenate([best, k])
            if len(best) > kc:
                best = np.partition(best, len(best) - kc)[len(best) - kc:]
        return top_keys(best, kc)

    def all_keys(self):
        return f32_keys(self.dots().astype(np.float32) * self.inv, np.arange(self.n))


class Filt:
    """A rebert_filter_t (device) and its host model (allowed[local row])."""

    def __init__(self, ex, excl=None, bitmap_rows=None, row_filter=None, genre=None, year=None):
        st = ex.store
        n, base = ex.n, st.row_base
        self.allowed = np.ones(n, dtype=bool)
        if genre is not None:
            st.set_metadata(genre, year)
        self.f = st._filter_struct(row_filter) or nat.Filter()
        if row_filter is not None and row_filter.genre_any:
            self.allowed &= (genre & np.uint32(row_filter.genre_any)) != 0
        if row_filter is not None and (row_filter.year_lo, row_filter.year_hi) != (0, 65535):
            self.allowed &= (year >= row_filter.year_lo) & (year <= row_filter.year_hi)
        if bitmap_rows is not None:
            words = np.zeros((n + 31) // 32 + 1, dtype=np.uint32)
            np.bitwise_or.at(words, bitmap_rows >> 5, np.uint32(1) << (bitmap_rows & 31).astype(np.uint32))
            self.bitmap = torch.from_numpy(words.view(np.int32)).to(DEV)
            self.f.exclude_bitmap = self.bitmap.data_ptr()
            self.allowed[bitmap_rows] = False
        if excl is not None:
            excl = np.unique(np.asarray(excl, dtype=np.int32))
            self.excl = torch.from_numpy(excl).to(DEV)
            self.f.exclude_rows, self.f.n_exclude = self.excl.data_ptr(), len(excl)
            local = excl.astype(np.int64) - base
            self.allowed[local[(local >= 0) & (local < n)]] = False


@pytest.fixture(scope="module")
def ws():
    """One zero-filled workspace for every launch (sized for kc = 256; every launch leaves its control words zero)."""
    return torch.zeros(nat.load().rebert_gemv_workspace_bytes(0, 256), dtype=torch.uint8, device=DEV)


def _stream():
    return torch.cuda.current_stream().cuda_stream


def qbuf(q, ld, dtype=torch.float32):
    """The query as the kernels read it: [ld], zero past d."""
    out = torch.zeros(ld, dtype=dtype, device=DEV)
    out[:len(q)] = torch.from_numpy(np.asarray(q, dtype=np.float64)).to(dtype)
    return out


def gemv_keys(ex, kc, ws, filt=None, shadow=False):
    lib = nat.load()
    cat = ex.store._c8 if shadow else ex.store._c
    q = qbuf(ex.q, max(cat.ld, ex.store.ld))
    cand = torch.zeros(kc, dtype=torch.int64, device=DEV)
    nat.check(lib.rebert_gemv_topk(C.byref(cat), q.data_ptr(), C.byref(filt.f if filt else nat.Filter()), kc, ws.data_ptr(),
                                   ws.numel(), cand.data_ptr(), _stream()))
    return cand.cpu().numpy().view(np.uint64)


def check_keys(ex, kc, ws, filt=None, shadow=False, what=""):
    got = gemv_keys(ex, kc, ws, filt, shadow)
    want = ex.keys(kc, None if filt is None else filt.allowed, shadow)
    if not np.array_equal(got, want):
        bad = int(np.nonzero(got != want)[0][0])
        raise AssertionError(f"{what} kc={kc}: {int((got != want).sum())} of {kc} keys differ, first at {bad}: "
                             f"got row {0xFFFFFFFF - (int(got[bad]) & 0xFFFFFFFF)} want row {0xFFFFFFFF - (int(want[bad]) & 0xFFFFFFFF)}")
    return want


def check_request_path(ex, kc, ws, want_keys, filt=None, shadow=False):
    """rebert_recommend_device with k = kc (its packed rows are the whole selected set) must equal rebert_finalize_topk run
    on the host's keys: rows (+ row_base), score bits, count and margin."""
    lib = nat.load()
    st = ex.store
    k = kc
    q32 = qbuf(ex.q, max(st.ld, st._c8.ld if shadow else 0))
    q64 = qbuf(ex.q, st.ld, torch.float64)
    fused = torch.zeros(2 * k + 2, dtype=torch.int64, device=DEV)
    nat.check(lib.rebert_recommend_device(C.byref(st._c), C.byref(st._c8) if shadow else None, q32.data_ptr(), q64.data_ptr(),
                                          C.byref(filt.f if filt else nat.Filter()), k, kc, ws.data_ptr(), ws.numel(),
                                          fused.data_ptr(), 0, None, None, _stream()))
    keys = torch.from_numpy(want_keys.view(np.int64).copy()).to(DEV)
    ref = torch.zeros(2 * k + 2, dtype=torch.int64, device=DEV)
    ob = ref.data_ptr()
    nat.check(lib.rebert_finalize_topk(C.byref(st._c), q64.data_ptr(), keys.data_ptr(), kc, k, ob, ob + 8 * k, ob + 16 * k,
                                       ob + 16 * k + 8, _stream()))
    got, want = fused.cpu().numpy(), ref.cpu().numpy()
    cnt = int(want[2 * k:2 * k + 1].view(np.int32)[0])
    assert cnt == int((want_keys != 0).sum())
    assert int(got[2 * k:2 * k + 1].view(np.int32)[0]) == cnt
    np.testing.assert_array_equal(got[:k], want[:k])                     # rows, global
    np.testing.assert_array_equal(got[k:2 * k], want[k:2 * k])           # fp64 score bits
    assert got[2 * k + 1] == want[2 * k + 1]                              # margin bits
    local = (np.uint64(0xFFFFFFFF) - (want_keys[:cnt] & np.uint64(0xFFFFFFFF))).astype(np.int64)
    assert sorted(got[:cnt].tolist()) == sorted((local + st.row_base).tolist())


def random_exact(rng, dtype, d, n, row_base=0, lo=-8, hi=9):
    q = rng.integers(lo, hi, size=d)
    q[0] = 5
    return Exact(rng.integers(lo, hi, size=(n, d)), np.arange(n), q, dtype, row_base=row_base)


def i8_exact(rng, d, n, row_base=0):
    """bf16 rows and a query whose int8 shadow is exact: one entry of +-127 per row / query, the rest in [-2, 2].  Then the
    row scale is 1, q8 = x, the query planes are (q, 0) with dh = 1, and the shadow score is fl32(float(dot) * factor[r])."""
    T = rng.integers(-2, 3, size=(n, d))
    T[np.arange(n), rng.integers(0, d, size=n)] = rng.choice([-127, 127], size=n)
    q = rng.integers(-2, 3, size=d)
    q[rng.integers(0, d)] = 127
    ex = Exact(T, np.arange(n), q, "bf16", row_base=row_base)
    ex.store.enable_prefilter()
    return ex


# ------------------------------------------------------------------ 1. every instantiation ----------------------------
def test_row_layout_restatement_matches_the_library():
    for dtype in ("fp32", "bf16", "i8"):
        for d in list(range(1, 300)) + [511, 512, 513, 1000, 1536, 2049, 2100, 2560, 3000, 4096, 5632, 6000, 6144]:
            assert CatalogStore.layout(10, d, dtype)[0] == row_layout(d, dtype)[2], (dtype, d)
    assert {kernel_class(d, t) for t, d in PLAIN_WIDTHS} == PLAIN_CLASSES
    assert {kernel_class(d, "i8") for d in I8_WIDTHS} == I8_CLASSES


@pytest.mark.parametrize("dtype,d", PLAIN_WIDTHS)
def test_every_plain_instantiation_returns_the_exact_candidate_keys(dtype, d, ws):
    rng = np.random.default_rng(d)
    n = 2000 + d % 13
    ex = random_exact(rng, dtype, d, n)
    for kc in KCS:
        check_keys(ex, kc, ws, what=f"{dtype} d={d} {kernel_class(d, dtype)}")


@pytest.mark.parametrize("d", I8_WIDTHS)
def test_every_int8_instantiation_returns_the_exact_candidate_keys(d, ws):
    rng = np.random.default_rng(d + 1)
    ex = i8_exact(rng, d, 3000 + d % 7)
    check_keys(ex, 256, ws, shadow=True, what=f"i8 d={d} {kernel_class(d, 'i8')}")


# ------------------------------------------------------------------ 2. adversarial arrangements -----------------------
LAYOUTS = [("bf16", 50), ("fp32", 600)]          # LANES 8 (four rows per warp step), generic (CPL 5)


def _query(rng, d):
    q = rng.integers(-8, 9, size=d)
    q[0] = 7
    return q


def arrangement(name, dtype, d, kc, rng):
    """(templates, idx, exps, q) of one adversarial catalog."""
    q = _query(rng, d)
    T, _ = score_pool(rng, d, q, 12000)
    lo, hi = 0, len(T) - 1                            # lowest / highest template
    if name == "rising":                              # every row beats the warp's threshold: every row is an insert
        n = min(len(T), 6000)
        return T, np.arange(len(T) - n, len(T)), None, q
    if name == "falling":
        n = min(len(T), 6000)
        return T, np.arange(len(T) - 1, len(T) - 1 - n, -1), None, q
    if name == "ragged_last_tile":                    # winners only in the last tile; the best three in its last n % 4 rows
        n = 5000 + 4 * kc
        n += 3 - n % 4 if n % 4 == 0 else 0
        p = plan_gemv(d, dtype, n, kc)
        idx = np.full(n, lo)
        start = (p["tiles"] - 1) * p["tile_rows"]
        assert n - start > 3 and n % 4 in (1, 2, 3)
        idx[start:] = rng.permutation(np.arange(hi - (n - start) + 1, hi + 1))
        idx[n - n % 4:] = np.arange(hi - n % 4 + 1, hi + 1)
        return T, idx, None, q
    if name == "one_cta":                             # 2 kc winners, all in the tiles of one CTA (static rounds)
        tr = plan_gemv(d, dtype, 1 << 24, kc)["tile_rows"]
        n = max(3, -(-2 * kc // tr) + 1) * num_sms() * tr
        p = plan_gemv(d, dtype, n, kc)
        assert p["tile_rows"] == tr and p["rounds"] == p["static_rounds"]
        c = p["grid"] // 3
        idx = rng.integers(lo, lo + 200, size=n)
        mine = np.concatenate([np.arange(t * p["tile_rows"], (t + 1) * p["tile_rows"]) for t in range(c, p["tiles"], p["grid"])])
        pick = rng.choice(mine, size=min(len(mine), 2 * kc), replace=False)
        idx[pick] = np.arange(hi - len(pick) + 1, hi + 1)
        return T, idx, None, q
    if name == "all_negative":
        Tn, _ = score_pool(rng, d, q, 12000, sign=-1)
        return Tn, rng.integers(0, len(Tn), size=4000), None, q
    if name == "zero_rows":                           # kc / 2 positive rows, then a block of zero rows (score +0) straddles place kc
        Tn, _ = score_pool(rng, d, q, 4000, sign=-1)
        Tp, _ = score_pool(rng, d, q, 4000, sign=1)
        T = np.concatenate([np.zeros((1, d), dtype=np.int64), Tn, Tp[-kc // 2:]])
        n = 5000
        idx = rng.integers(1, 1 + len(Tn), size=n)
        idx[rng.choice(n, size=3 * kc, replace=False)] = 0
        idx[rng.choice(n, size=kc // 2, replace=False)] = np.arange(1 + len(Tn), len(T))
        return T, idx, None, q
    if name == "ties_at_kc":                          # kc / 2 distinct best rows, then copies of one row tie across place kc
        n = 6000
        idx = rng.integers(lo, hi - 2 * kc, size=n)
        tied = rng.choice(n, size=4 * kc, replace=False)
        idx[tied] = hi - kc
        exps = np.zeros(n, dtype=np.int64)
        exps[tied] = rng.integers(0, 3, size=len(tied))  # power-of-two copies: the same fp32 (and fp64) score
        idx[rng.choice(np.setdiff1d(np.arange(n), tied), size=kc // 2, replace=False)] = np.arange(hi - kc // 2 + 1, hi + 1)
        return T, idx, exps, q
    if name == "all_tied":
        n = 5000
        return T[hi:hi + 1], np.zeros(n, dtype=np.int64), rng.integers(0, 3, size=n), q
    raise ValueError(name)


ARRANGEMENTS = ["rising", "falling", "ragged_last_tile", "one_cta", "all_negative", "zero_rows", "ties_at_kc", "all_tied"]


@pytest.mark.parametrize("dtype,d", LAYOUTS)
@pytest.mark.parametrize("name", ARRANGEMENTS)
def test_adversarial_arrangements(name, dtype, d, ws):
    for kc in (32, 256):
        rng = np.random.default_rng(kc + len(name))
        T, idx, exps, q = arrangement(name, dtype, d, kc, rng)
        ex = Exact(T, idx, q, dtype, exps)
        want = check_keys(ex, kc, ws, what=f"{name} {dtype} d={d}")
        if name == "all_negative":
            assert np.all(want >> np.uint64(63) == 0)              # every candidate scores below zero
        if name in ("zero_rows", "ties_at_kc"):                     # the tie block really straddles place kc
            scores = want >> np.uint64(32)
            assert scores[kc // 2 - 1] != scores[kc - 1] and (ex.all_keys() >> np.uint64(32) == scores[kc - 1]).sum() > kc


def test_winners_only_in_dynamically_claimed_tail_tiles(ws):
    """rows of 6 KB (tile = 8 rows): 59 rounds of tiles, the last 8 of them claimed from the grid-wide counter."""
    dtype, d, kc = "bf16", 3000, 256
    rng = np.random.default_rng(11)
    q = _query(rng, d)
    T, _ = score_pool(rng, d, q, 600)
    grid = num_sms()
    n = 59 * grid * 8 - 5
    p = plan_gemv(d, dtype, n, kc)
    assert p["tile_rows"] == 8 and p["grid"] == grid
    tail0 = p["static_rounds"] * p["grid"] * p["tile_rows"]
    assert p["rounds"] - p["static_rounds"] >= 8                      # a retune must not quietly make this case static
    idx = np.zeros(n, dtype=np.int64)
    win = rng.choice(np.arange(tail0, n), size=2 * kc, replace=False)
    idx[win] = rng.integers(len(T) - 300, len(T), size=len(win))       # ties among the winners too
    ex = Exact(T, idx, q, dtype)
    for k in (32, 256):
        want = check_keys(ex, k, ws, what="dynamic tail")
        assert np.all(0xFFFFFFFF - (want & np.uint64(0xFFFFFFFF)) >= tail0)


@pytest.mark.parametrize("kc", [32, 64])
def test_tied_rows_behind_a_lagging_warp_are_kept(kc, ws):
    """Warp 0 of every CTA inserts every row of its first tile (rising scores) while warps 1-7 fill their lists early and run
    ahead through the next tiles, where copies of one row bring the CTA's hint up to that row's score.  When warp 0 reaches
    its second tile, the copies there are the lowest-indexed rows of that score and belong to the result: `sa >= hint` must
    keep rows that equal the hint."""
    dtype, d = "fp32", 7                               # LANES 2: 16 rows per warp step, 1536-row tiles
    rng = np.random.default_rng(kc)
    q = _query(rng, d)
    T, _ = score_pool(rng, d, q, 20000)
    p = plan_gemv(d, dtype, 4 * num_sms() * 1536, kc)
    tr, grid, rpw = p["tile_rows"], p["grid"], p["rpw"]
    n = 4 * grid * tr
    assert p == plan_gemv(d, dtype, n, kc) and p["rounds"] == 4 == p["static_rounds"]
    r = np.arange(n)
    rnd, pos = r // tr // grid, r % tr
    warp0 = (pos // rpw) % 8 == 0
    s_row, low = len(T) - kc, 0                        # the tied score; kc / 2 distinct better rows sit in the last tile
    idx = np.full(n, low)
    first = rnd == 0
    idx[first & warp0] = 1 + (pos[first & warp0] // (8 * rpw)) * rpw + pos[first & warp0] % rpw   # rising, below s_row
    idx[(rnd == 1) & warp0] = s_row
    idx[(rnd >= 2) & ~warp0] = s_row
    idx[n - kc // 2:] = np.arange(len(T) - kc // 2, len(T))
    assert idx[first & warp0].max() < s_row
    ex = Exact(T, idx, q, dtype, exps=np.where(idx == s_row, rng.integers(0, 3, size=n), 0))
    want = check_keys(ex, kc, ws, what="lagging warp")
    rows = 0xFFFFFFFF - (want & np.uint64(0xFFFFFFFF)).astype(np.int64)
    assert np.all((rows[kc // 2:] // tr // grid == 1) & ((rows[kc // 2:] % tr // rpw) % 8 == 0))


# ------------------------------------------------------------------ filters, sizes, row_base --------------------------
@pytest.mark.parametrize("dtype,d", LAYOUTS)
def test_filters_that_remove_every_true_winner(dtype, d, ws):
    rng = np.random.default_rng(d)
    n, base = 20000, 700
    ex = random_exact(rng, dtype, d, n, row_base=base)
    for kc in (32, 256):
        winners = (0xFFFFFFFF - (ex.keys(kc) & np.uint64(0xFFFFFFFF))).astype(np.int64)
        others = np.setdiff1d(np.arange(n), winners)
        for length in (4096, 4097):                    # staged in shared memory / searched in global memory
            outside = np.array([0, base - 1, base + n, base + n + 12345])   # global rows outside the shard
            fill = rng.choice(others, size=length - len(winners) - len(outside), replace=False)
            excl = np.concatenate([winners, fill]) + base
            f = Filt(ex, excl=np.concatenate([excl, outside]))
            assert f.f.n_exclude == length
            got = check_keys(ex, kc, ws, f, what=f"exclusions {length}")
            assert not np.intersect1d(got, ex.keys(kc)[:kc]).size
            check_request_path(ex, kc, ws, got, f)
        bm = Filt(ex, bitmap_rows=np.union1d(winners, rng.choice(n, size=n // 3, replace=False)))
        check_keys(ex, kc, ws, bm, what="bitmap")
        genre = rng.integers(0, 1 << 20, size=n).astype(np.uint32)
        year = rng.integers(1900, 2030, size=n).astype(np.uint16)
        genre[winners] &= ~np.uint32(0b1010)
        year[winners[::2]] = 1950
        gy = Filt(ex, row_filter=RowFilter(genre_any=0b1010, year_lo=1960, year_hi=2020), genre=genre, year=year)
        assert not gy.allowed[winners].any()
        check_keys(ex, kc, ws, gy, what="genre and year")


@pytest.mark.parametrize("kc", [32, 256])
def test_tiny_shards_with_a_row_base(kc, ws):
    """n in {0, 1, kc - 1, kc, kc + 1} on a shard starting at global row 1000, exclusions inside and outside it: the fast pass
    offsets the exclusion list by row_base and the packed result carries global rows."""
    rng = np.random.default_rng(kc)
    base = 1000
    for n in (0, 1, kc - 1, kc, kc + 1):
        ex = random_exact(rng, "bf16", 100, n, row_base=base)
        excl = [base - 5, base - 1, base + n, base + n + 7] + ([base + n // 2] if n > 1 else [])
        f = Filt(ex, excl=excl)
        want = check_keys(ex, kc, ws, f, what=f"n={n}")
        assert int((want != 0).sum()) == int(f.allowed.sum())
        check_request_path(ex, kc, ws, want, f)


# ------------------------------------------------------------------ 3. selection regimes ------------------------------
def regimes(ex, kc, p, allowed):
    """An all-tied catalog on a fully static launch: no key falls below the hint, so CTA b publishes its kc lowest allowed
    rows.  Restated selection (test_selection_math._select) -> which branch select_winners takes in the last-CTA merge
    (rebert_gemv_topk, buffer merge_cap) and in the request path's cluster kernel (buffer >= 1024; kc >= 128: split)."""
    keys = ex.all_keys()
    tr, grid = p["tile_rows"], p["grid"]
    published = []
    for b in range(grid):
        rows = np.concatenate([np.arange(t * tr, min(ex.n, (t + 1) * tr)) for t in range(b, p["tiles"], grid)] or [np.zeros(0, int)])
        rows = rows[allowed[rows]][:kc]
        published.append(keys[rows])
    T, surv, out, _ = _select(published, kc)
    np.testing.assert_array_equal(out, ex.keys(kc, allowed))          # the restatement itself selects the right keys
    cnt = len(surv)

    def branch(cap):
        return "merge_all_regions" if cnt > cap else "rank" if cnt <= 512 else "sort_survivors"

    ccap = 1024
    while ccap < max(2 * kc, kc + grid):
        ccap <<= 1
    if kc >= 128:
        stage = max(3 * kc, kc + grid)
        owned = [sum(int((published[l] >= T).sum()) for l in range(grid) if l % 16 in (2 * c, 2 * c + 1)) for c in range(8)]
        fused = "stage_overflow" if max(owned) > stage else ("merge_all_regions" if cnt > ccap else "rank")
    else:
        fused = branch(ccap)
    return branch(p["merge_cap"]), fused


def test_every_selection_regime_is_reached_and_exact(ws):
    """One tile per CTA: d = 256 tiles shrink to 12 / 24 / 96 rows (partial lists: the threshold comes from the list heads
    and lets thousands of keys through); d = 100 rows are short enough for the survivors to exceed even the last-CTA merge's
    buffer; d = 50 tiles hold full lists (tight threshold)."""
    dtype = "bf16"
    rng = np.random.default_rng(3)
    sms = num_sms()
    seen_direct, seen_fused = set(), set()
    for d, rows_per_cta in ((256, 12), (256, 24), (256, 96), (100, 96), (50, 384)):
        q = _query(rng, d)
        T, _ = score_pool(rng, d, q, 50)
        for kc in KCS:
            n = sms * rows_per_cta
            p = plan_gemv(d, dtype, n, kc)
            assert p["tile_rows"] == rows_per_cta and p["rounds"] == p["static_rounds"] == 1
            ex = Exact(T[-1:], np.zeros(n, dtype=np.int64), q, dtype, exps=rng.integers(0, 3, size=n))
            excl = rng.choice(n, size=n // 10, replace=False)
            f = Filt(ex, excl=excl)
            direct, fused = regimes(ex, kc, plan_gemv(d, dtype, n, kc, len(excl)), f.allowed)
            seen_direct.add(direct)
            seen_fused.add((fused, kc >= 128))
            want = check_keys(ex, kc, ws, f, what=f"all tied n={n} ({direct})")
            check_request_path(ex, kc, ws, want, f)
    assert seen_direct == {"rank", "sort_survivors", "merge_all_regions"}
    assert {("rank", False), ("sort_survivors", False), ("merge_all_regions", False), ("rank", True),
            ("stage_overflow", True)} <= seen_fused


# ------------------------------------------------------------------ 4. the request path's selection -------------------
@pytest.mark.parametrize("dtype,d", [("bf16", 1536), ("fp32", 300)])
def test_request_path_selection_equals_the_host_keys(dtype, d, ws):
    rng = np.random.default_rng(d)
    ex = random_exact(rng, dtype, d, 30011)
    for kc in KCS:                                       # kc < 128: every CTA of the cluster selects; kc >= 128: split
        check_request_path(ex, kc, ws, check_keys(ex, kc, ws))


def test_request_path_selection_on_the_int8_shadow(ws):
    rng = np.random.default_rng(17)
    ex = i8_exact(rng, 700, 30011, row_base=5)
    check_request_path(ex, 256, ws, check_keys(ex, 256, ws, shadow=True), shadow=True)


# ------------------------------------------------------------------ 5. the margin -------------------------------------
@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
def test_margin_of_the_public_request(dtype):
    """A query of exactly 64 entries of +-1 has norm 8, so its normalised fp32 copy is exact and the fast pass can be modelled
    through recommend(): margin = exact k-th - F - 4 max|fast - exact| over the kc candidates, F = the kc-th fast score."""
    rng = np.random.default_rng(7)
    n, d, k = 20000, 100, 10
    q = np.zeros(d, dtype=np.int64)
    q[rng.choice(d, size=64, replace=False)] = rng.choice([-1, 1], size=64)
    ex = Exact(rng.integers(-8, 9, size=(n, d)), np.arange(n), q, dtype)
    rows, scores, info = ex.store.recommend(query=q.astype(np.float32), k=k, return_info=True)
    assert info["proven_exact"] and not info["prefilter"] and not info["exact_sweep"]
    kc = info["kc"]
    fast = ex.dots().astype(np.float32) * np.float32(0.125) * ex.inv
    keys = top_keys(f32_keys(fast, np.arange(n)), kc)
    cand = (0xFFFFFFFF - (keys & np.uint64(0xFFFFFFFF))).astype(np.int64)
    exact = ex.dots()[cand] * 0.125 / ex.store.norm64[:n].cpu().numpy()[cand]
    F = float(fast[cand[-1]])
    want = np.sort(exact)[::-1][k - 1] - F - 4.0 * np.abs(exact - fast[cand].astype(np.float64)).max()
    assert abs(info["margin"] - want) <= 1e-12
    want_rows, want_scores = ora.query_rows(ex.store.rows[:n, :d].to(torch.float64).cpu().numpy(), q.astype(np.float64), None, k)
    np.testing.assert_array_equal(rows, want_rows)
    np.testing.assert_allclose(scores, want_scores, rtol=1e-9)


# ------------------------------------------------------------------ 6. int8 rows with no streaming kernel -------------
@pytest.mark.parametrize("dtype,d", [("bf16", 2100), ("bf16", 4096), ("fp32", 2100)])
def test_shadow_without_a_streaming_kernel_leaves_requests_to_the_plain_path(dtype, d, ws):
    """int8 rows of 5 or 7-11 chunks per lane (d = 2049-2560, 3073-5632) have no streaming kernel: after enable_prefilter()
    single requests must still answer, from the plain path; direct calls on that shadow report UNSUPPORTED."""
    assert kernel_class(d, "i8") == ("generic",)
    n, k = 3000, 10
    store = CatalogStore.synthetic(0, n, d, dtype, scale_rows=True)
    store.enable_prefilter()
    m = store.rows[:n, :d].to(torch.float64).cpu().numpy()
    q = synth.query_f32(1, d)
    excl = np.random.default_rng(5).choice(n, size=133, replace=False)
    for prefilter in (None, True):
        rows, scores, info = store.recommend(query=q, exclude_rows=excl, k=k, return_info=True, prefilter=prefilter)
        assert info["prefilter"] is False
        want_rows, want_scores = ora.query_rows(m, q.astype(np.float64), excl, k)
        np.testing.assert_array_equal(rows, want_rows)
        np.testing.assert_allclose(scores, want_scores, rtol=1e-9)
    (rated, rts), = synth.user_ratings(2, n, 1)
    liked = rated[rts >= 3.5] if (rts >= 3.5).any() else rated[:1]
    rows, scores, info = store.recommend(liked_rows=liked, exclude_rows=rated, k=k, return_info=True)
    assert info["prefilter"] is False
    want_rows, want_scores = ora.recommend_rows(m, liked, rated, k)
    np.testing.assert_array_equal(rows, want_rows)
    np.testing.assert_allclose(scores, want_scores, rtol=1e-9)
    lib = nat.load()
    s = store._scratch()
    cand = torch.zeros(256, dtype=torch.int64, device=DEV)
    assert lib.rebert_gemv_topk(C.byref(store._c8), s.qn32.data_ptr(), C.byref(nat.Filter()), 256, ws.data_ptr(), ws.numel(),
                                cand.data_ptr(), _stream()) == nat.ERR_UNSUPPORTED
    out = torch.zeros(2 * k + 2, dtype=torch.int64, device=DEV)
    assert lib.rebert_recommend_device(C.byref(store._c), C.byref(store._c8), s.qn32.data_ptr(), s.qn64.data_ptr(),
                                       C.byref(nat.Filter()), k, 256, ws.data_ptr(), ws.numel(), out.data_ptr(), 0, None, None,
                                       _stream()) == nat.ERR_UNSUPPORTED
