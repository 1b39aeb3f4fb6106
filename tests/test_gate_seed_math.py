"""numpy restatement of the gate's seed (gemv_topk.cu: gate_seed_kernel, DESIGN.md §4.5).

The seed scores a strided sample of the int8 rows (S), keeps the best allowed rows by S per warp and per CTA, takes the kc
best of what the CTAs kept, and writes the smallest fast score F of those kc rows as a lower bound of the final kc-th best
fast score.  Whatever S says, the bound is reached by kc distinct allowed rows, so it never exceeds the kc-th best F of
the allowed rows; with fewer than kc rows to choose from there is no bound.
"""
import numpy as np
import pytest

GRID, WARPS = 148, 8


def orderable(f):
    b = np.asarray(f, dtype=np.float32).view(np.uint32).astype(np.uint64)
    return np.where(b & 0x80000000, ~b & 0xFFFFFFFF, b | 0x80000000)


def make_keys(s, rows):
    return (orderable(s) << np.uint64(32)) | (np.uint64(0xFFFFFFFF) - rows.astype(np.uint64))


def seed_rows(n):
    m = min(max(n // 64, 16384), 131072)
    m = min(m, n)
    return np.arange(m, dtype=np.int64) * (n // m)


def seed_bound(S, F, allowed, kc, grid=GRID):
    """(bound, rows it was taken from) or (None, None)."""
    n = S.size
    rows = seed_rows(n)
    P = min(32, 2 * -(-kc // grid))
    W = grid * WARPS
    idx = np.arange(rows.size)
    ok = allowed[rows]
    rows, idx = rows[ok], idx[ok]
    keys = make_keys(S[rows], rows)
    warp = idx % W
    kept = []
    for c in range(grid):                               # each warp's P best, then the CTA's P best of those
        cta = []
        for w in range(c * WARPS, (c + 1) * WARPS):
            kw = np.sort(keys[warp == w])[::-1][:P]
            cta.extend(kw.tolist())
        kept.extend(sorted(cta, reverse=True)[:P])
    if len(kept) < kc:
        return None, None
    best = np.sort(np.array(kept, dtype=np.uint64))[::-1][:kc]
    sel = (np.uint64(0xFFFFFFFF) - (best & np.uint64(0xFFFFFFFF))).astype(np.int64)
    return float(F[sel].min()), sel


def kth_best(F, allowed, kc):
    f = np.sort(F[allowed])[::-1]
    return f[kc - 1] if f.size >= kc else None


def test_sample_sizes():
    assert seed_rows(10_000_000).size == 131072 and seed_rows(10_000_000)[-1] == 131071 * 76
    assert seed_rows(1_000_000).size == 16384 and seed_rows(40_000).size == 16384
    assert seed_rows(300).size == 300
    for n in (1, 16385, 999_999, 8_388_607, 50_000_000):
        r = seed_rows(n)
        assert r[-1] < n and np.all(np.diff(r) > 0)


@pytest.mark.parametrize("kc", [32, 64, 128, 256])
@pytest.mark.parametrize("case", ["gauss", "s_reversed", "ties", "most_excluded"])
def test_bound_is_reached_by_kc_allowed_rows(kc, case):
    rng = np.random.default_rng(kc)
    n = 60_000
    F = rng.standard_normal(n).astype(np.float32)
    S = (F + 0.05 * rng.standard_normal(n)).astype(np.float32)
    allowed = rng.random(n) > 0.1
    if case == "s_reversed":                            # the int8 order says nothing about the fast score
        S = -F
    elif case == "ties":                                # whole blocks of rows with the same score
        F = np.round(F * 4).astype(np.float32) / 4
        S = F.copy()
    elif case == "most_excluded":
        allowed[seed_rows(n)[rng.random(seed_rows(n).size) > 0.02]] = False
    bound, sel = seed_bound(S, F, allowed, kc)
    assert bound is not None
    assert np.unique(sel).size == kc and allowed[sel].all()
    assert np.count_nonzero(F[allowed] >= bound) >= kc
    assert bound <= kth_best(F, allowed, kc)


@pytest.mark.parametrize("kc", [32, 256])
def test_no_bound_from_fewer_than_kc_rows(kc):
    rng = np.random.default_rng(3)
    n = 40_000
    F = rng.standard_normal(n).astype(np.float32)
    allowed = np.ones(n, dtype=bool)
    s = seed_rows(n)
    allowed[s] = False
    allowed[s[8 * np.arange(kc - 1)]] = True           # one row per CTA
    assert seed_bound(F, F, allowed, kc) == (None, None)
    allowed[s[8 * (kc - 1)]] = True
    assert seed_bound(F, F, allowed, kc)[0] is not None
    assert seed_bound(F[:kc - 1], F[:kc - 1], np.ones(kc - 1, dtype=bool), kc) == (None, None)
