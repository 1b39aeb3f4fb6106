"""Plans of the batched tensor-core path for long lists (241 <= k <= 2048), on the CPU.

rebert_gemm_plan / rebert_gemm_plan_i8 give k > 240 its own regime: sample rank 64 and a survivor target
E = max(3 kc, 50 x 64) per query.  Under the Gamma(rank) model of the survivor count (the rank-th best of a random sample of
S rows leaves Gamma(rank, n / S) rows above it), the probability that fewer than kc rows pass is gammainc(64, 64 kc / E),
and the sample costs S / n of the full GEMM's flops.  Plans for k <= 240 must stay exactly as recorded before the regime
was added (tests/golden/gemm_plans_k240.json: every k in 1..240 at four catalog sizes, b = 4096).
"""
import ctypes as C
import json
import os

import numpy as np
import pytest
from scipy.special import gammainc

from robot_ebert_b200 import _native as nat

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "gemm_plans_k240.json")
PLANS = {"bf16": "rebert_gemm_plan", "int8": "rebert_gemm_plan_i8"}
SAMPLE_FLOPS_MAX = 0.02       # sample GEMM / full GEMM
TAIL_MAX = 1e-9               # P(fewer than kc survivors)


def _plan(which, n, b, k):
    lib = nat.load()
    p = nat.GemmPlan()
    rc = getattr(lib, PLANS[which])(n, b, k, C.byref(p))
    return rc, p


def _kc(which, k):
    need = max(k + 16, k + (k + 3) // 4) if which == "bf16" else k + max(k, 64)
    return (need + 31) // 32 * 32


def _min_rows(which, k):
    return int(64 * max(3 * _kc(which, k), 50 * 64))


@pytest.mark.parametrize("which", ["bf16", "int8"])
@pytest.mark.parametrize("k", [241, 256, 500, 1000, 2048])
@pytest.mark.parametrize("n_over", [1.0, 1.7, 40.0])
def test_long_list_plan(which, k, n_over):
    n = int(_min_rows(which, k) * n_over) + 13
    rc, p = _plan(which, n, 4096, k)
    assert rc == nat.OK, nat.load().rebert_last_error()
    assert (p.b, p.k, p.kc) == (4096, k, _kc(which, k))
    assert p.kc <= (2560 if which == "bf16" else 4096)
    assert p.sample_rank == 64
    assert p.sample_rows % 256 == 0 and p.sample_rows > 0
    tiles = (n + 255) // 256
    frac = p.sample_rows / (tiles * 256.0)
    assert frac <= SAMPLE_FLOPS_MAX, frac
    e = p.sample_rank * n / p.sample_rows          # expected survivors per query
    assert e >= 3 * p.kc
    tail = gammainc(p.sample_rank, p.sample_rank * p.kc / e)
    assert tail <= TAIL_MAX, tail
    # the candidate buffer: 2 kc doubled until it holds 4 x the survivor target
    e_target = max(3 * p.kc, 50 * 64)
    steps = p.cand_cap // (2 * p.kc)
    assert p.cand_cap % (2 * p.kc) == 0 and steps & (steps - 1) == 0
    assert p.cand_cap >= 4 * e_target and (steps == 1 or p.cand_cap // 2 < 4 * e_target)


@pytest.mark.parametrize("which", ["bf16", "int8"])
def test_k_above_2048_is_unsupported(which):
    for k in (2049, 5000):
        rc, _ = _plan(which, 10_000_000, 64, k)
        assert rc == nat.ERR_UNSUPPORTED


@pytest.mark.parametrize("which", ["bf16", "int8"])
@pytest.mark.parametrize("k", [241, 1000, 2048])
def test_too_small_catalog_is_refused(which, k):
    n = _min_rows(which, k)
    rc, _ = _plan(which, n - 1, 64, k)
    assert rc == nat.ERR_UNSUPPORTED and b"too small" in nat.load().rebert_last_error()
    rc, _ = _plan(which, n, 64, k)
    assert rc == nat.OK


def test_plans_up_to_k240_are_unchanged():
    with open(GOLDEN) as f:
        g = json.load(f)
    assert g["fields"] == [f for f, _ in nat.GemmPlan._fields_]
    checked = 0
    for key, rows in g["plans"].items():
        fn, n = key.split(":")
        which = "bf16" if fn == "rebert_gemm_plan" else "int8"
        for k, want in enumerate(rows, start=1):
            rc, p = _plan(which, int(n), 4096, k)
            assert rc == want[0], (key, k)
            if rc == nat.OK:
                assert [getattr(p, f) for f in g["fields"]] == want[1:], (key, k)
            checked += 1
    assert checked == 2 * 4 * 240


def test_workspace_at_b4096_k2048():
    """The numbers DESIGN.md §4.3 quotes: workspace of the largest plans at b = 4096 over 1M rows."""
    lib = nat.load()
    got = {}
    for which in PLANS:
        rc, p = _plan(which, 1 << 20, 4096, 2048)
        assert rc == nat.OK
        ws = lib.rebert_gemm_workspace_bytes(None, C.byref(p))
        a = lambda x: (x + 255) // 256 * 256
        want = (a(4096 * p.sample_rows * 4) + 2 * a(4096 * 4) + a(4096 * p.cand_cap * 8) + a(4096 * p.kc * 8) + a(4096 * 8) + 256)
        assert ws == want
        got[which] = ws
    assert got["bf16"] < 1.6 * 2 ** 30 and got["int8"] < 2.4 * 2 ** 30


# numpy restatement of select_candidates_large_kernel's bucket arithmetic (csrc/gemm_topk.cu)
BUCKETS = 2048


def _bucket(hi32, lo, range_):
    return ((hi32.astype(np.uint64) - np.uint64(lo)) * np.uint64(BUCKETS)) // np.uint64(range_)


def _select_restated(keys, kc):
    """Returns (sorted best kc keys or None when the gathered set does not fit, gathered count)."""
    gather_cap = 2
    while gather_cap < 2 * kc:
        gather_cap <<= 1
    valid = keys[keys != 0]
    hi32 = (valid >> np.uint64(32)).astype(np.uint64)
    lo, hi = (int(hi32.min()), int(hi32.max())) if len(valid) else (0xFFFFFFFF, 0)
    range_ = (hi - lo) + 1 if len(valid) else 2
    m, bstar = len(valid), 0
    if len(valid) > gather_cap and hi > lo:
        hist = np.bincount(_bucket(hi32, lo, range_).astype(np.int64), minlength=BUCKETS)
        cum = np.cumsum(hist[::-1])
        j = int(np.argmax(cum >= kc))
        bstar, m = BUCKETS - 1 - j, int(cum[j])
    elif len(valid) > gather_cap:
        m = len(valid)
    if m > gather_cap:
        return None, m
    top = valid[_bucket(hi32, lo, range_) >= bstar] if len(valid) else valid
    assert len(top) == m
    return np.sort(top)[::-1][:kc], m


@pytest.mark.parametrize("kc", [320, 1280, 4096])
def test_bucket_select_restatement_keeps_the_best_kc(kc):
    rng = np.random.default_rng(kc)
    for spread in (1e-1, 1e-3, 1e-6):
        scores = (0.3 + spread * rng.standard_normal(3 * kc)).astype(np.float32)
        bits = scores.view(np.uint32).astype(np.uint64) | np.uint64(0x80000000)     # positive floats: orderable form
        rows = rng.choice(1 << 20, size=len(scores), replace=False).astype(np.uint64)
        keys = (bits << np.uint64(32)) | (np.uint64(0xFFFFFFFF) - rows)
        keys[rng.choice(len(keys), size=kc // 4, replace=False)] = 0                  # excluded rows
        got, m = _select_restated(keys, kc)
        assert got is not None and m <= 2 * kc + kc
        np.testing.assert_array_equal(got, np.sort(keys[keys != 0])[::-1][:kc])


def test_bucket_select_restatement_flags_mass_ties():
    kc = 320
    keys = (np.uint64(0xBE99999A) << np.uint64(32)) | (np.uint64(0xFFFFFFFF) - np.arange(4 * kc, dtype=np.uint64))
    got, m = _select_restated(keys, kc)
    assert got is None and m == 4 * kc      # status bit 16: the caller re-runs the query, no key is dropped silently
