"""CPU: the exact int8 score model (tests/int8_score_model.py) against exact rational arithmetic."""
from fractions import Fraction

import numpy as np
import pytest

from tests.int8_score_model import fmaf32, query_planes, score_from_sums


def f32_round(x: Fraction) -> np.float32:
    """x rounded to the nearest fp32, ties to even (float(x) is within one fp32 ulp of it: check the neighbours)."""
    f = np.float32(float(x))
    cands = [np.nextafter(f, np.float32(-np.inf)), f, np.nextafter(f, np.float32(np.inf))]
    dist = [abs(Fraction(float(c)) - x) for c in cands]
    best = min(dist)
    tied = [c for c, e in zip(cands, dist) if e == best]
    if len(tied) == 1:
        return tied[0]
    return next(c for c in tied if (np.array(c, dtype=np.float32).view(np.uint32) & 1) == 0)


def fma_ref(a, b, c):
    return f32_round(Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c)))


def _same(x, y):
    return np.array(x, dtype=np.float32).view(np.uint32) == np.array(y, dtype=np.float32).view(np.uint32)


def test_fmaf32_on_random_inputs():
    rng = np.random.default_rng(0)
    n = 3000
    a = (rng.standard_normal(n) * np.exp2(rng.integers(-20, 20, n))).astype(np.float32)
    b = (rng.standard_normal(n) * np.exp2(rng.integers(-20, 20, n))).astype(np.float32)
    c = (rng.standard_normal(n) * np.exp2(rng.integers(-40, 40, n))).astype(np.float32)
    c[::3] = (-(a[::3].astype(np.float64) * b[::3]) * (1 + rng.standard_normal(len(c[::3])) * 1e-6)).astype(np.float32)  # cancellation
    got = fmaf32(a, b, c)
    for i in range(n):
        assert _same(got[i], fma_ref(a[i], b[i], c[i])), (a[i], b[i], c[i])


def test_fmaf32_on_halfway_cases():
    """a * b = 1 + 2^-11 + 2^-24 lies exactly half way between two fp32 values; a tiny c decides the rounding.  A float64
    sum rounds the tail away and then ties to even: one rounding too many.  The model must not."""
    a = np.float32(1 + 2.0 ** -12)
    naive_wrong = 0
    cases = 0
    for scale in (1.0, 2.0 ** -30, 2.0 ** 40):
        for sign in (1.0, -1.0):
            for b in (np.float32(1 + 2.0 ** -12), np.float32(1 + 2.0 ** -12 + 2.0 ** -23)):
                for tail in (0.0, 2.0 ** -80, -(2.0 ** -80), 2.0 ** -60, -(2.0 ** -60)):
                    aa = np.float32(sign * scale * a)
                    cc = np.float32(sign * scale * tail)
                    want = fma_ref(aa, b, cc)
                    assert _same(fmaf32(aa, b, cc), want), (aa, b, cc)
                    naive_wrong += not _same(np.float32(np.float64(aa) * np.float64(b) + np.float64(cc)), want)
                    cases += 1
    assert cases == 60 and naive_wrong >= 12             # the cases do reach the double-rounding trap


def test_score_from_sums_rounds_like_the_kernel():
    rng = np.random.default_rng(1)
    n = 2000
    dh = np.float32(rng.uniform(1e-4, 1e-1))
    dl = np.float32(dh / np.float32(254))
    hs = rng.integers(-(1 << 28), 1 << 28, n)              # beyond 2^24: (float)hs rounds
    ls = rng.integers(-(1 << 28), 1 << 28, n)
    fac = rng.uniform(1e-3, 1.0, n).astype(np.float32)
    got = score_from_sums(dh, dl, hs, ls, fac)
    for i in range(0, n, 7):
        c = f32_round(Fraction(float(dl)) * Fraction(float(f32_round(Fraction(int(ls[i]))))))
        s = f32_round(Fraction(float(dh)) * Fraction(float(f32_round(Fraction(int(hs[i]))))) + Fraction(float(c)))
        assert _same(got[i], f32_round(Fraction(float(s)) * Fraction(float(fac[i]))))


def test_query_planes_reconstruct_the_query_and_use_the_fused_residual():
    rng = np.random.default_rng(2)
    d, differ = 1536, 0
    for t in range(200):
        q = rng.standard_normal(d)
        q = (q / np.linalg.norm(q)).astype(np.float32)
        dh, dl, h, l = query_planes(q)
        assert np.abs(h).max() <= 127 and np.abs(l).max() <= 127 and np.abs(h).max() == 127
        err = np.abs(q.astype(np.float64) - (np.float64(dh) * h + np.float64(dl) * l))
        assert err.max() <= 0.5 * float(dl) * (1 + 1e-5)
        # the residual rounded twice (q - fl(h * dh)) gives other low-plane values for some queries: the model must not use it
        r2 = (q - (h.astype(np.float32) * dh).astype(np.float32)).astype(np.float32)
        differ += not np.array_equal(np.clip(np.rint(r2 / dl), -127, 127).astype(np.int32), l)
    assert differ > 0


@pytest.mark.parametrize("d", [1, 20, 1536])
def test_query_planes_of_the_zero_query_and_padding(d):
    q = np.zeros(d + 64, dtype=np.float32)
    dh, dl, h, l = query_planes(q, d)
    assert dh == 1 and dl == np.float32(1) / np.float32(254) and not h.any() and not l.any()
    q[d:] = 5.0                                           # past d the kernel reads zero
    q[0] = -0.25
    dh, dl, h, l = query_planes(q, d)
    assert dh == np.float32(np.float32(0.25) / np.float32(127)) and h[0] == -127 and not h[d:].any() and not l[d:].any()
