"""Exact restatement of the single-query int8 score S (csrc/gemv_topk.cu: i8_steps, quant_planes, i8_dot4 / i8_dot4_32,
i8_score), the number every int8 path of the single-query kernel computes: the prefilter shadow, the gate, the gate's seed.

The query is split into two int8 planes, q ~ dh * h + dl * l with dl = dh / 254, each row is scored against both with exact
integer sums (hs, ls), and S = fmaf(dh, (float)hs, dl * (float)ls) * factor.  Every step here rounds where the kernel rounds
and nowhere else, so S comes out bit for bit:
  * dh = fl32(max|q[:d]| / 127) (1 for the zero query), dl = fl32(dh / 254);
  * h = clamp(rint_even(fl32(q / dh)), +-127);
  * l = clamp(rint_even(fl32(r / dl)), +-127) with r = fl32(q - h * dh) rounded ONCE (quant_planes forms it with fmaf);
  * hs, ls: integer dot products against the device's own int8 rows (a float64 GEMM of int8 values is exact: every partial
    sum is an integer far below 2^53);
  * (float)hs, (float)ls round to nearest; c = fl32(dl * fl32(ls)); fmaf(dh, fl32(hs), c) is emulated exactly (fmaf32);
  * finally one fp32 multiply by the row's factor.
"""
import numpy as np


def fmaf32(a, b, c):
    """fmaf on fp32 arrays, exactly: a * b is exact in float64 (24 + 24 bits); the float64 sum is taken with round-to-odd
    (TwoSum gives its error; an inexact sum with an even last bit steps one ulp toward the error), and rounding that to fp32
    is the correctly rounded a * b + c because 53 >= 2 * 24 + 2."""
    a, b, c = (np.asarray(x, dtype=np.float32).astype(np.float64) for x in (a, b, c))
    p = a * b
    s = p + c
    bb = s - p
    err = (p - (s - bb)) + (c - bb)
    even = (np.asarray(s).view(np.int64) & 1) == 0
    toward = np.where(err > 0, np.inf, -np.inf)
    s = np.where((err != 0) & even, np.nextafter(s, toward), s)
    return np.asarray(s).astype(np.float32)


def query_planes(q, d=None):
    """(dh, dl, h, l) of the query exactly as the kernel reads it: fp32, zero past d.  h and l cover the whole buffer."""
    q = np.asarray(q, dtype=np.float32)
    d = len(q) if d is None else d
    qv = q.copy()
    qv[d:] = 0
    qmax = np.float32(np.abs(qv[:d]).max()) if d else np.float32(0)
    dh = np.float32(qmax / np.float32(127)) if qmax > 0 else np.float32(1)
    dl = np.float32(dh / np.float32(254))
    h = np.clip(np.rint(qv / dh), -127, 127)
    r = (qv.astype(np.float64) - h.astype(np.float64) * np.float64(dh)).astype(np.float32)   # one rounding (fmaf)
    l = np.clip(np.rint(r / dl), -127, 127)
    return dh, dl, h.astype(np.int32), l.astype(np.int32)


def plane_sums(rows8, h, l, chunk=1 << 15):
    """Exact (hs, ls) of int8 rows [n, ld8] against the planes (zero-extended or cut to ld8), as float64 integers."""
    rows8 = np.asarray(rows8)
    ld8 = rows8.shape[1]
    planes = np.zeros((ld8, 2), dtype=np.float64)
    m = min(ld8, len(h))
    planes[:m, 0], planes[:m, 1] = h[:m], l[:m]
    out = np.empty((rows8.shape[0], 2), dtype=np.float64)
    for s in range(0, rows8.shape[0], chunk):
        out[s:s + chunk] = rows8[s:s + chunk].astype(np.float64) @ planes
    return out[:, 0], out[:, 1]


def score_from_sums(dh, dl, hs, ls, factor):
    """i8_score: fmaf(dh, (float)hs, dl * (float)ls) * factor, in fp32."""
    fhs = np.asarray(hs, dtype=np.float64).astype(np.float32)
    fls = np.asarray(ls, dtype=np.float64).astype(np.float32)
    c = (np.float32(dl) * fls).astype(np.float32)
    return (fmaf32(dh, fhs, c) * np.asarray(factor, dtype=np.float32)).astype(np.float32)


def int8_scores(rows8, factor, q, d=None):
    """S of every int8 row [n, ld8] with its fp32 factor [n] (the shadow's inv_norm / the gate's factor) against the fp32
    query q (zero past d)."""
    dh, dl, h, l = query_planes(q, d)
    hs, ls = plane_sums(rows8, h, l)
    return score_from_sums(dh, dl, hs, ls, np.asarray(factor, dtype=np.float32)[:len(hs)])


def round_up_f32(x):
    """__double2float_ru."""
    f = np.float32(x)
    return np.nextafter(f, np.float32(np.inf)) if float(f) < x else f


def gate_delta(q, d, row_err, epl):
    """gemv_topk.cu gate_delta for the query the kernel is passed: ||q||, the real error of its two planes, the gate rows'
    row error and the record's elements per lane, rounded up to fp32."""
    q = np.asarray(q, dtype=np.float32)[:d]
    dh, dl, h, l = query_planes(q)
    r = q.astype(np.float64) - (np.float64(dh) * h + np.float64(dl) * l)
    qn, eq = np.sqrt((q.astype(np.float64) ** 2).sum()), np.sqrt((r ** 2).sum())
    u = 2.0 ** -24
    shadow = row_err * (qn + eq) + eq + 32.0 * u * (1.0 + row_err) * (qn + eq)
    fast = (epl + 12) * u * qn
    return round_up_f32((shadow + fast) * (1.0 + 1e-6) + 1e-6 * qn + 1e-30)
