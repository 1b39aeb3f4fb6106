"""CPU: the gate's delta (csrc/gemv_topk.cu gate_delta, DESIGN.md §4.5) restated in numpy.

The gated fast pass skips a row when its int8 score S falls below L - delta, L a lower bound of the kc-th best fp32 fast
score F.  That is sound only if S >= F - delta for every row and every query the kernel may be passed (also non-unit
ones).  Here the int8 rows, the two query planes, S and F are formed the way the kernels form them (rebert_catalog_quantize_i8,
S bit for bit from tests/int8_score_model.py, the per-lane fmaf chains and the xor-shuffle tree of the plain kernel, delta
rounded up as gate_delta rounds it), and the inequality is checked
for every row over gaussian, scaled, spiky, one-hot and non-unit queries and catalogs with a dominant column.
"""
import zlib

import numpy as np
import pytest

from tests import int8_score_model as model

def quantize_rows(x):
    """rebert_catalog_quantize_i8: int8 rows, fp32 factor, max relative row error (fp64)."""
    mx = np.abs(x).max(axis=1).astype(np.float32)
    scale = np.where(mx > 0, mx / np.float32(127), np.float32(1)).astype(np.float32)
    q8 = np.clip(np.rint(x / scale[:, None]), -127, 127).astype(np.int32)
    err = np.sqrt(((x.astype(np.float64) - q8 * scale[:, None].astype(np.float64)) ** 2).sum(axis=1))
    nrm = np.sqrt((x.astype(np.float64) ** 2).sum(axis=1))
    nrm = np.where(nrm > 0, nrm, 1.0)
    factor = (scale.astype(np.float64) / nrm).astype(np.float32)
    return q8, factor, float((err / nrm).max()), (1.0 / nrm).astype(np.float32)


def query_planes(q):
    """The consumers' planes: q ~ dh * h + dl * l (gemv_topk.cu quant_planes, residual rounded once)."""
    return model.query_planes(q)


def shadow_scores(q8, factor, dh, dl, h, l):
    """S bit for bit (tests/int8_score_model.py)."""
    hs, ls = model.plane_sums(q8, h, l)
    return model.score_from_sums(dh, dl, hs, ls, factor)


def fast_scores(x, q, inv, epc):
    """The plain kernel's fp32 score: lane c holds chunks j*32 + c, chunk j accumulates into a[j & 1] with fmaf in
    element order, then a0 + a1, the xor-shuffle tree over 32 lanes, times inv_norm."""
    n, ld = x.shape
    cpl = ld // (32 * epc)
    xv = x.reshape(n, cpl, 32, epc)
    qv = q.reshape(cpl, 32, epc)
    acc = np.zeros((2, n, 32), dtype=np.float32)
    for j in range(cpl):
        for e in range(epc):
            acc[j & 1] = model.fmaf32(xv[:, j, :, e], qv[j, :, e], acc[j & 1])
    s = (acc[0] + acc[1]).astype(np.float32)
    o = 16
    while o:
        s = (s + s[:, np.arange(32) ^ o]).astype(np.float32)
        o >>= 1
    return (s[:, 0] * inv).astype(np.float32)


def catalog(kind, rng, n, d):
    x = rng.standard_normal((n, d)).astype(np.float32)
    if kind == "scaled":
        x *= rng.uniform(0.01, 100.0, size=(n, 1)).astype(np.float32)
    elif kind == "dominant_column":
        x[:, 0] += 60.0
    elif kind == "shared_mean":                        # rows ~0.7 cosine apart, like text-embedding catalogs
        m = rng.standard_normal(d)
        m /= np.linalg.norm(m)
        x = (np.sqrt(0.7) * m + np.sqrt(0.3) * x / np.sqrt(d)).astype(np.float32)
    return x


def query(kind, rng, d):
    g = rng.standard_normal(d)
    if kind == "gauss":
        q = g / np.linalg.norm(g)
    elif kind == "scaled_up":
        q = 7.5 * g / np.linalg.norm(g)
    elif kind == "scaled_down":
        q = 1e-3 * g / np.linalg.norm(g)
    elif kind == "spiky":
        q = 0.01 * g
        q[rng.integers(d)] = 3.0
        q /= np.linalg.norm(q)
    elif kind == "one_hot":
        q = np.zeros(d)
        q[rng.integers(d)] = 1.0
    else:                                              # non-unit, uneven magnitudes
        q = g * rng.uniform(0, 4, size=d)
    return q.astype(np.float32)


@pytest.mark.parametrize("dtype,d", [("bf16", 300), ("fp32", 700), ("bf16", 1536), ("fp32", 1536)])
@pytest.mark.parametrize("rows", ["gauss", "scaled", "dominant_column", "shared_mean"])
@pytest.mark.parametrize("qkind", ["gauss", "scaled_up", "scaled_down", "spiky", "one_hot", "non_unit"])
def test_shadow_never_falls_below_fast_minus_delta(dtype, d, rows, qkind):
    rng = np.random.default_rng(zlib.crc32(f"{dtype}{d}{rows}{qkind}".encode()))
    n = 600
    epc = 8 if dtype == "bf16" else 4
    ld = -(-d // (32 * epc)) * 32 * epc
    x = np.zeros((n, ld), dtype=np.float32)
    x[:, :d] = catalog(rows, rng, n, d)
    if dtype == "bf16":                               # stored values are bf16 (round to nearest even)
        b = x.view(np.uint32)
        x = ((b + 0x7FFF + ((b >> 16) & 1)) & 0xFFFF0000).astype(np.uint32).view(np.float32)
    q = np.zeros(ld, dtype=np.float32)
    q[:d] = query(qkind, rng, d)
    q8, factor, row_err, inv = quantize_rows(x[:, :d])
    dh, dl, h, l = query_planes(q[:d])
    delta = float(model.gate_delta(q, d, row_err, (ld // 32 // epc) * epc))
    S = shadow_scores(q8, factor, dh, dl, h, l).astype(np.float64)
    F = fast_scores(x, q, inv, epc).astype(np.float64)
    gap = F - S
    assert gap.max() <= delta, (gap.max(), delta)
    # delta is a bound, not a guess: the worst row uses a fair share of it (rows x query error, not slack alone)
    assert delta < 0.5 * np.sqrt((q.astype(np.float64) ** 2).sum()) + 1e-6
