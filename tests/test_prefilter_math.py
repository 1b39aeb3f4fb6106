"""CPU check of the int8 prefilter's error bound (the arithmetic of quantize_i8_kernel restated in numpy, the shadow score S
bit for bit from tests/int8_score_model.py): |S - true cosine| never exceeds the bound CatalogStore.enable_prefilter adds to
the proof margin."""
import numpy as np
import pytest

from tests import int8_score_model as model


def _quantize_rows(x, nrm=None):
    """x: fp32 rows [n, d]; nrm: fp64 row norms (zero -> 1), recomputed here when not given."""
    mx = np.abs(x).max(axis=1).astype(np.float32)
    scale = np.where(mx > 0, mx / np.float32(127), np.float32(1)).astype(np.float32)
    q8 = np.clip(np.rint(x / scale[:, None]), -127, 127).astype(np.int32)
    if nrm is None:
        nrm = np.linalg.norm(x.astype(np.float64), axis=1)
        nrm[nrm == 0] = 1.0
    err = np.linalg.norm(x.astype(np.float64) - q8 * scale[:, None].astype(np.float64), axis=1) / nrm
    factor = (scale.astype(np.float64) / nrm).astype(np.float32)
    return q8, factor, err.max()


@pytest.mark.parametrize("d", [1, 7, 32, 50, 768, 1536])
@pytest.mark.parametrize("kind", ["gauss", "scaled", "spiky", "onehot_query"])
def test_shadow_score_error_is_within_the_proven_bound(d, kind):
    rng = np.random.default_rng(d * 7 + len(kind))
    n = 400
    x = rng.standard_normal((n, d)).astype(np.float32)
    if kind == "scaled":
        x *= (10.0 ** rng.integers(-4, 5, size=(n, 1))).astype(np.float32)
    if kind == "spiky":
        x[::3, rng.integers(0, d)] = 300.0
    x[5] = 0.0                                                   # an all-zero row scores 0 in both worlds
    q = rng.standard_normal(d).astype(np.float64)
    if kind == "onehot_query":
        q[:] = 1e-3 * q
        q[rng.integers(0, d)] = 1.0
    qn = (q / np.linalg.norm(q)).astype(np.float32)              # what query_normalize hands the kernel
    q8, factor, row_err = _quantize_rows(x)
    dh, dl, hi, lo = model.query_planes(qn)
    shadow = model.int8_scores(q8, factor, qn)                    # S bit for bit, as the kernel forms it
    nrm = np.linalg.norm(x.astype(np.float64), axis=1)
    nrm[nrm == 0] = 1.0
    true = (x.astype(np.float64) @ qn.astype(np.float64)) / nrm
    query_err = np.sqrt(d) / (127.0 * 254.0 * 2.0)
    bound = row_err + 1.01 * (1.0 + row_err) * query_err + 4e-6  # CatalogStore.enable_prefilter's q8_eps
    assert np.abs(shadow.astype(np.float64) - true).max() <= bound
    assert np.abs(q8).max() <= 127 and np.abs(hi).max() <= 127 and np.abs(lo).max() <= 127
    # the int32 accumulators cannot overflow: d * 127 * 127 < 2^31 up to d = 133k (rows are <= 12 KB)
    assert 12288 * 127 * 127 < 2 ** 31
