"""The gate's seed as the prologue of the gated kernel (DESIGN.md §4.5): every CTA scores its share of the sample, the last
one forms the bound, and the others wait for it (bounded) before they stream.  Gated requests must equal the plain pass
bit for bit (packed result, candidate keys, the same seed word from both entry points) and the float64 oracle on:
  * a crowded shared-mean catalog with a forced gate, where most rows pass the gate test;
  * a shard where fewer than kc sampled rows are allowed, so the seed writes no bound and the waiting CTAs go on without it;
  * a catalog whose gated grid is smaller than the SM count, where gate_seed_kernel still runs ahead of the gated kernel;
  * int8 rows of 6 chunks per lane (d = 3000), which keep gate_seed_kernel too.
"""
import numpy as np
import pytest
import torch

from robot_ebert_b200 import CatalogStore, synth
from robot_ebert_b200 import _native as nat
from tests.test_gpu_gate_edges import DEV, check, num_sms, oracle_check, seed_rows

pytestmark = pytest.mark.gpu


def shared_mean(store, seed, cos=0.7):
    """Rows and a query around one shared unit direction (pairwise cosine ~cos), norms recomputed."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    d = store.d
    m = torch.randn(d, generator=g, device=DEV)
    m /= m.norm()
    noise = torch.randn((store.n, d), generator=g, device=DEV) / np.sqrt(d)
    store.rows[:store.n, :d] = (np.sqrt(cos) * m + np.sqrt(1 - cos) * noise).to(store.rows.dtype)
    nat.check(nat.load().rebert_catalog_norms(store.rows.data_ptr(), store.n, store.ld, nat.DTYPES[store.dtype],
                                              store.inv_norm.data_ptr(), store.norm64.data_ptr(),
                                              torch.cuda.current_stream().cuda_stream))
    torch.cuda.current_stream().synchronize()
    q = np.sqrt(cos) * m + np.sqrt(1 - cos) * torch.randn(d, generator=g, device=DEV) / np.sqrt(d)
    return q.cpu().numpy().astype(np.float32)


@pytest.mark.parametrize("k", [10, 240])
def test_crowded_catalog_forced_gate(k):
    st = CatalogStore.synthetic(3, 400_000, 1536, "bf16", device=DEV)
    q = shared_mean(st, 11)
    excl = np.sort(np.random.default_rng(1).choice(st.n, size=133, replace=False))
    word, _, packed = check(st, k, query=q, excl=excl)
    assert word != 0
    oracle_check(st, packed, k, q=q, excl=excl)


def test_no_bound_when_few_sampled_rows_are_allowed():
    """Every sampled row excluded: no bound (word 21 stays 0), and the CTAs that waited for it still stream every row."""
    st = CatalogStore.synthetic(4, 300_000, 1536, "bf16", device=DEV)
    q = synth.query_f32(5, st.d)
    excl = seed_rows(st.n)
    word, _, packed = check(st, 10, query=q, excl=excl)
    assert word == 0
    oracle_check(st, packed, 10, q=q, excl=excl)


@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
def test_standalone_seed_on_a_small_grid(dtype):
    """Fewer int8 tiles than SMs (32 rows a tile at d = 1536): the gated grid is smaller than the SM count."""
    n = 32 * (num_sms() // 2)
    st = CatalogStore.synthetic(6, n, 1536, dtype, device=DEV)
    q = synth.query_f32(7, st.d)
    _, _, packed = check(st, 10, query=q)
    oracle_check(st, packed, 10, q=q)


def test_standalone_seed_for_six_chunk_rows():
    st = CatalogStore.synthetic(8, 200_000, 3000, "bf16", device=DEV)
    q = synth.query_f32(9, st.d)
    word, _, packed = check(st, 100, query=q)
    assert word != 0
    oracle_check(st, packed, 100, q=q)
