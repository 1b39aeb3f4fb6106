"""Row-sharded recommend_batch with a genre / year filter per user equals the single-GPU result (needs >= 2 GPUs; skips
otherwise).  Every rank installs its own shard's metadata on backend.store and reports the plan its tensor-core pass used:
the per-query fallback answers correctly too, so without that check a broken batched pass would go unnoticed."""
import socket

import numpy as np
import pytest
import torch

from tests.test_multigpu_batched_large_k import _collect, _csr_users

pytestmark = pytest.mark.gpu

D = 128
K = 50


def _run_guarded(name, rank, world, port, *args):
    """Picklable worker entry (spawn): runs the named worker of this module; an exception becomes a queue item."""
    import traceback
    out_q = args[-1]
    try:
        globals()[name](rank, world, port, *args)
    except BaseException:  # noqa: BLE001
        out_q.put((rank, "ERROR", traceback.format_exc()))
        raise


def _filters(b):
    """Unrestricted, broad (~50 %), narrow (~1 %) and zero-row users in turn."""
    from robot_ebert_b200 import QueryFilters
    rng = np.random.default_rng(b)
    ga, lo, hi = [], [], []
    for u in range(b):
        y0 = int(rng.integers(1920, 1972))
        f = [(0, 0, 65535), (0, y0, y0 + 51), (1 << int(rng.integers(0, 19)), y0, y0 + 7), (0, 2000, 1999)][u % 4]
        ga.append(f[0]); lo.append(f[1]); hi.append(f[2])
    return QueryFilters(ga, lo, hi)


def _filter_worker(rank, world, port, n, b, out_q):
    import os

    import torch.distributed as dist
    from robot_ebert_b200 import synth
    from robot_ebert_b200.sharding import ShardedCatalog
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        sc = ShardedCatalog.synthetic(0, n, D, "bf16", scale_rows=True, device=torch.device("cuda", rank))
        store = sc.backend.store
        store.set_metadata(*synth.movie_metadata(3, store.row_base, store.n))      # this rank's rows only
        lp, lc, ep, ec = _csr_users(n, b)
        r = sc.recommend_batch(liked_ptr=lp, liked_col=lc, excl_ptr=ep, excl_col=ec, k=K, query_filters=_filters(b), return_info=True)
        out_q.put((rank, store.n, r[0].tolist(), r[1].tolist(), r[2].tolist(), r[3]["plan"], int((r[3]["status"] != 0).sum())))
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_sharded_batch_with_user_filters_equals_single_gpu():
    world = min(torch.cuda.device_count(), 8)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    from robot_ebert_b200 import CatalogStore, synth
    n, b = 70_000 * world + 17, 130                  # every shard above the bf16 minimum at k = 50 (49,152 rows)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    out_q = ctx.Queue()
    procs = [ctx.Process(target=_run_guarded, args=("_filter_worker", r, world, port, n, b, out_q)) for r in range(world)]
    for p in procs:
        p.start()
    results = _collect(out_q, procs, world)
    store = CatalogStore.synthetic(0, n, D, "bf16", scale_rows=True, device="cuda:0")
    store.set_metadata(*synth.movie_metadata(3, 0, n))
    lp, lc, ep, ec = _csr_users(n, b)
    want = store.recommend_batch(liked_ptr=lp, liked_col=lc, excl_ptr=ep, excl_col=ec, k=K, query_filters=_filters(b), prefilter=False)
    assert (want[2][3::4] == 0).all() and (want[2][::4] == K).all()          # zero-row and unrestricted users
    for rank, shard_n, rows, scores, counts, plan, n_status in results:
        assert shard_n >= 49_152
        assert plan is not None and plan["k"] == K, (rank, plan)
        assert n_status <= 0.05 * b, (rank, n_status)
        assert rows == want[0].tolist() and counts == want[2].tolist(), rank
        np.testing.assert_allclose(scores, want[1], rtol=1e-12)
