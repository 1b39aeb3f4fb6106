"""Row-sharded recommend_batch for long lists (k = 500, 2048) equals the single-GPU result (needs >= 2 GPUs; skips otherwise).

Every shard is above the long-list plan minimum, and each rank reports the plan its tensor-core pass used: the per-query
fallback answers correctly too, so without that check a broken batched pass would go unnoticed.
"""
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

D = 128


def _run_guarded(name, rank, world, port, *args):
    """Picklable worker entry (spawn): runs the named worker; an exception becomes a queue item, so the parent fails at
    once instead of waiting for a timeout."""
    import traceback
    out_q = args[-1]
    try:
        globals()[name](rank, world, port, *args)
    except BaseException:  # noqa: BLE001
        out_q.put((rank, "ERROR", traceback.format_exc()))
        raise


def _collect(out_q, procs, world, timeout=600):
    results = []
    for _ in range(world):
        item = out_q.get(timeout=timeout)
        if len(item) >= 2 and item[1] == "ERROR":
            for p in procs:
                p.kill()
            pytest.fail(f"worker {item[0]} raised:\n{item[2]}")
        results.append(item)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    return results


def _csr_users(n, b):
    from robot_ebert_b200 import synth
    lp, lc, ep, ec = [0], [], [0], []
    for rated, rts in synth.user_ratings(2, n, b):
        liked = rated[rts >= 3.5]
        if len(liked) == 0:
            liked = rated[:1]
        lc.append(liked); lp.append(lp[-1] + len(liked)); ec.append(rated); ep.append(ep[-1] + len(rated))
    return np.array(lp), np.concatenate(lc), np.array(ep), np.concatenate(ec)


def _batch_worker(rank, world, port, n, b, ks, out_q):
    import torch.distributed as dist
    from robot_ebert_b200.sharding import ShardedCatalog
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        sc = ShardedCatalog.synthetic(0, n, D, "bf16", scale_rows=True, device=torch.device("cuda", rank))
        lp, lc, ep, ec = _csr_users(n, b)
        out = []
        for k in ks:
            r = sc.recommend_batch(liked_ptr=lp, liked_col=lc, excl_ptr=ep, excl_col=ec, k=k, return_info=True)
            out.append((k, r[0].tolist(), r[1].tolist(), r[2].tolist(), r[3]["plan"], int((r[3]["status"] != 0).sum())))
        out_q.put((rank, sc.backend.store.n, out))
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_sharded_long_list_batch_equals_single_gpu():
    world = min(torch.cuda.device_count(), 8)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    from robot_ebert_b200 import CatalogStore
    ks = (500, 2048)
    n, b = 500_000 * world + 17, 130                 # every shard above the bf16 minimum at k = 2048 (491,520 rows)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    out_q = ctx.Queue()
    procs = [ctx.Process(target=_run_guarded, args=("_batch_worker", r, world, port, n, b, ks, out_q)) for r in range(world)]
    for p in procs:
        p.start()
    results = _collect(out_q, procs, world)
    store = CatalogStore.synthetic(0, n, D, "bf16", scale_rows=True, device="cuda:0")
    lp, lc, ep, ec = _csr_users(n, b)
    for i, k in enumerate(ks):
        want = store.recommend_batch(liked_ptr=lp, liked_col=lc, excl_ptr=ep, excl_col=ec, k=k, prefilter=False)
        for rank, shard_n, out in results:
            kk, rows, scores, counts, plan, n_status = out[i]
            assert kk == k and shard_n >= 491_520
            assert plan is not None and plan["k"] == k and plan["sample_rank"] == 64, (rank, plan)
            assert n_status <= 0.05 * b, (rank, k, n_status)
            assert rows == want[0].tolist() and counts == want[2].tolist(), (rank, k)
            np.testing.assert_allclose(scores, want[1], rtol=1e-12)
