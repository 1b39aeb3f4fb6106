"""Row shards with an int8 gate (needs >= 2 GPUs): every rank's shard streams its gate, seeds its own bound and reads rows
of record only where they can reach its candidate list; the sharded result must equal one GPU's plain pass (ids exact,
scores to 1e-12).  Harness as in test_multigpu.py."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

KS = (10, 100, 240)


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


def _spawn(name, world, *args):
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    out_q = ctx.Queue()
    procs = [ctx.Process(target=_run_guarded, args=(name, r, world, port, *args, out_q)) for r in range(world)]
    for p in procs:
        p.start()
    return _collect(out_q, procs, world)


def _world():
    world = min(torch.cuda.device_count(), 8)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    return world


def _requests(n, world, d):
    """Query and profile requests at every k, with exclusions of global ids on both sides of every shard boundary."""
    from robot_ebert_b200 import synth
    from robot_ebert_b200.sharding import ShardPlan
    plan = ShardPlan(n, world)
    edges = [plan.range(r)[0] for r in range(1, world)]
    rng = np.random.default_rng(3)
    excl = np.unique(np.concatenate([rng.choice(n, size=400, replace=False)] + [e + np.arange(-3, 3) for e in edges]))
    (rated, rts), = synth.user_ratings(2, n, 1)
    liked = rated[rts >= 3.5] if (rts >= 3.5).any() else rated[:1]
    reqs = []
    for k in KS:
        reqs.append(dict(query=synth.query_f32(1, d), exclude_rows=excl, k=k))
        reqs.append(dict(liked_rows=liked, exclude_rows=np.union1d(rated, excl), k=k))
    return reqs


def _fetches(backend):
    """Rows of record read by the gated pass on channel 0.  Sharded requests on the peer-memory path run on the channel's
    pre-allocated scratch, whose gemv workspace is the first region of its device block (csrc/host_api.cu, host_layout:
    off_ws = 0).  None on the NCCL fallback: there a request may widen kc and move to a freshly allocated workspace, so no
    single workspace holds its count."""
    from robot_ebert_b200 import _native as nat
    if backend.exchange != "p2p":
        return None
    ws = backend._chan_scratch[0].hdev
    out = C.c_uint32(0)
    nat.check(nat.load().rebert_gate_fetches(ws.data_ptr(), ws.numel(), C.byref(out), torch.cuda.current_stream().cuda_stream))
    return out.value


def _init(rank, world, port):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    return dist


def _gate_worker(rank, world, port, n, d, dtype, gated_ranks, out_q):
    dist = _init(rank, world, port)
    try:
        from robot_ebert_b200.sharding import ShardedCatalog
        sc = ShardedCatalog.synthetic(0, n, d, dtype, scale_rows=True, device=torch.device("cuda", rank))
        st = sc.backend.store
        if rank in gated_ranks:
            assert st.build_gate()
        sc.warm_up()                  # collective: the gated kernels' first launches before any request is in flight
        out, fetched = [], 0
        for r in _requests(n, world, d):
            f0 = _fetches(sc.backend)
            rows, scores = sc.recommend(**r)
            fetched = None if f0 is None else fetched + (_fetches(sc.backend) - f0)
            out.append((rows.tolist(), scores.tolist()))
        out_q.put((rank, st.has_gate, fetched, out))
        dist.barrier()
    finally:
        dist.destroy_process_group()


def _single_gpu(n, d, dtype, reqs):
    from robot_ebert_b200 import CatalogStore
    store = CatalogStore.synthetic(0, n, d, dtype, scale_rows=True, device="cuda:0")
    store.drop_gate()                                    # the plain pass
    want = [store.recommend(**r) for r in reqs]
    del store
    torch.cuda.empty_cache()
    return want


def _compare(results, want):
    for rank, _, _, out in results:
        for i, ((rows, scores), (wr, ws)) in enumerate(zip(out, want)):
            assert rows == wr.tolist(), (rank, i)
            np.testing.assert_allclose(scores, ws, rtol=1e-12)


@pytest.mark.parametrize("gated", ["every_rank", "rank0_only"])
@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
def test_gated_shards_equal_one_gpu(dtype, gated):
    world = _world()
    n, d = 200_003, 1536
    gated_ranks = tuple(range(world)) if gated == "every_rank" else (0,)
    results = _spawn("_gate_worker", world, n, d, dtype, gated_ranks)
    for rank, has_gate, fetched, _ in results:
        assert has_gate == (rank in gated_ranks), rank
        if fetched is not None:                        # peer-memory path: the channel's fetch count is readable
            assert (fetched > 0) == (rank in gated_ranks), (rank, fetched)
    _compare(results, _single_gpu(n, d, dtype, _requests(n, world, d)))


def _ctor_worker(rank, world, port, n, d, out_q):
    dist = _init(rank, world, port)
    try:
        from robot_ebert_b200.sharding import ShardedCatalog
        sc = ShardedCatalog.synthetic(0, n, d, "bf16", scale_rows=True, device=torch.device("cuda", rank))
        st = sc.backend.store
        reqs = _requests(n, world, d)[:2]                   # k = 10: a query and a profile
        out = [sc.recommend(**r) for r in reqs]
        out_q.put((rank, st.has_gate, st.n * st.ld, [(r.tolist(), s.tolist()) for r, s in out]))
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_constructor_built_gates_on_bench_sized_shards():
    """Shards large enough that each one's constructor builds its gate (GATE_MIN_SAVED_BYTES), as the bench's 2-GPU
    catalog's do."""
    from robot_ebert_b200 import CatalogStore
    world = _world()
    d = 1536
    per_shard = CatalogStore.GATE_MIN_SAVED_BYTES // d + 8192       # bf16 rows of 1536: d bytes saved per row
    n = world * per_shard
    results = _spawn("_ctor_worker", world, n, d)
    for rank, has_gate, saved, _ in results:
        assert saved >= CatalogStore.GATE_MIN_SAVED_BYTES, rank
        assert has_gate, f"rank {rank}: the constructor did not build the gate"
    _compare(results, _single_gpu(n, d, "bf16", _requests(n, world, d)[:2]))
