"""Multi-GPU parity (needs >= 2 GPUs: `gpurun --gpus 2`): row-sharded result == single-GPU result, ids bit-exact."""
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


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


def _collect(out_q, procs, world, timeout=300):
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


def _worker(rank, world, port, n, d, dtype, out_q):
    import torch.distributed as dist
    from robot_ebert_b200 import synth
    from robot_ebert_b200.sharding import ShardedCatalog
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        sc = ShardedCatalog.synthetic(0, n, d, dtype, scale_rows=True, device=torch.device("cuda", rank))
        q = synth.query_f32(1, d)
        excl = np.random.default_rng(3).choice(n, size=133, replace=False)
        r1 = sc.recommend(query=q, exclude_rows=excl, k=10)
        (rated, rts), = synth.user_ratings(2, n, 1)
        r2 = sc.recommend(liked_rows=rated[rts >= 3.5], exclude_rows=rated, k=50)
        r3 = sc.recommend(query=q, exclude_rows=excl, k=300)                 # k > 240: sharded bisection + sweep route
        r4 = sc.recommend(liked_rows=rated[rts >= 3.5], exclude_rows=rated, k=1000)
        out_q.put((rank, r1[0].tolist(), r1[1].tolist(), r2[0].tolist(), r2[1].tolist(), r3[0].tolist(), r3[1].tolist(),
                   r4[0].tolist(), r4[1].tolist()))
        dist.barrier()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
def test_sharded_equals_single_gpu(dtype):
    world = min(torch.cuda.device_count(), 8)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    from robot_ebert_b200 import CatalogStore, synth
    n, d = 200_003, 1536
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    out_q = ctx.Queue()
    procs = [ctx.Process(target=_run_guarded, args=("_worker", r, world, port, n, d, dtype, out_q)) for r in range(world)]
    for p in procs:
        p.start()
    results = _collect(out_q, procs, world)
    store = CatalogStore.synthetic(0, n, d, dtype, scale_rows=True, device="cuda:0")
    q = synth.query_f32(1, d)
    excl = np.random.default_rng(3).choice(n, size=133, replace=False)
    w1 = store.recommend(query=q, exclude_rows=excl, k=10)
    (rated, rts), = synth.user_ratings(2, n, 1)
    w2 = store.recommend(liked_rows=rated[rts >= 3.5], exclude_rows=rated, k=50)
    w3 = store.recommend(query=q, exclude_rows=excl, k=300)
    w4 = store.recommend(liked_rows=rated[rts >= 3.5], exclude_rows=rated, k=1000)
    assert len(w3[0]) == 300 and len(w4[0]) == 1000
    for rank, r1r, r1s, r2r, r2s, r3r, r3s, r4r, r4s in results:
        assert r1r == w1[0].tolist() and r2r == w2[0].tolist(), rank
        np.testing.assert_allclose(r1s, w1[1], rtol=1e-12)
        np.testing.assert_allclose(r2s, w2[1], rtol=1e-12)
        assert r3r == w3[0].tolist() and r4r == w4[0].tolist(), rank
        np.testing.assert_allclose(r3s, w3[1], rtol=1e-12)
        np.testing.assert_allclose(r4s, w4[1], rtol=1e-12)


def _batch_worker(rank, world, port, n, d, b, k, out_q):
    import torch.distributed as dist
    from robot_ebert_b200 import synth
    from robot_ebert_b200.sharding import ShardedCatalog
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        sc = ShardedCatalog.synthetic(0, n, d, "bf16", scale_rows=True, device=torch.device("cuda", rank))
        lp, lc, ep, ec = _csr_users(n, b)
        from robot_ebert_b200 import RowFilter
        g, y = synth.movie_metadata(3, sc.backend.store.row_base, sc.backend.store.n)      # this shard's slice of the side columns
        sc.backend.store.set_metadata(g, y)
        r = sc.recommend_batch(liked_ptr=lp, liked_col=lc, excl_ptr=ep, excl_col=ec, k=k,
                               row_filter=RowFilter(genre_any=0b1011, year_lo=1960, year_hi=2000))
        out_q.put((rank, r[0].tolist(), r[1].tolist(), r[2].tolist()))
        dist.barrier()
    finally:
        dist.destroy_process_group()


def _csr_users(n, b):
    from robot_ebert_b200 import synth
    lp, lc, ep, ec = [0], [], [0], []
    for rated, rts in synth.user_ratings(2, n, b):
        liked = rated[rts >= 3.5]
        if len(liked) == 0:
            liked = rated[:1]
        lc.append(liked); lp.append(lp[-1] + len(liked)); ec.append(rated); ep.append(ep[-1] + len(rated))
    return np.array(lp), np.concatenate(lc), np.array(ep), np.concatenate(ec)


def test_sharded_batch_equals_single_gpu_batch():
    """BASELINE config 5 shape at test size: CSR profiles + exclusions, sharded tcgen05 pass == one-GPU result."""
    world = min(torch.cuda.device_count(), 8)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    from robot_ebert_b200 import CatalogStore
    n, d, b, k = 140_000, 512, 200, 50
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    out_q = ctx.Queue()
    procs = [ctx.Process(target=_run_guarded, args=("_batch_worker", r, world, port, n, d, b, k, out_q)) for r in range(world)]
    for p in procs:
        p.start()
    results = _collect(out_q, procs, world)
    store = CatalogStore.synthetic(0, n, d, "bf16", scale_rows=True, device="cuda:0")
    lp, lc, ep, ec = _csr_users(n, b)
    from robot_ebert_b200 import RowFilter, synth
    g, y = synth.movie_metadata(3, 0, n)
    store.set_metadata(g, y)
    want = store.recommend_batch(liked_ptr=lp, liked_col=lc, excl_ptr=ep, excl_col=ec, k=k,
                                 row_filter=RowFilter(genre_any=0b1011, year_lo=1960, year_hi=2000))
    keep = ((g & 0b1011) != 0) & (y >= 1960) & (y <= 2000)
    assert keep[want[0][want[0] >= 0]].all()
    for rank, rows, scores, counts in results:
        assert rows == want[0].tolist() and counts == want[2].tolist(), rank
        np.testing.assert_allclose(scores, want[1], rtol=1e-12)


def _tie_worker(rank, world, port, out_q):
    import torch.distributed as dist
    from robot_ebert_b200 import CatalogStore
    from robot_ebert_b200.sharding import CudaShardBackend, ShardedCatalog, ShardPlan
    from robot_ebert_b200 import synth
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        n = 3000
        m = synth.catalog_rows_f32(0, 0, n, 1, scale_rows=True)                    # d = 1: every cosine is exactly +-1
        row0, cnt = ShardPlan(n, world).range(rank)
        store = CatalogStore.from_host(None, m[row0:row0 + cnt], "fp32", device=torch.device("cuda", rank), row_base=row0)
        backend = CudaShardBackend(store)
        backend.setup_p2p()
        sc = ShardedCatalog(backend, n)
        rows, scores, info = sc.recommend(query=np.ones(1, dtype=np.float32), exclude_rows=np.arange(0, n, 7), k=10, return_info=True)
        out_q.put((rank, rows.tolist(), scores.tolist(), bool(info["proven_exact"])))
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_sharded_mass_ties_use_the_exact_sweep():
    world = min(torch.cuda.device_count(), 8)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    from oracle import reference_scoring as ora
    from robot_ebert_b200 import synth
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    out_q = ctx.Queue()
    procs = [ctx.Process(target=_run_guarded, args=("_tie_worker", r, world, port, out_q)) for r in range(world)]
    for p in procs:
        p.start()
    results = _collect(out_q, procs, world)
    m = synth.catalog_rows_f32(0, 0, 3000, 1, scale_rows=True).astype(np.float64)
    want_rows, want_scores = ora.query_rows(m, np.ones(1), np.arange(0, 3000, 7), 10)
    for rank, rows, scores, proven in results:
        assert proven and rows == want_rows.tolist(), rank
        np.testing.assert_allclose(scores, want_scores, rtol=1e-12)


def test_sharded_batch_small_shards_fall_back_to_single_query_path():
    """Shards below the tensor-core path's minimum size: recommend_batch must still answer (per-query sharded path)."""
    world = min(torch.cuda.device_count(), 8)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    from robot_ebert_b200 import CatalogStore, RowFilter, synth
    n, d, b, k = 9_000 * world, 128, 6, 10
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    out_q = ctx.Queue()
    procs = [ctx.Process(target=_run_guarded, args=("_batch_worker", r, world, port, n, d, b, k, out_q)) for r in range(world)]
    for p in procs:
        p.start()
    results = _collect(out_q, procs, world)
    store = CatalogStore.synthetic(0, n, d, "bf16", scale_rows=True, device="cuda:0")
    lp, lc, ep, ec = _csr_users(n, b)
    g, y = synth.movie_metadata(3, 0, n)
    store.set_metadata(g, y)
    want = store.recommend_batch(liked_ptr=lp, liked_col=lc, excl_ptr=ep, excl_col=ec, k=k,
                                 row_filter=RowFilter(genre_any=0b1011, year_lo=1960, year_hi=2000))
    for rank, rows, scores, counts in results:
        assert rows == want[0].tolist() and counts == want[2].tolist(), rank
        np.testing.assert_allclose(scores, want[1], rtol=1e-12)


# ---------------------------------------------------------------------------------------------------------------------
# round 2: one C call per rank for liked-rows requests, from_host + the lib.py contract on shards, the int8 prefilter on
# shards, concurrent serving threads on their own exchange channels, and diverged request order
# ---------------------------------------------------------------------------------------------------------------------
def _spawn(name, world, *args, timeout=420):
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    out_q = ctx.Queue()
    procs = [ctx.Process(target=_run_guarded, args=(name, r, world, port, *args, out_q)) for r in range(world)]
    for p in procs:
        p.start()
    return _collect(out_q, procs, world, timeout=timeout)


def _init(rank, world, port):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    return dist


def _requests(n, d, count):
    """A fixed mix of query / liked-rows requests (with and without weights), identical in every process."""
    from robot_ebert_b200 import synth
    users = synth.user_ratings(7, n, count)
    reqs = []
    for i in range(count):
        rated, rts = users[i]
        liked = rated[rts >= 3.5] if (rts >= 3.5).any() else rated[:1]
        if i % 3 == 0:
            reqs.append(dict(query=synth.query_f32(100 + i, d), exclude_rows=rated, k=10))
        elif i % 3 == 1:
            reqs.append(dict(liked_rows=liked, exclude_rows=rated, k=10))
        else:
            reqs.append(dict(liked_rows=liked, weights=(1.0 + np.arange(len(liked)) % 3).astype(np.float32), exclude_rows=rated, k=25))
    return reqs


def _threads_worker(rank, world, port, n, d, nthreads, per_thread, out_q):
    import threading
    os.environ["REBERT_EXCHANGE_TIMEOUT_MS"] = "3000"        # fail fast if a peer never delivers
    dist = _init(rank, world, port)
    from robot_ebert_b200.sharding import ShardedCatalog
    try:
        sc = ShardedCatalog.synthetic(0, n, d, "bf16", scale_rows=True, device=torch.device("cuda", rank))
        assert sc.backend.exchange == "p2p", getattr(sc.backend, "_p2p_error", None)
        reqs = _requests(n, d, nthreads * per_thread)
        results, errors = [None] * len(reqs), []

        def serve(t):                                   # thread t of every rank serves the same requests on channel t
            try:
                torch.cuda.set_device(rank)             # a new thread starts on device 0
                with torch.cuda.stream(torch.cuda.Stream()):
                    for j in range(per_thread):
                        i = t * per_thread + j
                        r, s = sc.recommend(channel=t, **reqs[i])
                        results[i] = (r.tolist(), s.tolist())
            except BaseException as e:  # noqa: BLE001
                errors.append((t, repr(e)))

        th = [threading.Thread(target=serve, args=(t,)) for t in range(nthreads)]
        for x in th:
            x.start()
        for x in th:
            x.join()
        out_q.put((rank, results, errors))
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_sharded_serving_threads_on_their_own_channels():
    """FastAPI's threadpool (api/users.py:151) on row shards: 8 threads per rank, thread t on exchange channel t, a mix of
    query / profile / weighted-profile requests; every answer must equal the single-GPU answer."""
    world = min(torch.cuda.device_count(), 8)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    from robot_ebert_b200 import CatalogStore
    n, d, nthreads, per_thread = 120_001, 256, 8, 12
    results = _spawn("_threads_worker", world, n, d, nthreads, per_thread)
    assert not any(errs for _, _, errs in results), [(rank, errs) for rank, _, errs in results]
    store = CatalogStore.synthetic(0, n, d, "bf16", scale_rows=True, device="cuda:0")
    want = [store.recommend(**r) for r in _requests(n, d, nthreads * per_thread)]
    for rank, got, _ in results:
        for i, ((rows, scores), (wr, ws)) in enumerate(zip(got, want)):
            assert rows == wr.tolist(), (rank, i)
            np.testing.assert_allclose(scores, ws, rtol=1e-12)


def _contract_worker(rank, world, port, n, d, out_q):
    dist = _init(rank, world, port)
    from robot_ebert_b200 import lib as rlib, synth
    from robot_ebert_b200.sharding import ShardedCatalog
    from tests.helpers import FakeSql, fake_movie
    try:
        m = synth.catalog_rows_f32(0, 0, n, d, scale_rows=True)
        ids = [str(i * 7919 % 100003) for i in range(n)]             # unsorted ids: from_host sorts them as strings (notebook order)
        sc = ShardedCatalog.from_host(ids, m, "fp32", device=torch.device("cuda", rank))
        sql = FakeSql()
        for i in ids:
            sql.movies[i] = fake_movie(i)
        (rated, rts), = synth.user_ratings(5, n, 1)
        sql.ratings["u"] = [(ids[r], float(x)) for r, x in zip(rated, rts)] + [("not-in-catalog", 5.0)]
        rlib.configure(catalog=sc, sql=sql)
        recs = rlib.get_user_recs("u", k=10)
        eps = sc.enable_prefilter()
        q = synth.query_f32(1, d)
        pr, ps, info = sc.recommend(query=q, exclude_rows=np.arange(0, n, 11), k=10, return_info=True, prefilter=True)
        out_q.put((rank, [(r.movie.tmdb_id, r.score) for r in recs], pr.tolist(), ps.tolist(), bool(info.get("prefilter")), eps))
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_sharded_from_host_lib_contract_and_prefilter():
    """ShardedCatalog.from_host as the catalog behind lib.get_user_recs (the reference's real route, lib.py:32-63), and the
    int8 prefilter on shards: same answers as one GPU / the oracle."""
    world = min(torch.cuda.device_count(), 8)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    from oracle import reference_scoring as ora
    from robot_ebert_b200 import CatalogStore, synth
    n, d = 90_001, 96
    results = _spawn("_contract_worker", world, n, d)
    m = synth.catalog_rows_f32(0, 0, n, d, scale_rows=True)
    ids = [str(i * 7919 % 100003) for i in range(n)]
    order = sorted(range(n), key=ids.__getitem__)
    ms, sids = m[np.asarray(order)].astype(np.float64), [ids[i] for i in order]
    row_of = {i: r for r, i in enumerate(sids)}
    (rated, rts), = synth.user_ratings(5, n, 1)
    rated_rows = np.array([row_of[ids[r]] for r in rated])
    want_rows, want_scores = ora.recommend_rows(ms, rated_rows[rts >= 3.5], rated_rows, 10)
    store = CatalogStore.from_host(ids, m, "fp32", device="cuda:0")
    q = synth.query_f32(1, d)
    wq = store.recommend(query=q, exclude_rows=np.arange(0, n, 11), k=10)
    for rank, recs, pr, ps, used_prefilter, eps in results:
        assert [i for i, _ in recs] == [sids[r] for r in want_rows], rank
        np.testing.assert_allclose([s for _, s in recs], want_scores, rtol=1e-9)
        assert pr == wq[0].tolist() and ps == wq[1].tolist(), rank               # query request: same bits as one GPU
        assert 0.0 < eps < 0.05


def _diverge_worker(rank, world, port, n, d, out_q):
    dist = _init(rank, world, port)
    from robot_ebert_b200 import synth
    from robot_ebert_b200.sharding import ShardedCatalog
    try:
        sc = ShardedCatalog.synthetic(0, n, d, "bf16", device=torch.device("cuda", rank))
        q = synth.query_f32(1, d)
        first = sc.recommend(query=q, k=10)
        # the ranks now disagree about the request on channel 0: the merge must refuse, on every rank
        bad = synth.query_f32(50 + (rank % 2), d)
        try:
            sc.recommend(query=bad, k=10)
            refused = False
        except Exception as e:  # noqa: BLE001
            refused = "different request" in str(e)
        again = sc.recommend(query=q, k=10)                # ... and the channel keeps working afterwards
        out_q.put((rank, refused, first[0].tolist() == again[0].tolist() and first[1].tolist() == again[1].tolist()))
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_sharded_diverged_request_order_is_refused():
    world = min(torch.cuda.device_count(), 8)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    for rank, refused, recovered in _spawn("_diverge_worker", world, 50_000, 128):
        assert refused and recovered, rank


def _routing_batch_worker(rank, world, port, n, d, dtype, b, k, out_q):
    dist = _init(rank, world, port)
    from robot_ebert_b200 import synth
    from robot_ebert_b200.sharding import ShardedCatalog
    try:
        sc = ShardedCatalog.synthetic(0, n, d, dtype, scale_rows=True, device=torch.device("cuda", rank))
        lp, lc, ep, ec = _csr_users(n, b)
        rq = sc.recommend_batch(queries=synth.catalog_rows_f32(11, 0, b, d), excl_ptr=ep, excl_col=ec, k=k)
        rp = sc.recommend_batch(liked_ptr=lp, liked_col=lc, excl_ptr=ep, excl_col=ec, k=k)
        out_q.put((rank, [x.tolist() for x in rq], [x.tolist() for x in rp]))
        dist.barrier()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("dtype,d", [("fp32", 64), ("bf16", 32)])
def test_sharded_batch_on_shards_the_gemm_cannot_take(dtype, d):
    """fp32 shards, and bf16 shards of 32-element rows, each above gemm_plan's minimum size: the tcgen05 GEMM takes
    neither, so recommend_batch must serve them through the sharded single-query path, with the single-GPU answer."""
    world = min(torch.cuda.device_count(), 8)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    from robot_ebert_b200 import CatalogStore, synth
    n, b, k = 20_000 * world, 12, 10
    results = _spawn("_routing_batch_worker", world, n, d, dtype, b, k)
    store = CatalogStore.synthetic(0, n, d, dtype, scale_rows=True, device="cuda:0")
    lp, lc, ep, ec = _csr_users(n, b)
    wq = store.recommend_batch(queries=synth.catalog_rows_f32(11, 0, b, d), excl_ptr=ep, excl_col=ec, k=k)
    wp = store.recommend_batch(liked_ptr=lp, liked_col=lc, excl_ptr=ep, excl_col=ec, k=k)
    for rank, rq, rp in results:
        for got, want in ((rq, wq), (rp, wp)):
            assert got[0] == want[0].tolist() and got[2] == want[2].tolist(), rank
            np.testing.assert_allclose(got[1], want[1], rtol=1e-12)
