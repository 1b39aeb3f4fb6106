"""Row-sharding layer: one process per GPU, catalog split row-wise, local top-k + all-gather + merge.

SURVEY.md §8(e): score(j) depends only on catalog row j and the replicated query, so rank g owns the contiguous
rows [g*N/G, (g+1)*N/G) and the only exchange step is an all-gather of each rank's k best (row, score) pairs
(k*16+16 bytes per rank), followed by the same (score desc, row asc) merge on every rank — so every rank returns
the result a single GPU would.  Building a user profile from liked rows scattered over the shards adds one
all-reduce(sum) of the fp64 partial profile [ld+1].

The collective plumbing is torch.distributed (NCCL on GPUs).  The arithmetic is behind a small backend object so
the host logic can be exercised with gloo on CPU in tests; the product backend (`CudaShardBackend`) is CUDA-only.
"""
from __future__ import annotations

import ctypes as C
import logging
import threading
from typing import Optional, Sequence, Tuple

import numpy as np
import torch
import torch.distributed as dist

from . import _native as nat
from .catalog import (EMPTY_PROFILE, CatalogStore, QueryFilters, RowFilter, close_proof, large_k_search, sorted_csr, unpack_result,
                      user_row_filter, validated_table, widen_until_proven)

log = logging.getLogger("robot_ebert_b200")


class ShardPlan:
    """Contiguous, balanced row ranges; rank g owns [start(g), start(g+1))."""

    def __init__(self, n_total: int, world: int):
        if n_total < 0 or world <= 0:
            raise ValueError("bad shard plan")
        self.n_total, self.world = int(n_total), int(world)

    def start(self, g: int) -> int:
        return (self.n_total * g) // self.world

    def range(self, g: int) -> Tuple[int, int]:
        """(row0, nrows) of rank g."""
        return self.start(g), self.start(g + 1) - self.start(g)

    def owner(self, row: int) -> int:
        if not 0 <= row < self.n_total:
            raise ValueError("row out of range")
        g = min(self.world - 1, (row * self.world) // max(self.n_total, 1))
        while row < self.start(g):
            g -= 1
        while row >= self.start(g + 1):
            g += 1
        return g


class CudaShardBackend:
    """Product backend: the local shard is a CatalogStore; every step is a kernel enqueued on the current stream.

    Exchange paths: "p2p" (after setup_p2p: NVLink peer memory, the whole request is ONE C call per rank, no NCCL and no
    torch op on the request path) or "nccl" (fallback when the platform cannot map peer buffers)."""

    K_MAX = 240          # largest k of the single-query path
    CHANNELS = 16        # independent request streams of the peer-mapped buffers (one per serving thread)

    def __init__(self, store: CatalogStore):
        self.store = store
        self.device = store.device
        self._merged = {}
        self._host = {}
        self.exchange = "nccl"       # becomes "p2p" once setup_p2p() has mapped the peers' buffers
        self.channels = 1
        self._seq = [0]
        self._nccl_lock = threading.Lock()      # the NCCL fallback keeps per-process buffers: one request at a time
        self._err = {}
        self._xstructs = {}                     # channel -> its reusable rebert_exchange_t

    def setup_p2p(self, group=None, channels: Optional[int] = None) -> bool:
        """Map one symmetric buffer per rank (torch symmetric memory = CUDA VMM + fabric handles) holding `channels`
        independent exchange channels, so that the exchange steps become P2P stores + flags inside the request's kernels.
        Falls back to NCCL (and says so in the log) if the platform cannot provide peer mappings.
        Collective: every rank must call it."""
        lib = nat.load()
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        channels = int(channels or self.CHANNELS)
        ok = torch.zeros(1, dtype=torch.int32, device=self.device)
        try:
            import torch.distributed._symmetric_memory as symm
            nbytes = lib.rebert_exchange_buffer_bytes(world, self.K_MAX, self.store.ld, channels)
            if nbytes == 0:
                raise RuntimeError("world size not supported by the exchange kernels")
            buf = symm.empty(nbytes // 8, dtype=torch.int64, device=self.device)
            buf.zero_()
            hdl = symm.rendezvous(buf, group if group is not None else dist.group.WORLD)
            self._symm_buf, self._symm_hdl = buf, hdl
            self._peer_ptrs = (C.c_uint64 * world)(*[int(p) for p in hdl.buffer_ptrs])
            self._p2p_out = {}
            self._xstructs = {}
            self._p2p_world, self._p2p_rank = world, rank
            ok.fill_(1)
        except Exception as e:  # noqa: BLE001 - any failure of the plumbing means: keep NCCL
            self._p2p_error = repr(e)
            log.warning("rank %d: peer-memory exchange unavailable (%s)", rank, self._p2p_error)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)      # all or nothing, and a barrier after the zero-fill
        torch.cuda.synchronize(self.device)
        self.exchange = "p2p" if int(ok.item()) == 1 else "nccl"
        if self.exchange == "p2p":
            self.channels = channels
            self._seq = [0] * channels
            # One request scratch (pinned + device) per channel, allocated NOW, while no request is in flight: a CUDA
            # allocation may synchronise the device, and a device synchronisation while another channel's kernel is waiting
            # for a peer — whose own progress may hang on the mirrored allocation — stalls both ranks until the timeout.
            from .catalog import _Scratch
            self._chan_scratch = []
            with torch.cuda.device(self.device):
                for _ in range(channels):
                    sc = _Scratch(self.store)
                    sc.ensure_host(1, 1, 1)
                    self._chan_scratch.append(sc)
                torch.cuda.synchronize(self.device)
        log.info("rank %d/%d: row-shard exchange path = %s%s", rank, world, self.exchange,
                 f" ({channels} channels)" if self.exchange == "p2p" else " (all-gather + merge kernel; requests are serialised)")
        return self.exchange == "p2p"

    def exchange_struct(self, channel: int, seq: int) -> "nat.Exchange":
        """This rank's rebert_exchange_t for one call on `channel` (the caller holds the channel's lock, so the channel's
        struct is reused: only the sequence number changes from call to call)."""
        x = self._xstructs.get(channel)
        if x is None:
            x = self._xstructs[channel] = nat.Exchange()
            x.peer_buffers = C.cast(self._peer_ptrs, C.c_void_p)
            x.world, x.rank, x.k_max, x.prof_len = self._p2p_world, self._p2p_rank, self.K_MAX, self.store.ld
            x.channels, x.channel = self.channels, channel
        x.seq = (seq & 0xFFFFFFFF) or 1
        return x

    def next_seq(self, channel: int, n: int = 1) -> int:
        """First of n fresh sequence numbers on `channel` (the caller holds the channel's lock)."""
        first = self._seq[channel] + 1
        self._seq[channel] += n
        return first

    def recommend_host(self, query, liked_rows, weights, exclude_rows, k: int, kc: int, row_filter: Optional[RowFilter],
                       channel: int = 0, shadow_max_k: int = 0, shadow_eps=None):
        """One C call per rank for a whole request on the P2P path (rebert_recommend_host with an exchange): zero-copy
        request, query normalisation or profile build + partial-profile exchange, local fast + exact pass and the result
        exchange + merge inside the scoring launch, proof loop, result written into pinned memory.  Collective in effect:
        every rank must call it with the same arguments on the same channel.  Returns (rows, scores, info)."""
        st = self.store
        x = self.exchange_struct(channel, self._seq[channel] + 1)
        scratch = self._chan_scratch[channel]                      # pre-allocated; the caller holds the channel's lock
        scratch.last_attempts = 0
        try:
            rows, scores, info = st._recommend_host(query, liked_rows, weights, exclude_rows, k, kc, row_filter, shadow_max_k,
                                                    exchange=x, shadow_eps=shadow_eps, scratch=scratch)
        finally:
            # every attempt that reached the exchange consumed one sequence number on every rank, whether it succeeded or
            # failed (peer timeout, diverged request order); argument errors are raised before any exchange (0 attempts)
            self._seq[channel] += scratch.last_attempts
        return rows, scores, info

    def exchange_merge(self, local: torch.Tensor, k: int, channel: int = 0) -> torch.Tensor:
        """P2P exchange + merge of a packed local result (int64 [2k+2]) -> packed merged result (+1 word: error flag)."""
        lib = nat.load()
        out = self._p2p_out.get((k, channel))
        if out is None:
            out = self._p2p_out[(k, channel)] = torch.zeros(2 * k + 3, dtype=torch.int64, device=self.device)   # last word: error flag
        x = self.exchange_struct(channel, self.next_seq(channel))
        nat.check(lib.rebert_exchange_merge(C.byref(x), k, local.data_ptr(), out.data_ptr(), out.data_ptr() + 8 * (2 * k + 2),
                                            torch.cuda.current_stream().cuda_stream))
        return out

    def enqueue_fused(self, k: int, kc: int, row_filter: Optional[RowFilter], channel: int = 0) -> torch.Tensor:
        """Device-resident sharded step for an already staged query (bench `value` loop): ONE launch per rank — local fast +
        exact pass, exchange and merge in the kernel's tail.  Returns the packed merged result (+1 word: error flag)."""
        ptr, ne = self._excl
        out = self._p2p_out.get((k, channel))
        if out is None:
            out = self._p2p_out[(k, channel)] = torch.zeros(2 * k + 3, dtype=torch.int64, device=self.device)
        x = self.exchange_struct(channel, self.next_seq(channel))
        self.store.enqueue_fused(k, kc, ptr, ne, row_filter, exchange=x, err_ptr=out.data_ptr() + 8 * (2 * k + 2), out_ptr=out.data_ptr())
        return out

    def stage(self, query, liked_rows, weights, exclude_rows, k, kc):
        st = self.store
        self._excl = st.stage_inputs(query, liked_rows, weights, exclude_rows, k, kc, profile_partial_only=True)
        if liked_rows is None:
            return None
        s = st._scratch()
        return torch.cat([s.sum64, s.wsum])                      # fp64 [ld + 1] partial profile

    def set_profile(self, summed: torch.Tensor):
        st = self.store
        s = st._scratch()
        s.sum64.copy_(summed[:st.ld])
        # wsum is summed over ranks too, but every rank added the full weight sum: divide it back
        s.wsum.copy_(summed[st.ld:] / self._world)
        st.finalize_profile()

    def sweep_local(self, threshold: float, row_filter: Optional[RowFilter]):
        ptr, ne = self._excl
        return self.store.sweep_above(threshold, ptr, ne, row_filter)

    def count_local(self, threshold: float, row_filter: Optional[RowFilter]) -> int:
        ptr, ne = self._excl
        return self.store.count_above(threshold, ptr, ne, row_filter)

    def local_topk(self, k: int, kc: int, row_filter: Optional[RowFilter]) -> torch.Tensor:
        ptr, ne = self._excl
        return self.store.enqueue_fused(k, kc, ptr, ne, row_filter)

    def merge(self, gathered: torch.Tensor, k: int) -> torch.Tensor:
        """gathered int64 [G, 2k+2] packed per-rank results -> packed merged result int64 [2k+2] (margin = min)."""
        lib = nat.load()
        g = gathered.shape[0]
        out = self._merged.get(k)
        if out is None:
            out = self._merged[k] = torch.empty(2 * k + 2, dtype=torch.int64, device=self.device)
        base, w = gathered.data_ptr(), 2 * k + 2
        ob = out.data_ptr()
        nat.check(lib.rebert_merge_topk(base, base + 8 * k, base + 16 * k, w, w, 2 * w, g, 1, k, ob, ob + 8 * k, ob + 16 * k,
                                        torch.cuda.current_stream().cuda_stream))
        out[2 * k + 1:2 * k + 2].view(torch.float64).copy_(gathered[:, 2 * k + 1].view(torch.float64).min().reshape(1))
        return out

    def fetch(self, packed: torch.Tensor, k: int):
        """ONE pinned D2H copy of the packed result (and, on the P2P path, its trailing error word), then a stream sync."""
        n = packed.numel()
        host = self._host.get(n)
        if host is None:
            host = self._host[n] = torch.empty(n, dtype=torch.int64).pin_memory()
        host.copy_(packed, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        words = host.numpy()
        if n == 2 * k + 3 and int(words[2 * k + 2:].view(np.int32)[0]) != 0:
            code = int(words[2 * k + 2:].view(np.int32)[0])
            raise RuntimeError(f"rank {code - 101} answered a different request on this channel" if code > 100
                               else f"peer {code - 1} did not deliver its result to the exchange kernel")
        return unpack_result(words, k)


class ShardedCatalog:
    """The sharding layer.  Every rank calls recommend() with the same arguments and gets the same answer.

    Drop-in for CatalogStore under robot_ebert_b200.lib (row_of / id_of / recommend / build_profiles / score_subset).
    Thread safety: requests on one `channel` are serialised by a lock and must be issued in the same order by every
    rank (each serving thread of a rank uses its own channel, the same one as its counterparts on the other ranks);
    requests on different channels run concurrently.  A request tag travels with every rank's result, so ranks whose
    request order on a channel diverged get an error instead of a merged answer to two different requests."""

    def __init__(self, backend, n_total: int, group=None, ids: Optional[Sequence[str]] = None):
        self.backend = backend
        self.group = group
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self.plan = ShardPlan(n_total, self.world)
        backend._world = self.world
        self._gather = {}
        self.ids = list(ids) if ids is not None else None
        self._row_of = None
        self._locks = [threading.Lock() for _ in range(max(1, getattr(backend, "channels", 1)))]
        self._kc_for_k = {}
        self.q8_eps = None

    @classmethod
    def synthetic(cls, seed: int, n_total: int, d: int, dtype: str = "bf16", scale_rows: bool = False, device=None,
                  group=None) -> "ShardedCatalog":
        plan = ShardPlan(n_total, dist.get_world_size(group))
        row0, n = plan.range(dist.get_rank(group))
        store = CatalogStore.synthetic(seed, n, d, dtype, scale_rows=scale_rows, device=device, row0=row0)
        backend = CudaShardBackend(store)
        backend.setup_p2p(group)
        sc = cls(backend, n_total, group)
        sc.warm_up()
        return sc

    @classmethod
    def from_host(cls, ids: Optional[Sequence[str]], matrix: np.ndarray, dtype: str = "fp32", device=None, group=None,
                  sort_ids: bool = True) -> "ShardedCatalog":
        """Every rank passes the SAME [N, D] host matrix (what Chroma's collection.get returns, constants.py:55) and keeps
        only its contiguous slice of the id-sorted rows in HBM; the id table stays whole on every rank."""
        ids, matrix = validated_table(ids, matrix, sort_ids)
        n = matrix.shape[0]
        plan = ShardPlan(n, dist.get_world_size(group))
        row0, cnt = plan.range(dist.get_rank(group))
        store = CatalogStore.from_host(None, matrix[row0:row0 + cnt], dtype, device=device, row_base=row0)
        backend = CudaShardBackend(store)
        backend.setup_p2p(group)
        sc = cls(backend, n, group, ids)
        sc.warm_up()
        return sc

    def warm_up(self) -> None:
        """Run one request through every kernel variant the request path can take (candidate lists of 32 / 64 / 128 / 256
        keys, query / liked rows / weighted liked rows) on every channel's scratch.  Collective; called by the constructors,
        BEFORE any serving thread exists.  Why: the first launch of a kernel loads its module (CUDA lazy loading) and the
        first use of a scratch allocates — both may synchronise the device, and a device synchronisation while another
        channel's kernel is waiting for a peer (whose progress may hang on the mirrored event) stalls both ranks until the
        exchange times out.  After the warm-up the request path makes no such call."""
        if getattr(self.backend, "exchange", "nccl") != "p2p":
            return
        st = self.backend.store
        n = self.plan.n_total
        q = np.ones(st.d, dtype=np.float32)
        liked = np.arange(min(3, n), dtype=np.int64)
        for k in (10, 40, 100, 200):
            kk = max(1, min(k, n))
            self.recommend(query=q, k=kk)
            self.recommend(liked_rows=liked, exclude_rows=liked, k=kk)
        self.recommend(liked_rows=liked, weights=np.ones(len(liked), dtype=np.float32), k=max(1, min(10, n)))
        for ch in range(1, self.backend.channels):          # every channel's flags and scratch have been through one request
            self.recommend(query=q, k=max(1, min(10, n)), channel=ch)
        torch.cuda.synchronize(self.backend.device)
        dist.barrier(group=self.group)

    # ------------------------------------------------------------------ id map (global rows) ----
    def row_of(self, tmdb_id: str) -> Optional[int]:
        if self._row_of is None:
            if self.ids is None:
                raise ValueError("catalog has no id table")
            self._row_of = {i: r for r, i in enumerate(self.ids)}
        return self._row_of.get(tmdb_id)

    def id_of(self, row: int) -> str:
        return self.ids[row] if self.ids is not None else str(row)

    def build_profiles(self, row_ptr, col, w=None):
        """Sharded CatalogStore.build_profiles: fp64 partial sums all-reduced before the division (identical on every rank)."""
        return self.backend.store.build_profiles(
            row_ptr, col, w, reduce_fn=lambda t: dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group))

    def score_subset(self, p64: torch.Tensor, sub_rows: np.ndarray) -> np.ndarray:
        """fp64 scores of `sub_rows` (global ids, any shard) against prepared profiles (lib.py:105-106): each rank scores
        the rows it owns, one all-reduce puts them together."""
        st = self.backend.store
        local = torch.from_numpy(st.score_subset(p64, sub_rows)).to(st.device)
        local = torch.nan_to_num(local, nan=0.0)                   # rows of other shards come back NaN
        dist.all_reduce(local, op=dist.ReduceOp.SUM, group=self.group)
        return local.cpu().numpy()

    def enable_prefilter(self) -> float:
        """Build every rank's int8 prefilter shadow (CatalogStore.enable_prefilter).  The proof bound is the LARGEST bound
        over the ranks, so that every rank takes the same proven / not-proven decision.  Collective."""
        eps = self.backend.store.enable_prefilter()
        t = torch.tensor([eps], dtype=torch.float64, device=self.backend.device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
        self.q8_eps = float(t.item())
        if getattr(self.backend, "exchange", "nccl") == "p2p":          # warm the shadow's kernel variants up too (see warm_up)
            self.recommend(query=np.ones(self.backend.store.d, dtype=np.float32), k=max(1, min(10, self.plan.n_total)), prefilter=True)
            torch.cuda.synchronize(self.backend.device)
            dist.barrier(group=self.group)
        return self.q8_eps

    def _gather_buf(self, k: int, like: torch.Tensor) -> torch.Tensor:
        buf = self._gather.get(k)
        if buf is None:
            buf = self._gather[k] = torch.empty((self.world, 2 * k + 2), dtype=torch.int64, device=like.device)
        return buf

    def enqueue(self, k: int, kc: int, row_filter=None, channel: int = 0) -> torch.Tensor:
        """Device-resident step for an already staged query: local top-k -> exchange -> merge (packed result)."""
        if getattr(self.backend, "exchange", "nccl") == "p2p":
            return self.backend.enqueue_fused(k, kc, row_filter, channel)   # one launch: fast + exact pass + exchange + merge
        local = self.backend.local_topk(k, kc, row_filter)
        buf = self._gather_buf(k, local)
        dist.all_gather_into_tensor(buf.view(-1), local, group=self.group)
        return self.backend.merge(buf, k)

    def recommend(self, *, query=None, liked_rows=None, weights=None, exclude_rows=None, k: int = 10, row_filter=None,
                  return_info: bool = False, prefilter: Optional[bool] = None, channel: int = 0):
        if (query is None) == (liked_rows is None):
            raise ValueError("pass exactly one of query / liked_rows")
        if k <= 0:
            raise ValueError("k must be positive")
        if liked_rows is not None and len(liked_rows) == 0:
            raise ValueError(EMPTY_PROFILE)
        p2p = getattr(self.backend, "exchange", "nccl") == "p2p"
        if not 0 <= channel < len(self._locks):
            raise ValueError(f"channel must be in [0, {len(self._locks)})")
        lock = self._locks[channel] if p2p else getattr(self.backend, "_nccl_lock", self._locks[0])
        with lock:
            return self._recommend_locked(query, liked_rows, weights, exclude_rows, k, row_filter, return_info, prefilter,
                                          channel, p2p)

    def _recommend_locked(self, query, liked_rows, weights, exclude_rows, k, row_filter, return_info, prefilter, channel, p2p):
        kc = self._kc_for_k.get(k)
        if kc is None:
            kc = self._kc_for_k[k] = nat.load().rebert_candidates_for_k(k)
        eps = getattr(getattr(self.backend, "store", None), "fast_eps", 0.0)
        if kc == 0:
            # k beyond the register-list kernel (k > 240): sharded threshold bisection + sweep, still exact (slower route)
            rows, scores = self._recommend_large_k(query, liked_rows, weights, exclude_rows, k, row_filter, eps)
            if return_info:
                return rows, scores, {"kc": 0, "margin": float("inf"), "proven_exact": True, "exact_sweep": True}
            return rows, scores
        if prefilter and self.q8_eps is None:
            raise ValueError("prefilter=True needs enable_prefilter()")
        if p2p:
            # the whole request is ONE C call per rank (no torch ops, no NCCL): staging, profile exchange, fused scoring
            # launch with the result exchange in its tail, proof loop
            rows, scores, info = self.backend.recommend_host(query, liked_rows, weights, exclude_rows, k, kc, row_filter, channel,
                                                             CatalogStore.shadow_max_k(self.q8_eps is not None, prefilter),
                                                             self.q8_eps)
            margin, proven, kc = info["margin"], info["proven_exact"], info["kc"]
        else:
            def attempt(kc):
                self._stage(query, liked_rows, weights, exclude_rows, k, kc)
                return self.backend.fetch(self.enqueue(k, kc, row_filter), k)

            rows, scores, margin, kc = widen_until_proven(attempt, kc, eps)
            proven = margin > eps
            info = {"kc": kc, "margin": margin, "proven_exact": proven, "exact_sweep": False}
        if not proven:
            # Fail closed (close_proof).  The margin is the same on every rank, so all ranks take this branch together, and
            # every branch inside it depends on all-reduced counts and all-gathered sweeps: the collectives stay aligned.
            self._stage(query, liked_rows, weights, exclude_rows, k, kc)         # the sweeps read torch scratch
            rows, scores = close_proof(rows, scores, k, eps, margin, *self._sweeps(row_filter))
            info = dict(info, proven_exact=True, exact_sweep=True)
        if return_info:
            return rows, scores, info
        return rows, scores

    def _stage(self, query, liked_rows, weights, exclude_rows, k, kc):
        """Collective: stage the request on every rank; a liked-rows profile is completed by an all-reduce of the partials."""
        partial = self.backend.stage(query, liked_rows, weights, exclude_rows, k, kc)
        if partial is not None:
            dist.all_reduce(partial, op=dist.ReduceOp.SUM, group=self.group)
            self.backend.set_profile(partial)

    def _recommend_large_k(self, query, liked_rows, weights, exclude_rows, k, row_filter, eps):
        """Sharded form of CatalogStore._recommend_large_k: large_k_search over the whole catalog (see _sweeps)."""
        CatalogStore._check_large_k(k)
        self._stage(query, liked_rows, weights, exclude_rows, 1, 32)
        return large_k_search(*self._sweeps(row_filter), k, eps)

    def _sweeps(self, row_filter):
        """(count, sweep) of large_k_search / close_proof over every shard, for the staged request: the count is all-reduced
        and the survivors all-gathered, so every rank sees the same values, takes the same branches and orders alike."""
        dev = self.backend.device

        def count(thr):
            c = torch.tensor([self.backend.count_local(thr, row_filter)], dtype=torch.int64, device=dev)
            dist.all_reduce(c, op=dist.ReduceOp.SUM, group=self.group)
            return int(c.item())

        return count, lambda thr: self._sweep_gather(thr, row_filter)

    def _sweep_gather(self, threshold: float, row_filter):
        """(global rows, exact fp64 scores) of every allowed row of ANY shard whose fast score >= threshold, identical on
        every rank; None if some shard overflowed its sweep buffer."""
        local = self.backend.sweep_local(threshold, row_filter)
        dev = self.backend.device
        n_loc = torch.tensor([-1 if local is None else len(local[0])], dtype=torch.int64, device=dev)
        counts = torch.empty(self.world, dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(counts, n_loc, group=self.group)
        counts = counts.cpu().numpy()
        if (counts < 0).any():
            return None
        cap = int(counts.max())
        if cap == 0:
            return np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.float64)
        mine = torch.zeros(2 * cap, dtype=torch.int64, device=dev)
        if len(local[0]):
            mine[:len(local[0])] = torch.from_numpy(np.ascontiguousarray(local[0], dtype=np.int64)).to(dev)
            mine[cap:cap + len(local[0])] = torch.from_numpy(np.ascontiguousarray(local[1], dtype=np.float64).view(np.int64)).to(dev)
        allr = torch.empty((self.world, 2 * cap), dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(allr.view(-1), mine, group=self.group)
        allr = allr.cpu().numpy()
        rr = np.concatenate([allr[g, :counts[g]] for g in range(self.world)])
        sc = np.concatenate([allr[g, cap:cap + counts[g]].view(np.float64) for g in range(self.world)])
        return rr, sc

    # ------------------------------------------------------------------ batched (tensor-core) path ----------
    def batch_context(self, qbf: torch.Tensor, qn64: torch.Tensor, k: int, excl_ptr=None, excl_col=None, row_filter=None, qn32=None,
                      query_filters: Optional[QueryFilters] = None):
        """Allocate everything a batched step needs (device tensors only) for prepared queries [b, ld].  With qn32 given and
        an int8 shadow the GEMM can use (enable_prefilter), the step runs on int8 operands.  query_filters: one genre / year
        test per query, tested against this rank's own metadata (set_metadata on backend.store)."""
        import ctypes as C
        store: CatalogStore = self.backend.store
        lib = nat.load()
        dev = store.device
        b = qbf.shape[0]
        if query_filters is not None:
            query_filters.validate(b, row_filter, store.genre_bits, store.year)
        shadow = store.quantize_queries(qn32) if (qn32 is not None and store.batch_shadow_ok) else None
        if shadow is None and not store.batch_gemm_ok:
            raise nat.NativeError(nat.ERR_UNSUPPORTED, f"batch_context: the tcgen05 GEMM takes neither this {store.dtype} shard "
                                                       f"(ld={store.ld}) nor an int8 shadow of it")
        plan = store.gemm_plan(b, k, shadow=shadow is not None)
        ep = ec = None
        if excl_ptr is not None:
            excl_ptr, excl_col = sorted_csr(excl_ptr, excl_col)
            ep = torch.from_numpy(excl_ptr).to(dev)
            ec = torch.from_numpy(excl_col).to(dev)
        hb = (b + 1) // 2
        words = 2 * b * k + 2 * hb                                       # rows | scores | counts | status
        ctx = {"b": b, "k": k, "plan": plan, "row_filter": row_filter, "query_filters": query_filters, "qbf": qbf, "qn64": qn64, "ep": ep, "ec": ec, "hb": hb, "words": words,
               "shadow": shadow,
               "ws": torch.empty(lib.rebert_gemm_workspace_bytes(C.byref(store._c), C.byref(plan)), dtype=torch.uint8, device=dev),
               "local": torch.empty(words, dtype=torch.int64, device=dev),
               "gathered": torch.empty((self.world, words), dtype=torch.int64, device=dev),
               "m_rows": torch.empty((b, k), dtype=torch.int64, device=dev),
               "m_scores": torch.empty((b, k), dtype=torch.float64, device=dev),
               "m_count": torch.empty(b, dtype=torch.int32, device=dev)}
        return ctx

    def batch_step(self, ctx) -> None:
        """Device-resident batched step: per-rank tcgen05 pass -> ONE packed all-gather -> merge.  No host sync."""
        store: CatalogStore = self.backend.store
        lib = nat.load()
        b, k, hb, words, local = ctx["b"], ctx["k"], ctx["hb"], ctx["words"], ctx["local"]
        o_rows, o_scores = local[:b * k], local[b * k:2 * b * k].view(torch.float64)
        o_count = local[2 * b * k:2 * b * k + hb].view(torch.int32)
        o_status = local[2 * b * k + hb:].view(torch.int32)
        store.enqueue_batch(ctx["plan"], ctx["qbf"], ctx["qn64"], ctx["ep"], ctx["ec"], ctx["ws"], o_rows, o_scores, o_count, o_status,
                            ctx.get("row_filter"), shadow=ctx.get("shadow"), query_filters=ctx.get("query_filters"))
        dist.all_gather_into_tensor(ctx["gathered"].view(-1), local, group=self.group)
        base = ctx["gathered"].data_ptr()
        nat.check(lib.rebert_merge_topk(base, base + 8 * b * k, base + 16 * b * k, words, words, 2 * words, self.world, b, k,
                                        ctx["m_rows"].data_ptr(), ctx["m_scores"].data_ptr(), ctx["m_count"].data_ptr(),
                                        torch.cuda.current_stream().cuda_stream))

    def batch_collect(self, ctx, queries, excl_ptr=None, excl_col=None, *, liked_ptr=None, liked_col=None, liked_w=None,
                      prefilter: Optional[bool] = False):
        """Second half of a batched step: read the merged results and the per-query status back, and re-run every query some
        rank could not prove through the sharded single-query route (identical decisions on every rank), with `prefilter`.
        The batch is queries [b, d] or, with queries None, the liked CSR (+ optional weights) its profiles were built from.
        Returns (rows [b, k], scores [b, k], counts [b], status [b])."""
        b, k, hb = ctx["b"], ctx["k"], ctx["hb"]
        status = ctx["gathered"][:, 2 * b * k + hb:].contiguous().view(torch.int32)[:, :b].max(dim=0).values   # any rank unsure
        rows, scores = ctx["m_rows"].cpu().numpy(), ctx["m_scores"].cpu().numpy()
        counts, status = ctx["m_count"].cpu().numpy(), status.cpu().numpy()
        self._rerun(np.nonzero(status)[0], queries, liked_ptr, liked_col, liked_w, excl_ptr, excl_col, k, ctx.get("row_filter"),
                    prefilter, rows, scores, counts, ctx.get("query_filters"))
        return rows, scores, counts, status

    def _rerun(self, users, queries, liked_ptr, liked_col, liked_w, excl_ptr, excl_col, k, row_filter, prefilter,
               rows, scores, counts, query_filters=None):
        """Sharded single-query route (recommend) for `users` of a batch of queries or of a liked CSR with optional weights,
        each with its segment of the exclusion CSR and its own filter (user_row_filter).  `users` must be the same on every rank (the collectives stay aligned).
        Overwrites those users' rows / scores / counts."""
        ecp = None if excl_ptr is None else np.asarray(excl_ptr, dtype=np.int64)
        eca = None if excl_col is None else np.asarray(excl_col)
        if queries is None:
            lpn, lcol = np.asarray(liked_ptr, dtype=np.int64), np.asarray(liked_col)
            lw = None if liked_w is None else np.asarray(liked_w)
        for u in users:
            ex = None if ecp is None else eca[ecp[u]:ecp[u + 1]]
            rf = user_row_filter(query_filters, u, row_filter)
            if queries is not None:
                r, sc = self.recommend(query=np.asarray(queries[u]), exclude_rows=ex, k=k, row_filter=rf, prefilter=prefilter)
            else:
                seg = slice(lpn[u], lpn[u + 1])
                r, sc = self.recommend(liked_rows=lcol[seg], weights=None if lw is None else lw[seg], exclude_rows=ex, k=k,
                                       row_filter=rf, prefilter=prefilter)
            rows[u, :], scores[u, :] = -1, -np.inf
            rows[u, :len(r)], scores[u, :len(r)], counts[u] = r, sc, len(r)

    def recommend_batch(self, *, queries=None, liked_ptr=None, liked_col=None, liked_w=None, excl_ptr=None, excl_col=None,
                        k: int = 10, row_filter=None, return_info: bool = False, query_filters: Optional[QueryFilters] = None):
        """Sharded form of CatalogStore.recommend_batch: every rank runs the tcgen05 pass over its rows, the per-rank
        [b, k] results are all-gathered in ONE packed buffer and merged on every rank.  CUDA backend only.
        k up to 2048 runs on the tensor cores when every shard is above the plan minimum (rebert_gemm_plan); the packed buffer
        is 2 b k + b words per rank (128 MiB at b = 4096, k = 2048).  Larger k, and smaller shards, take the per-query loop."""
        store: CatalogStore = self.backend.store
        with torch.cuda.device(store.device):
            qn32, qn64, qbf = store.prepare_batch(queries, liked_ptr, liked_col, liked_w,
                                                  reduce_fn=lambda t: dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group))
            try:
                ctx = self.batch_context(qbf, qn64, k, excl_ptr, excl_col, row_filter, qn32=qn32, query_filters=query_filters)
            except nat.NativeError as e:
                if e.code != nat.ERR_UNSUPPORTED:
                    raise
                ctx = None           # shard too small for the tensor-core scheme, or of a dtype / width it does not take (same
                                     # verdict on every rank: equal shard sizes, one dtype and width)
            if ctx is None:
                return self._recommend_batch_loop(queries, liked_ptr, liked_col, liked_w, excl_ptr, excl_col, k, row_filter,
                                                  return_info, query_filters)
            self.batch_step(ctx)
            rows, scores, counts, status = self.batch_collect(ctx, queries, excl_ptr, excl_col, liked_ptr=liked_ptr,
                                                              liked_col=liked_col, liked_w=liked_w, prefilter=None)
        if return_info:
            plan = ctx["plan"]
            return rows, scores, counts, {"status": status, "plan": {f: getattr(plan, f) for f, _ in plan._fields_}}
        return rows, scores, counts

    def _recommend_batch_loop(self, queries, liked_ptr, liked_col, liked_w, excl_ptr, excl_col, k, row_filter, return_info,
                              query_filters=None):
        """Small shards: every query of the batch goes through the sharded single-query path (identical on all ranks)."""
        b = len(queries) if queries is not None else len(liked_ptr) - 1
        if query_filters is not None:
            query_filters.validate(b, row_filter, self.backend.store.genre_bits, self.backend.store.year)
        rows = np.full((b, k), -1, dtype=np.int64)
        scores = np.full((b, k), -np.inf, dtype=np.float64)
        counts = np.zeros(b, dtype=np.int32)
        self._rerun(range(b), queries, liked_ptr, liked_col, liked_w, excl_ptr, excl_col, k, row_filter, None, rows, scores, counts,
                    query_filters)
        if return_info:
            return rows, scores, counts, {"status": np.zeros(b, dtype=np.int32), "plan": None}
        return rows, scores, counts
