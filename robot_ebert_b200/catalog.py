"""HBM-resident catalog store and the single-request scoring call.

Replaces the process-global DataFrame `movies_collab_embeddings` (reference
src/backend/app/constants.py:55-56) and the pandas/sklearn expressions at src/backend/app/lib.py:44-55.
torch is used for device memory, pinned staging and streams only; all arithmetic happens in
librebert_b200.so (hand-written sm_100a kernels) through the C ABI in include/rebert_b200.h.
There is no CPU path: without a CUDA device and the built library every call raises.
"""
from __future__ import annotations

import ctypes as C
import threading
from typing import Optional, Sequence, Tuple

import numpy as np
import torch

from . import _native as nat


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _align(x: int, a: int = 16) -> int:
    return (x + a - 1) // a * a


class RowFilter:
    """Optional row predicate beside the seen-movie exclusion (BASELINE config 5: genre / year)."""

    def __init__(self, genre_any: int = 0, year_lo: int = 0, year_hi: int = 65535,
                 exclude_bitmap: Optional[torch.Tensor] = None):
        self.genre_any, self.year_lo, self.year_hi = int(genre_any), int(year_lo), int(year_hi)
        self.exclude_bitmap = exclude_bitmap

    @property
    def has_genre_or_year(self) -> bool:
        return bool(self.genre_any) or (self.year_lo, self.year_hi) != (0, 65535)


def _unsigned_column(x, name: str, dtype, hi: int) -> np.ndarray:
    a = np.asarray(x)
    if a.ndim != 1 or len(a) == 0:
        raise ValueError(f"QueryFilters.{name} must be a non-empty 1-D array, got shape {a.shape}")
    if not np.issubdtype(a.dtype, np.integer):
        raise ValueError(f"QueryFilters.{name} must hold integers, got {a.dtype}")
    if a.min() < 0 or a.max() > hi:
        raise ValueError(f"QueryFilters.{name} out of range [0, {hi}]")
    return a.astype(dtype)


class QueryFilters:
    """One genre / year predicate per user of a batch (recommend_batch(query_filters=...)).  User u keeps row r iff
    (genre_any[u] == 0 or genre_bits[r] & genre_any[u] != 0) and year_lo[u] <= year[r] <= year_hi[u], on top of its
    exclusion CSR and a shared exclude_bitmap.  (0, 0, 65535) leaves a user unrestricted; year_lo > year_hi allows no row.
    year_lo / year_hi default to the whole range."""

    def __init__(self, genre_any, year_lo=None, year_hi=None):
        self.genre_any = _unsigned_column(genre_any, "genre_any", np.uint32, 0xFFFFFFFF)
        b = len(self.genre_any)
        self.year_lo = _unsigned_column(np.zeros(b, np.uint16) if year_lo is None else year_lo, "year_lo", np.uint16, 65535)
        self.year_hi = _unsigned_column(np.full(b, 65535, np.uint16) if year_hi is None else year_hi, "year_hi", np.uint16, 65535)
        if len(self.year_lo) != b or len(self.year_hi) != b:
            raise ValueError(f"QueryFilters: genre_any, year_lo and year_hi must have one entry per user ({b}, {len(self.year_lo)}, "
                             f"{len(self.year_hi)})")
        self.has_genre = bool(self.genre_any.any())
        self.has_year = bool((self.year_lo != 0).any() or (self.year_hi != 65535).any())
        self._dev = {}

    def __len__(self) -> int:
        return len(self.genre_any)

    def row_filter(self, u: int, exclude_bitmap: Optional[torch.Tensor] = None) -> RowFilter:
        """User u's predicate as the RowFilter of a single request (the per-query route of a batch)."""
        return RowFilter(int(self.genre_any[u]), int(self.year_lo[u]), int(self.year_hi[u]), exclude_bitmap)

    def subset(self, users) -> "QueryFilters":
        users = np.asarray(users, dtype=np.int64)
        return QueryFilters(self.genre_any[users], self.year_lo[users], self.year_hi[users])

    def validate(self, b: int, row_filter: Optional[RowFilter], genre_bits, year) -> None:
        """ValueError unless these filters fit a batch of b users with `row_filter` shared and the catalog's metadata columns
        genre_bits / year (None when set_metadata was not called).  A shared genre or year test is refused: the per-query
        route takes one RowFilter, which cannot hold the AND of two genre masks.  A shared exclude_bitmap is fine."""
        if len(self) != b:
            raise ValueError(f"query_filters has {len(self)} users, the batch {b}")
        if row_filter is not None and row_filter.has_genre_or_year:
            raise ValueError("query_filters cannot be combined with a shared row_filter genre or year test "
                             "(put the shared test into every user's filter instead)")
        if self.has_genre and genre_bits is None:
            raise ValueError("query_filters genre_any needs set_metadata()")
        if self.has_year and year is None:
            raise ValueError("query_filters year range needs set_metadata()")

    def device_arrays(self, dev: torch.device):
        """(genre_any, year_lo, year_hi) on `dev`, copied once per device and kept (int32 / int16 views of the unsigned data)."""
        key = str(dev)
        if key not in self._dev:
            self._dev[key] = tuple(torch.from_numpy(a.view(np.int32 if a.dtype == np.uint32 else np.int16)).to(dev)
                                   for a in (self.genre_any, self.year_lo, self.year_hi))
        return self._dev[key]


def user_row_filter(query_filters: Optional[QueryFilters], u: int, row_filter: Optional[RowFilter]) -> Optional[RowFilter]:
    """The RowFilter the per-query route applies to user u of a batch: the shared row_filter, or with query_filters the
    user's own test plus the shared exclude_bitmap."""
    if query_filters is None:
        return row_filter
    return query_filters.row_filter(u, None if row_filter is None else row_filter.exclude_bitmap)


class _Scratch:
    """Per-thread staging + device scratch so concurrent requests (FastAPI's threadpool) never share buffers."""

    def __init__(self, store: "CatalogStore"):
        self.store = store
        self.in_cap = 0
        self.kc = 0
        self.k_cap = 0
        self.nl_cap = self.ne_cap = self.hk_cap = 0
        dev = store.device
        ld = store.ld
        self.qn32 = torch.zeros(ld, dtype=torch.float32, device=dev)
        self.qn64 = torch.zeros(ld, dtype=torch.float64, device=dev)
        self.sum64 = torch.zeros(ld, dtype=torch.float64, device=dev)
        self.wsum = torch.zeros(1, dtype=torch.float64, device=dev)
        self.info = nat.RequestInfo()                 # reused: one request at a time per scratch (thread / channel)
        self.info_addr = C.addressof(self.info)
        self.last_attempts = 0

    def ensure_host(self, n_liked: int, n_excl: int, k: int):
        """Pinned + device scratch of rebert_recommend_host.  Sized once for any k of the single-request path (256) and lists
        of 4096 entries; longer lists grow it geometrically.  (Growing allocates, and CUDA allocations may synchronise the
        device — harmless on one GPU, but on a row shard a kernel waiting for a peer may be running: the sharding layer
        therefore pre-allocates its channels' scratch while no request is in flight.)"""
        if n_liked > self.nl_cap or n_excl > self.ne_cap or k > self.hk_cap:
            self.nl_cap = max(self.nl_cap, 4096, 1 << max(n_liked - 1, 0).bit_length())
            self.ne_cap = max(self.ne_cap, 4096, 1 << max(n_excl - 1, 0).bit_length())
            self.hk_cap = max(self.hk_cap, 256, 1 << (k - 1).bit_length())
            self.hpin, self.hdev = self._host_scratch(self.nl_cap, self.ne_cap, self.hk_cap)
            self.h_rows = np.empty(self.hk_cap, dtype=np.int64)
            self.h_scores = np.empty(self.hk_cap, dtype=np.float64)
            # raw addresses / sizes, looked up once: the per-request wrapper is on the latency path of small catalogs
            self.host_args = (self.hpin.data_ptr(), self.hpin.numel(), self.hdev.data_ptr(), self.hdev.numel())
            self.out_args = (self.h_rows.ctypes.data, self.h_scores.ctypes.data)

    def _host_scratch(self, nl_cap: int, ne_cap: int, k_cap: int):
        lib = nat.load()
        pb, db = C.c_size_t(0), C.c_size_t(0)
        nat.check(lib.rebert_recommend_host_scratch(C.byref(self.store._c), nl_cap, ne_cap, k_cap, C.byref(pb), C.byref(db)))
        pinned = torch.empty(pb.value, dtype=torch.uint8).pin_memory()
        device = torch.zeros(db.value, dtype=torch.uint8, device=self.store.device)   # zero once (ticket / claim counters)
        return pinned, device

    def ensure_in(self, nbytes: int):
        if nbytes > self.in_cap:
            cap = max(4096, 1 << (nbytes - 1).bit_length())
            self.h_in = torch.empty(cap, dtype=torch.uint8).pin_memory()
            self.d_in = torch.empty(cap, dtype=torch.uint8, device=self.store.device)
            self.h_in_np = self.h_in.numpy()
            self.in_cap = cap

    def ensure_out(self, k: int, kc: int):
        if kc != self.kc:
            lib = nat.load()
            wsb = lib.rebert_gemv_workspace_bytes(self.store.n, kc)
            self.ws = torch.zeros(wsb, dtype=torch.uint8, device=self.store.device)   # zero once: holds the ticket counter
            self.cand = torch.empty(kc, dtype=torch.int64, device=self.store.device)   # u64 keys
            self.kc = kc
        if k != self.k_cap:
            # packed result, int64 words: rows[k] | scores[k] (fp64 bits) | count (int32, low half) | margin (fp64 bits)
            self.d_out = torch.empty(2 * k + 2, dtype=torch.int64, device=self.store.device)
            self.h_out = torch.empty(2 * k + 2, dtype=torch.int64).pin_memory()
            self.h_out_np = self.h_out.numpy()
            self.k_cap = k


def sorted_unique_i32(rows) -> np.ndarray:
    """Sorted, duplicate-free int32 copy of an exclusion list; already strictly increasing input (what the id->row
    lookup of lib.get_user_recs produces) is passed through without the sort."""
    ex = np.ascontiguousarray(rows, dtype=np.int32)
    if ex.ndim != 1:
        ex = ex.reshape(-1)
    if ex.size > 1 and not np.all(ex[1:] > ex[:-1]):
        ex = np.unique(ex)
    return ex


def _raw_stream(dev_index: int) -> int:
    """cudaStream_t of torch's current stream on the device (the request path's launches go there)."""
    return _get_raw_stream(dev_index) if _get_raw_stream is not None else torch.cuda.current_stream(dev_index).cuda_stream


# building a torch.cuda.Stream object per request costs ~2 us; torch exposes the raw handle directly (what its own compiled
# graphs use), with the public API as the fallback
_get_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


class _on_device:
    """`with torch.cuda.device(dev)` only when dev is not already current (the context manager costs ~8 us per request)."""

    __slots__ = ("ctx",)

    def __init__(self, dev: torch.device):
        self.ctx = None if torch.cuda.current_device() == (dev.index or 0) else torch.cuda.device(dev)

    def __enter__(self):
        if self.ctx is not None:
            self.ctx.__enter__()

    def __exit__(self, *a):
        if self.ctx is not None:
            self.ctx.__exit__(*a)


def sorted_csr(ptr, col):
    """Validate a ragged CSR (ptr monotone, within bounds) and return it with every segment sorted ascending, as the
    device-side binary searches require.  Already-sorted input (the common case) is returned without copying."""
    ptr = np.asarray(ptr, dtype=np.int64)
    col = np.asarray(col, dtype=np.int32)
    if ptr.ndim != 1 or ptr.size < 1 or ptr[0] != 0 or ptr[-1] != col.size or np.any(np.diff(ptr) < 0):
        raise ValueError("malformed CSR: ptr must start at 0, be non-decreasing and end at len(col)")
    if col.size > 1:
        desc = np.nonzero(np.diff(col) < 0)[0] + 1                 # positions where the order drops ...
        bad = np.setdiff1d(desc, ptr[1:-1], assume_unique=False)   # ... other than at a segment boundary
        if bad.size:
            col = col.copy()
            for u in np.unique(np.searchsorted(ptr, bad, side="right") - 1):
                col[ptr[u]:ptr[u + 1]].sort()
    return ptr, col


def unpack_result(words: np.ndarray, k: int):
    """Split a packed result (see _Scratch.ensure_out) into (rows int64[k'], scores f64[k'], margin)."""
    cnt = int(words[2 * k:2 * k + 1].view(np.int32)[0])
    margin = float(words[2 * k + 1:2 * k + 2].view(np.float64)[0])
    return words[:cnt].copy(), words[k:k + cnt].view(np.float64).copy(), margin


# same failure the reference hits: sklearn's check_array on an empty frame (SURVEY.md §3.2)
EMPTY_PROFILE = "Found array with 0 sample(s): user has no liked movies in the catalog"


def validated_table(ids, matrix, sort_ids: bool):
    """Host catalog as fp32 [N, D] and its id table (str) checked against it; with sort_ids, both in ascending id order."""
    matrix = np.asarray(matrix, dtype=np.float32)
    if matrix.ndim != 2:
        raise ValueError("matrix must be [N, D]")
    n = matrix.shape[0]
    if ids is not None:
        if len(ids) != n:
            raise ValueError("len(ids) != rows")
        ids = [str(i) for i in ids]
        if len(set(ids)) != n:
            raise ValueError("duplicate ids")
        if sort_ids:
            order = sorted(range(n), key=ids.__getitem__)
            if order != list(range(n)):
                matrix = matrix[np.asarray(order)]
                ids = [ids[i] for i in order]
    return ids, matrix


def topk_order(rows: np.ndarray, scores: np.ndarray, k: int):
    """The first k of (rows, scores) in result order: score desc, row asc."""
    order = np.lexsort((rows, -scores))[:k]
    return rows[order], scores[order]


def widen_until_proven(attempt, kc: int, eps: float):
    """attempt(kc) -> (rows, scores, margin) with 4x more candidates each time, until the margin clears eps or kc reaches
    256.  Returns (rows, scores, margin, kc) of the last attempt; the caller checks margin > eps."""
    while True:
        rows, scores, margin = attempt(kc)
        if margin > eps or kc >= 256:
            return rows, scores, margin, kc
        kc = min(256, kc * 4)


def close_proof(rows, scores, k: int, eps: float, margin: float, count, sweep):
    """Fail closed: the exact top-k of a request whose candidate list (rows, scores) did not prove itself (margin <= eps),
    or RuntimeError.  count / sweep as in large_k_search, over the staged request.

    Mass ties: more rows than any candidate list holds sit within fp32 noise of the k-th score.  The sweep collects every
    allowed row that could still belong to the top-k (fast score >= k-th exact score - 2 eps) and orders them by fp64
    score: provably exact.  If it overflows (or fewer than k rows are allowed), the bisection route of large_k_search
    handles any tie mass it can hold."""
    if len(rows) == k:
        res = sweep(float(scores[k - 1]) - 2.0 * eps)
        if res is not None and len(res[0]) >= k:
            return topk_order(res[0], res[1], k)
    try:
        return large_k_search(count, sweep, k, eps)
    except RuntimeError as e:
        raise RuntimeError(f"top-{k}: the result cannot be proven exact (margin {margin:.3e} <= {eps:.3e}) and the "
                           f"exhaustive route failed: {e}") from e


def large_k_search(count, sweep, k: int, eps: float):
    """Exact top-k for k beyond the register-list kernel (k > 240), on one shard or across shards.

    count(thr) -> number of allowed rows whose fast score >= thr;  sweep(thr) -> (global rows int64, exact fp64 scores) of
    those rows, or None on overflow.  Bisection finds a threshold that at least k (and at most ~2k) rows reach; the
    collected rows are ordered by (exact score desc, row asc) and the threshold is lowered until the k-th exact score
    clears it by 2 eps (eps = bound on |fast - exact|) — then no row outside the collected set can belong to the top-k."""
    total = count(-2.0)                                   # every allowed row (scores live in [-1, 1])
    if total <= k:
        thr = -2.0
    else:
        lo, hi = -2.0, 1.5                                # count(lo) >= k, count(hi) = 0
        for _ in range(40):
            mid = 0.5 * (lo + hi)
            c = count(mid)
            if c >= k:
                lo = mid
                if c <= 2 * k:
                    break
            else:
                hi = mid
        thr = lo
    while True:
        res = sweep(thr)
        if res is None:
            raise RuntimeError("large-k sweep overflow: more than SWEEP_CAP rows within the threshold band")
        rr, sc = topk_order(res[0], res[1], k)
        if len(res[0]) >= total or len(rr) < k or sc[-1] - 2.0 * eps > thr:
            return rr, sc
        thr = float(sc[-1]) - 4.0 * eps - 1e-6            # k-th exact score too close to the cut: widen


class CatalogStore:
    """One catalog shard in HBM: rows [n, ld] (fp32 or bf16), fp32 inv_norm[n], fp64 norm64[n].

    Rows are kept in ascending tmdb_id *string* order, so "row ascending" is the tie-break of lib.py:55,63.
    """

    def __init__(self, rows: torch.Tensor, inv_norm: torch.Tensor, norm64: torch.Tensor, n: int, d: int, ld: int,
                 dtype: str, row_base: int = 0, ids: Optional[Sequence[str]] = None):
        self.rows, self.inv_norm, self.norm64 = rows, inv_norm, norm64
        self.n, self.d, self.ld, self.dtype, self.row_base = int(n), int(d), int(ld), dtype, int(row_base)
        self.device = rows.device
        self.ids = list(ids) if ids is not None else None
        self._row_of = None
        self.genre_bits: Optional[torch.Tensor] = None
        self.year: Optional[torch.Tensor] = None
        self._tls = threading.local()
        self._c = nat.Catalog(rows=rows.data_ptr(), inv_norm=inv_norm.data_ptr(), norm64=norm64.data_ptr(), n=self.n,
                              row_base=self.row_base, d=self.d, ld=self.ld, dtype=nat.DTYPES[dtype], reserved=0)
        esize = 2 if dtype == "bf16" else 4
        chunks, epc = self.ld * esize // 16, 16 // esize
        self.elements_per_lane = epc if chunks <= 16 else (chunks // 32) * epc   # mirrors csrc row_layout()
        # fp32 error bound of the fast pass on a unit-vector dot (DESIGN.md §exactness)
        self.fast_eps = float((self.elements_per_lane + 12) * 2.0 ** -24)
        self._c8 = None            # int8 prefilter shadow (enable_prefilter)
        self.q8_eps = float("inf")
        self._dev_index = self.device.index if self.device.index is not None else 0
        self._c_addr = C.addressof(self._c)
        self._plain_proof = nat.Proof()      # read-only, shared by every request that does not try the shadow
        self._plain_proof.fast_eps, self._plain_proof.widen = self.fast_eps, 1
        self._kc_for_k = {}
        self._gate = None          # (int8 rows, factors) the fast pass streams as its gate (build_gate)
        self._q8_versions = None   # version counters of rows / inv_norm / norm64 when the int8 rows were last quantized
        if self.n * self.ld * (esize - 1) >= self.GATE_MIN_SAVED_BYTES and self.build_gate() and not self._gate_pays():
            self.drop_gate()

    # ------------------------------------------------------------------ int8 gate ---------------
    # When the gate pays (DESIGN.md §4.5, tools/bench_gate.py on a B200 at 1000 W): its cost is the rows it fetches from the
    # catalog of record, ~2 ns each in aggregate (one L2/HBM round trip of one warp; 8k per request at 10M synthetic rows
    # once the seed kernel has set the bound, 87k without it); its gain is the bytes it does not stream, at ~7 TB/s.  A catalog that saves fewer bytes
    # than GATE_MIN_SAVED_BYTES cannot win; a larger one keeps its gate when a probe request fetches fewer rows than
    # saved bytes / GATE_BYTES_PER_FETCH (half the break-even), so catalogs whose rows crowd together (text embeddings with
    # a shared mean direction, where a quarter of the rows pass) keep the plain pass.
    GATE_MIN_SAVED_BYTES = 2 << 30
    GATE_BYTES_PER_FETCH = 56_000

    @property
    def gate_layout_ok(self) -> bool:
        """True when the gated fast pass takes this catalog's rows: more than 256 bytes per row in int8 and in the catalog's
        own dtype (32 lanes per row), and an int8 row length with a gated kernel (512 x 1, 2, 3, 4 or 6 bytes; mirrors
        gate_applies in csrc/gemv_topk.cu)."""
        ld8, _ = self.layout(max(self.n, 1), self.d, "i8")
        return self.d > 256 and ld8 % 512 == 0 and ld8 // 512 in (1, 2, 3, 4, 6)

    @property
    def has_gate(self) -> bool:
        return self._gate is not None

    def build_gate(self) -> bool:
        """Give the single-request fast pass an int8 gate of this shard (n x ld8 bytes + one fp32 factor per row): it then
        streams the int8 rows and reads a row of record only where its int8 score can still reach the candidate list.
        Results, margins and kc are those of the plain pass, bit for bit (DESIGN.md §4.5).  The constructor builds it when
        it pays (GATE_MIN_SAVED_BYTES, _gate_pays).  Returns False, leaving the plain pass, when the layout has no gated kernel
        or the memory is not there."""
        if self._gate is not None:
            return True
        if not self.gate_layout_ok:
            return False
        try:
            rows8, factor = self._int8_buffers()
        except torch.cuda.OutOfMemoryError:
            return False
        self._gate = (rows8, factor)
        self._c.gate_rows, self._c.gate_factor, self._c.gate_err = rows8.data_ptr(), factor.data_ptr(), self.q8_row_err
        return True

    def _gate_pays(self) -> bool:
        """One probe request through the gated pass: a profile-like query (the mean of 64 rows spread over the catalog) with
        k = 10; True when it fetched few enough rows (GATE_BYTES_PER_FETCH)."""
        lib = nat.load()
        with torch.cuda.device(self.device):
            idx = torch.linspace(0, self.n - 1, 64, device=self.device).long()
            q = self.rows[idx, :self.d].float().mean(0).cpu().numpy()
            kc = lib.rebert_candidates_for_k(10)
            s = self._scratch()
            s.ensure_out(10, kc)
            before = self.gate_fetches()
            excl_ptr, ne = self.stage_inputs(q, None, None, None, 10, kc)
            self.enqueue_fused(10, kc, excl_ptr, ne)
            fetched = (self.gate_fetches() - before) & 0xFFFFFFFF
        self.last_probe_fetches = fetched
        return fetched * self.GATE_BYTES_PER_FETCH < self.n * self.ld * (self.rows.element_size() - 1)

    def gate_fetches(self) -> int:
        """Rows the gated pass has read from the catalog of record on this thread's scratch (a wrapping 32-bit count;
        diagnostics: tools/bench_gate.py, tests)."""
        s = self._scratch()
        if not s.kc:
            return 0
        out = C.c_uint32(0)
        nat.check(nat.load().rebert_gate_fetches(s.ws.data_ptr(), s.ws.numel(), C.byref(out), torch.cuda.current_stream().cuda_stream))
        return out.value

    def drop_gate(self) -> None:
        """Back to the plain fast pass (the int8 rows stay allocated while the prefilter shadow uses them)."""
        self._gate = None
        self._c.gate_rows, self._c.gate_factor, self._c.gate_err = None, None, 0.0

    def _int8_buffers(self):
        """The int8 rows + factors of this shard: the gate's or the prefilter shadow's when one exists (one copy serves
        both), else newly quantized."""
        if self._gate is not None:
            return self._gate
        if self._c8 is not None:
            return self._q8_rows, self._q8_factor
        ld8, _ = self.layout(self.n, self.d, "i8")
        rows8 = torch.empty((max(self.n, 1), ld8), dtype=torch.int8, device=self.device)
        factor = torch.empty(_align(max(self.n, 1), 4), dtype=torch.float32, device=self.device)
        self._quantize_into(rows8, factor)
        return rows8, factor

    def _row_versions(self):
        return self.rows._version, self.inv_norm._version, self.norm64._version

    def _quantize_into(self, rows8: torch.Tensor, factor: torch.Tensor) -> None:
        lib = nat.load()
        with torch.cuda.device(self.device):
            max_err = torch.zeros(1, dtype=torch.float64, device=self.device)
            nat.check(lib.rebert_catalog_quantize_i8(C.byref(self._c), rows8.data_ptr(), rows8.shape[1], factor.data_ptr(),
                                                     max_err.data_ptr(), torch.cuda.current_stream().cuda_stream))
            self.q8_row_err = float(max_err.item())
        self._q8_versions = self._row_versions()

    def _fresh_int8(self) -> None:
        """Re-quantize the int8 rows (gate and prefilter shadow) if rows / inv_norm / norm64 were written since they were
        built: a stale gate could hide a row that now belongs to the result.  About 24 ms at 10M x 1536."""
        if self._q8_versions is None or self._q8_versions == self._row_versions():
            return
        if self._gate is None and self._c8 is None:     # both given up: nothing left to refresh
            self._q8_versions = None
            return
        rows8, factor = self._gate if self._gate is not None else (self._q8_rows, self._q8_factor)
        self._quantize_into(rows8, factor)
        if self._gate is not None:
            self._c.gate_err = self.q8_row_err
        if self._c8 is not None:
            self.q8_eps = self._shadow_eps(self.q8_row_err)

    # ------------------------------------------------------------------ construction -----------
    @staticmethod
    def _require_cuda(device) -> torch.device:
        if not torch.cuda.is_available():
            raise RuntimeError("robot_ebert_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        dev = torch.device(device if device is not None else "cuda:0")
        lib = nat.load()
        with torch.cuda.device(dev):
            nat.check(lib.rebert_check_device())
        return dev

    @staticmethod
    def layout(n: int, d: int, dtype: str) -> Tuple[int, int]:
        lib = nat.load()
        ld, nbytes = C.c_int32(0), C.c_size_t(0)
        nat.check(lib.rebert_catalog_layout(n, d, nat.DTYPES[dtype], C.byref(ld), C.byref(nbytes)))
        return ld.value, nbytes.value

    @classmethod
    def _alloc(cls, n: int, d: int, dtype: str, dev: torch.device):
        ld, _ = cls.layout(n, d, dtype)
        tdt = torch.bfloat16 if dtype == "bf16" else torch.float32
        rows = torch.empty((max(n, 1), ld), dtype=tdt, device=dev)
        inv_norm = torch.empty(_align(max(n, 1), 4), dtype=torch.float32, device=dev)
        norm64 = torch.empty(max(n, 1), dtype=torch.float64, device=dev)
        return ld, rows, inv_norm, norm64

    @classmethod
    def from_host(cls, ids: Optional[Sequence[str]], matrix: np.ndarray, dtype: str = "fp32", device=None,
                  row_base: int = 0, chunk_rows: int = 1 << 18, sort_ids: bool = True) -> "CatalogStore":
        """Upload an [N, D] host matrix (what Chroma's collection.get returns, constants.py:55) and build the store."""
        dev = cls._require_cuda(device)
        lib = nat.load()
        ids, matrix = validated_table(ids, matrix, sort_ids)
        n, d = matrix.shape
        ld, rows, inv_norm, norm64 = cls._alloc(n, d, dtype, dev)
        with torch.cuda.device(dev):
            st = torch.cuda.current_stream().cuda_stream
            esize = rows.element_size()
            for s in range(0, n, chunk_rows):
                e = min(n, s + chunk_rows)
                src = torch.from_numpy(np.ascontiguousarray(matrix[s:e])).to(dev)
                nat.check(lib.rebert_catalog_store_rows(src.data_ptr(), e - s, d, nat.DTYPES[dtype],
                                                        rows.data_ptr() + s * ld * esize, ld, st))
                torch.cuda.current_stream().synchronize()
            if n:
                nat.check(lib.rebert_catalog_norms(rows.data_ptr(), n, ld, nat.DTYPES[dtype], inv_norm.data_ptr(),
                                                   norm64.data_ptr(), st))
            torch.cuda.current_stream().synchronize()
        return cls(rows, inv_norm, norm64, n, d, ld, dtype, row_base, ids)

    @classmethod
    def synthetic(cls, seed: int, n: int, d: int, dtype: str = "bf16", scale_rows: bool = False, device=None,
                  row0: int = 0, row_base: Optional[int] = None) -> "CatalogStore":
        """Rows [row0, row0+n) of the counter-based synthetic catalog (robot_ebert_b200/synth.py), generated in HBM."""
        dev = cls._require_cuda(device)
        lib = nat.load()
        ld, rows, inv_norm, norm64 = cls._alloc(n, d, dtype, dev)
        with torch.cuda.device(dev):
            st = torch.cuda.current_stream().cuda_stream
            nat.check(lib.rebert_synth_rows(seed, row0, n, d, int(scale_rows), nat.DTYPES[dtype], rows.data_ptr(), ld, st))
            nat.check(lib.rebert_catalog_norms(rows.data_ptr(), n, ld, nat.DTYPES[dtype], inv_norm.data_ptr(),
                                               norm64.data_ptr(), st))
            torch.cuda.current_stream().synchronize()
        return cls(rows, inv_norm, norm64, n, d, ld, dtype, row0 if row_base is None else row_base, None)

    def enable_prefilter(self) -> float:
        """Build the int8 PREFILTER SHADOW of this shard (n x ld8 bytes + one fp32 factor per row): the single-request fast
        pass then streams 1 byte per element instead of 2 (bf16) or 4 (fp32), keeps 256 candidates, and the exact pass
        re-scores them from the catalog of record as always.  Returns the proven bound on |shadow score - true score|:
        max_r ||x_r - dequant(q8_r)|| / ||x_r|| (Cauchy-Schwarz, any unit query) plus the worst-case error of the two
        int8 query planes.  A request whose proof margin does not clear that bound silently takes the standard path, so
        results never depend on the shadow.  The streaming kernel has no int8 variant for rows of 5 or 7-11 chunks per lane
        (d = 2049-2560 and 3073-5632, d = 4096 among them): there single requests always take the standard path, and the
        shadow serves only the batched int8 GEMM.  With a gate (build_gate) the shadow is the gate's int8 rows."""
        self._fresh_int8()
        rows8, factor = self._int8_buffers()
        self._q8_rows, self._q8_factor = rows8, factor
        self._c8 = nat.Catalog(rows=rows8.data_ptr(), inv_norm=factor.data_ptr(), norm64=self.norm64.data_ptr(), n=self.n,
                               row_base=self.row_base, d=self.d, ld=rows8.shape[1], dtype=nat.DTYPES["i8"], reserved=0)
        self.q8_eps = self._shadow_eps(self.q8_row_err)
        return self.q8_eps

    def _shadow_eps(self, row_err: float) -> float:
        # query planes: |q - (dh*hi + dl*lo)| <= dl/2 per element with dl = max|q| / (127*254) <= 1 / (127*254) for ||q|| <= 1
        query_err = float(np.sqrt(self.d)) / (127.0 * 254.0 * 2.0)
        return row_err + 1.01 * (1.0 + row_err) * query_err + 4e-6      # + fp32 rounding of factor / int->float / final products

    def set_metadata(self, genre_bits: np.ndarray, year: np.ndarray) -> None:
        """Per-row side columns for the genre/year predicate (local row order)."""
        self.genre_bits = torch.from_numpy(np.ascontiguousarray(genre_bits, dtype=np.uint32).view(np.int32)).to(self.device)
        self.year = torch.from_numpy(np.ascontiguousarray(year, dtype=np.uint16).view(np.int16)).to(self.device)

    # ------------------------------------------------------------------ id map ------------------
    def row_of(self, tmdb_id: str) -> Optional[int]:
        if self._row_of is None:
            if self.ids is None:
                raise ValueError("catalog has no id table")
            self._row_of = {i: r + self.row_base for r, i in enumerate(self.ids)}
        return self._row_of.get(tmdb_id)

    def id_of(self, row: int) -> str:
        return self.ids[row - self.row_base] if self.ids is not None else str(row)

    # ------------------------------------------------------------------ scoring -----------------
    def _scratch(self) -> _Scratch:
        s = getattr(self._tls, "s", None)
        if s is None:
            s = self._tls.s = _Scratch(self)
        return s

    def recommend(self, *, query: Optional[np.ndarray] = None, liked_rows: Optional[np.ndarray] = None,
                  weights: Optional[np.ndarray] = None, exclude_rows: Optional[np.ndarray] = None, k: int = 10,
                  row_filter: Optional[RowFilter] = None, return_info: bool = False, prefilter: Optional[bool] = None):
        """Top-k rows by cosine to `query`, or by mean cosine to `liked_rows` (lib.py:51-55).

        query        fp32 [D] host vector (not normalised), OR
        liked_rows   global row ids of the liked movies (+ optional weights; default 1 = the reference)
        exclude_rows global row ids that must not be returned (the user's rated movies, lib.py:48)
        Returns (rows int64[k'], scores float64[k']), k' = min(k, #allowed rows), ordered (score desc, row asc).
        Host buffers in, host buffers out: one C call (rebert_recommend_host) packs the request into pinned memory, the
        kernels read it from there and write the result back there.
        prefilter: None = use the int8 shadow when enable_prefilter() has built one and k <= PREFILTER_MAX_K; True = try it
        for any k <= 240; False = never.  The result is the same either way.
        The ids are PROVEN exact or the call raises: a request no candidate list can prove (mass ties) takes the exhaustive
        sweep, then the threshold-bisection route; if even that cannot decide, RuntimeError.
        """
        if (query is None) == (liked_rows is None):
            raise ValueError("pass exactly one of query / liked_rows")
        if k <= 0:
            raise ValueError("k must be positive")
        lib = nat.load()
        kc = self._kc_for_k.get(k)
        if kc is None:
            kc = self._kc_for_k[k] = lib.rebert_candidates_for_k(k)
        if kc == 0:
            # k beyond the register-list kernel (k > 240): threshold bisection + sweep, still exact (rare, slower path)
            rows, scores = self._recommend_large_k(query, liked_rows, weights, exclude_rows, k, row_filter)
            if return_info:
                return rows, scores, {"kc": 0, "margin": float("inf"), "proven_exact": True, "exact_sweep": True}
            return rows, scores
        if prefilter and self._c8 is None:
            raise ValueError("prefilter=True needs enable_prefilter()")
        rows, scores, info = self._recommend_host(query, liked_rows, weights, exclude_rows, k, kc, row_filter,
                                                  self.shadow_max_k(self._c8 is not None, prefilter))
        if not info["proven_exact"]:
            # fail closed: the margin proved nothing, so the exhaustive routes answer (close_proof) or the call raises
            with torch.cuda.device(self.device):
                excl_ptr, ne = self.stage_inputs(query, liked_rows, weights, exclude_rows, k, kc)   # the sweeps read qn32 / qn64
                rows, scores = close_proof(rows, scores, k, self.fast_eps, info["margin"], *self._sweeps(excl_ptr, ne, row_filter))
            info = dict(info, proven_exact=True, exact_sweep=True)
        if return_info:
            return rows, scores, info
        return rows, scores

    # 256 candidates absorb the shadow's proven error bound (~0.009 for gaussian rows) only while the k-th and the 256-th
    # best scores are far enough apart; beyond k ~ 16 the proof usually fails and the attempt would be wasted work.
    PREFILTER_MAX_K = 16

    @classmethod
    def shadow_max_k(cls, has_shadow: bool, prefilter: Optional[bool]) -> int:
        """Largest k for which a single request tries the int8 shadow first (0 = never); see recommend()'s `prefilter`."""
        if not has_shadow or prefilter is False:
            return 0
        return 240 if prefilter else cls.PREFILTER_MAX_K

    SWEEP_CAP = 1 << 16

    def _recommend_large_k(self, query, liked_rows, weights, exclude_rows, k, row_filter):
        """k > 240: see large_k_search — count-only sweeps for the bisection, then collect + fp64 re-score."""
        self._check_large_k(k)
        with torch.cuda.device(self.device):
            excl_ptr, ne = self.stage_inputs(query, liked_rows, weights, exclude_rows, 1, 32)
            return self.topk_prepared_large_k(k, excl_ptr, ne, row_filter)

    @classmethod
    def _check_large_k(cls, k: int):
        if k > cls.SWEEP_CAP // 2:
            raise ValueError(f"k={k} is too large (limit {cls.SWEEP_CAP // 2})")

    def topk_prepared_large_k(self, k: int, excl_ptr=None, n_excl: int = 0, row_filter: Optional[RowFilter] = None):
        """Exact top-k for k > 240 (up to SWEEP_CAP / 2) for the query / profile already in this thread's scratch (qn32, qn64):
        large_k_search over count_above / sweep_above.  About 10-20 count-only passes over the catalog plus a sweep per
        call, so the batched path sends only the queries its own passes could not prove."""
        self._check_large_k(k)
        return large_k_search(*self._sweeps(excl_ptr, n_excl, row_filter), k, self.fast_eps)

    def _sweeps(self, excl_ptr, n_excl: int, row_filter: Optional[RowFilter]):
        """(count, sweep) of large_k_search / close_proof over this shard, for the request staged in this thread's scratch."""
        return (lambda thr: self.count_above(thr, excl_ptr, n_excl, row_filter),
                lambda thr: self.sweep_above(thr, excl_ptr, n_excl, row_filter))

    def count_above(self, threshold: float, excl_ptr=None, n_excl: int = 0, row_filter: Optional[RowFilter] = None) -> int:
        """Number of allowed rows of this shard whose fast score >= threshold (count-only sweep; query / profile from this
        thread's scratch)."""
        lib = nat.load()
        s = self._scratch()
        f = self._filter_struct(row_filter) or nat.Filter()
        if n_excl:
            f.exclude_rows, f.n_exclude = excl_ptr, n_excl
        dummy = torch.empty(1, dtype=torch.int32, device=self.device)
        cnt_t = torch.zeros(1, dtype=torch.int32, device=self.device)
        nat.check(lib.rebert_collect_above(C.byref(self._c), s.qn32.data_ptr(), C.byref(f), C.c_float(threshold), dummy.data_ptr(), 1,
                                           cnt_t.data_ptr(), torch.cuda.current_stream().cuda_stream))
        return int(cnt_t.item())

    def sweep_above(self, threshold: float, excl_ptr=None, n_excl: int = 0, row_filter: Optional[RowFilter] = None):
        """(global rows int64, exact fp64 scores) of every allowed row of this shard whose fast score >= threshold, for
        the query / profile in this thread's scratch; None if more than SWEEP_CAP rows qualify."""
        lib = nat.load()
        s = self._scratch()
        stream = torch.cuda.current_stream()
        f = self._filter_struct(row_filter) or nat.Filter()
        if n_excl:
            f.exclude_rows, f.n_exclude = excl_ptr, n_excl
        out_rows = torch.empty(self.SWEEP_CAP, dtype=torch.int32, device=self.device)
        out_count = torch.zeros(1, dtype=torch.int32, device=self.device)
        nat.check(lib.rebert_collect_above(C.byref(self._c), s.qn32.data_ptr(), C.byref(f), C.c_float(threshold), out_rows.data_ptr(),
                                           self.SWEEP_CAP, out_count.data_ptr(), stream.cuda_stream))
        cnt = int(out_count.item())
        if cnt > self.SWEEP_CAP:
            return None
        if cnt == 0:
            return np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.float64)
        sub = out_rows[:cnt].contiguous()
        exact = torch.empty((1, cnt), dtype=torch.float64, device=self.device)
        nat.check(lib.rebert_score_subset(C.byref(self._c), s.qn64.data_ptr(), 1, sub.data_ptr(), cnt, exact.data_ptr(),
                                          stream.cuda_stream))
        return sub.cpu().numpy().astype(np.int64), exact[0].cpu().numpy()

    def _recommend_host(self, query, liked_rows, weights, exclude_rows, k, kc, row_filter, shadow_max_k=0, exchange=None,
                        shadow_eps=None, scratch=None):
        """One rebert_recommend_host call: host buffers in, host buffers out; staging, kernels, proof loop and stream sync
        inside.  exchange: a nat.Exchange for one rank of a row-sharded catalog (sharding.py); scratch: an explicit _Scratch
        instead of the calling thread's own (the sharding layer pre-allocates one per exchange channel).
        Returns (rows, scores, info)."""
        lib = nat.load()
        self._fresh_int8()
        d = self.d
        q = lk = w = ex = None
        nl = ne = 0
        if query is not None:
            q = np.ascontiguousarray(query, dtype=np.float32)
            if q.shape != (d,):
                raise ValueError(f"query must have shape ({d},)")
        else:
            lk = np.ascontiguousarray(liked_rows, dtype=np.int32)
            nl = int(lk.shape[0])
            if weights is not None:
                w = np.ascontiguousarray(weights, dtype=np.float32)
                if w.shape != lk.shape:
                    raise ValueError("weights must match liked_rows")
        if exclude_rows is not None and len(exclude_rows):
            ex = np.ascontiguousarray(exclude_rows, dtype=np.int32).reshape(-1)     # the C entry sorts / de-duplicates its copy
            ne = int(ex.shape[0])
        f = None if row_filter is None else self._filter_struct(row_filter)
        if shadow_max_k and self._c8 is not None:
            proof = nat.Proof()
            proof.fast_eps, proof.widen = self.fast_eps, 1
            proof.shadow = C.pointer(self._c8)
            proof.shadow_eps = self.q8_eps if shadow_eps is None else shadow_eps
            proof.shadow_max_k = shadow_max_k
        else:
            proof = self._plain_proof
        # bytes the kernels fetch from / write to the pinned block over PCIe (zero-copy: no copy-engine operation)
        self.last_h2d_bytes = (4 * d if lk is None else 4 * nl * (2 if w is not None else 1)) + 4 * ne
        self.last_d2h_bytes = 8 * (2 * k + 2)
        with _on_device(self.device):                 # a serving thread's current device is 0 until it says otherwise
            s = scratch if scratch is not None else self._scratch()
            s.ensure_host(nl, ne, k)
            info = s.info
            info.attempts = 0                         # an argument error returns before the C entry writes it
            fast = nat.fast_recommend_host()
            if fast is not None:
                # same C entry point, called through the CPython module instead of ctypes (csrc/pycall.c)
                rc, n = fast(self._c_addr, q, lk, w, ex, 0 if f is None else C.addressof(f), k, kc, s.nl_cap, s.ne_cap, *s.host_args,
                             C.addressof(proof), 0 if exchange is None else C.addressof(exchange), *s.out_args, s.info_addr,
                             _raw_stream(self._dev_index))
            else:
                cnt = C.c_int32(0)
                rc = lib.rebert_recommend_host(
                    C.byref(self._c), None if q is None else q.ctypes.data, None if lk is None else lk.ctypes.data,
                    None if w is None else w.ctypes.data, nl, None if ex is None else ex.ctypes.data, ne,
                    None if f is None else C.byref(f), k, kc, s.nl_cap, s.ne_cap, *s.host_args,
                    C.byref(proof), None if exchange is None else C.byref(exchange), *s.out_args, C.byref(cnt), C.byref(info),
                    _raw_stream(self._dev_index))
                n = cnt.value
        s.last_attempts = int(info.attempts)         # exchange sequence numbers consumed, also when the call failed (per thread)
        nat.check(rc)
        return s.h_rows[:n].copy(), s.h_scores[:n].copy(), {
            "kc": info.kc, "margin": info.margin, "proven_exact": bool(info.proven), "exact_sweep": False,
            "prefilter": bool(info.used_shadow), "attempts": info.attempts,
            "host_us": {"pack": info.host_pack_us, "enqueue": info.host_enqueue_us, "wait": info.host_wait_us,
                        "unpack": info.host_unpack_us}}

    def _filter_struct(self, row_filter: Optional[RowFilter]):
        """rebert_filter_t for the device-resident predicates of a RowFilter (None when there are none)."""
        if row_filter is None:
            return None
        f = nat.Filter()
        if row_filter.exclude_bitmap is not None:
            f.exclude_bitmap = row_filter.exclude_bitmap.data_ptr()
        if row_filter.genre_any:
            if self.genre_bits is None:
                raise ValueError("row_filter.genre_any needs set_metadata()")
            f.genre_bits, f.genre_any = self.genre_bits.data_ptr(), row_filter.genre_any
        if (row_filter.year_lo, row_filter.year_hi) != (0, 65535):
            if self.year is None:
                raise ValueError("row_filter year range needs set_metadata()")
            f.year, f.year_lo, f.year_hi = self.year.data_ptr(), row_filter.year_lo, row_filter.year_hi
        return f

    def _query_filter_struct(self, query_filters: Optional[QueryFilters]):
        """rebert_query_filter_t for the tests some user of the batch actually has (None when no user has one: the kernels
        then run exactly as without query filters)."""
        if query_filters is None or not (query_filters.has_genre or query_filters.has_year):
            return None
        genre_any, year_lo, year_hi = query_filters.device_arrays(self.device)
        f = nat.QueryFilter()
        if query_filters.has_genre:
            f.genre_bits, f.genre_any = self.genre_bits.data_ptr(), genre_any.data_ptr()
        if query_filters.has_year:
            f.year, f.year_lo, f.year_hi = self.year.data_ptr(), year_lo.data_ptr(), year_hi.data_ptr()
        return f

    def stage_inputs(self, query, liked_rows, weights, exclude_rows, k, kc, profile_partial_only: bool = False):
        """Pack the request into one pinned buffer, issue ONE H2D copy, and enqueue query normalisation or the
        profile build on the current stream.  Returns (device pointer of the exclusion list, its length)."""
        lib = nat.load()
        s = self._scratch()
        d, ld = self.d, self.ld
        excl = None
        if exclude_rows is not None and len(exclude_rows):
            excl = np.unique(np.asarray(exclude_rows, dtype=np.int32))
        ne = 0 if excl is None else int(excl.shape[0])
        nl = 0
        if liked_rows is not None:
            liked = np.asarray(liked_rows, dtype=np.int32)
            nl = int(liked.shape[0])
            if nl == 0:
                raise ValueError(EMPTY_PROFILE)
        off_rp = _align(4 * d)
        off_e = off_rp + 16
        off_c = off_e + _align(4 * ne)
        off_w = off_c + _align(4 * nl)
        total = off_w + _align(4 * nl)
        s.ensure_in(total)
        s.ensure_out(k, kc)
        h = s.h_in_np
        if query is not None:
            q = np.asarray(query, dtype=np.float32)
            if q.shape != (d,):
                raise ValueError(f"query must have shape ({d},)")
            h[0:4 * d].view(np.float32)[:] = q
        else:
            h[off_rp:off_rp + 16].view(np.int64)[:] = (0, nl)
            h[off_c:off_c + 4 * nl].view(np.int32)[:] = liked
            if weights is not None:
                h[off_w:off_w + 4 * nl].view(np.float32)[:] = np.asarray(weights, dtype=np.float32)
        if ne:
            h[off_e:off_e + 4 * ne].view(np.int32)[:] = excl
        self.last_h2d_bytes = total
        st = torch.cuda.current_stream().cuda_stream
        s.d_in[:total].copy_(s.h_in[:total], non_blocking=True)
        base = s.d_in.data_ptr()
        if query is not None:
            nat.check(lib.rebert_query_normalize(base, 1, d, ld, s.qn32.data_ptr(), s.qn64.data_ptr(), None, st))
        else:
            nat.check(lib.rebert_profile_accumulate(C.byref(self._c), base + off_rp, base + off_c,
                                                    (base + off_w) if weights is not None else None, 1,
                                                    s.sum64.data_ptr(), s.wsum.data_ptr(), st))
            if not profile_partial_only:
                self.finalize_profile()
        return (base + off_e) if ne else None, ne

    def finalize_profile(self):
        """scratch.sum64 / scratch.wsum -> scratch.qn32 / qn64 (the mean of unit rows, lib.py:52)."""
        lib = nat.load()
        s = self._scratch()
        nat.check(lib.rebert_profile_finalize(s.sum64.data_ptr(), s.wsum.data_ptr(), 1, self.ld, s.qn32.data_ptr(),
                                              s.qn64.data_ptr(), None, torch.cuda.current_stream().cuda_stream))

    def enqueue_topk(self, k: int, kc: int, excl_ptr=None, n_excl: int = 0, row_filter: Optional[RowFilter] = None,
                     prefilter: bool = False):
        """Device-resident step: fused score+mask+top-k over the shard, then the exact fp64 pass, for the query /
        profile already sitting in this thread's scratch (qn32, qn64).  Result lands packed in scratch.d_out.
        Nothing is copied and nothing synchronises."""
        lib = nat.load()
        self._fresh_int8()
        s = self._scratch()
        s.ensure_out(k, kc)
        st = torch.cuda.current_stream().cuda_stream
        f = self._filter_struct(row_filter) or nat.Filter()
        if n_excl:
            f.exclude_rows, f.n_exclude = excl_ptr, n_excl
        # prefilter: the fast pass streams the int8 shadow (kc must be 256); the exact pass below always reads the real rows
        nat.check(lib.rebert_gemv_topk(C.byref(self._c8 if prefilter else self._c), s.qn32.data_ptr(), C.byref(f), kc, s.ws.data_ptr(),
                                       s.ws.numel(), s.cand.data_ptr(), st))
        ob = s.d_out.data_ptr()
        nat.check(lib.rebert_finalize_topk(C.byref(self._c), s.qn64.data_ptr(), s.cand.data_ptr(), kc, k, ob,
                                           ob + 8 * k, ob + 16 * k, ob + 16 * k + 8, st))
        return s.d_out

    def enqueue_fused(self, k: int, kc: int, excl_ptr=None, n_excl: int = 0, row_filter: Optional[RowFilter] = None,
                      prefilter: bool = False, exchange=None, err_ptr=None, out_ptr=None):
        """Device-resident request in ONE launch (rebert_recommend_device): fused score+mask+top-k, fp64 exact pass and
        ranking in the tail of the same kernel (+ the NVLink exchange and merge when `exchange` is given), for the query /
        profile already sitting in this thread's scratch.  Result lands packed in scratch.d_out (or at out_ptr)."""
        lib = nat.load()
        self._fresh_int8()
        s = self._scratch()
        s.ensure_out(k, kc)
        f = self._filter_struct(row_filter) or nat.Filter()
        if n_excl:
            f.exclude_rows, f.n_exclude = excl_ptr, n_excl
        nat.check(lib.rebert_recommend_device(C.byref(self._c), C.byref(self._c8) if prefilter else None, s.qn32.data_ptr(),
                                              s.qn64.data_ptr(), C.byref(f), k, kc, s.ws.data_ptr(), s.ws.numel(),
                                              s.d_out.data_ptr() if out_ptr is None else out_ptr, 0,
                                              None if exchange is None else C.byref(exchange), err_ptr,
                                              torch.cuda.current_stream().cuda_stream))
        return s.d_out

    def topk_prepared(self, k: int, excl_ptr=None, n_excl: int = 0, row_filter: Optional[RowFilter] = None):
        """PROVEN top-k for the query / profile already in this thread's scratch (qn32, qn64): the fused launch with
        4x more candidates until the margin clears the fp32 bound, then the exhaustive routes of close_proof; raises if
        none proves the ids.  Used for the queries a batched pass hands back."""
        lib = nat.load()
        s = self._scratch()
        kc = lib.rebert_candidates_for_k(k)
        if kc == 0:
            raise ValueError(f"k={k} is outside the supported range (1..240)")

        def attempt(kc):
            self.enqueue_fused(k, kc, excl_ptr, n_excl, row_filter)
            return unpack_result(s.d_out.cpu().numpy(), k)

        r, sc, margin, _ = widen_until_proven(attempt, kc, self.fast_eps)
        if not margin > self.fast_eps:
            r, sc = close_proof(r, sc, k, self.fast_eps, margin, *self._sweeps(excl_ptr, n_excl, row_filter))
        return r, sc

    # ------------------------------------------------------------------ batched (tensor cores) --
    def prepare_queries(self, queries: np.ndarray):
        """Host fp32 [b, d] query matrix -> device (qn32, qn64, qnbf16) unit vectors [b, ld]."""
        lib = nat.load()
        q = torch.from_numpy(np.ascontiguousarray(queries, dtype=np.float32)).to(self.device)
        b = q.shape[0]
        if q.shape[1] != self.d:
            raise ValueError(f"queries must be [b, {self.d}]")
        qn32 = torch.empty((b, self.ld), dtype=torch.float32, device=self.device)
        qn64 = torch.empty((b, self.ld), dtype=torch.float64, device=self.device)
        qbf = torch.empty((b, self.ld), dtype=torch.bfloat16, device=self.device)
        with torch.cuda.device(self.device):
            nat.check(lib.rebert_query_normalize(q.data_ptr(), b, self.d, self.ld, qn32.data_ptr(), qn64.data_ptr(),
                                                 qbf.data_ptr(), torch.cuda.current_stream().cuda_stream))
        return qn32, qn64, qbf

    def prepare_batch(self, queries, liked_ptr, liked_col, liked_w, reduce_fn=None):
        """Device (qn32, qn64, qnbf16) [b, ld] for a batch given as queries [b, d] OR a ragged CSR of liked rows (+ optional
        weights): prepare_queries or build_profiles (reduce_fn as there)."""
        if (queries is None) == (liked_ptr is None):
            raise ValueError("pass exactly one of queries / liked CSR")
        if queries is not None:
            return self.prepare_queries(queries)
        lp = np.asarray(liked_ptr, dtype=np.int64)
        if np.any(np.diff(lp) == 0):
            raise ValueError(EMPTY_PROFILE)
        return self.build_profiles(lp, liked_col, liked_w, reduce_fn)

    def gemm_scores(self, qbf16: torch.Tensor, row0: int, nrows: int) -> torch.Tensor:
        """fp32 scores [b, nrows] of rows [row0, row0+nrows) on the tensor cores (bf16 catalogs; multiples of 256)."""
        lib = nat.load()
        b = qbf16.shape[0]
        out = torch.empty((b, nrows), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            nat.check(lib.rebert_gemm_scores(C.byref(self._c), qbf16.data_ptr(), b, row0, nrows, out.data_ptr(),
                                             torch.cuda.current_stream().cuda_stream))
        return out

    def gemm_plan(self, b: int, k: int, shadow: bool = False) -> "nat.GemmPlan":
        lib = nat.load()
        plan = nat.GemmPlan()
        nat.check((lib.rebert_gemm_plan_i8 if shadow else lib.rebert_gemm_plan)(self.n, b, k, C.byref(plan)))
        return plan

    @property
    def batch_shadow_ok(self) -> bool:
        """True when the batched path can run on int8 operands: enable_prefilter() has built the shadow and its rows are
        whole 128-byte k-blocks (tcgen05 kind::i8, K = 32 per instruction, 128-byte swizzled tiles)."""
        return self._c8 is not None and self._c8.ld % 128 == 0

    @property
    def batch_gemm_ok(self) -> bool:
        """True when the batched path can run on bf16 operands: a bf16 catalog whose rows are whole 64-element (128-byte)
        k-blocks.  bf16 rows of d <= 32 are stored 16 or 32 elements wide, which the tcgen05 GEMM does not take."""
        return self.dtype == "bf16" and self.ld % 64 == 0

    def quantize_queries(self, qn32: torch.Tensor):
        """Unit queries / profiles [b, ld] fp32 -> (q8 int8 [b, ld8], qscale fp32 [b], qeps fp64 [b]) for the int8 batched path."""
        lib = nat.load()
        b, ld8 = qn32.shape[0], self._c8.ld
        q8 = torch.empty((b, ld8), dtype=torch.int8, device=self.device)
        qscale = torch.empty(b, dtype=torch.float32, device=self.device)
        qeps = torch.empty(b, dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            nat.check(lib.rebert_query_quantize_i8(qn32.data_ptr(), b, self.d, self.ld, ld8, C.c_double(self.q8_row_err), q8.data_ptr(),
                                                   qscale.data_ptr(), qeps.data_ptr(), torch.cuda.current_stream().cuda_stream))
        return q8, qscale, qeps

    def enqueue_batch(self, plan, qbf16, q64, excl_ptr, excl_col, ws, out_rows, out_scores, out_count, out_status,
                      row_filter: Optional[RowFilter] = None, shadow=None, query_filters: Optional[QueryFilters] = None):
        """Device-resident batched step (sample -> thresholds -> filtered GEMM -> select -> exact pass).
        shadow = (q8, qscale, qeps) from quantize_queries: the GEMMs run on int8 operands over the prefilter shadow (plan
        from gemm_plan(shadow=True)); the exact pass reads the catalog of record either way.
        query_filters: one genre / year test per query (QueryFilters), applied inside the threshold sample and the GEMM epilogue."""
        lib = nat.load()
        if shadow is not None:
            self._fresh_int8()
        if query_filters is not None:
            query_filters.validate(plan.b, row_filter, self.genre_bits, self.year)
        f = self._filter_struct(row_filter)
        qf = self._query_filter_struct(query_filters)
        fp, qfp = (None if f is None else C.byref(f)), (None if qf is None else C.byref(qf))
        st = torch.cuda.current_stream().cuda_stream
        if shadow is not None:
            q8, qscale, qeps = shadow
            nat.check(lib.rebert_gemm_topk_i8_filtered(C.byref(self._c), C.byref(self._c8), q8.data_ptr(), qscale.data_ptr(),
                                                       qeps.data_ptr(), q64.data_ptr(), _ptr(excl_ptr), _ptr(excl_col), fp, qfp,
                                                       C.byref(plan), ws.data_ptr(), ws.numel(), out_rows.data_ptr(), out_scores.data_ptr(),
                                                       out_count.data_ptr(), out_status.data_ptr(), st))
            return
        nat.check(lib.rebert_gemm_topk_filtered(C.byref(self._c), qbf16.data_ptr(), q64.data_ptr(), _ptr(excl_ptr), _ptr(excl_col), fp,
                                                qfp, C.byref(plan), ws.data_ptr(), ws.numel(), out_rows.data_ptr(), out_scores.data_ptr(),
                                                out_count.data_ptr(), out_status.data_ptr(), st))

    def recommend_batch(self, *, queries: Optional[np.ndarray] = None, liked_ptr: Optional[np.ndarray] = None,
                        liked_col: Optional[np.ndarray] = None, liked_w: Optional[np.ndarray] = None,
                        excl_ptr: Optional[np.ndarray] = None, excl_col: Optional[np.ndarray] = None, k: int = 10,
                        row_filter: Optional[RowFilter] = None, return_info: bool = False, prefilter: Optional[bool] = None,
                        query_filters: Optional[QueryFilters] = None):
        """Top-k for many users at once (lib.py:51-55 per user) on the tcgen05 path.
        row_filter: optional per-row predicate (genre / year / bitmap) shared by the whole batch.
        query_filters: optional genre / year test per user (QueryFilters), applied in the same tensor-core pass.  It may be
        combined with a shared exclude_bitmap, not with a shared genre or year test (ValueError).
        prefilter: None = int8 operands (twice the tensor rate) when enable_prefilter() has built a shadow the GEMM can use;
        True = require that; False = bf16 operands.  The result is the same either way.

        queries [b, d] fp32, OR a ragged CSR of liked rows (liked_ptr[b+1], liked_col, optional weights).
        excl_ptr/excl_col: per-user CSR of GLOBAL rows that must not be returned (sorted within a user).
        Returns rows int64 [b, k] (-1 padded), scores float64 [b, k], counts int32 [b].  Queries the batched pass could
        not prove exact (status != 0) are transparently re-run through the single-query kernel.
        """
        lib = nat.load()
        long_list = k > 0 and lib.rebert_candidates_for_k(k) == 0       # k > 240: beyond the single-query kernel
        if long_list:
            self._check_large_k(k)
        dev = self.device
        with torch.cuda.device(dev):
            qn32, qn64, qbf = self.prepare_batch(queries, liked_ptr, liked_col, liked_w)
            b = qbf.shape[0]
            if query_filters is not None:
                query_filters.validate(b, row_filter, self.genre_bits, self.year)
            if prefilter and not self.batch_shadow_ok:
                raise ValueError("prefilter=True needs enable_prefilter() and rows of whole 128-byte int8 k-blocks")
            use_shadow = self.batch_shadow_ok and prefilter is not False
            plan = None
            if use_shadow or self.batch_gemm_ok:
                try:
                    plan = self.gemm_plan(b, k, shadow=use_shadow)
                except nat.NativeError as e:
                    if e.code != nat.ERR_UNSUPPORTED:
                        raise    # ERR_UNSUPPORTED: catalog too small for the sampled-threshold scheme, plan stays None
            if plan is None:        # too small, or neither operand type fits the GEMM: one fused GEMV per user instead
                return self._recommend_batch_loop(qn32, qn64, excl_ptr, excl_col, k, return_info, row_filter, query_filters)
            ep = ec = None
            if excl_ptr is not None:
                excl_ptr, excl_col = sorted_csr(excl_ptr, excl_col)
                if len(excl_ptr) != b + 1:
                    raise ValueError("exclusion CSR must have one segment per query")
                ep = torch.from_numpy(excl_ptr).to(dev)
                ec = torch.from_numpy(excl_col).to(dev)
            rows, scores, counts, status = self._run_batch(plan, qbf, qn64, qn32, ep, ec, row_filter, use_shadow, query_filters)
            redo = np.nonzero(status)[0]
            if len(redo) and long_list:
                redo = self._widened_retry(redo, k, use_shadow, qbf, qn64, qn32, excl_ptr, excl_col, row_filter, rows, scores, counts,
                                           query_filters)
            # proven single-query route for the ones the batch could not prove
            self._rerun_prepared(redo, qn32, qn64, excl_ptr, ec, k, row_filter, rows, scores, counts, query_filters)
        if return_info:
            return rows, scores, counts, {"status": status, "plan": {f: getattr(plan, f) for f, _ in plan._fields_}, "int8_operands": use_shadow,
                                          "per_query": len(redo)}
        return rows, scores, counts

    # Largest k of the tensor-core path (rebert_gemm_plan); also the cap of the widened retry of long lists.
    BATCH_MAX_K = 2048

    def _run_batch(self, plan, qbf, qn64, qn32, ep, ec, row_filter, use_shadow, query_filters=None):
        """One batched pass with freshly allocated workspace and outputs; returns host (rows, scores, counts, status)."""
        lib = nat.load()
        dev = self.device
        b, k = plan.b, plan.k
        ws = torch.empty(lib.rebert_gemm_workspace_bytes(C.byref(self._c), C.byref(plan)), dtype=torch.uint8, device=dev)
        out_rows = torch.empty((b, k), dtype=torch.int64, device=dev)
        out_scores = torch.empty((b, k), dtype=torch.float64, device=dev)
        out_count = torch.empty(b, dtype=torch.int32, device=dev)
        out_status = torch.empty(b, dtype=torch.int32, device=dev)
        self.enqueue_batch(plan, qbf, qn64, ep, ec, ws, out_rows, out_scores, out_count, out_status, row_filter,
                           shadow=self.quantize_queries(qn32) if use_shadow else None, query_filters=query_filters)
        return out_rows.cpu().numpy(), out_scores.cpu().numpy(), out_count.cpu().numpy(), out_status.cpu().numpy()

    def _widened_retry(self, redo, k, use_shadow, qbf, qn64, qn32, excl_ptr, excl_col, row_filter, rows, scores, counts,
                       query_filters=None):
        """Long lists: the queries the batched pass could not prove run once more, as a sub-batch at k' = min(2k, 2048) with
        its longer candidate list, and keep the first k results (a proven top-k' starts with the proven top-k).  Much cheaper
        than the per-query route when it works.  Fills rows / scores / counts in place; returns the queries still unproven."""
        k2 = min(2 * k, self.BATCH_MAX_K)
        if k2 <= k:
            return redo
        try:
            plan = self.gemm_plan(len(redo), k2, shadow=use_shadow)
        except nat.NativeError as e:
            if e.code != nat.ERR_UNSUPPORTED:
                raise
            return redo                          # catalog too small for the plan at k'
        dev = self.device
        idx = torch.from_numpy(redo).to(dev)
        ep = ec = None
        if excl_ptr is not None:                 # excl_ptr / excl_col: the sorted CSR of the whole batch
            segs = [np.asarray(excl_col[excl_ptr[u]:excl_ptr[u + 1]], dtype=np.int32) for u in redo]
            sub_ptr = np.zeros(len(redo) + 1, dtype=np.int64)
            np.cumsum([len(x) for x in segs], out=sub_ptr[1:])
            ep = torch.from_numpy(sub_ptr).to(dev)
            ec = torch.from_numpy(np.concatenate(segs) if sub_ptr[-1] else np.zeros(1, dtype=np.int32)).to(dev)
        r2, s2, c2, st2 = self._run_batch(plan, qbf[idx].contiguous(), qn64[idx].contiguous(), qn32[idx].contiguous(), ep, ec,
                                          row_filter, use_shadow, None if query_filters is None else query_filters.subset(redo))
        ok = st2 == 0
        for i in np.nonzero(ok)[0]:
            u = redo[i]
            rows[u], scores[u], counts[u] = r2[i, :k], s2[i, :k], min(int(c2[i]), k)
        return redo[~ok]

    def _recommend_batch_loop(self, qn32, qn64, excl_ptr, excl_col, k, return_info, row_filter=None, query_filters=None):
        """Small catalogs, catalogs neither GEMM operand type takes, and k > 2048: the batch is served one prepared query at
        a time, by the single-query kernel for k <= 240 and by topk_prepared_large_k above."""
        b = qn32.shape[0]
        rows = np.full((b, k), -1, dtype=np.int64)
        scores = np.full((b, k), -np.inf, dtype=np.float64)
        counts = np.zeros(b, dtype=np.int32)
        ecp = ec = None
        if excl_ptr is not None:
            ecp, ecol = sorted_csr(excl_ptr, excl_col)
            ec = torch.from_numpy(ecol).to(self.device)
        self._rerun_prepared(range(b), qn32, qn64, ecp, ec, k, row_filter, rows, scores, counts, query_filters)
        if return_info:
            return rows, scores, counts, {"status": np.zeros(b, dtype=np.int32), "plan": None, "per_query": b}
        return rows, scores, counts

    def _rerun_prepared(self, users, qn32, qn64, excl_ptr, excl_col_dev, k, row_filter, rows, scores, counts, query_filters=None):
        """Proven single-query route for `users` of a prepared batch (qn32 / qn64 [b, ld]): topk_prepared, or
        topk_prepared_large_k for k > 240, over the user's segment of the sorted exclusion CSR (host excl_ptr, device
        excl_col_dev) and the user's own filter (user_row_filter).  Overwrites those users' rows / scores / counts."""
        large = nat.load().rebert_candidates_for_k(k) == 0
        s = self._scratch()
        for u in users:
            s.qn32.copy_(qn32[u])
            s.qn64.copy_(qn64[u])
            ptr, ne = None, 0
            if excl_ptr is not None and excl_ptr[u + 1] > excl_ptr[u]:
                ptr, ne = excl_col_dev.data_ptr() + 4 * int(excl_ptr[u]), int(excl_ptr[u + 1] - excl_ptr[u])
            r, sc = (self.topk_prepared_large_k if large else self.topk_prepared)(k, ptr, ne, user_row_filter(query_filters, u, row_filter))
            rows[u, :], scores[u, :] = -1, -np.inf
            rows[u, :len(r)], scores[u, :len(r)], counts[u] = r, sc, len(r)

    # ------------------------------------------------------------------ diagnostics -------------
    def scores_dense(self, q32: torch.Tensor) -> torch.Tensor:
        """Materialised fp32 score rows for b pre-normalised queries [b, ld] (test / diagnostics only)."""
        lib = nat.load()
        b = q32.shape[0]
        out = torch.empty((b, self.n), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            nat.check(lib.rebert_scores_dense(C.byref(self._c), q32.data_ptr(), b, out.data_ptr(),
                                              torch.cuda.current_stream().cuda_stream))
        return out

    def score_subset(self, p64: torch.Tensor, sub_rows: np.ndarray) -> np.ndarray:
        """fp64 scores of `sub_rows` (global ids) against b prepared profiles [b, ld] (lib.py:105-106)."""
        lib = nat.load()
        sub = torch.from_numpy(np.asarray(sub_rows, dtype=np.int32)).to(self.device)
        b, m = p64.shape[0], sub.shape[0]
        out = torch.empty((b, m), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            nat.check(lib.rebert_score_subset(C.byref(self._c), p64.data_ptr(), b, sub.data_ptr(), m, out.data_ptr(),
                                              torch.cuda.current_stream().cuda_stream))
        return out.cpu().numpy()

    def build_profiles(self, row_ptr: np.ndarray, col: np.ndarray, w: Optional[np.ndarray] = None, reduce_fn=None):
        """Batched profile build from a ragged CSR of liked rows: returns (p32, p64, pbf16) device tensors [b, ld].

        On a row shard only the local liked rows contribute; `reduce_fn(sum64)` (an in-place all-reduce) completes the
        fp64 partial sums before they are divided by the weight sums."""
        lib = nat.load()
        dev = self.device
        rp = torch.from_numpy(np.asarray(row_ptr, dtype=np.int64)).to(dev)
        cl = torch.from_numpy(np.asarray(col, dtype=np.int32)).to(dev)
        wt = None if w is None else torch.from_numpy(np.asarray(w, dtype=np.float32)).to(dev)
        b = rp.shape[0] - 1
        sum64 = torch.empty((b, self.ld), dtype=torch.float64, device=dev)
        wsum = torch.empty(b, dtype=torch.float64, device=dev)
        p32 = torch.empty((b, self.ld), dtype=torch.float32, device=dev)
        p64 = torch.empty((b, self.ld), dtype=torch.float64, device=dev)
        pbf = torch.empty((b, self.ld), dtype=torch.bfloat16, device=dev)
        with torch.cuda.device(dev):
            st = torch.cuda.current_stream().cuda_stream
            nat.check(lib.rebert_profile_accumulate(C.byref(self._c), rp.data_ptr(), cl.data_ptr(), _ptr(wt), b,
                                                    sum64.data_ptr(), wsum.data_ptr(), st))
            if reduce_fn is not None:
                reduce_fn(sum64)
            nat.check(lib.rebert_profile_finalize(sum64.data_ptr(), wsum.data_ptr(), b, self.ld, p32.data_ptr(),
                                                  p64.data_ptr(), pbf.data_ptr(), st))
        return p32, p64, pbf
