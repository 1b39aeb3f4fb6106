"""ctypes binding of include/rebert_b200.h.  No fallback: if the library is missing this raises."""
from __future__ import annotations

import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
# REBERT_DEBUG=1 loads the assertion-carrying twin (build.py --debug): device-side bounds checks at every computed index
LIB_PATH = os.path.join(_PKG, "librebert_b200_debug.so" if os.environ.get("REBERT_DEBUG") == "1" else "librebert_b200.so")

F32, BF16 = 0, 1
I8 = 2          # prefilter shadow only (rebert_catalog_quantize_i8)
DTYPES = {"fp32": F32, "bf16": BF16, "i8": I8}

ABI_VERSION = 5
OK, ERR_INVALID, ERR_UNSUPPORTED, ERR_WORKSPACE, ERR_CUDA, ERR_DEVICE = 0, -1, -2, -3, -4, -5


class NativeError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"rebert_b200 error {code}: {msg}")
        self.code = code


class Catalog(C.Structure):
    _fields_ = [("rows", C.c_void_p), ("inv_norm", C.c_void_p), ("norm64", C.c_void_p), ("n", C.c_int64),
                ("row_base", C.c_int64), ("d", C.c_int32), ("ld", C.c_int32), ("dtype", C.c_int32),
                ("reserved", C.c_int32), ("gate_rows", C.c_void_p), ("gate_factor", C.c_void_p), ("gate_err", C.c_double)]


class Filter(C.Structure):
    _fields_ = [("exclude_bitmap", C.c_void_p), ("exclude_rows", C.c_void_p), ("n_exclude", C.c_int32),
                ("genre_any", C.c_uint32), ("genre_bits", C.c_void_p), ("year", C.c_void_p),
                ("year_lo", C.c_uint16), ("year_hi", C.c_uint16), ("reserved", C.c_uint32)]


class QueryFilter(C.Structure):
    """rebert_query_filter_t: per-query genre / year tests of a batch (catalog columns [n] + per-query arrays [b])."""
    _fields_ = [("genre_bits", C.c_void_p), ("year", C.c_void_p), ("genre_any", C.c_void_p), ("year_lo", C.c_void_p),
                ("year_hi", C.c_void_p)]


class Exchange(C.Structure):
    """rebert_exchange_t: one rank's view of the peer-mapped exchange buffers of a row-sharded catalog."""
    _fields_ = [("peer_buffers", C.c_void_p), ("world", C.c_int32), ("rank", C.c_int32), ("k_max", C.c_int32),
                ("prof_len", C.c_int32), ("channels", C.c_int32), ("channel", C.c_int32), ("seq", C.c_uint32),
                ("reserved", C.c_uint32)]


class Proof(C.Structure):
    """rebert_proof_t: which fast passes rebert_recommend_host may try and their proven error bounds."""
    _fields_ = [("shadow", C.POINTER(Catalog)), ("shadow_eps", C.c_double), ("fast_eps", C.c_double),
                ("shadow_max_k", C.c_int32), ("widen", C.c_int32)]


class RequestInfo(C.Structure):
    _fields_ = [("kc", C.c_int32), ("attempts", C.c_int32), ("proven", C.c_int32), ("used_shadow", C.c_int32),
                ("margin", C.c_double), ("host_pack_us", C.c_double), ("host_enqueue_us", C.c_double),
                ("host_wait_us", C.c_double), ("host_unpack_us", C.c_double)]


class GemmPlan(C.Structure):
    _fields_ = [("b", C.c_int32), ("k", C.c_int32), ("kc", C.c_int32), ("sample_rows", C.c_int32),
                ("sample_rank", C.c_int32), ("cand_cap", C.c_int32)]


_P = C.c_void_p
_SIGS = {
    "rebert_abi_version": (C.c_int, []),
    "rebert_last_error": (C.c_char_p, []),
    "rebert_check_device": (C.c_int, []),
    "rebert_catalog_layout": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_size_t)]),
    "rebert_catalog_store_rows": (C.c_int, [_P, C.c_int64, C.c_int32, C.c_int32, _P, C.c_int32, _P]),
    "rebert_catalog_quantize_i8": (C.c_int, [C.POINTER(Catalog), _P, C.c_int32, _P, _P, _P]),
    "rebert_catalog_norms": (C.c_int, [_P, C.c_int64, C.c_int32, C.c_int32, _P, _P, _P]),
    "rebert_query_normalize": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    "rebert_profile_accumulate": (C.c_int, [C.POINTER(Catalog), _P, _P, _P, C.c_int32, _P, _P, _P]),
    "rebert_profile_finalize": (C.c_int, [_P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    "rebert_candidates_for_k": (C.c_int32, [C.c_int32]),
    "rebert_gemv_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int32]),
    "rebert_gemv_topk": (C.c_int, [C.POINTER(Catalog), _P, C.POINTER(Filter), C.c_int32, _P, C.c_size_t, _P, _P]),
    "rebert_finalize_topk": (C.c_int, [C.POINTER(Catalog), _P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P]),
    "rebert_recommend_host_scratch": (C.c_int, [C.POINTER(Catalog), C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "rebert_recommend_host": (C.c_int, [C.POINTER(Catalog), _P, _P, _P, C.c_int32, _P, C.c_int32, C.POINTER(Filter), C.c_int32, C.c_int32,
                                        C.c_int32, C.c_int32, _P, C.c_size_t, _P, C.c_size_t, C.POINTER(Proof), C.POINTER(Exchange),
                                        _P, _P, _P, C.POINTER(RequestInfo), _P]),
    "rebert_recommend_device": (C.c_int, [C.POINTER(Catalog), C.POINTER(Catalog), _P, _P, C.POINTER(Filter), C.c_int32, C.c_int32, _P,
                                          C.c_size_t, _P, C.c_uint32, C.POINTER(Exchange), _P, _P]),
    "rebert_workspace_reset": (C.c_int, [_P, C.c_size_t, _P]),
    "rebert_gate_fetches": (C.c_int, [_P, C.c_size_t, C.POINTER(C.c_uint32), _P]),
    "rebert_merge_topk": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    "rebert_exchange_buffer_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    "rebert_exchange_merge": (C.c_int, [C.POINTER(Exchange), C.c_int32, _P, _P, _P, _P]),
    "rebert_profile_exchange": (C.c_int, [C.POINTER(Exchange), C.c_int32, _P, _P, _P, _P, _P, _P]),
    "rebert_score_subset": (C.c_int, [C.POINTER(Catalog), _P, C.c_int32, _P, C.c_int32, _P, _P]),
    "rebert_collect_above": (C.c_int, [C.POINTER(Catalog), _P, C.POINTER(Filter), C.c_float, _P, C.c_int32, _P, _P]),
    "rebert_scores_dense": (C.c_int, [C.POINTER(Catalog), _P, C.c_int32, _P, _P]),
    "rebert_gemm_plan": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, C.POINTER(GemmPlan)]),
    "rebert_gemm_workspace_bytes": (C.c_size_t, [C.POINTER(Catalog), C.POINTER(GemmPlan)]),
    "rebert_gemm_topk": (C.c_int, [C.POINTER(Catalog), _P, _P, _P, _P, C.POINTER(Filter), C.POINTER(GemmPlan), _P, C.c_size_t, _P, _P, _P, _P, _P]),
    "rebert_gemm_scores": (C.c_int, [C.POINTER(Catalog), _P, C.c_int32, C.c_int64, C.c_int64, _P, _P]),
    "rebert_gemm_plan_i8": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, C.POINTER(GemmPlan)]),
    "rebert_query_quantize_i8": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_double, _P, _P, _P, _P]),
    "rebert_gemm_topk_i8": (C.c_int, [C.POINTER(Catalog), C.POINTER(Catalog), _P, _P, _P, _P, _P, _P, C.POINTER(Filter), C.POINTER(GemmPlan),
                                      _P, C.c_size_t, _P, _P, _P, _P, _P]),
    "rebert_gemm_topk_filtered": (C.c_int, [C.POINTER(Catalog), _P, _P, _P, _P, C.POINTER(Filter), C.POINTER(QueryFilter),
                                            C.POINTER(GemmPlan), _P, C.c_size_t, _P, _P, _P, _P, _P]),
    "rebert_gemm_topk_i8_filtered": (C.c_int, [C.POINTER(Catalog), C.POINTER(Catalog), _P, _P, _P, _P, _P, _P, C.POINTER(Filter),
                                               C.POINTER(QueryFilter), C.POINTER(GemmPlan), _P, C.c_size_t, _P, _P, _P, _P, _P]),
    "rebert_gemm_scores_i8": (C.c_int, [C.POINTER(Catalog), _P, _P, C.c_int32, C.c_int64, C.c_int64, _P, _P]),
    "rebert_synth_rows": (C.c_int, [C.c_uint64, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32, _P, C.c_int32, _P]),
}

_lib = None


def load() -> C.CDLL:
    """Load librebert_b200.so (built in-tree by robot_ebert_b200/build.py).  Raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU or PyTorch fallback for the scoring path)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGS.items():
        fn = getattr(lib, name)          # AttributeError if the header and the library disagree
        fn.restype = res
        fn.argtypes = args
    if lib.rebert_abi_version() != ABI_VERSION:
        raise ImportError("rebert_b200 ABI version mismatch")
    _lib = lib
    return lib


_fast_call = False      # False = not looked up yet, None = unavailable


def fast_recommend_host():
    """robot_ebert_b200._pycall.recommend_host bound to the loaded library's rebert_recommend_host (csrc/pycall.c), or None
    when that optional module has not been built — the caller then makes the same call through ctypes.
    REBERT_PYCALL=0 forces the ctypes route."""
    global _fast_call
    if _fast_call is False:
        _fast_call = None
        if os.environ.get("REBERT_PYCALL", "1") != "0":
            try:
                from . import _pycall
                _pycall.set_entry(C.cast(load().rebert_recommend_host, C.c_void_p).value)
                _fast_call = _pycall.recommend_host
            except ImportError:
                pass
    return _fast_call


def exported_symbols():
    return list(_SIGS)


def check(rc: int) -> None:
    if rc != OK:
        msg = load().rebert_last_error().decode("utf-8", "replace")
        if rc == ERR_INVALID:
            raise ValueError(f"rebert_b200: {msg}")
        raise NativeError(rc, msg)
