"""CPU-only: per-user genre / year filters of a batch (QueryFilters) and the argument checks of the filtered batched entry
points, which must refuse half-specified predicates before any CUDA call."""
import ctypes as C

import numpy as np
import pytest

from robot_ebert_b200 import QueryFilters, RowFilter, _native as nat
from robot_ebert_b200.catalog import user_row_filter


def test_query_filters_hold_validated_unsigned_columns():
    qf = QueryFilters([0, 0b1011, 0xFFFFFFFF], [0, 1960, 2000], [65535, 2000, 1999])
    assert qf.genre_any.dtype == np.uint32 and qf.year_lo.dtype == np.uint16 and qf.year_hi.dtype == np.uint16
    assert len(qf) == 3 and qf.has_genre and qf.has_year
    only_genre = QueryFilters(np.array([1, 0], dtype=np.int64))            # years default to the whole range
    assert only_genre.has_genre and not only_genre.has_year
    assert only_genre.year_lo.tolist() == [0, 0] and only_genre.year_hi.tolist() == [65535, 65535]
    none = QueryFilters([0, 0], [0, 0], [65535, 65535])
    assert not none.has_genre and not none.has_year


@pytest.mark.parametrize("args,match", [
    (([0.5, 1.0],), "integers"),
    (([[1, 2]],), "1-D"),
    (([],), "non-empty"),
    (([-1],), "out of range"),
    (([1 << 32],), "out of range"),
    (([1], [0], [70000]), "out of range"),
    (([1], [-5], [10]), "out of range"),
    (([1, 2], [0], [10, 20]), "one entry per user"),
    (([1, 2], [0, 0], [10]), "one entry per user"),
])
def test_query_filters_refuse_bad_dtype_shape_and_range(args, match):
    with pytest.raises(ValueError, match=match):
        QueryFilters(*args)


def test_row_filter_of_one_user():
    qf = QueryFilters([0, 0b1011, 4], [0, 1960, 1990], [65535, 2000, 1989])
    r0 = qf.row_filter(0)
    assert isinstance(r0, RowFilter) and (r0.genre_any, r0.year_lo, r0.year_hi) == (0, 0, 65535) and not r0.has_genre_or_year
    r1 = qf.row_filter(1)
    assert (r1.genre_any, r1.year_lo, r1.year_hi) == (0b1011, 1960, 2000) and r1.exclude_bitmap is None
    bitmap = object()
    r2 = qf.row_filter(2, exclude_bitmap=bitmap)
    assert (r2.genre_any, r2.year_lo, r2.year_hi) == (4, 1990, 1989) and r2.exclude_bitmap is bitmap
    assert all(type(x) is int for x in (r2.genre_any, r2.year_lo, r2.year_hi))
    sub = qf.subset([2, 0])
    assert sub.genre_any.tolist() == [4, 0] and sub.year_lo.tolist() == [1990, 0] and sub.year_hi.tolist() == [1989, 65535]
    # the per-query route: the shared row_filter without query filters, else the user's own test plus the shared bitmap
    shared = RowFilter(exclude_bitmap=bitmap)
    assert user_row_filter(None, 1, shared) is shared
    u1 = user_row_filter(qf, 1, shared)
    assert (u1.genre_any, u1.year_lo, u1.year_hi) == (0b1011, 1960, 2000) and u1.exclude_bitmap is bitmap
    assert user_row_filter(qf, 1, None).exclude_bitmap is None


def test_validate_batch_size_shared_filter_and_metadata():
    cols = (object(), object())                                            # stand-ins for set_metadata's device columns
    qf = QueryFilters([1, 0], [0, 1990], [65535, 2000])
    qf.validate(2, None, *cols)
    qf.validate(2, RowFilter(exclude_bitmap=object()), *cols)              # a shared bitmap is fine
    qf.validate(2, RowFilter(), *cols)                                     # so is an empty shared filter
    with pytest.raises(ValueError, match="2 users, the batch 3"):
        qf.validate(3, None, *cols)
    with pytest.raises(ValueError, match="shared row_filter"):
        qf.validate(2, RowFilter(genre_any=1), *cols)
    with pytest.raises(ValueError, match="shared row_filter"):
        qf.validate(2, RowFilter(year_lo=1900), *cols)
    with pytest.raises(ValueError, match="genre_any needs set_metadata"):
        qf.validate(2, None, None, cols[1])
    with pytest.raises(ValueError, match="year range needs set_metadata"):
        qf.validate(2, None, cols[0], None)
    QueryFilters([1, 2]).validate(2, None, cols[0], None)                  # genre tests only: no year column needed
    QueryFilters([0, 0], [0, 1990], [65535, 2000]).validate(2, None, None, cols[1])
    QueryFilters([0], [0], [65535]).validate(1, None, None, None)          # nobody restricted: no metadata needed


def _fake_catalogs():
    """Descriptors that pass the catalog checks (aligned non-null pointers, whole k-blocks) without any device memory: the
    calls below must fail on the query filter before they touch CUDA."""
    cat = nat.Catalog(rows=128, inv_norm=128, norm64=128, n=100_000, row_base=0, d=64, ld=64, dtype=nat.BF16, reserved=0)
    shadow = nat.Catalog(rows=128, inv_norm=128, norm64=128, n=100_000, row_base=0, d=64, ld=128, dtype=nat.I8, reserved=0)
    return cat, shadow


@pytest.mark.parametrize("fields,match", [
    (dict(genre_any=256), b"per-query genre test"),                       # genre_any without the catalog's genre_bits
    (dict(genre_bits=256), b"per-query genre test"),                      # the column without the per-query array
    (dict(year_lo=256, year_hi=256), b"per-query year test"),             # bounds without the catalog's year
    (dict(year=256, year_lo=256), b"per-query year test"),                # year_hi missing
    (dict(year=256, year_hi=256), b"per-query year test"),                # year_lo missing
    (dict(genre_bits=256, genre_any=256, year_lo=256, year_hi=256), b"per-query year test"),
])
def test_filtered_entry_points_refuse_half_a_predicate_before_cuda(fields, match):
    lib = nat.load()
    cat, shadow = _fake_catalogs()
    qf = nat.QueryFilter(**fields)
    plan = nat.GemmPlan(b=4, k=10, kc=32, sample_rows=256, sample_rank=16, cand_cap=1024)
    rc = lib.rebert_gemm_topk_filtered(C.byref(cat), 128, 128, None, None, None, C.byref(qf), C.byref(plan), 128, 1 << 30,
                                       128, 128, 128, 128, None)
    assert rc == nat.ERR_INVALID and match in lib.rebert_last_error()
    rc = lib.rebert_gemm_topk_i8_filtered(C.byref(cat), C.byref(shadow), 128, 128, 128, 128, None, None, None, C.byref(qf),
                                          C.byref(plan), 128, 1 << 30, 128, 128, 128, 128, None)
    assert rc == nat.ERR_INVALID and match in lib.rebert_last_error()


def test_unfiltered_entry_points_keep_their_checks():
    """rebert_gemm_topk / _i8 are the filtered entry points with a NULL query filter: same argument checks."""
    lib = nat.load()
    cat, shadow = _fake_catalogs()
    plan = nat.GemmPlan(b=4, k=10, kc=32, sample_rows=256, sample_rank=16, cand_cap=1024)
    assert lib.rebert_gemm_topk(C.byref(cat), None, 128, None, None, None, C.byref(plan), 128, 1 << 30, 128, 128, 128, 128,
                                None) == nat.ERR_INVALID
    assert b"null argument" in lib.rebert_last_error()
    assert lib.rebert_gemm_topk_filtered(C.byref(cat), None, 128, None, None, None, None, C.byref(plan), 128, 1 << 30, 128, 128,
                                         128, 128, None) == nat.ERR_INVALID
    assert b"null argument" in lib.rebert_last_error()
    assert lib.rebert_gemm_topk_i8(C.byref(cat), C.byref(cat), 128, 128, 128, 128, None, None, None, C.byref(plan), 128, 1 << 30,
                                   128, 128, 128, 128, None) == nat.ERR_INVALID
    assert b"int8 prefilter shadow" in lib.rebert_last_error()
    empty = nat.QueryFilter()                                              # all pairs NULL: no test, nothing to refuse
    assert lib.rebert_gemm_topk_filtered(C.byref(cat), None, 128, None, None, None, C.byref(empty), C.byref(plan), 128, 1 << 30,
                                         128, 128, 128, 128, None) == nat.ERR_INVALID
    assert b"null argument" in lib.rebert_last_error()
