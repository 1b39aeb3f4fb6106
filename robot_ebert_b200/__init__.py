"""robot_ebert_b200 — B200-native recommendation scoring path for robot-ebert (see DESIGN.md).

Only the scoring hot path lives here: catalog store, profile build, fused cosine + mask + top-k kernels,
the row-sharding layer, and a host-side mirror of the reference's lib.get_user_recs / run_search.
"""
from .catalog import CatalogStore, QueryFilters, RowFilter  # noqa: F401

__all__ = ["CatalogStore", "QueryFilters", "RowFilter"]
