"""Mirror of `shot_fpfh.matching`: the names pipeline.py imports (pipeline.py:24-30, matching/__init__.py:1-19)."""

from .filters import FilterFunction, left_median_filter, quantile_filter, threshold_filter
from .matching import basic_matching, double_matching_with_rejects, match_descriptors
from .ransac import ransac_on_matches, ransac_on_matches_adaptive

__all__ = [
    "FilterFunction",
    "threshold_filter",
    "quantile_filter",
    "left_median_filter",
    "match_descriptors",
    "basic_matching",
    "double_matching_with_rejects",
    "ransac_on_matches",
    "ransac_on_matches_adaptive",
]
