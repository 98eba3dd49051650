"""Mirror of `shot_fpfh.descriptors` for the hot path: the names pipeline.py imports (pipeline.py:15) + compute_normals
(+ orient_normals, which the reference does not have)."""

from .fpfh import compute_fpfh_descriptor
from .pca_based_descriptors import compute_normals, orient_normals
from .shot_parallelization import ShotMultiprocessor

__all__ = ["compute_fpfh_descriptor", "compute_normals", "orient_normals", "ShotMultiprocessor"]
