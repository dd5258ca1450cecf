"""deepmerge_b200 -- B200-native (sm_100a) region-merging hot path of lvxianwei/DeepMerge.

Python host code over a C-ABI CUDA library (include/deepmerge_b200.h).  Importing the package
does not touch CUDA; the first kernel call loads libdeepmerge_b200.so and fails loudly if it
has not been built (`python -m deepmerge_b200.build`).  See DESIGN.md / INTEGRATION.md.
"""
from .raster import (RAG, MergeEngine, MergeResult, build_rag, compact_roots, csr_from_region_of_point,  # noqa: F401
                     merge_edge_lists, merge_graph, merge_scene, points_region, pool_bands, pool_dense, pool_points,
                     pool_points_csr, region_mean, relabel, score_l2, PackedMLP, score_mlp, mlp_forward, pool_boundary, ScenePipeline,
                     score_spectral, merge_scene_spectral)
from .polygons import Lines, Polygons, boundary_lines, polygonize, rasterize  # noqa: F401

__version__ = "0.1.0"
