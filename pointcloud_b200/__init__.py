"""pointcloud_b200 -- the point-cloud reconstruction-loss hot path of JoongWonSeo/pointcloud
(Chamfer distance and auction EMD, forward + backward) re-built for NVIDIA B200 (sm_100a).

Python host layer (this package) mirrors the reference's loss interface
(pointcloud_vision/utils.py:207-309, pointcloud_vision/loss/emd/emd_module.py); all arithmetic runs in
hand-written CUDA kernels behind the C ABI of include/pcl.h (libpcl_b200.so).  No CPU fallback.
"""
from . import cfg
from .ball_query import ball_query, ball_query_forward_raw
from .chamfer import chamfer_distance, chamfer_forward_raw
from .emd_module import emdFunction, emdModule, emd_forward_raw, set_emd_path
from .knn import knn_forward_raw, knn_gather, knn_points
from .losses import (ChamferDistance, EarthMoverDistance, FilterClasses, FilteringChamferDistance,
                     SegmentingChamferDistance, chamfer_emd_loss)
from .normals import estimate_pointcloud_local_coord_frames, estimate_pointcloud_normals, frames_forward_raw
from .points_alignment import (ICPSolution, SimilarityTransform, corresponding_points_alignment, icp_forward_raw,
                               iterative_closest_point, points_alignment_forward_raw)
from .points_to_volumes import add_points_features_to_volume_densities_features, points_to_volumes_forward_raw
from .compositing import alpha_composite, composite_forward_raw, norm_weighted_sum, weighted_sum
from .rasterize_points import rasterize_points, rasterize_points_backward_raw, rasterize_points_forward_raw
from .sampling import farthest_point_sample, fps_forward_raw, query_ball_point, sample_farthest_points
from .sharded import ShardedChamferEmdStep, ShardedLoss, shard_bounds

__all__ = [
    "cfg", "chamfer_distance", "chamfer_forward_raw", "emdFunction", "emdModule", "emd_forward_raw", "set_emd_path",
    "ChamferDistance", "FilteringChamferDistance", "SegmentingChamferDistance", "EarthMoverDistance",
    "FilterClasses", "chamfer_emd_loss", "ShardedLoss", "ShardedChamferEmdStep", "shard_bounds",
    "farthest_point_sample", "sample_farthest_points", "fps_forward_raw", "query_ball_point", "knn_points", "knn_gather", "knn_forward_raw",
    "ball_query", "ball_query_forward_raw",
    "estimate_pointcloud_normals", "estimate_pointcloud_local_coord_frames", "frames_forward_raw",
    "corresponding_points_alignment", "iterative_closest_point", "SimilarityTransform", "ICPSolution", "icp_forward_raw",
    "points_alignment_forward_raw", "add_points_features_to_volume_densities_features", "points_to_volumes_forward_raw",
    "rasterize_points", "rasterize_points_forward_raw", "rasterize_points_backward_raw", "alpha_composite", "norm_weighted_sum",
    "weighted_sum", "composite_forward_raw",
]
