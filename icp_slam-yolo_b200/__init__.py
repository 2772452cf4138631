"""icp_slam-yolo_b200: B200-native (sm_100a) 2D ICP scan matching.

Drop-in for the registration path of DucVuUET04/ICP_SLAM-YOLO
(labels_segmentation/icp.py:5-53 fed by duc/ICP_LIDAR/process.py:9-52).  Hand-written CUDA
behind a C ABI (include/b200icp.h); PyTorch only carries device memory and streams.
"""
from ._cabi import B200IcpError, lib, library_path          # noqa: F401
from .icp import (IcpOutput, best_fit_transform, icp, icp_full, nearest_neighbors,   # noqa: F401
                  registration_p2p)
from .registration import (AlignResult, ScanTable, align_pairs, alloc_outputs,   # noqa: F401
                           best_fit, ffma_probe, nn_search, polar_to_cartesian)
from .odometry import align_consecutive, chain_poses         # noqa: F401
from .gicp import estimate_covariances, gicp_consecutive, gicp_pairs, registration_gicp   # noqa: F401
from .sharding import shard_range, triangle_pair, triangle_pair_count   # noqa: F401
from .scan_to_map import MapShard, ScanToMap, ScanToMapResult, scan_to_map_icp   # noqa: F401
from .mapping import crop_local_map, remove_dynamic_points, voxel_down_sample   # noqa: F401
from .occupancy import OccupancyGrid                           # noqa: F401
from .slam import OfflineSlam, SlamConfig                      # noqa: F401
from . import hostmem, map_io, scan_io                         # noqa: F401

__all__ = [
    "B200IcpError", "lib", "library_path", "IcpOutput", "icp", "icp_full", "nearest_neighbors",
    "registration_p2p", "best_fit_transform", "best_fit", "AlignResult", "ScanTable", "align_pairs", "alloc_outputs", "ffma_probe",
    "nn_search", "polar_to_cartesian", "align_consecutive", "chain_poses", "shard_range",
    "triangle_pair", "triangle_pair_count", "scan_io", "MapShard", "ScanToMap", "ScanToMapResult",
    "scan_to_map_icp", "crop_local_map", "remove_dynamic_points", "voxel_down_sample",
    "OccupancyGrid", "map_io", "hostmem", "OfflineSlam", "SlamConfig",
    "estimate_covariances", "gicp_pairs", "gicp_consecutive", "registration_gicp",
]
