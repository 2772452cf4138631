"""The two point-selection steps that sit either side of registration in the reference's SLAM
loop, on the device: the local-map radius crop (duc/ICP_LIDAR/mainn.py:297-308) and dynamic-point
removal (duc/ICP_LIDAR/process.py:75-84).  Both keep the input order."""
from __future__ import annotations

from typing import Optional

import torch

from . import _cabi
from .registration import _DTYPES, ScanTable, _compact_scratch, _ptr, _require_cuda, _stream_ptr, _workspace, nn_search


def _select(points: torch.Tensor, mode: int, key: Optional[torch.Tensor], cx: float, cy: float,
            threshold: float, stream=None) -> torch.Tensor:
    if points.dim() != 2 or points.shape[1] != 2 or points.dtype not in _DTYPES:
        raise ValueError("points must be [n, 2] float32/float64")
    _require_cuda(points, "points")
    n = int(points.shape[0])
    out = torch.empty_like(points)
    count = torch.zeros(1, dtype=torch.int64, device=points.device)
    with torch.cuda.device(points.device):
        rc = _cabi.lib().b200icp_select_points(_ptr(points), _DTYPES[points.dtype], n, mode, _ptr(key),
                                               float(cx), float(cy), float(threshold), _ptr(out),
                                               _ptr(count), _ptr(_compact_scratch(n, points.device)), _stream_ptr(stream))
    _cabi.check(rc, "b200icp_select_points")
    return out[: int(count.item())]


def crop_local_map(map_points: torch.Tensor, center_xy, radius: float, min_points: int = 50) -> torch.Tensor:
    """Map points within ``radius`` of the robot position; the whole map if fewer than
    ``min_points`` survive (mainn.py:300-308)."""
    kept = _select(map_points, 1, None, float(center_xy[0]), float(center_xy[1]), float(radius) ** 2)
    return map_points if kept.shape[0] < min_points else kept


def remove_dynamic_points(current_points: torch.Tensor, prev_points: Optional[torch.Tensor],
                          distance_threshold: float = 250.0) -> torch.Tensor:
    """Keep the points of ``current_points`` whose nearest neighbour in ``prev_points`` is closer
    than ``distance_threshold`` (process.py:75-84; Open3D's compute_point_cloud_distance is the
    NN distance).  Empty / missing previous scan returns the input (process.py:76-77)."""
    if prev_points is None or prev_points.shape[0] == 0 or current_points.shape[0] == 0:
        return current_points
    lib = _cabi.lib()
    n, m = int(current_points.shape[0]), int(prev_points.shape[0])
    if n <= lib.b200icp_max_src_pitch() and m <= lib.b200icp_max_tgt_pitch():
        if prev_points.dtype != current_points.dtype:
            prev_points = prev_points.to(current_points.dtype)
        _, d2 = nn_search(ScanTable(current_points[None].contiguous()), ScanTable(prev_points[None].contiguous()), n_pairs=1)
        key = d2[0].contiguous()
    else:                       # large sets: one search of the sharded-map path
        from .scan_to_map import MapShard, ScanToMap
        s2m = ScanToMap(MapShard(prev_points.contiguous()), n, local_only=True)
        s2m.init(current_points.contiguous())
        s2m.search()
        key = s2m.records[:, 0].contiguous()
    return _select(current_points, 0, key, 0.0, 0.0, float(distance_threshold) ** 2)


def voxel_down_sample(points: torch.Tensor, voxel_size: float, stream=None) -> torch.Tensor:
    """One point per occupied 2D cell ``floor(p / voxel_size)`` (the mean of its points), cells
    ordered by (cell_y, cell_x): ``point_cloud.voxel_down_sample(voxel_size)`` as the reference
    applies it before registration (gicp_lidar.py:8-11,20-21) and in remove_duplicate_points
    (process.py:68-73)."""
    if points.dim() != 2 or points.shape[1] != 2 or points.dtype not in _DTYPES:
        raise ValueError("points must be [n, 2] float32/float64")
    _require_cuda(points, "points")
    n = int(points.shape[0])
    if n == 0:
        return points
    ws, wb = _workspace(_cabi.lib().b200icp_voxel_workspace_bytes, n, device=points.device)
    out = torch.empty_like(points)
    count = torch.zeros(1, dtype=torch.int64, device=points.device)
    with torch.cuda.device(points.device):
        rc = _cabi.lib().b200icp_voxel_downsample(_ptr(points), _DTYPES[points.dtype], n, float(voxel_size),
                                                  _ptr(out), _ptr(count), _ptr(ws), wb, _stream_ptr(stream))
    _cabi.check(rc, "b200icp_voxel_downsample")
    return out[: int(count.item())]
