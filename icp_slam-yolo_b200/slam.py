"""The reference's offline SLAM loop composed from the device primitives of this package.

Mirrors ``duc/ICP_LIDAR/slam_offline.py:318-455`` step by step -- same order, same thresholds
(``Config.py``), same early ``continue`` on a rejected registration -- with one substitution: the
registration call ``gicp(points, local_map, threshold, voxel, trans_init)`` (Open3D Generalized
ICP, slam_offline.py:108-144,382) is, by default, the point-to-point loop of
``labels_segmentation/icp.py:28-53`` behind the same call shape (``registration_p2p``);
``SlamConfig(registration="gicp")`` selects the 2D Generalized ICP of ``gicp.py`` instead.  Open3D is not vendored by the reference, so the
loop as a whole is parity-UNPINNED; every step in it is pinned on its own (DESIGN.md §2), and
``tests/test_slam_gpu.py`` replays it against the same composition of the CPU oracles.

Per frame the numeric work -- local-map crop, voxel down-sampling, ICP, dynamic-point removal,
occupancy filter, ray casting, map pruning -- runs in ``libb200icp.so``; the loop itself (frame
order, the 3 x 3 pose, list bookkeeping) is host glue exactly as in the reference.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import map_io
from .gicp import registration_gicp
from .icp import registration_p2p
from .mapping import crop_local_map, remove_dynamic_points, voxel_down_sample
from .occupancy import OccupancyGrid


@dataclass
class SlamConfig:
    """duc/ICP_LIDAR/Config.py:7-21."""
    resolution_mm_per_pixel: float = 30
    map_width_mm: float = 30000
    map_height_mm: float = 25000
    icp_voxel_size: float = 25.0
    icp_threshold: float = 180.0
    max_rmse_threshold: float = 50.0
    dynamic_distance_threshold: float = 300.0
    local_map_radius_mm: float = 9000.0
    min_icp_map_points: int = 50
    max_map_points_before_downsample: int = 1000        # slam_offline.py:409
    min_scan_points: int = 10                           # slam_offline.py:353
    max_iteration: int = 50                             # gicp_lidar.py:27 (ICPConvergenceCriteria)
    tolerance: float = 1e-5
    registration: str = "p2p"                           # "p2p" (registration_p2p) or "gicp" (registration_gicp)

    @property
    def map_width_pixels(self) -> int:
        return int(self.map_width_mm / self.resolution_mm_per_pixel)

    @property
    def map_height_pixels(self) -> int:
        return int(self.map_height_mm / self.resolution_mm_per_pixel)


@dataclass
class FrameResult:
    accepted: bool
    rmse: float
    pose: np.ndarray                 # (4, 4) global pose after the frame
    map_points: int


def transform_points(points: np.ndarray, rotation_matrix: np.ndarray, translation_vector: np.ndarray) -> np.ndarray:
    """slam_offline.py:105-107 (host glue, as in the reference)."""
    return np.dot(np.asarray(points), rotation_matrix.T) + translation_vector


@dataclass
class OfflineSlam:
    config: SlamConfig = field(default_factory=SlamConfig)
    device: str = "cuda"

    def __post_init__(self):
        c = self.config
        if c.registration not in ("p2p", "gicp"):
            raise ValueError(f"SlamConfig.registration must be 'p2p' or 'gicp', got {c.registration!r}")
        self.map_center_px = (c.map_width_pixels // 2, c.map_height_pixels // 2)          # :320
        self.grid = OccupancyGrid(c.map_height_pixels, c.map_width_pixels, self.map_center_px,
                                  c.resolution_mm_per_pixel, device=self.device)           # :319
        self.global_map = torch.zeros((0, 2), dtype=torch.float64, device=self.device)     # :322
        self.global_pose = np.eye(4)                                                        # :323
        self.prev_points_global: Optional[torch.Tensor] = None
        self.current_points_global = np.zeros((0, 3))
        self.pose_history: List[np.ndarray] = []
        self.mapped = False              # the reference's hasattr(update_occupancy_map, "occupancy_probs")

    def _cuda(self, pts: np.ndarray) -> torch.Tensor:
        return torch.from_numpy(np.ascontiguousarray(np.asarray(pts, dtype=np.float64)[:, :2])).to(self.device)

    def _update_occupancy(self):
        if len(self.current_points_global) == 0:
            return
        self.grid.update(self.current_points_global, self.global_pose[:3, 3])
        self.mapped = True

    # ---- slam_offline.py:333-342 -------------------------------------------------------------------
    def first_scan(self, points: np.ndarray) -> None:
        """``points``: (N, 3) Cartesian scan (``load_and_prepare_scan``)."""
        if points is None or len(points) == 0:
            raise ValueError("the first scan is empty")
        self.global_map = self._cuda(points)
        self.current_points_global = np.asarray(points, dtype=np.float64)
        self._update_occupancy()
        self.pose_history.append(self.global_pose[:3, 3][:2].copy())

    # ---- slam_offline.py:344-430 -------------------------------------------------------------------
    def step(self, points: Optional[np.ndarray]) -> Optional[FrameResult]:
        c = self.config
        if points is None or len(points) == 0 or len(points) < c.min_scan_points:          # :348-360
            return None
        current_points = np.asarray(points, dtype=np.float64)
        robot = self.global_pose[:3, 3]
        if self.global_map.shape[0] > 0:                                                   # :366-373
            map_for_icp = crop_local_map(self.global_map, robot[:2], c.local_map_radius_mm, c.min_icp_map_points)
        else:
            map_for_icp = self.global_map
        if c.registration == "gicp":                                                       # :382
            rmse, T = registration_gicp(current_points, map_for_icp, c.icp_threshold, c.icp_voxel_size,
                                        trans_init=self.global_pose, max_iteration=c.max_iteration)
        else:
            rmse, T = registration_p2p(current_points, map_for_icp, c.icp_threshold, c.icp_voxel_size,
                                       trans_init=self.global_pose, max_iteration=c.max_iteration,
                                       tolerance=c.tolerance)
        if rmse > c.max_rmse_threshold:                                                     # :386-387: `continue`
            return FrameResult(False, float(rmse), self.global_pose.copy(), int(self.global_map.shape[0]))
        self.global_pose = T                                                                # :390
        self.current_points_global = transform_points(current_points, T[:3, :3], T[:3, 3])  # :391
        cur = self._cuda(self.current_points_global)
        to_add = remove_dynamic_points(cur, self.prev_points_global, c.dynamic_distance_threshold)   # :394
        if self.mapped and to_add.shape[0] > 0:                                             # :399-405
            to_add = self.grid.filter_points(to_add)
        if to_add.shape[0] > 0:                                                             # :407-408
            self.global_map = torch.cat([self.global_map, to_add.contiguous()], dim=0)
        if self.global_map.shape[0] > c.max_map_points_before_downsample:                   # :409-410
            self.global_map = voxel_down_sample(self.global_map.contiguous(), c.icp_voxel_size)
        self.pose_history.append(self.global_pose[:3, 3][:2].copy())                        # :413-414
        self.prev_points_global = cur                                                       # :416
        self._update_occupancy()                                                            # :418
        if self.mapped and self.global_map.shape[0] > 0:                                    # :420-428
            self.global_map = self.grid.filter_points(self.global_map.contiguous())
        return FrameResult(True, float(rmse), self.global_pose.copy(), int(self.global_map.shape[0]))

    def run(self, scans: Sequence[np.ndarray]) -> List[Optional[FrameResult]]:
        """``scans``: Cartesian (N, 3) arrays in recording order; the first one seeds the map."""
        self.first_scan(scans[0])
        return [self.step(s) for s in scans[1:]]

    # ---- slam_offline.py:445-453 -------------------------------------------------------------------
    def save(self, pcd_path: str, png_path: str) -> None:
        final_map = self.global_map
        if final_map.shape[0] > 0:
            final_map = voxel_down_sample(final_map.contiguous(), self.config.icp_voxel_size)
        map_io.write_pcd(pcd_path, final_map.cpu().numpy())
        map_io.write_png(png_path, self.grid.image_numpy())
