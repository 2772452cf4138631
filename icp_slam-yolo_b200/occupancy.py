"""Occupancy-grid mapping on the device: the step that follows registration in the reference's
SLAM loop (duc/ICP_LIDAR/process.py:86-249; called at mainn.py:322-351,749 and
slam_offline.py:341,400-428).

``OccupancyGrid`` owns what the reference keeps in two places -- the probabilities in the
function attribute ``update_occupancy_map.occupancy_probs`` (process.py:122-125) and the
``(h, w, 3) uint8`` picture passed as ``occupancy_map`` -- as CUDA tensors; ``update`` is
``update_occupancy_map``, ``filter_points`` is ``filter_new_points_by_occupancy`` /
``prune_global_map``.  All arithmetic runs in ``libb200icp.so`` (csrc/occupancy.cu) and is
bit-identical to the reference under NumPy 2 scalar rules; there is no CPU fallback.
"""
from __future__ import annotations

from typing import Optional, Sequence

import numpy as np
import torch

from . import _cabi
from .registration import _DTYPES, _compact_scratch, _ptr, _require_cuda, _stream_ptr

THRESHOLD_UP = 0.65              # process.py:158


def _f32(v: float) -> float:
    """The float32 value NumPy 2 uses for a Python float next to an ``np.float32``."""
    return float(np.float32(v))


class OccupancyGrid:
    """``n_maps`` independent grids of ``h x w`` cells on one GPU.

    probs : [n_maps, h, w] float32, 0.5 everywhere at creation (process.py:123)
    image : [n_maps, h, w, 3] uint8, 128 everywhere at creation (slam_offline.py:319)
    """

    def __init__(self, h: int, w: int, map_center_px: Sequence[float], resolution: float, *,
                 n_maps: int = 1, device="cuda", with_image: bool = True):
        _cabi.lib()                                   # fail loudly when the CUDA library is missing
        self.h, self.w, self.n_maps = int(h), int(w), int(n_maps)
        self.center = (float(map_center_px[0]), float(map_center_px[1]))
        self.resolution = float(resolution)
        dev = torch.device(device)
        if dev.type != "cuda":
            raise _cabi.B200IcpError("OccupancyGrid lives on a CUDA device: this path has no CPU fallback")
        self.probs = torch.full((self.n_maps, self.h, self.w), 0.5, dtype=torch.float32, device=dev)
        self.image = (torch.full((self.n_maps, self.h, self.w, 3), 128, dtype=torch.uint8, device=dev)
                      if with_image else None)

    # ---- update_occupancy_map (process.py:114-177) -------------------------------------------
    def _grid(self, p_occ_inc, p_free_dec, area) -> _cabi.OccGrid:
        g = _cabi.OccGrid()
        g.probs = self.probs.data_ptr()
        g.image = 0 if self.image is None else self.image.data_ptr()
        g.h, g.w = self.h, self.w
        g.center_x, g.center_y = self.center
        g.resolution = self.resolution
        g.area = int(area)
        g.p_occ_inc, g.p_free_dec, g.threshold_up = _f32(p_occ_inc), _f32(p_free_dec), _f32(THRESHOLD_UP)
        return g

    def update_frames(self, points: torch.Tensor, lengths: Optional[torch.Tensor], robot_xy: torch.Tensor,
                      p_occ_inc: float = 0.2, p_free_dec: float = 0.9, area: int = 140, stream=None) -> None:
        """Apply frames in order to every map in one launch.

        points   [n_maps, n_frames, pitch, 2] float32/float64 CUDA, map-frame coordinates
        lengths  [n_maps, n_frames] int32 CUDA or None (all rows full)
        robot_xy [n_maps, n_frames, 2] float64 CUDA (``global_pose[:2, 3]`` per frame)
        """
        if points.dim() != 4 or points.shape[0] != self.n_maps or points.shape[3] != 2 or points.dtype not in _DTYPES:
            raise ValueError("points must be [n_maps, n_frames, pitch, 2] float32/float64")
        n_frames, pitch = int(points.shape[1]), int(points.shape[2])
        if robot_xy.dtype != torch.float64 or tuple(robot_xy.shape) != (self.n_maps, n_frames, 2):
            raise ValueError("robot_xy must be [n_maps, n_frames, 2] float64")
        _require_cuda(points, "points")
        _require_cuda(robot_xy, "robot_xy")
        if lengths is not None:
            if lengths.dtype != torch.int32 or tuple(lengths.shape) != (self.n_maps, n_frames):
                raise ValueError("lengths must be [n_maps, n_frames] int32")
            _require_cuda(lengths, "lengths")
        g = self._grid(p_occ_inc, p_free_dec, area)
        with torch.cuda.device(self.probs.device):
            rc = _cabi.lib().b200icp_occ_update(g, self.n_maps, _ptr(points), _DTYPES[points.dtype], _ptr(lengths),
                                                _ptr(robot_xy), n_frames, pitch, _stream_ptr(stream))
        _cabi.check(rc, "b200icp_occ_update")

    def update(self, points_global, robot_pos, p_occ_inc: float = 0.2, p_free_dec: float = 0.9,
               area: int = 140, map_index: int = 0) -> None:
        """``update_occupancy_map(occupancy_map, points_global, robot_pos, map_center_px,
        resolution, p_occ_inc, p_free_dec, area)`` for one frame of map ``map_index``.
        ``points_global``: (N, 2) or (N, 3) NumPy array or CUDA tensor; ``robot_pos``: (>=2,)."""
        if len(points_global) == 0:                                   # process.py:116-117
            return
        dev = self.probs.device
        if isinstance(points_global, torch.Tensor):
            pts = points_global[:, :2].to(device=dev).contiguous()
            if pts.dtype not in _DTYPES:
                pts = pts.to(torch.float64)
        else:
            pts = torch.from_numpy(np.ascontiguousarray(np.asarray(points_global, dtype=np.float64)[:, :2])).to(dev)
        rob = torch.tensor([[[float(robot_pos[0]), float(robot_pos[1])]]], dtype=torch.float64, device=dev)
        one = OccupancyGrid.__new__(OccupancyGrid)                    # view of one map, same memory
        one.__dict__.update(self.__dict__)
        one.n_maps = 1
        one.probs = self.probs[map_index:map_index + 1]
        one.image = None if self.image is None else self.image[map_index:map_index + 1]
        one.update_frames(pts[None, None], None, rob, p_occ_inc, p_free_dec, area)

    # ---- filter_new_points_by_occupancy / prune_global_map (process.py:203-249) ----------------
    def filter_points(self, points, free_threshold: float = 0.2, map_index: int = 0, stream=None):
        """Rows of ``points`` ((N, 2) or (N, 3)) that do not fall into a cell with probability
        below ``free_threshold``; rows outside the grid are kept.  Order preserved.  NumPy in ->
        NumPy out, CUDA tensor in -> CUDA tensor out."""
        if len(points) == 0:                                          # process.py:207-208
            return points
        dev = self.probs.device
        as_numpy = not isinstance(points, torch.Tensor)
        pts = torch.from_numpy(np.ascontiguousarray(points)).to(dev) if as_numpy else points
        if pts.dtype not in _DTYPES:
            pts = pts.to(torch.float64)
        if pts.dim() != 2 or pts.shape[1] < 2:
            raise ValueError("points must be [n, >= 2]")
        _require_cuda(pts, "points")
        n, cols = int(pts.shape[0]), int(pts.shape[1])
        kept = torch.empty(n, dtype=torch.int64, device=dev)
        count = torch.zeros(1, dtype=torch.int64, device=dev)
        with torch.cuda.device(dev):
            rc = _cabi.lib().b200icp_occ_filter_points(
                _ptr(pts), _DTYPES[pts.dtype], cols, n, _ptr(self.probs[map_index]), self.h, self.w,
                self.center[0], self.center[1], self.resolution, _f32(free_threshold), _ptr(kept),
                _ptr(count), _ptr(_compact_scratch(n, dev)), _stream_ptr(stream))
        _cabi.check(rc, "b200icp_occ_filter_points")
        idx = kept[: int(count.item())]
        return points[idx.cpu().numpy()] if as_numpy else points[idx]

    # ---- host copies -------------------------------------------------------------------------
    def probs_numpy(self, map_index: int = 0) -> np.ndarray:
        return self.probs[map_index].cpu().numpy()

    def image_numpy(self, map_index: int = 0) -> np.ndarray:
        if self.image is None:
            raise ValueError("grid was created with with_image=False")
        return self.image[map_index].cpu().numpy()
