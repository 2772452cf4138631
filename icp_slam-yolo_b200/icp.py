"""Drop-in mirror of the reference's ICP call surface, executed on the B200.

Same names, argument meaning and return shapes as
``labels_segmentation/icp.py`` (``icp`` :28-53, ``best_fit_transform`` :5-26) and the
Open3D-shaped wrapper ``gicp`` (duc/ICP_LIDAR/gicp_lidar.py:12-36), with NumPy arrays in
and out like the reference.  All arithmetic runs in the CUDA library through the C ABI;
nothing here computes on the host and nothing falls back to the CPU.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional, Tuple

import numpy as np
import torch

from . import _cabi
from .registration import ScanTable, _registration_4x4, _rmse_pose, align_pairs, best_fit, nn_search


@dataclass
class IcpOutput:
    R: np.ndarray            # (2,2) cumulative rotation,  src = R A + t
    t: np.ndarray            # (2,)
    error: float             # mean NN distance of the last search (lagged, icp.py:48)
    iterations: int
    R_last: np.ndarray       # last increment (what the reference's icp() returns)
    t_last: np.ndarray
    rmse: float
    fitness: float
    indices: np.ndarray      # (N,) correspondences of the last search
    src: np.ndarray          # (N,2) transformed source


def _as_points(a, name: str) -> np.ndarray:
    a = np.asarray(a, dtype=np.float64)
    if a.ndim != 2 or a.shape[1] < 2:
        raise ValueError(f"{name} must be an (N, 2) array, got shape {a.shape}")
    if a.shape[0] == 0:
        # the reference fails inside SciPy on empty input (SURVEY.md quirk Q5)
        raise ValueError(f"{name} is empty")
    return np.ascontiguousarray(a[:, :2])


def _pose6_host(init_pose) -> torch.Tensor:
    """(R, t) / 3x3 / 4x4 -> host tensor [6] = R00 R01 R10 R11 tx ty."""
    if isinstance(init_pose, (tuple, list)) and len(init_pose) == 2:
        R0, t0 = np.asarray(init_pose[0], dtype=np.float64), np.asarray(init_pose[1], dtype=np.float64)
    else:
        T = np.asarray(init_pose, dtype=np.float64)
        if T.shape == (4, 4):            # Open3D trans_init (gicp_lidar.py:12)
            R0, t0 = T[:2, :2], T[:2, 3]
        elif T.shape == (3, 3):
            R0, t0 = T[:2, :2], T[:2, 2]
        else:
            raise ValueError("init_pose must be (R, t), a 3x3 or a 4x4 homogeneous matrix")
    return torch.from_numpy(np.ascontiguousarray(np.concatenate([R0.reshape(4), t0.reshape(2)])))


def _pose6(init_pose) -> Optional[torch.Tensor]:
    if init_pose is None:
        return None
    return _pose6_host(init_pose)[None, :].cuda()


class _CallBuffers:
    """Pinned host + device staging for ONE alignment of an (n, m) problem: both point sets travel
    in one host-to-device copy and every output comes back in one device-to-host copy, so a call costs
    two copies, one launch and one synchronisation (the reference's call is synchronous too)."""

    def __init__(self, n: int, m: int, device):
        self.n, self.m = n, m
        n_idx = ((n + 1) // 2 + 1) // 2 * 2        # float64 slots that hold n int32 indices; even, so that
                                                   # the points behind them stay 16-byte aligned (double2 stores)
        self.h_in = torch.empty(2 * (n + m), dtype=torch.float64).pin_memory()
        self.d_in = torch.empty(2 * (n + m), dtype=torch.float64, device=device)
        self.h_pose = torch.zeros(6, dtype=torch.float64).pin_memory()
        self.d_pose = torch.empty((1, 6), dtype=torch.float64, device=device)
        size = 16 + n_idx + 2 * n
        self.h_out = torch.empty(size, dtype=torch.float64).pin_memory()
        self.d_out = torch.empty(size, dtype=torch.float64, device=device)
        d = self.d_out
        ints = d[14:15].view(torch.int32)
        from .registration import AlignResult
        self.out = AlignResult(
            pose_total=d[0:6].view(1, 6), pose_last=d[6:12].view(1, 6), error=d[12:13], rmse=d[13:14],
            inliers=ints[0:1], iterations=ints[1:2],
            indices=d[16:16 + n_idx].view(torch.int32)[:n].view(1, n),
            src_final=d[16 + n_idx:].view(1, n, 2))
        self.src = ScanTable(self.d_in[:2 * n].view(1, n, 2), None)
        self.tgt = ScanTable(self.d_in[2 * n:].view(1, m, 2), None)
        self.n_idx = n_idx


_buffers: "dict[tuple, _CallBuffers]" = {}


def _call_buffers(n: int, m: int) -> _CallBuffers:
    dev = torch.device("cuda", torch.cuda.current_device())
    key = (n, m, dev.index)
    buf = _buffers.get(key)
    if buf is None:
        if len(_buffers) >= 16:                    # a handful of shapes (the SLAM loop sees few)
            _buffers.pop(next(iter(_buffers)))
        buf = _buffers[key] = _CallBuffers(n, m, dev)
    return buf


def icp_full(A, B, max_iterations: int = 20, tolerance: float = 1e-5, *, init_pose=None,
             max_corr_dist: Optional[float] = None) -> IcpOutput:
    """One alignment with every output of the new call surface (SURVEY.md §8b)."""
    A = _as_points(A, "A")
    B = _as_points(B, "B")
    lib = _cabi.lib()
    if len(A) > lib.b200icp_max_src_pitch() or len(B) > lib.b200icp_max_tgt_pitch():
        return _icp_full_large(A, B, max_iterations, tolerance, init_pose, max_corr_dist)
    n, m = len(A), len(B)
    buf = _call_buffers(n, m)
    hin = buf.h_in.numpy()
    hin[:2 * n] = A.reshape(-1)
    hin[2 * n:] = B.reshape(-1)
    buf.d_in.copy_(buf.h_in, non_blocking=True)
    pose = None
    if init_pose is not None:
        buf.h_pose.copy_(_pose6_host(init_pose))
        buf.d_pose.copy_(buf.h_pose.view(1, 6), non_blocking=True)
        pose = buf.d_pose
    align_pairs(buf.src, buf.tgt, n_pairs=1, max_iterations=max_iterations, tolerance=tolerance,
                init_pose=pose, max_corr_dist=max_corr_dist, out=buf.out)
    buf.h_out.copy_(buf.d_out, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    o = buf.h_out.numpy()
    ints = o[14:15].view(np.int32)
    return IcpOutput(
        R=o[0:4].reshape(2, 2).copy(), t=o[4:6].copy(),
        error=float(o[12]), iterations=int(ints[1]),
        R_last=o[6:10].reshape(2, 2).copy(), t_last=o[10:12].copy(),
        rmse=float(o[13]), fitness=int(ints[0]) / float(n),
        indices=o[16:16 + buf.n_idx].view(np.int32)[:n].astype(np.intp),
        src=o[16 + buf.n_idx:].reshape(n, 2).copy(),
    )


def _icp_full_large(A, B, max_iterations, tolerance, init_pose, max_corr_dist) -> IcpOutput:
    """Point sets beyond the fused per-pair kernel (> 1,024 source or > 4,096 target points, e.g. a
    scan against the 11 k-point local map of the reference's SLAM loop): the sharded-map path with
    a single shard -- same loop, same exactness, any size."""
    from .scan_to_map import MapShard, ScanToMap
    s2m = ScanToMap(MapShard(torch.from_numpy(B).cuda()), len(A), want_indices=True, local_only=True)
    ip = None
    if init_pose is not None:
        ip = _pose6(init_pose)[0].cpu().numpy()
    r = s2m.run(torch.from_numpy(A).cuda(), max_iterations=max_iterations, tolerance=tolerance,
                init_pose=ip, max_corr_dist=max_corr_dist)
    return IcpOutput(R=r.R, t=r.t, error=r.error, iterations=r.iterations, R_last=r.R_last, t_last=r.t_last,
                     rmse=r.rmse, fitness=r.inliers / float(len(A)),
                     indices=r.indices.cpu().numpy().astype(np.intp), src=r.src.cpu().numpy())


def icp(A, B, max_iterations: int = 20, tolerance: float = 1e-5, *, init_pose=None,
        max_corr_dist: Optional[float] = None) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """``icp(A, B, max_iterations=20, tolerance=1e-5) -> (src, R, t)``.

    Positional-compatible with labels_segmentation/icp.py:28.  Like the reference, the
    returned ``R, t`` are the LAST incremental update (icp.py:42,53), not the cumulative
    pose; use :func:`icp_full` for the cumulative pose, error and iteration count.
    """
    o = icp_full(A, B, max_iterations, tolerance, init_pose=init_pose, max_corr_dist=max_corr_dist)
    return o.src, o.R_last, o.t_last


def best_fit_transform(A, B) -> Tuple[np.ndarray, np.ndarray]:
    """``best_fit_transform(A, B) -> (R, t)`` for matched rows (labels_segmentation/icp.py:5-26)."""
    A = _as_points(A, "A")
    B = _as_points(B, "B")
    if len(A) != len(B):
        raise ValueError("A and B must have the same number of rows")     # NumPy would fail to broadcast
    pose = best_fit(ScanTable(torch.from_numpy(A[None]).cuda()), ScanTable(torch.from_numpy(B[None]).cuda()),
                    n_pairs=1)[0].cpu().numpy()
    return pose[:4].reshape(2, 2).copy(), pose[4:6].copy()


def nearest_neighbors(src, tgt) -> Tuple[np.ndarray, np.ndarray]:
    """``distances, indices = KDTree(tgt).query(src)`` (icp.py:37-38) on the device."""
    A = _as_points(src, "src")
    B = _as_points(tgt, "tgt")
    s = ScanTable(torch.from_numpy(A[None]).cuda(), None)
    t = ScanTable(torch.from_numpy(B[None]).cuda(), None)
    idx, d2 = nn_search(s, t, n_pairs=1)
    return np.sqrt(d2[0].cpu().numpy()), idx[0].cpu().numpy().astype(np.intp)


def registration_p2p(points1, points2, threshold: float = 200.0, voxel_size: Optional[float] = None,
                     trans_init=None, max_iteration: int = 50, tolerance: float = 1e-5):
    """Open3D-shaped point-to-point adapter: ``(rmse, T4x4)``.

    Positional-compatible with ``gicp(points1, points2, threshold, voxel_size, trans_init)``.
    Mirrors the call shape of ``gicp(points1, points2, threshold, voxel, trans_init)``
    (duc/ICP_LIDAR/gicp_lidar.py:12-36; caller duc/ICP_LIDAR/mainn.py:311) and of
    ``icp(...)`` in duc/code python/b.py:219-236, including the ``< 10`` points guard
    (gicp_lidar.py:13-15).  Gate / rmse semantics are parity-unpinned (Open3D is not
    vendored by the reference) and are defined by oracle.icp_oracle.icp_extended.
    ``points1`` / ``points2`` may be NumPy arrays or CUDA tensors ((N, 2) or (N, 3)); tensors stay
    on the device from the voxel grid to the pose (the SLAM loop passes its map that way).
    """
    def solve(p1, p2):
        lib = _cabi.lib()
        if p1.shape[0] > lib.b200icp_max_src_pitch() or p2.shape[0] > lib.b200icp_max_tgt_pitch():
            o = _icp_full_large(p1.cpu().numpy(), p2.cpu().numpy(), max_iteration, tolerance,
                                None if trans_init is None else np.asarray(trans_init), threshold)
            return o.rmse, o.R, o.t
        return _rmse_pose(align_pairs(ScanTable(p1[None].contiguous()), ScanTable(p2[None].contiguous()), n_pairs=1,
                                      max_iterations=max_iteration, tolerance=tolerance,
                                      init_pose=None if trans_init is None else _pose6(np.asarray(trans_init)),
                                      max_corr_dist=threshold))

    return _registration_4x4(points1, points2, voxel_size, solve)
