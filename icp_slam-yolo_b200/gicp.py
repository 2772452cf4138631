"""2D Generalized ICP (line-to-line) on the device: the registration objective of the reference's
``gicp(points1, points2, threshold, voxel, trans_init)`` (duc/ICP_LIDAR/gicp_lidar.py:12-36, called at
duc/ICP_LIDAR/slam_offline.py:382 and mainn.py:311).

Open3D is not vendored, so the model is defined by ``oracle/gicp_oracle.py`` (DESIGN.md §4.8):
per-point covariances regularised to (1, epsilon) on their principal axes, then Open3D's
RegistrationICP loop with one float64 Gauss-Newton step per update.  Every computation runs in
``libb200icp.so`` (``b200icp_estimate_covariances``, ``b200icp_gicp_batch``).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np
import torch

from . import _cabi
from .registration import (_DTYPES, AlignResult, ScanTable, _check_out, _check_pairs, _default_pairs, _init_pose_ptr,
                           _outputs, _problem, _ptr, _registration_4x4, _require_cuda, _rmse_pose, _stream_ptr,
                           alloc_outputs)


def estimate_covariances(table: ScanTable, k: int = 20, epsilon: float = 1e-3, stream=None) -> torch.Tensor:
    """Regularised covariance of every point from its k nearest points in the same row:
    float64 [rows, pitch, 3] (cxx, cxy, cyy), zeros past each row's length.  3 <= k <= 32."""
    out = torch.empty((table.rows, table.pitch, 3), dtype=torch.float64, device=table.points.device)
    with torch.cuda.device(table.points.device):
        rc = _cabi.lib().b200icp_estimate_covariances(_ptr(table.points), _ptr(table.lengths), table.rows, table.pitch,
                                                      _DTYPES[table.points.dtype], int(k), float(epsilon), _ptr(out),
                                                      _stream_ptr(stream))
    _cabi.check(rc, "b200icp_estimate_covariances")
    return out


def _check_cov(cov: torch.Tensor, table: ScanTable, name: str) -> None:
    if cov.dtype != torch.float64 or tuple(cov.shape) != (table.rows, table.pitch, 3):
        raise ValueError(f"{name} must be float64 [{table.rows}, {table.pitch}, 3] (estimate_covariances of "
                         f"the same table), got {cov.dtype} {tuple(cov.shape)}")
    _require_cuda(cov, name)
    if cov.device != table.points.device:
        raise ValueError(f"{name} must live on the device of its table")


def gicp_pairs(src: ScanTable, tgt: ScanTable, src_cov: torch.Tensor, tgt_cov: torch.Tensor, *,
               n_pairs: Optional[int] = None, pairing: str = "rowwise", src_row=None, tgt_row=None,
               first_pair: int = 0, max_iterations: int = 30, max_corr_dist: Optional[float] = None,
               init_pose: Optional[torch.Tensor] = None, relative_fitness: float = 1e-6,
               relative_rmse: float = 1e-6, want_indices: bool = False, want_src: bool = False,
               want_history: bool = False, out: Optional[AlignResult] = None, validate_rows: bool = False,
               stream=None) -> AlignResult:
    """The whole GICP loop of every pair on the device (one launch, one CTA per pair).

    Same pairings, row checks and output buffers as :func:`align_pairs`.  ``src_cov`` / ``tgt_cov``
    come from :func:`estimate_covariances` of the two tables.  Outputs: ``pose_total``;
    ``pose_last`` = last applied increment; ``error`` (mean inlier distance), ``rmse``, ``inliers``
    and ``indices`` at the final pose (+inf errors when no pair survived the gate);
    ``iterations`` = applied updates; ``index_history[:, it]`` = the correspondences update ``it`` used.
    Source rows hold up to 1,024 points, target rows up to 65,536.
    """
    pr = _problem(src, tgt, pairing, src_row, tgt_row, first_pair)
    b = _default_pairs(src, tgt, pairing, src_row, first_pair) if n_pairs is None else int(n_pairs)
    dev = src.points.device
    _check_pairs(src, tgt, pairing, src_row, tgt_row, b, validate_rows)
    _check_cov(src_cov, src, "src_cov")
    _check_cov(tgt_cov, tgt, "tgt_cov")
    if out is not None:
        _check_out(out, b, src.pitch, int(max_iterations), dev)
    else:
        out = alloc_outputs(b, src.pitch, dev, max_iterations=max_iterations, want_indices=want_indices,
                            want_src=want_src, want_history=want_history)
    opt = _cabi.GicpOptions()
    opt.max_iterations = int(max_iterations)
    opt.max_corr_dist = 0.0 if max_corr_dist is None else float(max_corr_dist)
    opt.relative_fitness, opt.relative_rmse = float(relative_fitness), float(relative_rmse)
    opt.init_pose = _init_pose_ptr(init_pose, b)
    with torch.cuda.device(dev):
        rc = _cabi.lib().b200icp_gicp_batch(C.byref(pr), b, C.byref(opt), _ptr(src_cov), _ptr(tgt_cov),
                                            C.byref(_outputs(out)), _stream_ptr(stream))
    _cabi.check(rc, "b200icp_gicp_batch")
    return out


def gicp_consecutive(table: ScanTable, k: int = 20, epsilon: float = 1e-3, *, max_iterations: int = 30,
                     max_corr_dist=None, out=None, stream=None, **kw) -> AlignResult:
    """Sequence odometry with GICP: pair p aligns row p+1 (source) onto row p (target).  The
    covariances are estimated once for the table and shared by both roles."""
    cov = estimate_covariances(table, k, epsilon, stream=stream)
    return gicp_pairs(table.slice_rows(1), table.slice_rows(0, table.rows - 1), cov[1:], cov[:-1],
                      n_pairs=table.rows - 1, max_iterations=max_iterations, max_corr_dist=max_corr_dist,
                      out=out, stream=stream, **kw)


def registration_gicp(points1, points2, threshold: float = 200.0, voxel_size: Optional[float] = None,
                      trans_init=None, max_iteration: int = 50, k: int = 20, epsilon: float = 1e-3,
                      relative_fitness: float = 1e-6, relative_rmse: float = 1e-6):
    """Open3D-shaped Generalized ICP: ``(rmse, T4x4)``, registering ``points1`` onto ``points2``.

    Positional-compatible with ``gicp(points1, points2, threshold, voxel_size, trans_init)``
    (duc/ICP_LIDAR/gicp_lidar.py:12-36), including the ``< 10`` points guard (gicp_lidar.py:13-15)
    and the voxel filter of both clouds (gicp_lidar.py:20-21).  NumPy arrays or CUDA tensors,
    (N, 2) or (N, 3); one device-to-host read.  rmse is +inf when no pair lies within ``threshold``.
    """
    def solve(p1, p2):
        s, t = ScanTable(p1[None].contiguous()), ScanTable(p2[None].contiguous())
        init = None
        if trans_init is not None:
            from .icp import _pose6
            init = _pose6(np.asarray(trans_init))
        return _rmse_pose(gicp_pairs(s, t, estimate_covariances(s, k, epsilon), estimate_covariances(t, k, epsilon),
                                     n_pairs=1, max_iterations=max_iteration, max_corr_dist=threshold, init_pose=init,
                                     relative_fitness=relative_fitness, relative_rmse=relative_rmse))

    return _registration_4x4(points1, points2, voxel_size, solve)
