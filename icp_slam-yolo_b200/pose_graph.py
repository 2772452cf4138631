"""Loop closure on the device: loop candidates from a trajectory, the information matrix of each
alignment, graph edges from verified alignments and a batched SE(2) pose-graph optimiser.

The reference has no loop closure; ``oracle/pose_graph_oracle.py`` defines the results (DESIGN.md
§4.9, conventions in include/b200icp.h).  Every computation runs in ``libb200icp.so``
(``b200icp_loop_candidates``, ``b200icp_information_batch``, ``b200icp_loop_edges``,
``b200icp_odometry_edges``, ``b200icp_pose_graph_optimize``); this module checks arguments and
allocates.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import List, Optional, Sequence, Union

import numpy as np
import torch

from . import _cabi
from .registration import AlignResult, ScanTable, _check_pairs, _compact_scratch, _default_pairs, _problem, _ptr, \
    _require_cuda, _stream_ptr, _workspace, align_pairs


def _pose_table(t: torch.Tensor, name: str) -> None:
    if t.dtype != torch.float64 or t.dim() != 2 or t.shape[1] != 6:
        raise ValueError(f"{name} must be float64 [n, 6], got {t.dtype} {tuple(t.shape)}")
    _require_cuda(t, name)


def loop_candidates(poses: torch.Tensor, min_gap: int, radius: float, *, capacity: Optional[int] = None,
                    strict: bool = False, stream=None):
    """Pairs (i < j) with j - i >= min_gap and |t_i - t_j|^2 <= radius^2, in PAIR_TRIANGLE order:
    ``(src_row = j, tgt_row = i, init_pose = X_i^-1 X_j)`` ready for ``align_pairs(pairing="explicit",
    init_pose=...)``.  poses: float64 [n, 6] CUDA.  With more candidates than ``capacity`` (default
    4 n) the buffers are re-allocated and the call repeated, or ``strict=True`` raises."""
    _pose_table(poses, "poses")
    n, dev = int(poses.shape[0]), poses.device
    cap = 4 * n if capacity is None else int(capacity)
    if cap < 0:
        raise ValueError("capacity < 0")
    count = torch.empty(1, dtype=torch.int64, device=dev)
    scratch = _compact_scratch(n * (n - 1) // 2, dev)
    while True:
        src = torch.empty(cap, dtype=torch.int32, device=dev)
        tgt = torch.empty(cap, dtype=torch.int32, device=dev)
        rel = torch.empty((cap, 6), dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            rc = _cabi.lib().b200icp_loop_candidates(_ptr(poses), n, int(min_gap), float(radius), cap, _ptr(src),
                                                     _ptr(tgt), _ptr(rel), _ptr(count), _ptr(scratch),
                                                     _stream_ptr(stream))
        _cabi.check(rc, "b200icp_loop_candidates")
        k = int(count.item())
        if k <= cap:
            return src[:k], tgt[:k], rel[:k]
        if strict:
            raise _cabi.B200IcpError(f"{k} loop candidates exceed the capacity {cap}")
        cap = k


def information_matrices(src: ScanTable, tgt: ScanTable, pose: torch.Tensor, indices: torch.Tensor,
                         max_corr_dist: Optional[float] = None, *, n_pairs: Optional[int] = None,
                         pairing: str = "rowwise", src_row=None, tgt_row=None, first_pair: int = 0,
                         stream=None):
    """Information matrix of every aligned pair, the 2D analogue of Open3D's
    ``get_information_matrix_from_point_clouds``: ``(info float64 [b, 6] = upper triangle (xx, xy, xt,
    yy, yt, tt), inliers int32 [b])``.  ``pose`` / ``indices`` as ``align_pairs(want_indices=True)`` or
    ``gicp_pairs`` return them (the indices of ``align_pairs`` are those of its last search, one update
    behind ``pose_total``)."""
    pr = _problem(src, tgt, pairing, src_row, tgt_row, first_pair)
    b = _default_pairs(src, tgt, pairing, src_row, first_pair) if n_pairs is None else int(n_pairs)
    _check_pairs(src, tgt, pairing, src_row, tgt_row, b, False)
    dev = src.points.device
    if pose.dtype != torch.float64 or pose.dim() != 2 or pose.shape[0] < b or pose.shape[1] != 6:
        raise ValueError(f"pose must be float64 [>={b}, 6]")
    if indices is None or indices.dtype != torch.int32 or indices.dim() != 2 or indices.shape[0] < b or \
            indices.shape[1] != src.pitch:
        raise ValueError(f"indices must be int32 [>={b}, {src.pitch}] (align_pairs(..., want_indices=True))")
    _require_cuda(pose, "pose")
    _require_cuda(indices, "indices")
    info = torch.empty((b, 6), dtype=torch.float64, device=dev)
    inl = torch.empty(b, dtype=torch.int32, device=dev)
    gate = 0.0 if max_corr_dist is None else float(max_corr_dist)
    with torch.cuda.device(dev):
        rc = _cabi.lib().b200icp_information_batch(C.byref(pr), b, _ptr(pose), _ptr(indices), gate, _ptr(info),
                                                   _ptr(inl), _stream_ptr(stream))
    _cabi.check(rc, "b200icp_information_batch")
    return info, inl


def _edge_buffers(b: int, dev):
    return (torch.empty(b, dtype=torch.int32, device=dev), torch.empty(b, dtype=torch.int32, device=dev),
            torch.empty((b, 6), dtype=torch.float64, device=dev), torch.empty((b, 6), dtype=torch.float64, device=dev),
            torch.empty(1, dtype=torch.int64, device=dev))


def _info_ptr(info, b, name="info"):
    if info is None:
        return None
    _pose_table(info, name)
    if info.shape[0] < b:
        raise ValueError(f"{name} must hold {b} rows")
    return _ptr(info)


@dataclass
class PoseGraph:
    """Edges of one SE(2) pose graph (CUDA tensors): edge (i, j) measures Z_ij ~ X_i^-1 X_j with
    information ``info`` (upper triangle [6]).  ``n_nodes`` poses; ``dropped`` = odometry pairs left
    out because their alignment failed."""
    n_nodes: int
    edge_i: torch.Tensor
    edge_j: torch.Tensor
    meas: torch.Tensor
    info: torch.Tensor
    dropped: int = 0

    def __post_init__(self):
        self.validate()

    def validate(self) -> None:
        """The optimiser reads the edge tensors blindly: int32 [e] ``edge_i`` / ``edge_j`` and float64
        [e, 6] ``meas`` / ``info``, contiguous CUDA tensors on one device (endpoints are range-checked on
        the device, status bad_edge)."""
        if isinstance(self.n_nodes, bool) or not isinstance(self.n_nodes, (int, np.integer)) or self.n_nodes < 0:
            raise ValueError(f"n_nodes must be an int >= 0, got {self.n_nodes!r}")
        e = None
        for name in ("edge_i", "edge_j", "meas", "info"):
            t = getattr(self, name)
            if not isinstance(t, torch.Tensor):
                raise ValueError(f"{name} must be a tensor")
            want = (torch.int32, 1) if name.startswith("edge") else (torch.float64, 2)
            if t.dtype != want[0] or t.dim() != want[1] or (want[1] == 2 and t.shape[1] != 6):
                shape = "[n_edges]" if want[1] == 1 else "[n_edges, 6]"
                raise ValueError(f"{name} must be {want[0]} {shape}, got {t.dtype} {tuple(t.shape)}")
            if e is None:
                e = int(t.shape[0])
            elif int(t.shape[0]) != e:
                raise ValueError(f"edge_i, edge_j, meas and info must have one row per edge ({e}), "
                                 f"{name} has {int(t.shape[0])}")
        for name in ("edge_i", "edge_j", "meas", "info"):
            _require_cuda(getattr(self, name), name)
        if len({getattr(self, n).device for n in ("edge_i", "edge_j", "meas", "info")}) != 1:
            raise ValueError("edge_i, edge_j, meas and info must live on one device")

    @property
    def n_edges(self) -> int:
        return int(self.edge_i.shape[0])

    @staticmethod
    def from_odometry(result: AlignResult, info: Optional[torch.Tensor] = None, stream=None) -> "PoseGraph":
        """Edges (p, p + 1, pose_total[p], info[p]) of a sequence-odometry result (``align_consecutive``
        / ``gicp_consecutive``); pairs with iterations == 0 or error == +inf are dropped.  info None:
        identity information."""
        b, dev = int(result.pose_total.shape[0]), result.pose_total.device
        ei, ej, meas, inf, count = _edge_buffers(b, dev)
        with torch.cuda.device(dev):
            rc = _cabi.lib().b200icp_odometry_edges(b, _ptr(result.pose_total), _ptr(result.error),
                                                    _ptr(result.iterations), _info_ptr(info, b), _ptr(ei), _ptr(ej),
                                                    _ptr(meas), _ptr(inf), _ptr(count), _ptr(_compact_scratch(b, dev)),
                                                    _stream_ptr(stream))
        _cabi.check(rc, "b200icp_odometry_edges")
        k = int(count.item())
        return PoseGraph(b + 1, ei[:k], ej[:k], meas[:k], inf[:k], b - k)

    def add_loops(self, result: AlignResult, src_row: torch.Tensor, tgt_row: torch.Tensor,
                  info: Optional[torch.Tensor], *, min_fitness: float, max_rmse: float,
                  src_lengths: Optional[torch.Tensor] = None, src_pitch: Optional[int] = None,
                  stream=None) -> int:
        """Append the verified loop candidates: pair p is kept when its rmse is finite and <= max_rmse
        and inliers / source points >= min_fitness (source points = src_lengths[src_row[p]], capped at
        src_pitch).  Returns the number of edges added."""
        b, dev = int(result.pose_total.shape[0]), result.pose_total.device
        for name, t in (("src_row", src_row), ("tgt_row", tgt_row)):
            if t.dtype != torch.int32 or t.dim() != 1 or t.shape[0] < b:
                raise ValueError(f"{name} must be int32 [>={b}]")
            _require_cuda(t, name)
        if result.rmse is None or result.inliers is None:
            raise ValueError("result needs rmse and inliers")
        pitch = int(src_pitch) if src_pitch is not None else (int(result.indices.shape[1]) if result.indices is not None else 0)
        if pitch < 1:
            raise ValueError("src_pitch is required when result has no indices")
        ei, ej, meas, inf, count = _edge_buffers(b, dev)
        with torch.cuda.device(dev):
            rc = _cabi.lib().b200icp_loop_edges(b, _ptr(result.pose_total), _ptr(result.rmse), _ptr(result.inliers),
                                                _ptr(src_lengths), pitch, _ptr(src_row), _ptr(tgt_row),
                                                _info_ptr(info, b), float(min_fitness), float(max_rmse), _ptr(ei),
                                                _ptr(ej), _ptr(meas), _ptr(inf), _ptr(count), _ptr(_compact_scratch(b, dev)),
                                                _stream_ptr(stream))
        _cabi.check(rc, "b200icp_loop_edges")
        k = int(count.item())
        self.edge_i = torch.cat([self.edge_i, ei[:k]])
        self.edge_j = torch.cat([self.edge_j, ej[:k]])
        self.meas = torch.cat([self.meas, meas[:k]])
        self.info = torch.cat([self.info, inf[:k]])
        return k


@dataclass
class PoseGraphResult:
    """Per call: ``poses`` [sum n, 6] (graphs concatenated; ``split()`` per graph) and per graph
    ``chi2_initial``, ``chi2_final``, ``iterations`` (Gauss-Newton steps), ``pcg_iterations``,
    ``status`` (0 converged, 1 max_iterations, 2 pcg_limit, 3 non_finite, 4 bad_edge, 5 pcg_breakdown),
    ``isolated`` (nodes no edge touches) and ``anchored`` (components without the gauge node, each held
    at its lowest-index node)."""
    poses: torch.Tensor
    chi2_initial: torch.Tensor
    chi2_final: torch.Tensor
    iterations: torch.Tensor
    pcg_iterations: torch.Tensor
    status: torch.Tensor
    isolated: torch.Tensor
    anchored: torch.Tensor
    node_offset: List[int]

    def split(self) -> List[torch.Tensor]:
        o = self.node_offset
        return [self.poses[o[k]:o[k + 1]] for k in range(len(o) - 1)]


def optimize_pose_graph(graphs: Union[PoseGraph, Sequence[PoseGraph]],
                        poses: Union[torch.Tensor, Sequence[torch.Tensor]], *,
                        fixed: Union[int, Sequence[int]] = 0, max_iterations: int = 20, tolerance: float = 1e-9,
                        pcg_max_iterations: int = 20000, pcg_tolerance: float = 1e-14, damping: float = 0.0,
                        stream=None) -> PoseGraphResult:
    """Gauss-Newton on every graph of the batch in one launch (one CTA per graph), PCG solves on the
    device.  ``poses``: initial float64 [n_g, 6] per graph (e.g. ``chain_poses_device`` of the
    odometry); ``fixed``: the gauge node of every graph, or one per graph.  Every other connected
    component of a graph is held at its lowest-index node (counted in ``anchored``)."""
    single = isinstance(graphs, PoseGraph)
    gl = [graphs] if single else list(graphs)
    pl = [poses] if isinstance(poses, torch.Tensor) else list(poses)
    if len(gl) != len(pl):
        raise ValueError("one initial pose table per graph")
    fx = [int(fixed)] * len(gl) if isinstance(fixed, int) else [int(f) for f in fixed]
    if len(fx) != len(gl):
        raise ValueError("one fixed node per graph")
    if not gl:
        raise ValueError("no graph")
    for g in gl:
        if not isinstance(g, PoseGraph):
            raise ValueError("graphs must be PoseGraph objects")
        g.validate()                       # again: the fields may have been replaced since construction
    dev = pl[0].device
    for g, p, f in zip(gl, pl, fx):
        _pose_table(p, "poses")
        if int(p.shape[0]) != g.n_nodes:
            raise ValueError(f"a graph of {g.n_nodes} nodes needs {g.n_nodes} initial poses, got {int(p.shape[0])}")
        if p.device != dev or g.edge_i.device != dev:
            raise ValueError("every graph and pose table must live on one device")
        if f < 0 or (g.n_nodes > 0 and f >= g.n_nodes):
            raise ValueError(f"fixed node {f} is outside the graph of {g.n_nodes} nodes")
    node_off = np.zeros(len(gl) + 1, dtype=np.int64)
    edge_off = np.zeros(len(gl) + 1, dtype=np.int64)
    node_off[1:] = np.cumsum([g.n_nodes for g in gl])
    edge_off[1:] = np.cumsum([g.n_edges for g in gl])
    fixed_np = np.asarray(fx, dtype=np.int32)
    P = torch.cat(pl).contiguous() if len(pl) > 1 else pl[0].contiguous()
    ei = torch.cat([g.edge_i for g in gl]).contiguous()
    ej = torch.cat([g.edge_j for g in gl]).contiguous()
    meas = torch.cat([g.meas for g in gl]).contiguous()
    info = torch.cat([g.info for g in gl]).contiguous()
    batch = _cabi.PoseGraphBatch()
    batch.n_graphs = len(gl)
    batch.node_offset = node_off.ctypes.data
    batch.edge_offset = edge_off.ctypes.data
    batch.fixed_node = fixed_np.ctypes.data
    batch.poses_in, batch.edge_i, batch.edge_j = P.data_ptr(), ei.data_ptr(), ej.data_ptr()
    batch.meas, batch.info = meas.data_ptr(), info.data_ptr()
    opt = _cabi.PoseGraphOptions()
    opt.max_iterations, opt.pcg_max_iterations = int(max_iterations), int(pcg_max_iterations)
    opt.tolerance, opt.pcg_tolerance, opt.damping = float(tolerance), float(pcg_tolerance), float(damping)
    G = len(gl)
    f64 = dict(dtype=torch.float64, device=dev)
    i32 = dict(dtype=torch.int32, device=dev)
    res = PoseGraphResult(torch.empty_like(P), torch.empty(G, **f64), torch.empty(G, **f64), torch.empty(G, **i32),
                          torch.empty(G, **i32), torch.empty(G, **i32), torch.empty(G, **i32), torch.empty(G, **i32),
                          node_off.tolist())
    out = _cabi.PoseGraphOutputs()
    out.poses, out.chi2_initial, out.chi2_final = res.poses.data_ptr(), res.chi2_initial.data_ptr(), res.chi2_final.data_ptr()
    out.iterations, out.pcg_iterations = res.iterations.data_ptr(), res.pcg_iterations.data_ptr()
    out.status, out.isolated, out.anchored = res.status.data_ptr(), res.isolated.data_ptr(), res.anchored.data_ptr()
    L = _cabi.lib()
    try:
        ws, nbytes = _workspace(L.b200icp_pose_graph_workspace_bytes, C.byref(batch), device=dev)
    except _cabi.B200IcpError:              # the optimiser's own checks say what is wrong with the batch
        _cabi.check(L.b200icp_pose_graph_optimize(C.byref(batch), C.byref(opt), C.byref(out), None, 0, None),
                    "b200icp_pose_graph_optimize")
        raise
    with torch.cuda.device(dev):
        rc = L.b200icp_pose_graph_optimize(C.byref(batch), C.byref(opt), C.byref(out), _ptr(ws), nbytes,
                                           _stream_ptr(stream))
    _cabi.check(rc, "b200icp_pose_graph_optimize")
    return res


def close_loops(table: ScanTable, odometry_result: AlignResult, *, min_gap: int, radius: float,
                max_corr_dist: float, min_fitness: float, max_rmse: float, registration: str = "p2p",
                max_iterations: int = 30, gicp_k: int = 20, gicp_epsilon: float = 1e-3, optimize_kw=None,
                stream=None):
    """Close the loops of a sequence: odometry edges from ``odometry_result`` (``align_consecutive`` or
    ``gicp_consecutive`` over ``table`` with ``want_indices=True``), loop candidates from the chained
    trajectory, verification of every candidate by ``align_pairs`` ("p2p") or ``gicp_pairs`` ("gicp")
    from its relative pose, the accepted loop edges, and the optimised trajectory.  A stretch of the
    trajectory cut off by a dropped odometry pair that no accepted loop bridges is held at its first node
    and keeps its odometry placement (``stats["anchored"]`` counts such stretches).
    Returns ``(poses float64 [rows, 6], graph, stats)``."""
    from .odometry import chain_poses_device
    if registration not in ("p2p", "gicp"):
        raise ValueError(f"registration must be 'p2p' or 'gicp', got {registration!r}")
    if odometry_result.indices is None:
        raise ValueError("odometry_result needs its correspondences (want_indices=True)")
    rows = table.rows
    if int(odometry_result.pose_total.shape[0]) != rows - 1:
        raise ValueError(f"odometry_result must hold the {rows - 1} consecutive pairs of the table")
    srcs, tgts = table.slice_rows(1), table.slice_rows(0, rows - 1)
    odo_info, _ = information_matrices(srcs, tgts, odometry_result.pose_total, odometry_result.indices, max_corr_dist,
                                       n_pairs=rows - 1, stream=stream)
    graph = PoseGraph.from_odometry(odometry_result, odo_info, stream=stream)
    poses0 = chain_poses_device(odometry_result.pose_total, stream=stream)
    src_row, tgt_row, init = loop_candidates(poses0, min_gap, radius, stream=stream)
    k = int(src_row.shape[0])
    loops = 0
    if k > 0:
        kw = dict(n_pairs=k, pairing="explicit", src_row=src_row, tgt_row=tgt_row, init_pose=init,
                  max_iterations=max_iterations, max_corr_dist=max_corr_dist, want_indices=True, stream=stream)
        if registration == "p2p":
            res = align_pairs(table, table, **kw)
        else:
            from .gicp import estimate_covariances, gicp_pairs
            cov = estimate_covariances(table, gicp_k, gicp_epsilon, stream=stream)
            res = gicp_pairs(table, table, cov, cov, **kw)
        info, _ = information_matrices(table, table, res.pose_total, res.indices, max_corr_dist, n_pairs=k,
                                       pairing="explicit", src_row=src_row, tgt_row=tgt_row, stream=stream)
        loops = graph.add_loops(res, src_row, tgt_row, info, min_fitness=min_fitness, max_rmse=max_rmse,
                                src_lengths=table.lengths, src_pitch=table.pitch, stream=stream)
    r = optimize_pose_graph(graph, poses0, stream=stream, **(optimize_kw or {}))
    stats = {"candidates": k, "loop_edges": loops, "odometry_edges": graph.n_edges - loops,
             "dropped_odometry": graph.dropped, "chi2_initial": float(r.chi2_initial[0]),
             "chi2_final": float(r.chi2_final[0]), "iterations": int(r.iterations[0]),
             "pcg_iterations": int(r.pcg_iterations[0]), "status": _cabi.PG_STATUS_NAMES[int(r.status[0])],
             "isolated": int(r.isolated[0]), "anchored": int(r.anchored[0])}
    return r.poses, graph, stats
