"""Batched device-side registration: PyTorch tensors in and out, CUDA through the C ABI.

This is the host-side mirror of the reference's registration boundary
(labels_segmentation/icp.py:28-53) for *batches* of scan pairs.  Tensors only carry
device memory and the stream; every computation happens in ``libb200icp.so``.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np
import torch

from . import _cabi

_DTYPES = {torch.float32: _cabi.F32, torch.float64: _cabi.F64}
# kernel="auto" takes the CTA-per-pair kernel up to this many pairs, the W-warps-per-pair kernel above
# (kAutoCtaPairs in csrc/b200icp.cu)
_AUTO_CTA_PAIRS = 512
_PAIRINGS = {"rowwise": _cabi.PAIR_ROWWISE, "explicit": _cabi.PAIR_EXPLICIT,
             "triangle": _cabi.PAIR_TRIANGLE}


def _require_cuda(t: torch.Tensor, name: str) -> None:
    if not t.is_cuda:
        raise _cabi.B200IcpError(f"{name} must be a CUDA tensor: this path has no CPU fallback")
    if not t.is_contiguous():
        raise _cabi.B200IcpError(f"{name} must be contiguous")


@dataclass
class ScanTable:
    """Ragged scans padded to a common pitch in HBM.

    points  : [rows, pitch, 2] float32/float64 CUDA tensor, (x, y) interleaved
    lengths : [rows] int32 CUDA tensor of valid points per row, or None (= all full)
    """
    points: torch.Tensor
    lengths: Optional[torch.Tensor] = None

    def __post_init__(self):
        p = self.points
        if p.dim() != 3 or p.shape[2] != 2:
            raise ValueError(f"points must be [rows, pitch, 2], got {tuple(p.shape)}")
        if p.dtype not in _DTYPES:
            raise ValueError("points must be float32 or float64")
        _require_cuda(p, "points")
        if self.lengths is not None:
            l = self.lengths
            if l.dtype != torch.int32 or l.dim() != 1 or l.shape[0] != p.shape[0]:
                raise ValueError("lengths must be int32 [rows]")
            _require_cuda(l, "lengths")

    @property
    def rows(self) -> int:
        return int(self.points.shape[0])

    @property
    def pitch(self) -> int:
        return int(self.points.shape[1])

    def slice_rows(self, start: int, stop: Optional[int] = None) -> "ScanTable":
        """Row view sharing memory (e.g. rows 1.. as the sources of sequence odometry)."""
        pts = self.points[start:stop]
        lens = None if self.lengths is None else self.lengths[start:stop]
        return ScanTable(pts, lens)

    @staticmethod
    def pack_host(scans: Sequence[np.ndarray], dtype=np.float64, pitch: Optional[int] = None,
                  pin: bool = False):
        """Pad a list of (Ni, >=2) arrays into host tensors (points, lengths)."""
        n = len(scans)
        longest = max((len(s) for s in scans), default=1)
        pitch = max(1, longest) if pitch is None else int(pitch)
        if longest > pitch:
            raise ValueError(f"scan with {longest} points does not fit pitch {pitch}")
        pts = np.zeros((n, pitch, 2), dtype=dtype)
        lens = np.zeros(n, dtype=np.int32)
        for i, s in enumerate(scans):
            s = np.asarray(s)
            if s.size:
                pts[i, : len(s)] = s[:, :2]
            lens[i] = len(s)
        tp, tl = torch.from_numpy(pts), torch.from_numpy(lens)
        if pin:
            tp, tl = tp.pin_memory(), tl.pin_memory()
        return tp, tl

    @staticmethod
    def from_list(scans: Sequence[np.ndarray], dtype=np.float64, device="cuda",
                  pitch: Optional[int] = None) -> "ScanTable":
        tp, tl = ScanTable.pack_host(scans, dtype, pitch)
        return ScanTable(tp.to(device), tl.to(device))


@dataclass
class AlignResult:
    """Device tensors, one row per pair.  Poses are [R00 R01 R10 R11 tx ty]."""
    pose_total: torch.Tensor          # cumulative: src_final = R A + t
    pose_last: torch.Tensor           # last increment: what the reference icp() returns
    error: torch.Tensor               # lagged mean NN distance (icp.py:48)
    rmse: torch.Tensor
    inliers: torch.Tensor
    iterations: torch.Tensor
    indices: Optional[torch.Tensor] = None
    src_final: Optional[torch.Tensor] = None
    index_history: Optional[torch.Tensor] = None
    evaluated_pairs: Optional[torch.Tensor] = None   # int64: pair-evals the sweep executed

    def rotation(self, which: str = "total") -> torch.Tensor:
        p = self.pose_total if which == "total" else self.pose_last
        return p[:, :4].reshape(-1, 2, 2)

    def translation(self, which: str = "total") -> torch.Tensor:
        p = self.pose_total if which == "total" else self.pose_last
        return p[:, 4:6]

    def theta(self, which: str = "total") -> torch.Tensor:
        p = self.pose_total if which == "total" else self.pose_last
        return torch.atan2(p[:, 2], p[:, 0])


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream_ptr(stream) -> C.c_void_p:
    s = torch.cuda.current_stream() if stream is None else stream
    return C.c_void_p(s.cuda_stream)


def _compact_scratch(n: int, device) -> torch.Tensor:
    return torch.empty((n + 1023) // 1024 + 1, dtype=torch.int64, device=device)   # compact.cuh: a count per 1,024


def _workspace(query, *args, device):        # query: a b200icp_*_workspace_bytes function
    nbytes = int(query(*args))
    if nbytes < 0:
        raise _cabi.B200IcpError(f"{query.__name__} failed")
    return torch.empty(max(nbytes, 1), dtype=torch.uint8, device=device), nbytes


def _problem(src: ScanTable, tgt: ScanTable, pairing: str, src_row, tgt_row, first_pair: int):
    if src.points.dtype != tgt.points.dtype:
        raise ValueError("source and target tables must share a dtype")
    if src.points.device != tgt.points.device:
        raise ValueError("source and target tables must live on the same device")
    pr = _cabi.Problem()
    pr.src_points = src.points.data_ptr()
    pr.tgt_points = tgt.points.data_ptr()
    pr.src_len = None if src.lengths is None else src.lengths.data_ptr()
    pr.tgt_len = None if tgt.lengths is None else tgt.lengths.data_ptr()
    pr.src_pitch, pr.tgt_pitch = src.pitch, tgt.pitch
    pr.dtype = _DTYPES[src.points.dtype]
    pr.pairing = _PAIRINGS[pairing]
    if pairing == "explicit":
        for name, t in (("src_row", src_row), ("tgt_row", tgt_row)):
            if t is None or t.dtype != torch.int32:
                raise ValueError(f"{name} must be an int32 CUDA tensor for explicit pairing")
            _require_cuda(t, name)
        pr.src_row, pr.tgt_row = src_row.data_ptr(), tgt_row.data_ptr()
    if pairing == "triangle":
        if src.points.data_ptr() != tgt.points.data_ptr():
            raise ValueError("triangle pairing enumerates pairs of ONE table")
        pr.n_rows = src.rows
        pr.first_pair = int(first_pair)
    return pr


def _default_pairs(src, tgt, pairing, src_row, first_pair):
    if pairing == "rowwise":
        return min(src.rows, tgt.rows)
    if pairing == "explicit":
        return int(src_row.shape[0])
    r = src.rows
    return r * (r - 1) // 2 - int(first_pair)


def _check_pairs(src, tgt, pairing, src_row, tgt_row, b, validate_rows):
    """The C side sees pointers only: row counts are checked here."""
    if b < 0:
        raise ValueError("n_pairs < 0")
    if pairing == "rowwise" and b > min(src.rows, tgt.rows):
        raise ValueError(f"n_pairs = {b} exceeds the tables ({src.rows} source rows, {tgt.rows} target rows)")
    if pairing == "explicit":
        for name, t, rows in (("src_row", src_row, src.rows), ("tgt_row", tgt_row, tgt.rows)):
            if t.dim() != 1 or t.shape[0] < b:
                raise ValueError(f"{name} must hold at least n_pairs = {b} entries")
            if validate_rows and b > 0:          # one device synchronisation: opt-in
                lo, hi = int(t[:b].min()), int(t[:b].max())
                if lo < 0 or hi >= rows:
                    raise ValueError(f"{name} has entries outside [0, {rows})")


def _check_out(out: "AlignResult", b: int, src_pitch: int, max_iterations: int, device) -> None:
    """A caller-supplied result buffer is written blindly by the kernel: shapes must fit."""
    def need(t, name, shape, dtype):
        if t is None:
            return
        if t.dtype != dtype or t.device != device or not t.is_contiguous():
            raise ValueError(f"out.{name} must be a contiguous {dtype} tensor on {device}")
        if t.dim() != len(shape) or t.shape[0] < shape[0] or tuple(t.shape[1:]) != tuple(shape[1:]):
            raise ValueError(f"out.{name} has shape {tuple(t.shape)}, needs [>={shape[0]}{''.join(', %d' % d for d in shape[1:])}]")
    for name in ("pose_total", "pose_last"):
        need(getattr(out, name), name, (b, 6), torch.float64)
    for name in ("error", "rmse"):
        need(getattr(out, name), name, (b,), torch.float64)
    for name in ("inliers", "iterations"):
        need(getattr(out, name), name, (b,), torch.int32)
    need(out.indices, "indices", (b, src_pitch), torch.int32)
    need(out.src_final, "src_final", (b, src_pitch, 2), torch.float64)
    need(out.evaluated_pairs, "evaluated_pairs", (b,), torch.int64)
    if out.index_history is not None:
        h = out.index_history
        if (h.dtype != torch.int32 or h.device != device or not h.is_contiguous() or h.dim() != 3 or
                h.shape[0] < b or h.shape[1] != max_iterations or h.shape[2] != src_pitch):
            raise ValueError(f"out.index_history must be int32 [>={b}, {max_iterations}, {src_pitch}] "
                             f"(the kernel strides it by max_iterations), got {tuple(h.shape)}")


def _kernel_flags(kernel: str, dense_sweep: bool, sweep_reuse: bool = True, pair_warps: int = 0) -> int:
    """b200icp_options.flags / the flags of b200icp_nn_batch for the Python-side kernel choice."""
    return ((_cabi.FLAG_DENSE_SWEEP if dense_sweep else 0) | (0 if sweep_reuse else _cabi.FLAG_NO_SWEEP_REUSE) |
            {"auto": 0, "warp": _cabi.FLAG_WARP_KERNEL, "cta": _cabi.FLAG_CTA_KERNEL}[kernel] |
            ((int(pair_warps) & 7) << _cabi.FLAG_PAIR_WARPS_SHIFT))


def _init_pose_ptr(init_pose: Optional[torch.Tensor], b: int):
    """Device pointer of an optional float64 [b, 6] initial pose (None: identity)."""
    if init_pose is None:
        return None
    if init_pose.dtype != torch.float64 or tuple(init_pose.shape) != (b, 6):
        raise ValueError("init_pose must be float64 [n_pairs, 6]")
    _require_cuda(init_pose, "init_pose")
    return init_pose.data_ptr()


def _outputs(out: "AlignResult") -> "_cabi.Outputs":
    """The b200icp_outputs view of a result buffer; pose_total, error and iterations are required."""
    o = _cabi.Outputs()
    o.pose_total, o.error, o.iterations = out.pose_total.data_ptr(), out.error.data_ptr(), out.iterations.data_ptr()
    o.pose_last, o.rmse, o.inliers = _ptr(out.pose_last), _ptr(out.rmse), _ptr(out.inliers)
    o.indices, o.src_final, o.index_history = _ptr(out.indices), _ptr(out.src_final), _ptr(out.index_history)
    o.evaluated_pairs = _ptr(out.evaluated_pairs)
    return o


def _device_points(p) -> torch.Tensor:
    """NumPy array or tensor, (N, 2) or (N, 3) -> contiguous float64 (N, 2) CUDA tensor."""
    if isinstance(p, torch.Tensor):
        t = p[:, :2].to(device="cuda", dtype=torch.float64)
    else:
        t = torch.from_numpy(np.ascontiguousarray(np.asarray(p, dtype=np.float64)[:, :2])).cuda()
    return t.contiguous()


def _registration_4x4(points1, points2, voxel_size, solve):
    """The Open3D-shaped ``(rmse, T4x4)`` call around ``solve(p1, p2) -> (rmse, R, t)``: the ``< 10``
    points guard (gicp_lidar.py:13-15), both clouds on the device as float64 (N, 2), and the voxel
    filter of both clouds (gicp_lidar.py:20-21)."""
    if len(points1) < 10 or len(points2) < 10:
        return float("inf"), np.eye(4)
    p1, p2 = _device_points(points1), _device_points(points2)
    if voxel_size:
        from .mapping import voxel_down_sample
        p1, p2 = voxel_down_sample(p1, voxel_size), voxel_down_sample(p2, voxel_size)
    rmse, R, t = solve(p1, p2)
    T = np.eye(4)
    T[:2, :2] = R
    T[:2, 3] = t
    return rmse, T


def _rmse_pose(res: "AlignResult"):
    """(rmse, R, t) of pair 0, in one device-to-host read."""
    host = torch.cat([res.pose_total[0], res.rmse]).cpu().numpy()
    return float(host[6]), host[:4].reshape(2, 2), host[4:6]


def nn_search(src: ScanTable, tgt: ScanTable, *, n_pairs: Optional[int] = None,
              pairing: str = "rowwise", src_row=None, tgt_row=None, first_pair: int = 0,
              want_dist2: bool = True, out_idx=None, out_dist2=None, validate_rows: bool = False,
              kernel: str = "auto", dense_sweep: bool = False, stream=None):
    """Nearest target index for every source point of every pair.

    Replaces ``KDTree(B).query(src)`` (icp.py:37-38): returns (idx int32 [B,pitch],
    dist2 float64 [B,pitch] or None); idx = -1 beyond a row's length.  ``kernel``: "auto" (by
    batch size), "warp" or "cta"; ``dense_sweep`` disables the culling of target groups (A/B).
    """
    pr = _problem(src, tgt, pairing, src_row, tgt_row, first_pair)
    b = _default_pairs(src, tgt, pairing, src_row, first_pair) if n_pairs is None else int(n_pairs)
    dev = src.points.device
    _check_pairs(src, tgt, pairing, src_row, tgt_row, b, validate_rows)
    for name, t, dt in (("out_idx", out_idx, torch.int32), ("out_dist2", out_dist2, torch.float64)):
        if t is not None and (t.dtype != dt or t.device != dev or not t.is_contiguous() or t.dim() != 2 or
                              t.shape[0] < b or t.shape[1] != src.pitch):
            raise ValueError(f"{name} must be a contiguous {dt} [>={b}, {src.pitch}] tensor on {dev}")
    idx = out_idx if out_idx is not None else torch.empty((b, src.pitch), dtype=torch.int32, device=dev)
    d2 = out_dist2
    if d2 is None and want_dist2:
        d2 = torch.empty((b, src.pitch), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        rc = _cabi.lib().b200icp_nn_batch(C.byref(pr), b, _ptr(idx), _ptr(d2), _kernel_flags(kernel, dense_sweep),
                                          _stream_ptr(stream))
    _cabi.check(rc, "b200icp_nn_batch")
    return idx, d2


def alloc_outputs(n_pairs: int, src_pitch: int, device, *, max_iterations: int = 0,
                  want_indices=False, want_src=False, want_history=False,
                  want_stats=False) -> AlignResult:
    f64 = dict(dtype=torch.float64, device=device)
    i32 = dict(dtype=torch.int32, device=device)
    return AlignResult(
        pose_total=torch.empty((n_pairs, 6), **f64),
        pose_last=torch.empty((n_pairs, 6), **f64),
        error=torch.empty(n_pairs, **f64),
        rmse=torch.empty(n_pairs, **f64),
        inliers=torch.empty(n_pairs, **i32),
        iterations=torch.empty(n_pairs, **i32),
        indices=torch.empty((n_pairs, src_pitch), **i32) if want_indices else None,
        src_final=torch.empty((n_pairs, src_pitch, 2), **f64) if want_src else None,
        index_history=(torch.full((n_pairs, max_iterations, src_pitch), -1, **i32)
                       if want_history else None),
        evaluated_pairs=torch.zeros(n_pairs, dtype=torch.int64, device=device) if want_stats else None,
    )


def align_pairs(src: ScanTable, tgt: ScanTable, *, n_pairs: Optional[int] = None,
                pairing: str = "rowwise", src_row=None, tgt_row=None, first_pair: int = 0,
                max_iterations: int = 20, tolerance: float = 1e-5,
                init_pose: Optional[torch.Tensor] = None, max_corr_dist: Optional[float] = None,
                want_indices: bool = False, want_src: bool = False, want_history: bool = False,
                want_stats: bool = False, dense_sweep: bool = False, sweep_reuse: bool = True,
                kernel: str = "auto", pair_warps: int = 0, out: Optional[AlignResult] = None,
                validate_rows: bool = False, stream=None) -> AlignResult:
    """Run the whole ICP loop of every pair on the device (one kernel launch).

    Replaces ``icp(A, B, max_iterations, tolerance)`` (icp.py:28-53) for a batch:
    same defaults, same convergence rule, same lagged error.  ``init_pose`` is
    [B,6] float64 (R row-major, t); ``max_corr_dist`` None = exactly the reference.
    ``dense_sweep`` evaluates every source-target pair instead of culling target groups that are
    provably out of reach (identical results; only worth it for spatially unordered point sets).
    ``sweep_reuse=False`` sweeps every pass in every iteration instead of skipping the sweep of a
    pass whose points provably keep their nearest neighbour's group (identical results; A/B knob).
    ``kernel``: "auto" (CTA-per-pair fused kernel up to 512 pairs -- lowest latency --, the
    W-warps-per-pair throughput kernel above), "warp" (throughput kernel) or "cta".
    ``pair_warps`` forces W (1..4; 0 = auto).
    """
    pr = _problem(src, tgt, pairing, src_row, tgt_row, first_pair)
    b = _default_pairs(src, tgt, pairing, src_row, first_pair) if n_pairs is None else int(n_pairs)
    dev = src.points.device
    _check_pairs(src, tgt, pairing, src_row, tgt_row, b, validate_rows)
    if out is not None:
        _check_out(out, b, src.pitch, int(max_iterations), dev)
    if out is None:
        out = alloc_outputs(b, src.pitch, dev, max_iterations=max_iterations,
                            want_indices=want_indices, want_src=want_src, want_history=want_history,
                            want_stats=want_stats)
    opt = _cabi.Options()
    opt.max_iterations = int(max_iterations)
    opt.flags = _kernel_flags(kernel, dense_sweep, sweep_reuse, pair_warps)
    opt.tolerance = float(tolerance)
    opt.max_corr_dist = 0.0 if max_corr_dist is None else float(max_corr_dist)
    opt.init_pose = _init_pose_ptr(init_pose, b)
    o = _outputs(out)
    with torch.cuda.device(dev):
        rc = _cabi.lib().b200icp_align_batch(C.byref(pr), b, C.byref(opt), C.byref(o),
                                             _stream_ptr(stream))
    _cabi.check(rc, "b200icp_align_batch")
    return out


def best_fit(src: ScanTable, tgt: ScanTable, *, n_pairs: Optional[int] = None, stream=None) -> torch.Tensor:
    """Rigid least-squares fit of matched rows, batched: ``best_fit_transform(A, B)``
    (icp.py:5-26) for every pair; returns poses [B,6] (R row-major, t)."""
    pr = _problem(src, tgt, "rowwise", None, None, 0)
    b = min(src.rows, tgt.rows) if n_pairs is None else int(n_pairs)
    _check_pairs(src, tgt, "rowwise", None, None, b, False)
    pose = torch.empty((b, 6), dtype=torch.float64, device=src.points.device)
    with torch.cuda.device(src.points.device):
        rc = _cabi.lib().b200icp_best_fit_batch(C.byref(pr), b, _ptr(pose), _stream_ptr(stream))
    _cabi.check(rc, "b200icp_best_fit_batch")
    return pose


POLAR_FILTERS = {
    # name: (min_dist, max_dist, min_quality, arc_lo, arc_hi, use_arc, y_sign)
    "process": (1000.0, 9000.0, 10.0, 135.0, 225.0, 1, -1),        # duc/ICP_LIDAR/process.py:45-49 (canonical)
    "slam_offline": (0.0, 10000.0, 13.0, 135.0, 225.0, 1, -1),      # duc/ICP_LIDAR/slam_offline.py:68-72
    "realtime_2": (0.0, 5000.0, 5.0, 135.0, 225.0, 0, -1),          # duc/code python/realtime_2.py:159-163
    "realtime_1": (0.0, 5000.0, 5.0, 135.0, 225.0, 0, 1),           # duc/code python/realtime_1.py:164-167, b.py:173-177
}


def polar_to_cartesian(raw: torch.Tensor, raw_len: Optional[torch.Tensor] = None,
                       out_pitch: Optional[int] = None, stream=None, filter="process") -> ScanTable:
    """Device scan preparation (process.py:38-52): raw [S, pitch, 3] float64 rows of
    (quality, angle_deg, distance_mm) -> filtered Cartesian ScanTable (float64).  ``filter``: the name
    of one of the reference's copies of the function (POLAR_FILTERS) or a 7-tuple
    (min_dist, max_dist, min_quality, arc_lo, arc_hi, use_arc, y_sign)."""
    if raw.dim() != 3 or raw.shape[2] != 3 or raw.dtype != torch.float64:
        raise ValueError("raw must be float64 [scans, pitch, 3]")
    _require_cuda(raw, "raw")
    s, pitch = int(raw.shape[0]), int(raw.shape[1])
    out_pitch = pitch if out_pitch is None else int(out_pitch)
    xy = torch.empty((s, out_pitch, 2), dtype=torch.float64, device=raw.device)
    lens = torch.empty(s, dtype=torch.int32, device=raw.device)
    with torch.cuda.device(raw.device):
        fv = POLAR_FILTERS[filter] if isinstance(filter, str) else tuple(filter)
        pf = _cabi.PolarFilter(float(fv[0]), float(fv[1]), float(fv[2]), float(fv[3]), float(fv[4]), int(fv[5]), int(fv[6]))
        rc = _cabi.lib().b200icp_polar_to_cartesian(_ptr(raw), _ptr(raw_len), s, pitch, C.byref(pf), _ptr(xy),
                                                    _ptr(lens), out_pitch, _stream_ptr(stream))
    _cabi.check(rc, "b200icp_polar_to_cartesian")
    return ScanTable(xy, lens)


def ffma_probe(inner_iters: int = 4096, repeats: int = 5, device="cuda") -> float:
    """Measured FP32 FFMA throughput in TFLOP/s (roofline denominator of the NN phase)."""
    sink = torch.zeros(4, dtype=torch.float32, device=device)
    flop = C.c_int64(0)
    best = 0.0
    with torch.cuda.device(sink.device):
        for _ in range(repeats + 1):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rc = _cabi.lib().b200icp_ffma_probe(_ptr(sink), inner_iters, C.byref(flop), _stream_ptr(None))
            e1.record()
            _cabi.check(rc, "b200icp_ffma_probe")
            e1.synchronize()
            ms = e0.elapsed_time(e1)
            best = max(best, flop.value / (ms * 1e-3) / 1e12)
    return best


class HostPipeline:
    """End-to-end batched alignment from HOST buffers: the call a user with NumPy-side scans
    makes.  Pinned host tables are streamed to the device in chunks (sizes: ``chunk_schedule``) on a
    copy stream while the previous chunk's ICP kernel runs, and each chunk's poses / errors / iteration counts
    are copied back to pinned host memory, so host<->device traffic overlaps the compute.
    Consecutive chunks run on alternating compute streams (one per staging buffer, three by default):
    the next chunk's CTAs fill the SMs that the tail wave of the current chunk leaves idle.

    Device staging buffers and pinned result buffers are allocated once and reused.

    ``graph=True``: a run (~16 chunks, ~100 enqueue calls from Python) is captured once per (host
    buffers, arguments) as a CUDA graph -- on the second call with the same pinned tensors, after an
    eager first call -- and replayed afterwards: one launch per run, the same kernels, copies and
    dependencies, the same bits.  Off by default: on the benchmark the host keeps ahead of the GPU
    either way (9.087 vs 9.088 ms per run); it pays when the host thread is busy with other work.
    """

    def __init__(self, n_pairs: int, src_pitch: int, tgt_pitch: int, dtype=torch.float32,
                 chunks: int = 8, device="cuda", graph: bool = False, buffers: int = 3):
        self.n_pairs, self.src_pitch, self.tgt_pitch = int(n_pairs), int(src_pitch), int(tgt_pitch)
        self.device = torch.device(device)
        self.use_graph = bool(graph)
        # Staging buffers = compute streams.  The copy of chunk i may start once the kernel of chunk
        # i - buffers has ended.  With two buffers it ends only ~0.25 ms before the kernel of chunk i - 1
        # does (copy 0.86 ms, kernel 1.11 ms per 8,192 pairs), which is the length of that kernel's
        # tail wave: the next kernel arrived too late to fill it, and a run cost the sum of the
        # ISOLATED chunk times (9.8 ms) instead of the work (8.9 ms).  Three buffers give the slack.
        self.nbuf = max(2, int(buffers))
        self._graphs, self._seen, self._graph_launches = {}, set(), 0
        sizes = self.chunk_schedule(self.n_pairs, chunks)
        self.chunk = max(sizes)
        self.bounds = [0]
        for sz in sizes:
            self.bounds.append(self.bounds[-1] + sz)
        self.dtype = dtype
        c = self.chunk
        mk = lambda *shape, dt=dtype: torch.empty(shape, dtype=dt, device=self.device)
        self.bufs = [dict(src=mk(c, src_pitch, 2), tgt=mk(c, tgt_pitch, 2),
                          slen=mk(c, dt=torch.int32), tlen=mk(c, dt=torch.int32),
                          out=alloc_outputs(c, src_pitch, self.device)) for _ in range(self.nbuf)]
        self.copy_stream = torch.cuda.Stream(device=self.device)
        self.out_stream = torch.cuda.Stream(device=self.device)
        self.compute_streams = [torch.cuda.Stream(device=self.device) for _ in range(self.nbuf)]
        # one fused kernel for every chunk, chosen on the size of the whole batch: results must not
        # depend on how the batch is cut (the two kernels agree to ~1e-12, not bit for bit)
        self.kernel = "warp" if self.n_pairs > _AUTO_CTA_PAIRS else "cta"
        pin = lambda *shape, dt: torch.empty(shape, dtype=dt, pin_memory=True)
        from . import hostmem
        with hostmem.near_gpu(self.device.index if self.device.index is not None else torch.cuda.current_device()):
            self.h_pose = pin(self.n_pairs, 6, dt=torch.float64)       # result buffers on the GPU's NUMA node
            self.h_error = pin(self.n_pairs, dt=torch.float64)
            self.h_iters = pin(self.n_pairs, dt=torch.int32)
        self.launches = 0
        self.done_event = None

    @staticmethod
    def chunk_schedule(n_pairs: int, chunks: int = 8, growth: float = 1.25):
        """Chunk sizes of one run.  ``chunks`` sets the LARGEST chunk (n_pairs / chunks).  Two parts of
        the pipeline cannot be hidden: the first host-to-device copy (nothing to compute yet) and the
        last kernel (nothing left to copy).  So the sizes ramp up geometrically from 1/8 of the largest
        chunk -- a copy must end before the kernel ahead of it does, which holds while the chunks grow
        by no more than the kernel / copy time ratio (1.3 on the headline workload) -- and the run ends
        with shrinking chunks (1/2 and 1/4 of the
        largest), which is what a copy-bound run (several GPUs sharing the host's memory bandwidth)
        exposes after its last copy."""
        n_pairs, chunks = int(n_pairs), max(1, int(chunks))
        if chunks == 1:
            return [n_pairs]
        big = max(1, -(-n_pairs // chunks))
        tail = [t for t in (big // 2, big // 4) if t >= 1]
        avail = n_pairs - sum(tail)
        if avail <= 0:
            tail, avail = [], n_pairs
        head, sz = [], max(1.0, big / 8.0)
        while int(sz) < big and sum(head) + int(sz) <= avail:
            head.append(int(sz))
            sz *= growth
        rest = avail - sum(head)
        body = [big] * (rest // big)
        if rest % big:                    # the remainder joins the shrinking end of the run
            tail = sorted(tail + [rest % big], reverse=True)
        return head + body + tail

    def bytes_per_run(self, ragged: bool):
        elt = 4 if self.dtype == torch.float32 else 8
        h2d = self.n_pairs * (self.src_pitch + self.tgt_pitch) * 2 * elt + (8 * self.n_pairs if ragged else 0)
        d2h = self.n_pairs * (6 * 8 + 8 + 4)
        return h2d, d2h

    def _check_host(self, t, name, shape, dtype):
        if t.is_cuda or tuple(t.shape) != shape or t.dtype != dtype or not t.is_contiguous():
            raise ValueError(f"{name} must be a contiguous host tensor of shape {shape}, dtype {dtype}")
        if not t.is_pinned():
            raise ValueError(f"{name} must live in pinned host memory (tensor.pin_memory()): the copies are asynchronous")

    def run(self, h_src: torch.Tensor, h_tgt: torch.Tensor, h_src_len=None, h_tgt_len=None, *,
            max_iterations: int = 20, tolerance: float = 1e-5, max_corr_dist=None):
        """h_src [B,src_pitch,2], h_tgt [B,tgt_pitch,2] pinned host tensors (row-wise pairs);
        h_src_len / h_tgt_len: both int32 [B] pinned host tensors, or both None (all rows full).
        Returns pinned host tensors (pose_total [B,6], error [B], iterations [B]); they are valid
        once ``self.done_event`` (recorded on the caller's current stream, which has been made to
        wait for every copy of this run) has completed, or after a device synchronize.  Calls may
        be issued back to back without synchronising: a run starts its copies only after the
        previous run on the caller's stream has drained."""
        if (h_src_len is None) != (h_tgt_len is None):
            raise ValueError("pass both h_src_len and h_tgt_len, or neither")
        self._check_host(h_src, "h_src", (self.n_pairs, self.src_pitch, 2), self.dtype)
        self._check_host(h_tgt, "h_tgt", (self.n_pairs, self.tgt_pitch, 2), self.dtype)
        ragged = h_src_len is not None
        if ragged:
            self._check_host(h_src_len, "h_src_len", (self.n_pairs,), torch.int32)
            self._check_host(h_tgt_len, "h_tgt_len", (self.n_pairs,), torch.int32)
        key = (h_src.data_ptr(), h_tgt.data_ptr(), h_src_len.data_ptr() if ragged else 0,
               h_tgt_len.data_ptr() if ragged else 0, int(max_iterations), float(tolerance),
               None if max_corr_dist is None else float(max_corr_dist))
        args = (h_src, h_tgt, h_src_len, h_tgt_len, ragged, max_iterations, tolerance, max_corr_dist)
        g = self._graphs.get(key) if self.use_graph else None
        if g is None and self.use_graph and key in self._seen:
            # second run on these buffers: capture (the first one ran eagerly: lazy one-time set-up of
            # the kernels is done).  The captured graph holds the tensors' addresses, not the tensors.
            g = torch.cuda.CUDAGraph()
            with torch.cuda.device(self.device), torch.cuda.graph(g):
                self._enqueue(*args)
            self._graphs[key] = g
            self._graph_launches = self.launches
        main = torch.cuda.current_stream(self.device)
        if g is not None:
            with torch.cuda.device(self.device):
                g.replay()
            self.launches = self._graph_launches
        else:
            if self.use_graph:
                if len(self._seen) > 64:              # callers that never reuse their buffers: stop tracking
                    self._seen.clear()
                self._seen.add(key)
            self._enqueue(*args)
        self.done_event = torch.cuda.Event()
        self.done_event.record(main)
        return self.h_pose, self.h_error, self.h_iters

    def _enqueue(self, h_src, h_tgt, h_src_len, h_tgt_len, ragged, max_iterations, tolerance, max_corr_dist):
        """One run's copies and kernels, enqueued on the side streams (forked from and joined back to the
        current stream, so the whole of it can be captured in a CUDA graph)."""
        main = torch.cuda.current_stream(self.device)
        # the previous run() ended with `main` waiting for all of its copies and kernels; ordering
        # the side streams after `main` keeps this run's first copies out of staging buffers that
        # the previous run's kernels may still be reading
        self.copy_stream.wait_stream(main)
        self.out_stream.wait_stream(main)
        nb_ = self.nbuf
        ready = [None] * nb_       # compute-done events per staging buffer
        drained = [None] * nb_     # results-copied events per staging buffer
        self.launches = 0
        for ci in range(len(self.bounds) - 1):
            b0, b1 = self.bounds[ci], self.bounds[ci + 1]
            nb = b1 - b0
            bi = ci % nb_
            buf = self.bufs[bi]
            with torch.cuda.stream(self.copy_stream):
                if ready[bi] is not None:
                    self.copy_stream.wait_event(ready[bi])          # kernel finished reading it
                buf["src"][:nb].copy_(h_src[b0:b1], non_blocking=True)
                buf["tgt"][:nb].copy_(h_tgt[b0:b1], non_blocking=True)
                if ragged:
                    buf["slen"][:nb].copy_(h_src_len[b0:b1], non_blocking=True)
                    buf["tlen"][:nb].copy_(h_tgt_len[b0:b1], non_blocking=True)
                copied = torch.cuda.Event()
                copied.record(self.copy_stream)
            cs = self.compute_streams[bi]
            if ci < nb_:
                cs.wait_stream(main)                                # work queued by the caller before run()
            cs.wait_event(copied)
            if drained[bi] is not None:
                cs.wait_event(drained[bi])                          # previous results left the buffer
            s = ScanTable(buf["src"][:nb], buf["slen"][:nb] if ragged else None)
            t = ScanTable(buf["tgt"][:nb], buf["tlen"][:nb] if ragged else None)
            with torch.cuda.stream(cs):
                align_pairs(s, t, n_pairs=nb, max_iterations=max_iterations, tolerance=tolerance,
                            max_corr_dist=max_corr_dist, kernel=self.kernel, out=buf["out"], stream=cs)
            self.launches += 1
            done = torch.cuda.Event()
            done.record(cs)
            ready[bi] = done
            with torch.cuda.stream(self.out_stream):
                self.out_stream.wait_event(done)
                self.h_pose[b0:b1].copy_(buf["out"].pose_total[:nb], non_blocking=True)
                self.h_error[b0:b1].copy_(buf["out"].error[:nb], non_blocking=True)
                self.h_iters[b0:b1].copy_(buf["out"].iterations[:nb], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(self.out_stream)
                drained[bi] = ev
        for ev in drained:
            if ev is not None:
                main.wait_event(ev)
        for cs in self.compute_streams:
            main.wait_stream(cs)
        main.wait_stream(self.copy_stream)
        main.wait_stream(self.out_stream)
