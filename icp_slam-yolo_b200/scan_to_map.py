"""Scan-to-map ICP with the map sharded across GPUs (one process per GPU).

Call shape of the reference's SLAM step -- register the current scan against the (local) map
(duc/ICP_LIDAR/mainn.py:297-318, slam_offline.py:366-392) -- with the point-to-point loop of
labels_segmentation/icp.py:28-53.  The map is split into contiguous index ranges, one per
rank.  Once per map the bounding circles of every 1,024-point chunk of every rank are gathered
(32 bytes per chunk), so each rank can bound a scan point's nearest-neighbour distance over the
whole map on its own.  Per iteration two kernels run on every rank: the search finds the exact
nearest point of ITS shard for every scan point that can have its neighbour there (exact scan
of the few chunks within the bound) and stores the 32-byte record straight into every rank's
inbox over NVLink; the update waits for all ranks' flags, picks the global winner per point and
solves the pose -- on the same records everywhere, so poses, errors and the stop decision are
bit-identical on every rank without a second exchange.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional

import numpy as np
import torch

from . import _cabi
from .registration import _DTYPES, _ptr, _require_cuda, _stream_ptr, _workspace

RECORD_BYTES = 32
STATE_BYTES = 136


def _lib():
    return _cabi.lib()


class MapShard:
    """One rank's contiguous slice of the map and its circle tables.

    ``spatial_sort``: the culling works on runs of 1,024 consecutive map points, so it needs an
    order in which neighbours in memory are neighbours in space.  True builds a Morton-sorted copy
    of the shard once (indices and tie-breaking still refer to the original order); False scans the
    map as given (accumulated LiDAR scans are ordered along the walls already); "auto" sorts when
    the chunks of the given order are spread out (mean chunk radius above 5 % of the shard's extent)."""

    def __init__(self, points: torch.Tensor, global_offset: int = 0, stream=None, spatial_sort="auto"):
        if points.dim() != 2 or points.shape[1] != 2 or points.dtype not in _DTYPES:
            raise ValueError("map points must be [m, 2] float32/float64")
        _require_cuda(points, "map points")
        if points.shape[0] < 1:
            raise ValueError("empty map shard")
        self.points = points
        self.m = int(points.shape[0])
        self.global_offset = int(global_offset)
        self.n_chunks = int(_lib().b200icp_s2m_padded_chunks(self.m))      # padded to a multiple of 32
        dev = points.device
        self.chunk_circle = torch.empty((self.n_chunks, 4), dtype=torch.float64, device=dev)
        self.super_circle = torch.empty((self.n_chunks // 32, 4), dtype=torch.float64, device=dev)
        self.desc = _cabi.S2MShard()
        self.desc.points = points.data_ptr()
        self.desc.m = self.m
        self.desc.global_offset = self.global_offset
        self.desc.dtype = _DTYPES[points.dtype]
        self.desc.chunk_circle = self.chunk_circle.data_ptr()
        self.desc.super_circle = self.super_circle.data_ptr()
        self.sorted_points = self.order = None
        if spatial_sort is not True:               # circles of the given order (also the test of "auto")
            self._prepare(stream)
        if spatial_sort == "auto" and self.m >= 4 * 1024:
            valid = self.chunk_circle[:, 2] >= 0
            extent = float((points.max(dim=0).values - points.min(dim=0).values).max())
            spatial_sort = bool(float(self.chunk_circle[valid, 2].mean()) > 0.05 * extent)
        if spatial_sort is True and self.m < 2 ** 31:
            self.sorted_points = torch.empty_like(points)
            self.order = torch.empty(self.m, dtype=torch.int32, device=dev)
            self.desc.sorted_points, self.desc.order = self.sorted_points.data_ptr(), self.order.data_ptr()
            self._prepare(stream)

    def _prepare(self, stream):
        ws, nbytes = (None, 0) if self.order is None else \
            _workspace(_lib().b200icp_s2m_prepare_workspace_bytes, self.m, device=self.points.device)
        with torch.cuda.device(self.points.device):
            rc = _lib().b200icp_s2m_prepare_map(C.byref(self.desc), _ptr(ws), nbytes, _stream_ptr(stream))
        _cabi.check(rc, "b200icp_s2m_prepare_map")
        if ws is not None:
            torch.cuda.current_stream().synchronize()          # the workspace is freed on return


class CircleTables:
    """The circle tables of the whole map (every rank's, concatenated in rank order) plus where
    one rank's chunks sit in them."""

    def __init__(self, chunk_circle: torch.Tensor, super_circle: torch.Tensor, first_local: int, n_local: int):
        self.chunk_circle, self.super_circle = chunk_circle.contiguous(), super_circle.contiguous()
        self.desc = _cabi.S2MTables()
        self.desc.chunk_circle = self.chunk_circle.data_ptr()
        self.desc.super_circle = self.super_circle.data_ptr()
        self.desc.n_chunks_total = int(self.chunk_circle.shape[0])
        self.desc.first_local_chunk = int(first_local)
        self.desc.n_local_chunks = int(n_local)

    @staticmethod
    def local(shard: MapShard) -> "CircleTables":
        return CircleTables(shard.chunk_circle, shard.super_circle, 0, shard.n_chunks)

    @staticmethod
    def gathered(shard: MapShard, group, world: int, rank: int) -> "CircleTables":
        """All-gather of the per-rank tables (once per map; the only use of the library collective)."""
        import torch.distributed as dist
        dev = shard.points.device
        counts = torch.zeros(world, dtype=torch.int64, device=dev)
        counts[rank] = shard.n_chunks
        dist.all_reduce(counts, group=group)
        counts = [int(c) for c in counts.cpu()]
        cap = max(counts)
        pad = torch.zeros((cap, 4), dtype=torch.float64, device=dev)
        pad[:, 2] = -1.0                                       # padding circles hold no points
        pad[:shard.n_chunks] = shard.chunk_circle
        everyone = torch.empty((world, cap, 4), dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(everyone.view(world * cap, 4), pad, group=group)
        spad = torch.zeros((cap // 32, 4), dtype=torch.float64, device=dev)
        spad[:, 2] = -1.0
        spad[:shard.n_chunks // 32] = shard.super_circle
        severyone = torch.empty((world, cap // 32, 4), dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(severyone.view(world * (cap // 32), 4), spad, group=group)
        chunks = torch.cat([everyone[r, :counts[r]] for r in range(world)])
        supers = torch.cat([severyone[r, :counts[r] // 32] for r in range(world)])
        return CircleTables(chunks, supers, sum(counts[:rank]), shard.n_chunks)

    @staticmethod
    def concatenated(shards) -> list:
        """Tables of several shards resident on ONE device (ScanToMapLocalShards)."""
        chunks = torch.cat([s.chunk_circle for s in shards])
        supers = torch.cat([s.super_circle for s in shards])
        out, first = [], 0
        for s in shards:
            out.append(CircleTables(chunks, supers, first, s.n_chunks))
            first += s.n_chunks
        return out


@dataclass
class ScanToMapResult:
    R: np.ndarray             # cumulative rotation (2,2)
    t: np.ndarray             # cumulative translation (2,)
    R_last: np.ndarray
    t_last: np.ndarray
    error: float              # lagged mean NN distance (icp.py:48)
    rmse: float
    inliers: int
    iterations: int
    indices: Optional[torch.Tensor]      # [n] int32 global map index of the last search
    src: torch.Tensor                    # [n,2] float64 transformed scan (device)


class PeerInboxes:
    """Peer-visible inboxes of all ranks (CUDA IPC) for the store-to-every-peer all-gather in the
    epilogue of b200icp_s2m_search.  Layout per rank: [2 slots][world][n] records, [2][world] int64
    flags, one int64 exchange counter.  NCCL is used once, to exchange the 64-byte IPC handles."""

    def __init__(self, n: int, world: int, rank: int, group, device):
        import torch.distributed as dist
        self.n, self.world, self.rank, self.device = n, world, rank, device
        lib = _lib()
        nbytes = lib.b200icp_s2m_inbox_bytes(n, world)
        if nbytes < 0:
            raise _cabi.B200IcpError("b200icp_s2m_inbox_bytes failed (world too large?)")
        ptr, handle = C.c_void_p(), C.create_string_buffer(64)
        with torch.cuda.device(device):
            _cabi.check(lib.b200icp_peer_alloc(nbytes, C.byref(ptr), handle), "b200icp_peer_alloc")
            mine = torch.frombuffer(bytearray(handle.raw), dtype=torch.uint8).to(device)
            everyone = torch.empty(world * 64, dtype=torch.uint8, device=device)
            dist.all_gather_into_tensor(everyone, mine, group=group)
            handles = everyone.cpu().numpy().reshape(world, 64)
            self.base = int(ptr.value)
            self.opened = []
            addrs = []
            for r in range(world):
                if r == rank:
                    addrs.append(self.base)
                    continue
                p = C.c_void_p()
                _cabi.check(lib.b200icp_peer_open(handles[r].tobytes(), C.byref(p)), "b200icp_peer_open")
                self.opened.append(int(p.value))
                addrs.append(int(p.value))
            self.peers = torch.tensor(addrs, dtype=torch.int64, device=device)
            torch.cuda.synchronize()
            dist.barrier(group=group)

    def close(self):
        import torch.distributed as dist
        lib = _lib()
        torch.cuda.synchronize()
        if dist.is_initialized():
            dist.barrier()
        for p in self.opened:
            lib.b200icp_peer_close(C.c_void_p(p))
        self.opened = []
        if self.base:
            lib.b200icp_peer_free(C.c_void_p(self.base))
            self.base = 0


class ScanToMap:
    """Reusable buffers for registering n-point scans against one shard (per rank).

    exchange = "peer" (default with several ranks): the search kernel stores its records into
    every rank's inbox over NVLink and raises a flag; the update kernel waits for the flags.  No
    library collective and no host synchronisation inside the loop.
    exchange = "nccl": records all-gathered with torch.distributed between the two kernels.
    ``graph=True`` captures the whole fixed-length loop of a ``run`` in a CUDA graph (peer or
    single-rank exchange only) and replays it for the same arguments."""

    def __init__(self, shard: MapShard, n_scan: int, group=None, want_indices: bool = False,
                 exchange: str = "peer", local_only: bool = False, graph: bool = False):
        import torch.distributed as dist
        self.shard, self.n = shard, int(n_scan)
        self.group = group
        self.world = (dist.get_world_size(group)
                      if (not local_only and dist.is_available() and dist.is_initialized()) else 1)
        self.rank = dist.get_rank(group) if self.world > 1 else 0
        if exchange not in ("nccl", "peer"):
            raise ValueError("exchange must be 'nccl' or 'peer'")
        self.exchange = exchange if self.world > 1 else "local"
        dev = shard.points.device
        self.dev = dev
        self.src64 = torch.empty((self.n, 2), dtype=torch.float64, device=dev)
        self.prev_nn = torch.empty((self.n, 2), dtype=torch.float64, device=dev)
        self.state = torch.zeros(STATE_BYTES // 8, dtype=torch.float64, device=dev)
        self.records = torch.empty((self.n, 4), dtype=torch.float64, device=dev)          # 32 B each
        self.records_all = (torch.empty((self.world, self.n, 4), dtype=torch.float64, device=dev)
                            if self.exchange == "nccl" else None)
        sb = _lib().b200icp_s2m_scratch_bytes(self.n)
        if sb < 0:
            raise _cabi.B200IcpError("b200icp_s2m_scratch_bytes failed")
        self.scratch = torch.zeros(sb, dtype=torch.uint8, device=dev)
        self.indices = torch.empty(self.n, dtype=torch.int32, device=dev) if want_indices else None
        self.tables = (CircleTables.gathered(shard, group, self.world, self.rank) if self.world > 1
                       else CircleTables.local(shard))
        self.peer = PeerInboxes(self.n, self.world, self.rank, group, dev) if self.exchange == "peer" else None
        self.launches = 0
        self.use_graph = bool(graph) and self.exchange != "nccl"
        self._graphs = {}
        self._ip = torch.zeros(6, dtype=torch.float64, device=dev)
        self._scan_f32 = torch.empty((self.n, 2), dtype=torch.float32, device=dev)
        self._scan_f64 = torch.empty((self.n, 2), dtype=torch.float64, device=dev)

    # ---- single steps -----------------------------------------------------------------------
    def init(self, scan: torch.Tensor, init_pose: Optional[torch.Tensor] = None, stream=None):
        rc = _lib().b200icp_s2m_init(_ptr(scan), _DTYPES[scan.dtype], self.n, _ptr(init_pose),
                                     _ptr(self.src64), _ptr(self.prev_nn), _ptr(self.state), _stream_ptr(stream))
        _cabi.check(rc, "b200icp_s2m_init")

    def search(self, stream=None, records: Optional[torch.Tensor] = None, tables: Optional[CircleTables] = None):
        """Exact nearest point of this shard for every scan point that can have its neighbour here
        (the others get "none" records).  With the peer exchange the records go to every rank's inbox."""
        tb = self.tables if tables is None else tables
        peers = self.peer.peers if self.peer is not None else None
        rec = self.records if records is None else records
        rc = _lib().b200icp_s2m_search(C.byref(self.shard.desc), C.byref(tb.desc), _ptr(self.src64),
                                       _ptr(self.prev_nn), self.n, _ptr(rec), _ptr(peers), self.world,
                                       self.rank, _ptr(self.state), _ptr(self.scratch), _stream_ptr(stream))
        _cabi.check(rc, "b200icp_s2m_search")
        self.launches += 1

    def update(self, max_iterations: int, tolerance: float, max_corr_dist=None, stream=None,
               records_all: Optional[torch.Tensor] = None, n_ranks: Optional[int] = None):
        if records_all is None:
            records_all = self.records_all if self.exchange == "nccl" else self.records
        inbox = C.c_void_p(self.peer.base) if self.peer is not None else None
        rc = _lib().b200icp_s2m_update(_ptr(records_all), inbox, self.world if n_ranks is None else int(n_ranks),
                                       _ptr(self.src64), _ptr(self.prev_nn), self.n, int(max_iterations),
                                       float(tolerance), 0.0 if max_corr_dist is None else float(max_corr_dist),
                                       _ptr(self.indices), _ptr(self.state), _ptr(self.scratch), _stream_ptr(stream))
        _cabi.check(rc, "b200icp_s2m_update")
        self.launches += 1

    def finish(self, stream=None):
        rc = _lib().b200icp_s2m_finish(_ptr(self.src64), self.n, _ptr(self.state), _ptr(self.scratch),
                                       _stream_ptr(stream))
        _cabi.check(rc, "b200icp_s2m_finish")
        self.launches += 1

    # ---- the loop ------------------------------------------------------------------------------
    def _loop(self, scan, ip, max_iterations, tolerance, max_corr_dist, events=None):
        import torch.distributed as dist

        def mark():
            if events is not None:
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                events.append(e)

        self.init(scan, ip)
        self.launches += 1
        for _ in range(int(max_iterations)):
            mark()
            self.search()
            mark()
            if self.exchange == "nccl":
                dist.all_gather_into_tensor(self.records_all.view(self.world * self.n, 4), self.records,
                                            group=self.group)
            self.update(max_iterations, tolerance, max_corr_dist)
        mark()
        self.finish()

    def run(self, scan: torch.Tensor, *, max_iterations: int = 20, tolerance: float = 1e-5,
            init_pose=None, max_corr_dist: Optional[float] = None, sync: bool = True, events=None):
        """Full loop.  No host synchronisation inside; kernels no-op once converged.  ``events``: a
        list that receives CUDA events recorded before every search, before every update (the peer
        wait is part of the update) and after the last update (profiling; not with ``graph``)."""
        if scan.dim() != 2 or scan.shape != (self.n, 2) or scan.dtype not in _DTYPES:
            raise ValueError(f"scan must be [{self.n}, 2] float32/float64")
        _require_cuda(scan, "scan")
        ip = None
        if init_pose is not None:
            self._ip.copy_(torch.as_tensor(np.asarray(init_pose, dtype=np.float64).reshape(6)), non_blocking=False)
            ip = self._ip
        self.launches = 0
        with torch.cuda.device(self.dev):
            if not self.use_graph or events is not None:
                self._loop(scan, ip, max_iterations, tolerance, max_corr_dist, events)
            else:
                staged = self._scan_f32 if scan.dtype == torch.float32 else self._scan_f64
                staged.copy_(scan)
                key = (scan.dtype, int(max_iterations), float(tolerance), max_corr_dist, ip is not None)
                g = self._graphs.get(key)
                if g is None:
                    torch.cuda.synchronize()
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):
                        self._loop(staged, ip, max_iterations, tolerance, max_corr_dist)
                    self._graphs[key] = g
                    self._graph_launches = self.launches
                g.replay()
                self.launches = self._graph_launches
        return self.result() if sync else None

    def result(self) -> ScanToMapResult:
        st = self.state.cpu().numpy()
        ints = st[15:17].view(np.int32)           # iterations, inliers, done, applied
        if int(ints[2]) == 2:
            self.scratch.zero_()
            raise _cabi.B200IcpError(
                "scan-to-map: a peer's records did not arrive within 2 s (rank missing, or the ranks issued "
                "different call sequences); the state of this alignment is invalid")
        mean_d2 = st[13]
        return ScanToMapResult(
            R=st[0:4].reshape(2, 2).copy(), t=st[4:6].copy(),
            R_last=st[6:10].reshape(2, 2).copy(), t_last=st[10:12].copy(),
            error=float(st[12]), rmse=float(np.sqrt(mean_d2)) if np.isfinite(mean_d2) else float("inf"),
            inliers=int(ints[1]), iterations=int(ints[0]), indices=self.indices, src=self.src64)


def scan_to_map_icp(scan: torch.Tensor, shard: MapShard, max_iterations: int = 20,
                    tolerance: float = 1e-5, *, init_pose=None, max_corr_dist=None, group=None,
                    want_indices: bool = False) -> ScanToMapResult:
    """One-shot convenience wrapper around :class:`ScanToMap`."""
    s2m = ScanToMap(shard, int(scan.shape[0]), group=group, want_indices=want_indices)
    return s2m.run(scan, max_iterations=max_iterations, tolerance=tolerance, init_pose=init_pose,
                   max_corr_dist=max_corr_dist)


class ScanToMapLocalShards:
    """The multi-rank protocol with every shard resident on ONE GPU: each shard is searched in
    turn against the concatenated circle tables, the records are stacked where the all-gather
    would put them, and the same update kernel runs.  Used to split a map that is built
    incrementally into pieces, and by the tests to check the sharded path (global bounds, shard
    offsets, "none" records, record merge, lowest-global-index ties) without several GPUs.
    ``step()`` runs one iteration so callers can inspect per-iteration state."""

    def __init__(self, shards, n_scan: int, want_indices: bool = True):
        self.workers = [ScanToMap(s, n_scan, local_only=True) for s in shards]
        self.tables = CircleTables.concatenated(shards)
        self.n, self.dev = int(n_scan), shards[0].points.device
        self.w0 = self.workers[0]
        self.src64, self.state = self.w0.src64, self.w0.state
        self.records_all = torch.empty((len(shards), self.n, 4), dtype=torch.float64, device=self.dev)
        self.indices = torch.empty(self.n, dtype=torch.int32, device=self.dev) if want_indices else None
        self.w0.indices = self.indices
        for w in self.workers[1:]:               # one scan state, one scratch, one neighbour memory
            w.src64, w.prev_nn, w.state, w.scratch = self.w0.src64, self.w0.prev_nn, self.w0.state, self.w0.scratch

    def init(self, scan: torch.Tensor, init_pose=None):
        ip = None
        if init_pose is not None:
            ip = torch.as_tensor(np.asarray(init_pose, dtype=np.float64).reshape(6)).to(self.dev)
        self.w0.init(scan, ip)

    def step(self, max_iterations: int, tolerance: float, max_corr_dist=None):
        for g, w in enumerate(self.workers):
            w.search(records=self.records_all[g], tables=self.tables[g])
        self.w0.update(max_iterations, tolerance, max_corr_dist, records_all=self.records_all,
                       n_ranks=len(self.workers))

    def run(self, scan, *, max_iterations=20, tolerance=1e-5, init_pose=None, max_corr_dist=None):
        self.init(scan, init_pose)
        for _ in range(int(max_iterations)):
            self.step(max_iterations, tolerance, max_corr_dist)
        return self.result()

    def result(self) -> ScanToMapResult:
        self.w0.finish()
        return self.w0.result()
