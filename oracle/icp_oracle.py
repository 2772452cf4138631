"""NumPy/SciPy restatement of the reference's 2D point-to-point ICP path.

TEST INFRASTRUCTURE (see ``oracle/__init__.py``) -- never imported by the product.

Reference anchors (relative to /root/reference):
  * ``labels_segmentation/icp.py:5-26``   best_fit_transform  -> :func:`best_fit_transform`
  * ``labels_segmentation/icp.py:28-53``  icp                 -> :func:`icp_reference_form`
  * ``duc/ICP_LIDAR/process.py:38-52``    polar_to_cartesian_3d -> :func:`polar_to_cartesian`
  * ``duc/ICP_LIDAR/process.py:9-36``     load_and_prepare_scan -> :func:`load_and_prepare_scan`

:func:`icp_extended` is the same loop with the bookkeeping the new call surface
needs (per-iteration correspondence history, cumulative pose, lagged error,
iteration count, optional initial pose and correspondence gate).  With
``init_pose=None`` and ``max_corr_dist=None`` it performs the same floating
point operations in the same order as the reference, so ``src`` is bitwise equal.
"""
from __future__ import annotations

import math
import os
from dataclasses import dataclass, field

import numpy as np
from scipy.spatial import KDTree


# ----------------------------------------------------------------------------
# best_fit_transform  (icp.py:5-26)
# ----------------------------------------------------------------------------
def best_fit_transform(P, Q):
    """Least-squares rigid (R, t) taking matched rows of P onto Q.

    icp.py:10-11 centroids, :13-14 centring, :16 H = PP^T QQ, :17 SVD,
    :18 R = V U^T, :21-23 reflection repair on the last row of Vt, :25 t.
    """
    cP = np.mean(P, axis=0)
    cQ = np.mean(Q, axis=0)
    H = (P - cP).T @ (Q - cQ)
    U, _, Vt = np.linalg.svd(H)
    R = Vt.T @ U.T
    if np.linalg.det(R) < 0:
        Vt[1, :] *= -1
        R = Vt.T @ U.T
    t = cQ.T - R @ cP.T
    return R, t


def best_fit_transform_closed_form(P, Q):
    """Closed-form 2D Kabsch: theta = atan2(H01 - H10, H00 + H11).

    Equals the proper-rotation SVD result of icp.py:17-23 to ~1e-16 rad
    (SURVEY.md §8 a5); this is the form the CUDA kernel evaluates, restated
    here so tests can separate "SVD vs closed form" from "CPU vs GPU".
    """
    cP = np.mean(P, axis=0)
    cQ = np.mean(Q, axis=0)
    H = (P - cP).T @ (Q - cQ)
    num = H[0, 1] - H[1, 0]
    den = H[0, 0] + H[1, 1]
    hyp = math.hypot(num, den)
    if hyp == 0.0:
        c, s = 1.0, 0.0
    else:
        c, s = den / hyp, num / hyp
    R = np.array([[c, -s], [s, c]])
    t = cQ - R @ cP
    return R, t


# ----------------------------------------------------------------------------
# icp  (icp.py:28-53), reference form: returns (src, R_last, t_last)
# ----------------------------------------------------------------------------
def icp_reference_form(A, B, max_iterations=20, tolerance=1e-5):
    """Same signature and return as the reference's ``icp`` (icp.py:28)."""
    res = icp_extended(A, B, max_iterations, tolerance)
    return res.src, res.R_last, res.t_last


@dataclass
class IcpResult:
    src: np.ndarray            # (N,2) transformed source            icp.py:45
    R_last: np.ndarray         # last incremental rotation           icp.py:42,53 (quirk Q1)
    t_last: np.ndarray
    R_tot: np.ndarray          # cumulative pose: src = R_tot A + t_tot
    t_tot: np.ndarray
    error: float               # lagged mean NN distance             icp.py:48 (quirk Q2)
    iterations: int            # i+1 at break else max_iterations    (quirk Q4)
    rmse: float = float("nan")     # sqrt(mean d^2) over inliers, last search
    fitness: float = float("nan")  # inliers / N, last search
    indices: list = field(default_factory=list)   # per-iteration (N,) intp
    errors: list = field(default_factory=list)    # per-iteration mean distance
    inlier_masks: list = field(default_factory=list)


def nn_kdtree(src, tgt):
    """icp.py:37-38: tree rebuilt per call, k=1 Euclidean query."""
    d, i = KDTree(tgt).query(src)
    return d, i


def nn_bruteforce(src, tgt, chunk=2048):
    """float64 argmin_j |src_i - tgt_j|^2, lowest j on exact ties.

    Stand-in for the KD-tree when M is huge; identical to ``KDTree.query`` on
    all 1.86 M real queries of Scan_data_1 (SURVEY.md §7.1-1c).
    """
    src = np.asarray(src, dtype=np.float64)
    tgt = np.asarray(tgt, dtype=np.float64)
    n = src.shape[0]
    idx = np.empty(n, dtype=np.intp)
    d2 = np.empty(n, dtype=np.float64)
    for s in range(0, n, chunk):
        e = min(n, s + chunk)
        dx = src[s:e, None, 0] - tgt[None, :, 0]
        dy = src[s:e, None, 1] - tgt[None, :, 1]
        dd = dx * dx + dy * dy
        k = np.argmin(dd, axis=1)
        idx[s:e] = k
        d2[s:e] = dd[np.arange(e - s), k]
    return np.sqrt(d2), idx


def icp_extended(A, B, max_iterations=20, tolerance=1e-5, *, init_pose=None,
                 max_corr_dist=None, nn="kdtree", solver="svd", keep_history=True):
    """The reference loop (icp.py:32-53) plus bookkeeping.

    init_pose      (R0 (2,2), t0 (2,)): pre-transforms A and is left-composed into
                   the cumulative pose (Open3D ``trans_init`` convention,
                   gicp_lidar.py:32).  PARITY-UNPINNED extension (Q7).
    max_corr_dist  finite => only pairs with distance < max_corr_dist enter the
                   fit and the error mean (Open3D ``max_correspondence_distance``
                   shape).  PARITY-UNPINNED extension (Q5).  If no pair survives
                   the loop stops: that search is not counted, error = +inf.
    """
    A = np.asarray(A, dtype=np.float64)
    B = np.asarray(B, dtype=np.float64)
    search = nn_kdtree if nn == "kdtree" else nn_bruteforce
    fit = best_fit_transform if solver == "svd" else best_fit_transform_closed_form

    src = np.copy(A)                                   # icp.py:32
    R_tot = np.eye(2)
    t_tot = np.zeros(2)
    if init_pose is not None:
        R0 = np.asarray(init_pose[0], dtype=np.float64)
        t0 = np.asarray(init_pose[1], dtype=np.float64)
        src = (R0 @ src.T).T + t0
        R_tot, t_tot = R0.copy(), t0.copy()
    prev_error = 0                                     # icp.py:33 (quirk Q3)
    res = IcpResult(src, np.eye(2), np.zeros(2), R_tot, t_tot, float("inf"), 0)

    for i in range(max_iterations):                    # icp.py:35
        dist, idx = search(src, B)                     # icp.py:37-38
        if max_corr_dist is None:
            keep = None
            P, Q, dsel = src, B[idx], dist             # icp.py:39
        else:
            keep = dist < max_corr_dist
            if not np.any(keep):
                res.error = float("inf")
                res.fitness = 0.0
                break
            P, Q, dsel = src[keep], B[idx[keep]], dist[keep]
        R, t = fit(P, Q)                               # icp.py:42
        src = (R @ src.T).T + t                        # icp.py:45
        R_tot = R @ R_tot
        t_tot = R @ t_tot + t
        mean_error = np.mean(dsel)                     # icp.py:48
        res.R_last, res.t_last = R, t
        res.error = float(mean_error)
        res.rmse = float(np.sqrt(np.mean(dsel * dsel)))
        res.fitness = float(len(dsel)) / float(len(src))
        res.iterations = i + 1
        if keep_history:
            res.indices.append(np.asarray(idx))
            res.errors.append(float(mean_error))
            res.inlier_masks.append(keep)
        if np.abs(prev_error - mean_error) < tolerance:   # icp.py:49-50
            break
        prev_error = mean_error                        # icp.py:51

    res.src, res.R_tot, res.t_tot = src, R_tot, t_tot
    return res


# ----------------------------------------------------------------------------
# scan preparation  (process.py:9-52)
# ----------------------------------------------------------------------------
def polar_to_cartesian_loop(scan):
    """Row loop as in process.py:38-52 (math.radians/cos/sin per kept row)."""
    if scan is None or len(scan) == 0:
        return np.array([])
    out = []
    for quality, angle, distance in scan:
        front = (angle <= 135) or (angle >= 225)                       # :45
        if distance > 1000 and distance < 9000 and quality > 10 and front:   # :46
            a = math.radians(angle)
            out.append([distance * math.cos(a), -distance * math.sin(a), 0.0])  # :47-50
    return np.array(out)


def polar_keep_mask(scan):
    """Row filter of process.py:45-46."""
    q, a, d = scan[:, 0], scan[:, 1], scan[:, 2]
    return ((a <= 135) | (a >= 225)) & (d > 1000) & (d < 9000) & (q > 10)


def polar_to_cartesian(scan):
    """Vectorised process.py:38-52; bitwise equal to the row loop on all
    1,831 Scan_data_1 files (checked in tests when the reference is present)."""
    scan = np.asarray(scan, dtype=np.float64)
    if scan.size == 0:
        return np.zeros((0, 3))
    rows = scan[polar_keep_mask(scan)]
    rad = np.radians(rows[:, 1])      # == math.radians: x * (pi/180) in C doubles
    x = rows[:, 2] * np.cos(rad)
    y = -rows[:, 2] * np.sin(rad)
    return np.stack([x, y, np.zeros_like(x)], axis=1)


# The reference's other copies of polar_to_cartesian_3d differ from process.py:45-49 only in
# constants: (min_dist, max_dist, min_quality, use_arc, y_sign)
POLAR_VARIANTS = {
    "process": (1000, 9000, 10, True, -1),          # duc/ICP_LIDAR/process.py:45-49 (canonical)
    "slam_offline": (0, 10000, 13, True, -1),       # duc/ICP_LIDAR/slam_offline.py:68-72
    "realtime_2": (0, 5000, 5, False, -1),          # duc/code python/realtime_2.py:159-163
    "realtime_1": (0, 5000, 5, False, 1),           # duc/code python/realtime_1.py:164-167, b.py:173-177
}


def polar_to_cartesian_variant(scan, variant):
    """Row loop of the named copy of polar_to_cartesian_3d (same statements, its constants)."""
    lo, hi, qmin, use_arc, ysign = POLAR_VARIANTS[variant]
    out = []
    for quality, angle, distance in scan:
        front = (not use_arc) or (angle <= 135) or (angle >= 225)
        if distance > lo and distance < hi and quality > qmin and front:
            a = math.radians(angle)
            out.append([distance * math.cos(a), ysign * distance * math.sin(a), 0.0])
    return np.array(out) if out else np.zeros((0, 3))


def scan_path(directory, k):
    """Scan_data_1 mixes ``Scan_data_{k}.npy`` (k<=219) and ``scan_data_{k}.npy``
    (SURVEY.md §8 a1); resolve either spelling."""
    for stem in ("Scan_data_", "scan_data_", "scan_"):
        p = os.path.join(directory, f"{stem}{k}.npy")
        if os.path.exists(p):
            return p
    return None


def load_and_prepare_scan(path):
    """process.py:9-36: (N,3) polar rows -> Cartesian, (N,2) -> append z=0,
    anything else / missing file -> None."""
    if path is None or not os.path.exists(path):
        return None
    try:
        raw = np.load(path)
        if raw.ndim != 2 or raw.shape[1] not in (2, 3):
            return None
        raw = np.asarray(raw, dtype=np.float64)
        if raw.shape[1] == 3:
            return polar_to_cartesian(raw)
        return np.hstack((raw, np.zeros((raw.shape[0], 1))))
    except Exception:
        return None


# ----------------------------------------------------------------------------
# synthetic workloads (SURVEY.md §8d, configs 3-5).  Kept here so that the
# tests, the bench's CPU arm and the GPU arm all draw the *same* arrays.
# ----------------------------------------------------------------------------
def synth_room_pair(pair_index, n_points=360, dtype=np.float32):
    """One scan pair of config 3 (see :func:`synth_room_batch`): returns (src, tgt, theta, t)."""
    src, tgt, theta, t = synth_room_batch(pair_index, 1, n_points, dtype, with_truth=True)
    return src[0], tgt[0], float(theta[0]), t[0]


def synth_room_batch(first_pair, count, n_points=360, dtype=np.float32, with_truth=False):
    """Config 3 generator (SURVEY.md §8d): ``count`` scan pairs starting at ``first_pair``.

    Target = n_points beams at equal angular spacing on a star-convex room
    r(phi) = 3000 + sum_{k=1..4} a_k sin(k phi + psi_k) mm, a_k ~ U(0,600), psi_k ~ U(0,2pi),
    plus N(0, 5 mm) range noise (no exact ties).  Source = the same room sampled at
    phi + theta, expressed in a frame rotated by theta ~ U(-0.1,0.1) rad and shifted by
    t ~ U(-100,100)^2 mm, with independent noise.  Pair b draws from
    ``PCG64(1234 + first_pair + b)`` in a fixed order, so any batch split yields the same
    values.  Generated in float64, cast to ``dtype``.  All math is elementwise (no BLAS), so
    results do not depend on ``count``.
    """
    amp = np.empty((count, 4)); psi = np.empty((count, 4)); theta = np.empty(count)
    t = np.empty((count, 2)); nz_t = np.empty((count, n_points)); nz_s = np.empty((count, n_points))
    for b in range(count):
        rng = np.random.Generator(np.random.PCG64(1234 + int(first_pair) + b))
        amp[b] = rng.uniform(0.0, 600.0, size=4)
        psi[b] = rng.uniform(0.0, 2.0 * np.pi, size=4)
        theta[b] = rng.uniform(-0.1, 0.1)
        t[b] = rng.uniform(-100.0, 100.0, size=2)
        nz_t[b] = rng.normal(0.0, 5.0, size=n_points)
        nz_s[b] = rng.normal(0.0, 5.0, size=n_points)
    phi = np.deg2rad(np.arange(n_points, dtype=np.float64) * (360.0 / n_points))[None, :]

    def room(ph):                       # ph [count, n]
        r = np.full(ph.shape, 3000.0)
        for k in range(4):
            r = r + amp[:, k:k + 1] * np.sin((k + 1.0) * ph + psi[:, k:k + 1])
        return r

    r_t = room(np.broadcast_to(phi, (count, n_points))) + nz_t
    tgt = np.stack([r_t * np.cos(phi), r_t * np.sin(phi)], axis=2)
    ph_s = phi + theta[:, None]
    r_s = room(ph_s) + nz_s
    wx = r_s * np.cos(ph_s) - t[:, 0:1]
    wy = r_s * np.sin(ph_s) - t[:, 1:2]
    c, s = np.cos(theta)[:, None], np.sin(theta)[:, None]
    src = np.stack([wx * c + wy * s, wy * c - wx * s], axis=2)       # R^T (world - t)
    src, tgt = src.astype(dtype), tgt.astype(dtype)
    if with_truth:
        return src, tgt, theta, t
    return src, tgt


# ----------------------------------------------------------------------------
# config 5: scan-to-map (SURVEY.md §8d)
# ----------------------------------------------------------------------------
def _polyline_world(seed, n_vertices=24):
    rng = np.random.Generator(np.random.PCG64(seed))
    ang = np.sort(rng.uniform(0.0, 2.0 * np.pi, size=n_vertices))
    rad = rng.uniform(8000.0, 20000.0, size=n_vertices)
    v = np.stack([rad * np.cos(ang), rad * np.sin(ang)], axis=1)
    seg = np.roll(v, -1, axis=0) - v
    length = np.hypot(seg[:, 0], seg[:, 1])
    return rng, v, seg, np.concatenate([[0.0], np.cumsum(length)])


def _sample_polyline(v, seg, cum, s):
    k = np.clip(np.searchsorted(cum, s, side="right") - 1, 0, len(seg) - 1)
    f = (s - cum[k]) / (cum[k + 1] - cum[k])
    return v[k] + seg[k] * f[:, None]


def synth_map(m, seed=5, dtype=np.float32):
    """Map of config 5: m points in order along a seeded closed random polyline (a room of
    8-20 m radius), N(0, 5 mm) noise on both coordinates.  Generated in float64, cast."""
    rng, v, seg, cum = _polyline_world(seed)
    s = (np.arange(m, dtype=np.float64) + 0.5) * (cum[-1] / m)
    pts = _sample_polyline(v, seg, cum, s) + rng.normal(0.0, 5.0, size=(m, 2))
    return pts.astype(dtype)


def synth_scan_for_map(n, seed=5, scan_seed=77, theta=0.02, t=(35.0, -20.0), dtype=np.float32):
    """n noisy observations of the same polyline, expressed in a sensor frame that is rotated by
    ``theta`` and shifted by ``t`` against the map frame (so ICP should recover about that)."""
    _, v, seg, cum = _polyline_world(seed)
    rng = np.random.Generator(np.random.PCG64(scan_seed))
    s = np.sort(rng.uniform(0.0, cum[-1], size=n))
    world = _sample_polyline(v, seg, cum, s) + rng.normal(0.0, 5.0, size=(n, 2))
    c, sn = np.cos(theta), np.sin(theta)
    wx, wy = world[:, 0] - t[0], world[:, 1] - t[1]
    return np.stack([wx * c + wy * sn, wy * c - wx * sn], axis=1).astype(dtype)


# ----------------------------------------------------------------------------
# config 4: all-pairs loop-closure candidates (SURVEY.md §8d)
# ----------------------------------------------------------------------------
def synth_trajectory_scans(n_scans, n_points=360, seed=4096, dtype=np.float32):
    """n_scans scans of ONE star-convex room (same family as config 3) seen from a seeded
    random-walk trajectory: step ~ N(0, 30 mm), heading step ~ N(0, 0.01 rad); every scan is
    the room boundary at n_points world directions + N(0, 5 mm) range noise, expressed in the
    sensor frame.  Returns [n_scans, n_points, 2]."""
    rng = np.random.Generator(np.random.PCG64(seed))
    amp = rng.uniform(0.0, 600.0, size=4)
    psi = rng.uniform(0.0, 2.0 * np.pi, size=4)
    steps = rng.normal(0.0, 30.0, size=(n_scans, 2))
    dth = rng.normal(0.0, 0.01, size=n_scans)
    pos = np.cumsum(steps, axis=0)
    th = np.cumsum(dth)
    phi = np.deg2rad(np.arange(n_points, dtype=np.float64) * (360.0 / n_points))[None, :]
    r = np.full((1, n_points), 3000.0)
    for k in range(4):
        r = r + amp[k] * np.sin((k + 1.0) * phi + psi[k])
    r = r + rng.normal(0.0, 5.0, size=(n_scans, n_points))
    wx = r * np.cos(phi) - pos[:, 0:1]
    wy = r * np.sin(phi) - pos[:, 1:2]
    c, s = np.cos(th)[:, None], np.sin(th)[:, None]
    return np.stack([wx * c + wy * s, wy * c - wx * s], axis=2).astype(dtype)


# ----------------------------------------------------------------------------
# voxel-grid down-sampling as the reference applies it before registration
# (gicp_lidar.py:8-11,20-21 -> Open3D voxel_down_sample; 2D grid as in d.py:10-16)
# ----------------------------------------------------------------------------
def voxel_down_sample_2d(points, voxel_size):
    """One point per occupied cell floor(p / voxel_size): the mean of its points, cells ordered by
    (cell_y, cell_x), int64 per axis.  Points whose cell is not an int64 (non-finite coordinates,
    |p / voxel_size| >= 2^63) are skipped.  PARITY-UNPINNED against Open3D (not vendored; its output
    order is the iteration order of a hash map); this function is the definition the CUDA path is
    held to."""
    p = np.asarray(points, dtype=np.float64)[:, :2]
    inv = 1.0 / float(voxel_size)
    f = np.floor(p * inv)
    keep = np.all(np.abs(f) < 2.0 ** 63, axis=1)
    p, f = p[keep], f[keep]
    if len(p) == 0:
        return p.copy()
    gx, gy = f[:, 0].astype(np.int64), f[:, 1].astype(np.int64)
    order = np.lexsort((np.arange(len(p)), gx, gy))            # stable: (gy, gx), then input order
    gxs, gys = gx[order], gy[order]
    head = np.ones(len(p), dtype=bool)
    head[1:] = (gxs[1:] != gxs[:-1]) | (gys[1:] != gys[:-1])
    seg = np.cumsum(head) - 1
    out = np.zeros((seg[-1] + 1, 2))
    cnt = np.bincount(seg).astype(np.float64)
    np.add.at(out, seg, p[order])                              # unbuffered, in index order: sequential
    return out * (1.0 / cnt)[:, None]
