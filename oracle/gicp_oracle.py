"""CPU oracle of 2D Generalized ICP (TEST INFRASTRUCTURE ONLY, see oracle/__init__.py).

The reference registers each frame with Open3D's Generalized ICP (gicp(scan, local_map, threshold,
voxel, trans_init), duc/ICP_LIDAR/slam_offline.py:382, mainn.py:311, gicp_lidar.py:12-36).  Open3D is
not vendored, so this module DEFINES the 2D model the CUDA path is held to (parity-UNPINNED,
DESIGN.md §4.8): line-to-line GICP, the 2D analogue of Open3D's plane-to-plane.

  estimate_covariances_2d  per point: the k nearest points of the same cloud under the order
                           (d^2, index), the point itself included; population covariance with the
                           sums taken sequentially in that order; regularised to
                           u u^T + eps (I - u u^T), u = the principal direction
                           (phi = atan2(2 cxy, cxx - cyy) / 2); identity when |N| < 3 or cxx + cyy = 0.
  gicp_extended            Open3D's RegistrationICP loop shape: evaluate at the initial pose, then
                           solve / apply / evaluate until |d fitness| < relative_fitness and
                           |d rmse| < relative_rmse, or max_iterations.  One Gauss-Newton step in
                           (dtheta, dx, dy) per update, float64, about the pivot c = current pose
                           applied to the centroid of the original source.
"""
from dataclasses import dataclass, field

import numpy as np
from scipy.spatial import cKDTree

from . import icp_oracle as orc
from .slam_oracle import OracleSlam


def _knn_small(P, kk):
    """Stable argsort of the exact float64 d^2 = (lexicographic (d^2, index))."""
    dx = P[:, None, 0] - P[None, :, 0]
    dy = P[:, None, 1] - P[None, :, 1]
    d2 = dx * dx + dy * dy
    return np.argsort(d2, axis=1, kind="stable")[:, :kk]


def _knn_large(P, kk):
    """The same sets for large clouds: a KD-tree ball slightly larger than its kk-th distance is a
    superset of the kk nearest points; the selection among it is made on the exact float64 d^2."""
    tree = cKDTree(P)
    dk, _ = tree.query(P, k=kk)
    dk = np.asarray(dk).reshape(len(P), -1)[:, -1]
    balls = tree.query_ball_point(P, dk * (1.0 + 1e-9) + 1e-300, return_sorted=True)
    out = np.empty((len(P), kk), dtype=np.intp)
    for i, cand in enumerate(balls):
        cand = np.asarray(cand, dtype=np.intp)
        dx = P[i, 0] - P[cand, 0]
        dy = P[i, 1] - P[cand, 1]
        d2 = dx * dx + dy * dy
        out[i] = cand[np.argsort(d2, kind="stable")[:kk]]
    return out


def knn_2d(P, k):
    """Indices [n, min(k, n)] of the k nearest points of the cloud itself, ordered by (d^2, index)."""
    P = np.asarray(P, dtype=np.float64)
    kk = min(int(k), len(P))
    if len(P) == 0:
        return np.zeros((0, 0), dtype=np.intp)
    return _knn_small(P, kk) if len(P) <= 2048 else _knn_large(P, kk)


def regularise(cxx, cxy, cyy, eps, count):
    """C_reg = u u^T + eps (I - u u^T) as (cxx, cxy, cyy); identity when count < 3 or cxx + cyy = 0."""
    phi = 0.5 * np.arctan2(2.0 * cxy, cxx - cyy)
    c, s = np.cos(phi), np.sin(phi)
    out = np.stack([c * c + eps * (s * s), (1.0 - eps) * (c * s), s * s + eps * (c * c)], axis=-1)
    iso = (np.asarray(count) < 3) | ((cxx + cyy) == 0.0)
    out[iso] = (1.0, 0.0, 1.0)
    return out


def estimate_covariances_2d(P, k=20, eps=1e-3):
    """[n, 3] (cxx, cxy, cyy) regularised covariances of one cloud (see the module docstring)."""
    P = np.asarray(P, dtype=np.float64)[:, :2]
    n = len(P)
    if n == 0:
        return np.zeros((0, 3))
    nb = P[knn_2d(P, k)]                                   # [n, kk, 2] in (d^2, index) order
    kk = nb.shape[1]
    sx, sy = np.zeros(n), np.zeros(n)
    for j in range(kk):                                    # sequential sums, as the kernel adds them
        sx = sx + nb[:, j, 0]
        sy = sy + nb[:, j, 1]
    mx, my = sx / kk, sy / kk
    cxx, cxy, cyy = np.zeros(n), np.zeros(n), np.zeros(n)
    for j in range(kk):
        dx, dy = nb[:, j, 0] - mx, nb[:, j, 1] - my
        cxx = cxx + dx * dx
        cxy = cxy + dx * dy
        cyy = cyy + dy * dy
    return regularise(cxx / kk, cxy / kk, cyy / kk, float(eps), kk)


def nn_exact(src, tgt, tree=None):
    """float64 argmin_j |src_i - tgt_j|^2 with the lowest j on exact ties (= orc.nn_bruteforce), via a
    KD-tree where its two best distances are clearly apart and brute force for the rest."""
    src = np.asarray(src, dtype=np.float64)
    tgt = np.asarray(tgt, dtype=np.float64)
    if len(tgt) < 2:
        return orc.nn_bruteforce(src, tgt)
    tree = cKDTree(tgt) if tree is None else tree
    d, i = tree.query(src, k=2)
    idx = i[:, 0].astype(np.intp)
    amb = ~(d[:, 1] > d[:, 0] * (1.0 + 1e-9) + 1e-300)
    if np.any(amb):
        _, idx[amb] = orc.nn_bruteforce(src[amb], tgt)
    dx = src[:, 0] - tgt[idx, 0]
    dy = src[:, 1] - tgt[idx, 1]
    return np.sqrt(dx * dx + dy * dy), idx


@dataclass
class GicpResult:
    R_tot: np.ndarray
    t_tot: np.ndarray
    R_last: np.ndarray            # last applied increment p -> R_last p + t_last
    t_last: np.ndarray
    src: np.ndarray               # source at the final pose
    iterations: int               # applied updates
    rmse: float                   # at the final pose; +inf when no pair survived the gate
    error: float                  # mean inlier distance at the final pose
    fitness: float
    inliers: int
    indices: np.ndarray           # correspondences at the final pose
    history: list = field(default_factory=list)    # history[it]: the correspondences update `it` used
    poses: list = field(default_factory=list)      # (R, t) after each update
    fitness_history: list = field(default_factory=list)   # per evaluation
    rmse_history: list = field(default_factory=list)


def _apply(R, t, P):
    """R p + t elementwise in the kernel's operation order (no contraction)."""
    return np.stack([R[0, 0] * P[:, 0] + R[0, 1] * P[:, 1] + t[0],
                     R[1, 0] * P[:, 0] + R[1, 1] * P[:, 1] + t[1]], axis=1)


def cholesky_solve3(H, g):
    """Solve H x = g with a 3x3 Cholesky factorisation; None on a non-positive / non-finite pivot."""
    H00, H01, H02, H11, H12, H22 = H
    if not (np.isfinite(H00) and H00 > 0.0):
        return None
    L00 = np.sqrt(H00)
    L10, L20 = H01 / L00, H02 / L00
    p1 = H11 - L10 * L10
    if not (np.isfinite(p1) and p1 > 0.0):
        return None
    L11 = np.sqrt(p1)
    L21 = (H12 - L20 * L10) / L11
    p2 = H22 - L20 * L20 - L21 * L21
    if not (np.isfinite(p2) and p2 > 0.0):
        return None
    L22 = np.sqrt(p2)
    y0 = g[0] / L00
    y1 = (g[1] - L10 * y0) / L11
    y2 = (g[2] - L20 * y0 - L21 * y1) / L22
    x2 = y2 / L22
    x1 = (y1 - L21 * x2) / L11
    x0 = (y0 - L10 * x1 - L20 * x2) / L00
    return np.array([x0, x1, x2])


def gn_system(S, Bm, CA, CB, R, c):
    """H (6 sums: 00 01 02 11 12 22) and g (3 sums) of one Gauss-Newton step for matched inliers:
    J = [[-(sy - cy), 1, 0], [sx - cx, 0, 1]], r = b - s, M = (C_B + R C_A R^T)^-1."""
    r00, r01, r10, r11 = R[0, 0], R[0, 1], R[1, 0], R[1, 1]
    a, b, d = CA[:, 0], CA[:, 1], CA[:, 2]
    # R C R^T
    u00, u01, u10, u11 = r00 * a + r01 * b, r00 * b + r01 * d, r10 * a + r11 * b, r10 * b + r11 * d
    sa = CB[:, 0] + (u00 * r00 + u01 * r01)
    sb = CB[:, 1] + (u00 * r10 + u01 * r11)
    sd = CB[:, 2] + (u10 * r10 + u11 * r11)
    inv = 1.0 / (sa * sd - sb * sb)
    m00, m01, m11 = sd * inv, -sb * inv, sa * inv
    rx, ry = S[:, 0] - c[0], S[:, 1] - c[1]
    e0, e1 = Bm[:, 0] - S[:, 0], Bm[:, 1] - S[:, 1]
    w0 = m01 * rx - m00 * ry                               # M [-ry, rx]
    w1 = m11 * rx - m01 * ry
    v0 = m00 * e0 + m01 * e1                               # M r
    v1 = m01 * e0 + m11 * e1
    H = np.array([np.sum(rx * w1 - ry * w0), np.sum(w0), np.sum(w1), np.sum(m00), np.sum(m01), np.sum(m11)])
    g = np.array([np.sum(rx * v1 - ry * v0), np.sum(v0), np.sum(v1)])
    return H, g


def gicp_extended(A, B, max_iterations=30, *, init_pose=None, max_corr_dist=None, relative_fitness=1e-6,
                  relative_rmse=1e-6, cov_A=None, cov_B=None, k=20, eps=1e-3, pivot=None):
    """2D GICP of source A onto target B (module docstring).  ``pivot``: override the lever-arm
    origin (the result does not depend on it, up to rounding) -- a fixed point in the target frame."""
    A = np.asarray(A, dtype=np.float64)[:, :2]
    B = np.asarray(B, dtype=np.float64)[:, :2]
    R, t = np.eye(2), np.zeros(2)
    if init_pose is not None:
        R = np.asarray(init_pose[0], dtype=np.float64).copy()
        t = np.asarray(init_pose[1], dtype=np.float64).copy()
    n, m = len(A), len(B)
    res = GicpResult(R, t, np.eye(2), np.zeros(2), _apply(R, t, A) if n else A.copy(), 0,
                     float("inf"), float("inf"), 0.0, 0, np.full(n, -1, dtype=np.intp))
    if n == 0 or m == 0:
        return res
    CA = estimate_covariances_2d(A, k, eps) if cov_A is None else np.asarray(cov_A, dtype=np.float64)
    CB = estimate_covariances_2d(B, k, eps) if cov_B is None else np.asarray(cov_B, dtype=np.float64)
    gate = max_corr_dist is not None and 0.0 < max_corr_dist < np.inf
    tree = cKDTree(B)
    cA = A.mean(axis=0)
    src = _apply(R, t, A)

    def evaluate(S):
        d, idx = nn_exact(S, B, tree)
        keep = d < max_corr_dist if gate else np.ones(n, dtype=bool)
        cnt = int(keep.sum())
        if cnt == 0:
            return idx, keep, 0.0, float("inf"), float("inf")
        dk = d[keep]
        return idx, keep, cnt / n, float(np.sqrt(np.mean(dk * dk))), float(np.mean(dk))

    idx, keep, fit, rmse, err = evaluate(src)
    res.fitness_history.append(fit)
    res.rmse_history.append(rmse)
    it = 0
    while np.isfinite(rmse) and it < max_iterations:
        c = _apply(R, t, cA[None])[0] if pivot is None else np.asarray(pivot, dtype=np.float64)
        H, g = gn_system(src[keep], B[idx[keep]], CA[keep], CB[idx[keep]], R, c)
        x = cholesky_solve3(H, g)
        if x is None:
            break
        # applied as increments, s + ((R(dtheta) - I)(s - c) + dt) with cos - 1 = -2 sin^2(dtheta / 2):
        # a zero step leaves points and pose bit for bit unchanged
        sh, ch = np.sin(0.5 * x[0]), np.cos(0.5 * x[0])
        st, cm1 = 2.0 * sh * ch, -2.0 * sh * sh
        ex, ey = src[:, 0] - c[0], src[:, 1] - c[1]
        src = np.stack([src[:, 0] + ((cm1 * ex - st * ey) + x[1]), src[:, 1] + ((st * ex + cm1 * ey) + x[2])], axis=1)
        tx, ty = t[0] - c[0], t[1] - c[1]
        t = np.array([t[0] + ((cm1 * tx - st * ty) + x[1]), t[1] + ((st * tx + cm1 * ty) + x[2])])
        R = R + np.array([[cm1 * R[0, 0] - st * R[1, 0], cm1 * R[0, 1] - st * R[1, 1]],
                          [st * R[0, 0] + cm1 * R[1, 0], st * R[0, 1] + cm1 * R[1, 1]]])
        res.R_last = np.array([[1.0 + cm1, -st], [st, 1.0 + cm1]])
        res.t_last = np.array([x[1] - (cm1 * c[0] - st * c[1]), x[2] - (st * c[0] + cm1 * c[1])])
        res.history.append(np.asarray(idx))
        res.poses.append((R.copy(), t.copy()))
        it += 1
        idx2, keep2, fit2, rmse2, err2 = evaluate(src)
        res.fitness_history.append(fit2)
        res.rmse_history.append(rmse2)
        converged = abs(fit2 - fit) < relative_fitness and abs(rmse2 - rmse) < relative_rmse
        idx, keep, fit, rmse, err = idx2, keep2, fit2, rmse2, err2
        if converged:
            break
    res.R_tot, res.t_tot, res.src, res.iterations = R, t, src, it
    res.rmse, res.error, res.fitness, res.inliers, res.indices = rmse, err, fit, int(keep.sum()) if np.isfinite(rmse) else 0, idx
    return res


class GicpOracleSlam(OracleSlam):
    """OracleSlam whose registration follows ``cfg.registration`` ("p2p", the default, or "gicp")."""

    def _gicp(self, p1, p2):
        c = self.c
        if getattr(c, "registration", "p2p") != "gicp":
            return super()._gicp(p1, p2)
        if len(p1) < 10 or len(p2) < 10:
            return float("inf"), np.eye(4)
        a, b = orc.voxel_down_sample_2d(p1[:, :2], c.icp_voxel_size), orc.voxel_down_sample_2d(p2[:, :2], c.icp_voxel_size)
        o = gicp_extended(a, b, c.max_iteration, init_pose=(self.pose[:2, :2], self.pose[:2, 3]),
                          max_corr_dist=c.icp_threshold)
        T = np.eye(4)
        T[:2, :2], T[:2, 3] = o.R_tot, o.t_tot
        return o.rmse, T
