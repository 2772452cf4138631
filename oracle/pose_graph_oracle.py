"""CPU oracle of the loop-closure back end (TEST INFRASTRUCTURE ONLY, see oracle/__init__.py).

The reference has no loop closure, so this module DEFINES what the CUDA path computes
(parity-UNPINNED, DESIGN.md §4.9; conventions in include/b200icp.h):

  loop_candidates     pairs (i < j) of a trajectory in PAIR_TRIANGLE order with j - i >= min_gap and
                      d^2 <= radius * radius (every product and sum rounded on its own), and the
                      initial relative pose X_i^-1 X_j rounded the same way.
  information         per aligned pair, sum of G^T G, G = [[1, 0, -q_y], [0, 1, q_x]] over the gated
                      correspondences, in the kernel's order: lane l takes the points l, l + 32, ...,
                      then v += v[lane ^ o] for o = 16, 8, 4, 2, 1.
  loop_edges / odometry_edges
                      acceptance of verified candidates, and odometry edges without failed pairs.
  optimize            Gauss-Newton on SE(2) with the same error, Jacobians, assembly order, damping,
                      gauge, per-component anchor and isolated-node rules as the device; the linear solve is exact
                      (scipy.sparse.linalg.spsolve and one step of iterative refinement) where the
                      device runs PCG.
"""
from dataclasses import dataclass, field

import numpy as np
import scipy.sparse as sp
from scipy.sparse.csgraph import connected_components
from scipy.sparse.linalg import spsolve

IDENTITY = np.array([1.0, 0.0, 0.0, 1.0, 0.0, 0.0])
STATUS = {"converged": 0, "max_iterations": 1, "pcg_limit": 2, "non_finite": 3, "bad_edge": 4}


# ----------------------------------------------------------------------------------------------
# poses [R00 R01 R10 R11 tx ty]
# ----------------------------------------------------------------------------------------------
def v2t(x, y, th):
    c, s = np.cos(th), np.sin(th)
    return np.array([c, -s, s, c, x, y])


def compose(a, b):
    """a o b (first b, then a)."""
    Ra, Rb = a[:4].reshape(2, 2), b[:4].reshape(2, 2)
    return np.concatenate([(Ra @ Rb).reshape(4), Ra @ b[4:6] + a[4:6]])


def inverse(a):
    R = a[:4].reshape(2, 2)
    return np.concatenate([R.T.reshape(4), -R.T @ a[4:6]])


def theta(a):
    return float(np.arctan2(a[2], a[0]))


def chain(rel):
    """Prefix composition: out[0] = identity, out[k + 1] = out[k] o rel[k]."""
    out = [IDENTITY.copy()]
    for z in rel:
        out.append(compose(out[-1], z))
    return np.array(out)


# ----------------------------------------------------------------------------------------------
# loop candidates
# ----------------------------------------------------------------------------------------------
def relative_pose(a, b):
    """X_a^-1 X_b with every product and sum rounded on its own (the device has no FMA here)."""
    dx, dy = b[4] - a[4], b[5] - a[5]
    return np.array([a[0] * b[0] + a[2] * b[2], a[0] * b[1] + a[2] * b[3],
                     a[1] * b[0] + a[3] * b[2], a[1] * b[1] + a[3] * b[3],
                     a[0] * dx + a[2] * dy, a[1] * dx + a[3] * dy])


def loop_candidates(poses, min_gap, radius):
    """(src_row j, tgt_row i, rel_pose) in PAIR_TRIANGLE order (i outer, j inner)."""
    P = np.asarray(poses, dtype=np.float64).reshape(-1, 6)
    n = len(P)
    r2 = float(radius) * float(radius)
    src, tgt = [], []
    for i in range(n):
        j = np.arange(i + 1, n)
        j = j[j - i >= min_gap]
        dx, dy = P[i, 4] - P[j, 4], P[i, 5] - P[j, 5]
        keep = j[dx * dx + dy * dy <= r2]
        src.extend(keep.tolist())
        tgt.extend([i] * len(keep))
    rel = np.array([relative_pose(P[i], P[j]) for i, j in zip(tgt, src)]).reshape(-1, 6)
    return np.array(src, dtype=np.int32), np.array(tgt, dtype=np.int32), rel


# ----------------------------------------------------------------------------------------------
# information matrix of an alignment
# ----------------------------------------------------------------------------------------------
def information(src, tgt, pose, indices, max_corr_dist=None):
    """Upper triangle (xx, xy, xt, yy, yt, tt) and the inlier count of one aligned pair.
    src [n, 2], tgt [m, 2], pose [6], indices [>= n] (-1: no correspondence).  The gate compares the
    moved source point; the device moves it with contracted multiply-adds, so a point within an ulp of
    the gate may be decided differently there."""
    src, tgt = np.asarray(src, dtype=np.float64), np.asarray(tgt, dtype=np.float64)
    n = len(src)
    idx = np.asarray(indices[:n], dtype=np.int64)
    ok = (idx >= 0) & (idx < len(tgt))
    q = tgt[np.where(ok, idx, 0)]
    if max_corr_dist is not None and max_corr_dist > 0 and np.isfinite(max_corr_dist):
        s = src @ pose[:4].reshape(2, 2).T + pose[4:6]
        d = q - s
        ok &= np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) < max_corr_dist
    lanes = np.zeros((32, 4))
    for i in np.nonzero(ok)[0]:
        qx, qy = q[i]
        v = lanes[i % 32]
        v[0] += 1.0
        v[1] -= qy
        v[2] += qx
        v[3] += qx * qx + qy * qy
    for o in (16, 8, 4, 2, 1):
        lanes = lanes + lanes[np.arange(32) ^ o]
    c, sy, sx, tt = lanes[0]
    return np.array([c, 0.0, sy, c, sx, tt]), int(c)


# ----------------------------------------------------------------------------------------------
# edges
# ----------------------------------------------------------------------------------------------
def loop_edges(pose_total, rmse, inliers, n_src, src_row, tgt_row, info, min_fitness, max_rmse):
    """Accepted pairs -> (edge_i, edge_j, meas, info).  n_src: source points of each pair."""
    rmse, n_src = np.asarray(rmse, dtype=np.float64), np.asarray(n_src)
    fit = np.where(n_src > 0, np.asarray(inliers, dtype=np.float64) / np.maximum(n_src, 1), 0.0)
    keep = np.isfinite(rmse) & (rmse <= max_rmse) & (fit >= min_fitness)
    return (np.asarray(tgt_row)[keep].astype(np.int32), np.asarray(src_row)[keep].astype(np.int32),
            np.asarray(pose_total)[keep], np.asarray(info)[keep])


def odometry_edges(pose_total, error, iterations, info=None):
    """Pair p -> (p, p + 1); pairs with iterations == 0 or error == +inf are dropped."""
    pose_total = np.asarray(pose_total)
    n = len(pose_total)
    if info is None:
        info = np.tile([1.0, 0.0, 0.0, 1.0, 0.0, 1.0], (n, 1))
    keep = (np.asarray(iterations) > 0) & (np.asarray(error) != np.inf)
    p = np.nonzero(keep)[0]
    return p.astype(np.int32), (p + 1).astype(np.int32), pose_total[keep], np.asarray(info)[keep]


# ----------------------------------------------------------------------------------------------
# Gauss-Newton
# ----------------------------------------------------------------------------------------------
def linearise_edge(Xi, Xj, Z, inf):
    """(e, A, B, e'We) of e = t2v(Z^-1 (Xi^-1 Xj)), theta wrapped to (-pi, pi]."""
    ri00, ri01, ri10, ri11 = Xi[:4]
    rz00, rz01, rz10, rz11 = Z[:4]
    dx, dy = Xj[4] - Xi[4], Xj[5] - Xi[5]
    ux, uy = ri00 * dx + ri10 * dy - Z[4], ri01 * dx + ri11 * dy - Z[5]
    q00, q10 = ri00 * Xj[0] + ri10 * Xj[2], ri01 * Xj[0] + ri11 * Xj[2]
    m00, m10 = rz00 * q00 + rz10 * q10, rz01 * q00 + rz11 * q10
    eth = np.arctan2(m10, m00)
    if eth == -np.pi:
        eth = np.pi
    e = np.array([rz00 * ux + rz10 * uy, rz01 * ux + rz11 * uy, eth])
    S = np.array([[rz00 * ri00 + rz10 * ri01, rz00 * ri10 + rz10 * ri11],
                  [rz01 * ri00 + rz11 * ri01, rz01 * ri10 + rz11 * ri11]])
    w0, w1 = -ri10 * dx + ri00 * dy, -ri00 * dx - ri10 * dy
    v = np.array([rz00 * w0 + rz10 * w1, rz01 * w0 + rz11 * w1])
    A = np.zeros((3, 3))
    A[:2, :2], A[:2, 2], A[2, 2] = -S, v, -1.0
    B = np.zeros((3, 3))
    B[:2, :2], B[2, 2] = S, 1.0
    W = info_matrix(inf)
    return e, A, B, float(e @ W @ e)


def info_matrix(u):
    return np.array([[u[0], u[1], u[2]], [u[1], u[3], u[4]], [u[2], u[4], u[5]]])


def chi2(poses, ei, ej, meas, info):
    return sum(linearise_edge(poses[i], poses[j], z, w)[3] for i, j, z, w in zip(ei, ej, meas, info))


def apply_step(X, x):
    """X (+) x: t + (x0, x1), R R(x2); a zero step leaves the pose as it is."""
    if x[0] == 0.0 and x[1] == 0.0 and x[2] == 0.0:
        return X.copy()
    c, s = np.cos(x[2]), np.sin(x[2])
    r00, r01, r10, r11 = X[:4]
    return np.array([r00 * c + r01 * s, r01 * c - r00 * s, r10 * c + r11 * s, r11 * c - r10 * s,
                     X[4] + x[0], X[5] + x[1]])


def normal_equations(poses, ei, ej, meas, info, fixed=0, damping=0.0):
    """(H, rhs, active) of one Gauss-Newton step: H and -b reduced to the nodes that are neither the
    gauge nor untouched (`active`, the device gives those an identity block and no step)."""
    n = len(poses)
    diag = np.zeros((n, 3, 3))
    g = np.zeros((n, 3))
    touched = np.zeros(n, dtype=bool)
    rows, cols, vals = [], [], []
    # slots in ascending edge order per node = the device's CSR order
    for i, j, z, w in zip(ei, ej, meas, info):
        e, A, B, _ = linearise_edge(poses[i], poses[j], z, w)
        W = info_matrix(w)
        diag[i] += A.T @ W @ A
        diag[j] += B.T @ W @ B
        g[i] += A.T @ W @ e
        g[j] += B.T @ W @ e
        touched[i] = touched[j] = True
        C = A.T @ W @ B
        for r in range(3):
            for c in range(3):
                rows += [3 * i + r, 3 * j + c]
                cols += [3 * j + c, 3 * i + r]
                vals += [C[r, c], C[r, c]]
    active = touched & ~held_nodes(n, ei, ej, fixed)
    for k in range(n):
        if active[k]:
            diag[k] += damping * np.eye(3)
        for r in range(3):
            for c in range(3):
                rows.append(3 * k + r)
                cols.append(3 * k + c)
                vals.append(diag[k, r, c])
    H = sp.csr_matrix((vals, (rows, cols)), shape=(3 * n, 3 * n))
    keep = np.repeat(active, 3)
    return H[keep][:, keep].tocsc(), -g.reshape(-1)[keep], active


def held_nodes(n, ei, ej, fixed=0):
    """The nodes whose row and column are eliminated: the gauge, and the lowest-index node of every
    connected component that does not contain it (isolated nodes included)."""
    held = np.zeros(n, dtype=bool)
    if n == 0:
        return held
    A = sp.coo_matrix((np.ones(len(ei)), (np.asarray(ei), np.asarray(ej))), shape=(n, n))
    _, comp = connected_components(A, directed=False)
    first = {}
    for k in range(n):
        first.setdefault(comp[k], k)
    for c, k in first.items():
        if c != comp[fixed]:
            held[k] = True
    held[fixed] = True
    return held


def anchored_count(n, ei, ej, fixed=0):
    """Components with edges that do not contain the gauge (each held at its lowest node)."""
    touched = np.zeros(n, dtype=bool)
    touched[np.asarray(ei, dtype=np.int64)] = True
    touched[np.asarray(ej, dtype=np.int64)] = True
    h = held_nodes(n, ei, ej, fixed)
    if n:
        h[fixed] = False
    return int((h & touched).sum())


def exact_solve(H, rhs):
    """spsolve and one step of iterative refinement on its float64 residual: on the graphs of the
    tests the refinement moves the solution by up to ~1e-5 mm (the angle and metre scales of H make
    its LU pivots lose digits); a second step changes it by less than 1e-8 mm."""
    x = spsolve(H, rhs)
    return x + spsolve(H, rhs - H @ x)


def gauss_newton_step(poses, ei, ej, meas, info, fixed=0, damping=0.0):
    """The step x [n, 3] of one Gauss-Newton iteration (exact sparse solve)."""
    n = len(poses)
    H, rhs, active = normal_equations(poses, ei, ej, meas, info, fixed, damping)
    x = np.zeros(3 * n)
    keep = np.repeat(active, 3)
    if keep.any():
        x[keep] = exact_solve(H, rhs)
    return x.reshape(n, 3)


@dataclass
class GraphResult:
    poses: np.ndarray
    chi2_initial: float
    chi2_final: float
    iterations: int
    status: int
    isolated: int
    anchored: int = 0
    history: list = field(default_factory=list)       # poses after every step
    chi2_history: list = field(default_factory=list)  # chi2 before the first and after every step


def optimize(poses, ei, ej, meas, info, *, fixed=0, max_iterations=20, tolerance=1e-9, damping=0.0):
    """Gauss-Newton with the device's loop and stopping rule (include/b200icp.h)."""
    X = np.array(poses, dtype=np.float64).reshape(-1, 6).copy()
    ei, ej = np.asarray(ei, dtype=np.int64), np.asarray(ej, dtype=np.int64)
    meas, info = np.asarray(meas, dtype=np.float64).reshape(-1, 6), np.asarray(info, dtype=np.float64).reshape(-1, 6)
    n = len(X)
    touched = np.zeros(n, dtype=bool)
    touched[ei[(ei >= 0) & (ei < n)]] = True
    touched[ej[(ej >= 0) & (ej < n)]] = True
    isolated = int(sum(1 for k in range(n) if not touched[k] and k != fixed))
    if ((ei < 0) | (ej < 0) | (ei >= n) | (ej >= n) | (ei == ej)).any():
        return GraphResult(X, 0.0, 0.0, 0, STATUS["bad_edge"], isolated)
    c = chi2(X, ei, ej, meas, info)
    res = GraphResult(X, c, c, 0, STATUS["converged"], isolated, anchored_count(n, ei, ej, fixed), [], [c])
    if not np.isfinite(c):
        res.status = STATUS["non_finite"]
        return res
    converged = c == 0.0
    while not converged and res.iterations < max_iterations:
        x = gauss_newton_step(X, ei, ej, meas, info, fixed, damping)
        if not np.isfinite(x).all():
            res.status = STATUS["non_finite"]
            break
        X = np.array([apply_step(X[k], x[k]) for k in range(n)])
        res.iterations += 1
        cn = chi2(X, ei, ej, meas, info)
        res.history.append(X.copy())
        res.chi2_history.append(cn)
        if not np.isfinite(cn):
            res.status, c = STATUS["non_finite"], cn
            break
        converged = abs(c - cn) <= tolerance * c or cn == 0.0
        c = cn
    if res.status == STATUS["converged"] and not converged:
        res.status = STATUS["max_iterations"]
    res.poses, res.chi2_final = X, c
    return res


# ----------------------------------------------------------------------------------------------
# synthetic graph with ground truth
# ----------------------------------------------------------------------------------------------
def random_walk(n, seed=4096):
    """The ground-truth poses of the sensor in oracle.icp_oracle.synth_trajectory_scans (configs[3]):
    the same generator and draw order, so scan k of that table was taken from pose k."""
    rng = np.random.Generator(np.random.PCG64(seed))
    rng.uniform(0.0, 600.0, size=4)
    rng.uniform(0.0, 2.0 * np.pi, size=4)
    steps = rng.normal(0.0, 30.0, size=(n, 2))
    dth = rng.normal(0.0, 0.01, size=n)
    pos, th = np.cumsum(steps, axis=0), np.cumsum(dth)
    return np.array([v2t(pos[k, 0], pos[k, 1], th[k]) for k in range(n)])


def synth_graph(n=4096, seed=4096, noise_seed=7, sigma_t=5.0, sigma_th=2e-3, min_gap=50, radius=60.0,
                max_loops=2000, loop_sigma_t=2.0, loop_sigma_th=5e-4):
    """Ground truth from random_walk(n), noisy odometry edges (p, p + 1) and noisy loop edges between
    poses at most `radius` mm apart and at least `min_gap` steps apart (a seeded subset of at most
    max_loops).  Information = diag(1 / sigma^2).  Returns (truth, initial = chained odometry,
    edge_i, edge_j, meas, info)."""
    truth = random_walk(n, seed)
    rng = np.random.default_rng(noise_seed)

    def noisy(a, b, st, sth):
        z = compose(inverse(a), b)
        return compose(z, v2t(rng.normal(0, st), rng.normal(0, st), rng.normal(0, sth)))

    odo = [noisy(truth[k], truth[k + 1], sigma_t, sigma_th) for k in range(n - 1)]
    src, tgt, _ = loop_candidates(truth, min_gap, radius)
    if len(src) > max_loops:
        pick = np.sort(rng.choice(len(src), max_loops, replace=False))
        src, tgt = src[pick], tgt[pick]
    loops = [noisy(truth[i], truth[j], loop_sigma_t, loop_sigma_th) for i, j in zip(tgt, src)]
    w_odo = [1 / sigma_t ** 2, 0.0, 0.0, 1 / sigma_t ** 2, 0.0, 1 / sigma_th ** 2]
    w_loop = [1 / loop_sigma_t ** 2, 0.0, 0.0, 1 / loop_sigma_t ** 2, 0.0, 1 / loop_sigma_th ** 2]
    ei = np.concatenate([np.arange(n - 1), tgt]).astype(np.int32)
    ej = np.concatenate([np.arange(1, n), src]).astype(np.int32)
    meas = np.array(odo + loops).reshape(-1, 6)
    info = np.array([w_odo] * (n - 1) + [w_loop] * len(loops)).reshape(-1, 6)
    return truth, chain(odo), ei, ej, meas, info


def trajectory_error(poses, truth):
    """RMS position error (mm) and RMS heading error (rad) after aligning node 0 of both."""
    T = compose(truth[0], inverse(poses[0]))
    al = np.array([compose(T, p) for p in poses])
    dp = al[:, 4:6] - truth[:, 4:6]
    dth = np.array([theta(compose(inverse(t), a)) for a, t in zip(al, truth)])
    return float(np.sqrt(np.mean(np.sum(dp * dp, axis=1)))), float(np.sqrt(np.mean(dth * dth)))
