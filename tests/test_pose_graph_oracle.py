"""CPU checks of the loop-closure oracle (oracle/pose_graph_oracle.py), the definition the CUDA path is
held to, and argument / shape rejection of its C ABI (no GPU needed)."""
import ctypes
import math

import numpy as np
import pytest

from oracle import pose_graph_oracle as pg


def _ring(n, radius=2000.0):
    """Ground truth on a circle; odometry (k, k + 1) and one loop edge (0, n - 1)."""
    truth = np.array([pg.v2t(radius * math.cos(2 * math.pi * k / n), radius * math.sin(2 * math.pi * k / n),
                             2 * math.pi * k / n + math.pi / 2) for k in range(n)])
    ei = np.array(list(range(n - 1)) + [0], dtype=np.int32)
    ej = np.array(list(range(1, n)) + [n - 1], dtype=np.int32)
    meas = np.array([pg.compose(pg.inverse(truth[i]), truth[j]) for i, j in zip(ei, ej)])
    info = np.tile([1.0, 0.0, 0.0, 1.0, 0.0, 100.0], (len(ei), 1))
    return truth, ei, ej, meas, info


def test_noise_free_edges_recover_the_ground_truth():
    truth, ei, ej, meas, info = _ring(24)
    rng = np.random.default_rng(1)
    init = np.array([pg.compose(t, pg.v2t(*rng.normal(0, [30.0, 30.0, 0.05]))) for t in truth])
    init[0] = truth[0]                                               # the gauge node sits on the truth
    r = pg.optimize(init, ei, ej, meas, info, max_iterations=30, tolerance=0.0)
    assert r.chi2_final < 1e-16 * r.chi2_initial
    assert np.allclose(r.poses[:, 4:], truth[:, 4:], atol=1e-8, rtol=0)
    assert np.allclose(r.poses[:, :4], truth[:, :4], atol=1e-12, rtol=0)


def test_chi2_never_increases_on_the_synthetic_graphs():
    for n, seed in ((512, 4096), (4096, 4096), (1000, 11)):
        truth, init, ei, ej, meas, info = pg.synth_graph(n, seed=seed, max_loops=400)
        r = pg.optimize(init, ei, ej, meas, info, max_iterations=8)
        h = r.chi2_history
        assert all(b <= a * (1 + 1e-12) for a, b in zip(h, h[1:])), h
        assert r.chi2_final < 0.01 * r.chi2_initial
        assert pg.trajectory_error(r.poses, truth)[0] < pg.trajectory_error(init, truth)[0]


def test_angle_error_wraps_across_pi():
    a = pg.v2t(0.0, 0.0, math.pi - 0.01)
    b = pg.v2t(0.0, 0.0, -math.pi + 0.01)                           # 0.02 rad further, across +-pi
    e, _, _, _ = pg.linearise_edge(a, b, pg.v2t(0.0, 0.0, 0.0), [1, 0, 0, 1, 0, 1])
    assert abs(e[2] - 0.02) < 1e-12
    e, _, _, _ = pg.linearise_edge(a, b, pg.v2t(0.0, 0.0, 0.03), [1, 0, 0, 1, 0, 1])
    assert abs(e[2] + 0.01) < 1e-12
    # exactly pi apart: (-pi, pi] keeps +pi
    e, _, _, _ = pg.linearise_edge(pg.v2t(0, 0, 0), np.array([-1.0, -0.0, 0.0, -1.0, 0, 0]), pg.IDENTITY, [1, 0, 0, 1, 0, 1])
    assert e[2] == math.pi
    # a graph whose headings cross +-pi converges like any other
    n = 16
    truth = np.array([pg.v2t(100.0 * k, 0.0, math.pi - 0.2 + 0.03 * k) for k in range(n)])
    ei, ej = np.arange(n - 1, dtype=np.int32), np.arange(1, n, dtype=np.int32)
    meas = np.array([pg.compose(pg.inverse(truth[i]), truth[j]) for i, j in zip(ei, ej)])
    init = truth.copy()
    init[1:] = [pg.compose(t, pg.v2t(5.0, -3.0, 0.02)) for t in truth[1:]]
    r = pg.optimize(init, ei, ej, meas, np.tile([1, 0, 0, 1, 0, 1.0], (n - 1, 1)), max_iterations=20, tolerance=0.0)
    assert np.allclose(r.poses, truth, atol=1e-8)


def test_jacobians_match_finite_differences():
    rng = np.random.default_rng(2)
    for _ in range(20):
        Xi, Xj, Z = (pg.v2t(*rng.normal(0, [500, 500, 2])) for _ in range(3))
        e, A, B, _ = pg.linearise_edge(Xi, Xj, Z, [1, 0, 0, 1, 0, 1])
        for J, which in ((A, 0), (B, 1)):
            for c in range(3):
                d = np.zeros(3)
                d[c] = 1e-6
                ev = []
                for sgn in (1.0, -1.0):                                  # central difference
                    Xp = [Xi, Xj]
                    Xp[which] = pg.apply_step(Xp[which], sgn * d)
                    ev.append(pg.linearise_edge(Xp[0], Xp[1], Z, [1, 0, 0, 1, 0, 1])[0])
                assert np.allclose((ev[0] - ev[1]) / 2e-6, J[:, c], rtol=1e-6, atol=1e-4)


def test_gauge_node_and_isolated_nodes_keep_their_pose():
    truth, ei, ej, meas, info = _ring(10)
    init = np.array([pg.compose(t, pg.v2t(10.0, -5.0, 0.01)) for t in truth])
    extra = pg.v2t(7.0, 8.0, 0.3)                                    # node 10: no edge touches it
    init = np.vstack([init, extra])
    for fixed in (0, 4):
        r = pg.optimize(init, ei, ej, meas, info, fixed=fixed, max_iterations=10)
        assert np.array_equal(r.poses[fixed], init[fixed]) and np.array_equal(r.poses[10], extra)
        assert r.isolated == 1 and r.status in (0, 1)           # noise-free: chi2 ends at round-off level
        for k in range(10):                                          # relative poses are the truth's
            rel = pg.compose(pg.inverse(r.poses[fixed]), r.poses[k])
            want = pg.compose(pg.inverse(truth[fixed]), truth[k])
            assert np.allclose(rel, want, atol=1e-7)


def test_degenerate_graphs():
    r = pg.optimize(np.zeros((0, 6)), [], [], np.zeros((0, 6)), np.zeros((0, 6)))
    assert r.status == 0 and r.iterations == 0 and r.chi2_final == 0.0
    P = np.tile(pg.IDENTITY, (3, 1))
    r = pg.optimize(P, [], [], np.zeros((0, 6)), np.zeros((0, 6)))
    assert r.status == 0 and r.isolated == 2 and np.array_equal(r.poses, P)
    r = pg.optimize(P, [0], [5], [pg.IDENTITY], [[1, 0, 0, 1, 0, 1]])
    assert r.status == pg.STATUS["bad_edge"]
    bad = pg.IDENTITY.copy()
    bad[4] = np.nan
    r = pg.optimize(P, [0], [1], [bad], [[1, 0, 0, 1, 0, 1]])
    assert r.status == pg.STATUS["non_finite"] and r.iterations == 0 and np.array_equal(r.poses, P)


def test_candidates_are_in_triangle_order_with_crop_rounding():
    rng = np.random.default_rng(3)
    P = np.array([pg.v2t(*rng.uniform(-300, 300, 2), rng.uniform(-3, 3)) for _ in range(60)])
    src, tgt, rel = pg.loop_candidates(P, 5, 200.0)
    want = [(j, i) for i in range(60) for j in range(i + 5, 60)
            if (P[i, 4] - P[j, 4]) ** 2 + (P[i, 5] - P[j, 5]) ** 2 <= 200.0 ** 2]
    assert list(zip(src.tolist(), tgt.tolist())) == want
    for (j, i), r in zip(want, rel):
        assert np.allclose(r, pg.compose(pg.inverse(P[i]), P[j]), atol=1e-9)
    # on the circle and one ulp either side
    r2 = 150.0 * 150.0
    Q = np.tile(pg.IDENTITY, (4, 1))
    Q[1, 4] = 150.0
    Q[2, 4] = np.nextafter(150.0, np.inf)
    Q[3, 4] = np.nextafter(150.0, 0.0)
    src, tgt, _ = pg.loop_candidates(Q, 1, 150.0)
    assert (1, 0) in zip(src, tgt) and (2, 0) not in zip(src, tgt) and (3, 0) in zip(src, tgt)
    assert Q[1, 4] * Q[1, 4] == r2
    assert pg.loop_candidates(Q, 10, 1e9)[0].size == 0


def test_information_order_and_gate():
    rng = np.random.default_rng(4)
    tgt = rng.uniform(-3000, 3000, size=(300, 2))
    src = tgt[:200] + rng.normal(0, 5, size=(200, 2))
    idx = np.arange(200)
    idx[::7] = -1
    info, n = pg.information(src, tgt, pg.IDENTITY, idx)
    q = tgt[:200][idx >= 0]
    assert n == len(q) and info[0] == info[3] == n and info[1] == 0.0
    assert np.isclose(info[2], -q[:, 1].sum(), rtol=1e-14) and np.isclose(info[4], q[:, 0].sum(), rtol=1e-14)
    assert np.isclose(info[5], (q * q).sum(), rtol=1e-14)
    G = np.zeros((3, 3))
    for x, y in q:
        g = np.array([[1, 0, -y], [0, 1, x]])
        G += g.T @ g
    assert np.allclose(info, G[np.triu_indices(3)], rtol=1e-12)
    assert pg.information(src, tgt, pg.v2t(1e5, 0, 0), idx, 100.0) == (pytest.approx(np.zeros(6)), 0)


def test_edge_acceptance():
    pose = np.tile(pg.IDENTITY, (5, 1))
    rmse = np.array([10.0, np.inf, 30.0, 10.0, np.nan])
    inl = np.array([90, 90, 90, 40, 90])
    ei, ej, _, _ = pg.loop_edges(pose, rmse, inl, np.full(5, 100), np.arange(5) + 10, np.arange(5),
                                 np.zeros((5, 6)), 0.5, 20.0)
    assert ei.tolist() == [0] and ej.tolist() == [10]
    ei, ej, _, _ = pg.odometry_edges(pose, np.array([1.0, np.inf, 2.0, 3.0, 4.0]), np.array([5, 5, 0, 5, 5]))
    assert ei.tolist() == [0, 3, 4] and ej.tolist() == [1, 4, 5]


def test_cabi_rejects_bad_pose_graph_arguments_without_touching_the_gpu():
    import __graft_entry__ as ge
    ge.build()
    from icp_slam_yolo_b200 import _cabi
    L = _cabi.lib()
    p = ctypes.c_void_p(4096)
    # candidates
    assert L.b200icp_loop_candidates(p, 10, 1, 5.0, 4, p, p, p, None, p, None) == 1
    assert L.b200icp_loop_candidates(p, 10, 0, 5.0, 4, p, p, p, p, p, None) == 1
    assert L.b200icp_loop_candidates(p, 10, 1, -1.0, 4, p, p, p, p, p, None) == 1
    assert L.b200icp_loop_candidates(p, 10, 1, float("nan"), 4, p, p, p, p, p, None) == 1
    assert L.b200icp_loop_candidates(p, 10, 1, 5.0, 4, None, p, p, p, p, None) == 1
    assert L.b200icp_loop_candidates(p, 65537, 1, 5.0, 4, p, p, p, p, p, None) == 2
    # information
    pr = _cabi.Problem()
    assert L.b200icp_information_batch(None, 1, p, p, 0.0, p, None, None) == 1
    pr.src_points = pr.tgt_points = 4096
    pr.src_pitch, pr.tgt_pitch, pr.dtype = 16, 16, _cabi.F64
    assert L.b200icp_information_batch(ctypes.byref(pr), 1, None, p, 0.0, p, None, None) == 1
    assert L.b200icp_information_batch(ctypes.byref(pr), 1, p, None, 0.0, p, None, None) == 1
    assert L.b200icp_information_batch(ctypes.byref(pr), -1, p, p, 0.0, p, None, None) == 1
    # edges
    assert L.b200icp_loop_edges(1, p, p, p, None, 16, p, p, None, 0.5, 1.0, p, p, p, p, None, p, None) == 1
    assert L.b200icp_loop_edges(1, p, p, p, None, 0, p, p, None, 0.5, 1.0, p, p, p, p, p, p, None) == 1
    assert L.b200icp_loop_edges(1, p, p, p, None, 16, p, p, None, float("nan"), 1.0, p, p, p, p, p, p, None) == 1
    assert L.b200icp_odometry_edges(1, None, p, p, None, p, p, p, p, p, p, None) == 1
    assert L.b200icp_odometry_edges(-1, p, p, p, None, p, p, p, p, p, p, None) == 1
    # optimiser
    opt, out = _cabi.PoseGraphOptions(), _cabi.PoseGraphOutputs()
    opt.max_iterations, opt.pcg_max_iterations, opt.pcg_tolerance = 5, 100, 1e-12
    out.poses = out.status = 4096

    def batch(nodes, edges, fixed=None):
        b = _cabi.PoseGraphBatch()
        no, eo = np.asarray(nodes, dtype=np.int64), np.asarray(edges, dtype=np.int64)
        b.n_graphs = len(no) - 1
        b.node_offset, b.edge_offset = no.ctypes.data, eo.ctypes.data
        if fixed is not None:
            f = np.asarray(fixed, dtype=np.int32)
            b.fixed_node = f.ctypes.data
        b.poses_in = b.edge_i = b.edge_j = b.meas = b.info = 4096
        return b, no, eo, (f if fixed is not None else None)

    def call(b, o=opt, ws=p, nbytes=1 << 40):
        return L.b200icp_pose_graph_optimize(ctypes.byref(b), ctypes.byref(o), ctypes.byref(out), ws, nbytes, None)

    assert L.b200icp_pose_graph_optimize(None, ctypes.byref(opt), ctypes.byref(out), p, 1 << 40, None) == 1
    keep = batch([0, 65537], [0, 10])
    assert call(keep[0]) == 2 and L.b200icp_pose_graph_workspace_bytes(ctypes.byref(keep[0])) == -1
    keep = batch([0, 10], [0, (1 << 20) + 1])
    assert call(keep[0]) == 2
    keep = batch([0, 10, 5], [0, 4, 8])                   # decreasing node offsets
    assert call(keep[0]) == 1
    keep = batch([1, 10], [0, 4])                         # offsets must start at 0
    assert call(keep[0]) == 1
    keep = batch([0, 10], [0, 4], fixed=[10])             # gauge outside the graph
    assert call(keep[0]) == 1
    keep = batch([0, 10], [0, 4])
    assert L.b200icp_pose_graph_workspace_bytes(ctypes.byref(keep[0])) > 0
    assert call(keep[0], nbytes=16) == 1                  # workspace too small
    assert call(keep[0], ws=None) == 1
    bad = _cabi.PoseGraphOptions()
    bad.max_iterations, bad.pcg_max_iterations, bad.damping = 5, 100, -1.0
    assert call(keep[0], o=bad) == 1
    bad.damping, bad.tolerance = 0.0, float("nan")
    assert call(keep[0], o=bad) == 1
    b = keep[0]
    b.meas = None
    assert call(b) == 1
    assert b"NULL" in L.b200icp_last_error()


def _split_chain():
    """Two chains 0-1-2-3 and 4-5-6 with no edge between them (a dropped odometry pair, no loop)."""
    truth = np.array([pg.v2t(100.0 * k, 10.0 * k, 0.05 * k) for k in range(7)])
    ei = np.array([0, 1, 2, 4, 5], dtype=np.int32)
    ej = ei + 1
    meas = np.array([pg.compose(pg.inverse(truth[i]), truth[j]) for i, j in zip(ei, ej)])
    info = np.tile([1.0, 0.0, 0.0, 1.0, 0.0, 100.0], (len(ei), 1))
    init = np.array([pg.compose(t, pg.v2t(3.0 * k, -2.0, 0.01 * k)) for k, t in enumerate(truth)])
    return truth, init, ei, ej, meas, info


def test_a_component_without_the_gauge_is_held_at_its_lowest_node():
    truth, init, ei, ej, meas, info = _split_chain()
    assert pg.held_nodes(7, ei, ej, 0).tolist() == [True, False, False, False, True, False, False]
    assert pg.held_nodes(7, ei, ej, 5).tolist() == [True, False, False, False, False, True, False]
    r = pg.optimize(init, ei, ej, meas, info, max_iterations=20, tolerance=0.0)
    assert r.anchored == 1 and r.isolated == 0 and np.isfinite(r.chi2_final) and r.chi2_final < 1e-12
    assert np.array_equal(r.poses[0], init[0]) and np.array_equal(r.poses[4], init[4])
    for a, k in ((0, 2), (4, 6)):                                   # each chain is rigid again
        assert np.allclose(pg.compose(pg.inverse(r.poses[a]), r.poses[k]),
                           pg.compose(pg.inverse(truth[a]), truth[k]), atol=1e-8)
    # an isolated node is not an anchored component
    assert pg.anchored_count(8, ei, ej, 0) == 1


def test_pose_graph_rejects_malformed_edge_tensors_before_any_launch():
    import torch
    from icp_slam_yolo_b200 import B200IcpError, PoseGraph, optimize_pose_graph
    i32, f64 = torch.zeros(3, dtype=torch.int32), torch.zeros((3, 6), dtype=torch.float64)
    bad = [
        dict(edge_i=torch.zeros(3, dtype=torch.int64)),              # int64 indices (torch.arange)
        dict(edge_j=torch.zeros((3, 1), dtype=torch.int32)),         # not 1-D
        dict(meas=torch.zeros((3, 6), dtype=torch.float32)),         # float32 measurements
        dict(info=torch.zeros((3, 3), dtype=torch.float64)),         # not [e, 6]
        dict(meas=torch.zeros((2, 6), dtype=torch.float64)),         # fewer rows than edges
        dict(edge_j=torch.zeros(4, dtype=torch.int32)),              # lengths disagree
        dict(info=[[0.0] * 6] * 3),                                  # not a tensor
    ]
    for change in bad:
        with pytest.raises(ValueError):
            PoseGraph(10, **{**dict(edge_i=i32, edge_j=i32, meas=f64, info=f64), **change})
    with pytest.raises(ValueError, match="n_nodes"):
        PoseGraph(-1, i32, i32, f64, f64)
    with pytest.raises(B200IcpError, match="CUDA"):                 # right shapes, host memory
        PoseGraph(10, i32, i32, f64, f64)
    # fields replaced after construction are checked again by the optimiser
    g = PoseGraph.__new__(PoseGraph)
    g.n_nodes, g.edge_i, g.edge_j, g.meas, g.info, g.dropped = 10, i32, i32, f64.float(), f64, 0
    with pytest.raises(ValueError, match="meas"):
        optimize_pose_graph(g, torch.zeros((10, 6), dtype=torch.float64))
