"""Loop closure on the B200 against oracle/pose_graph_oracle.py: candidates, information, edges and the
batched pose-graph optimiser (after every Gauss-Newton step), determinism and degenerate graphs."""
import math

import numpy as np
import pytest
import torch

from oracle import pose_graph_oracle as pg

pytestmark = pytest.mark.gpu

MAX_CORR = 300.0
# PCG stops at a preconditioned residual of 1e-14 of the first one.  Against the oracle's exact solve
# (spsolve + one refinement step) the tests below assert every step to 1e-6 mm, 1e-9 rad and 1e-9
# relative chi2, so passing them shows that this tolerance holds that bound on these graphs.
PCG_TOL = 1e-14


@pytest.fixture(scope="module")
def m():
    import __graft_entry__ as ge
    ge.build()
    import icp_slam_yolo_b200 as mod
    return mod


def _dev(a, dtype=torch.float64):
    return torch.from_numpy(np.ascontiguousarray(a)).to(device="cuda", dtype=dtype)


def _graph(m, n, ei, ej, meas, info):
    return m.PoseGraph(n, _dev(ei, torch.int32), _dev(ej, torch.int32), _dev(meas).reshape(-1, 6),
                       _dev(info).reshape(-1, 6))


def _assert_close_poses(got, want, what=""):
    got, want = np.asarray(got), np.asarray(want)
    assert np.abs(got[:, 4:] - want[:, 4:]).max(initial=0.0) < 1e-6, what
    dth = [abs(pg.theta(pg.compose(pg.inverse(w), g))) for g, w in zip(got, want)]
    assert max(dth, default=0.0) < 1e-9, what


def _per_step_parity(m, n, ei, ej, meas, info, init, steps, fixed=0):
    """Device after k steps == oracle after k steps, for every k."""
    o = pg.optimize(init, ei, ej, meas, info, fixed=fixed, max_iterations=steps)
    g = _graph(m, n, ei, ej, meas, info)
    P = _dev(init).reshape(-1, 6)
    for k in range(1, o.iterations + 1):
        r = m.optimize_pose_graph(g, P, fixed=fixed, max_iterations=k, pcg_tolerance=PCG_TOL)
        assert int(r.iterations[0]) == k and int(r.status[0]) in (0, 1)
        _assert_close_poses(r.poses.cpu().numpy(), o.history[k - 1], f"step {k}")
        # relative, with a floor at round-off of the starting chi2 (an odometry-only chain converges to ~1e-25)
        assert abs(float(r.chi2_final[0]) - o.chi2_history[k]) <= 1e-9 * o.chi2_history[k] + 1e-18 * o.chi2_initial
    assert abs(float(r.chi2_initial[0]) - o.chi2_initial) <= 1e-12 * o.chi2_initial
    return o, r


# ------------------------------------------------------------------------------------------------
# candidates
# ------------------------------------------------------------------------------------------------
def test_candidates_bit_exact_with_ulp_neighbours(m):
    rng = np.random.default_rng(11)
    P = np.array([pg.v2t(*rng.uniform(-400, 400, 2), rng.uniform(-3, 3)) for _ in range(300)])
    # pairs exactly on the circle and one ulp either side
    P[200, 4:6], P[250, 4:6] = [0.0, 0.0], [150.0, 0.0]
    P[201, 4:6], P[260, 4:6] = [0.0, 0.0], [np.nextafter(150.0, np.inf), 0.0]
    P[202, 4:6], P[270, 4:6] = [0.0, 0.0], [np.nextafter(150.0, 0.0), 0.0]
    for gap, radius in ((1, 150.0), (20, 150.0), (5, 90.0)):
        s, t, rel = m.loop_candidates(_dev(P), gap, radius)
        ws, wt, wrel = pg.loop_candidates(P, gap, radius)
        assert np.array_equal(s.cpu().numpy(), ws) and np.array_equal(t.cpu().numpy(), wt)
        assert np.array_equal(rel.cpu().numpy().view(np.uint64), wrel.view(np.uint64))
    s, t, _ = m.loop_candidates(_dev(P), 1, 150.0)
    pairs = set(zip(s.tolist(), t.tolist()))
    assert (250, 200) in pairs and (260, 201) not in pairs and (270, 202) in pairs


def test_candidates_small_overflow_and_gap(m):
    for n in (0, 1, 2):
        P = np.tile(pg.IDENTITY, (n, 1))
        s, t, rel = m.loop_candidates(_dev(P).reshape(-1, 6), 1, 10.0)
        assert s.shape[0] == (1 if n == 2 else 0) and rel.shape == (s.shape[0], 6)
    P = np.tile(pg.IDENTITY, (40, 1))                      # every pair within the radius: 780
    s, t, _ = m.loop_candidates(_dev(P), 1, 1.0, capacity=10)
    ws, wt, _ = pg.loop_candidates(P, 1, 1.0)
    assert s.shape[0] == 780 and np.array_equal(s.cpu().numpy(), ws) and np.array_equal(t.cpu().numpy(), wt)
    with pytest.raises(m.B200IcpError, match="capacity"):
        m.loop_candidates(_dev(P), 1, 1.0, capacity=10, strict=True)
    assert m.loop_candidates(_dev(P), 41, 1.0)[0].shape[0] == 0


# ------------------------------------------------------------------------------------------------
# information and edges on the recording
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def recording(m, cart_scans):
    table = m.ScanTable.from_list(cart_scans)
    odo = m.align_consecutive(table, max_iterations=30, tolerance=1e-5, max_corr_dist=MAX_CORR, want_indices=True)
    torch.cuda.synchronize()
    return table, odo


def test_information_on_the_recording_equals_the_oracle(m, recording, cart_scans):
    table, odo = recording
    n = table.rows - 1
    srcs, tgts = table.slice_rows(1), table.slice_rows(0, n)
    pose, idx = odo.pose_total.cpu().numpy(), odo.indices.cpu().numpy()
    for gate in (MAX_CORR, None):
        info, inl = m.information_matrices(srcs, tgts, odo.pose_total, odo.indices, gate)
        info, inl = info.cpu().numpy(), inl.cpu().numpy()
        bad = []
        for p in range(n):
            w, c = pg.information(cart_scans[p + 1], cart_scans[p], pose[p], idx[p], gate)
            if inl[p] != c or not np.array_equal(info[p], w):
                bad.append((p, int(inl[p]), c, float(np.max(np.abs(info[p] - w) / np.maximum(np.abs(w), 1.0)))))
        assert not bad, f"gate {gate}: {len(bad)} pairs differ, first {bad[:5]}"
    far = odo.pose_total.clone()
    far[:, 4] += 1e7                                       # every moved source point lands outside the gate
    info, inl = m.information_matrices(srcs, tgts, far, odo.indices, MAX_CORR)
    assert not info.any() and not inl.any()


def test_edges_equal_the_oracle(m, recording, cart_scans):
    table, odo = recording
    res = m.alloc_outputs(odo.pose_total.shape[0], table.pitch, "cuda")
    for f in ("pose_total", "pose_last", "error", "rmse", "inliers", "iterations"):
        getattr(res, f).copy_(getattr(odo, f))
    res.iterations[::97] = 0                               # failed pairs
    res.error[5::131] = float("inf")
    g = m.PoseGraph.from_odometry(res)
    ei, ej, meas, _ = pg.odometry_edges(res.pose_total.cpu().numpy(), res.error.cpu().numpy(), res.iterations.cpu().numpy())
    assert np.array_equal(g.edge_i.cpu().numpy(), ei) and np.array_equal(g.edge_j.cpu().numpy(), ej)
    assert torch.equal(g.meas.cpu(), torch.from_numpy(meas)) and g.dropped == res.pose_total.shape[0] - len(ei)
    assert g.dropped > 0
    # loop acceptance over odometry results posing as verified candidates
    b = odo.pose_total.shape[0]
    src_row = torch.arange(1, b + 1, dtype=torch.int32, device="cuda")
    tgt_row = torch.arange(0, b, dtype=torch.int32, device="cuda")
    info = torch.rand((b, 6), dtype=torch.float64, device="cuda")
    lens = table.lengths.cpu().numpy()[1:]
    rmse = odo.rmse.cpu().numpy()
    for fit, mr in ((0.5, 40.0), (0.9, 15.0), (0.0, float(np.median(rmse)))):
        k = g.add_loops(odo, src_row, tgt_row, info, min_fitness=fit, max_rmse=mr, src_lengths=table.lengths,
                        src_pitch=table.pitch)
        wi, wj, wm, wf = pg.loop_edges(odo.pose_total.cpu().numpy(), rmse, odo.inliers.cpu().numpy(), lens,
                                       src_row.cpu().numpy(), tgt_row.cpu().numpy(), info.cpu().numpy(), fit, mr)
        assert k == len(wi) and 0 < k < b
        assert np.array_equal(g.edge_i[-k:].cpu().numpy(), wi) and np.array_equal(g.edge_j[-k:].cpu().numpy(), wj)
        assert np.array_equal(g.info[-k:].cpu().numpy(), wf) and np.array_equal(g.meas[-k:].cpu().numpy(), wm)


# ------------------------------------------------------------------------------------------------
# optimiser against the oracle, after every step
# ------------------------------------------------------------------------------------------------
def test_chain_and_ring_per_step(m):
    rng = np.random.default_rng(5)
    n = 200
    truth = np.array([pg.v2t(2000 * math.cos(2 * math.pi * k / n), 2000 * math.sin(2 * math.pi * k / n),
                             2 * math.pi * k / n + math.pi / 2) for k in range(n)])
    odo = [pg.compose(pg.compose(pg.inverse(truth[k]), truth[k + 1]), pg.v2t(*rng.normal(0, [3.0, 3.0, 2e-3])))
           for k in range(n - 1)]
    init = pg.chain(odo)
    init[1:] = [pg.compose(p, pg.v2t(*rng.normal(0, [20.0, 20.0, 0.01]))) for p in init[1:]]
    w = [0.1, 0.0, 0.0, 0.1, 0.0, 2.5e5]
    ei, ej = np.arange(n - 1), np.arange(1, n)
    _per_step_parity(m, n, ei, ej, np.array(odo), np.tile(w, (n - 1, 1)), init, 10)                      # chain
    loop = pg.compose(pg.inverse(truth[0]), truth[n - 1])
    _per_step_parity(m, n, np.append(ei, 0), np.append(ej, n - 1), np.array(odo + [loop]),
                     np.tile(w, (n, 1)), init, 10, fixed=17)                                                  # ring


@pytest.fixture(scope="module")
def synthetic():
    return pg.synth_graph(4096)


def test_synthetic_graph_per_step_and_against_ground_truth(m, synthetic):
    truth, init, ei, ej, meas, info = synthetic
    o, r = _per_step_parity(m, len(truth), ei, ej, meas, info, init, 6)
    err_odo = pg.trajectory_error(init, truth)
    err = pg.trajectory_error(r.poses.cpu().numpy(), truth)
    assert err[0] < 0.5 * err_odo[0] and err[1] < err_odo[1]


def test_recording_with_loop_edges_per_step(m, recording):
    table, odo = recording
    poses, graph, stats = m.close_loops(table, odo, min_gap=100, radius=300.0, max_corr_dist=MAX_CORR,
                                        min_fitness=0.6, max_rmse=60.0, optimize_kw={"pcg_tolerance": PCG_TOL})
    assert stats["loop_edges"] > 0 and stats["chi2_final"] < stats["chi2_initial"]
    init = m.chain_poses(odo.pose_total)
    _per_step_parity(m, graph.n_nodes, graph.edge_i.cpu().numpy(), graph.edge_j.cpu().numpy(),
                     graph.meas.cpu().numpy(), graph.info.cpu().numpy(), init, 4)


# ------------------------------------------------------------------------------------------------
# determinism and degenerate graphs
# ------------------------------------------------------------------------------------------------
def test_alone_and_in_a_batch_of_eight_bit_identical(m, synthetic):
    truth, init, ei, ej, meas, info = synthetic
    big = _graph(m, len(truth), ei, ej, meas, info)
    others, inits = [], []
    for k in range(7):
        t2, i2, a, b, z, w = pg.synth_graph(300 + 150 * k, seed=100 + k, max_loops=100 + 20 * k)
        others.append(_graph(m, len(t2), a, b, z, w))
        inits.append(_dev(i2))
    alone = m.optimize_pose_graph(big, _dev(init), max_iterations=5)
    graphs, ps = others[:3] + [big] + others[3:], inits[:3] + [_dev(init)] + inits[3:]
    for _ in range(2):
        r = m.optimize_pose_graph(graphs, ps, max_iterations=5)
        assert torch.equal(r.split()[3], alone.poses)
        assert torch.equal(r.chi2_final[3], alone.chi2_final[0]) and int(r.pcg_iterations[3]) == int(alone.pcg_iterations[0])
    again = m.optimize_pose_graph(big, _dev(init), max_iterations=5)
    assert torch.equal(again.poses, alone.poses)


def test_degenerate_graphs(m):
    I = pg.IDENTITY
    empty = m.PoseGraph(0, *(torch.empty(0, dtype=torch.int32, device="cuda"),) * 2,
                        torch.empty((0, 6), dtype=torch.float64, device="cuda"),
                        torch.empty((0, 6), dtype=torch.float64, device="cuda"))
    P3 = np.array([pg.v2t(1.0, 2.0, 0.3), pg.v2t(5.0, -1.0, 1.0), pg.v2t(-3.0, 4.0, -2.0)])
    edgeless = m.PoseGraph(3, empty.edge_i, empty.edge_j, empty.meas, empty.info)
    single = m.PoseGraph(1, empty.edge_i, empty.edge_j, empty.meas, empty.info)
    # nodes 0-1-2 joined, node 3 isolated
    Z = pg.v2t(10.0, 0.0, 0.1)
    P4 = np.vstack([pg.chain([Z, Z]), pg.v2t(7.0, 7.0, 0.7)])
    P4[1, 4] += 3.0
    iso = _graph(m, 4, [0, 1], [1, 2], np.array([Z, Z]), np.tile([1, 0, 0, 1, 0, 100.0], (2, 1)))
    bad = I.copy()
    bad[5] = np.inf
    nonfinite = _graph(m, 2, [0], [1], bad[None], np.array([[1, 0, 0, 1, 0, 1.0]]))
    badedge = _graph(m, 2, [0], [2], I[None], np.array([[1, 0, 0, 1, 0, 1.0]]))
    graphs = [empty, edgeless, single, iso, nonfinite, badedge]
    poses = [torch.empty((0, 6), dtype=torch.float64, device="cuda"), _dev(P3), _dev(P3[:1]), _dev(P4),
             _dev(np.tile(I, (2, 1))), _dev(np.tile(I, (2, 1)))]
    r = m.optimize_pose_graph(graphs, poses, max_iterations=10)
    st = r.status.tolist()
    assert st[:4] == [0, 0, 0, 0] and st[4] == 3 and st[5] == 4
    assert r.isolated.tolist()[:4] == [0, 2, 0, 1] and r.anchored.tolist()[:4] == [0, 0, 0, 0]
    out = r.split()
    assert torch.equal(out[1], poses[1]) and torch.equal(out[2], poses[2]) and torch.equal(out[3][3], poses[3][3])
    assert torch.equal(out[3][0], poses[3][0])
    _assert_close_poses(out[3][:3].cpu().numpy(), pg.chain([Z, Z]))
    assert torch.equal(out[4], poses[4]) and torch.equal(out[5], poses[5])
    assert r.iterations.tolist()[4] == 0 and not math.isfinite(float(r.chi2_initial[4]))
    o = pg.optimize(P4, [0, 1], [1, 2], np.array([Z, Z]), np.tile([1, 0, 0, 1, 0, 100.0], (2, 1)), max_iterations=10)
    _assert_close_poses(out[3].cpu().numpy(), o.poses)
    with pytest.raises(m.B200IcpError, match="UNSUPPORTED_SHAPE"):
        m.optimize_pose_graph(m.PoseGraph(65537, empty.edge_i, empty.edge_j, empty.meas, empty.info),
                              torch.zeros((65537, 6), dtype=torch.float64, device="cuda"))


def test_component_without_the_gauge_is_anchored_per_step(m):
    """Two chains with no edge between them (a dropped odometry pair that no loop bridges): the second
    is held at its lowest node, H stays regular, and every step matches the oracle."""
    truth = np.array([pg.v2t(100.0 * k, 10.0 * k, 0.05 * k) for k in range(60)])
    ei = np.array([k for k in range(59) if k != 29], dtype=np.int32)
    ej = ei + 1
    meas = np.array([pg.compose(pg.inverse(truth[i]), truth[j]) for i, j in zip(ei, ej)])
    info = np.tile([1.0, 0.0, 0.0, 1.0, 0.0, 100.0], (len(ei), 1))
    rng = np.random.default_rng(9)
    init = np.array([pg.compose(t, pg.v2t(*rng.normal(0, [20.0, 20.0, 0.01]))) for t in truth])
    o, r = _per_step_parity(m, 60, ei, ej, meas, info, init, 6, fixed=40)
    assert o.anchored == 1 and int(r.anchored[0]) == 1 and int(r.isolated[0]) == 0
    got = r.poses.cpu().numpy()
    assert np.array_equal(got[40], init[40]) and np.array_equal(got[0], init[0])   # gauge and anchor


def test_pcg_iteration_limit_is_reported(m, synthetic):
    truth, init, ei, ej, meas, info = synthetic
    g = _graph(m, len(truth), ei, ej, meas, info)
    r = m.optimize_pose_graph(g, _dev(init), max_iterations=2, pcg_max_iterations=3)
    assert int(r.status[0]) == 2 and int(r.iterations[0]) == 2 and int(r.pcg_iterations[0]) == 6
    assert float(r.chi2_final[0]) < float(r.chi2_initial[0])


def test_close_loops_with_gicp_verification(m, recording):
    table, odo = recording
    poses, graph, stats = m.close_loops(table, odo, min_gap=100, radius=300.0, max_corr_dist=MAX_CORR,
                                        min_fitness=0.6, max_rmse=60.0, registration="gicp")
    assert stats["candidates"] > 0 and stats["loop_edges"] > 0 and stats["anchored"] == 0
    assert stats["status"] in ("converged", "max_iterations") and stats["chi2_final"] < stats["chi2_initial"]
    assert poses.shape == (table.rows, 6) and bool(torch.isfinite(poses).all())
    assert graph.n_edges == stats["odometry_edges"] + stats["loop_edges"]


def test_mixed_devices_are_rejected_before_any_launch(m):
    i32 = torch.zeros(3, dtype=torch.int32)
    f64 = torch.zeros((3, 6), dtype=torch.float64, device="cuda")
    with pytest.raises(m.B200IcpError, match="CUDA"):
        m.PoseGraph(10, i32, i32.cuda(), f64, f64)
