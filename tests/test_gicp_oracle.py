"""CPU checks of the 2D GICP oracle (oracle/gicp_oracle.py), the definition the CUDA path is held
to, and argument rejection of the GICP C ABI (no GPU needed)."""
import ctypes
import math

import numpy as np
import pytest
from scipy.spatial import cKDTree

from oracle import gicp_oracle as g
from oracle import icp_oracle as orc


def _rot(th):
    return np.array([[math.cos(th), -math.sin(th)], [math.sin(th), math.cos(th)]])


def test_knn_sets_match_the_kd_tree_where_there_are_no_ties():
    rng = np.random.default_rng(3)
    for n in (7, 300, 2500):                      # 2,500 > 2,048 takes the KD-tree-superset path
        P = rng.uniform(-5000.0, 5000.0, size=(n, 2))
        for k in (3, 20, 32):
            kk = min(k, n)
            _, want = cKDTree(P).query(P, k=kk)
            got = g.knn_2d(P, k)
            assert got.shape == (n, kk)
            assert np.array_equal(np.sort(got, axis=1), np.sort(np.asarray(want).reshape(n, kk), axis=1))


def test_knn_large_path_equals_brute_force_with_ties():
    P = np.stack(np.meshgrid(np.arange(60.0), np.arange(50.0)), axis=-1).reshape(-1, 2) * 25.0   # 3,000, many ties
    P = np.concatenate([P, P[:40]])                                                              # and duplicates
    assert np.array_equal(g._knn_large(P, 20), g._knn_small(P, 20))


def test_nn_exact_equals_brute_force():
    rng = np.random.default_rng(4)
    tgt = np.round(rng.uniform(0, 100, size=(4000, 2)))          # integer lattice: exact ties
    src = np.round(rng.uniform(0, 100, size=(700, 2))) + 0.5
    d, i = g.nn_exact(src, tgt)
    d0, i0 = orc.nn_bruteforce(src, tgt)
    assert np.array_equal(i, i0) and np.array_equal(d, d0)


def test_regularised_covariance_matches_an_eigh_construction():
    rng = np.random.default_rng(5)
    for _ in range(200):
        th = rng.uniform(-math.pi, math.pi)
        line = rng.uniform(-500, 500, size=(40, 1)) * np.array([[math.cos(th), math.sin(th)]])
        P = line + rng.normal(0, rng.uniform(1, 40), size=(40, 2)) + rng.uniform(-1e4, 1e4, size=2)
        eps = 10.0 ** rng.uniform(-4, -1)
        C = g.estimate_covariances_2d(P, 20, eps)
        for i in range(0, 40, 7):
            nb = P[g.knn_2d(P, 20)[i]]
            cov = np.cov(nb.T, bias=True)
            w, V = np.linalg.eigh(cov)
            if w[1] - w[0] < 1e-6 * w[1]:
                continue                                          # near-isotropic: axis ill-defined
            u = V[:, 1]
            want = np.outer(u, u) + eps * (np.eye(2) - np.outer(u, u))
            assert np.allclose(C[i], [want[0, 0], want[0, 1], want[1, 1]], rtol=0, atol=1e-9)


def test_isotropic_and_degenerate_neighbourhoods_give_the_stated_rule():
    eps = 1e-3
    square = np.array([[0.0, 0.0], [1.0, 0.0], [0.0, 1.0], [1.0, 1.0]])     # cxx = cyy, cxy = 0: phi = 0
    assert np.array_equal(g.estimate_covariances_2d(square, 20, eps), np.tile([1.0, 0.0, eps], (4, 1)))
    two = np.array([[0.0, 0.0], [3.0, 4.0]])                                # fewer than 3 neighbours
    assert np.array_equal(g.estimate_covariances_2d(two, 20, eps), np.tile([1.0, 0.0, 1.0], (2, 1)))
    same = np.zeros((5, 2)) + 7.0                                           # cxx + cyy = 0
    assert np.array_equal(g.estimate_covariances_2d(same, 3, eps), np.tile([1.0, 0.0, 1.0], (5, 1)))
    assert g.estimate_covariances_2d(np.zeros((0, 2)), 20, eps).shape == (0, 3)
    diag = np.array([[0.0, 0.0], [1.0, 1.0], [2.0, 2.0]])                   # along (1, 1) / sqrt(2)
    assert np.allclose(g.estimate_covariances_2d(diag, 3, eps)[0], [(1 + eps) / 2, (1 - eps) / 2, (1 + eps) / 2])


def test_one_step_with_identity_covariances_is_the_point_to_point_gauss_newton_step():
    rng = np.random.default_rng(6)
    B = orc.synth_map(600, dtype=np.float64)
    A = (B[::3] - [30.0, -12.0]) @ _rot(0.02) + rng.normal(0, 3.0, size=(200, 2))
    I = np.tile([1.0, 0.0, 1.0], (len(A), 1)), np.tile([1.0, 0.0, 1.0], (len(B), 1))
    o = g.gicp_extended(A, B, 1, cov_A=I[0], cov_B=I[1], max_corr_dist=150.0)
    d, idx = orc.nn_bruteforce(A, B)
    keep = d < 150.0
    s, b = A[keep], B[idx[keep]]
    c = A.mean(axis=0)
    J = np.zeros((2 * len(s), 3))
    J[0::2, 0], J[0::2, 1] = -(s[:, 1] - c[1]), 1.0
    J[1::2, 0], J[1::2, 2] = s[:, 0] - c[0], 1.0
    x = np.linalg.solve(J.T @ J, J.T @ (b - s).reshape(-1))
    R = _rot(x[0])
    assert o.iterations == 1 and np.array_equal(o.history[0], idx)
    assert np.allclose(o.R_tot, R, atol=1e-13)
    assert np.allclose(o.t_tot, c + x[1:] - R @ c, atol=1e-9)


@pytest.mark.parametrize("th,t", [(0.05, (120.0, -80.0)), (-0.2, (10.0, 300.0))])
def test_noise_free_clouds_recover_the_transform(th, t):
    B = orc.synth_map(3000, dtype=np.float64)
    A = (B[::4] - np.asarray(t)) @ _rot(th)               # R A + t = B exactly
    o = g.gicp_extended(A, B, 50, max_corr_dist=1000.0)
    assert o.rmse < 1e-8 and o.fitness == 1.0
    assert np.allclose(o.R_tot, _rot(th), atol=1e-9) and np.allclose(o.t_tot, t, atol=1e-9)


def test_converged_result_does_not_depend_on_the_pivot():
    # the linear step is the same least-squares problem in other coordinates; applying its rotation
    # about another pivot differs at O(dtheta^2 |c - c'|), so the iterates differ and the fixed point not
    rng = np.random.default_rng(7)
    B = orc.synth_map(2000, dtype=np.float64)
    A = (B[::5] - [50.0, 20.0]) @ _rot(0.04) + rng.normal(0, 4.0, size=(400, 2))
    kw = dict(max_corr_dist=300.0, relative_fitness=0.0, relative_rmse=0.0)
    o1 = g.gicp_extended(A, B, 40, **kw)
    o2 = g.gicp_extended(A, B, 40, pivot=(4000.0, -3000.0), **kw)
    assert np.array_equal(o1.indices, o2.indices) and abs(o1.rmse - o2.rmse) < 1e-9 * o1.rmse
    assert np.allclose(o1.R_tot, o2.R_tot, atol=1e-12) and np.allclose(o1.t_tot, o2.t_tot, atol=1e-8)


def test_a_zero_step_leaves_identical_clouds_exactly_in_place():
    B = orc.synth_map(800, dtype=np.float64)
    o = g.gicp_extended(B[::2], B[::2], 30, max_corr_dist=180.0)
    assert o.iterations == 1 and o.rmse == 0.0 and o.rmse_history == [0.0, 0.0]
    assert np.array_equal(o.R_tot, np.eye(2)) and np.array_equal(o.t_tot, np.zeros(2))
    assert np.array_equal(o.src, B[::2])


def test_degenerate_inputs_of_the_oracle():
    B = orc.synth_map(500, dtype=np.float64)
    o = g.gicp_extended(np.zeros((0, 2)), B, 10, init_pose=(_rot(0.1), np.array([1.0, 2.0])))
    assert o.iterations == 0 and np.isinf(o.rmse) and np.allclose(o.R_tot, _rot(0.1))
    o = g.gicp_extended(B[:50], B + 1e5, 10, max_corr_dist=100.0)         # all gated out
    assert o.iterations == 0 and np.isinf(o.rmse) and o.inliers == 0
    o = g.gicp_extended(B[:1], B, 10)                                      # one point: H is singular
    assert o.iterations == 0 and np.isfinite(o.rmse)


def test_cabi_rejects_bad_gicp_arguments_without_touching_the_gpu():
    import __graft_entry__ as ge
    ge.build()
    from icp_slam_yolo_b200 import _cabi
    L = _cabi.lib()
    p = ctypes.c_void_p(4096)
    assert L.b200icp_estimate_covariances(None, None, 1, 8, _cabi.F64, 20, 1e-3, p, None) == 1
    assert L.b200icp_estimate_covariances(p, None, 1, 8, _cabi.F64, 20, 1e-3, None, None) == 1
    assert L.b200icp_estimate_covariances(p, None, 1, 8, _cabi.F64, 2, 1e-3, p, None) == 1
    assert L.b200icp_estimate_covariances(p, None, 1, 8, _cabi.F64, 33, 1e-3, p, None) == 1
    assert L.b200icp_estimate_covariances(p, None, 1, 8, _cabi.F64, 20, 0.0, p, None) == 1
    assert L.b200icp_estimate_covariances(p, None, 1, 8, 7, 20, 1e-3, p, None) == 1
    assert L.b200icp_estimate_covariances(p, None, -1, 8, _cabi.F64, 20, 1e-3, p, None) == 1
    assert L.b200icp_estimate_covariances(p, None, 1, 65537, _cabi.F64, 20, 1e-3, p, None) == 2
    assert b"pitch" in L.b200icp_last_error()
    opt, out = _cabi.GicpOptions(), _cabi.Outputs()
    assert L.b200icp_gicp_batch(None, 1, ctypes.byref(opt), p, p, ctypes.byref(out), None) == 1
    pr = _cabi.Problem()
    pr.src_points = pr.tgt_points = 4096
    pr.src_pitch, pr.tgt_pitch, pr.dtype = 16, 65536, _cabi.F64
    assert L.b200icp_gicp_batch(ctypes.byref(pr), 1, None, p, p, ctypes.byref(out), None) == 1
    assert L.b200icp_gicp_batch(ctypes.byref(pr), 1, ctypes.byref(opt), None, p, ctypes.byref(out), None) == 1
    assert L.b200icp_gicp_batch(ctypes.byref(pr), 1, ctypes.byref(opt), p, p, ctypes.byref(out), None) == 1
    assert b"required" in L.b200icp_last_error()
    pr.tgt_pitch = 65537
    assert L.b200icp_gicp_batch(ctypes.byref(pr), 1, ctypes.byref(opt), p, p, ctypes.byref(out), None) == 2
    pr.src_pitch, pr.tgt_pitch = 1025, 16
    assert L.b200icp_gicp_batch(ctypes.byref(pr), 1, ctypes.byref(opt), p, p, ctypes.byref(out), None) == 2
    pr.src_pitch, pr.pairing, pr.n_rows = 16, _cabi.PAIR_TRIANGLE, 4
    assert L.b200icp_gicp_batch(ctypes.byref(pr), 7, ctypes.byref(opt), p, p, ctypes.byref(out), None) == 1
    pr.pairing = _cabi.PAIR_EXPLICIT
    assert L.b200icp_gicp_batch(ctypes.byref(pr), 1, ctypes.byref(opt), p, p, ctypes.byref(out), None) == 1
    out.pose_total = out.error = out.iterations = 4096
    pr.pairing = _cabi.PAIR_ROWWISE
    opt.max_iterations = -1
    assert L.b200icp_gicp_batch(ctypes.byref(pr), 1, ctypes.byref(opt), p, p, ctypes.byref(out), None) == 1


def test_slam_config_rejects_an_unknown_registration():
    from icp_slam_yolo_b200.slam import OfflineSlam, SlamConfig
    assert SlamConfig().registration == "p2p"
    with pytest.raises(ValueError, match="registration"):
        OfflineSlam(SlamConfig(registration="plane"))
