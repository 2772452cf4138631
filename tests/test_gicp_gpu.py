"""2D Generalized ICP on the device (b200icp_estimate_covariances, b200icp_gicp_batch and the Python
layer in icp_slam-yolo_b200/gicp.py) against the CPU oracle oracle/gicp_oracle.py."""
import ctypes

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import gicp_oracle as g        # noqa: E402
from oracle import icp_oracle as orc       # noqa: E402


@pytest.fixture(scope="module")
def pkg():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import icp_slam_yolo_b200 as m
    m.lib()
    return m


def _cov_close(got, want):
    assert got.shape == want.shape
    assert np.all(np.abs(got - want) <= 1e-12 * np.maximum(1.0, np.abs(want)))


def _check_table_covariances(pkg, scans, dtype, k=20, eps=1e-3):
    t = pkg.ScanTable.from_list(scans, dtype=dtype)
    got = pkg.estimate_covariances(t, k, eps).cpu().numpy()
    for r, s in enumerate(scans):
        s = np.asarray(s, dtype=dtype).astype(np.float64)
        _cov_close(got[r, :len(s)], g.estimate_covariances_2d(s, k, eps))
        assert np.all(got[r, len(s):] == 0.0)


def test_covariances_of_the_recording(pkg, cart_scans):
    _check_table_covariances(pkg, cart_scans, np.float64)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_covariances_of_ties_duplicates_and_short_rows(pkg, dtype):
    lattice = np.stack(np.meshgrid(np.arange(13.0), np.arange(11.0)), axis=-1).reshape(-1, 2) * 25.0
    rng = np.random.default_rng(1)
    dup = np.repeat(rng.uniform(-100, 100, size=(30, 2)), 3, axis=0)
    rows = [lattice, dup, lattice[:19], lattice[:5], lattice[:2], lattice[:1], np.zeros((0, 2)),
            rng.uniform(-1e4, 1e4, size=(300, 2))]
    for k in (3, 20, 32):
        _check_table_covariances(pkg, rows, dtype, k=k, eps=1e-2)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_covariances_of_a_large_map(pkg, dtype):
    _check_table_covariances(pkg, [orc.synth_map(18700, dtype=dtype)], dtype)


def _host(res):
    return {k: getattr(res, k).cpu().numpy() for k in ("iterations", "index_history", "pose_total", "rmse", "inliers")}


def _compare(h, p, o, what):
    it = int(h["iterations"][p])
    assert it == o.iterations, f"{what}: iterations {it} vs {o.iterations}"
    for i in range(it):
        n = len(o.history[i])
        assert np.array_equal(h["index_history"][p, i, :n], o.history[i]), f"{what}: correspondences of update {i}"
    pt = h["pose_total"][p]
    th, tho = np.arctan2(pt[2], pt[0]), np.arctan2(o.R_tot[1, 0], o.R_tot[0, 0])
    assert abs(th - tho) < 1e-9 and np.all(np.abs(pt[4:] - o.t_tot) < 1e-6), what
    rm = float(h["rmse"][p])
    assert (np.isinf(rm) and np.isinf(o.rmse)) or abs(rm - o.rmse) <= 1e-9 * max(o.rmse, 1e-9), what
    assert int(h["inliers"][p]) == o.inliers, what


@pytest.mark.parametrize("which", ["scan_data_1", "scan_data_3"])
def test_gicp_consecutive_on_the_recordings(pkg, which, request):
    scans = request.getfixturevalue("cart_scans" if which == "scan_data_1" else "cart_scans3")
    t = pkg.ScanTable.from_list(scans)
    res = pkg.gicp_consecutive(t, max_iterations=30, max_corr_dist=180.0, want_history=True)
    h = _host(res)
    covs = [g.estimate_covariances_2d(s) for s in scans]
    for p in range(len(scans) - 1):
        o = g.gicp_extended(scans[p + 1], scans[p], 30, max_corr_dist=180.0, cov_A=covs[p + 1], cov_B=covs[p])
        _compare(h, p, o, f"{which} pair {p}")


def _single(pkg, A, B, max_iterations, gate, init):
    s, t = pkg.ScanTable(torch.from_numpy(A[None]).cuda()), pkg.ScanTable(torch.from_numpy(B[None]).cuda())
    ip = torch.from_numpy(np.concatenate([init[0].reshape(4), init[1]])[None]).cuda()
    return pkg.gicp_pairs(s, t, pkg.estimate_covariances(s), pkg.estimate_covariances(t), n_pairs=1,
                          max_iterations=max_iterations, max_corr_dist=gate, init_pose=ip, want_history=True,
                          want_indices=True, want_src=True)


@pytest.mark.parametrize("m", [4095, 4096, 4097, 12000, 18700])
def test_single_registrations_of_slam_shape(pkg, m):
    B = orc.synth_map(m, dtype=np.float64)
    A = orc.synth_scan_for_map(194, dtype=np.float64)
    init = (np.array([[np.cos(0.015), -np.sin(0.015)], [np.sin(0.015), np.cos(0.015)]]), np.array([30.0, -15.0]))
    res = _single(pkg, A, B, 50, 180.0, init)
    o = g.gicp_extended(A, B, 50, max_corr_dist=180.0, init_pose=init)
    _compare(_host(res), 0, o, f"m = {m}")
    assert np.array_equal(res.indices[0].cpu().numpy(), o.indices)
    assert np.allclose(res.src_final[0].cpu().numpy(), o.src, atol=1e-6)
    assert o.iterations > 2 and o.fitness > 0.9


def test_a_duplicate_in_a_later_tile_loses_to_the_lower_index(pkg):
    B = orc.synth_map(9000, dtype=np.float64)
    B[6000] = B[100]                                  # tile 1 holds an exact copy of a tile-0 point
    B[8500] = B[5000]                                 # tile 2 holds a copy of a tile-1 point
    A = np.concatenate([B[[100, 5000]], orc.synth_scan_for_map(60, dtype=np.float64)])
    res = _single(pkg, A, B, 0, 0.0, (np.eye(2), np.zeros(2)))
    idx = res.indices[0].cpu().numpy()
    assert idx[0] == 100 and idx[1] == 5000
    assert np.array_equal(idx, g.nn_exact(A, B)[1])
    assert int(res.iterations[0]) == 0 and float(res.rmse[0]) >= 0.0


def test_degenerate_pairs(pkg):
    dev = "cuda"
    B = orc.synth_map(600, dtype=np.float64)
    eye = (np.eye(2), np.zeros(2))
    # n = 0 and m = 0 in one ragged batch, with an initial pose
    src = pkg.ScanTable.from_list([np.zeros((0, 2)), B[:50]], pitch=64)
    tgt = pkg.ScanTable.from_list([B, np.zeros((0, 2))], pitch=600)
    ip = torch.tensor([[0.0, -1.0, 1.0, 0.0, 5.0, 6.0]] * 2, dtype=torch.float64, device=dev)
    res = pkg.gicp_pairs(src, tgt, pkg.estimate_covariances(src), pkg.estimate_covariances(tgt), init_pose=ip,
                         want_src=True)
    assert res.iterations.tolist() == [0, 0] and torch.isinf(res.rmse).all() and torch.isinf(res.error).all()
    assert torch.equal(res.pose_total, ip)
    assert np.allclose(res.src_final[1, :50].cpu().numpy(), B[:50] @ np.array([[0.0, -1.0], [1.0, 0.0]]).T + [5, 6])
    cases = {
        "gated out": (B[:50] + 1e5, B, 100.0),
        "identical": (B, B, 180.0),
        "collinear": (np.c_[np.arange(40.0) * 10, np.zeros(40)], np.c_[np.arange(60.0) * 10 - 97, np.zeros(60) + 3], 180.0),
        "one point": (B[7:8] + 2.0, B, 180.0),
    }
    for name, (A, Bt, gate) in cases.items():
        res = _single(pkg, A, Bt, 30, gate, eye)
        o = g.gicp_extended(A, Bt, 30, max_corr_dist=gate)
        _compare(_host(res), 0, o, name)
    assert g.gicp_extended(B[:50] + 1e5, B, 30, max_corr_dist=100.0).iterations == 0
    assert g.gicp_extended(B[7:8] + 2.0, B, 30).iterations == 0           # singular H: no update
    # a source pitch beyond the CTA is rejected before any launch
    s = pkg.ScanTable(torch.zeros((1, 1025, 2), dtype=torch.float64, device=dev))
    t = pkg.ScanTable(torch.zeros((1, 16, 2), dtype=torch.float64, device=dev))
    with pytest.raises(pkg.B200IcpError, match="UNSUPPORTED_SHAPE"):
        pkg.gicp_pairs(s, t, torch.zeros((1, 1025, 3), dtype=torch.float64, device=dev),
                       torch.zeros((1, 16, 3), dtype=torch.float64, device=dev))
    from icp_slam_yolo_b200 import _cabi
    pr = _cabi.Problem()
    pr.src_points = pr.tgt_points = s.points.data_ptr()
    pr.src_pitch, pr.tgt_pitch, pr.dtype = 1025, 16, _cabi.F64
    opt, out = _cabi.GicpOptions(), _cabi.Outputs()
    assert pkg.lib().b200icp_gicp_batch(ctypes.byref(pr), 1, ctypes.byref(opt), ctypes.c_void_p(4096),
                                        ctypes.c_void_p(4096), ctypes.byref(out), None) == 2


def test_registration_gicp_and_the_slam_loop(pkg, cart_scans):
    from icp_slam_yolo_b200.slam import OfflineSlam, SlamConfig
    cfg = SlamConfig(registration="gicp")
    scans = [np.c_[s, np.zeros(len(s))] for s in cart_scans[2:132]]     # scans 3 .. 132 of Scan_data_1
    rm, T = pkg.registration_gicp(scans[1], scans[0], 180.0, 25.0)
    a, b = orc.voxel_down_sample_2d(scans[1][:, :2], 25.0), orc.voxel_down_sample_2d(scans[0][:, :2], 25.0)
    o = g.gicp_extended(a, b, 50, max_corr_dist=180.0)
    assert abs(rm - o.rmse) < 1e-6 and np.allclose(T[:2, :2], o.R_tot, atol=1e-9) and np.allclose(T[:2, 3], o.t_tot, atol=1e-6)
    rm9, T9 = pkg.registration_gicp(scans[1][:9], scans[0])
    assert np.isinf(rm9) and np.array_equal(T9, np.eye(4))
    dev, ora = OfflineSlam(cfg), g.GicpOracleSlam(cfg)
    dev.first_scan(scans[0])
    ora.first(scans[0])
    accepted = 0
    for k, s in enumerate(scans[1:]):
        r = dev.step(s)
        o = ora.step(s)
        assert (r is None) == (o is None), f"frame {k}"
        if r is None:
            continue
        assert r.accepted == o[0], f"frame {k}: rmse {r.rmse} vs {o[1]}"
        assert abs(r.rmse - o[1]) < 1e-6 or (np.isinf(r.rmse) and np.isinf(o[1])), f"frame {k}"
        assert np.allclose(r.pose, ora.pose, atol=1e-6), f"frame {k}"
        got = dev.global_map.cpu().numpy()
        assert got.shape == ora.map.shape and np.allclose(got, ora.map, atol=1e-6), f"frame {k}"
        accepted += int(r.accepted)
    assert accepted >= 100
    assert np.array_equal(dev.grid.probs_numpy().view(np.uint32), ora.occ.view(np.uint32))
