"""CPU: the oracle restatement against the reference's golden vectors (parity pin)."""
import math
import os
import zlib

import numpy as np

from oracle import icp_oracle as orc


def test_circle_demo_matches_reference_bitwise(golden):
    """icp.py:55-67 known-answer test: outputs recorded from the unmodified reference."""
    r = orc.icp_extended(golden["demo_A"], golden["demo_B"])          # defaults 20 / 1e-5
    assert r.iterations == 7
    assert np.array_equal(r.src, golden["demo_A_aligned"])
    assert np.array_equal(r.R_last, golden["demo_R_est"])
    assert np.array_equal(r.t_last, golden["demo_t_est"])
    # SURVEY.md §4 spot values
    assert abs(r.errors[0] - 0.34609498386935730) < 1e-15
    assert abs(r.errors[4] - 0.02567312646578419) < 1e-15
    assert np.allclose(r.src[0], [0.8713187041233889, 0.49071755200393774], atol=1e-15)
    Rc, tc = orc.best_fit_transform(golden["demo_A"], r.src)
    assert abs(math.degrees(math.atan2(Rc[1, 0], Rc[0, 0])) - (-0.6122448979591766)) < 1e-9
    assert np.allclose(tc, [-0.502108551471, -0.194645838741], atol=1e-9)


def test_all_scan_pairs_match_reference_bitwise(golden, cart_scans, oracle_pairs):
    """Every consecutive Scan_data_1 pair: src bitwise equal to the reference's icp() output."""
    assert len(oracle_pairs) == 1830
    crc = golden["pair_src_crc32"]
    for p, r in enumerate(oracle_pairs):
        assert zlib.crc32(np.ascontiguousarray(r.src).tobytes()) == crc[p], f"pair {p + 1}"
        assert np.array_equal(r.R_last, golden["pair_R_last"][p])
        assert np.array_equal(r.t_last, golden["pair_t_last"][p])
        assert len(cart_scans[p + 1]) == golden["pair_n_src"][p]
    its = np.array([r.iterations for r in oracle_pairs])
    assert its.min() == 1 and its.max() == 30 and abs(its.mean() - 7.38) < 0.01   # SURVEY.md §6


def test_second_recording_matches_reference_bitwise(golden3, cart_scans3, oracle_pairs3):
    """scan_data_3/ (2,042 consecutive pairs): the oracle reproduces what the unmodified reference
    icp() returned (tests/golden/make_golden_scan3.py) bit for bit."""
    assert len(oracle_pairs3) == 2042
    crc = golden3["pair_src_crc32"]
    for p, r in enumerate(oracle_pairs3):
        assert zlib.crc32(np.ascontiguousarray(r.src).tobytes()) == crc[p], f"pair {p}"
        assert np.array_equal(r.R_last, golden3["pair_R_last"][p]) and np.array_equal(r.t_last, golden3["pair_t_last"][p])
        assert len(cart_scans3[p + 1]) == golden3["pair_n_src"][p] and len(cart_scans3[p]) == golden3["pair_n_tgt"][p]


def test_spot_pairs_full_src(golden, oracle_pairs):
    for k in golden["spot_pairs"]:
        assert np.array_equal(oracle_pairs[k - 1].src, golden[f"spot_src_{k}"])


def test_cumulative_pose_consistent_with_reference_src(golden, cart_scans, oracle_pairs):
    """Quirk Q1: the cumulative pose is implicit in src; the oracle's composed pose must
    reproduce what best_fit_transform(A, src_ref) of the REFERENCE gave."""
    for p in (2, 349, 1074, 0):
        r = oracle_pairs[p]
        th = math.atan2(r.R_tot[1, 0], r.R_tot[0, 0])
        assert abs(th - golden["pair_theta_tot"][p]) < 1e-12
        assert np.allclose(r.t_tot, golden["pair_t_tot"][p], atol=1e-8)
    # SURVEY.md §8c spot values: scan 4->3 and 2->1
    r = oracle_pairs[2]
    assert r.iterations == 8 and abs(r.error - 33.027300367) < 1e-8
    assert abs(math.atan2(r.R_tot[1, 0], r.R_tot[0, 0]) - (-7.511402722180e-03)) < 1e-12
    assert np.allclose(r.t_tot, [-7.273582873339, -4.273236454951], atol=1e-9)
    r = oracle_pairs[0]
    assert r.iterations == 1 and r.error == 0.0 and np.linalg.norm(r.t_tot) < 2e-12


def test_closed_form_and_bruteforce_variants_agree(cart_scans, oracle_pairs):
    """The forms the CUDA kernel evaluates (closed-form Kabsch, brute-force argmin) walk the
    same index history as SVD + KD-tree on real data."""
    for p in list(range(0, 1830, 37)) + [184, 250, 672, 1006, 1062]:
        a = oracle_pairs[p]
        b = orc.icp_extended(cart_scans[p + 1], cart_scans[p], 30, 1e-5, nn="brute", solver="closed")
        assert a.iterations == b.iterations
        assert all(np.array_equal(x, y) for x, y in zip(a.indices, b.indices))
        assert np.allclose(a.R_tot, b.R_tot, atol=1e-13) and np.allclose(a.t_tot, b.t_tot, atol=1e-9)


def test_polar_to_cartesian_vectorised_equals_row_loop(raw_scans):
    for k in list(range(0, 1831, 29)) + [0, 1, 1830]:
        L, V = orc.polar_to_cartesian_loop(raw_scans[k]), orc.polar_to_cartesian(raw_scans[k])
        assert L.shape == V.shape and np.array_equal(L, V)
    assert orc.polar_to_cartesian_loop(np.zeros((0, 3))).size == 0
    assert orc.polar_to_cartesian(np.zeros((0, 3))).shape == (0, 3)


def test_polar_filter_counts(raw_scans, cart_scans):
    n = np.array([len(c) for c in cart_scans])
    assert n.min() == 11 and n.max() == 196 and abs(n.mean() - 136.6) < 0.1    # SURVEY.md §8 a2
    assert np.array_equal(raw_scans[0], raw_scans[1])                          # files 1 and 2 identical


def test_extended_options(cart_scans):
    A, B = cart_scans[3], cart_scans[2]
    base = orc.icp_extended(A, B, 30, 1e-5)
    # identity init pose == no init pose
    same = orc.icp_extended(A, B, 30, 1e-5, init_pose=(np.eye(2), np.zeros(2)))
    # (memory order of the pre-transformed array changes NumPy's summation order: ~1e-13)
    assert np.allclose(base.src, same.src, rtol=0, atol=1e-9) and same.iterations == base.iterations
    # a huge gate keeps everything
    wide = orc.icp_extended(A, B, 30, 1e-5, max_corr_dist=1e9)
    assert np.allclose(base.src, wide.src, rtol=0, atol=1e-9) and wide.fitness == 1.0
    # a tiny gate removes every pair: nothing is counted
    none = orc.icp_extended(A, B, 30, 1e-5, max_corr_dist=1e-9)
    assert none.iterations == 0 and math.isinf(none.error) and np.array_equal(none.src, A)
    gated = orc.icp_extended(A, B, 30, 1e-5, max_corr_dist=150.0)
    assert 0 < gated.fitness <= 1.0 and gated.rmse >= gated.error
    assert orc.icp_extended(A, B, 0).iterations == 0


def test_synthetic_generator_is_seeded_and_recoverable():
    s1, t1, th, tr = orc.synth_room_pair(7)
    s2, t2, _, _ = orc.synth_room_pair(7)
    assert np.array_equal(s1, s2) and np.array_equal(t1, t2) and s1.dtype == np.float32
    r = orc.icp_extended(s1, t1, 30, 1e-5)
    # near-circular rooms sampled at 1 degree let ICP snap to the beam spacing (as in the
    # reference's own circle demo, SURVEY.md §4): recovery is only good to a few degrees
    assert abs(math.atan2(r.R_tot[1, 0], r.R_tot[0, 0]) - th) < 0.06
    assert np.linalg.norm(r.t_tot - tr) < 30.0


def test_reference_form_and_best_fit_match_recorded_reference(golden, cart_scans):
    """icp_reference_form returns what the unmodified icp() returned, and best_fit_transform
    reproduces the reference's best_fit_transform(A, src) (tests/golden/make_golden.py) bit for
    bit, on the reference's own full src arrays of the spot pairs."""
    for p in (2, 99, 672, 1062, 1500):
        A, B = cart_scans[p + 1], cart_scans[p]
        src, R, t = orc.icp_reference_form(A, B, 30, 1e-5)
        assert zlib.crc32(np.ascontiguousarray(src).tobytes()) == golden["pair_src_crc32"][p], f"pair {p}"
        assert np.array_equal(R, golden["pair_R_last"][p]) and np.array_equal(t, golden["pair_t_last"][p])
    for k in golden["spot_pairs"]:
        Rc, tc = orc.best_fit_transform(cart_scans[k], golden[f"spot_src_{k}"])
        assert np.arctan2(Rc[1, 0], Rc[0, 0]) == golden["pair_theta_tot"][k - 1], f"pair {k}"
        assert np.array_equal(tc, golden["pair_t_tot"][k - 1]), f"pair {k}"


def test_c_oracle_matches_numpy_oracle(cart_scans):
    """oracle/icp_oracle.c (brute force + closed form) walks the same index history as the
    SciPy/SVD restatement on real scans, incl. gate and initial pose."""
    from oracle import c_oracle
    for p in (2, 350, 672, 1062):
        A, B = cart_scans[p + 1], cart_scans[p]
        o = orc.icp_extended(A, B, 30, 1e-5)
        c = c_oracle.icp(A, B, 30, 1e-5, history=True)
        assert c["iterations"] == o.iterations
        assert all(np.array_equal(c["history"][i], o.indices[i]) for i in range(o.iterations))
        assert np.allclose(c["pose_total"][:4].reshape(2, 2), o.R_tot, atol=1e-12)
        assert np.allclose(c["pose_total"][4:], o.t_tot, atol=1e-8) and abs(c["error"] - o.error) < 1e-9
    A, B = cart_scans[100], cart_scans[99]
    init = [math.cos(0.01), -math.sin(0.01), math.sin(0.01), math.cos(0.01), 5.0, -3.0]
    o = orc.icp_extended(A, B, 30, 1e-5, init_pose=(np.array(init[:4]).reshape(2, 2), np.array(init[4:])), max_corr_dist=120.0)
    c = c_oracle.icp(A, B, 30, 1e-5, init_pose=init, max_corr_dist=120.0)
    assert c["iterations"] == o.iterations and c["inliers"] == round(o.fitness * len(A))
    assert np.allclose(c["pose_total"][4:], o.t_tot, atol=1e-8) and abs(c["rmse"] - o.rmse) < 1e-9
    idx, d2 = c_oracle.nn_bruteforce(A, B)
    d, i = orc.nn_kdtree(A, B)
    assert np.array_equal(idx, i) and np.allclose(np.sqrt(d2), d, rtol=1e-15)


def test_polar_to_cartesian_restatement_matches_recorded_reference(raw_scans):
    """process.py:38-52: the UNMODIFIED polar_to_cartesian_3d was run on all 1,831 scans of
    Scan_data_1 (tests/golden/make_golden_occupancy.py, process.py imported with a stub open3d);
    point counts and CRC32 of its float64 output must equal the oracle's vectorised and loop
    restatements bit for bit."""
    import zlib
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_occupancy_golden.npz"))
    assert len(raw_scans) == len(g["p2c_count"]) == 1831
    for f, raw in enumerate(raw_scans):
        v = orc.polar_to_cartesian(raw)
        assert len(v) == int(g["p2c_count"][f]), f"scan {f}"
        if len(v):
            assert zlib.crc32(np.ascontiguousarray(v).tobytes()) == int(g["p2c_crc32"][f]), f"scan {f}"
        if f % 97 == 0:
            l = orc.polar_to_cartesian_loop(raw)
            assert np.array_equal(np.asarray(l).reshape(-1, 3), v), f"scan {f} (loop form)"
