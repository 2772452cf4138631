"""The occupancy-grid oracle (oracle/occupancy_oracle.py + .c) against the outputs of the
UNMODIFIED reference (duc/ICP_LIDAR/process.py:86-249) recorded in
tests/golden/reference_occupancy_golden.npz by tests/golden/make_golden_occupancy.py.
Everything here is bit-exact: float32 probabilities, uint8 grey levels, integer cells."""
import os
import zlib

import numpy as np
import pytest

from oracle import occupancy_oracle as occ

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
MAP_H, MAP_W, RES = 833, 1000, 30              # Config.py:7-9,25-26
CENTER = (MAP_W // 2, MAP_H // 2)              # slam_offline.py:320


@pytest.fixture(scope="module")
def gold():
    return np.load(os.path.join(GOLDEN, "reference_occupancy_golden.npz"))


@pytest.fixture(scope="module")
def packed():
    return dict(np.load(os.path.join(GOLDEN, "scan_data_1_packed.npz")))


def _crc(a):
    return zlib.crc32(np.ascontiguousarray(a).tobytes())


def small_case(gold, i):
    par = gold[f"small_{i}_par"]
    return dict(occ=gold[f"small_{i}_occ_in"].copy(), pts=gold[f"small_{i}_pts"], robot=gold[f"small_{i}_robot"],
                center=(int(par[0]), int(par[1])), res=float(par[2]) if par[2] != int(par[2]) else int(par[2]),
                area=int(par[3]), p_occ_inc=float(par[4]), p_free_dec=float(par[5]),
                occ_out=gold[f"small_{i}_occ_out"], img_out=gold[f"small_{i}_img_out"])


def test_bresenham_restatement_and_closed_form(gold):
    ends, offs, cells = gold["bres_ends"], gold["bres_offsets"], gold["bres_cells"]
    for i, e in enumerate(ends):
        e = [int(v) for v in e]
        want = [tuple(int(v) for v in c) for c in cells[offs[i]:offs[i + 1]]]
        assert occ.bresenham_line(*e) == want
        got = [occ.bresenham_cell(*e, k) for k in range(len(want))]
        assert got == want, (e, got[:5], want[:5])
        assert len(want) == max(abs(e[2] - e[0]), abs(e[3] - e[1])) + 1


@pytest.mark.parametrize("impl", ["python", "c"])
def test_small_cases_bit_exact(gold, impl):
    fn = occ.update_occupancy_map if impl == "python" else occ.update_occupancy_map_c
    for i in range(int(gold["small_count"])):
        c = small_case(gold, i)
        image = np.full(c["occ"].shape + (3,), 128, dtype=np.uint8)
        fn(c["occ"], image, c["pts"], c["robot"], c["center"], c["res"],
           p_occ_inc=c["p_occ_inc"], p_free_dec=c["p_free_dec"], area=c["area"])
        assert np.array_equal(c["occ"].view(np.uint32), c["occ_out"].view(np.uint32)), f"case {i}"
        assert np.array_equal(image[:, :, 0], c["img_out"]), f"case {i}"
        assert np.array_equal(image[:, :, 1], c["img_out"]) and np.array_equal(image[:, :, 2], c["img_out"])


def test_replay_of_the_recording_bit_exact(gold, packed):
    """200 frames of Scan_data_1 on the reference's map geometry: the C restatement on every
    frame (CRC at the recorded frames + final arrays), the Python restatement on the first 12."""
    poses = gold["replay_poses"]
    want = {int(f): (int(a), int(b)) for f, a, b in gold["replay_crc"]}
    o_c = np.full((MAP_H, MAP_W), 0.5, dtype=np.float32)
    i_c = np.full((MAP_H, MAP_W, 3), 128, dtype=np.uint8)
    o_p, i_p = o_c.copy(), i_c.copy()
    for f in range(len(poses)):
        pts, robot = occ.replay_frame(packed, poses, f)
        if len(pts) == 0:
            continue
        occ.update_occupancy_map_c(o_c, i_c, pts, robot, CENTER, RES)
        if f < 12:
            occ.update_occupancy_map(o_p, i_p, pts, robot, CENTER, RES)
            assert np.array_equal(o_p.view(np.uint32), o_c.view(np.uint32)) and np.array_equal(i_p, i_c)
        if f in want:
            assert (_crc(o_c), _crc(i_c)) == want[f], f"frame {f}"
    assert np.array_equal(o_c.view(np.uint32), gold["replay_occ_final"].view(np.uint32))
    assert np.array_equal(i_c[:, :, 0], gold["replay_image_final"])
    assert o_c.max() >= 0.65 and o_c.min() < 0.2          # walls stop rays, free space is carved


def test_filter_points_bit_exact(gold):
    for i in range(int(gold["filter_count"])):
        par = gold[f"filter_{i}_par"]
        res = float(par[2]) if par[2] != int(par[2]) else int(par[2])
        kept = occ.filter_points_by_occupancy(gold[f"filter_{i}_pts"], gold[f"filter_{i}_grid"],
                                              (int(par[0]), int(par[1])), res, float(par[3]))
        # the reference returns the kept rows themselves (process.py:226)
        assert np.array_equal(gold[f"filter_{i}_pts"][kept], gold[f"filter_{i}_kept"]), f"case {i}"
        assert 0 < len(kept) < len(gold[f"filter_{i}_pts"])


def test_slam_oracle_composition_tracks_the_recording(packed):
    """oracle/slam_oracle.py (the order of slam_offline.py:318-455 over the pinned oracles): the
    first 80 scans are all registered, the map grows and is re-sampled, free space is carved."""
    from oracle import icp_oracle as orc
    from oracle.slam_oracle import OracleSlam

    class Cfg:                                   # duc/ICP_LIDAR/Config.py:7-21
        resolution_mm_per_pixel = 30; map_width_pixels = 1000; map_height_pixels = 833
        icp_voxel_size = 25.0; icp_threshold = 180.0; max_rmse_threshold = 50.0
        dynamic_distance_threshold = 300.0; local_map_radius_mm = 9000.0; min_icp_map_points = 50
        max_map_points_before_downsample = 1000; min_scan_points = 10; max_iteration = 50; tolerance = 1e-5

    scans = [orc.polar_to_cartesian(occ.unpack_scan(packed, f)) for f in range(2, 82)]
    slam = OracleSlam(Cfg)
    slam.first(scans[0])
    out = [slam.step(s) for s in scans[1:]]
    assert all(o is not None and o[0] and o[1] < 50.0 for o in out)
    assert len(slam.map) > 1000 and np.hypot(*slam.pose[:2, 3]) > 20.0
    assert slam.occ.max() >= 0.65 and slam.occ.min() < 0.2


def test_closed_form_bresenham_randomised():
    """The closed form the device evaluates (floor((2 k minor + major - 1) / (2 major)) minor steps
    after k major steps) against the reference's stepping walk on 4,000 random segments, incl.
    axis-aligned, diagonal and single-cell ones."""
    rng = np.random.Generator(np.random.PCG64(86112))
    for q in range(4000):
        span = [3, 40, 400, 3000][q % 4]
        x0, y0, x1, y1 = (int(v) for v in rng.integers(-span, span + 1, size=4))
        if q % 10 == 0:
            y1 = y0
        elif q % 10 == 1:
            x1 = x0
        elif q % 10 == 2:
            x1, y1 = x0 + (y1 - y0), y1                      # exact diagonal
        line = occ.bresenham_line(x0, y0, x1, y1)
        assert len(line) == max(abs(x1 - x0), abs(y1 - y0)) + 1
        ks = range(len(line)) if len(line) < 64 else list(rng.integers(0, len(line), size=48)) + [0, len(line) - 1]
        for k in ks:
            assert occ.bresenham_cell(x0, y0, x1, y1, int(k)) == line[int(k)], (x0, y0, x1, y1, k)


def test_python_and_c_occupancy_oracles_agree_on_random_cases():
    """300 seeded frames on small grids with arbitrary float32 probabilities (not only the values the
    update itself produces), robots inside / on the border / outside, random parameters."""
    rng = np.random.Generator(np.random.PCG64(172))
    for q in range(300):
        h, w = int(rng.integers(8, 48)), int(rng.integers(8, 48))
        area = int(rng.integers(0, 30))
        res = float(rng.choice([10.0, 30.0, 37.5]))
        center = (int(rng.integers(0, w)), int(rng.integers(0, h)))
        o_p = rng.random((h, w), dtype=np.float32)
        o_p[rng.random((h, w)) < 0.2] = np.float32(0.65)
        i_p = rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8)
        o_c, i_c = o_p.copy(), i_p.copy()
        robot = np.array([rng.uniform(-1.5, 1.5) * w * res, rng.uniform(-1.5, 1.5) * h * res, 0.0])
        pts = np.zeros((int(rng.integers(0, 25)), 3))
        pts[:, :2] = robot[:2] + rng.normal(0, (area + 2) * res, size=(len(pts), 2))
        kw = dict(p_occ_inc=float(rng.choice([0.2, 0.35, 1.5])), p_free_dec=float(rng.choice([0.9, 0.5, 1.0])), area=area)
        occ.update_occupancy_map(o_p, i_p, pts, robot, center, res, **kw)
        occ.update_occupancy_map_c(o_c, i_c, pts, robot, center, res, **kw)
        assert np.array_equal(o_p.view(np.uint32), o_c.view(np.uint32)) and np.array_equal(i_p, i_c), f"case {q}"
