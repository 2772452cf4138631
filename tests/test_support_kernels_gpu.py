"""Edge cases of the kernels around registration in the SLAM loop: point selection (local-map crop,
dynamic-point removal), the voxel grid, pose chaining, matched-row best fit and scan preparation.

Every case compares the CUDA result with a plain high-precision reference of the same operation:
NumPy float64 in the reference's operation order where the kernel claims bit-equality, np.longdouble
(64-bit significand) where its claim is a tolerance.  The cases sit where such kernels go wrong:
decision boundaries, integer ranges, the multi-segment paths of the single-CTA scans and degenerate
geometry.
"""
import math
from fractions import Fraction

import numpy as np
import pytest
import torch

from oracle import icp_oracle as orc

pytestmark = pytest.mark.gpu

EPS = float(np.finfo(np.float64).eps)
LD = np.longdouble


@pytest.fixture(scope="module")
def b200():
    import icp_slam_yolo_b200 as m
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    m.lib()
    assert np.finfo(LD).eps < 1e-18, "the longdouble references need a 64-bit significand"
    return m


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


# ---------------------------------------------------------------------------------------
# A. point selection: b200icp_select_points (crop_local_map: mode 1, remove_dynamic_points: mode 0)
# ---------------------------------------------------------------------------------------
def _crop_ref(pts, centre, radius):
    """mainn.py:300-303 in NumPy's order: (p - c)**2 rounded per axis, then one add."""
    p = np.asarray(pts, dtype=np.float64)
    return np.asarray(pts)[np.sum((p - np.array(centre, dtype=np.float64)) ** 2, axis=1) < float(radius) ** 2]


def _fma_keep(pts, centre, thr):
    """keep/drop of the contracted form fma(dx, dx, dy*dy) < thr, evaluated exactly (one rounding)."""
    out = np.empty(len(pts), dtype=bool)
    for i, (x, y) in enumerate(np.asarray(pts, dtype=np.float64)):
        dx, dy = float(x) - centre[0], float(y) - centre[1]
        out[i] = float(Fraction(dx) * Fraction(dx) + Fraction(dy * dy)) < thr
    return out


def _ring(rng, centre, radius, n, quadrant, ulps=4):
    """n points whose squared distance from `centre` lies within a few ulps of radius**2."""
    th = rng.uniform(quadrant * np.pi / 2, (quadrant + 1) * np.pi / 2, n)
    rr = radius * (1.0 + rng.integers(-ulps, ulps + 1, n) * EPS)
    return np.stack([centre[0] + rr * np.cos(th), centre[1] + rr * np.sin(th)], axis=1)


_BAND_CIRCLES = [((1500.0, -700.0), 6000.0), ((0.0, 0.0), 1000.0),
                 ((-12345.678, 9876.54321), 250.0), ((100000.1, -30000.0), 37.5)]


def test_crop_boundary_band_float64(b200):
    """Points within a few ulps of the crop circle: the kept rows equal NumPy's, in order, and the
    set provably separates the rounded form from the contracted (FMA) one."""
    rng = np.random.default_rng(11)
    fma_disagree = 0
    for centre, radius in _BAND_CIRCLES:
        pts = np.concatenate([_ring(rng, centre, radius, 1000, q) for q in range(4)])
        if centre == (1500.0, -700.0):       # kept by fma(dx, dx, dy*dy), dropped by NumPy
            pts = np.concatenate([pts, [[-2991.0520870178234, -4678.749948374847]]])
        rng.shuffle(pts)
        ref = _crop_ref(pts, centre, radius)
        assert 0 < len(ref) < len(pts)
        got = b200.crop_local_map(_dev(pts), centre, radius, min_points=0).cpu().numpy()
        assert np.array_equal(got, ref), f"centre {centre}, radius {radius}"
        d2 = np.sum((pts - np.array(centre)) ** 2, axis=1)
        fma_disagree += int(np.sum(_fma_keep(pts, centre, radius ** 2) != (d2 < radius ** 2)))
    assert fma_disagree > 0, "the point set does not probe the band where an FMA would decide differently"


def test_crop_boundary_float32(b200):
    """float32 tables are measured in float64 of the float32 values: radii whose square lands on
    (or one ulp next to) a point's squared distance."""
    rng = np.random.default_rng(12)
    centre = (1234.5678901, -987.654321)
    pts = _ring(rng, centre, 3000.0, 4000, 0).astype(np.float32)
    pts = np.concatenate([pts] + [_ring(rng, centre, 3000.0, 1000, q).astype(np.float32) for q in (1, 2, 3)])
    d2 = np.sum((pts.astype(np.float64) - np.array(centre)) ** 2, axis=1)
    t = _dev(pts)
    for j in rng.choice(len(pts), 12, replace=False):
        r0 = math.sqrt(d2[j])
        for radius in (np.nextafter(r0, 0.0), r0, np.nextafter(r0, np.inf)):
            ref = _crop_ref(pts, centre, float(radius))
            got = b200.crop_local_map(t, centre, float(radius), min_points=0).cpu().numpy()
            assert got.dtype == np.float32 and np.array_equal(got, ref), f"radius {radius!r}"


def _lattice_rings(rng, d, centres, per):
    """Previous scan: a lattice of spacing 8 d.  Current scan: `per` points at distance ~d around
    each lattice point (so that point is the unique nearest neighbour), plus 4 at exactly d on the
    axes.  Returns (current, previous, squared NN distance in NumPy's order)."""
    g = int(math.ceil(math.sqrt(centres)))
    ij = np.stack(np.meshgrid(np.arange(g), np.arange(g), indexing="ij"), -1).reshape(-1, 2)[:centres]
    prev = (ij * 8.0 * d - 4000.0).astype(np.float64)
    th = rng.uniform(-np.pi, np.pi, (centres, per))
    off = np.concatenate([d * np.stack([np.cos(th), np.sin(th)], -1),
                          np.broadcast_to([[d, 0.0], [-d, 0.0], [0.0, d], [0.0, -d]], (centres, 4, 2))], axis=1)
    cur = (prev[:, None, :] + off).reshape(-1, 2)
    own = np.repeat(prev, per + 4, axis=0)
    key = (cur[:, 0] - own[:, 0]) ** 2 + (cur[:, 1] - own[:, 1]) ** 2
    perm = rng.permutation(len(cur))
    return cur[perm], prev, key[perm]


@pytest.mark.parametrize("route,centres,per", [("pair-kernel NN", 64, 12), ("scan-to-map search", 4900, 3)])
def test_dynamic_point_removal_at_the_threshold(b200, route, centres, per):
    """mode 0 keeps key < d**2: NN distances exactly d (dropped) and one ulp either side, through
    both searches that produce the key (<= 1,024 x 4,096 points: the pair kernel; larger: scan-to-map)."""
    d = 250.0
    cur, prev, key = _lattice_rings(np.random.default_rng(13), d, centres, per)
    lib = b200.lib()
    small = len(cur) <= lib.b200icp_max_src_pitch() and len(prev) <= lib.b200icp_max_tgt_pitch()
    assert small == (route == "pair-kernel NN")
    thr = d * d
    for k in (np.nextafter(thr, 0.0), thr, np.nextafter(thr, np.inf)):
        assert np.sum(key == k) > 0, f"no point with squared NN distance {k!r}"
    got = b200.remove_dynamic_points(_dev(cur), _dev(prev), d).cpu().numpy()
    assert np.array_equal(got, cur[key < thr])


_SIZES = [0, 1, 255, 256, 1023, 1024, 1025, 3_000_017]


@pytest.mark.parametrize("n", _SIZES)
def test_select_sizes_and_paths(b200, n):
    """Every path of count -> scan -> scatter: a partial last CTA, exactly full CTAs, and more than
    1,024 CTAs (3,000,017 points: the scan gives every thread a segment of 3 blocks).  Crop
    (mode 1) with some, all and none kept; key threshold (mode 0)."""
    rng = np.random.default_rng(100 + n)
    pts = rng.uniform(-1e4, 1e4, (n, 2))
    t = _dev(pts)
    for centre, radius in (((123.4, -567.8), 7000.0), ((0.0, 0.0), 1e6), ((5e4, 5e4), 1.0)):
        got = b200.crop_local_map(t, centre, radius, min_points=0).cpu().numpy()
        assert np.array_equal(got, _crop_ref(pts, centre, radius)), f"n={n}, radius {radius}"
    if n >= 1024:
        assert 0 < len(_crop_ref(pts, (123.4, -567.8), 7000.0)) < n
    key = rng.uniform(0.0, 1.0, n)
    got = b200.mapping._select(t, 0, _dev(key), 0.0, 0.0, 0.5).cpu().numpy()
    assert np.array_equal(got, pts[key < 0.5])
    if n <= 1025:
        p32 = pts.astype(np.float32)
        got = b200.crop_local_map(_dev(p32), (123.4, -567.8), 7000.0, min_points=0).cpu().numpy()
        assert np.array_equal(got, _crop_ref(p32, (123.4, -567.8), 7000.0))


@pytest.mark.parametrize("inside", [49, 50])
def test_crop_min_points_fallback(b200, inside):
    """Fewer than min_points = 50 survivors: the whole map (mainn.py:305-308)."""
    rng = np.random.default_rng(inside)
    near = rng.uniform(-100.0, 100.0, (inside, 2))
    far = rng.uniform(5000.0, 9000.0, (500, 2))
    pts = np.concatenate([near, far])
    rng.shuffle(pts)
    got = b200.crop_local_map(_dev(pts), (0.0, 0.0), 200.0).cpu().numpy()
    want = pts if inside < 50 else _crop_ref(pts, (0.0, 0.0), 200.0)
    assert np.array_equal(got, want) and len(want) == (len(pts) if inside < 50 else 50)


# ---------------------------------------------------------------------------------------
# B. voxel grid: b200icp_voxel_downsample against oracle.icp_oracle.voxel_down_sample_2d
# ---------------------------------------------------------------------------------------
def _voxel_check(b200, pts, voxel):
    """float64: bit-exact (both sides sum each cell sequentially in input order and scale by
    1/count).  float32: the same float64 means rounded once to float32."""
    pts = np.ascontiguousarray(pts, dtype=np.float64)
    ref = orc.voxel_down_sample_2d(pts, voxel)
    got = b200.voxel_down_sample(_dev(pts), voxel).cpu().numpy()
    assert got.shape == ref.shape and np.array_equal(got, ref), f"float64, voxel {voxel}"
    p32 = pts.astype(np.float32)
    ref32 = orc.voxel_down_sample_2d(p32, voxel).astype(np.float32)
    got32 = b200.voxel_down_sample(_dev(p32), voxel).cpu().numpy()
    assert got32.dtype == np.float32 and got32.shape == ref32.shape and np.array_equal(got32, ref32), \
        f"float32, voxel {voxel}"
    return ref


def test_voxel_signs_and_cell_edges(b200):
    """Negative coordinates, -0.0 and points exactly on cell edges k * voxel for both signs."""
    k = np.arange(-6, 7, dtype=np.float64)
    for voxel in (0.25, 0.1, 25.0):
        edges = np.stack(np.meshgrid(k * voxel, k[::-1] * voxel), -1).reshape(-1, 2)
        rng = np.random.default_rng(int(voxel * 100))
        inner = rng.uniform(-6 * voxel, 6 * voxel, (300, 2))
        zeros = np.array([[-0.0, 0.0], [0.0, -0.0], [-0.0, -0.0], [np.nextafter(0.0, -1.0), -0.0]])
        ref = _voxel_check(b200, np.concatenate([edges, inner, zeros, edges[::3]]), voxel)
        assert len(ref) > 100


def test_voxel_one_cell_and_all_distinct(b200):
    rng = np.random.default_rng(21)
    one = rng.uniform(0.0, 25.0, (200_000, 2)) - [50.0, 75.0]      # all in cell (-2, -3)
    assert len(_voxel_check(b200, one, 25.0)) == 1
    ij = rng.permutation(np.stack(np.meshgrid(np.arange(-300, 300), np.arange(-200, 200)), -1).reshape(-1, 2))
    distinct = (ij + rng.uniform(0.01, 0.99, ij.shape)) * 25.0
    assert len(_voxel_check(b200, distinct, 25.0)) == len(distinct)


@pytest.mark.parametrize("n", [1, 256, 257, 1025, 2_000_003])
def test_voxel_sizes(b200, n):
    """The rank scan is one CTA: 2,000,003 points give every thread ~1,954 flags."""
    rng = np.random.default_rng(n)
    pts = rng.normal(0.0, 4000.0, (n, 2))
    ref = _voxel_check(b200, pts, 20.0)
    if n > 1000:
        assert len(ref) < n


def test_voxel_cells_beyond_32_bits(b200):
    """Cell indices are int64 per axis: cells 2^32 apart stay apart, and the output is ordered by
    the full (cell_y, cell_x)."""
    a = np.array([[0.0005, 0.0], [0.0005 + 4294.967296, 0.0], [0.0, 0.0005 + 4294.967296], [0.0005, 0.0]])
    ref = _voxel_check(b200, a, 1e-6)
    assert len(ref) == 3
    rng = np.random.default_rng(22)
    cloud = rng.uniform(-1e4, 1e4, (50_000, 2))
    shifted = np.concatenate([cloud[:2000], cloud[:2000] + [4294.967296, 0.0], cloud[:2000] - [0.0, 4294.967296]])
    for pts in (cloud, shifted):
        _voxel_check(b200, pts, 1e-6)


def test_voxel_skips_non_finite(b200):
    rng = np.random.default_rng(23)
    pts = rng.uniform(-100.0, 100.0, (3000, 2))
    bad = rng.choice(len(pts), 300, replace=False)
    pts[bad[:100], 0] = np.nan
    pts[bad[100:150], 1] = np.inf
    pts[bad[150:200], 0] = -np.inf
    pts[bad[200:], :] = [np.nan, -np.inf]
    pts[0] = [0.5, 0.5]
    pts[1] = [np.nan, 0.5]                  # same cell as row 0 if NaN were cast to cell 0
    ref = _voxel_check(b200, pts, 10.0)
    assert np.all(np.isfinite(ref))
    only_bad = np.array([[np.nan, 1.0], [np.inf, np.inf], [1.0, -np.inf]])
    assert _voxel_check(b200, only_bad, 10.0).shape == (0, 2)


# ---------------------------------------------------------------------------------------
# C. pose chaining: b200icp_chain_poses and the NumPy branch of chain_poses
# ---------------------------------------------------------------------------------------
def _poses(rng, n):
    th = rng.uniform(-np.pi, np.pi, n)
    c, s = np.cos(th), np.sin(th)
    t = rng.uniform(-1e4, 1e4, (n, 2))
    return np.stack([c, -s, s, c, t[:, 0], t[:, 1]], axis=1), th


def _chain_ref(p):
    """out[0] = I, out[k+1] = out[k] o p[k] in longdouble, as an inclusive Hillis-Steele scan: each
    entry is an associative regrouping of the same product, with rounding ~log2(n) * 2^-64."""
    n = len(p)
    R = p[:, :4].astype(LD).reshape(n, 2, 2)
    t = p[:, 4:].astype(LD)
    s = 1
    while s < n:
        Ra, ta = R[:-s], t[:-s]                    # earlier prefix: applied after (left factor)
        Rb, tb = R[s:], t[s:]
        t = np.concatenate([t[:s], np.einsum("kij,kj->ki", Ra, tb) + ta])
        R = np.concatenate([R[:s], np.einsum("kij,kjl->kil", Ra, Rb)])
        s *= 2
    out = np.zeros((n + 1, 6), dtype=LD)
    out[0] = [1, 0, 0, 1, 0, 0]
    out[1:, :4] = R.reshape(n, 4)
    out[1:, 4:] = t
    return out


# A composed entry r = a b + c d with unit rows/columns is within sqrt(2) eps of the exact value of
# its rounded factors (one FMA + one rounding); an output of depth k is the product of k factors, so
# its rotation is within ~sqrt(2) k eps and its translation within ~sqrt(2) k eps * sum |t_j| (the
# rotation error of every prefix scales each later translation).  CHAIN_C = 4 leaves 2x for the
# shuffle-scan regrouping and the reference's own (2^-64) rounding.
CHAIN_C = 4.0


@pytest.mark.parametrize("n", [0, 1, 2, 31, 32, 33, 1023, 1024, 1025, 2049, 5000, 1_000_003])
def test_chain_poses_every_row(b200, n):
    rng = np.random.default_rng(1000 + n)
    p, th = _poses(rng, n)
    ref = _chain_ref(p)
    got = b200.chain_poses(_dev(p))
    host = b200.chain_poses(p)
    assert got.shape == host.shape == (n + 1, 6)
    assert np.array_equal(got[0], [1, 0, 0, 1, 0, 0]) and np.array_equal(host[0], [1, 0, 0, 1, 0, 0])
    k = np.arange(n + 1, dtype=np.float64)
    tol_r = CHAIN_C * (k + 1) * EPS
    tsum = np.concatenate([[0.0], np.cumsum(np.abs(p[:, 4:]).sum(axis=1))])
    tol_t = CHAIN_C * (k + 1) * EPS * np.maximum(1.0, tsum)
    for name, out in (("device", got), ("host", host)):
        er = np.abs(out[:, :4] - ref[:, :4]).max(axis=1).astype(np.float64)
        et = np.abs(out[:, 4:] - ref[:, 4:]).max(axis=1).astype(np.float64)
        assert np.all(er <= tol_r), f"{name}: rotation of row {int(np.argmax(er / tol_r))}"
        assert np.all(et <= tol_t), f"{name}: translation of row {int(np.argmax(et / tol_t))}"
    er = np.abs(got - host)
    assert np.all(er[:, :4].max(axis=1) <= 2 * tol_r) and np.all(er[:, 4:].max(axis=1) <= 2 * tol_t)
    # the angle of every row against the exact sum of the input angles, modulo 2 pi
    rows = np.unique(np.linspace(0, n, min(n + 1, 2000)).astype(np.int64))
    for r in rows:
        want = math.fsum(th[:r])
        a = math.atan2(got[r, 2], got[r, 0])
        diff = math.remainder(a - want, 2 * math.pi)
        assert abs(diff) <= CHAIN_C * (r + 1) * EPS + 4 * EPS * abs(want), f"angle of row {r}"


# ---------------------------------------------------------------------------------------
# D. matched-row best fit: b200icp_best_fit_batch (best_fit, best_fit_transform)
# ---------------------------------------------------------------------------------------
def _fit_ref(A, B):
    """Closed-form 2D Kabsch in longdouble with two-pass centring; A, B [n, 2] (rows matched).
    Returns (R 2x2, t, tolerance on R, tolerance on t) as float64.

    The kernel sums the products of the points taken relative to each cloud's first point in
    float64: ceil(n/32) sequential terms per lane and 5 shuffle levels.  Its error on (num, den) is
    within depth * eps times the sum of the magnitudes it adds, so the rotation is within
    4 (depth + 4) eps kappa, kappa = those magnitudes over hypot(num, den); the translation adds the
    rotation error times |cA| and a few roundings of the centroids."""
    a, b = np.asarray(A, dtype=np.float64), np.asarray(B, dtype=np.float64)
    n = len(a)
    al, bl = a.astype(LD), b.astype(LD)
    ca, cb = al.mean(axis=0), bl.mean(axis=0)
    p, q = al - ca, bl - cb
    h = p.T @ q
    num, den = h[0, 1] - h[1, 0], h[0, 0] + h[1, 1]
    hyp = np.sqrt(num * num + den * den)
    c, s = (LD(1), LD(0)) if hyp == 0 else (den / hyp, num / hyp)
    R = np.array([[c, -s], [s, c]], dtype=LD)
    t = cb - R @ ca
    ax, qx = np.abs(a - a[0]), np.abs(b - b[0])
    mag = float(np.sum(np.hypot(ax[:, 0], ax[:, 1]) * np.hypot(qx[:, 0], qx[:, 1])) +
                np.hypot(*ax.sum(0)) * np.hypot(*qx.sum(0)) / n)
    kappa = mag / float(hyp) if hyp > 0 else 0.0
    depth = -(-n // 32) + 5
    tol_r = 4 * (depth + 4) * EPS * max(kappa, 1.0)
    tol_t = tol_r * float(np.hypot(*ca)) + 8 * EPS * (float(np.hypot(*ca) + np.hypot(*cb))) + \
        2 * depth * EPS * float(np.mean(np.hypot(ax[:, 0], ax[:, 1])) + np.mean(np.hypot(qx[:, 0], qx[:, 1])))
    return R.astype(np.float64), t.astype(np.float64), tol_r, max(tol_t, 4 * EPS)


def _check_fit(pose, A, B, what, svd=True):
    R, t, tol_r, tol_t = _fit_ref(A, B)
    Rg, tg = pose[:4].reshape(2, 2), pose[4:]
    assert np.abs(Rg - R).max() <= tol_r, f"{what}: R off by {np.abs(Rg - R).max():.3g} > {tol_r:.3g}"
    assert np.abs(tg - t).max() <= tol_t, f"{what}: t off by {np.abs(tg - t).max():.3g} > {tol_t:.3g}"
    if svd:                 # the reference's own SVD solve (float64, icp.py:5-26)
        Ro, to = orc.best_fit_transform(np.asarray(A, np.float64), np.asarray(B, np.float64))
        scale = 1.0 + np.abs(np.asarray(B, np.float64)).max() + np.abs(np.asarray(A, np.float64)).max()
        assert np.abs(Rg - Ro).max() <= 1e-10 and np.abs(tg - to).max() <= 1e-10 * scale, f"{what}: SVD oracle"


def _rigid(A, theta, t):
    c, s = math.cos(theta), math.sin(theta)
    return A @ np.array([[c, -s], [s, c]]).T + t


def test_best_fit_degenerate_and_special_geometry(b200):
    rng = np.random.default_rng(31)
    cases = []
    a1 = np.array([[123.25, -77.5]])
    cases.append(("n = 1", a1, np.array([[-5.0, 1000.125]]), True))
    same = np.repeat([[300.5, -20.25]], 40, axis=0)
    cases.append(("identical points (H = 0)", same, same + [7.0, -3.0], True))
    line = np.outer(rng.uniform(-2000, 2000, 60), [0.6, 0.8]) + [10.0, 20.0]
    cases.append(("collinear", line, _rigid(line, 0.7, [40.0, -15.0]), True))
    cloud = rng.normal(0.0, 1500.0, (300, 2))
    cases.append(("180 degree turn", cloud, -cloud, True))
    aniso = rng.normal(0.0, 1.0, (400, 2)) * [3000.0, 700.0]
    aniso = _rigid(aniso, 0.4, [0.0, 0.0])
    mirror = aniso * [-1.0, 1.0] + [250.0, -90.0]
    cases.append(("mirrored cloud", aniso, mirror, True))
    far = rng.uniform(0.0, 1.0, (500, 2)) + [7e5, 7e5]
    cases.append(("clouds 1e6 mm apart, 1 mm spread", far, _rigid(far, 0.3, [-7e5, -2e5]), True))
    noisy = rng.normal(0, 2000, (1000, 2))
    cases.append(("noisy rigid motion", noisy, _rigid(noisy, -2.5, [30.0, 40.0]) + rng.normal(0, 5, (1000, 2)), True))
    poses = b200.best_fit(b200.ScanTable.from_list([c[1] for c in cases]),
                          b200.ScanTable.from_list([c[2] for c in cases])).cpu().numpy()
    for k, (what, A, B, svd) in enumerate(cases):
        _check_fit(poses[k], A, B, what, svd)
    assert np.array_equal(poses[0], [1, 0, 0, 1, -5.0 - 123.25, 1000.125 + 77.5])
    assert np.array_equal(poses[1, :4], [1, 0, 0, 1])
    R, t = b200.best_fit_transform(cases[5][1], cases[5][2])          # the single-pair wrapper
    _check_fit(np.concatenate([R.reshape(4), t]), cases[5][1], cases[5][2], "best_fit_transform, far")


def test_best_fit_ragged_and_float32(b200):
    """Rows of different lengths use the first min(src_len, tgt_len) points of each."""
    rng = np.random.default_rng(32)
    P, Q = [], []
    for ns, nt in ((100, 37), (5, 300), (64, 64), (33, 1), (1000, 999)):
        A, B = rng.normal(0, 3000, (ns, 2)), rng.normal(0, 3000, (nt, 2))
        m = min(ns, nt)
        B[:m] = _rigid(A[:m], rng.uniform(-3, 3), rng.uniform(-1e3, 1e3, 2))
        P.append(A); Q.append(B)
    for dt in (np.float64, np.float32):
        Pd, Qd = [p.astype(dt) for p in P], [q.astype(dt) for q in Q]
        poses = b200.best_fit(b200.ScanTable.from_list(Pd, dtype=dt),
                              b200.ScanTable.from_list(Qd, dtype=dt)).cpu().numpy()
        for k in range(len(P)):
            m = min(len(P[k]), len(Q[k]))
            _check_fit(poses[k], Pd[k][:m], Qd[k][:m], f"{dt.__name__} pair {k}", svd=m > 1)


def test_best_fit_large_pitch_and_many_pairs(b200):
    rng = np.random.default_rng(33)
    A = rng.normal(0, 5000, (200_000, 2))
    B = _rigid(A, 1.1, [-300.0, 4000.0]) + rng.normal(0, 3, A.shape)
    pose = b200.best_fit(b200.ScanTable(_dev(A[None])), b200.ScanTable(_dev(B[None]))).cpu().numpy()
    _check_fit(pose[0], A, B, "200,000 points")
    n_pairs = 10_000
    A3 = rng.uniform(-3000, 3000, (n_pairs, 3, 2))
    th = rng.uniform(-np.pi, np.pi, n_pairs)
    c, s = np.cos(th), np.sin(th)
    Rm = np.stack([np.stack([c, -s], -1), np.stack([s, c], -1)], -2)
    B3 = np.einsum("pij,pkj->pki", Rm, A3) + rng.uniform(-1e4, 1e4, (n_pairs, 1, 2))
    poses = b200.best_fit(b200.ScanTable(_dev(A3)), b200.ScanTable(_dev(B3))).cpu().numpy()
    for p in range(n_pairs):
        _check_fit(poses[p], A3[p], B3[p], f"3-point pair {p}", svd=p % 50 == 0)


# ---------------------------------------------------------------------------------------
# E. scan preparation: b200icp_polar_to_cartesian at the thresholds of every filter
# ---------------------------------------------------------------------------------------
def _polar_ref(rows, fv):
    """process.py:45-49 row loop with the filter's constants (registration.POLAR_FILTERS)."""
    lo, hi, qmin, arc_lo, arc_hi, use_arc, ysign = fv
    out = []
    for quality, angle, distance in rows:
        front = (not use_arc) or (angle <= arc_lo) or (angle >= arc_hi)
        if distance > lo and distance < hi and quality > qmin and front:
            a = math.radians(angle)
            out.append([distance * math.cos(a), ysign * distance * math.sin(a)])
    return np.array(out, dtype=np.float64).reshape(-1, 2)


def _around(v, step):
    return [np.nextafter(v, -np.inf), v, np.nextafter(v, np.inf), v - step, v + step]


def _threshold_rows(fv, rng):
    """Rows at every threshold of the filter (one ulp and one recording quantum, 1/4 mm or 1/64
    degree, either side) with the other fields comfortably inside, plus NaN in every field."""
    lo, hi, qmin, arc_lo, arc_hi, use_arc, ysign = fv
    good_d, good_q, good_a = 0.5 * (max(lo, 1.0) + hi), qmin + 20.0, 30.0
    rows = []
    for d in _around(lo, 0.25) + _around(hi, 0.25) + [np.nan]:
        rows.append([good_q, good_a, d])
    for q in _around(qmin, 1.0) + [np.nan]:
        rows.append([q, good_a, good_d])
    for a in _around(arc_lo, 1 / 64) + _around(arc_hi, 1 / 64) + [np.nan, 0.0, 359.984375, 180.0]:
        rows.append([good_q, a, good_d])
    rows = np.array(rows, dtype=np.float64)
    filler = np.stack([rng.integers(0, 60, 1000).astype(np.float64), rng.integers(0, 360 * 64, 1000) / 64.0,
                       rng.integers(0, 4 * 12000, 1000) / 4.0], axis=1)
    return np.concatenate([rows, filler, rows[::-1]])[rng.permutation(len(rows) * 2 + 1000)]


def _check_polar(got_xy, got_len, ref, what):
    assert int(got_len) == len(ref), f"{what}: {int(got_len)} kept, want {len(ref)}"
    g = got_xy[:len(ref)]
    assert np.array_equal(np.isnan(g), np.isnan(ref)), f"{what}: NaN rows"
    ok = ~np.isnan(ref)
    assert np.all(np.abs(g[ok] - ref[ok]) <= 1e-9), f"{what}: coordinates"


@pytest.mark.parametrize("name", ["process", "slam_offline", "realtime_2", "realtime_1"])
def test_polar_filter_thresholds(b200, name):
    """Counts and order exact, coordinates within 1e-9 mm (device sincos is not libm); more than
    256 rows per scan (several block trips); raw_len 0, short, and beyond raw_pitch (clamped)."""
    fv = b200.registration.POLAR_FILTERS[name]
    rng = np.random.default_rng(sum(map(ord, name)))
    scans = [_threshold_rows(fv, rng) for _ in range(3)]
    pitch = max(len(s) for s in scans)
    raw = np.zeros((5, pitch, 3))
    for k, s in enumerate(scans):
        raw[k, :len(s)] = s
    raw[3] = raw[0]
    raw[4] = raw[1]
    lens = np.array([len(scans[0]), len(scans[1]), len(scans[2]), 0, pitch + 100], dtype=np.int32)
    used = [scans[0], scans[1], scans[2], scans[0][:0], raw[4]]
    tab = b200.polar_to_cartesian(_dev(raw), _dev(lens), filter=name)
    xy, ln = tab.points.cpu().numpy(), tab.lengths.cpu().numpy()
    for k, rows in enumerate(used):
        ref = _polar_ref(rows, fv)
        if name in orc.POLAR_VARIANTS:           # the oracle's copy of the same function
            o = orc.polar_to_cartesian_variant(rows, name)[:, :2].reshape(-1, 2)
            assert np.array_equal(o, ref, equal_nan=True)
        _check_polar(xy[k], ln[k], ref, f"{name} scan {k}")
        assert np.all(xy[k, len(ref):] == 0.0), f"{name} scan {k}: padding"
    assert len(scans[0]) > 3 * 256 and np.any(np.isnan(_polar_ref(scans[0], fv))) == (not fv[5])


def test_polar_out_pitch_smaller_than_kept(b200):
    """out_pitch below the kept count: the first out_pitch kept points, len = out_pitch."""
    fv = b200.registration.POLAR_FILTERS["process"]
    rows = _threshold_rows(fv, np.random.default_rng(41))
    ref = _polar_ref(rows, fv)
    for out_pitch in (1, 100, len(ref) - 1, len(ref), len(ref) + 7):
        tab = b200.polar_to_cartesian(_dev(rows[None]), out_pitch=out_pitch)
        xy, ln = tab.points.cpu().numpy(), tab.lengths.cpu().numpy()
        assert xy.shape == (1, out_pitch, 2)
        m = min(out_pitch, len(ref))
        _check_polar(xy[0], ln[0], ref[:m], f"out_pitch {out_pitch}")
        assert np.all(xy[0, m:] == 0.0)
