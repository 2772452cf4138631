"""CPU property tests of the two FP32 guard-band formulas the exactness of the CUDA kernels rests on.

They restate, in NumPy float32 / float64 arithmetic, (a) the skip test of the scan-to-map FP32 filter
(`Fp32Filter`, `filter_threshold`, `scan_round` in csrc/scan2map.cu) and (b) the bounds of the 16-target
decision of the pair kernel (`in_group_decide` in csrc/align_pair.cu: low mantissa byte replaced by the
slot number), and check on adversarial inputs the properties the kernels' proofs use:
  (a) a skipped point is farther than the best so far in the EXACT float64 arithmetic of `consider`;
  (b) `ubd` >= the exact distance to the winner, `los` <= the exact distance to every other target, and
      whenever the FP32 winner is not the float64 winner the near-tie flag is raised.
"""
import numpy as np

F32 = np.float32


def _f32(x):
    return np.asarray(x, dtype=np.float32)


def _next_up_f32(x):
    return np.nextafter(_f32(x), F32(np.inf))


def _filter_threshold(best, slack):
    """filter_threshold(): RU_f32(((sqrt(best) + slack) * 1.000004)^2), +inf without a bound."""
    best = np.asarray(best, dtype=np.float64)
    r = (np.sqrt(best) + slack) * 1.000004
    r2 = r * r
    t = r2.astype(np.float32)
    t = np.where(t.astype(np.float64) < r2, _next_up_f32(t), t)          # round up
    return np.where(np.isfinite(best), t, F32(np.inf)).astype(np.float32)


def _d32(q, s):
    """scan_round(): dx = q.x - RN(s.x), dy = ...; d32 = fmaf(dx, dx, dy * dy), all float32."""
    sx, sy = _f32(s[..., 0]), _f32(s[..., 1])
    dx, dy = _f32(q[..., 0] - sx), _f32(q[..., 1] - sy)
    t = _f32(dy * dy)
    return (dx.astype(np.float64) * dx.astype(np.float64) + t.astype(np.float64)).astype(np.float32)


def _dist2_f64(s, q):
    """dist2_f64(): NumPy's operation order, no contraction."""
    dx, dy = s[..., 0] - q[..., 0].astype(np.float64), s[..., 1] - q[..., 1].astype(np.float64)
    return dx * dx + dy * dy


def test_fp32_filter_never_skips_a_point_that_could_win():
    rng = np.random.default_rng(2024)
    checked = skipped = 0
    for scale in (1e-3, 1.0, 37.0, 2.5e3, 2e4, 1e6):
        for spread in (1e-4, 1e-2, 1.0, 50.0, 3e3):
            n = 40000
            s = rng.uniform(-scale, scale, size=(n, 2))                       # float64 scan points
            # the best so far: a map point at distance ~spread; candidates around that distance, many of
            # them within a few ulps of it (the adversarial band), on both sides
            ang = rng.uniform(0, 2 * np.pi, size=n)
            best_pt = _f32(s + spread * rng.uniform(0.2, 1.0, size=(n, 1)) * np.stack([np.cos(ang), np.sin(ang)], 1))
            best = _dist2_f64(s, best_pt)
            rel = np.concatenate([rng.uniform(-3e-5, 3e-5, size=n // 2), rng.uniform(-0.5, 2.0, size=n - n // 2)])
            ang2 = rng.uniform(0, 2 * np.pi, size=n)
            rad = np.sqrt(best) * (1.0 + rel)
            cand = _f32(s + rad[:, None] * np.stack([np.cos(ang2), np.sin(ang2)], 1))
            slack = 5e-7 * (np.abs(s[:, 0]) + np.abs(s[:, 1])) + 1e-20
            thr = _filter_threshold(best, slack)
            skip = _d32(cand, s) > thr
            exact = _dist2_f64(s, cand)
            assert not np.any(skip & (exact <= best)), (scale, spread)         # (a)
            checked += n
            skipped += int(skip.sum())
    assert skipped > 0.3 * checked                                             # the filter does filter


def test_fp32_filter_passes_exact_ties_and_duplicates():
    rng = np.random.default_rng(5)
    s = rng.uniform(-2e4, 2e4, size=(20000, 2))
    q = _f32(s + rng.normal(0, 20.0, size=s.shape))
    best = _dist2_f64(s, q)                                                    # the point itself is the best so far
    slack = 5e-7 * (np.abs(s[:, 0]) + np.abs(s[:, 1])) + 1e-20
    assert np.all(_d32(q, s) <= _filter_threshold(best, slack))                # a duplicate of the NN is never skipped
    # the bound of the first trip: ub = sqrt(d2 * kUp) * kUp, best := ub^2 * kUp
    k_up = 1.000000000001
    ub = np.sqrt(best * k_up) * k_up
    assert np.all(_d32(q, s) <= _filter_threshold(ub * ub * k_up, slack))
    assert np.all(_filter_threshold(np.array([np.inf]), 1.0) == np.inf)


def _in_group_bounds(tile_x, tile_y, fx, fy, tmax):
    """in_group_decide() for ONE source against 16 targets (float32 tile, centred)."""
    u = _f32(tile_x - fx)
    v = _f32(tile_y - fy)
    uu = _f32(u * u)
    d = (v.astype(np.float64) * v.astype(np.float64) + uu.astype(np.float64)).astype(np.float32)    # ffma(v, v, u*u)
    key = (d.view(np.uint32) & np.uint32(0xFFFFFF00)) | np.arange(16, dtype=np.uint32)
    order = np.argsort(key, kind="stable")
    best, second = key[order[0]], key[order[1]]
    bd = (best & np.uint32(0xFFFFFF00)).view(np.float32)
    sd = (second & np.uint32(0xFFFFFF00)).view(np.float32)
    cs = max(abs(float(fx)), abs(float(fy)))
    guard = F32((F32(cs) + F32(tmax)) * F32(4.76837158e-7))
    ubd = F32(F32(np.sqrt(bd)) * F32(1.00002) + guard)
    near_tie = bool(sd <= F32(F32(ubd * ubd) * F32(1.000001)))
    los = F32(F32(np.sqrt(sd)) * F32(0.999996) - guard)
    return int(best & np.uint32(15)), float(ubd), float(los), near_tie


def test_in_group_decision_bounds_hold_in_float64():
    rng = np.random.default_rng(11)
    worst_u = worst_l = np.inf
    for trial in range(6000):
        scale = 10.0 ** rng.uniform(1.0, 4.2)                                   # 10 mm .. 16 m from the tile origin
        gap = 10.0 ** rng.uniform(-4.0, 1.5)
        tx = rng.uniform(-scale, scale, size=16)
        ty = rng.uniform(-scale, scale, size=16)
        k = rng.integers(16)
        ang = rng.uniform(0, 2 * np.pi)
        r = 10.0 ** rng.uniform(-1.0, 2.5)
        sx, sy = tx[k] + r * np.cos(ang), ty[k] + r * np.sin(ang)               # near target k ...
        j = (k + 1 + rng.integers(15)) % 16
        ang2 = rng.uniform(0, 2 * np.pi)
        tx[j], ty[j] = sx + (r + gap * rng.uniform(-1, 1)) * np.cos(ang2), sy + (r + gap) * np.sin(ang2)   # ... and a rival
        tile_x, tile_y = _f32(tx), _f32(ty)
        fx, fy = F32(sx), F32(sy)                                               # the kernel's (float)(s - origin)
        tmax = float(max(np.abs(tile_x).max(), np.abs(tile_y).max()))
        slot, ubd, los, near_tie = _in_group_bounds(tile_x, tile_y, fx, fy, tmax)
        # exact distances from the float64 source (the float32 centring error of the source is inside `guard`)
        ex = np.hypot(tile_x.astype(np.float64) - sx, tile_y.astype(np.float64) - sy)
        winner = int(np.argmin(ex))
        if slot != winner:
            assert near_tie, (trial, slot, winner, ex[slot], ex[winner])        # a wrong FP32 winner is always flagged
            continue
        if near_tie:
            continue                                                            # re-decided in float64: no bound is used
        others = np.delete(ex, slot)
        assert ubd >= ex[slot], (trial, ubd, ex[slot])
        assert los <= others.min(), (trial, los, others.min())
        worst_u = min(worst_u, ubd - ex[slot])
        worst_l = min(worst_l, others.min() - los)
    assert worst_u >= 0.0 and worst_l >= 0.0
