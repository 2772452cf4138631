"""2D Generalized ICP on the device: covariances, batched odometry, one SLAM-shaped registration and
the offline SLAM replay, each next to its point-to-point counterpart.

    python tools/gicp_bench.py [--out profiles/r3_gicp_bench.json] [--repeats 20]

Kernel-level rows are timed with CUDA events around each call after warm-up launches (median, min
and max over --repeats); single registrations and the replay include their host work and one
device-to-host read each, so they are timed with a host clock (every call ends in a
synchronisation).  Outputs at the timed sizes are checked against oracle/gicp_oracle.py.  The
device name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import icp_slam_yolo_b200 as m                       # noqa: E402
from oracle import gicp_oracle as g                  # noqa: E402  (checker only)
from oracle import icp_oracle as orc                 # noqa: E402  (scan unpacking, synthetic map)


def load_scans():
    z = np.load(os.path.join(ROOT, "tests", "golden", "scan_data_1_packed.npz"))
    off = z["offsets"]
    rows = np.stack([z["quality"].astype(np.float64), z["angle64"].astype(np.float64) / 64.0,
                     z["dist4"].astype(np.float64) / 4.0], axis=1)
    return [np.ascontiguousarray(orc.polar_to_cartesian(rows[off[i]:off[i + 1]])[:, :2]) for i in range(len(off) - 1)]


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def events(fn, repeats, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(repeats):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    return {"median_ms": float(np.median(ts)), "min_ms": float(min(ts)), "max_ms": float(max(ts)), "repeats": repeats}


def wall(fn, repeats, warmup=3):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return {"median_ms": float(np.median(ts)), "min_ms": float(min(ts)), "max_ms": float(max(ts)), "repeats": repeats}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_gicp_bench.json"))
    ap.add_argument("--repeats", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gicp_bench needs a CUDA device")
    rep = args.repeats
    res = {"device": device_info()}
    scans = load_scans()
    table = m.ScanTable.from_list(scans)

    # ---- covariances: the whole recording as one ragged table, and one local-map-sized cloud
    cov = m.estimate_covariances(table)
    got = cov.cpu().numpy()
    worst = max(float(np.max(np.abs(got[r, :len(s)] - g.estimate_covariances_2d(s)))) for r, s in enumerate(scans[::61]))
    mp = orc.synth_map(18678, dtype=np.float64)
    mt = m.ScanTable(torch.from_numpy(mp[None]).cuda())
    worst_map = float(np.max(np.abs(m.estimate_covariances(mt).cpu().numpy()[0] - g.estimate_covariances_2d(mp))))
    res["covariances"] = {
        "recording_table": {"rows": table.rows, "pitch": table.pitch, "points": int(sum(map(len, scans))),
                            **events(lambda: m.estimate_covariances(table), rep),
                            "max_abs_diff_vs_oracle_every_61st_row": worst},
        "map_18678": {**events(lambda: m.estimate_covariances(mt), rep), "max_abs_diff_vs_oracle": worst_map},
    }

    # ---- odometry: all 1,830 consecutive pairs, gate 180, 30 iterations
    gi = m.gicp_consecutive(table, max_iterations=30, max_corr_dist=180.0)
    ok = 0
    for p in range(0, len(scans) - 1, 61):
        o = g.gicp_extended(scans[p + 1], scans[p], 30, max_corr_dist=180.0)
        ok += int(int(gi.iterations[p]) == o.iterations and
                  np.allclose(gi.pose_total[p, 4:].cpu().numpy(), o.t_tot, atol=1e-6))
    res["odometry_1830_pairs"] = {
        "gicp_consecutive_incl_covariances": events(
            lambda: m.gicp_consecutive(table, max_iterations=30, max_corr_dist=180.0), rep),
        "align_consecutive": events(lambda: m.align_consecutive(table, max_iterations=30, max_corr_dist=180.0), rep),
        "gicp_mean_iterations": float(gi.iterations.double().mean()),
        "oracle_checked_pairs": len(range(0, len(scans) - 1, 61)), "oracle_agreeing_pairs": ok,
    }

    # ---- one registration of SLAM shape: 194 x 18,678, gate 180, 50 iterations, from an initial pose
    A = orc.synth_scan_for_map(194, dtype=np.float64)
    T0 = np.eye(4)
    T0[:2, :2] = [[np.cos(0.015), -np.sin(0.015)], [np.sin(0.015), np.cos(0.015)]]
    T0[:2, 3] = [30.0, -15.0]
    rm, T = m.registration_gicp(A, mp, 180.0, None, T0, 50)
    o = g.gicp_extended(A, mp, 50, max_corr_dist=180.0, init_pose=(T0[:2, :2], T0[:2, 3]))
    res["single_194x18678"] = {
        "registration_gicp": wall(lambda: m.registration_gicp(A, mp, 180.0, None, T0, 50), rep),
        "registration_p2p": wall(lambda: m.registration_p2p(A, mp, 180.0, None, T0, 50), rep),
        "gicp_iterations": o.iterations, "gicp_rmse": rm,
        "matches_oracle": bool(abs(rm - o.rmse) < 1e-9 * o.rmse and np.allclose(T[:2, 3], o.t_tot, atol=1e-6)),
    }

    # ---- the offline SLAM loop over the whole recording
    from icp_slam_yolo_b200.slam import OfflineSlam, SlamConfig
    frames = [np.c_[s, np.zeros(len(s))] for s in scans]
    replay = {}
    for reg in ("p2p", "gicp"):
        slam = OfflineSlam(SlamConfig(registration=reg))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = slam.run(frames)
        torch.cuda.synchronize()
        replay[reg] = {"wall_s": time.perf_counter() - t0, "frames": len(out),
                       "accepted": sum(1 for r in out if r is not None and r.accepted),
                       "rejected": sum(1 for r in out if r is not None and not r.accepted),
                       "final_map_points": int(slam.global_map.shape[0])}
    res["replay_scan_data_1"] = replay
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
