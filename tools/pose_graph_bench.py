"""Loop closure on the device, stage by stage, on Scan_data_1 and on synthetic graphs with ground truth.

    python tools/pose_graph_bench.py [--out profiles/r3_pose_graph_bench.json] [--repeats 10]

Scan_data_1 stages (odometry, candidates, verification, information, edges, optimisation) are timed
with CUDA events around each call after warm-up calls; the stages whose Python wrapper reads a
count back to the host (candidates, edges) include that synchronisation.  The synthetic graph is
the 4,096-pose seeded random walk of configs[3] (oracle.pose_graph_oracle.synth_graph) with noisy
odometry and loop edges; it is optimised alone and as one of a batch of 8 graphs.  The oracle
(NumPy/SciPy, one spsolve per Gauss-Newton step) is timed on the host for the same graphs, in total
and for its spsolve calls alone.  The device name and power limit are read in the same run.
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
from oracle import icp_oracle as orc                 # noqa: E402  (scan unpacking)
from oracle import pose_graph_oracle as pg           # noqa: E402  (checker and host baseline)

MAX_CORR = 300.0


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


def events(fn, repeats, warmup=2):
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


def oracle_time(init, ei, ej, meas, info, max_iterations):
    """Wall time of the oracle's Gauss-Newton and of its spsolve calls alone."""
    spent = [0.0]
    solve = pg.spsolve

    def timed(*a, **k):
        t0 = time.perf_counter()
        try:
            return solve(*a, **k)
        finally:
            spent[0] += time.perf_counter() - t0

    pg.spsolve = timed
    try:
        t0 = time.perf_counter()
        o = pg.optimize(init, ei, ej, meas, info, max_iterations=max_iterations)
        total = time.perf_counter() - t0
    finally:
        pg.spsolve = solve
    return o, {"total_ms": total * 1e3, "spsolve_ms": spent[0] * 1e3, "iterations": o.iterations}


def graph(n, ei, ej, meas, info):
    d = lambda a, t=torch.float64: torch.from_numpy(np.ascontiguousarray(a)).to("cuda", t)   # noqa: E731
    return m.PoseGraph(n, d(ei, torch.int32), d(ej, torch.int32), d(meas).reshape(-1, 6), d(info).reshape(-1, 6))


def summary(r, k=0):
    return {"status": int(r.status[k]), "iterations": int(r.iterations[k]), "pcg_iterations": int(r.pcg_iterations[k]),
            "chi2_initial": float(r.chi2_initial[k]), "chi2_final": float(r.chi2_final[k])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_pose_graph_bench.json"))
    ap.add_argument("--repeats", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("pose_graph_bench needs a CUDA device")
    rep = args.repeats
    res = {"device": device_info()}

    # ---- Scan_data_1: every stage of close_loops on its own
    scans = load_scans()
    table = m.ScanTable.from_list(scans)
    rows = table.rows
    odo_fn = lambda: m.align_consecutive(table, max_iterations=30, max_corr_dist=MAX_CORR, want_indices=True)  # noqa: E731
    odo = odo_fn()
    poses0 = m.odometry.chain_poses_device(odo.pose_total)
    gap, radius, fit, rmse = 100, 300.0, 0.6, 60.0
    src_row, tgt_row, init = m.loop_candidates(poses0, gap, radius)
    k = int(src_row.shape[0])
    ver_fn = lambda: m.align_pairs(table, table, n_pairs=k, pairing="explicit", src_row=src_row,  # noqa: E731
                                   tgt_row=tgt_row, init_pose=init, max_iterations=30, max_corr_dist=MAX_CORR,
                                   want_indices=True)
    ver = ver_fn()
    srcs, tgts = table.slice_rows(1), table.slice_rows(0, rows - 1)
    info_odo_fn = lambda: m.information_matrices(srcs, tgts, odo.pose_total, odo.indices, MAX_CORR)  # noqa: E731
    info_loop_fn = lambda: m.information_matrices(table, table, ver.pose_total, ver.indices, MAX_CORR,  # noqa: E731
                                                  n_pairs=k, pairing="explicit", src_row=src_row, tgt_row=tgt_row)
    info_odo, _ = info_odo_fn()
    info_loop, _ = info_loop_fn()

    def edges():
        g = m.PoseGraph.from_odometry(odo, info_odo)
        g.add_loops(ver, src_row, tgt_row, info_loop, min_fitness=fit, max_rmse=rmse, src_lengths=table.lengths,
                    src_pitch=table.pitch)
        return g

    g = edges()
    opt_fn = lambda: m.optimize_pose_graph(g, poses0)  # noqa: E731
    r = opt_fn()
    ei, ej = g.edge_i.cpu().numpy(), g.edge_j.cpu().numpy()
    meas, info = g.meas.cpu().numpy(), g.info.cpu().numpy()
    init_np = poses0.cpu().numpy()
    o, host = oracle_time(init_np, ei, ej, meas, info, 20)
    dev = r.poses.cpu().numpy()
    res["scan_data_1"] = {
        "params": {"max_corr_dist": MAX_CORR, "min_gap": gap, "radius": radius, "min_fitness": fit, "max_rmse": rmse},
        "nodes": rows, "candidates": k, "odometry_edges": g.n_edges - int((ei + 1 != ej).sum()),
        "loop_edges": int((ei + 1 != ej).sum()), "dropped_odometry": g.dropped,
        "stages": {"odometry": events(odo_fn, rep),
                   "candidates": events(lambda: m.loop_candidates(poses0, gap, radius), rep),
                   "verification": events(ver_fn, rep),
                   "information": events(lambda: (info_odo_fn(), info_loop_fn()), rep),
                   "edges": events(edges, rep),
                   "optimisation": events(opt_fn, rep)},
        "device_result": summary(r), "oracle_host": host, "oracle_chi2_final": o.chi2_final,
        "max_position_diff_vs_oracle_mm": float(np.abs(dev[:, 4:] - o.poses[:, 4:]).max()),
    }

    # ---- synthetic 4,096-node graph with ground truth, alone and in a batch of 8
    truth, init, ei, ej, meas, info = pg.synth_graph(4096)
    big = graph(len(truth), ei, ej, meas, info)
    P = torch.from_numpy(init).cuda()
    r = m.optimize_pose_graph(big, P)
    o, host = oracle_time(init, ei, ej, meas, info, 20)
    dev = r.poses.cpu().numpy()
    res["synthetic_4096"] = {
        "nodes": len(truth), "edges": len(ei), "loop_edges": len(ei) - (len(truth) - 1),
        "optimisation": events(lambda: m.optimize_pose_graph(big, P), rep),
        "device_result": summary(r), "oracle_host": host, "oracle_chi2_final": o.chi2_final,
        "max_position_diff_vs_oracle_mm": float(np.abs(dev[:, 4:] - o.poses[:, 4:]).max()),
        "rms_error_vs_truth": {"odometry_only": pg.trajectory_error(init, truth),
                               "optimised": pg.trajectory_error(dev, truth)},
    }
    batch, inits, host_total, host_solve = [], [], 0.0, 0.0
    for s in range(8):
        t2, i2, a, b, z, w = pg.synth_graph(4096, seed=4096 + s, noise_seed=7 + s)
        batch.append(graph(len(t2), a, b, z, w))
        inits.append(torch.from_numpy(i2).cuda())
        _, h = oracle_time(i2, a, b, z, w, 20)
        host_total += h["total_ms"]
        host_solve += h["spsolve_ms"]
    rb = m.optimize_pose_graph(batch, inits)
    res["synthetic_batch_8x4096"] = {
        "optimisation": events(lambda: m.optimize_pose_graph(batch, inits), rep),
        "status": rb.status.tolist(), "iterations": rb.iterations.tolist(), "pcg_iterations": rb.pcg_iterations.tolist(),
        "oracle_host_total_ms": host_total, "oracle_host_spsolve_ms": host_solve,
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
