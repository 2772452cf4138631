#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native 2D ICP path.

Workload (BASELINE.json configs[2], the configuration the metric is quoted on): batched
synthetic 2D LiDAR pairs, 65,536 pairs x 360 points, 30 forced iterations
(tolerance = -1 so the work is deterministic), float32 point tables generated in float64
by oracle.icp_oracle.synth_room_batch (seed = 1234 + pair index).  Weak scaling: every
rank aligns its own 65,536 pairs (pair indices rank*65536 ...), no data-path collective.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--pairs P] [--dump-outputs DIR]
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference      # CPU arm: the oracle port on all host cores

One JSON line on stdout (rank 0).  A "step" = one pass of the fused ICP kernel over the
rank's whole batch (one launch).  `value` = alignments/s with inputs resident in HBM;
`e2e` = the same through HostPipeline (pinned host buffers, H2D + D2H inside the timed
region); `roofline` = algorithmic FP32 FLOP/s of the search (5 FLOP per pair-eval,
SURVEY.md §8d) over the FFMA peak measured live by the library's probe kernel.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_POINTS = 360
ITERS = 30
FLOP_PER_PAIR_EVAL = 5.0                       # SURVEY.md §8(d)
PAIR_EVALS_PER_ALIGNMENT = N_POINTS * N_POINTS * ITERS
ALG_BYTES_PER_ALIGNMENT = 2 * N_POINTS * 8 + 12 + 36   # SURVEY.md §8(d): 5,808 B
ALLPAIRS_SCANS = 4096


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--pairs", type=int, default=65536, help="pairs per GPU (weak scaling)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-sample", type=int, default=0, help="pairs in the CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="headline workload only (no `secondary` block)")
    ap.add_argument("--e2e-chunks", type=int, default=8)
    ap.add_argument("--e2e-buffers", type=int, default=3, help="e2e: staging buffers = compute streams of HostPipeline")
    ap.add_argument("--e2e-graph", action="store_true",
                    help="e2e: replay each run as one CUDA graph instead of enqueueing it from Python (measured: no "
                         "difference, 9.087 vs 9.088 ms; the host keeps ahead of the GPU either way)")
    ap.add_argument("--no-numa-bind", action="store_true",
                    help="A/B: allocate the pinned host tables wherever the process happens to run instead of on the "
                         "GPU's NUMA node (hostmem.near_gpu)")
    ap.add_argument("--workload", default="pairs", choices=["pairs", "odometry", "allpairs", "scan2map", "single", "nn", "occupancy", "slam"],
                    help="pairs = the headline configs[2] (default); the others are BASELINE.json "
                         "configs[1], [3] and [4], reported with the same JSON shape")
    ap.add_argument("--map-points", type=int, default=1 << 24, help="scan2map: total map points")
    ap.add_argument("--scan-points", type=int, default=8192)
    ap.add_argument("--s2m-exchange", default="peer", choices=["peer", "nccl"])
    ap.add_argument("--s2m-graph", dest="s2m_graph", action="store_true", default=True,
                    help="scan2map: replay the 30-iteration loop as one CUDA graph (default with the peer exchange)")
    ap.add_argument("--no-s2m-graph", dest="s2m_graph", action="store_false",
                    help="scan2map: launch the 60 kernels of an alignment from the host loop")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="pairs workload: write what the last timed step computed on rank 0 (the AlignResult "
                         "fields) to DIR/<field>.npy as float64, so that two builds can be compared on the same "
                         "seeded inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "pairs"):
        ap.error("--dump-outputs covers the headline workload only (--impl b200 --workload pairs)")
    return args


DUMP_BYTES = 60 << 20          # keeps the files, .npy headers included, under 64 MB (10^6 B)


def dump_outputs(directory, res):
    """Every [P, ...] field of ``res`` as float64 (int32 counts are exact in float64); above DUMP_BYTES
    in all, a fixed seeded sample of the pairs, whose indices go to pair_index.npy."""
    fields = {f: getattr(res, f).cpu().numpy().astype(np.float64)
              for f in ("pose_total", "pose_last", "error", "rmse", "inliers", "iterations")}
    n = len(fields["pose_total"])
    row_bytes = sum(a[0].nbytes for a in fields.values())
    if n * row_bytes > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_BYTES // (row_bytes + 8), replace=False))
        fields = {f: a[rows] for f, a in fields.items()}
        fields["pair_index"] = rows.astype(np.float64)
    os.makedirs(directory, exist_ok=True)
    for name, a in fields.items():
        np.save(os.path.join(directory, name + ".npy"), a)


# ------------------------------------------------------------------------------------------
# CPU arm: the UNMODIFIED reference icp() (labels_segmentation/icp.py:28-53), loaded from the
# reference tree or from the byte-identical build-time copy oracle/_ref/icp.py; the oracle port
# (kind "port") only when neither exists.
# ------------------------------------------------------------------------------------------
_REF = {}


def reference_icp():
    """(callable icp(A, B, max_iterations, tolerance) -> anything, kind, description)."""
    if not _REF:
        from oracle import ref_loader
        if ref_loader.reference_available():
            mod = ref_loader.load_reference_icp()
            _REF["f"] = (mod.icp, "reference",
                         "unmodified labels_segmentation/icp.py:28-53 (SciPy KDTree rebuilt every iteration + NumPy SVD), "
                         "loaded from " + os.path.relpath(ref_loader.reference_icp_path(), ROOT))
        else:
            from oracle import icp_oracle as orc
            _REF["f"] = (lambda A, B, it, tol: orc.icp_extended(A, B, it, tol, keep_history=False), "port",
                         "oracle port of labels_segmentation/icp.py:5-53 (oracle/_ref/icp.py absent: build() did not see the reference)")
    return _REF["f"]


def _cpu_worker(job):
    kind, first, count, tol = job
    from oracle import icp_oracle as orc
    icp, _, _ = reference_icp()
    try:                                    # one BLAS/OpenMP thread per worker process: the pool is the parallelism
        import threadpoolctl
        threadpoolctl.threadpool_limits(1)
    except Exception:
        pass
    if kind == "rooms":
        src, tgt = orc.synth_room_batch(first, count)
        pairs = [(src[p].astype(np.float64), tgt[p].astype(np.float64)) for p in range(count)]
    else:                                   # "trajectory": all-pairs candidates, row-major (i < j) from pair `first`
        scans = orc.synth_trajectory_scans(ALLPAIRS_SCANS).astype(np.float64)
        pairs = []
        for q in range(first, first + count):
            i, rem = 0, q                   # linear index -> (i, j), i < j (the CPU workers import no torch)
            while rem >= ALLPAIRS_SCANS - 1 - i:
                rem -= ALLPAIRS_SCANS - 1 - i
                i += 1
            pairs.append((scans[i + 1 + rem], scans[i]))
    t0 = time.perf_counter()
    for A, B in pairs:
        icp(A, B, ITERS, tol)
    return time.perf_counter() - t0


def cpu_pool_throughput(kind, sample_pairs, cores, tol=-1.0, first=0, stride=None):
    """alignments/s of the reference over `sample_pairs` pairs spread on `cores` processes (time of
    the icp() calls only: the slowest worker; generation excluded)."""
    import multiprocessing as mp
    reference_icp()                          # import once in the parent; the workers are forked from it
    per = max(1, sample_pairs // cores)
    stride = per if stride is None else stride
    jobs = [(kind, first + i * stride, per, tol) for i in range(cores)]
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        pool.map(_cpu_worker, [(kind, 0, 1, tol)] * cores)          # warm the workers
        out = pool.map(_cpu_worker, jobs)
    return per * cores / max(out), per * cores


def cpu_single_core(kind, count, tol=-1.0):
    """The reference as shipped: one process, one core."""
    return count / _cpu_worker((kind, 0, count, tol)), count


def default_cpu_sample(cores):
    """~15 s of single-core work (15 ms per 360x360x30 alignment), a multiple of the core count."""
    return max(1024 // cores, 4) * cores


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    sample = args.cpu_sample or default_cpu_sample(cores)
    _, kind, what = reference_icp()
    steps_ms, vals = [], []
    for i in range(args.warmup + args.steps):
        v, n = cpu_pool_throughput("rooms", sample, cores)
        if i >= args.warmup:
            vals.append(v)
            steps_ms.append(1e3 * n / v)
    value = float(np.mean(vals))
    one, n1 = cpu_single_core("rooms", 32)
    desc = f"{sample} pairs x {N_POINTS} pts x {ITERS} forced iterations per step, {cores} processes"
    line = {
        "impl": "reference", "metric": "ICP alignments/sec (360-pt 2D scans, 30 iters)",
        "value": value, "unit": "alignments/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": float(np.mean(steps_ms)), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "nn_pairs_per_s": value * PAIR_EVALS_PER_ALIGNMENT,
        "config": {"workload": "configs[2]: batched synthetic 2D LiDAR pairs, 360 x 360 points, 30 forced "
                               "iterations (tolerance=-1)", "sample_pairs_per_step": sample,
                   "implementation": what, "cpu": cpu_model()},
        "cpu_baseline": {"value": value, "unit": "alignments/s", "cores": cores, "kind": kind, "sample": desc,
                         "single_core_as_shipped": {"value": one, "unit": "alignments/s", "cores": 1,
                                                    "sample": f"{n1} pairs, one process"}},
        "e2e": {"value": value, "unit": "alignments/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


# ------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.QUERY}",
                 "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(mx)) if mx else None,
                "power_w_max": float(max(power)) if power else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_hbm_peak():
    try:
        d = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(d["hbm_gbs"]), "MEASURED_PEAKS.json"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_summary(name):
    """Counters of one committed `ncu --set full` capture (profiles/<name>.json, written by
    tools/ncu_summary.py from the .ncu-rep of the same kernel and command); None if absent."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", name + ".json")))
    except Exception:
        return None


def run_b200(args):
    import torch
    import torch.distributed as dist
    import icp_slam_yolo_b200 as m
    from oracle import icp_oracle as orc          # input generator + CPU baseline only

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # CPU legs that use a process pool run first: the workers are forked before CUDA is initialised
    cpu_base, cpu_sec = None, {}
    want_cpu = world == 1 and not args.no_cpu_baseline
    if want_cpu:
        cores = os.cpu_count() or 1
        _, kind, what = reference_icp()
        sample = args.cpu_sample or default_cpu_sample(cores)
        v, n = cpu_pool_throughput("rooms", sample, cores)
        one, n1 = cpu_single_core("rooms", 32)
        cpu_base = {
            "value": v, "unit": "alignments/s", "cores": cores, "kind": kind,
            "sample": f"{n} pairs of the same workload (360 x 360 x 30 forced iterations) on {cores} "
                      f"processes; {what}; {cpu_model()}",
            "single_core_as_shipped": {"value": one, "unit": "alignments/s", "cores": 1,
                                       "sample": f"{n1} pairs, one process (the reference has no parallelism of its own)"}}
        if not args.no_secondary:
            small = max(4, 128 // cores) * cores
            vt, nt = cpu_pool_throughput("rooms", small, cores, tol=1e-5)
            cpu_sec["tol"] = {"value": vt, "unit": "alignments/s", "cores": cores, "kind": kind,
                              "sample": f"{nt} pairs of the same batch, tolerance 1e-5 (early exit), {cores} processes"}
            total = ALLPAIRS_SCANS * (ALLPAIRS_SCANS - 1) // 2
            va, na = cpu_pool_throughput("trajectory", small, cores, first=0, stride=total // cores)
            cpu_sec["allpairs"] = {"value": va, "unit": "alignments/s", "cores": cores, "kind": kind,
                                   "sample": f"{na} of the {total} pairs ({na // cores} consecutive pairs at {cores} "
                                             f"evenly spaced offsets of the row-major enumeration), 30 forced iterations"}
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    m.lib()                                        # fail loudly if the CUDA library is missing

    P = args.pairs
    first = rank * P
    src_np, tgt_np = orc.synth_room_batch(first, P)              # float32, values generated in float64
    if args.no_numa_bind:
        h_src, h_tgt, numa = torch.from_numpy(src_np).pin_memory(), torch.from_numpy(tgt_np).pin_memory(), None
    else:                                   # pinned tables on the GPU's NUMA node (matters once 8 GPUs copy at once)
        h_src, numa = m.hostmem.pin_near_gpu(src_np, local)
        h_tgt, _ = m.hostmem.pin_near_gpu(tgt_np, local)
    src = m.ScanTable(h_src.to(dev))
    tgt = m.ScanTable(h_tgt.to(dev))
    out = m.alloc_outputs(P, N_POINTS, dev)

    def step():
        m.align_pairs(src, tgt, max_iterations=ITERS, tolerance=-1.0, out=out)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # FP32 peak of this GPU, measured live (MEASURED_PEAKS.json has no FP32 figure)
    fp32_peak = m.ffma_probe()

    for _ in range(max(3, args.warmup)):
        step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    t_all0, t_all1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_all0.record()
    for e0, e1 in evs:
        e0.record()
        step()
        e1.record()
    t_all1.record()
    barrier()
    total_ms = max_over_ranks(t_all0.elapsed_time(t_all1))
    kernel_ms = float(np.mean([e0.elapsed_time(e1) for e0, e1 in evs]))     # per-launch duration
    assert bool(torch.all(out.iterations == ITERS)), "forced-iteration run did not run 30 iterations"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)
    # untimed diagnostic launch: how many pair evaluations did the (exactly pruned) sweep execute?
    stats = m.align_pairs(src, tgt, max_iterations=ITERS, tolerance=-1.0, want_stats=True)
    torch.cuda.synchronize()
    executed = float(stats.evaluated_pairs.sum().item())
    assert torch.equal(stats.pose_total, out.pose_total)
    del stats
    # A/B outside the headline timing: the dense sweep of the same kernel (every source-target pair
    # evaluated in every iteration, no culling, no reuse) = the brute-force work SURVEY.md 8(d) counts;
    # this is the launch whose FLOP rate is a hardware utilisation.  Identical results required.
    dense_out = m.alloc_outputs(P, N_POINTS, dev)
    for _ in range(2):
        m.align_pairs(src, tgt, max_iterations=ITERS, tolerance=-1.0, dense_sweep=True, sweep_reuse=False, out=dense_out)
    d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    d0.record()
    for _ in range(3):
        m.align_pairs(src, tgt, max_iterations=ITERS, tolerance=-1.0, dense_sweep=True, sweep_reuse=False, out=dense_out)
    d1.record()
    torch.cuda.synchronize()
    dense_ms = d0.elapsed_time(d1) / 3
    assert torch.equal(dense_out.pose_total, out.pose_total), "dense and pruned sweeps disagree"
    del dense_out

    ms_per_step = total_ms / args.steps
    value = world * P / (ms_per_step * 1e-3)

    # ---- e2e: pinned host buffers -> chunked H2D || kernel || D2H, through HostPipeline
    e2e = None
    if not args.no_e2e:
        n_chunks = args.e2e_chunks
        pipe = m.registration.HostPipeline(P, N_POINTS, N_POINTS, dtype=torch.float32, chunks=n_chunks, device=dev,
                                           graph=args.e2e_graph, buffers=args.e2e_buffers)
        for _ in range(3):                     # eager, capture + replay, replay
            pipe.run(h_src, h_tgt, max_iterations=ITERS, tolerance=-1.0)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            hp, he, hi = pipe.run(h_src, h_tgt, max_iterations=ITERS, tolerance=-1.0)
        e1.record()
        barrier()
        e2e_ms = max_over_ranks(e0.elapsed_time(e1)) / args.steps
        assert torch.equal(hp, out.pose_total.cpu()), "e2e results differ from the resident-input run"
        h2d, d2h = pipe.bytes_per_run(ragged=False)
        # the floor of any end-to-end number: the same tables host -> device and nothing else, all ranks at once
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        c0.record()
        for _ in range(3):
            src.points.copy_(h_src, non_blocking=True)
            tgt.points.copy_(h_tgt, non_blocking=True)
        c1.record()
        barrier()
        h2d_ms = max_over_ranks(c0.elapsed_time(c1)) / 3
        e2e = {"value": world * P / (e2e_ms * 1e-3), "unit": "alignments/s", "ms_per_step": e2e_ms,
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "launches_per_step": pipe.launches,
               "h2d_only_ms": h2d_ms, "h2d_only_gbs_per_gpu": h2d / (h2d_ms * 1e-3) / 1e9,
               "host_numa": numa if numa is not None else "not bound (--no-numa-bind)",
               "limiter": ("host-to-device copy" if h2d_ms > 0.9 * e2e_ms else "kernel") +
                          ": e2e = max(kernel + the first chunk's copy, copy + the last chunk's kernel); h2d_only_ms is "
                          "the copy alone with every rank copying at once (GPUs share host memory and PCIe uplinks)",
               "cuda_graph": bool(pipe._graphs), "staging_buffers": pipe.nbuf,
               "chunk_pairs": [int(b1 - b0) for b0, b1 in zip(pipe.bounds[:-1], pipe.bounds[1:])],
               "api": "icp_slam_yolo_b200.registration.HostPipeline.run (largest chunk = 1/%d of the batch, ramped "
                      "chunk sizes, copy/compute overlap)" % n_chunks}
        del pipe

    clocks = sampler.stop() if rank == 0 else None      # sampled across both timed regions

    # ---- the other BASELINE configs, each timed by the same rules (CUDA events, barrier, max over ranks)
    secondary = None
    if not args.no_secondary:
        del src, tgt, out, h_src, h_tgt
        torch.cuda.empty_cache()
        ctx = BenchCtx(world, rank, local, dev, barrier, max_over_ranks, fp32_peak, cpu_sec, want_cpu)
        secondary = run_secondary(args, ctx, src_np, tgt_np)
    if rank != 0:
        return

    flops = P * PAIR_EVALS_PER_ALIGNMENT * FLOP_PER_PAIR_EVAL
    alg_tflops = flops / (kernel_ms * 1e-3) / 1e12
    dense_tflops = flops / (dense_ms * 1e-3) / 1e12
    hbm_peak, hbm_src = measured_hbm_peak()
    achieved_gbs = P * ALG_BYTES_PER_ALIGNMENT / (kernel_ms * 1e-3) / 1e9
    ncu = ncu_summary("r2_pair_kernel_ncu") if P == 65536 else None
    line = {
        "metric": "ICP alignments/sec (360-pt 2D scans, 30 iters)",
        "value": value, "unit": "alignments/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32 search + f64 state", "data": "synthetic",
        "nn_pairs_per_s": value * PAIR_EVALS_PER_ALIGNMENT,
        "config": {"workload": "configs[2]: batched synthetic 2D LiDAR pairs, %d pairs per GPU x 360 x 360 "
                               "points, 30 forced iterations (tolerance=-1), float32 tables" % P,
                   "pairs_per_gpu": P, "points": N_POINTS, "iterations": ITERS,
                   "l2": "inputs (%.0f MB per GPU) exceed the 126 MB L2; no flush needed" %
                         (P * N_POINTS * 16 / 1e6),
                   "parallelism": "pairs sharded by contiguous index range, no collective (weak scaling: "
                                  "%d pairs per GPU; the strong curve of 65,536 pairs in total is secondary."
                                  "configs2_strong)" % P},
        "gpu_launches": args.steps,
        "clocks": clocks,
        "roofline": {
            "bound": "fp32",
            "kernel": "icp_align_pair_kernel<6,dense,2 warps> (B200ICP_FLAG_DENSE_SWEEP | B200ICP_FLAG_NO_SWEEP_REUSE): "
                      "every one of the N_src x N_tgt x 30 pair evaluations SURVEY.md 8(d) counts is executed, so "
                      "achieved/peak is a hardware utilisation",
            "achieved": dense_tflops, "peak": fp32_peak, "unit": "TFLOP/s", "frac": dense_tflops / fp32_peak,
            "peak_source": "b200icp_ffma_probe measured live (dependent-FFMA chains, all SMs)",
            "algorithmic_flop_per_launch": flops, "kernel_ms": dense_ms,
            "traffic": (ncu or {}).get("dram_bytes"),
            "traffic_source": ("dram__bytes_read.sum + dram__bytes_write.sum of one launch of the SHIPPED kernel, "
                               "profiles/r2_pair_kernel_ncu.json (ncu --set full, same command)") if ncu else None,
            "shipped_kernel": {
                "kernel": "icp_align_pair_kernel<2,pruned,2 warps> (exact culling of target groups, two candidate groups "
                          "per source, movement-bound reuse; bit-identical results, asserted against the dense "
                          "launch in this run)",
                "kernel_ms": kernel_ms,
                "algorithmic_tflops": alg_tflops,
                "algorithmic_speedup_vs_dense": dense_ms / kernel_ms,
                "algorithmic_tflops_over_peak": alg_tflops / fp32_peak,
                "executed_pair_eval_fraction": executed / (P * PAIR_EVALS_PER_ALIGNMENT),
                "executed_tflops": executed * FLOP_PER_PAIR_EVAL / (kernel_ms * 1e-3) / 1e12,
                "ncu": ncu,
                "note": "algorithmic_tflops counts the brute-force work although most of it is skipped (pair "
                        "evaluations that are PROVEN irrelevant), so it may exceed the FP32 peak: it is a speed-up "
                        "figure, not a utilisation.  The utilisation of the shipped kernel is ncu's issue-slot figure."},
            "hbm": {"achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s",
                    "frac": achieved_gbs / hbm_peak, "peak_source": hbm_src,
                    "algorithmic_bytes_per_launch": P * ALG_BYTES_PER_ALIGNMENT}},
    }
    if e2e:
        line["e2e"] = e2e
    if cpu_base is not None:
        line["cpu_baseline"] = cpu_base
    if secondary is not None:
        line["secondary"] = secondary
    emit(line)
    if world > 1:
        dist.destroy_process_group()


class BenchCtx:
    def __init__(self, world, rank, local, dev, barrier, max_over_ranks, fp32_peak, cpu_sec, want_cpu):
        self.world, self.rank, self.local, self.dev = world, rank, local, dev
        self.barrier, self.max_over_ranks, self.fp32_peak = barrier, max_over_ranks, fp32_peak
        self.cpu_sec, self.want_cpu = cpu_sec, want_cpu


def _slim(line, keep=("metric", "value", "unit", "ms_per_step", "scaling", "config", "gpu_launches", "roofline", "e2e",
                      "cpu_baseline", "per_iteration_ms", "gpu_wall_fraction_of_cpu", "subset_first_1075", "n_gpus")):
    return {k: line[k] for k in keep if k in line}


def run_secondary(args, ctx, src_np, tgt_np):
    """Every other BASELINE.json config at this N, two timed steps each (they are not the headline):
    configs[2] strong (65,536 pairs in total), its tolerance = 1e-5 variant, configs[3] all-pairs
    (strong), configs[4] scan-to-map (strong), and at N = 1 configs[1] odometry and configs[0]."""
    import torch
    import icp_slam_yolo_b200 as m
    sec = {}
    steps, warm = 3, 3
    world, rank, dev = ctx.world, ctx.rank, ctx.dev
    # ---- configs[2] as BASELINE words it: 65,536 pairs sharded across the GPUs (strong scaling)
    total = 65536
    b, e = m.shard_range(total, rank, world)
    lo = rank * args.pairs                      # this rank generated pairs [lo, lo + args.pairs)
    if world == 1:
        s_np, t_np = src_np[b:e], tgt_np[b:e]
    else:
        from oracle import icp_oracle as orc
        s_np, t_np = orc.synth_room_batch(b, e - b)
    s, t = m.ScanTable(torch.from_numpy(np.ascontiguousarray(s_np)).to(dev)), m.ScanTable(torch.from_numpy(np.ascontiguousarray(t_np)).to(dev))
    out = m.alloc_outputs(e - b, N_POINTS, dev)
    ms = _timed(lambda: m.align_pairs(s, t, max_iterations=ITERS, tolerance=-1.0, kernel="warp", out=out),
                steps, warm, ctx.barrier, ctx.max_over_ranks)
    sec["configs2_strong"] = {
        "metric": "ICP alignments/sec (65,536 pairs in total sharded across the GPUs)", "value": total / (ms * 1e-3),
        "unit": "alignments/s", "ms_per_step": ms, "scaling": "strong", "n_gpus": world,
        "config": {"pairs_total": total, "pairs_this_rank": e - b,
                   "waves_of_resident_ctas": (e - b) / (148 * 12.0)}}
    if world == 1:
        ms_t = _timed(lambda: m.align_pairs(s, t, max_iterations=ITERS, tolerance=1e-5, kernel="warp", out=out),
                      steps, warm, ctx.barrier, ctx.max_over_ranks)
        its = out.iterations.double()
        sec["configs2_tolerance_1e-5"] = {
            "metric": "ICP alignments/sec (configs[2] tables, tolerance 1e-5: the reference's own stopping rule)",
            "value": total / (ms_t * 1e-3), "unit": "alignments/s", "ms_per_step": ms_t,
            "config": {"iterations_mean": float(its.mean()), "iterations_min": int(its.min()), "iterations_max": int(its.max())},
            "cpu_baseline": ctx.cpu_sec.get("tol")}
    del s, t, out
    # ---- configs[3], configs[4], configs[1], configs[0]
    sub = argparse.Namespace(**vars(args))
    sub.steps, sub.warmup = steps, warm
    if world == 1:                  # the NN phase alone ("NN pairs/sec"): one search per pair of the same tables
        sec["nn_search"] = _slim(run_nn(sub, ctx, tables=(src_np, tgt_np)) or {})
        torch.cuda.empty_cache()
    sec["allpairs"] = _slim(run_allpairs(sub, ctx) or {})
    torch.cuda.empty_cache()
    sec["scan2map"] = _slim(run_scan2map(sub, ctx) or {})
    torch.cuda.empty_cache()
    if world == 1:
        sec["odometry"] = _slim(run_odometry(sub, ctx) or {})
        sec["single_alignment"] = run_single(sub, ctx)
    return sec


# ------------------------------------------------------------------------------------------
# secondary workloads (BASELINE.json configs[1], [3], [4]); same timing rules, same JSON shape
# ------------------------------------------------------------------------------------------
def _dist_setup():
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    return world, rank, local, dev, barrier, max_over_ranks


def _timed(step, steps, warmup, barrier, max_over_ranks):
    import torch
    for _ in range(max(3, warmup)):
        step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    barrier()
    return max_over_ranks(e0.elapsed_time(e1)) / steps


def _fixture_scans():
    from icp_slam_yolo_b200 import scan_io
    return scan_io.unpack_fixture(os.path.join(ROOT, "tests", "golden", "scan_data_1_packed.npz"))


def run_odometry(args, ctx=None):
    """configs[1]: Scan_data_1 sequence odometry, all 1,830 consecutive pairs (k+1 -> k),
    max_iterations 30, tolerance 1e-5, one launch; the bundled recording ships as the lossless
    fixture tests/golden/scan_data_1_packed.npz.  Also the first-1,075-pair subset BASELINE.json
    words ("~1075 consecutive scan pairs")."""
    import torch
    import icp_slam_yolo_b200 as m
    from oracle import icp_oracle as orc
    raw = _fixture_scans()
    # CPU: the unmodified reference icp() on one core (the reference as shipped); iteration counts
    # from the oracle port (the reference does not return them)
    icp_ref, kind, what = reference_icp()
    cart = [np.ascontiguousarray(orc.polar_to_cartesian(r)[:, :2]) for r in raw]
    walls = np.zeros(len(cart) - 1)
    for p in range(len(cart) - 1):
        t0 = time.perf_counter()
        icp_ref(cart[p + 1], cart[p], 30, 1e-5)
        walls[p] = time.perf_counter() - t0
    cpu_wall, cpu_wall_1075 = float(walls.sum()), float(walls[:1075].sum())
    its = sum(orc.icp_extended(cart[p + 1], cart[p], 30, 1e-5, keep_history=False).iterations
              for p in range(len(cart) - 1))
    t0 = time.perf_counter()
    for r in raw[:200]:
        orc.polar_to_cartesian_loop(r)
    cpu_prep = (time.perf_counter() - t0) * len(raw) / 200.0
    if ctx is None:
        world, rank, local, dev, barrier, max_over_ranks = _dist_setup()
    else:
        world, rank, local, dev, barrier, max_over_ranks = ctx.world, ctx.rank, ctx.local, ctx.dev, ctx.barrier, ctx.max_over_ranks
    n_pairs = len(raw) - 1
    h_raw, h_len = m.scan_io.raw_table(raw, pin=True)
    table = m.scan_io.prepare_scans(raw, device=dev)
    out = m.alloc_outputs(n_pairs, table.pitch, dev)
    fp32_peak = m.ffma_probe()

    def step():
        m.align_consecutive(table, max_iterations=30, tolerance=1e-5, out=out)

    ms = _timed(step, args.steps, args.warmup, barrier, max_over_ranks)
    gpu_its = int(out.iterations.sum().item())

    def e2e_step():       # raw polar rows on the host -> poses on the host
        d_raw = h_raw.to(dev, non_blocking=True)
        d_len = h_len.to(dev, non_blocking=True)
        tb = m.polar_to_cartesian(d_raw, d_len)
        res = m.align_consecutive(tb, max_iterations=30, tolerance=1e-5, out=out)
        return m.chain_poses(res.pose_total)             # device prefix composition + D2H of [1831,6]

    e2e_ms = _timed(e2e_step, args.steps, args.warmup, barrier, max_over_ranks)
    # first 1,075 pairs (rows 0..1075 of the same table)
    sub_table = m.ScanTable(table.points[:1076].contiguous(), table.lengths[:1076].contiguous())
    sub_out = m.alloc_outputs(1075, table.pitch, dev)
    ms_1075 = _timed(lambda: m.align_consecutive(sub_table, max_iterations=30, tolerance=1e-5, out=sub_out),
                     args.steps, args.warmup, barrier, max_over_ranks)
    assert torch.equal(sub_out.pose_total, out.pose_total[:1075])
    lens = table.lengths.cpu().numpy().astype(np.int64)
    its_np = out.iterations.cpu().numpy().astype(np.int64)
    evals = float(np.sum(lens[1:] * lens[:-1] * its_np))
    if rank != 0:
        return None
    line = {
        "metric": "ICP alignments/sec (Scan_data_1 sequence odometry, 1,830 consecutive pairs)",
        "value": n_pairs / (ms * 1e-3), "unit": "alignments/s", "n_gpus": 1, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": ms, "higher_is_better": True, "scaling": "replicas",
        "vs_baseline": None, "dtype": "f32 search + f64 state", "data": "bundled recording (fixture)",
        "nn_pairs_per_s": evals / (ms * 1e-3),
        "config": {"workload": "configs[1]: full Scan_data_1 sequence odometry, 1,830 pairs, max_iterations 30, "
                               "tolerance 1e-5, ragged 11..196 points", "iterations_total": gpu_its,
                   "l2": "inputs (5.7 MB) fit L2: a 64 MB buffer is NOT flushed between steps; noted"},
        "gpu_launches": args.steps,
        "roofline": {"bound": "fp32", "kernel": "icp_align_pair_kernel<2,pruned,2 warps> (the dispatcher's choice above 512 pairs)",
                     "achieved": evals * 5 / (ms * 1e-3) / 1e12,
                     "peak": fp32_peak, "unit": "TFLOP/s", "frac": evals * 5 / (ms * 1e-3) / 1e12 / fp32_peak,
                     "traffic": None, "note": "tiny ragged problems, less than one wave: bound by the latency of the longest pair"},
        "e2e": {"value": n_pairs / (e2e_ms * 1e-3), "unit": "alignments/s", "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": int(h_raw.numel() * 8 + h_len.numel() * 4),
                "d2h_bytes_per_step": n_pairs * 48,
                "api": "raw polar rows (host) -> polar_to_cartesian -> align_consecutive -> chain_poses (device kernel) -> D2H of global poses"},
        "cpu_baseline": {"value": n_pairs / cpu_wall, "unit": "alignments/s", "cores": 1, "kind": kind,
                         "sample": f"all 1,830 pairs, {what}, {cpu_wall:.3f} s wall "
                                   f"(+ {cpu_prep:.3f} s for process.py:38-52's row loop); {its} iterations; {cpu_model()}",
                         "wall_s": cpu_wall, "prep_wall_s": cpu_prep},
        "gpu_wall_fraction_of_cpu": {"kernel_only": ms * 1e-3 / cpu_wall,
                                     "e2e_incl_prep": e2e_ms * 1e-3 / (cpu_wall + cpu_prep),
                                     "target": "< 0.01 (north_star)"},
        "subset_first_1075": {"pairs": 1075, "ms_per_step": ms_1075, "value": 1075 / (ms_1075 * 1e-3),
                              "cpu_wall_s": cpu_wall_1075, "gpu_wall_fraction_of_cpu": ms_1075 * 1e-3 / cpu_wall_1075},
    }
    assert gpu_its == its, (gpu_its, its)
    if ctx is None:
        emit(line)
    return line


def run_allpairs(args, ctx=None):
    """configs[3]: all-pairs loop-closure candidates over 4,096 synthetic scans (8,386,560 pairs),
    30 forced iterations, pairs enumerated row-major (i<j) and split into contiguous ranges."""
    import torch
    import icp_slam_yolo_b200 as m
    from oracle import icp_oracle as orc
    if ctx is None:
        world, rank, local, dev, barrier, max_over_ranks = _dist_setup()
    else:
        world, rank, local, dev, barrier, max_over_ranks = ctx.world, ctx.rank, ctx.local, ctx.dev, ctx.barrier, ctx.max_over_ranks
    n_scans = ALLPAIRS_SCANS
    scans = orc.synth_trajectory_scans(n_scans)
    h_table = torch.from_numpy(scans).pin_memory()
    table = m.ScanTable(h_table.to(dev))
    total = m.triangle_pair_count(n_scans) if args.pairs == 65536 else min(args.pairs, m.triangle_pair_count(n_scans))
    b, e = m.shard_range(total, rank, world)
    mine = e - b
    out = m.alloc_outputs(mine, N_POINTS, dev)
    fp32_peak = m.ffma_probe()

    def step():
        m.align_pairs(table, table, pairing="triangle", first_pair=b, n_pairs=mine,
                      max_iterations=ITERS, tolerance=-1.0, out=out)

    ms = _timed(step, args.steps, args.warmup, barrier, max_over_ranks)
    # e2e: scan table on the host -> device, this rank's share of the pairs, poses / errors / counts back
    h_pose = torch.empty((mine, 6), dtype=torch.float64).pin_memory()
    h_err = torch.empty(mine, dtype=torch.float64).pin_memory()
    h_it = torch.empty(mine, dtype=torch.int32).pin_memory()

    def e2e_step():
        tb = m.ScanTable(h_table.to(dev, non_blocking=True))
        m.align_pairs(tb, tb, pairing="triangle", first_pair=b, n_pairs=mine, max_iterations=ITERS, tolerance=-1.0, out=out)
        h_pose.copy_(out.pose_total, non_blocking=True)
        h_err.copy_(out.error, non_blocking=True)
        h_it.copy_(out.iterations, non_blocking=True)

    e2e_ms = _timed(e2e_step, max(1, args.steps - 1), 1, barrier, max_over_ranks)
    if rank != 0:
        return None
    value = total / (ms * 1e-3)
    line = {
        "metric": "ICP alignments/sec (all-pairs loop closure, 360-pt scans, 30 iters)",
        "value": value, "unit": "alignments/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32 search + f64 state", "data": "synthetic",
        "nn_pairs_per_s": value * PAIR_EVALS_PER_ALIGNMENT,
        "config": {"workload": "configs[3]: all-pairs loop-closure candidate ICP over 4,096 synthetic scans",
                   "pairs_total": total, "pairs_this_rank": mine, "scan_table_bytes": int(scans.nbytes),
                   "l2": "scan table (11.8 MB) is L2 resident by design; outputs 48 B/pair stream to HBM",
                   "parallelism": "triangular pair index split in contiguous ranges, no collective"},
        "gpu_launches": args.steps,
        "roofline": {"bound": "fp32", "kernel": "icp_align_pair_kernel<2,pruned,2 warps>",
                     "achieved": None, "peak": fp32_peak, "unit": "TFLOP/s", "frac": None, "traffic": None,
                     "algorithmic_tflops": mine * PAIR_EVALS_PER_ALIGNMENT * 5 / (ms * 1e-3) / 1e12,
                     "note": "same kernel as the headline; brute-force-equivalent rate, not a utilisation (see the "
                             "headline's roofline.shipped_kernel)"},
        "e2e": {"value": total / (e2e_ms * 1e-3), "unit": "alignments/s", "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": int(scans.nbytes), "d2h_bytes_per_step": mine * 60,
                "api": "host scan table -> device, align_pairs(pairing='triangle') on this rank's range, poses/errors/"
                       "iteration counts -> pinned host"},
        "cpu_baseline": (ctx.cpu_sec.get("allpairs") if ctx is not None else None),
    }
    if ctx is None:
        emit(line)
    return line


def run_single(args, ctx=None):
    """configs[0]: ONE alignment through the reference-shaped call icp(A, B, 30, 1e-5) with NumPy
    arrays in and out (host -> device -> host inside the timed region): scan 1 -> scan 2 of the
    bundled recording (byte-identical 11-point scans: 1 iteration) and scan 4 -> scan 3
    (169 x 176 points, 8 iterations), next to the unmodified reference on one core."""
    import torch
    import icp_slam_yolo_b200 as m
    from oracle import icp_oracle as orc
    raw = _fixture_scans()
    icp_ref, kind, what = reference_icp()
    out = {}
    for name, (a, b) in {"scan1_to_scan2": (0, 1), "scan4_to_scan3": (3, 2)}.items():
        A = np.ascontiguousarray(orc.polar_to_cartesian(raw[a])[:, :2])
        B = np.ascontiguousarray(orc.polar_to_cartesian(raw[b])[:, :2])
        for _ in range(5):
            m.icp(A, B, 30, 1e-5)
        torch.cuda.synchronize()
        reps = 50
        t0 = time.perf_counter()
        for _ in range(reps):
            r = m.icp_full(A, B, 30, 1e-5)
        gpu_ms = (time.perf_counter() - t0) / reps * 1e3
        t0 = time.perf_counter()
        for _ in range(20):
            icp_ref(A, B, 30, 1e-5)
        cpu_ms = (time.perf_counter() - t0) / 20 * 1e3
        out[name] = {"points": [len(A), len(B)], "iterations": int(r.iterations), "error_mm": float(r.error),
                     "gpu_ms_per_call_host_to_host": gpu_ms,
                     "cpu_baseline": {"value": 1e3 / cpu_ms, "unit": "alignments/s", "ms_per_call": cpu_ms, "cores": 1,
                                      "kind": kind, "sample": "20 calls; " + what}}
    out["note"] = ("replicas only (SURVEY.md 8e): a single small alignment is launch- and copy-latency bound on a GPU "
                   "(one CTA of work); reported for completeness, wall clock around the Python call")
    if ctx is None:
        emit({"metric": "single ICP alignment latency (configs[0])", "unit": "ms", **out})
    return out


def run_nn(args, ctx=None, tables=None):
    """The correspondence search alone (b200icp_nn_batch, icp.py:37-38): one search per pair on the
    configs[2] tables; the NN-phase number of the metric ("NN pairs/sec")."""
    import torch
    import icp_slam_yolo_b200 as m
    from oracle import icp_oracle as orc
    if ctx is None:
        world, rank, local, dev, barrier, max_over_ranks = _dist_setup()
    else:
        world, rank, local, dev, barrier, max_over_ranks = ctx.world, ctx.rank, ctx.local, ctx.dev, ctx.barrier, ctx.max_over_ranks
    P = args.pairs
    src_np, tgt_np = tables if tables is not None else orc.synth_room_batch(rank * P, P)
    src, tgt = m.ScanTable(torch.from_numpy(src_np).to(dev)), m.ScanTable(torch.from_numpy(tgt_np).to(dev))
    idx = torch.empty((P, N_POINTS), dtype=torch.int32, device=dev)
    d2 = torch.empty((P, N_POINTS), dtype=torch.float64, device=dev)
    fp32_peak = m.ffma_probe()

    def step():
        m.nn_search(src, tgt, out_idx=idx, out_dist2=d2)

    ms = _timed(step, args.steps, args.warmup, barrier, max_over_ranks)
    dense_ms = _timed(lambda: m.nn_search(src, tgt, out_idx=idx, out_dist2=d2, dense_sweep=True),
                      args.steps, args.warmup, barrier, max_over_ranks)
    if rank != 0:
        return None
    evals = float(P) * N_POINTS * N_POINTS
    line = {
        "metric": "NN pairs/sec (360 x 360 brute-force-equivalent searches)", "value": world * evals / (ms * 1e-3),
        "unit": "pair-evals/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 search + f64 re-decision", "data": "synthetic",
        "config": {"workload": "configs[2] tables, ONE search per pair (%d pairs per GPU x 360 x 360)" % P,
                   "l2": "inputs (377 MB) exceed L2; outputs idx + d2 = %.0f MB per step" % (P * N_POINTS * 12 / 1e6)},
        "gpu_launches": args.steps,
        "roofline": {"bound": "fp32", "kernel": "nn_warp_kernel<6,dense> (every pair evaluated: a utilisation)",
                     "achieved": evals * 5 / (dense_ms * 1e-3) / 1e12, "peak": fp32_peak, "unit": "TFLOP/s",
                     "frac": evals * 5 / (dense_ms * 1e-3) / 1e12 / fp32_peak, "kernel_ms": dense_ms, "traffic": None,
                     "shipped_kernel": {"kernel": "nn_warp_kernel<2,pruned>", "kernel_ms": ms,
                                        "algorithmic_tflops": evals * 5 / (ms * 1e-3) / 1e12,
                                        "algorithmic_speedup_vs_dense": dense_ms / ms},
                     "hbm": {"achieved": P * N_POINTS * (16 + 12) / (ms * 1e-3) / 1e9, "unit": "GB/s",
                             "peak": measured_hbm_peak()[0],
                             "frac": P * N_POINTS * (16 + 12) / (ms * 1e-3) / 1e9 / measured_hbm_peak()[0],
                             "note": "a single search per pair moves 28 B per source point (8 + 8 in, 4 + 8 out): the "
                                     "pruned search alone is closer to the HBM roof than to the FP32 one"}},
    }
    if ctx is None:
        emit(line)
    return line


def run_scan2map(args, ctx=None):
    """configs[4]: 8,192-point scan against a 2^24-point map sharded contiguously across the
    ranks; 30 forced iterations; one all-gather of 32-byte records per iteration."""
    import torch
    import icp_slam_yolo_b200 as m
    from oracle import icp_oracle as orc
    if ctx is None:
        world, rank, local, dev, barrier, max_over_ranks = _dist_setup()
    else:
        world, rank, local, dev, barrier, max_over_ranks = ctx.world, ctx.rank, ctx.local, ctx.dev, ctx.barrier, ctx.max_over_ranks
    M, N = args.map_points, args.scan_points
    b, e = m.shard_range(M, rank, world)
    full = orc.synth_map(M)                               # seeded: every rank draws the same map
    scan_np = orc.synth_scan_for_map(N)
    cpu = None
    if world == 1 and not args.no_cpu_baseline:           # ONE reference iteration: KD-tree over the full map
        icp_ref, kind, what = reference_icp()
        A64, B64 = scan_np.astype(np.float64), full.astype(np.float64)
        t0 = time.perf_counter()
        icp_ref(A64, B64, 1, -1.0)
        one_iter = time.perf_counter() - t0
        cpu = {"value": 1.0 / (one_iter * ITERS), "unit": "alignments/s", "cores": 1, "kind": kind,
               "sample": f"ONE of the 30 iterations of one alignment ({one_iter:.2f} s: KD-tree over all {M} map points "
                         f"rebuilt + {N} queries + best_fit_transform, icp.py:37-45), alignment time = 30 x that; {what}; "
                         f"{cpu_model()}"}
        del A64, B64
    shard = m.MapShard(torch.from_numpy(full[b:e]).to(dev), global_offset=b)
    del full
    h_scan = torch.from_numpy(scan_np).pin_memory()
    scan = h_scan.to(dev)
    exchange = args.s2m_exchange
    hbm_peak, hbm_src = measured_hbm_peak()
    s2m_ncu = ncu_summary("r2_s2m_search_ncu")
    shard_bytes = float(e - b) * 8.0
    use_graph = bool(args.s2m_graph) and exchange != "nccl"      # NCCL calls are not captured
    s2m = m.ScanToMap(shard, N, exchange=exchange, graph=use_graph)
    fp32_peak = m.ffma_probe()

    def step():
        s2m.run(scan, max_iterations=ITERS, tolerance=-1.0, sync=False)

    ms = _timed(step, args.steps, args.warmup, barrier, max_over_ranks)
    res = s2m.result()
    assert res.iterations == ITERS
    # per-kernel split of one alignment: CUDA events on the launching stream around every search / update
    evs = []
    s2m.run(scan, max_iterations=ITERS, tolerance=-1.0, sync=False, events=evs)
    torch.cuda.synchronize()
    search_ms = sum(evs[2 * i].elapsed_time(evs[2 * i + 1]) for i in range(ITERS)) / ITERS
    update_ms = sum(evs[2 * i + 1].elapsed_time(evs[2 * i + 2]) for i in range(ITERS)) / ITERS
    # e2e: scan on the host -> device, the whole loop, state (pose, error, counts) back to the host
    h_state = torch.empty_like(s2m.state, device="cpu").pin_memory()

    def e2e_step():
        d = h_scan.to(dev, non_blocking=True)
        s2m.run(d, max_iterations=ITERS, tolerance=-1.0, sync=False)
        h_state.copy_(s2m.state, non_blocking=True)

    e2e_ms = _timed(e2e_step, args.steps, args.warmup, barrier, max_over_ranks)
    if s2m.peer is not None:
        s2m.peer.close()
    if rank != 0:
        return None
    evals_per_iter = float(N) * float(M)
    line = {
        "metric": "scan-to-map ICP alignments/sec (8,192-pt scan vs 16M-pt map, 30 iters)",
        "value": 1.0 / (ms * 1e-3), "unit": "alignments/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32 search + f64 state", "data": "synthetic",
        "nn_pairs_per_s": evals_per_iter * ITERS / (ms * 1e-3),
        "config": {"workload": "configs[4]: scan-to-map ICP, %d-point scan vs %d-point map, 30 forced iterations" % (N, M),
                   "map_points_this_rank": e - b,
                   "l2": "map shard %.0f MB; a scan point touches ~7 chunks of 8 KB per iteration" % ((e - b) * 8 / 1e6),
                   "parallelism": "map sharded contiguously; %s all-gather of 32 B records per iteration (%d B per rank)" % (
                       "peer stores over NVLink in the search epilogue + flags" if (exchange == "peer" and world > 1) else ("NCCL" if world > 1 else "single rank: none"), N * 32),
                   "cuda_graph": use_graph,
                   "final_error_mm": res.error},
        "gpu_launches": args.steps * s2m.launches,
        "per_iteration_ms": {"search": search_ms, "update_incl_peer_wait": update_ms},
        # the search reads (almost) every chunk of the shard once per iteration -- the union of the
        # scan points' candidate chunks covers the map -- and little else: an HBM-latency-bound kernel
        "roofline": {"bound": "hbm", "kernel": "s2m_search_kernel",
                     "achieved": shard_bytes / (search_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                     "frac": shard_bytes / (search_ms * 1e-3) / 1e9 / hbm_peak, "peak_source": hbm_src,
                     "algorithmic_bytes_per_launch": shard_bytes,
                     "kernel_ms": search_ms,
                     "traffic": (s2m_ncu or {}).get("dram_bytes") if world == 1 else None,
                     "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of one search on ONE GPU, "
                                       "profiles/r2_s2m_search_ncu.json (ncu --set full)" if (s2m_ncu and world == 1) else None,
                     "brute_force_equivalent_tflops": float(N) * (e - b) * 5 / (search_ms * 1e-3) / 1e12,
                     "ffma_peak_tflops": fp32_peak,
                     "note": "algorithmic bytes = this rank's map shard read once per search (8 B per float32 point); "
                             "chunks of 1,024 map points whose bounding circle is provably farther than a point's "
                             "nearest neighbour are skipped, the rest are scanned exactly (FP32 filter + float64), so the "
                             "brute-force-equivalent FLOP rate is a speed-up figure, not a utilisation"},
        "e2e": {"value": 1.0 / (e2e_ms * 1e-3), "unit": "alignments/s", "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": int(h_scan.numel() * 4), "d2h_bytes_per_step": 136,
                "api": "pinned host scan -> device, ScanToMap.run (map shard and circle tables resident), state -> host"},
        "cpu_baseline": cpu,
    }
    if ctx is None:
        emit(line)
    return line


def run_occupancy(args):
    """SURVEY.md 8(f) rank 4: occupancy-grid ray casting (duc/ICP_LIDAR/process.py:114-177).
    (a) replay of the bundled recording: the 1,831 scans of Scan_data_1, poses from the device
        odometry chain, ONE map of the reference's geometry (833 x 1000 cells, 30 mm, +-140-cell
        window), all frames in one launch -- the order-dependent, latency-bound case;
    (b) 296 independent maps x 64 frames x 180 beams (one CTA per map, two per SM).
    value = frames (scans) integrated per second.  The CPU leg times the pure-Python port (the
    reference as shipped, on a bounded sample) and the C restatement, and the device result is
    checked against the C restatement bit for bit inside this run."""
    import torch
    import icp_slam_yolo_b200 as m
    from oracle import icp_oracle as orc
    from oracle import occupancy_oracle as occ
    H, W, RES, AREA = 833, 1000, 30, 140
    CENTER = (W // 2, H // 2)
    world, rank, local, dev, barrier, max_over_ranks = _dist_setup()
    raw = _fixture_scans()
    table = m.scan_io.prepare_scans(raw, device=dev)
    res = m.align_consecutive(table, max_iterations=30, tolerance=1e-5)
    poses = m.chain_poses(res.pose_total)                          # [1831, 6] global pose of every scan
    lens = table.lengths.cpu().numpy()
    xy = table.points.cpu().numpy().astype(np.float64)
    F, pitch = xy.shape[0], xy.shape[1]
    glob = np.zeros((1, F, pitch, 2))
    glob[0, :, :, 0] = poses[:, None, 0] * xy[:, :, 0] + poses[:, None, 1] * xy[:, :, 1] + poses[:, None, 4]
    glob[0, :, :, 1] = poses[:, None, 2] * xy[:, :, 0] + poses[:, None, 3] * xy[:, :, 1] + poses[:, None, 5]
    rob = np.ascontiguousarray(poses[None, :, 4:6])
    l32 = np.ascontiguousarray(lens[None].astype(np.int32))
    h_pts, h_len, h_rob = (torch.from_numpy(a).pin_memory() for a in (glob, l32, rob))
    d_pts, d_len, d_rob = h_pts.to(dev), h_len.to(dev), h_rob.to(dev)
    grid = m.OccupancyGrid(H, W, CENTER, RES, device=dev)

    def reset(g):
        g.probs.fill_(0.5)
        g.image.fill_(128)

    # correctness inside the run: device == C restatement, bit for bit
    grid.update_frames(d_pts, d_len, d_rob, area=AREA)
    o = np.full((H, W), 0.5, dtype=np.float32)
    im = np.full((H, W, 3), 128, dtype=np.uint8)
    t0 = time.perf_counter()
    cells = 0
    for f in range(F):
        occ.update_occupancy_map_c(o, im, glob[0, f, :lens[f]], rob[0, f], CENTER, RES, area=AREA)
    c_wall = time.perf_counter() - t0
    same = bool(np.array_equal(grid.probs_numpy().view(np.uint32), o.view(np.uint32)) and
                np.array_equal(grid.image_numpy(), im))
    assert same, "device occupancy map differs from the oracle"
    # the reference as shipped: pure-Python loops, bounded sample (frames 0..39 of the same replay)
    SAMPLE = 40
    o2 = np.full((H, W), 0.5, dtype=np.float32)
    im2 = np.full((H, W, 3), 128, dtype=np.uint8)
    t0 = time.perf_counter()
    for f in range(SAMPLE):
        occ.update_occupancy_map(o2, im2, glob[0, f, :lens[f]], rob[0, f], CENTER, RES, area=AREA)
    py_wall = time.perf_counter() - t0

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn, before):
        tot = 0.0
        for it in range(max(3, args.warmup) + args.steps):
            before()
            torch.cuda.synchronize()
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            if it >= max(3, args.warmup):
                tot += e0.elapsed_time(e1)
        return tot / args.steps

    ms = timed(lambda: grid.update_frames(d_pts, d_len, d_rob, area=AREA), lambda: reset(grid))
    h_img = torch.empty((H, W, 3), dtype=torch.uint8).pin_memory()

    def e2e():
        p, l, r = h_pts.to(dev, non_blocking=True), h_len.to(dev, non_blocking=True), h_rob.to(dev, non_blocking=True)
        grid.update_frames(p, l, r, area=AREA)
        h_img.copy_(grid.image[0], non_blocking=True)

    e2e_ms = timed(e2e, lambda: reset(grid))
    # (b) independent maps
    NM, NF, NB = 296, 64, 180
    bt = np.zeros((NM, NF, NB, 2))
    br = np.zeros((NM, NF, 2))
    for k in range(8):                                   # 8 distinct replays, tiled over the maps
        bt[k], br[k] = occ.synth_replay(200 + k, NF, beams=NB)
    for k in range(8, NM):
        bt[k], br[k] = bt[k % 8], br[k % 8]
    bg = m.OccupancyGrid(400, 400, (200, 200), RES, n_maps=NM, device=dev)
    b_pts, b_rob = torch.from_numpy(bt).to(dev), torch.from_numpy(br).to(dev)
    bms = timed(lambda: bg.update_frames(b_pts, None, b_rob, area=AREA), lambda: reset(bg))
    # algorithmic bytes: per ray cell one float32 read + write, per frame the window re-rendered
    # (4 B read + 3 B written per cell), 16 B per point
    rays_cells = 0
    for f in range(F):
        n = int(lens[f])
        if n == 0:
            continue
        rx = int(CENTER[0] + rob[0, f, 0] / RES); ry = int(CENTER[1] - rob[0, f, 1] / RES)
        px = (CENTER[0] + glob[0, f, :n, 0] / RES).astype(np.int64); py = (CENTER[1] - glob[0, f, :n, 1] / RES).astype(np.int64)
        ok = (np.abs(px - rx) <= AREA) & (np.abs(py - ry) <= AREA)
        rays_cells += int(np.sum(np.maximum(np.abs(px - rx), np.abs(py - ry))[ok] + 1))
    alg_bytes = rays_cells * 8 + F * (2 * AREA) ** 2 * 7 + int(lens.sum()) * 16
    hbm_peak, hbm_src = measured_hbm_peak()
    if rank != 0:
        return
    line = {
        "metric": "occupancy-grid frames/sec (Scan_data_1 replay, 833 x 1000 cells, +-140-cell window)",
        "value": F / (ms * 1e-3), "unit": "frames/s", "n_gpus": 1, "steps": args.steps, "warmup": max(3, args.warmup),
        "ms_per_step": ms, "higher_is_better": True, "scaling": "replicas", "vs_baseline": None,
        "dtype": "f32 probabilities, f64 cell coordinates, u8 picture", "data": "bundled recording (fixture) + device odometry poses",
        "config": {"workload": "SURVEY 8f-4: update_occupancy_map over the 1,831 scans of Scan_data_1 in order, one map, one launch",
                   "frames": F, "beams_total": int(lens.sum()), "ray_cells_total": rays_cells,
                   "l2": "one 3.3 MB map: L2/L1 resident by design (the update is a dependent chain); maps reset between steps"},
        "gpu_launches": args.steps, "bit_exact_vs_oracle": same,
        "roofline": {"bound": "hbm", "kernel": "occ_update_kernel", "achieved": alg_bytes / (ms * 1e-3) / 1e9,
                     "peak": hbm_peak, "unit": "GB/s", "frac": alg_bytes / (ms * 1e-3) / 1e9 / hbm_peak,
                     "peak_source": hbm_src, "traffic": None, "algorithmic_bytes_per_launch": alg_bytes,
                     "note": "one map is an order-dependent chain (one CTA): latency-bound, not bandwidth-bound; see batched_maps",
                     "us_per_frame": ms * 1e3 / F, "ns_per_beam": ms * 1e6 / float(lens.sum())},
        "batched_maps": {"maps": NM, "frames_per_map": NF, "beams_per_frame": NB, "ms_per_step": bms,
                         "frames_per_s": NM * NF / (bms * 1e-3), "beams_per_s": NM * NF * NB / (bms * 1e-3)},
        "e2e": {"value": F / (e2e_ms * 1e-3), "unit": "frames/s", "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": int(h_pts.numel() * 8 + h_len.numel() * 4 + h_rob.numel() * 8),
                "d2h_bytes_per_step": H * W * 3,
                "api": "OccupancyGrid.update_frames (pinned host points -> device) + D2H of the rendered map"},
        "cpu_baseline": {"value": SAMPLE / py_wall, "unit": "frames/s", "cores": 1, "kind": "port",
                         "sample": f"first {SAMPLE} frames of the same replay, pure-Python port of process.py:86-177 "
                                   f"({py_wall:.2f} s); C restatement, all {F} frames: {c_wall:.3f} s = {F / c_wall:.0f} frames/s; {cpu_model()}"},
    }
    emit(line)


def run_slam(args):
    """The reference's offline SLAM loop (duc/ICP_LIDAR/slam_offline.py:318-455) composed from the
    device primitives (icp_slam-yolo_b200/slam.py) over the first 400 scans of the bundled
    recording: per frame local-map crop, voxel grids, gated scan-to-map ICP with the previous pose,
    dynamic-point removal, occupancy filter, map growth / re-sampling, ray casting, pruning.  The
    loop is host-driven and sequential (every frame needs the previous pose), so the metric is
    wall-clock frames per second around the whole loop, device synchronised at both ends.  CPU
    leg: the same composition of the CPU oracles (oracle/slam_oracle.py), one core."""
    import torch
    import icp_slam_yolo_b200 as m
    from icp_slam_yolo_b200.slam import OfflineSlam, SlamConfig
    from oracle import icp_oracle as orc
    from oracle.slam_oracle import OracleSlam
    FRAMES = 400
    raw = _fixture_scans()[2:2 + FRAMES]
    scans = []
    for r in raw:
        xy = orc.polar_to_cartesian(r)
        scans.append(np.ascontiguousarray(xy))
    t0 = time.perf_counter()
    ora = OracleSlam(SlamConfig())
    ora.first(scans[0])
    o_acc = sum(int(bool(o and o[0])) for o in (ora.step(s) for s in scans[1:]))
    cpu_wall = time.perf_counter() - t0
    torch.cuda.set_device(0)
    walls = []
    for it in range(1 + args.steps):                     # first pass = warm-up
        dev = OfflineSlam(SlamConfig())
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = dev.run(scans)
        torch.cuda.synchronize()
        walls.append(time.perf_counter() - t0)
    wall = min(walls[1:])
    acc = sum(int(bool(r and r.accepted)) for r in res)
    same = bool(np.array_equal(dev.grid.probs_numpy().view(np.uint32), ora.occ.view(np.uint32)) and
                np.allclose(dev.global_pose, ora.pose, atol=1e-6) and acc == o_acc)
    line = {
        "metric": "offline SLAM loop frames/sec (Scan_data_1, first %d scans)" % FRAMES,
        "value": (FRAMES - 1) / wall, "unit": "frames/s", "n_gpus": 1, "steps": args.steps, "warmup": 1,
        "ms_per_step": wall * 1e3, "higher_is_better": True, "scaling": "replicas", "vs_baseline": None,
        "dtype": "f32 search + f64 state; f32 occupancy", "data": "bundled recording (fixture)",
        "config": {"workload": "slam_offline.py:318-455 composed from the device primitives; host-driven, sequential",
                   "frames": FRAMES, "accepted": acc, "map_points": int(dev.global_map.shape[0])},
        "matches_oracle_composition": same,
        "cpu_baseline": {"value": (FRAMES - 1) / cpu_wall, "unit": "frames/s", "cores": 1, "kind": "port",
                         "sample": f"the same {FRAMES} frames through oracle/slam_oracle.py (NumPy/SciPy + C occupancy), "
                                   f"{cpu_wall:.2f} s; {cpu_model()}"},
        "note": "launch- and synchronisation-bound (a dozen small launches and three device-to-host reads per "
                "frame); reported for completeness, not a roofline workload",
    }
    emit(line)


_RESULT_OUT = None


def emit(line):
    """The ONE JSON line of the contract, on the process's original stdout."""
    out = _RESULT_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def _keep_stdout_for_the_result():
    """Libraries print to fd 1 behind Python's back (NCCL's "NCCL version ..." banner when the box sets NCCL_DEBUG):
    point fd 1 at stderr for everything but the result line."""
    global _RESULT_OUT
    sys.stdout.flush()
    _RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def main():
    args = parse()
    _keep_stdout_for_the_result()
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "odometry":
        run_odometry(args)
    elif args.workload == "allpairs":
        run_allpairs(args)
    elif args.workload == "scan2map":
        run_scan2map(args)
    elif args.workload == "single":
        run_single(args)
    elif args.workload == "nn":
        run_nn(args)
    elif args.workload == "occupancy":
        run_occupancy(args)
    elif args.workload == "slam":
        run_slam(args)
    else:
        run_b200(args)
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            dist.destroy_process_group()
    except Exception:
        pass


if __name__ == "__main__":
    main()
