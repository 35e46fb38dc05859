#!/usr/bin/env python
"""Benchmark of the scan-to-map registration hot path (see DESIGN.md "Measurement").

One run measures every BASELINE.json config and prints ONE JSON line:

  headline (top-level keys)  C2/C4: point-to-plane ICP of synthetic 32-beam scans (32 x 940 rays, ~27.6 k points
                             each) against a 1 M-point synthetic map, device-resident Gauss-Newton loop,
                             max_iteration = 10, eps = 0 (exactly 10 iterations).  A step registers a batch of
                             `--scans-per-gpu` scans (default 512 = config 4's 4096 scans over 8 GPUs) on every GPU;
                             ranks hold a replica of the map and a disjoint block of scans, no collective on the data
                             path (weak scaling).  Single-scan tracking latency (config 2 proper) rides along ("track").
  configs.C4_strong          config 4 as written: 4096 scans FIXED, block-partitioned over the ranks, the poses of all
                             scans exchanged over NCCL inside liblocreg.so at the end (locreg_align_batch_sharded).
  configs.C3                 direct NDT (NEARBY6, 1 m voxels, 10 iterations) of a 128 x 1953-ray scan (~225 k points)
                             against a 20 M-point map; replicas only (SURVEY 8e).
  configs.C5                 global relocalisation: 65 536 pose hypotheses of one scan dealt over the ranks, 10
                             iterations + score pass each, ONE ncclAllReduce(MIN) + broadcast inside the timed region
                             (locreg_relocalise_sharded); strong scaling.

Every entry carries value (device-timed, inputs resident / kernels only), e2e (host buffers through the C ABI),
roofline, clocks sampled during its timed region, and - at N = 1 - a cpu_baseline (the oracle on the host cores).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--configs C4S,C3,C5]   our arm (one process per GPU under torchrun)
  python bench.py --impl reference [...]                                      CPU arm: the oracle's restatement of the
                                                                              reference loop on all host threads

--dump-outputs DIR writes what the headline's timed call returned in its last step as DIR/<name>.npy (float64): poses.npy
(S, 7) and one result_<field>.npy (S,) per locreg_result field, S = every scan of the step (all ranks, rank order; the
reference arm: its sample).  The inputs are seeded, so two builds run with the same arguments can be compared output for
output.
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

METRIC = "registered_points_per_sec"
UNIT = "points/s"
BYTES_PER_POINT_ITER = 96  # SURVEY.md §8d: 16 B source float4 + 5 x 16 B gathered neighbours
MAX_ITER = 10
C4_SCANS = 4096


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10,
                    help="timed steps of the headline, C4S and C3 (C5 times one relocalisation of more than 8192 hypotheses)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scans-per-gpu", type=int, default=512)
    ap.add_argument("--map-points", type=int, default=1_000_000)
    ap.add_argument("--cpu-sample-scans", type=int, default=32)  # ~11 s of one host core (the contract asks for 10-30 s)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--configs", default="C4S,C3,C5,LIO",
                    help="comma list of the extra measurements after the headline (C4S, C3, C5, LIO); 'none' = headline only")
    ap.add_argument("--hyp", type=int, default=65536, help="C5: number of pose hypotheses (64x64 xy grid x 16 yaws)")
    ap.add_argument("--ndt-map-points", type=int, default=20_000_000)
    ap.add_argument("--c4-scans", type=int, default=C4_SCANS)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the headline's outputs of its last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def make_world(args):
    from loc_lib_b200 import synth
    w = synth.World(200.0)
    return w, w.sample_map(args.map_points)


def make_scans(world, first, count, total):
    """Scans [first, first+count) of a `total`-long seeded random walk; returns (clouds (n,4), offsets, init poses, gt)."""
    from loc_lib_b200 import synth
    gt_all = world.poses(total)
    gt = gt_all[first:first + count]
    buf, counts = world.scan_batch(gt, seed=synth.SEED_SCAN + first)
    clouds = np.concatenate([buf[i, :counts[i]] for i in range(count)])
    del buf
    offsets = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    init = np.stack([synth.perturb_pose(g, synth.SEED_POSE + 7919 * (first + i)) for i, g in enumerate(gt)])
    return clouds, offsets, init, gt


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons of one GPU sampled every 100 ms for the whole run; every timed region asks
    for the samples that fell inside it (`window`)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.proc = index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))
        except OSError:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        self.join(timeout=2)

    def window(self, t0, t1):
        """Clocks under load between perf_counter() times t0 and t1.  A region shorter than the sampling period takes
        the samples next to it as well (the GPU is busy with the neighbouring warm-up / e2e passes of the same kernels)."""
        rows = [r for t, r in self.rows if t0 <= t <= t1]
        if len(rows) < 3:
            rows = [r for t, r in self.rows if t0 - 0.35 <= t <= t1 + 0.35]
        sm = [float(r[0]) for r in rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def _oracle():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_py as O
    return O


def _pose_delta(a, b):
    d = abs(float(np.dot(a[:4], b[:4]))) / (np.linalg.norm(a[:4]) * np.linalg.norm(b[:4]))
    return 2.0 * float(np.arccos(min(1.0, d))), float(np.linalg.norm(a[4:] - b[4:]))


MAX_DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, poses, results):
    """--dump-outputs: `poses` (S, 7) and `results` (result field -> S values) as float64 out_dir/<name>.npy.  Past
    MAX_DUMP_BYTES in all, a fixed seeded sample of the scans is written, their indices as scan_index.npy."""
    arrays = {"poses": np.asarray(poses, np.float64)}
    arrays.update({"result_" + k: np.asarray(v, np.float64) for k, v in results.items()})
    S = len(arrays["poses"])
    row_bytes = sum(a.nbytes for a in arrays.values()) // max(S, 1)
    if S * row_bytes > MAX_DUMP_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(S, MAX_DUMP_BYTES // (row_bytes + 8), replace=False))
        arrays = {k: a[keep] for k, a in arrays.items()}
        arrays["scan_index"] = keep.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def cpu_baseline_icp(map_cloud, clouds, offsets, init, n_scans, threads):
    """Times the oracle (std-only restatement of IcpRegistration, literal always-on ANN kd-tree search = what the
    reference runs) on `n_scans` scans with `threads` host threads.  Map build is not included (as for the GPU).
    Also reports quirk Q1's visible effect: how often the literal ANN search differs from the exact one, and the pose
    delta that causes (SURVEY.md 8a "contract for the build")."""
    O = _oracle()
    ref = O.OracleIcp(method=O.P2PLANE, max_iteration=MAX_ITER, eps=0.0, nn_mode=O.NN_LITERAL_ANN)
    t0 = time.perf_counter()
    ref.set_target(map_cloud)
    build_s = time.perf_counter() - t0
    S = min(n_scans, len(offsets) - 1)
    t0 = time.perf_counter()
    p_ann, _, used = ref.align_batch(clouds, offsets[:S + 1], init[:S], threads=threads)
    dt = time.perf_counter() - t0
    pts = int(offsets[S])
    out = {"value": pts / dt, "unit": UNIT, "cores": int(used), "kind": "port", "scans_per_s": S / dt,
           "sample": f"{S} scans ({pts} points) x {MAX_ITER} GN iterations, oracle ANN kd-tree (the reference's literal search), "
                     f"{used} thread(s), {dt:.1f} s; kd-tree build {build_s:.1f} s not included",
           "seconds": dt}
    # Q1: exact (this library's contract) vs literal ANN on the first two scans of the sample
    S2 = min(S, 2)
    ex = O.OracleIcp(method=O.P2PLANE, max_iteration=MAX_ITER, eps=0.0, nn_mode=O.NN_EXACT_TIEBREAK)
    ex.set_target(map_cloud)
    p_ex, _, _ = ex.align_batch(clouds, offsets[:S2 + 1], init[:S2], threads=threads)
    q = O.transform_cloud(clouds[:int(offsets[1])], init[0])
    nn_a = ref.knn(q, 5, O.NN_LITERAL_ANN)
    nn_e = ref.knn(q, 5, O.NN_EXACT_TIEBREAK)
    deltas = [_pose_delta(p_ann[i], p_ex[i]) for i in range(S2)]
    out["q1_ann_vs_exact"] = {"nn_rows_differing": float(np.mean(np.any(nn_a != nn_e, axis=1))),
                              "nn_entries_differing": float(np.mean(nn_a != nn_e)),
                              "final_pose_delta_rad_max": max(d[0] for d in deltas),
                              "final_pose_delta_m_max": max(d[1] for d in deltas),
                              "sample": f"5-NN of scan 0 at its initial pose ({len(q)} queries); final poses of {S2} scans"}
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world, map_cloud = make_world(args)
    threads = os.cpu_count() or 1
    S = max(4 * threads, 8)  # bounded sample of the workload: ~1-2 s of CPU work per step on all host threads
    clouds, offsets, init, _ = make_scans(world, 0, S, max(S, 4096))
    O = _oracle()
    ref = O.OracleIcp(method=O.P2PLANE, max_iteration=MAX_ITER, eps=0.0, nn_mode=O.NN_LITERAL_ANN)
    ref.set_target(map_cloud)
    for _ in range(min(args.warmup, 1)):  # one pass over the same sample the steps time (page-in, thread pool)
        ref.align_batch(clouds, offsets, init, threads=threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        poses, res, used = ref.align_batch(clouds, offsets, init, threads=threads)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, poses, {k: [r[k] for r in res] for k in res[0]})
    pts = int(offsets[-1]) * args.steps
    val = pts / dt
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, args.scans_per_gpu,
                                      note="reference arm: each step is a bounded sample of this workload, %d scans on %d host threads" % (S, used)),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": int(used), "kind": "port",
                             "sample": f"{S} scans x {args.steps} steps, oracle ANN kd-tree (reference semantics)"},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "scans_per_s": S * args.steps / dt}
    print(json.dumps(line))


def workload_config(args, scans_per_step, note=""):
    return {"workload": "C2/C4: point-to-plane ICP, 32x940-ray synthetic scans (~27.6k pts) vs 1M-pt synthetic map, "
                        "10 Gauss-Newton iterations (eps=0), device-resident loop",
            "scans_per_gpu_per_step": scans_per_step, "map_points": args.map_points, "max_iteration": MAX_ITER,
            "timing": "inputs larger than L2 (scan batch %.0f MB per step); CUDA events on the launch stream" %
                      (scans_per_step * 27600 * 16 / 1e6), "note": note}


def _peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except (OSError, KeyError, ValueError):
        return 6650.0, "fallback 6650 GB/s (B200_PROFILING.md)"


def _traffic(kernel_names, grid=None):
    """Mean dram__bytes_read + dram__bytes_write per launch over ALL launches of the named kernels (base names, at the
    batch's grid size) in one ncu pass of this command: profiles/roofline_traffic.json, written by
    tools/traffic_from_ncu.py from the launch list tools/profile_remote.sh captures."""
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
    except (OSError, ValueError):
        return None
    recs = [r for r in tj.get("launch_groups", []) if r["kernel"] in kernel_names]
    if not recs:
        return None
    if grid is None:
        grid = max(r["grid"] for r in recs)  # the whole batch (smaller grids = the e2e chunks and single scans)
    tot = sum(r["mean_bytes"] * r["launches"] for r in recs if r["grid"] == grid)
    cnt = sum(r["launches"] for r in recs if r["grid"] == grid)
    return tot / cnt if cnt else None


class Ctx:
    """Process group, device, stream, clocks and the collectives the harness itself needs (max / sum over ranks)."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.args = torch, dist, args
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.world_size = int(os.environ.get("WORLD_SIZE", "1"))
        if self.world_size > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.stream = torch.cuda.current_stream(self.dev)
        self.sampler = ClockSampler(self.local)
        self.sampler.start()
        self.peak, self.peak_src = _peak()

    def barrier(self):
        if self.world_size > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def reduce(self, values, op):
        t = self.torch.tensor(values, dtype=self.torch.float64, device=self.dev)
        if self.world_size > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX if op == "max" else self.dist.ReduceOp.SUM)
        return [float(x) for x in t.cpu()]

    def gather(self, t):
        """Rows of an equally shaped device tensor of every rank, in rank order, on the host."""
        if self.world_size > 1:
            out = self.torch.empty((self.world_size * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=self.dev)
            self.dist.all_gather_into_tensor(out, t.contiguous())
            t = out
        return t.cpu().numpy()

    def close(self):
        self.sampler.stop()
        if self.world_size > 1:
            self.dist.destroy_process_group()


# ---- headline: C2 / C4, weak scaling -------------------------------------------------------------------------------
def bench_icp(ctx, reg, map_cloud, clouds, offsets, init, gt, map_build):
    torch, args, dev, stream = ctx.torch, ctx.args, ctx.dev, ctx.stream
    B = len(offsets) - 1
    n_pts = int(offsets[-1])
    d_src = torch.from_numpy(clouds).to(dev)
    d_off = torch.from_numpy(offsets).to(dev)
    d_pin = torch.from_numpy(init).to(dev)
    d_pout = torch.zeros_like(d_pin)
    d_res = torch.zeros(B * 48, dtype=torch.uint8, device=dev)

    def step_resident():
        reg.ScanMatchBatchDevice(d_src.data_ptr(), d_off.data_ptr(), d_pin.data_ptr(), B, n_pts, d_pout.data_ptr(),
                                 d_res.data_ptr())
        return reg.last_timing()[1]

    # ---- pinned host inputs for `e2e` (the C-ABI call a MatchingInterface user makes, host buffers)
    h_src = torch.from_numpy(clouds).pin_memory()
    h2d = h_src.numel() * 4 + offsets.nbytes + 2 * init.nbytes
    d2h = B * 7 * 8 + B * 48

    def step_e2e():
        return reg.ScanMatchBatch(h_src.numpy(), offsets, init)[0]

    warm = max(args.warmup, 3)
    for _ in range(warm):
        step_resident()
    # sanity: the registered poses must be the right ones (median translation error vs ground truth)
    err = np.median(np.linalg.norm(d_pout.cpu().numpy()[:, 4:] - gt[:, 4:], axis=1))

    ctx.barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    wall0 = time.perf_counter()
    ev0.record(stream)
    launches = 0
    for _ in range(args.steps):
        launches += step_resident()
    ev1.record(stream)
    ctx.barrier()
    wall1 = time.perf_counter()
    dev_ms = ev0.elapsed_time(ev1)
    if args.dump_outputs:  # what the last timed step handed its caller: poses and locreg_result records
        from loc_lib_b200 import _lib
        poses, rec = ctx.gather(d_pout), ctx.gather(d_res.view(B, -1))
        rec = np.frombuffer(rec.tobytes(), np.dtype(_lib.Result))
        if ctx.rank == 0:
            dump_outputs(args.dump_outputs, poses, {k: rec[k] for k in rec.dtype.names if k != "pad_"})

    # ---- end to end through host buffers
    for _ in range(2):
        step_e2e()
    ctx.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    ctx.barrier()
    e2e_s = time.perf_counter() - t0
    clocks = ctx.sampler.window(wall0, wall1)

    # ---- kernel-class breakdown for the roofline (separate instrumented pass, not part of the timed steps)
    reg.profile(True)
    for _ in range(3):
        step_resident()
    prof = reg.profile(False)

    # ---- single-scan tracking latency (config 2)
    one = clouds[:int(offsets[1])]
    h_one = torch.from_numpy(one).pin_memory().numpy()
    lat_k, lat_w, n_launch = [], [], 0
    for i in range(40):
        t0 = time.perf_counter()
        reg.ScanMatch(h_one, init[0], want_cloud=True)
        lat_w.append((time.perf_counter() - t0) * 1e3)
        lat_k.append(reg.last_timing()[0])
        n_launch = reg.last_timing()[1]
    track = {"scan_points": int(offsets[1]), "kernel_ms": float(np.median(lat_k[10:])), "e2e_ms": float(np.median(lat_w[10:])),
             "points_per_s_e2e": int(offsets[1]) / (np.median(lat_w[10:]) * 1e-3), "launches_per_scan_match": int(n_launch),
             "roofline_frac": BYTES_PER_POINT_ITER * int(offsets[1]) * MAX_ITER / (np.median(lat_k[10:]) * 1e-3) / 1e9 / ctx.peak}

    dev_ms, e2e_ms = ctx.reduce([dev_ms, e2e_s * 1e3], "max")
    total_pts, = ctx.reduce([float(n_pts)], "sum")
    del d_src, h_src
    if ctx.rank != 0:
        return None
    W = ctx.world_size
    nn_ms, nn_launches = prof["search"]
    fit_ms, fit_launches = prof["fit"]
    ring_ms, _ = prof["rings"]
    solve_ms, _ = prof["solve"]
    per_launch_ms = nn_ms / max(nn_launches, 1)
    achieved = BYTES_PER_POINT_ITER * n_pts / (per_launch_ms * 1e-3) / 1e9 if per_launch_ms > 0 else None
    pipe_ms = (nn_ms + fit_ms + ring_ms + solve_ms) / max(nn_launches, 1)  # one whole Gauss-Newton iteration
    value = total_pts * args.steps / (dev_ms * 1e-3)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": W, "steps": args.steps, "warmup": warm,
        "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": workload_config(args, B),
        "scans_per_s": W * B * args.steps / (dev_ms * 1e-3),
        "point_iterations_per_s": value * MAX_ITER,
        "e2e": {"value": total_pts * args.steps / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": int(d2h), "scans_per_s": W * B * args.steps / (e2e_ms * 1e-3),
                "api": "locreg_align_batch (host buffers, pinned)"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"bound": "hbm", "kernel": "k_icp_nn<5> (neighbour search stage 1, %.0f%% of pipeline kernel time)" %
                     (100 * nn_ms / max(nn_ms + fit_ms + ring_ms + solve_ms, 1e-9)),
                     "achieved": achieved, "peak": ctx.peak, "unit": "GB/s", "frac": achieved / ctx.peak if achieved else None,
                     "traffic": _traffic(("k_icp_nn", "k_icp_nn_staged")) if B == 512 else None, "peak_source": ctx.peak_src,
                     "traffic_note": "mean dram read+write bytes per stage-1 search launch (k_icp_nn, k_icp_nn_staged) over ALL such launches of the batch in an ncu pass of this command (profiles/roofline_traffic.json; null when the pass was taken on another batch size)",
                     "algorithmic_bytes_per_launch": BYTES_PER_POINT_ITER * n_pts, "launch_ms": per_launch_ms,
                     "fit_kernel_launch_ms": fit_ms / max(fit_launches, 1),
                     "rings_kernel_launch_ms": ring_ms / max(nn_launches, 1),
                     "iteration_ms": pipe_ms,
                     "iteration_achieved": BYTES_PER_POINT_ITER * n_pts / (pipe_ms * 1e-3) / 1e9 if pipe_ms > 0 else None,
                     "iteration_frac": BYTES_PER_POINT_ITER * n_pts / (pipe_ms * 1e-3) / 1e9 / ctx.peak if pipe_ms > 0 else None,
                     "step_frac": BYTES_PER_POINT_ITER * n_pts * MAX_ITER / (dev_ms / args.steps * 1e-3) / 1e9 / ctx.peak,
                     "note": "96 B per point-iteration (SURVEY 8d) x points per launch; the map (16 MB of points + "
                             "neighbour lists) is mostly L2/L1 resident: the DRAM traffic is the scan points plus the "
                             "per-point search state, and stays below this.  step_frac = the same bytes for all ten "
                             "iterations over the measured ms_per_step (everything included)"},
        "track": track,
        "map_build": map_build,
        "check": {"median_translation_error_m": float(err), "wall_s_timed_region": wall1 - wall0},
    }
    if not args.no_cpu_baseline and W == 1:
        line["cpu_baseline"] = cpu_baseline_icp(map_cloud, clouds, offsets, init, args.cpu_sample_scans, 1)
    return line


# ---- C4 as written: 4096 scans fixed (strong scaling), poses exchanged over NCCL inside the library ------------------
def bench_c4_strong(ctx, reg, clouds, offsets, init, gt, S_global):
    torch, args, dev, stream = ctx.torch, ctx.args, ctx.dev, ctx.stream
    S_local = len(offsets) - 1
    n_pts = int(offsets[-1])
    d_src = torch.from_numpy(clouds).to(dev)
    d_off = torch.from_numpy(offsets).to(dev)
    d_pin = torch.from_numpy(init).to(dev)
    d_pout = torch.zeros_like(d_pin)
    d_res = torch.zeros(max(S_local, 1) * 48, dtype=torch.uint8, device=dev)
    steps = args.steps

    def step_resident():
        reg.ScanMatchBatchDevice(d_src.data_ptr(), d_off.data_ptr(), d_pin.data_ptr(), S_local, n_pts, d_pout.data_ptr(), d_res.data_ptr())
        return reg.last_timing()[1]

    h_src = torch.from_numpy(clouds).pin_memory()

    def step_e2e():
        return reg.ScanMatchBatchSharded(h_src.numpy(), offsets, init, S_global)[0]

    for _ in range(2):
        step_resident()
    ctx.barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    wall0 = time.perf_counter()
    ev0.record(stream)
    launches = 0
    for _ in range(steps):
        launches += step_resident()
    ev1.record(stream)
    ctx.barrier()
    wall1 = time.perf_counter()
    dev_ms = ev0.elapsed_time(ev1)
    poses = step_e2e()
    ctx.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        poses = step_e2e()
    ctx.barrier()
    e2e_s = time.perf_counter() - t0
    clocks = ctx.sampler.window(wall0, wall1)
    dev_ms, e2e_ms = ctx.reduce([dev_ms, e2e_s * 1e3], "max")
    total_pts, = ctx.reduce([float(n_pts)], "sum")
    # every rank holds the poses of ALL scans after the exchange: check its own block against ground truth, and that
    # foreign blocks arrived (non-zero quaternions)
    from loc_lib_b200 import dist as D
    lo, hi = D.shard_range(S_global, ctx.rank, ctx.world_size)
    err = float(np.median(np.linalg.norm(poses[lo:hi, 4:] - gt[:, 4:], axis=1))) if hi > lo else 0.0
    filled = bool(np.all(np.abs(np.linalg.norm(poses[:, :4], axis=1) - 1.0) < 1e-6))
    del d_src, h_src
    if ctx.rank != 0:
        return None
    W = ctx.world_size
    value = total_pts * steps / (dev_ms * 1e-3)
    return {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": W, "steps": steps, "warmup": 2,
            "ms_per_step": dev_ms / steps, "higher_is_better": True, "scaling": "strong", "dtype": "f64",
            "scans_per_s": S_global * steps / (dev_ms * 1e-3),
            "config": {"workload": "C4: batch offline mapping, %d scans FIXED, block-partitioned over %d rank(s) (%d on rank 0), "
                                   "P2Plane ICP 10 iterations vs 1M-pt map" % (S_global, W, S_local),
                       "timing": "scan block %.0f MB per rank (larger than L2); CUDA events on the launch stream" % (n_pts * 16 / 1e6)},
            "e2e": {"value": total_pts * steps / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(n_pts * 16 + offsets.nbytes + 2 * init.nbytes),
                    "d2h_bytes_per_step": int(S_global * (7 * 8 + 48)), "scans_per_s": S_global * steps / (e2e_ms * 1e-3),
                    "api": "locreg_align_batch_sharded (host block in, poses of ALL scans out)",
                    "collective": "grouped ncclBroadcast per rank (ragged all-gather) of %d poses + results on the handle's stream, inside the timed region" % S_global
                                  if W > 1 else "none (one rank)"},
            "gpu_launches": int(launches), "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "whole Gauss-Newton pipeline (10 iterations)",
                         "achieved": BYTES_PER_POINT_ITER * total_pts * MAX_ITER * steps / (dev_ms * 1e-3) / 1e9 / W, "peak": ctx.peak,
                         "unit": "GB/s per GPU", "frac": BYTES_PER_POINT_ITER * total_pts * MAX_ITER * steps / (dev_ms * 1e-3) / 1e9 / W / ctx.peak,
                         "traffic": None, "peak_source": ctx.peak_src},
            "check": {"median_translation_error_m": err, "all_blocks_received": filled}}


# ---- C3: direct NDT --------------------------------------------------------------------------------------------------
def bench_ndt(ctx):
    """Config 3: direct NDT (NEARBY6, 1 m voxels, 10 iterations) of a 128-beam scan (~225 k points) against a 20 M-point
    map; one scan in flight, whole AlignNdt loop in one cooperative launch.  Replicas only: every rank runs the same job."""
    import loc_lib_b200 as L
    from loc_lib_b200 import synth
    torch, args, dev = ctx.torch, ctx.args, ctx.dev
    w = synth.World(900.0)
    t0 = time.perf_counter()
    m = w.sample_map(args.ndt_map_points)
    gen_s = time.perf_counter() - t0
    gts = w.poses(4)
    scans = [w.scan(g, beams=128, azimuth=1953, seed=synth.SEED_SCAN + i) for i, g in enumerate(gts)]
    init = synth.perturb_poses(gts)
    reg = L.NdtRegistration(L.NdtOptions(max_iteration_=MAX_ITER, eps_=0.0), device=ctx.local)
    reg.set_stream(ctx.stream.cuda_stream)
    t0 = time.perf_counter()
    reg.SetInputTarget(m)
    build_wall = (time.perf_counter() - t0) * 1e3
    build_kernel = reg.last_timing()[0]
    nv = len(reg.Voxels()[3])
    pinned = [torch.from_numpy(s).pin_memory().numpy() for s in scans]
    warm = max(args.warmup, 3)
    for i in range(warm):
        reg.ScanMatch(pinned[i % 4], init[i % 4], want_cloud=False)
    ctx.barrier()
    # `value`: the handle's CUDA events around the kernels of each ScanMatch (the scan is in HBM by then; the 149 MB voxel
    # table and the four scans in rotation keep L2 from holding the inputs); `e2e`: the same calls by wall clock -
    # pinned host scan in, pose out
    hits, errs, k_ms, pts, launches = [], [], [], 0, 0
    wall0 = time.perf_counter()
    for i in range(args.steps):
        _, _, pose = reg.ScanMatch(pinned[i % 4], init[i % 4], want_cloud=False)
        k_ms.append(reg.last_timing()[0])
        launches += reg.last_timing()[1]
        pts += len(scans[i % 4])
        hits.append(reg.last_result["n_inlier"] / max(reg.last_result["n_effective"], 1))
        errs.append(float(np.linalg.norm(pose[4:] - gts[i % 4][4:])))
    ctx.barrier()
    wall1 = time.perf_counter()
    e2e_s = wall1 - wall0
    dev_ms = float(np.sum(k_ms))
    clocks = ctx.sampler.window(wall0, wall1)
    dev_ms, e2e_ms = ctx.reduce([dev_ms, e2e_s * 1e3], "max")
    total_pts, = ctx.reduce([float(pts)], "sum")
    out = None
    if ctx.rank == 0:
        W = ctx.world_size
        h = float(np.mean(hits))
        bytes_pt = 16 + 7 * 16 + h * 96
        dev_s = dev_ms * 1e-3
        out = {"metric": METRIC, "value": total_pts / dev_s, "unit": UNIT, "n_gpus": W, "steps": args.steps,
               "warmup": warm, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
               "scaling": "replicas only (one scan cannot amortise an exchange per iteration: SURVEY 8e)", "dtype": "f64",
               "config": {"workload": "C3: direct NDT (NEARBY6, voxel 1.0 m), 128x1953-ray synthetic scan vs %d-pt synthetic map, "
                                      "10 Gauss-Newton iterations (eps=0), one cooperative launch per ScanMatch" % len(m),
                          "scan_points": int(np.mean([len(s) for s in scans])), "voxels": nv,
                          "timing": "one scan in flight, four scans in rotation; the %d-voxel table (%.0f MB) exceeds L2; CUDA events on the launch stream" % (nv, nv * 112 / 1e6)},
               "e2e": {"value": total_pts / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(scans[0].nbytes), "d2h_bytes_per_step": 7 * 8 + 48,
                       "api": "locreg_align (pinned host scan in, pose out)"},
               "gpu_launches": int(launches), "clocks": clocks,
               "roofline": {"bound": "hbm", "kernel": "k_align_persist<NdtProblem> (10 iterations in one launch)",
                            "achieved": bytes_pt * pts * MAX_ITER / dev_s / 1e9, "peak": ctx.peak, "unit": "GB/s",
                            "frac": bytes_pt * pts * MAX_ITER / dev_s / 1e9 / ctx.peak, "traffic": _traffic("k_align_persist"), "peak_source": ctx.peak_src,
                            "bytes_per_point_iteration": bytes_pt, "hits_per_point": h,
                            "note": "16 B point + 7 x 16 B probes + hits x 96 B voxel records per point-iteration (SURVEY 8d)"},
               "map_build": {"wall_ms": build_wall, "kernel_ms": build_kernel, "points": int(len(m)), "gen_s": gen_s,
                             "points_per_s": len(m) / (build_kernel * 1e-3) if build_kernel else None},
               "check": {"median_translation_error_vs_ground_truth_m": float(np.median(errs)),
                         "note": "ten iterations of the reference's unweighted NDT Gauss-Newton (quirk Q8) from a 0.3 m / 2 deg error do not "
                                 "reach the ground truth on 1 m voxels; parity is against the oracle (cpu_baseline.pose_vs_gpu)"}}
        if not args.no_cpu_baseline and W == 1:
            # the oracle's AlignNdt only ever looks at voxels the scan reaches: build it from the part of the map within
            # 120 m of the sensor (scan range 100 m + initial error) - same result, a bounded build
            O = _oracle()
            c = gts[0][4:6]
            near = m[(np.abs(m[:, 0] - c[0]) < 120.0) & (np.abs(m[:, 1] - c[1]) < 120.0)]
            ref = O.OracleNdt(max_iteration=MAX_ITER, eps=0.0)
            t0 = time.perf_counter()
            ref.set_target(near)
            b_s = time.perf_counter() - t0
            t0 = time.perf_counter()
            p_ref, _, _, _ = ref.align(scans[0], init[0], want_cloud=False)
            dt = time.perf_counter() - t0
            _, _, p_gpu = reg.ScanMatch(pinned[0], init[0], want_cloud=False)
            drad, dm = _pose_delta(p_ref, p_gpu)
            out["cpu_baseline"] = {"value": len(scans[0]) / dt, "unit": UNIT, "cores": 1, "kind": "port", "seconds": dt,
                                   "sample": "1 scan (%d points) x %d iterations, oracle AlignNdt (std::unordered_map grid), 1 thread; grid built "
                                             "from the %d map points within 120 m of the sensor (%.1f s, not included)" % (len(scans[0]), MAX_ITER, len(near), b_s),
                                   "pose_vs_gpu": {"rad": drad, "m": dm}}
    del reg
    torch.cuda.empty_cache()
    if ctx.rank == 0:
        # the ICP search index over the same 20 M-point map (SURVEY 8a-1 at config 3's map size): build time and size
        icp = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE, max_iteration_=MAX_ITER, eps_=0.0), device=ctx.local)
        t0 = time.perf_counter()
        icp.SetInputTarget(m)
        w0 = (time.perf_counter() - t0) * 1e3
        t0 = time.perf_counter()
        icp.SetInputTarget(m)
        w1 = (time.perf_counter() - t0) * 1e3
        ib, ip, il = icp.index_info()
        out["icp_index_20M"] = {"first_build_wall_ms": w0, "rebuild_wall_ms": w1, "rebuild_device_ms": icp.last_timing()[0],
                                "index_bytes": int(ib), "index_bytes_per_point": ib / max(ip, 1), "neighbourhood_lists": int(il),
                                "note": "wall includes the H2D copy of the 320 MB cloud (pageable)"}
        del icp
        torch.cuda.empty_cache()
    return out


def reloc_hypotheses(gt, n_hyp):
    """64 x 64 xy grid (0.5 m pitch, centred on gt) x 16 yaws (22.5 deg), truncated / tiled to n_hyp (SURVEY 8d)."""
    g = (np.arange(64) - 31.5) * 0.5
    out = []
    ax, ay, az, aw = gt[:4]
    for k in range(16):
        a = k * np.pi / 8
        bz, bw = np.sin(a / 2), np.cos(a / 2)  # yaw about the sensor's z axis: q = q_gt * (0, 0, bz, bw)
        q = np.array([ax * bw + ay * bz, ay * bw - ax * bz, az * bw + aw * bz, aw * bw - az * bz])
        for y in g:
            for x in g:
                out.append(np.concatenate([q, [gt[4] + x, gt[5] + y, gt[6]]]))
    hyp = np.array(out)
    return hyp[np.resize(np.arange(len(hyp)), n_hyp)] if n_hyp != len(hyp) else hyp


# ---- C5: global relocalisation ---------------------------------------------------------------------------------------
def bench_reloc(ctx, reg, world, map_cloud):
    """Config 5: hypotheses dealt over the ranks, ONE ncclAllReduce(MIN) + broadcast on the handle's stream picks the
    winner - inside locreg_relocalise_sharded, inside the timed region."""
    args = ctx.args
    gt = world.poses(3)[2]
    scan = world.scan(gt)
    hyp = reloc_hypotheses(gt, args.hyp)
    warm = hyp[:: max(1, len(hyp) // (256 * ctx.world_size))][:256 * ctx.world_size]
    for _ in range(2):
        reg.RelocaliseSharded(scan, warm)
    steps = 1 if len(hyp) > 8192 else args.steps
    times, kernel, launches = [], [], 0
    ctx.barrier()
    wall0 = time.perf_counter()
    for _ in range(steps):
        ctx.barrier()
        t0 = time.perf_counter()
        pose, idx, score = reg.RelocaliseSharded(scan, hyp)
        ctx.barrier()
        times.append(time.perf_counter() - t0)
        kernel.append(reg.last_timing()[0])
        launches += reg.last_timing()[1]
    wall1 = time.perf_counter()
    clocks = ctx.sampler.window(wall0, wall1)
    step_s, kern_ms = ctx.reduce([float(np.mean(times)), float(np.mean(kernel))], "max")
    if ctx.rank != 0:
        return None
    W = ctx.world_size
    evals = MAX_ITER + 1  # ten Gauss-Newton iterations + the score pass
    algo = BYTES_PER_POINT_ITER * len(scan) * evals * len(hyp)
    out = {"metric": "relocalisation_hypotheses_per_sec", "value": len(hyp) / (kern_ms * 1e-3), "unit": "hypotheses/s",
           "n_gpus": W, "steps": steps, "warmup": 2, "ms_per_step": kern_ms, "higher_is_better": True,
           "scaling": "strong", "dtype": "f64",
           "registered_points_per_s": len(hyp) * len(scan) / (kern_ms * 1e-3),
           "config": {"workload": "C5: global relocalisation, %d pose hypotheses (64x64 xy grid 0.5 m x 16 yaws) of one 32-beam "
                                  "scan (%d pts) vs 1M-pt map, P2Plane ICP 10 iterations + score pass each, dealt round-robin over "
                                  "%d rank(s)" % (len(hyp), len(scan), W), "hypotheses": len(hyp),
                      "collective": "ncclAllReduce(MIN, uint64 (score bits << 32 | global index), count 1) + ncclBroadcast(8 doubles) "
                                    "on the handle's stream inside locreg_relocalise_sharded" if W > 1 else "none (one rank)",
                      "stage2_queue": "spatial order (counting sort of the queued queries by 1 m bin, Morton order inside hashed 8 m groups), waves of 4 GiB neighbour scratch",
                      "timing": "CUDA events of the handle (kernels + both collectives), max over ranks; per-point scratch of a wave ~20 GB (larger than L2)"},
           "e2e": {"value": len(hyp) / step_s, "unit": "hypotheses/s", "ms_per_step": step_s * 1e3,
                   "h2d_bytes_per_step": int(scan.nbytes + hyp.nbytes // W), "d2h_bytes_per_step": 8 + 8 * 8,
                   "api": "locreg_relocalise_sharded (host scan + hypotheses in, winner out; wall clock between barriers)"},
           "gpu_launches": int(launches), "clocks": clocks,
           "roofline": {"bound": "hbm", "kernel": "whole pipeline (stage-2 search k_icp_nn_finish on the spatially ordered queue dominates: far hypotheses)",
                        "achieved": algo / (kern_ms * 1e-3) / 1e9 / W, "peak": ctx.peak, "unit": "GB/s per GPU",
                        "frac": algo / (kern_ms * 1e-3) / 1e9 / W / ctx.peak, "traffic": None, "peak_source": ctx.peak_src,
                        "note": "96 B x scan points x 11 evaluations x hypotheses"},
           "best": {"index": int(idx), "score": float(score), "translation_error_m": float(np.linalg.norm(pose[4:] - gt[4:]))}}
    if not args.no_cpu_baseline and W == 1:
        O = _oracle()
        ref = O.OracleIcp(method=O.P2PLANE, max_iteration=MAX_ITER, eps=0.0, nn_mode=O.NN_LITERAL_ANN)
        ref.set_target(map_cloud)
        sample = hyp[:: max(1, len(hyp) // 16)][:16]
        clouds = np.concatenate([scan] * len(sample))
        offs = np.arange(len(sample) + 1, dtype=np.int64) * len(scan)
        t0 = time.perf_counter()
        _, _, used = ref.align_batch(clouds, offs, sample, threads=1)
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": len(sample) / dt, "unit": "hypotheses/s", "cores": int(used), "kind": "port", "seconds": dt,
                               "sample": "%d hypotheses (every %d-th) x 10 iterations of the same scan, oracle ANN kd-tree, 1 thread; "
                                         "no score pass (the reference has none: GetFitnessScore returns 0)" % (len(sample), max(1, len(hyp) // 16))}
    return out


# ---- Lio key-frame step (SURVEY 8f): incremental NDT voxel cache updated on the device ---------------------------------
def bench_lio_keyframe(ctx, world):
    """Lio::AddCloud's key-frame block for incremental NDT (lio.cpp:277-307, ndt_registration.cpp:150-236): transform the
    scan, add it to the LRU voxel cache (order, evictions, statistics: all kernels, nothing copied back), publish the
    table.  Timed per key frame through locreg_local_map_add_keyframe with a pinned host scan; the small-capacity run
    evicts on every key frame."""
    import loc_lib_b200 as L
    torch = ctx.torch
    gt = world.poses(40)
    scans = [torch.from_numpy(world.scan(g)).pin_memory().numpy() for g in gt]
    out = {}
    for name, capacity in (("capacity_100000", 100000), ("capacity_5000", 5000)):
        reg = L.NdtRegistration(L.NdtOptions(method_=L.NdtMethod.INCREMENTAL_NDT, capacity_=capacity), device=ctx.local)
        wall, kern = [], []
        for sc, g in zip(scans, gt):
            ctx.torch.cuda.synchronize(ctx.dev)
            t0 = time.perf_counter()
            reg.AddKeyFrame(sc, g, max_keyframes=10, leaf=0.5)
            ctx.torch.cuda.synchronize(ctx.dev)
            wall.append((time.perf_counter() - t0) * 1e3)
            kern.append(reg.last_timing()[0])
        out[name] = {"keyframe_wall_ms": float(np.median(wall[8:])), "cache_update_kernel_ms": float(np.median(kern[8:])),
                     "voxels_cached": int(len(reg.Voxels()[0])), "scan_points": int(len(scans[0])), "keyframes": len(scans)}
        del reg
    out["note"] = ("locreg_local_map_add_keyframe, method = incremental NDT: H2D of the scan, double-precision transform, LRU cache "
                   "update + statistics + table publish on the device (no D2H, no host LRU); median over key frames 9-40")
    return out


def run_ours(args):
    import loc_lib_b200 as L
    from loc_lib_b200 import dist as D
    ctx = Ctx(args)
    want = set() if args.configs.lower() == "none" else {c.strip().upper() for c in args.configs.split(",") if c.strip()}
    world, map_cloud = make_world(args)
    B = args.scans_per_gpu
    W = ctx.world_size
    reg = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE, max_iteration_=MAX_ITER, eps_=0.0), device=ctx.local)
    reg.set_stream(ctx.stream.cuda_stream)
    t0 = time.perf_counter()
    reg.SetInputTarget(map_cloud)
    map_build = {"wall_ms": (time.perf_counter() - t0) * 1e3, "kernel_ms": reg.last_timing()[0], "points": int(len(map_cloud))}
    # the same index again on warm buffers (what Loc's re-crop and Lio's key frames pay), and its size
    walls, spans = [], []
    for _ in range(3):
        t0 = time.perf_counter()
        reg.SetInputTarget(map_cloud)
        walls.append((time.perf_counter() - t0) * 1e3)
        spans.append(reg.last_timing()[0])
    ib, ip, il = reg.index_info()
    map_build.update({"rebuild_wall_ms": float(np.median(walls)), "rebuild_device_ms": float(np.median(spans)), "index_bytes": int(ib),
                      "index_bytes_per_point": ib / max(ip, 1), "neighbourhood_lists": int(il),
                      "note": "wall_ms / kernel_ms: first build (allocates the index); rebuild_*: warm buffers, H2D of the 16 MB cloud included in wall"})
    if ctx.rank == 0:
        nl = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE, max_iteration_=MAX_ITER, eps_=0.0, knn_lists=0), device=ctx.local)
        nl.SetInputTarget(map_cloud)
        t0 = time.perf_counter()
        nl.SetInputTarget(map_cloud)
        w_nl = (time.perf_counter() - t0) * 1e3
        nb, np_, _ = nl.index_info()
        map_build["knn_lists_0"] = {"rebuild_wall_ms": w_nl, "index_bytes_per_point": nb / max(np_, 1)}
        sc, so, si, _ = make_scans(world, 0, 64, 4096)
        nl.ScanMatchBatch(sc, so, si)
        t0 = time.perf_counter()
        nl.ScanMatchBatch(sc, so, si)
        map_build["knn_lists_0"]["points_per_s_64_scans"] = int(so[-1]) / max(nl.last_timing()[0] * 1e-3, 1e-9)
        map_build["knn_lists_0"]["note"] = "block tables only (no neighbourhood lists): every query takes the shell search; 64-scan batch, device time"
        del nl
    if W > 1:
        D.comm_init(reg, ctx.dev)  # NCCL communicator INSIDE liblocreg.so (the id travels over the torchrun process group)

    # the rank's block of config 4's 4096-scan walk; the headline batch is its first B scans
    S_global = args.c4_scans
    lo, hi = D.shard_range(S_global, ctx.rank, W)
    n_mine = max(hi - lo, B) if "C4S" in want else B
    clouds, offsets, init, gt = make_scans(world, lo, n_mine, max(S_global, lo + n_mine))
    line = bench_icp(ctx, reg, map_cloud, clouds[:int(offsets[B])], offsets[:B + 1], init[:B], gt[:B], map_build)
    extra = {}
    if "C4S" in want:
        S_loc = hi - lo
        extra["C4_strong"] = bench_c4_strong(ctx, reg, clouds[:int(offsets[S_loc])], offsets[:S_loc + 1], init[:S_loc], gt[:S_loc], S_global)
    del clouds
    if "C5" in want:
        extra["C5"] = bench_reloc(ctx, reg, world, map_cloud)
    del reg
    ctx.torch.cuda.empty_cache()
    if "C3" in want:
        extra["C3"] = bench_ndt(ctx)
    if "LIO" in want and ctx.rank == 0:
        extra["lio_keyframe"] = bench_lio_keyframe(ctx, world)
    if ctx.rank == 0:
        if extra:
            line["configs"] = extra
        print(json.dumps(line))
    ctx.close()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
