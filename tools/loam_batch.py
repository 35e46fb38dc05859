"""LOAM batch throughput: locreg_align_loam_batch (LoamRegistration.ScanMatchBatch, all scans in one device-resident
loop) against a loop of single locreg_align_loam calls (LoamRegistration.ScanMatch), one per scan.  C4-style workload:
S scans of World(200) at World.poses(S) (scan_batch), registered from perturb_poses against the 1 M-point map; each scan
is cut by a seeded permutation into 8192 surf and 2048 edge points, as in tools/loam_latency.py.  10 trips, eps 0.  The
two paths alternate in one process after a warm-up; both must give bit-identical poses and results.  Writes one JSON
file (--out)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import loc_lib_b200 as L  # noqa: E402
from loc_lib_b200 import synth  # noqa: E402

N_SURF, N_EDGE = 8192, 2048


def stats(v):
    v = np.asarray(v, float)
    return {"median": float(np.median(v)), "p10": float(np.percentile(v, 10)), "p90": float(np.percentile(v, 90)),
            "min": float(v.min()), "max": float(v.max())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scans", type=int, default=512)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default="r4_loam_batch.json")
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    S = args.scans
    w = synth.World(200.0)
    m = w.sample_map(1_000_000)
    gt = w.poses(S)
    buf, counts = w.scan_batch(gt)
    init = synth.perturb_poses(gt, synth.SEED_POSE)
    assert counts.min() >= N_SURF + N_EDGE, counts.min()
    rng = np.random.default_rng(7)
    surfs, edges = [], []
    for s in range(S):
        idx = rng.permutation(int(counts[s]))
        surfs.append(buf[s, idx[:N_SURF]])
        edges.append(buf[s, idx[N_SURF:N_SURF + N_EDGE]])
    surf, edge = np.ascontiguousarray(np.concatenate(surfs)), np.ascontiguousarray(np.concatenate(edges))
    so = np.arange(S + 1, dtype=np.int64) * N_SURF
    eo = np.arange(S + 1, dtype=np.int64) * N_EDGE
    del buf
    iters, eps = 10, 0.0
    loam = L.LoamRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE, max_iteration_=iters, eps_=eps),
                              L.IcpOptions(method_=L.IcpMethod.P2LINE, max_iteration_=iters, eps_=eps), iters, eps)
    loam.SetInputTarget(m, m)
    single = {"wall_ms": [], "kernel_ms": [], "launches": []}
    batch = {"wall_ms": [], "kernel_ms": [], "launches": []}
    for rep in range(args.warmup + args.reps):
        t0 = time.perf_counter()
        lp, lr, k_ms, k_n = np.empty((S, 7)), [], 0.0, 0
        for s in range(S):
            lp[s], r = loam.ScanMatch(surfs[s], edges[s], init[s])
            lr.append(r)
            ms, n = loam.last_timing()
            k_ms, k_n = k_ms + ms, k_n + n
        t1 = time.perf_counter()
        bp, br = loam.ScanMatchBatch(surf, so, edge, eo, init)
        t2 = time.perf_counter()
        assert np.array_equal(bp, lp) and br == lr, "batch and single calls differ"
        if rep < args.warmup:
            continue
        single["wall_ms"].append((t1 - t0) * 1e3)
        single["kernel_ms"].append(k_ms)
        single["launches"].append(k_n)
        ms, n = loam.last_timing()
        batch["wall_ms"].append((t2 - t1) * 1e3)
        batch["kernel_ms"].append(ms)
        batch["launches"].append(n)
    points = S * (N_SURF + N_EDGE)
    iters_done = [r[0]["iters"] for r in br]

    def rates(d):
        wall = np.median(d["wall_ms"]) * 1e-3
        return {"scans_per_s": S / wall, "points_per_s": points / wall}

    out = {
        "gpu": gpu,
        "setup": {"map_points": int(m.shape[0]), "scans": S, "surf_points_per_scan": N_SURF, "edge_points_per_scan": N_EDGE,
                  "points": points, "iterations": iters, "eps": eps, "warmup": args.warmup, "reps": args.reps,
                  "order": "loop of single calls then batch, alternating", "poses_bit_identical": True},
        "single_calls": {**{k: stats(v) for k, v in single.items()}, **rates(single)},
        "align_loam_batch": {**{k: stats(v) for k, v in batch.items()}, **rates(batch)},
        "speedup_wall_median": float(np.median(single["wall_ms"]) / np.median(batch["wall_ms"])),
        "iters": {"min": int(min(iters_done)), "max": int(max(iters_done))},
        "inliers_median": {"surf": float(np.median([r[0]["n_inlier"] for r in br])),
                           "edge": float(np.median([r[1]["n_inlier"] for r in br]))},
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"gpu": gpu, "single_wall_ms": out["single_calls"]["wall_ms"]["median"],
                      "batch_wall_ms": out["align_loam_batch"]["wall_ms"]["median"], "speedup": out["speedup_wall_median"],
                      "batch_points_per_s": out["align_loam_batch"]["points_per_s"]}))


if __name__ == "__main__":
    main()
