"""LOAM loop latency: the host loop LoamRegistration runs over two CudaIcpRegistration handles today (two
locreg_compute_hb round trips per Gauss-Newton trip, the 6x6 solve on the host) against locreg_align_loam (the whole loop
queued on the device).  C2 map (1 M points) and one C2 scan; surf = 8192 of its points, edge = 2048 others (sizes from
SURVEY row 11's bound of at most 3840 edge points for 32 beams; no LOAM feature counts have been measured), 10 trips,
eps 0.  The two paths alternate in one process after a warm-up.  Writes one JSON file (--out)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import loc_lib_b200 as L  # noqa: E402
from loc_lib_b200 import synth  # noqa: E402
from loam_cases import host_loop, rot_diff  # noqa: E402


def stats(v):
    v = np.asarray(v, float)
    return {"median": float(np.median(v)), "p10": float(np.percentile(v, 10)), "p90": float(np.percentile(v, 90)),
            "min": float(v.min()), "max": float(v.max())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default="r3_loam_latency.json")
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    w = synth.World(200.0)
    m = w.sample_map(1_000_000)
    gt = w.poses(1)[0]
    scan = w.scan(gt, seed=synth.SEED_SCAN)
    init = synth.perturb_pose(gt, synth.SEED_POSE)
    idx = np.random.default_rng(7).permutation(scan.shape[0])
    surf, edge = np.ascontiguousarray(scan[idx[:8192]]), np.ascontiguousarray(scan[idx[8192:8192 + 2048]])
    iters, eps = 10, 0.0
    loam = L.LoamRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE, max_iteration_=iters, eps_=eps),
                              L.IcpOptions(method_=L.IcpMethod.P2LINE, max_iteration_=iters, eps_=eps), iters, eps)
    loam.SetInputTarget(m, m)
    host = {"wall_ms": [], "kernel_ms": [], "launches": []}
    dev = {"wall_ms": [], "kernel_ms": [], "launches": []}
    for rep in range(args.warmup + args.reps):
        tl = []
        t0 = time.perf_counter()
        hpose, hres = host_loop(loam.surf, loam.edge, surf, edge, init, iters, eps, tl)
        t1 = time.perf_counter()
        dpose, dres = loam.ScanMatch(surf, edge, init)
        t2 = time.perf_counter()
        if rep < args.warmup:
            continue
        host["wall_ms"].append((t1 - t0) * 1e3)
        host["kernel_ms"].append(sum(t[0] for t in tl))
        host["launches"].append(sum(t[1] for t in tl))
        ms, n = loam.last_timing()
        dev["wall_ms"].append((t2 - t1) * 1e3)
        dev["kernel_ms"].append(ms)
        dev["launches"].append(n)
    dr, dt = rot_diff(hpose, dpose), float(np.linalg.norm(hpose[4:] - dpose[4:]))
    assert (hres["iters"], hres["updates"]) == (dres[0]["iters"], dres[0]["updates"]) and dr < 1e-9 and dt < 1e-8, (dr, dt)
    out = {
        "gpu": gpu,
        "setup": {"map_points": int(m.shape[0]), "scan_points": int(scan.shape[0]), "surf_points": int(surf.shape[0]),
                  "edge_points": int(edge.shape[0]), "iterations": iters, "eps": eps, "warmup": args.warmup,
                  "reps": args.reps, "order": "host loop then device loop, alternating"},
        "host_loop": {k: stats(v) for k, v in host.items()},
        "align_loam": {k: stats(v) for k, v in dev.items()},
        "speedup_wall_median": float(np.median(host["wall_ms"]) / np.median(dev["wall_ms"])),
        "pose_difference": {"rad": dr, "m": dt},
        "inliers": {"surf": int(dres[0]["n_inlier"]), "edge": int(dres[1]["n_inlier"])},
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"gpu": gpu, "host_wall_ms": out["host_loop"]["wall_ms"]["median"],
                      "loam_wall_ms": out["align_loam"]["wall_ms"]["median"], "speedup": out["speedup_wall_median"],
                      "host_launches": out["host_loop"]["launches"]["median"],
                      "loam_launches": out["align_loam"]["launches"]["median"]}))


if __name__ == "__main__":
    main()
