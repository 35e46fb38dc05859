"""Staged LOAM relocalisation: locreg_relocalise_loam_staged (LoamRegistration.RelocaliseStaged, rounds with the
worst-scoring hypotheses cut between them) against exhaustive locreg_relocalise_loam (LoamRegistration.Relocalise) on
tools/loam_reloc.py's workload: World(200), the 1 M-point map, gt = World.poses(3)[2] and its 32-beam scan cut by a
seeded permutation into 8192 surf + 2048 edge points, hypotheses from bench.reloc_hypotheses (64 x 64 xy grid of
0.5 m x 16 yaws, default 65 536), eps 0, 10 trips in total.  Arms, alternating in one process after a warm-up, all on
one LOAM pair:
  exhaustive  Relocalise with max_iteration 10;
  staged      RelocaliseStaged for each schedule trips / keep (tools/reloc_staged.py's four).
Per arm: wall time (host clock around the call, which ends in a device synchronise), kernel time and launches
(locreg_last_timing of the surf handle), scan evaluations counted from shapes (sum over rounds of alive * (trips + 1)),
the winner (index, score, error to the truth) and whether it is the exhaustive winner.  Writes one JSON file (--out)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tools")]
import loc_lib_b200 as L  # noqa: E402
from loc_lib_b200 import synth  # noqa: E402
from bench import reloc_hypotheses  # noqa: E402
from reloc_staged import SCHEDULES, evaluations, stats, winner  # noqa: E402

N_SURF, N_EDGE = 8192, 2048


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--hyp", type=int, default=65536)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default="r8_loam_reloc_staged.json")
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    w = synth.World(200.0)
    m = w.sample_map(1_000_000)
    gt = w.poses(3)[2]
    scan = w.scan(gt)
    assert len(scan) >= N_SURF + N_EDGE, len(scan)
    idx = np.random.default_rng(7).permutation(len(scan))  # tools/loam_reloc.py's cut
    surf = np.ascontiguousarray(scan[idx[:N_SURF]])
    edge = np.ascontiguousarray(scan[idx[N_SURF:N_SURF + N_EDGE]])
    hyp = reloc_hypotheses(gt, args.hyp)
    iters, eps = 10, 0.0
    loam = L.LoamRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE, max_iteration_=iters, eps_=eps),
                              L.IcpOptions(method_=L.IcpMethod.P2LINE, max_iteration_=iters, eps_=eps), iters, eps)
    loam.SetInputTarget(m, m)
    names = ["exhaustive"] + ["staged %s / %s" % (t, k) for t, k in SCHEDULES]
    arms = {n: {"wall_ms": [], "kernel_ms": [], "launches": []} for n in names}
    last = {}
    for rep in range(args.warmup + args.reps):
        for name, sched in zip(names, [None] + SCHEDULES):
            t0 = time.perf_counter()
            if sched is None:
                res = loam.Relocalise(surf, edge, hyp)
            else:
                res = loam.RelocaliseStaged(surf, edge, hyp, sched[0], sched[1])
            wall = time.perf_counter() - t0
            ms, n = loam.last_timing()
            if last.get(name) is not None and (last[name][1], last[name][2]) != (res[1], res[2]):
                raise SystemExit("%s: the winner changed between repetitions: %s vs %s" % (name, last[name][1:3], res[1:3]))
            last[name] = res
            if rep >= args.warmup:
                arms[name]["wall_ms"].append(wall * 1e3)
                arms[name]["kernel_ms"].append(ms)
                arms[name]["launches"].append(n)

    n_h = len(hyp)
    ex = last["exhaustive"]
    ex_wall = float(np.median(arms["exhaustive"]["wall_ms"]))
    results = {}
    for name, sched in zip(names, [None] + SCHEDULES):
        trips, keep = ((iters,), ()) if sched is None else sched
        res = last[name]
        wall = float(np.median(arms[name]["wall_ms"]))
        results[name] = {"trips": list(trips), "keep": list(keep),
                         **{k: stats(v) for k, v in arms[name].items()},
                         "scan_evaluations": evaluations(n_h, trips, keep),
                         "hypotheses_per_s_wall": n_h / (wall * 1e-3),
                         "speedup_vs_exhaustive_wall_median": ex_wall / wall,
                         "best": winner(res[0], res[1], res[2], gt),
                         "same_winner_as_exhaustive": bool(res[1] == ex[1])}
    out = {
        "gpu": gpu,
        "setup": {"map_points": int(m.shape[0]), "scan_points": int(len(scan)), "surf_points": N_SURF, "edge_points": N_EDGE,
                  "hypotheses": n_h, "hypothesis_grid": "bench.reloc_hypotheses: 64 x 64 xy grid of 0.5 m x 16 yaws",
                  "eps": eps, "warmup": args.warmup, "reps": args.reps,
                  "order": "exhaustive, then each staged schedule, alternating; one LOAM pair for all arms",
                  "timing": "wall: host clock around the call (it ends in a device synchronise); kernel: the surf "
                            "handle's CUDA events (locreg_last_timing)",
                  "scan_evaluations": "counted from shapes: sum over rounds of alive hypotheses x (trips + 1), each "
                                      "evaluation both halves"},
        "arms": results,
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"gpu": gpu, **{k: {"wall_ms": v["wall_ms"]["median"], "kernel_ms": v["kernel_ms"]["median"],
                                         "launches": v["launches"]["median"], "evals": v["scan_evaluations"],
                                         "best": v["best"]["index"], "same": v["same_winner_as_exhaustive"]}
                                     for k, v in results.items()}}))


if __name__ == "__main__":
    main()
