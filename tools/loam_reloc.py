"""LOAM global relocalisation: locreg_relocalise_loam (LoamRegistration.Relocalise, every hypothesis's LOAM loop and score
pass in one device-resident call) against what a LOAM user has without it.  C5-style workload: World(200), the 1 M-point
map, gt = World.poses(3)[2] and its 32-beam scan, as bench.py's C5; the scan is cut by a seeded permutation into 8192 surf
and 2048 edge points, as in tools/loam_batch.py; hypotheses from bench.reloc_hypotheses (64 x 64 xy grid of 0.5 m x 16
yaws, default 65 536).  10 trips, eps 0.  Arms, alternating in one process after a warm-up:
  loam   locreg_relocalise_loam on all hypotheses;
  icp    locreg_relocalise with a P2Plane handle on the whole scan (a second handle a LOAM user would keep for this).
Then a seeded sample of hypotheses through single locreg_align_loam calls plus two locreg_compute_hb calls at the
returned pose (the host loop a LOAM user has otherwise), which must agree with the batched call.  Writes one JSON file
(--out); an agreement failure is recorded there before the tool exits non-zero."""
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
from bench import BYTES_PER_POINT_ITER, reloc_hypotheses  # noqa: E402

N_SURF, N_EDGE = 8192, 2048


def stats(v):
    v = np.asarray(v, float)
    return {"median": float(np.median(v)), "p10": float(np.percentile(v, 10)), "p90": float(np.percentile(v, 90)),
            "min": float(v.min()), "max": float(v.max())}


def rot_err(a, b):
    d = abs(float(np.dot(a[:4], b[:4]))) / (np.linalg.norm(a[:4]) * np.linalg.norm(b[:4]))
    return 2.0 * float(np.arccos(min(1.0, d)))


def winner(pose, idx, score, gt):
    return {"index": int(idx), "score": float(score), "translation_error_m": float(np.linalg.norm(pose[4:] - gt[4:])),
            "rotation_error_rad": rot_err(pose, gt)}


def host_score(loam, surf, edge, pose):
    """(sum_sq_surf + sum_sq_edge) / (n_inlier_surf + n_inlier_edge) from two CaculateMatrixHAndB calls at pose."""
    _, Hs, _ = loam.surf.CaculateMatrixHAndB(surf, pose)
    rs = loam.surf.last_result
    _, He, _ = loam.edge.CaculateMatrixHAndB(edge, pose)
    re = loam.edge.last_result
    n = rs["n_inlier"] + re["n_inlier"]
    return np.inf if np.linalg.det(Hs + He) == 0 or n == 0 else (rs["sum_sq_res"] + re["sum_sq_res"]) / float(n)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--hyp", type=int, default=65536)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--sample", type=int, default=256)
    ap.add_argument("--out", default="r5_loam_reloc.json")
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    w = synth.World(200.0)
    m = w.sample_map(1_000_000)
    gt = w.poses(3)[2]
    scan = w.scan(gt)
    assert len(scan) >= N_SURF + N_EDGE, len(scan)
    idx = np.random.default_rng(7).permutation(len(scan))
    surf = np.ascontiguousarray(scan[idx[:N_SURF]])
    edge = np.ascontiguousarray(scan[idx[N_SURF:N_SURF + N_EDGE]])
    hyp = reloc_hypotheses(gt, args.hyp)
    iters, eps = 10, 0.0
    loam = L.LoamRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE, max_iteration_=iters, eps_=eps),
                              L.IcpOptions(method_=L.IcpMethod.P2LINE, max_iteration_=iters, eps_=eps), iters, eps)
    loam.SetInputTarget(m, m)
    icp = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE, max_iteration_=iters, eps_=eps))
    icp.SetInputTarget(m)
    arms = {"loam": {"wall_ms": [], "kernel_ms": [], "launches": []}, "icp": {"wall_ms": [], "kernel_ms": [], "launches": []}}
    for rep in range(args.warmup + args.reps):
        t0 = time.perf_counter()
        lres = loam.Relocalise(surf, edge, hyp, want_all=True)
        t1 = time.perf_counter()
        lt = loam.last_timing()
        ires = icp.Relocalise(scan, hyp)
        t2 = time.perf_counter()
        it = icp.last_timing()
        if rep < args.warmup:
            continue
        for name, wall, (ms, n) in (("loam", t1 - t0, lt), ("icp", t2 - t1, it)):
            arms[name]["wall_ms"].append(wall * 1e3)
            arms[name]["kernel_ms"].append(ms)
            arms[name]["launches"].append(n)
    best_pose, best_idx, best_score, scores, poses = lres

    # the host loop a LOAM user has otherwise: one locreg_align_loam + two locreg_compute_hb per hypothesis
    sample = np.sort(np.random.default_rng(11).choice(len(hyp), size=min(args.sample, len(hyp)), replace=False))
    walls, bad = [], []
    max_dr = {"near": 0.0, "far": 0.0}
    max_dt = {"near": 0.0, "far": 0.0}
    max_rel_score = 0.0
    for i in sample:
        t0 = time.perf_counter()
        pose, _ = loam.ScanMatch(surf, edge, hyp[i])
        sc = host_score(loam, surf, edge, pose)
        walls.append((time.perf_counter() - t0) * 1e3)
        dr, dt = rot_err(poses[i], pose), float(np.linalg.norm(poses[i][4:] - pose[4:]))
        near = np.linalg.norm(pose[4:] - gt[4:]) < 0.05 and rot_err(pose, gt) < 5e-3  # converged near the truth
        kind = "near" if near else "far"
        max_dr[kind], max_dt[kind] = max(max_dr[kind], dr), max(max_dt[kind], dt)
        rtol, atol = (1e-5, 1e-4) if near else (1e-4, 1e-3)
        ok = dr < rtol and dt < atol
        if near and np.isfinite(sc):
            rel = abs(scores[i] - sc) / sc
            max_rel_score = max(max_rel_score, rel)
            ok = ok and rel <= 1e-5
        elif near:
            ok = ok and scores[i] == sc
        if not ok:
            bad.append({"index": int(i), "kind": kind, "rad": dr, "m": dt, "score": float(scores[i]), "host_score": float(sc)})

    n_h = len(hyp)
    lw = np.median(arms["loam"]["wall_ms"]) * 1e-3
    lk = np.median(arms["loam"]["kernel_ms"]) * 1e-3
    iw = np.median(arms["icp"]["wall_ms"]) * 1e-3
    algo = BYTES_PER_POINT_ITER * (N_SURF + N_EDGE) * (iters + 1) * n_h
    near_sample = int(sum(1 for i in sample if np.linalg.norm(poses[i][4:] - gt[4:]) < 0.05))
    out = {
        "gpu": gpu,
        "setup": {"map_points": int(m.shape[0]), "scan_points": int(len(scan)), "surf_points": N_SURF, "edge_points": N_EDGE,
                  "hypotheses": n_h, "hypothesis_grid": "bench.reloc_hypotheses: 64 x 64 xy grid of 0.5 m x 16 yaws",
                  "iterations": iters, "eps": eps, "warmup": args.warmup, "reps": args.reps,
                  "order": "loam arm then icp arm, alternating", "timing": "wall: host clock around the call (it ends in a "
                  "device synchronise); kernel: the surf handle's CUDA events (locreg_last_timing)"},
        "relocalise_loam": {**{k: stats(v) for k, v in arms["loam"].items()},
                            "hypotheses_per_s_wall": n_h / lw, "hypotheses_per_s_kernel": n_h / lk,
                            "algorithmic_bytes_per_s_kernel": algo / lk,
                            "algorithmic_bytes_note": "96 B x (surf + edge points) x 11 evaluations x hypotheses",
                            "best": winner(best_pose, best_idx, best_score, gt),
                            "finite_scores": int(np.isfinite(scores).sum())},
        "relocalise_icp_p2plane_whole_scan": {**{k: stats(v) for k, v in arms["icp"].items()},
                                              "hypotheses_per_s_wall": n_h / iw,
                                              "best": winner(ires[0], ires[1], ires[2], gt)},
        "loam_vs_icp_wall_median": float(iw / lw),
        "single_calls_sample": {"hypotheses": int(len(sample)), "seed": 11, "near_truth_in_sample": near_sample,
                                "wall_ms_per_hypothesis": stats(walls),
                                "projected_s_for_all_hypotheses": float(np.median(walls) * 1e-3 * n_h),
                                "agreement": {"max_rad": max_dr, "max_m": max_dt, "max_rel_score_near": max_rel_score,
                                              "tolerances": "near the truth: 1e-5 rad / 1e-4 m / 1e-5 relative score; "
                                                            "far: 1e-4 rad / 1e-3 m", "failures": bad}},
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"gpu": gpu, "loam_wall_ms": out["relocalise_loam"]["wall_ms"]["median"],
                      "loam_kernel_ms": out["relocalise_loam"]["kernel_ms"]["median"],
                      "icp_wall_ms": out["relocalise_icp_p2plane_whole_scan"]["wall_ms"]["median"],
                      "loam_best": out["relocalise_loam"]["best"], "icp_best": out["relocalise_icp_p2plane_whole_scan"]["best"],
                      "single_ms_per_hyp": out["single_calls_sample"]["wall_ms_per_hypothesis"]["median"],
                      "agreement_failures": len(bad)}))
    assert not bad, "batched and single-call results disagree: %s" % bad[:5]


if __name__ == "__main__":
    main()
