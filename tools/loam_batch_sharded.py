"""LOAM batch offline mapping across ranks (BASELINE config 4 in LOAM form): locreg_align_loam_batch_sharded
(LoamRegistration.ScanMatchBatchSharded), strong scaling on a fixed batch.  Workload: 4096 scans of World(200) at
World.poses(4096), each cut by tools/loam_batch.py's seeded permutation into 8192 surf + 2048 edge points, registered
from perturb_poses against the 1 M-point map, 10 trips, eps 0, pageable host inputs.

    python tools/loam_batch_sharded.py --out f.jsonl                                   # one GPU
    python -m torch.distributed.run --standalone --nproc-per-node N tools/loam_batch_sharded.py --out f.jsonl

Every rank builds the whole batch (seeded) and passes its block (dist.shard_range); one LOAM pair per rank, its surf
handle holding an NCCL communicator over all ranks.  Arms, alternating after a warm-up: "sharded"
(ScanMatchBatchSharded) and, at N = 1 only, "align_loam_batch" (ScanMatchBatch of the whole batch on the same pair).
Per arm: wall time between barriers (host clock; the call ends in a stream synchronise), kernel ms
(locreg_last_timing(surf): kernels + exchange; max over ranks), launches (rank 0).  Outside the timed region rank 0
checks that every rank returned the same poses and results (digests) and that they are bit for bit one unsharded
ScanMatchBatch of the whole batch on rank 0; a mismatch ends the run with an error.  Rank 0 appends one JSON line to
--out, with the GPU name and power limit read in the same run.

--share-gpu0 runs every rank on GPU 0, each naming a host of its own to NCCL (NCCL_HOSTID) and talking over loopback
sockets (NCCL refuses two ranks of one host on one device).  That checks the cross-rank results of the real workload on
a box with fewer GPUs than ranks; its times measure ranks queueing on one GPU, not scaling, and its lines say so."""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import loc_lib_b200 as L  # noqa: E402
from loc_lib_b200 import dist as D, synth  # noqa: E402

N_SURF, N_EDGE = 8192, 2048
RESULT_KEYS = ("iters", "updates", "converged", "degenerate", "n_effective", "n_inlier", "sum_sq_res", "pose_written")


def stats(v):
    v = np.asarray(v, float)
    return {"median": float(np.median(v)), "p10": float(np.percentile(v, 10)), "p90": float(np.percentile(v, 90)),
            "min": float(v.min()), "max": float(v.max())}


def workload(S, chunk=256):
    """(map, surf (S * N_SURF, 4), edge (S * N_EDGE, 4), init (S, 7)): tools/loam_batch.py's batch, its scans generated
    `chunk` at a time (scan s is seeded SEED_SCAN + s either way) and cut by the same sequence of permutations."""
    w = synth.World(200.0)
    m = w.sample_map(1_000_000)
    gt = w.poses(S)
    init = synth.perturb_poses(gt, synth.SEED_POSE)
    surf = np.empty((S * N_SURF, 4), np.float32)
    edge = np.empty((S * N_EDGE, 4), np.float32)
    rng = np.random.default_rng(7)
    for c0 in range(0, S, chunk):
        buf, counts = w.scan_batch(gt[c0:c0 + chunk], seed=synth.SEED_SCAN + c0)
        assert counts.min() >= N_SURF + N_EDGE, counts.min()
        for i in range(len(counts)):
            s = c0 + i
            idx = rng.permutation(int(counts[i]))
            surf[s * N_SURF:(s + 1) * N_SURF] = buf[i, idx[:N_SURF]]
            edge[s * N_EDGE:(s + 1) * N_EDGE] = buf[i, idx[N_SURF:N_SURF + N_EDGE]]
    return m, surf, edge, init


def digest(poses, res):
    r = np.array([[pair[h][k] for h in (0, 1) for k in RESULT_KEYS] for pair in res], np.float64)
    return hashlib.sha256(np.ascontiguousarray(poses, np.float64).tobytes() + r.tobytes()).hexdigest()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scans", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default="r9_loam_batch_sharded.jsonl")
    ap.add_argument("--share-gpu0", action="store_true", help="every rank on GPU 0: checks results, does not measure scaling")
    args = ap.parse_args()
    if args.share_gpu0:  # before torch or liblocreg make their first NCCL call
        os.environ.update({"NCCL_HOSTID": "loam-batch-rank-%s" % os.environ.get("RANK", "0"), "NCCL_SOCKET_IFNAME": "lo",
                           "NCCL_NET": "Socket", "NCCL_IB_DISABLE": "1", "NCCL_MNNVL_ENABLE": "0"})

    import torch
    import torch.distributed as dist
    local, world_size = int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    if args.share_gpu0:
        local = 0
    if world_size > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    rank = dist.get_rank() if world_size > 1 else 0

    def barrier():
        if world_size > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def gather(obj):
        if world_size == 1:
            return [obj]
        out = [None] * world_size
        dist.all_gather_object(out, obj)
        return out

    S = args.scans
    m, surf, edge, init = workload(S)
    so_all = np.arange(S + 1, dtype=np.int64) * N_SURF
    eo_all = np.arange(S + 1, dtype=np.int64) * N_EDGE
    lo, hi = D.shard_range(S, rank, world_size)
    mine = (surf[lo * N_SURF:hi * N_SURF], so_all[lo:hi + 1] - so_all[lo], edge[lo * N_EDGE:hi * N_EDGE],
            eo_all[lo:hi + 1] - eo_all[lo], init[lo:hi])
    iters, eps = 10, 0.0
    loam = L.LoamRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE, max_iteration_=iters, eps_=eps),
                              L.IcpOptions(method_=L.IcpMethod.P2LINE, max_iteration_=iters, eps_=eps), iters, eps,
                              device=local)
    loam.SetInputTarget(m, m)
    D.comm_init(loam, dev)
    assert loam.CommInfo()[1] == world_size or world_size == 1

    arms = {"sharded": lambda: loam.ScanMatchBatchSharded(*mine, S)}
    if world_size == 1:
        arms["align_loam_batch"] = lambda: loam.ScanMatchBatch(surf, so_all, edge, eo_all, init)
    times = {n: {"wall_ms": [], "kernel_ms": [], "launches": []} for n in arms}
    last = {}
    for rep in range(args.warmup + args.reps):
        for name, run in arms.items():
            barrier()
            t0 = time.perf_counter()
            out = run()
            barrier()
            wall = time.perf_counter() - t0
            ms, n = loam.last_timing()
            ms = max(gather(ms))
            d = digest(*out)
            if name in last and last[name][0] != d:
                raise SystemExit("%s: the results changed between repetitions" % name)
            last[name] = (d, out)
            if rep >= args.warmup:
                times[name]["wall_ms"].append(wall * 1e3)
                times[name]["kernel_ms"].append(ms)
                times[name]["launches"].append(n)

    everyone = gather(last["sharded"][0])
    if rank == 0:
        for q, theirs in enumerate(everyone):
            if theirs != everyone[0]:
                raise SystemExit("rank %d returned other poses / results than rank 0" % q)
        ref = last["align_loam_batch"][1] if world_size == 1 else loam.ScanMatchBatch(surf, so_all, edge, eo_all, init)
        poses, res = last["sharded"][1]
        if not (np.array_equal(poses, ref[0]) and res == ref[1]):
            raise SystemExit("the sharded poses / results differ from the unsharded ScanMatchBatch of the whole batch")
    barrier()

    if rank == 0:
        gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(local)],
                             capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
        points = S * (N_SURF + N_EDGE)
        res = last["sharded"][1][1]
        iters_done = [r[0]["iters"] for r in res]
        results = {}
        for name, t in times.items():
            wall = float(np.median(t["wall_ms"])) * 1e-3
            results[name] = {**{k: stats(v) for k, v in t.items()}, "scans_per_s": S / wall, "points_per_s": points / wall}
        line = {"gpus": 1 if args.share_gpu0 else world_size, "ranks": world_size, "gpu": gpu,
                "ranks_share_gpu0": bool(args.share_gpu0),
                "setup": {"map_points": int(m.shape[0]), "scans": S, "surf_points_per_scan": N_SURF,
                          "edge_points_per_scan": N_EDGE, "points": points, "iterations": iters, "eps": eps,
                          "warmup": args.warmup, "reps": args.reps, "host_inputs": "pageable",
                          "order": "sharded, then (N = 1) align_loam_batch, alternating; one LOAM pair per rank",
                          "timing": "wall: host clock between barriers around the call; kernel: locreg_last_timing(surf) "
                                    "(kernels + exchange), max over ranks; launches: rank 0",
                          "checks": "poses and results identical on every rank, and bit for bit one unsharded "
                                    "ScanMatchBatch of the whole batch on rank 0"},
                "exchange_bytes": S * (7 * 8 + 3 * 48),
                "iters": {"min": int(min(iters_done)), "max": int(max(iters_done))},
                "bit_identical_to_align_loam_batch": True,
                "arms": results}
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            f.write(json.dumps(line) + "\n")
        print(json.dumps({"ranks": world_size, "share_gpu0": bool(args.share_gpu0), "gpu": gpu,
                          **{k: {"wall_ms": v["wall_ms"]["median"], "kernel_ms": v["kernel_ms"]["median"],
                                 "launches": v["launches"]["median"], "points_per_s": v["points_per_s"]}
                             for k, v in results.items()}}))
    if world_size > 1:
        loam.CommDestroy()
        dist.destroy_process_group()
    loam.close()


if __name__ == "__main__":
    main()
