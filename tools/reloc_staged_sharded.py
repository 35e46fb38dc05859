"""Staged global relocalisation across ranks: locreg_relocalise_staged_sharded (RelocaliseStagedSharded) against
exhaustive locreg_relocalise_sharded (RelocaliseSharded, BASELINE config 5) on C5's workload, built as
tools/reloc_staged.py builds it: World(200), the 1 M-point map, gt = World.poses(3)[2] and its 32-beam scan, 65 536
hypotheses of bench.reloc_hypotheses, P2Plane, eps 0, 10 trips in total.

    python tools/reloc_staged_sharded.py --out f.jsonl                                   # one GPU
    python -m torch.distributed.run --nproc-per-node N tools/reloc_staged_sharded.py --out f.jsonl

Arms, alternating after a warm-up, on one handle per rank with an NCCL communicator over all ranks:
  exhaustive  RelocaliseSharded with max_iteration 10;
  staged      RelocaliseStagedSharded for each schedule trips / keep of tools/reloc_staged.py.
Per arm: wall time between barriers (as bench.py's C5), kernel time and launches (locreg_last_timing; kernel time is the
max over ranks), scan evaluations counted from shapes.  Rank 0 checks that every rank returned the same winner (index,
score bits, pose) and that each staged winner equals one single-GPU RelocaliseStaged call of the same schedule, made on
rank 0 outside the timed region; a mismatch ends the run with an error.  Rank 0 appends one JSON line to --out, with
the GPU name and power limit.

--share-gpu0 runs every rank on GPU 0, each naming a host of its own to NCCL (NCCL_HOSTID) and talking over loopback
sockets (NCCL refuses two ranks of one host on one device).  That checks the cross-rank results of the real workload
on a box with fewer GPUs than ranks; its times measure ranks queueing on one GPU, not scaling, and its lines say so."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import loc_lib_b200 as L  # noqa: E402
from loc_lib_b200 import dist as D, synth  # noqa: E402
from bench import reloc_hypotheses  # noqa: E402
from reloc_staged import SCHEDULES, evaluations, stats, winner  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--hyp", type=int, default=65536)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default="r7_reloc_staged_sharded.jsonl")
    ap.add_argument("--share-gpu0", action="store_true", help="every rank on GPU 0: checks results, does not measure scaling")
    args = ap.parse_args()
    if args.share_gpu0:  # before torch or liblocreg make their first NCCL call
        os.environ.update({"NCCL_HOSTID": "reloc-staged-rank-%s" % os.environ.get("RANK", "0"), "NCCL_SOCKET_IFNAME": "lo",
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

    w = synth.World(200.0)
    m = w.sample_map(1_000_000)
    gt = w.poses(3)[2]
    scan = w.scan(gt)
    hyp = reloc_hypotheses(gt, args.hyp)
    iters = 10
    reg = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE, max_iteration_=iters, eps_=0.0), device=local)
    reg.SetInputTarget(m)
    D.comm_init(reg, dev)
    assert reg.CommInfo()[1] == world_size or world_size == 1

    names = ["exhaustive sharded"] + ["staged sharded %s / %s" % (t, k) for t, k in SCHEDULES]
    scheds = [None] + SCHEDULES
    arms = {n: {"wall_ms": [], "kernel_ms": [], "launches": []} for n in names}
    last = {}
    for rep in range(args.warmup + args.reps):
        for name, sched in zip(names, scheds):
            barrier()
            t0 = time.perf_counter()
            if sched is None:
                res = reg.RelocaliseSharded(scan, hyp)
            else:
                res = reg.RelocaliseStagedSharded(scan, hyp, sched[0], sched[1])[:3]
            barrier()
            wall = time.perf_counter() - t0
            ms, n = reg.last_timing()
            ms = max(gather(ms))
            if name in last and (last[name][1], last[name][2]) != (res[1], res[2]):
                raise SystemExit("%s: the winner changed between repetitions: %s vs %s" % (name, last[name][1:3], res[1:3]))
            last[name] = res
            if rep >= args.warmup:
                arms[name]["wall_ms"].append(wall * 1e3)
                arms[name]["kernel_ms"].append(ms)
                arms[name]["launches"].append(n)

    # every rank's winners, as bits
    mine = {name: (int(r[1]), np.float64(r[2]).tobytes().hex(), np.asarray(r[0], np.float64).tobytes().hex())
            for name, r in last.items()}
    everyone = gather(mine)
    single = {}
    if rank == 0:
        for q, theirs in enumerate(everyone):
            if theirs != mine:
                raise SystemExit("rank %d returned other winners than rank 0: %s vs %s" % (q, theirs, mine))
        for name, sched in zip(names[1:], scheds[1:]):  # one single-GPU staged call per schedule, outside the timed region
            bp, bi, bs = reg.RelocaliseStaged(scan, hyp, sched[0], sched[1])[:3]
            single[name] = bi == mine[name][0] and np.float64(bs).tobytes().hex() == mine[name][1] and \
                np.asarray(bp, np.float64).tobytes().hex() == mine[name][2]
            if not single[name]:
                raise SystemExit("%s: winner %s differs from the single-GPU RelocaliseStaged winner %s" % (
                    name, mine[name][:2], (bi, bs)))
    barrier()

    if rank == 0:
        gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(local)],
                             capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
        n_h = len(hyp)
        ex_wall = float(np.median(arms[names[0]]["wall_ms"]))
        results = {}
        for name, sched in zip(names, scheds):
            trips, keep = ((iters,), ()) if sched is None else sched
            res = last[name]
            wall = float(np.median(arms[name]["wall_ms"]))
            results[name] = {"trips": list(trips), "keep": list(keep),
                             **{k: stats(v) for k, v in arms[name].items()},
                             "scan_evaluations": evaluations(n_h, trips, keep),
                             "hypotheses_per_s_wall": n_h / (wall * 1e-3),
                             "speedup_vs_exhaustive_sharded_wall_median": ex_wall / wall,
                             "best": winner(res[0], res[1], res[2], gt),
                             "same_winner_on_every_rank": True,
                             "same_winner_as_exhaustive_sharded": bool(res[1] == last[names[0]][1])}
            if sched is not None:
                results[name]["same_winner_as_single_gpu_staged"] = bool(single[name])
        line = {"gpus": 1 if args.share_gpu0 else world_size, "ranks": world_size, "gpu": gpu,
                "ranks_share_gpu0": bool(args.share_gpu0),
                "setup": {"map_points": int(m.shape[0]), "scan_points": int(len(scan)), "hypotheses": n_h,
                          "method": "P2Plane", "eps": 0.0, "warmup": args.warmup, "reps": args.reps,
                          "order": "exhaustive sharded, then each staged schedule, alternating; one handle per rank",
                          "timing": "wall: host clock between barriers around the call; kernel: the handle's CUDA events "
                                    "(locreg_last_timing, kernels + collectives), max over ranks; launches: rank 0",
                          "checks": "winner (index, score bits, pose bits) identical on every rank; each staged winner "
                                    "equal to one single-GPU RelocaliseStaged call on rank 0"},
                "arms": results}
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            f.write(json.dumps(line) + "\n")
        print(json.dumps({"ranks": world_size, "share_gpu0": bool(args.share_gpu0), "gpu": gpu,
                          **{k: {"wall_ms": v["wall_ms"]["median"], "kernel_ms": v["kernel_ms"]["median"],
                                 "launches": v["launches"]["median"], "best": v["best"]["index"]}
                             for k, v in results.items()}}))
    if world_size > 1:
        reg.CommDestroy()
        dist.destroy_process_group()
    reg.close()


if __name__ == "__main__":
    main()
