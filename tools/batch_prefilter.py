"""Batch pre-filters and batch ScanMatch from raw scans, measured (profiles/r11_batch_prefilter.jsonl via
tools/batch_prefilter.sh).  One JSON line per run on stdout (and appended to --out).

--mode batch: config 4's synthetic scans (World(200), bench.py's seeded walk) at S = 512 and 4096 as PointXYZI
    (32 B: x y z 1 intensity 0 0 0) with ~10 % NaN rows at seeded positions (an organised driver cloud), 1 M-point map,
    leaf 1.0 m, P2Plane ICP with bench.py's options (10 trips, eps 0).
      filter:  a loop of S RemoveNanPoint + VoxelFilter calls (locreg_filter_remove_nan / _voxel_grid) against
               RemoveNanPointBatch + VoxelFilterBatch: wall time, kernel launches; the outputs must be equal.
      chain:   the single filters + ScanMatchBatch (locreg_align_batch) against ScanMatchBatchFiltered
               (locreg_align_batch_filtered): wall time; the poses and results must be bit-identical.
--mode single: the single-cloud filter of the package under --root (default: this tree; tools/batch_prefilter.sh
    alternates a built checkout of the parent commit with this tree): locreg_filter_voxel_grid of one C2 scan (leaf
    1.0) and of a 1 M-point local map (leaf 0.5), and bench.py's LIO key-frame step (incremental NDT, locreg_local_map_add_keyframe, leaf 0.5); a hash of
    the outputs goes with the times.
Stream synchronisations are counted from the code (filters.cu), not measured: a single call synchronises once
(NaN removal) or twice (voxel grid), the batch calls once and twice per batch."""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
L = synth = None  # loc_lib_b200 of --root, imported in main()

LEAF_SCAN, LEAF_MAP = 1.0, 0.5


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in q.split(",")]
    return {"gpu": name, "power_limit": power}


def stats(v):
    v = np.asarray(v, float)
    return {"median": float(np.median(v)), "min": float(v.min()), "max": float(v.max()), "n": int(len(v))}


def raw_scans(world, S):
    """bench.py's make_scans(world, 0, S, 4096) as PointXYZI with ~10 % NaN rows."""
    gt = world.poses(4096)[:S]
    buf, counts = world.scan_batch(gt, seed=synth.SEED_SCAN)
    init = np.stack([synth.perturb_pose(g, synth.SEED_POSE + 7919 * i) for i, g in enumerate(gt)])
    offsets = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    cloud = np.zeros((int(offsets[-1]), 8), np.float32)
    for i in range(S):
        c = cloud[offsets[i]:offsets[i + 1]]
        c[:, :3] = buf[i, :counts[i], :3]
        c[:, 3] = 1.0
        c[:, 4] = buf[i, :counts[i], 3]
    del buf
    rng = np.random.default_rng(11)
    cloud[rng.random(len(cloud)) < 0.1, :3] = np.nan
    return cloud, offsets, init


def timed(f):
    t0 = time.perf_counter()
    r = f()
    return (time.perf_counter() - t0) * 1e3, r


def run_batch(args, world, m):
    reg = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE, max_iteration_=10, eps_=0.0))
    reg.SetInputTarget(m)
    for S in args.scans:
        cloud, offs, init = raw_scans(world, S)
        scans = [cloud[offs[s]:offs[s + 1]] for s in range(S)]

        def single_filters():
            out, launches = [], 0
            for sc in scans:
                a = reg.RemoveNanPoint(sc)
                launches += reg.last_timing()[1]
                out.append(reg.VoxelFilter(a, LEAF_SCAN))
                launches += reg.last_timing()[1]
            return out, launches

        def batch_filters():
            a, ao = reg.RemoveNanPointBatch(cloud, offs)
            launches = reg.last_timing()[1]
            b, bo = reg.VoxelFilterBatch(a, ao, LEAF_SCAN)
            return (b, bo), launches + reg.last_timing()[1]

        t_single, t_batch, t_chain_single, t_chain_batch = [], [], [], []
        for rep in range(args.warmup + args.reps):
            ts, (filtered, l_single) = timed(single_filters)
            tb, ((bout, boffs), l_batch) = timed(batch_filters)
            if rep == 0:
                fo = np.concatenate([[0], np.cumsum([len(f) for f in filtered])]).astype(np.int64)
                assert np.array_equal(boffs, fo), "batch filter offsets differ from the single calls"
                assert np.array_equal(bout.view(np.uint32), np.concatenate(filtered).view(np.uint32)), "batch filter output differs"
            fc = np.ascontiguousarray(np.concatenate(filtered))

            def chain_single():
                f = [reg.VoxelFilter(reg.RemoveNanPoint(sc), LEAF_SCAN) for sc in scans]
                c = np.ascontiguousarray(np.concatenate(f))
                o = np.concatenate([[0], np.cumsum([len(x) for x in f])]).astype(np.int64)
                return reg.ScanMatchBatch(c, o, init)

            tcs, (p_ref, r_ref) = timed(chain_single)
            tcb, (p_got, r_got, n_f) = timed(lambda: reg.ScanMatchBatchFiltered(cloud, offs, init, LEAF_SCAN))
            chain_ms, chain_launches = reg.last_timing()
            assert np.array_equal(p_got, p_ref) and r_got == r_ref, "filtered batch poses differ"
            assert np.array_equal(n_f, np.diff(fo))
            if rep >= args.warmup:
                t_single.append(ts); t_batch.append(tb); t_chain_single.append(tcs); t_chain_batch.append(tcb)
        line = dict(gpu_info(), mode="batch", scans=S, raw_points=int(offs[-1]), filtered_points=int(fo[-1]), leaf=LEAF_SCAN,
                    filter_single_loop_ms=stats(t_single), filter_batch_ms=stats(t_batch),
                    filter_speedup=float(np.median(t_single) / np.median(t_batch)),
                    filter_single_launches=int(l_single), filter_batch_launches=int(l_batch),
                    filter_single_syncs=3 * S, filter_batch_syncs=3,
                    chain_single_filters_plus_align_batch_ms=stats(t_chain_single), chain_align_batch_filtered_ms=stats(t_chain_batch),
                    chain_speedup=float(np.median(t_chain_single) / np.median(t_chain_batch)),
                    chain_kernel_ms=float(chain_ms), chain_launches=int(chain_launches),
                    outputs_equal=True, poses_bit_identical=True)
        emit(args, line)
        del cloud, scans, filtered, fc


def run_single(args, world, m):
    h = hashlib.sha1()
    reg = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE, max_iteration_=10, eps_=0.0))
    scan = world.scan(world.poses(1)[0])
    lmap = np.ascontiguousarray(m)
    out = {}
    for name, cloud, leaf, reps in (("c2_scan", scan, LEAF_SCAN, 400), ("local_map_1M", lmap, LEAF_MAP, 40)):
        t = []
        for rep in range(reps + 10):
            dt, f = timed(lambda: reg.VoxelFilter(cloud, leaf))
            if rep >= 10:
                t.append(dt)
        h.update(f.tobytes())
        out[name] = dict(points=int(len(cloud)), out_points=int(len(f)), leaf=leaf, wall_ms=stats(t),
                         kernel_ms=float(reg.last_timing()[0]), launches=int(reg.last_timing()[1]))
    # bench.py's LIO key-frame step
    gt = world.poses(40)
    scans = [world.scan(g) for g in gt]
    wall = []
    reg = L.NdtRegistration(L.NdtOptions(method_=L.NdtMethod.INCREMENTAL_NDT, capacity_=100000))
    for sc, g in zip(scans, gt):
        dt, _ = timed(lambda: reg.AddKeyFrame(sc, g, max_keyframes=10, leaf=LEAF_MAP))
        wall.append(dt)
    h.update(reg.GetLocalMap().tobytes())
    out["lio_keyframe"] = dict(keyframe_wall_ms=stats(wall[8:]), local_map_points=int(len(reg.GetLocalMap())))
    emit(args, dict(gpu_info(), mode="single", build=args.tag, outputs_sha1=h.hexdigest(), **out))


def emit(args, line):
    s = json.dumps(line)
    print(s, flush=True)
    if args.out:
        with open(args.out, "a") as f:
            f.write(s + "\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", choices=("batch", "single"), default="batch")
    ap.add_argument("--scans", type=int, nargs="+", default=[512, 4096])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--tag", default="this")
    ap.add_argument("--out", default="")
    ap.add_argument("--root", default=ROOT, help="repository whose loc_lib_b200 is measured (--mode single)")
    args = ap.parse_args()
    global L, synth
    sys.path.insert(0, os.path.abspath(args.root))
    import loc_lib_b200
    from loc_lib_b200 import synth
    L = loc_lib_b200
    world = synth.World(200.0)
    m = world.sample_map(1_000_000)
    (run_batch if args.mode == "batch" else run_single)(args, world, m)


if __name__ == "__main__":
    main()
