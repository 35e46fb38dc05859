"""Multi-GPU entry points of the C ABI (SURVEY.md 8e): NCCL inside liblocreg.so.

A communicator of ONE rank exercises the whole code path (ncclAllReduce / ncclBroadcast on the handle's stream) on a
single-GPU box; the two-rank tests need two GPUs and are skipped otherwise."""
import multiprocessing as mp
import os
import subprocess

import numpy as np
import pytest

from conftest import GPU_COUNT, ROOT

pytestmark = pytest.mark.gpu


def _hypotheses(scene, n):
    rng = np.random.default_rng(7)
    hyp = np.repeat(scene.init[0][None], n, axis=0)
    hyp[:, 4:6] += rng.uniform(-2.0, 2.0, (n, 2))
    hyp[n // 3] = scene.init[0]
    return hyp


def _batch(scene):
    clouds = np.concatenate(scene.scans)
    offsets = np.concatenate([[0], np.cumsum([len(s) for s in scene.scans])]).astype(np.int64)
    return clouds, offsets, np.asarray(scene.init)


def test_world_of_one_equals_the_unsharded_calls(scene):
    import loc_lib_b200 as L
    reg = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE, max_iteration_=6, eps_=0.0))
    reg.SetInputTarget(scene.map)
    hyp = _hypotheses(scene, 41)
    pose0, idx0, score0, _, _ = reg.Relocalise(scene.scan, hyp)
    reg.CommInit(reg.CommUniqueId(), 0, 1)
    rank, world, version = reg.CommInfo()
    assert (rank, world) == (0, 1) and version >= 20000
    pose1, idx1, score1 = reg.RelocaliseSharded(scene.scan, hyp)
    assert idx1 == idx0 and score1 == score0 and np.array_equal(pose1, pose0)
    clouds, offsets, init = _batch(scene)
    p0, r0 = reg.ScanMatchBatch(clouds, offsets, init)
    p1, r1 = reg.ScanMatchBatchSharded(clouds, offsets, init, len(init))
    assert np.array_equal(p0, p1) and [r["n_inlier"] for r in r0] == [r["n_inlier"] for r in r1]
    reg.CommDestroy()
    assert reg.CommInfo()[:2] == (0, 1)
    with pytest.raises(Exception):
        reg.ScanMatchBatchSharded(clouds, offsets, init, len(init) + 3)  # not this rank's block of a 7-scan batch


def test_ndt_relocalisation_scores_every_hypothesis(scene):
    """locreg_relocalise with direct NDT: one CTA per hypothesis (k_align_batch) + score pass; the winner is the
    hypothesis a single ScanMatch + evaluation also ranks first."""
    import loc_lib_b200 as L
    reg = L.NdtRegistration(L.NdtOptions(max_iteration_=8, eps_=0.0))
    reg.SetInputTarget(scene.map)
    hyp = _hypotheses(scene, 24)
    pose, idx, score, scores, poses = reg.Relocalise(scene.scan, hyp, want_all=True)
    assert np.isfinite(score) and score == scores[idx] and idx == int(np.argmin(scores))
    for i in (0, idx, 23):
        _, _, p = reg.ScanMatch(scene.scan, hyp[i], want_cloud=False)
        assert np.allclose(p, poses[i], rtol=0, atol=1e-9)


def _rank_main(rank, world, uid, q):
    import sys
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import loc_lib_b200 as L
    from conftest import Scene
    from loc_lib_b200 import dist as D
    scene = Scene()
    reg = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE, max_iteration_=6, eps_=0.0), device=rank)
    reg.SetInputTarget(scene.map)
    reg.CommInit(uid, rank, world)
    hyp = _hypotheses(scene, 41)
    pose, idx, score = reg.RelocaliseSharded(scene.scan, hyp)
    clouds, offsets, init = _batch(scene)
    lo, hi = D.shard_range(len(init), rank, world)
    mine = clouds[offsets[lo]:offsets[hi]]
    poses, res = reg.ScanMatchBatchSharded(mine, offsets[lo:hi + 1] - offsets[lo], init[lo:hi], len(init))
    reg.CommDestroy()
    q.put((rank, pose, idx, score, poses, [r["n_inlier"] for r in res]))


@pytest.mark.skipif(GPU_COUNT < 2, reason="needs two GPUs")
def test_two_ranks_agree_with_one(scene):
    import loc_lib_b200 as L
    reg = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE, max_iteration_=6, eps_=0.0))
    reg.SetInputTarget(scene.map)
    hyp = _hypotheses(scene, 41)
    pose0, idx0, score0, _, _ = reg.Relocalise(scene.scan, hyp)
    clouds, offsets, init = _batch(scene)
    p0, r0 = reg.ScanMatchBatch(clouds, offsets, init)
    uid = reg.CommUniqueId()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_rank_main, args=(r, 2, uid, q)) for r in range(2)]
    for p in procs:
        p.start()
    outs = sorted([q.get(timeout=120) for _ in procs], key=lambda o: o[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, pose, idx, score, poses, inl in outs:
        assert idx == idx0 and score == score0 and np.array_equal(pose, pose0), rank
        assert np.array_equal(poses, p0), rank
        assert inl == [r["n_inlier"] for r in r0]


def test_cpp_host_drives_all_visible_gpus():
    """tests/cpp/sharded_host.cpp: one host thread per GPU, no Python / torch in the process."""
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "tests", "cpp")])
    r = subprocess.run([os.path.join(ROOT, "tests", "cpp", "_build", "sharded_host"), str(min(GPU_COUNT, 4))],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
