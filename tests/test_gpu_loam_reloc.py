"""GPU tests of locreg_relocalise_loam / LoamRegistration.Relocalise and their sharded forms: every hypothesis's loop and
score against the public single calls (ScanMatch + two CaculateMatrixHAndB), parity with the oracle's LOAM loop, the
argmin, waves, edge cases, argument errors, the handles staying usable, one caller stream, and the sharded entry point."""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_py as O
from conftest import GPU_COUNT, ROOT, pose_delta
from loam_cases import KatScene, oracle_loam_align, pose_from_rpy_t

pytestmark = pytest.mark.gpu

IDENTITY = np.array([0, 0, 0, 1, 0, 0, 0], np.float64)
EMPTY = np.zeros((0, 4), np.float32)


@pytest.fixture(scope="module", autouse=True)
def _torch_first():
    """torch is imported before the first sharded call loads NCCL: liblocreg.so then binds the NCCL torch brought
    (nccl_dyn.h), which a later torch import needs, instead of the system's."""
    import torch  # noqa: F401


def make(max_iteration=10, eps=0.0, device=0):
    import loc_lib_b200 as L
    so = L.IcpOptions(method_=L.IcpMethod.P2PLANE, max_iteration_=max_iteration, eps_=eps)
    eo = L.IcpOptions(method_=L.IcpMethod.P2LINE, max_iteration_=max_iteration, eps_=eps, max_line_distance_=0.5)
    return L.LoamRegistration(so, eo, max_iteration=max_iteration, eps=eps, device=device)


def halves(scene):
    return scene.scan[0::2], scene.scan[1::2]


def hypotheses(scene, n=48):
    from loc_lib_b200 import synth
    hyp = np.stack([synth.perturb_pose(scene.gt[0], 1000 + i, 1.5, 6.0) for i in range(n)])
    hyp[min(17, n - 1)] = scene.init[0]
    return hyp


def half_hb(reg, cloud, pose):
    """(H, sum_sq_res, n_inlier) of one half at pose, as locreg_compute_hb reports it (an empty half: zeros)."""
    if len(cloud) == 0:
        return np.zeros((6, 6)), 0.0, 0
    _, H, _ = reg.CaculateMatrixHAndB(cloud, pose)
    return H, reg.last_result["sum_sq_res"], reg.last_result["n_inlier"]


def host_score(loam, surf, edge, pose):
    """The score of the contract from two CaculateMatrixHAndB calls at pose."""
    Hs, ss, ns = half_hb(loam.surf, surf, pose)
    He, se, ne = half_hb(loam.edge, edge, pose)
    if np.linalg.det(Hs + He) == 0 or ns + ne == 0:
        return np.inf
    return (ss + se) / float(ns + ne)


def assert_equals_single_calls(loam, surf, edge, hyp):
    """Every hypothesis's pose bit for bit what ScanMatch gives from it, its score the host formula at that pose, and
    the winner the argmin of the float32 scores.

    The score is equal up to the last bits, not bit for bit, after a loop (max_iteration > 0): the score pass searches
    from the last trip's neighbours (kNnSeeds, as ICP relocalisation's), and a surf point whose neighbour SET did not
    change keeps the plane the last trip fitted (k_icp_fit's cache).  That fit summed the five points in the order of
    that trip's search; locreg_compute_hb searches afresh and fits in the current distance order, which differs when
    two neighbours swapped ranks.  Without a trip the score pass searches afresh too, and the scores are bit-identical."""
    best_pose, best_idx, best_score, scores, poses = loam.Relocalise(surf, edge, hyp, want_all=True)
    assert scores.shape == (len(hyp),) and poses.shape == (len(hyp), 7)
    rtol = 1e-12 if loam.max_iteration > 0 else 0.0
    for i, h in enumerate(hyp):
        pose, _ = loam.ScanMatch(surf, edge, h)
        assert np.array_equal(poses[i], pose), (i, poses[i], pose)
        sc = host_score(loam, surf, edge, poses[i])
        assert scores[i] == sc or abs(scores[i] - sc) <= rtol * sc, (i, scores[i], sc)
    assert best_idx == int(np.argmin(np.float32(scores)))
    assert best_score == scores[best_idx]
    assert np.array_equal(best_pose, poses[best_idx])
    return best_pose, best_idx, best_score, scores, poses


def test_loop_and_score_equal_the_public_single_calls(scene):
    """max_iteration = 2: both trips come before the tracked search (LOCREG_TRACK_FROM = 3), whose neighbour order is
    canonical, so every pose is bit-identical to the single calls' (the score: see assert_equals_single_calls)."""
    loam = make(max_iteration=2)
    loam.SetInputTarget(scene.map, scene.map)
    surf, edge = halves(scene)
    loam.Relocalise(surf, edge, hypotheses(scene))
    ms, launches = loam.last_timing()
    assert ms > 0 and launches > 10
    _, _, _, scores, _ = assert_equals_single_calls(loam, surf, edge, hypotheses(scene))
    assert np.isfinite(scores).any()


def test_argmin_and_ties(scene):
    loam = make(max_iteration=2)
    loam.SetInputTarget(scene.map, scene.map)
    surf, edge = halves(scene)
    hyp = hypotheses(scene)
    best_pose, best_idx, best_score, scores, poses = loam.Relocalise(surf, edge, hyp, want_all=True)
    assert best_idx == int(np.argmin(np.float32(scores))) and best_score == scores[best_idx]
    assert np.array_equal(best_pose, poses[best_idx])
    # the best hypothesis once more at a higher index: it scores the same and loses the tie
    dup = np.concatenate([hyp, hyp[best_idx][None]])
    p2, i2, s2, sc2, _ = loam.Relocalise(surf, edge, dup, want_all=True)
    assert sc2[-1] == sc2[best_idx] and i2 == best_idx and s2 == best_score and np.array_equal(p2, best_pose)
    # and without the optional outputs the winner is the same
    p3, i3, s3, sc3, ps3 = loam.Relocalise(surf, edge, hyp)
    assert sc3 is None and ps3 is None and (i3, s3) == (best_idx, best_score) and np.array_equal(p3, best_pose)


def oracle_pair(surf_map, edge_map):
    surf = O.OracleIcp(method=O.P2PLANE, nn_mode=O.NN_EXACT_TIEBREAK, skip_nonfinite=1)
    edge = O.OracleIcp(method=O.P2LINE, nn_mode=O.NN_EXACT_TIEBREAK, skip_nonfinite=1, max_line_distance=0.5)
    surf.set_target(surf_map)
    edge.set_target(edge_map)
    return surf, edge


def oracle_score(surf_o, edge_o, surf, edge, pose):
    _, Hs, _, rs, _, _ = surf_o.compute_hb(surf, pose, False, False)
    _, He, _, re, _, _ = edge_o.compute_hb(edge, pose, False, False)
    n = rs["n_inlier"] + re["n_inlier"]
    return np.inf if np.linalg.det(Hs + He) == 0 or n == 0 else (rs["sum_sq_res"] + re["sum_sq_res"]) / n


def assert_oracle_parity(surf_map, edge_map, surf, edge, hyp, near, poses, scores):
    so, eo = oracle_pair(surf_map, edge_map)
    for i, h in enumerate(hyp):
        rpose, _ = oracle_loam_align(so, eo, surf, edge, h, 10, 0.0)
        dr, dt = pose_delta(poses[i], rpose)
        if i in near:  # converges near the truth: the contract's tolerance
            assert dr < 1e-5 and dt < 1e-4, (i, dr, dt)
            sc = oracle_score(so, eo, surf, edge, rpose)
            assert abs(scores[i] - sc) <= 1e-5 * sc, (i, scores[i], sc)
        else:  # far hypotheses are ill-conditioned (test_relocalise's bound)
            assert dr < 1e-4 and dt < 1e-3, (i, dr, dt)


def test_parity_with_the_oracle(scene):
    from loc_lib_b200 import synth
    loam = make()
    loam.SetInputTarget(scene.map, scene.map)
    surf, edge = halves(scene)
    hyp = np.stack([scene.init[0], synth.perturb_pose(scene.gt[0], 5, 0.2, 1.0),
                    synth.perturb_pose(scene.gt[0], 1003, 1.5, 6.0), synth.perturb_pose(scene.gt[0], 1030, 1.5, 6.0)])
    _, _, _, scores, poses = loam.Relocalise(surf, edge, hyp, want_all=True)
    assert_oracle_parity(scene.map, scene.map, surf, edge, hyp, (0, 1), poses, scores)
    # KatScene: its own surf and edge targets, and neither half solves it alone
    k = KatScene()
    kat = make()
    kat.SetInputTarget(k.surf_map, k.edge_map)
    hyp = np.stack([k.init, pose_from_rpy_t([0.005, 0.0, -0.01], [0.02, 0.01, 0.0]),
                    pose_from_rpy_t([0.0, 0.0, 0.1], [0.2, -0.1, 0.05])])
    best_pose, best_idx, _, scores, poses = kat.Relocalise(k.surf, k.edge, hyp, want_all=True)
    assert_oracle_parity(k.surf_map, k.edge_map, k.surf, k.edge, hyp, (0, 1), poses, scores)
    dr, dt = pose_delta(best_pose, k.truth)
    assert dr < 1e-5 and dt < 1e-4, (dr, dt)


_WAVES = r"""
import sys
import numpy as np
sys.path[:0] = [{root!r}, {tests!r}]
from conftest import Scene
from test_gpu_loam_reloc import make, halves, hypotheses
scene = Scene()
loam = make(max_iteration=2)
loam.SetInputTarget(scene.map, scene.map)
surf, edge = halves(scene)
_, idx, score, scores, poses = loam.Relocalise(surf, edge, hypotheses(scene), want_all=True)
np.savez({out!r}, idx=idx, score=score, scores=scores, poses=poses, launches=loam.last_timing()[1])
"""


def test_waves_agree_bit_for_bit(scene, tmp_path):
    """LOCREG_RELOC_WAVE_GIB is read once per process: a subprocess runs the 48 hypotheses in waves of 3."""
    loam = make(max_iteration=2)
    loam.SetInputTarget(scene.map, scene.map)
    surf, edge = halves(scene)
    _, idx, score, scores, poses = loam.Relocalise(surf, edge, hypotheses(scene), want_all=True)
    launches = loam.last_timing()[1]
    out = str(tmp_path / "waves.npz")
    env = dict(os.environ, LOCREG_RELOC_WAVE_GIB="0.0005")
    code = _WAVES.format(root=ROOT, tests=os.path.join(ROOT, "tests"), out=out)
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    w = np.load(out)
    assert int(w["idx"]) == idx and float(w["score"]) == score
    assert np.array_equal(w["scores"], scores) and np.array_equal(w["poses"], poses)
    assert int(w["launches"]) > 4 * launches  # many waves really ran


def test_edge_cases(scene):
    loam = make(max_iteration=2)
    loam.SetInputTarget(scene.map, scene.map)
    surf, edge = halves(scene)
    hyp = hypotheses(scene, 8)
    assert_equals_single_calls(loam, surf, EMPTY, hyp)
    assert_equals_single_calls(loam, EMPTY, edge, hyp)
    best_pose, best_idx, best_score, scores, poses = assert_equals_single_calls(loam, EMPTY, EMPTY, hyp)
    assert np.all(np.isinf(scores)) and best_idx == 0 and best_score == np.inf
    assert np.array_equal(poses, hyp) and np.array_equal(best_pose, hyp[0])
    # one hypothesis
    assert_equals_single_calls(loam, surf, edge, hyp[:1])
    # max_iteration = 0: the score pass runs at the poses as given
    loam.max_iteration = 0
    _, _, _, scores, poses = assert_equals_single_calls(loam, surf, edge, hyp)
    assert np.array_equal(poses, hyp) and np.isfinite(scores).any()


def test_argument_errors(scene):
    import loc_lib_b200 as L
    from loc_lib_b200 import _lib
    a = np.ascontiguousarray(scene.scan[:1024], np.float32)
    hyp = np.stack([IDENTITY, IDENTITY])
    bp, bs = np.zeros(7), np.zeros(1)
    bi = np.zeros(1, np.int64)

    def call(sharded, s, e, n_hyp=2, stride=16, surf_xyz=a, edge_xyz=a, n_surf=1024, pin=hyp):
        ptr = lambda x: None if x is None else x.ctypes.data  # noqa: E731
        h = lambda r: None if r is None else r._h  # noqa: E731
        args = [h(s), h(e), ptr(surf_xyz), n_surf, ptr(edge_xyz), 1024, stride, ptr(pin), n_hyp, 2, 0.0, ptr(bp), ptr(bi), ptr(bs)]
        if sharded:
            return _lib.lib().locreg_relocalise_loam_sharded(*args)
        return _lib.lib().locreg_relocalise_loam(*args, None, None)

    def err():
        return _lib.lib().locreg_last_error()

    plane = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE))
    line = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2LINE))
    p2p = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2P))
    ndt = L.NdtRegistration(L.NdtOptions())
    p2p.SetInputTarget(scene.map)
    ndt.SetInputTarget(scene.map)
    other = None
    if GPU_COUNT > 1:
        other = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2LINE), device=1)
        other.SetInputTarget(scene.map)
    for sharded in (False, True):
        if not sharded:
            assert call(sharded, plane, line) == -3 and b"surf handle" in err()  # no target yet
            plane.SetInputTarget(scene.map)
            assert call(sharded, plane, line) == -3 and b"edge handle" in err()
            line.SetInputTarget(scene.map)
        assert call(sharded, plane, line) == 0
        assert call(sharded, None, line) == -1 and b"null handle" in err()
        assert call(sharded, plane, None) == -1 and b"null handle" in err()
        assert call(sharded, plane, plane) == -1 and call(sharded, line, line) == -1 and call(sharded, line, plane) == -1
        assert call(sharded, p2p, line) == -1 and call(sharded, plane, p2p) == -1
        assert call(sharded, plane, ndt) == -1 and call(sharded, ndt, line) == -1
        if other is not None:
            assert call(sharded, plane, other) == -1 and b"different devices" in err()
        assert call(sharded, plane, line, stride=8) == -1 and call(sharded, plane, line, stride=18) == -1
        assert call(sharded, plane, line, surf_xyz=None) == -1 and call(sharded, plane, line, edge_xyz=None) == -1
        assert call(sharded, plane, line, pin=None) == -1 and b"invalid hypotheses" in err()
        assert call(sharded, plane, line, n_hyp=0) == -1 and b"invalid hypotheses" in err()
        assert call(sharded, plane, line, n_hyp=1 << 31) == -1 and b"invalid hypotheses" in err()
        # an empty cloud may come as a null pointer
        assert call(sharded, plane, line, surf_xyz=None, n_surf=0) == 0
    fresh = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2LINE))
    assert call(True, plane, fresh) == -3 and b"edge handle" in err()


def test_handles_stay_usable(scene):
    loam = make()
    loam.SetInputTarget(scene.map, scene.map)
    surf, edge = halves(scene)
    init = scene.init[0]
    pairs = [(sc[0::2], sc[1::2]) for sc in scene.scans]
    so = np.concatenate([[0], np.cumsum([len(p[0]) for p in pairs])]).astype(np.int64)
    eo = np.concatenate([[0], np.cumsum([len(p[1]) for p in pairs])]).astype(np.int64)
    sb = np.ascontiguousarray(np.concatenate([p[0] for p in pairs]), np.float32)
    eb = np.ascontiguousarray(np.concatenate([p[1] for p in pairs]), np.float32)

    def everything():
        pose, res = loam.ScanMatch(surf, edge, init)
        bp, br = loam.ScanMatchBatch(sb, so, eb, eo, np.asarray(scene.init))
        return pose, res, bp, br, loam.surf.ScanMatch(surf, init)[2], loam.edge.ScanMatch(edge, init)[2]

    before = everything()
    r1 = loam.Relocalise(surf, edge, hypotheses(scene, 16), want_all=True)
    after = everything()
    for x, y in zip(before, after):
        assert (np.array_equal(x, y) if isinstance(x, np.ndarray) else x == y)
    r2 = loam.Relocalise(surf, edge, hypotheses(scene, 16), want_all=True)
    assert r1[1:3] == r2[1:3] and np.array_equal(r1[3], r2[3]) and np.array_equal(r1[4], r2[4])


def test_one_caller_stream_equals_two_streams(scene):
    import torch
    loam = make()
    loam.SetInputTarget(scene.map, scene.map)
    surf, edge = halves(scene)
    hyp = hypotheses(scene, 16)
    two = loam.Relocalise(surf, edge, hyp, want_all=True)
    s = torch.cuda.Stream()
    loam.surf.set_stream(s.cuda_stream)
    loam.edge.set_stream(s.cuda_stream)
    one = loam.Relocalise(surf, edge, hyp, want_all=True)
    loam.surf.set_stream(0)
    loam.edge.set_stream(0)
    assert one[1:3] == two[1:3] and np.array_equal(one[0], two[0])
    assert np.array_equal(one[3], two[3]) and np.array_equal(one[4], two[4])


def test_sharded_world_of_one_equals_unsharded(scene):
    loam = make()
    loam.SetInputTarget(scene.map, scene.map)
    surf, edge = halves(scene)
    hyp = hypotheses(scene, 41)
    pose0, idx0, score0, _, _ = loam.Relocalise(surf, edge, hyp)
    # without a communicator: a world of one
    pose1, idx1, score1 = loam.RelocaliseSharded(surf, edge, hyp)
    assert idx1 == idx0 and score1 == score0 and np.array_equal(pose1, pose0)
    loam.CommInit(loam.CommUniqueId(), 0, 1)
    assert loam.CommInfo()[:2] == (0, 1)
    pose2, idx2, score2 = loam.RelocaliseSharded(surf, edge, hyp)
    assert idx2 == idx0 and score2 == score0 and np.array_equal(pose2, pose0)
    ms, launches = loam.last_timing()
    assert ms > 0 and launches > 10
    loam.CommDestroy()
    assert loam.CommInfo()[:2] == (0, 1)


def _rank_main(rank, world, uid, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import Scene
    from test_gpu_loam_reloc import halves, hypotheses, make
    scene = Scene()
    loam = make(max_iteration=2, device=rank)
    loam.SetInputTarget(scene.map, scene.map)
    loam.CommInit(uid, rank, world)
    surf, edge = halves(scene)
    pose, idx, score = loam.RelocaliseSharded(surf, edge, hypotheses(scene, 41))
    loam.CommDestroy()
    q.put((rank, pose, idx, score))


@pytest.mark.skipif(GPU_COUNT < 2, reason="needs two GPUs")
def test_two_ranks_agree_with_one(scene):
    import multiprocessing as mp
    loam = make(max_iteration=2)
    loam.SetInputTarget(scene.map, scene.map)
    surf, edge = halves(scene)
    pose0, idx0, score0, _, _ = loam.Relocalise(surf, edge, hypotheses(scene, 41))
    uid = loam.CommUniqueId()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_rank_main, args=(r, 2, uid, q)) for r in range(2)]
    for p in procs:
        p.start()
    outs = sorted([q.get(timeout=300) for _ in procs], key=lambda o: o[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, pose, idx, score in outs:
        assert idx == idx0 and score == score0 and np.array_equal(pose, pose0), rank
