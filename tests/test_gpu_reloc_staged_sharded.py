"""GPU tests of locreg_relocalise_staged_sharded / RelocaliseStagedSharded: on every rank, all six outputs (winner pose,
index and score, every hypothesis's score, pose and rounds) are bit for bit what the single-GPU RelocaliseStaged
returns for the same scene and schedule.  A world of one (no communicator, or a one-rank one) is the single-GPU call;
two and four ranks run as spawned processes, one GPU each (skipped on a box with fewer GPUs), and two, four and eight
ranks also run sharing GPU 0, which needs one GPU only.  The handle is unchanged afterwards."""
import multiprocessing as mp
import os

import numpy as np
import pytest

from conftest import GPU_COUNT, ROOT
from reloc_staged_cases import chain

pytestmark = pytest.mark.gpu

P2PLANE, P2P, NDT = "p2plane", "p2p", "ndt"
STAGED_MAX_ITERATION = 7  # the handles' own max_iteration, which no schedule uses


def make(method, max_iteration, zero_t=False, device=0):
    import loc_lib_b200 as L
    if method == NDT:
        return L.NdtRegistration(L.NdtOptions(max_iteration_=max_iteration, eps_=0.0, remove_centroid_=zero_t), device=device)
    m = L.IcpMethod.P2PLANE if method == P2PLANE else L.IcpMethod.P2P
    return L.IcpRegistration(L.IcpOptions(method_=m, max_iteration_=max_iteration, eps_=0.0,
                                          use_initial_translation_=not zero_t), device=device)


_HANDLES = {}


@pytest.fixture(scope="module", autouse=True)
def _close_handles():
    yield
    for reg in _HANDLES.values():
        reg.close()
    _HANDLES.clear()


def handle(scene, method, max_iteration=STAGED_MAX_ITERATION, zero_t=False):
    """One handle with its target per (method, max_iteration, zero_t), kept for the module."""
    key = (method, max_iteration, zero_t)
    if key not in _HANDLES:
        _HANDLES[key] = make(method, max_iteration, zero_t)
        _HANDLES[key].SetInputTarget(scene.map)
    return _HANDLES[key]


def hypotheses(scene, n_far=16):
    """test_gpu_reloc_staged.py's 64 hypotheses: 48 near the truth (one of them the scene's initial pose), 16 far off."""
    from loc_lib_b200 import synth
    hyp = [synth.perturb_pose(scene.gt[0], 1000 + i, 1.5, 6.0) for i in range(48)]
    hyp[17] = scene.init[0]
    hyp += [synth.perturb_pose(scene.gt[0], 3000 + i, 15.0, 60.0) for i in range(n_far)]
    return np.stack(hyp)


# (name, method, zero_t, hypotheses (slice of hypotheses()), trips, keep)
TWO_RANK_CASES = [
    ("cuts", P2PLANE, False, slice(None), (1, 2, 3), (16, 4)),
    ("odd survivors", P2PLANE, False, slice(None), (1, 2), (7,)),
    ("last round below the ranks", P2PLANE, False, slice(None), (1, 2, 2), (5, 1)),
    ("one hypothesis", P2PLANE, False, slice(17, 18), (1, 2, 3), (4, 4)),
    ("ndt", NDT, False, slice(None), (1, 2, 3), (16, 4)),
    ("zero initial translation", P2PLANE, True, slice(0, 24), (2, 3), (6,)),
]
# 64 -> 13 -> 6 -> 3 alive: m mod 4 = 0, 1, 2, 3
FOUR_RANK_CASES = [("every remainder", P2PLANE, False, slice(None), (1, 1, 1, 1), (13, 6, 3))]


def assert_same(got, want, what):
    bp, bi, bs, scores, poses, rounds = got
    wbp, wbi, wbs, wscores, wposes, wrounds = want
    assert bi == wbi and np.array_equal(np.float64(bs), np.float64(wbs), equal_nan=True), (what, bi, wbi, bs, wbs)
    assert np.array_equal(bp, wbp), what
    assert np.array_equal(rounds, wrounds), what
    assert np.array_equal(scores, wscores, equal_nan=True), (what, np.flatnonzero(scores != wscores))
    assert np.array_equal(poses, wposes), (what, np.flatnonzero((poses != wposes).any(axis=1)))


def single_gpu(scene, cases):
    out = []
    for name, method, zero_t, sl, trips, keep in cases:
        reg = handle(scene, method, zero_t=zero_t)
        out.append(reg.RelocaliseStaged(scene.scan, hypotheses(scene)[sl], trips, keep, want_all=True))
    return out


@pytest.mark.parametrize("method", [P2PLANE, P2P, NDT])
def test_world_of_one_is_the_single_gpu_call(scene, method):
    hyp = hypotheses(scene)
    reg = handle(scene, method)
    schedules = [((1, 2, 3), (16, 4)), ((2, 3), (len(hyp),)), ((0, 2), (8,))]  # cuts, no cut, a score-only round
    for comm in (False, True):
        if comm:
            reg.CommInit(reg.CommUniqueId(), 0, 1)
            assert reg.CommInfo()[:2] == (0, 1)
        try:
            for trips, keep in schedules:
                want = reg.RelocaliseStaged(scene.scan, hyp, trips, keep, want_all=True)
                launches = reg.last_timing()[1]
                got = reg.RelocaliseStagedSharded(scene.scan, hyp, trips, keep, want_all=True)
                assert_same(got, want, (method, comm, trips, keep))
                assert reg.last_timing()[1] == launches  # the same launch sequence: no deal, pack or unpack
                # outputs may be left out, as in the single-GPU call
                bp, bi, bs, scores, poses, rounds = reg.RelocaliseStagedSharded(scene.scan, hyp, trips, keep)
                assert scores is None and bi == want[1] and bs == want[2] and np.array_equal(bp, want[0])
        finally:
            if comm:
                reg.CommDestroy()
    if method == P2PLANE:  # and the contract itself: the host chain of locreg_relocalise calls
        got = reg.RelocaliseStagedSharded(scene.scan, hyp, (1, 2, 3), (16, 4), want_all=True)
        cbest, cscores, cposes, crounds, _ = chain(lambda t: handle(scene, P2PLANE, t), scene.scan, hyp, (1, 2, 3), (16, 4))
        assert got[1] == cbest and np.array_equal(got[3], cscores) and np.array_equal(got[4], cposes)
        assert np.array_equal(got[5], crounds)


def test_the_handle_is_unchanged_afterwards(scene):
    hyp = hypotheses(scene)
    for zero_t in (False, True):
        reg = handle(scene, P2PLANE, 5, zero_t=zero_t)
        before = reg.Relocalise(scene.scan, hyp, want_all=True)
        before_sharded = reg.RelocaliseSharded(scene.scan, hyp)
        reg.RelocaliseStagedSharded(scene.scan, hyp, (0, 2, 9), (20, 5))
        ms, launches = reg.last_timing()
        assert ms > 0 and launches > 0
        after = reg.Relocalise(scene.scan, hyp, want_all=True)
        assert before[1:3] == after[1:3] and np.array_equal(before[0], after[0])
        assert np.array_equal(before[3], after[3]) and np.array_equal(before[4], after[4])
        after_sharded = reg.RelocaliseSharded(scene.scan, hyp)
        assert before_sharded[1:] == after_sharded[1:] and np.array_equal(before_sharded[0], after_sharded[0])


# Ranks that share one GPU: NCCL refuses two ranks of one host on one device, so each rank names a host of its own
# (NCCL_HOSTID) and the ranks talk over loopback sockets.  Slower than NVLink, but every rank runs the same deal, pack,
# ncclAllGather and unpack as on a GPU of its own; on a box with fewer GPUs than ranks this is how the cross-rank path
# runs at all.
def _shared_gpu_env(rank):
    return {"NCCL_HOSTID": "locreg-test-rank-%d" % rank, "NCCL_SOCKET_IFNAME": "lo", "NCCL_NET": "Socket",
            "NCCL_IB_DISABLE": "1", "NCCL_MNNVL_ENABLE": "0"}


def _rank_main(rank, world, shared, cases, uid_q, q):
    import sys
    sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
    if shared:
        os.environ.update(_shared_gpu_env(rank))  # before the first NCCL call of this process
    try:
        import loc_lib_b200 as L
        from conftest import Scene
        # one communicator per handle, with ids drawn on rank 0 and handed to the others
        keys = sorted({(m, z) for _, m, z, _, _, _ in cases} | {(P2PLANE, False)})
        if rank == 0:
            uid = {k: L.IcpRegistration.CommUniqueId() for k in keys}
            for _ in range(world - 1):
                uid_q.put(uid)
        else:
            uid = uid_q.get(timeout=300)
        scene = Scene()
        regs, outs = {}, []
        for k in keys:
            regs[k] = make(k[0], STAGED_MAX_ITERATION, k[1], device=0 if shared else rank)
            regs[k].SetInputTarget(scene.map)
            regs[k].CommInit(uid[k], rank, world)
            assert regs[k].CommInfo()[:2] == (rank, world)
        for name, method, zero_t, sl, trips, keep in cases:
            outs.append(regs[(method, zero_t)].RelocaliseStagedSharded(scene.scan, hypotheses(scene)[sl], trips, keep,
                                                                        want_all=True))
        # the handle afterwards: the exhaustive sharded and single-GPU calls as on a fresh handle
        reg = regs[(P2PLANE, False)]
        hyp = hypotheses(scene)
        after = (reg.RelocaliseSharded(scene.scan, hyp), reg.Relocalise(scene.scan, hyp)[:3])
        for reg in regs.values():
            reg.CommDestroy()
            reg.close()
        q.put((rank, outs, after, None))
    except Exception as e:  # noqa: BLE001 - reported to the parent, which fails the test with it
        q.put((rank, None, None, repr(e)))


def run_ranks(scene, world, cases, shared=False):
    """Every case on `world` spawned ranks (one GPU each, or all on GPU 0 with `shared`); every rank's outputs must
    equal the single-GPU call."""
    want = single_gpu(scene, cases)
    fresh = make(P2PLANE, STAGED_MAX_ITERATION)
    fresh.SetInputTarget(scene.map)
    hyp = hypotheses(scene)
    fresh_sharded, fresh_single = fresh.RelocaliseSharded(scene.scan, hyp), fresh.Relocalise(scene.scan, hyp)[:3]
    fresh.close()
    ctx = mp.get_context("spawn")
    q, uid_q = ctx.Queue(), ctx.Queue()
    procs = [ctx.Process(target=_rank_main, args=(r, world, shared, cases, uid_q, q)) for r in range(world)]
    try:
        for p in procs:
            p.start()
        outs = sorted([q.get(timeout=900) for _ in procs], key=lambda o: o[0])
        for p in procs:
            p.join(timeout=120)
            assert p.exitcode == 0
    finally:
        for p in procs:  # a rank that failed leaves the others waiting in a collective: end them all
            if p.is_alive():
                p.kill()
                p.join()
    for rank, got, after, err in outs:
        assert err is None, (rank, err)
        for case, g, w in zip(cases, got, want):
            assert_same(g, w, (rank, case[0]))
        (sp, si, ss), (p1, i1, s1) = after
        assert (si, ss) == fresh_sharded[1:] and np.array_equal(sp, fresh_sharded[0]), rank
        assert (i1, s1) == fresh_single[1:] and np.array_equal(p1, fresh_single[0]), rank
    return want


def check_two_rank_cases(want):
    """The two-rank cases cover what they are named for."""
    rounds = {c[0]: w[5] for c, w in zip(TWO_RANK_CASES, want)}
    assert int((rounds["odd survivors"] == 2).sum()) == 7
    assert int((rounds["last round below the ranks"] == 3).sum()) == 1
    assert rounds["one hypothesis"].tolist() == [3]


def check_four_rank_cases(want):
    alive = [int((want[0][5] > r).sum()) for r in range(4)]
    assert alive == [64, 13, 6, 3] and {a % 4 for a in alive} == {0, 1, 2, 3}


@pytest.mark.skipif(GPU_COUNT < 2, reason="needs two GPUs")
def test_two_ranks_agree_with_one_gpu(scene):
    check_two_rank_cases(run_ranks(scene, 2, TWO_RANK_CASES))


@pytest.mark.skipif(GPU_COUNT < 4, reason="needs four GPUs")
def test_four_ranks_agree_with_one_gpu(scene):
    check_four_rank_cases(run_ranks(scene, 4, FOUR_RANK_CASES))


# 64 -> 13 -> 6 -> 3 alive on 8 ranks: rounds with more, and with fewer, alive hypotheses than ranks
EIGHT_RANK_CASES = [("every remainder", P2PLANE, False, slice(None), (1, 1, 1, 1), (13, 6, 3)),
                    ("ndt", NDT, False, slice(None), (1, 2), (5,))]


def test_two_ranks_sharing_one_gpu_agree_with_one_gpu(scene):
    check_two_rank_cases(run_ranks(scene, 2, TWO_RANK_CASES, shared=True))


def test_four_ranks_sharing_one_gpu_agree_with_one_gpu(scene):
    check_four_rank_cases(run_ranks(scene, 4, FOUR_RANK_CASES, shared=True))


def test_eight_ranks_sharing_one_gpu_agree_with_one_gpu(scene):
    run_ranks(scene, 8, EIGHT_RANK_CASES, shared=True)
