"""GPU tests of locreg_relocalise_loam_staged[_sharded] / LoamRegistration.RelocaliseStaged[Sharded] against their
contract: a staged call equals the host chain of plain LoamRegistration.Relocalise calls (max_iteration = trips[r], each
round fed the poses the previous round left, the cut by reloc_staged_cases.survivors) bit for bit - poses, scores,
rounds and the winner - for cuts, score-only rounds, keep >= n, keep == 1 and one round; ties, empty halves, a scene
only both halves solve, waves, one caller stream, argument errors, the handles unchanged afterwards; and the sharded
form on a world of one and on 2, 4 and 8 ranks."""
import multiprocessing as mp
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import GPU_COUNT, ROOT, pose_delta
from loam_cases import KatScene, pose_from_rpy_t
from reloc_staged_cases import chain, survivors

pytestmark = pytest.mark.gpu

IDENTITY = np.array([0, 0, 0, 1, 0, 0, 0], np.float64)
EMPTY = np.zeros((0, 4), np.float32)
OWN_MAX_ITERATION = 7  # the LOAM object's own max_iteration, which no schedule uses


@pytest.fixture(scope="module", autouse=True)
def _torch_first():
    """torch is imported before the first sharded call loads NCCL: liblocreg.so then binds the NCCL torch brought
    (nccl_dyn.h), which a later torch import needs, instead of the system's."""
    import torch  # noqa: F401


def make(max_iteration=OWN_MAX_ITERATION, eps=0.0, device=0):
    import loc_lib_b200 as L
    so = L.IcpOptions(method_=L.IcpMethod.P2PLANE, max_iteration_=max_iteration, eps_=eps)
    eo = L.IcpOptions(method_=L.IcpMethod.P2LINE, max_iteration_=max_iteration, eps_=eps, max_line_distance_=0.5)
    return L.LoamRegistration(so, eo, max_iteration=max_iteration, eps=eps, device=device)


_LOAMS = {}


@pytest.fixture(scope="module", autouse=True)
def _close_handles():
    yield
    for loam in _LOAMS.values():
        loam.close()
    _LOAMS.clear()


def loam_for(scene, eps=0.0):
    """One LOAM pair with its targets per eps, kept for the module."""
    if eps not in _LOAMS:
        _LOAMS[eps] = make(eps=eps)
        _LOAMS[eps].SetInputTarget(scene.map, scene.map)
    return _LOAMS[eps]


def halves(scene):
    return scene.scan[0::2], scene.scan[1::2]


def hypotheses(scene, n_far=16):
    """48 hypotheses near the truth (one of them the scene's initial pose), then n_far far-off ones."""
    from loc_lib_b200 import synth
    hyp = [synth.perturb_pose(scene.gt[0], 1000 + i, 1.5, 6.0) for i in range(48)]
    hyp[17] = scene.init[0]
    hyp += [synth.perturb_pose(scene.gt[0], 3000 + i, 15.0, 60.0) for i in range(n_far)]
    return np.stack(hyp)


class LoamRounds:
    """reloc_staged_cases.chain's handle_for for LOAM: rounds(t).Relocalise((surf, edge), poses, want_all) is
    LoamRegistration.Relocalise with max_iteration = t, the object's own max_iteration restored afterwards."""

    def __init__(self, loam):
        self.loam, self.t = loam, None

    def __call__(self, t):
        self.t = t
        return self

    def Relocalise(self, clouds, hyp, want_all=False):
        own = self.loam.max_iteration
        self.loam.max_iteration = self.t
        try:
            return self.loam.Relocalise(clouds[0], clouds[1], hyp, want_all=want_all)
        finally:
            self.loam.max_iteration = own


def assert_equals_chain(loam, surf, edge, hyp, trips, keep):
    got = loam.RelocaliseStaged(surf, edge, hyp, trips, keep, want_all=True)
    bp, bi, bs, scores, poses, rounds = got
    cbest, cscores, cposes, crounds, history = chain(LoamRounds(loam), (surf, edge), hyp, trips, keep)
    assert np.array_equal(rounds, crounds), (rounds, crounds)
    for r in range(1, len(trips)):  # the survivors of every cut, as rounds_out shows them
        assert np.array_equal(np.flatnonzero(rounds > r), history[r]), r
    assert np.array_equal(scores, cscores), np.flatnonzero(scores != cscores)
    assert np.array_equal(poses, cposes), np.flatnonzero((poses != cposes).any(axis=1))
    assert bi == cbest and bs == scores[bi] and np.array_equal(bp, poses[bi])
    assert rounds[bi] == len(trips)
    assert loam.max_iteration == OWN_MAX_ITERATION
    return got


@pytest.mark.parametrize("trips, keep", [
    ((1, 2, 3), (16, 4)),     # cuts
    ((0, 2), (8,)),           # a score-only first round
    ((2, 0), (8,)),           # a score-only last round
    ((2, 3), (1000,)),        # keep >= n: no cut
    ((1, 2), (1,)),           # keep == 1: a single finalist
    ((3,), None),             # one round
])
def test_staged_equals_the_chain(scene, trips, keep):
    surf, edge = halves(scene)
    hyp = hypotheses(scene)
    _, bi, _, scores, _, rounds = assert_equals_chain(loam_for(scene), surf, edge, hyp, trips, keep)
    assert np.isfinite(scores).any()
    alive = len(hyp)
    for r in range(len(trips)):
        assert int((rounds > r).sum()) == alive, r
        if r < len(trips) - 1:
            alive = min(keep[r], alive)
    if keep == (1,):
        assert np.flatnonzero(rounds == 2).tolist() == [bi]


def test_eps_is_the_callers(scene):
    """eps > 0: hypotheses converge and stop inside a round; the staged call passes the object's eps to every round."""
    surf, edge = halves(scene)
    assert_equals_chain(loam_for(scene, 1e-2), surf, edge, hypotheses(scene), (2, 3, 5), (16, 4))


def test_one_round_equals_relocalise_loam(scene):
    loam = loam_for(scene)
    surf, edge = halves(scene)
    hyp = hypotheses(scene)
    loam.max_iteration = 4
    try:
        bp, bi, bs, scores, poses = loam.Relocalise(surf, edge, hyp, want_all=True)
    finally:
        loam.max_iteration = OWN_MAX_ITERATION
    sp, si, ss, sscores, sposes, rounds = loam.RelocaliseStaged(surf, edge, hyp, (4,), None, want_all=True)
    assert np.array_equal(sscores, scores) and np.array_equal(sposes, poses)
    assert (si, ss) == (bi, bs) and np.array_equal(sp, bp)
    assert np.all(rounds == 1) and np.isfinite(scores).any()
    ms, launches = loam.last_timing()
    assert ms > 0 and launches > 10


def test_a_tie_at_the_cut_goes_to_the_lower_index(scene):
    loam = loam_for(scene)
    surf, edge = halves(scene)
    hyp = hypotheses(scene)
    _, _, _, s0, _ = LoamRounds(loam)(1).Relocalise((surf, edge), hyp, want_all=True)
    keep = 10
    order = np.lexsort((np.arange(len(hyp)), np.float32(s0)))
    last_in = int(order[keep - 1])  # the last survivor of a cut at `keep`
    assert np.float32(s0[order[keep - 1]]) != np.float32(s0[order[keep]])
    assert last_in in survivors(s0, np.arange(len(hyp)), keep)
    dup = np.concatenate([hyp, hyp[last_in][None]])  # the same hypothesis at the highest index straddles the cut
    _, _, _, scores, _, rounds = assert_equals_chain(loam, surf, edge, dup, (1, 2), (keep,))
    assert scores[-1] == s0[last_in] and rounds[last_in] == 2 and rounds[-1] == 1


def test_a_tie_for_the_winner_goes_to_the_lower_index(scene):
    loam = loam_for(scene)
    surf, edge = halves(scene)
    hyp = hypotheses(scene)
    _, bi, bs, _, _, _ = loam.RelocaliseStaged(surf, edge, hyp, (1, 2), (8,))
    # the winner's copy at the highest index: one more survivor makes room for it
    dup = np.concatenate([hyp, hyp[bi][None]])
    _, bi2, bs2, scores, _, rounds = assert_equals_chain(loam, surf, edge, dup, (1, 2), (9,))
    assert rounds[-1] == 2 and scores[-1] == scores[bi]  # the copy reached the last round with the same score
    assert bi2 != len(dup) - 1  # ... and never wins: the lower index takes the tie
    if np.float32(bs) == np.float32(scores[rounds == 2]).min():
        assert (bi2, bs2) == (bi, bs)


def test_empty_halves(scene):
    loam = loam_for(scene)
    surf, edge = halves(scene)
    hyp = hypotheses(scene)
    assert_equals_chain(loam, surf, EMPTY, hyp, (1, 2), (8,))
    assert_equals_chain(loam, EMPTY, edge, hyp, (1, 2), (8,))
    bp, bi, bs, scores, poses, rounds = assert_equals_chain(loam, EMPTY, EMPTY, hyp, (1, 2), (8,))
    assert np.all(np.isinf(scores)) and bi == 0 and bs == np.inf
    assert np.array_equal(np.flatnonzero(rounds == 2), np.arange(8))  # all +inf: the lowest indices go on
    assert np.array_equal(poses, hyp) and np.array_equal(bp, hyp[0])


def test_a_scene_only_both_halves_solve():
    """KatScene: a plane (surf) and two poles (edge).  The staged LOAM winner reaches the truth; a staged P2Plane-only
    call on the surf half (a second handle a LOAM user would otherwise keep) cannot fix x, y or yaw."""
    import loc_lib_b200 as L
    k = KatScene()
    kat = make()
    kat.SetInputTarget(k.surf_map, k.edge_map)
    hyp = np.stack([k.init, pose_from_rpy_t([0.005, 0.0, -0.01], [0.02, 0.01, 0.0]),
                    pose_from_rpy_t([0.0, 0.0, 0.1], [0.2, -0.1, 0.05]), pose_from_rpy_t([0.02, 0.01, -0.05], [-0.1, 0.15, 0.1])])
    bp, bi, bs, scores, _, rounds = kat.RelocaliseStaged(k.surf, k.edge, hyp, (2, 8), (2,), want_all=True)
    dr, dt = pose_delta(bp, k.truth)
    assert np.isfinite(bs) and rounds[bi] == 2
    assert dr < 1e-4 and dt < 1e-3, (bi, dr, dt)
    plane = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE, max_iteration_=10, eps_=0.0))
    plane.SetInputTarget(k.surf_map)
    pp, pi, _, _, _, _ = plane.RelocaliseStaged(k.surf, hyp, (2, 8), (2,))
    assert np.linalg.norm(pp[4:6] - k.truth[4:6]) > 0.03, (pi, pp)  # x, y stay where the hypothesis put them
    plane.close()
    kat.close()


_WAVES = r"""
import sys
import numpy as np
sys.path[:0] = [{root!r}, {tests!r}]
from conftest import Scene
from test_gpu_loam_reloc_staged import make, halves, hypotheses
scene = Scene()
loam = make()
loam.SetInputTarget(scene.map, scene.map)
surf, edge = halves(scene)
bp, bi, bs, scores, poses, rounds = loam.RelocaliseStaged(surf, edge, hypotheses(scene), (1, 2, 3), (16, 4), want_all=True)
np.savez({out!r}, bp=bp, bi=bi, bs=bs, scores=scores, poses=poses, rounds=rounds, launches=loam.last_timing()[1])
loam.close()
"""


def test_waves_agree_bit_for_bit(scene, tmp_path):
    """LOCREG_RELOC_WAVE_GIB is read once per process: a subprocess runs every round in waves of a few hypotheses."""
    loam = loam_for(scene)
    surf, edge = halves(scene)
    bp, bi, bs, scores, poses, rounds = loam.RelocaliseStaged(surf, edge, hypotheses(scene), (1, 2, 3), (16, 4), want_all=True)
    launches = loam.last_timing()[1]
    out = str(tmp_path / "waves.npz")
    env = dict(os.environ, LOCREG_RELOC_WAVE_GIB="0.0005")
    code = _WAVES.format(root=ROOT, tests=os.path.join(ROOT, "tests"), out=out)
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    w = np.load(out)
    assert int(w["bi"]) == bi and float(w["bs"]) == bs and np.array_equal(w["bp"], bp)
    assert np.array_equal(w["scores"], scores) and np.array_equal(w["poses"], poses) and np.array_equal(w["rounds"], rounds)
    assert int(w["launches"]) > 2 * launches  # several waves per round really ran


def test_one_caller_stream_equals_two_streams(scene):
    import torch
    loam = loam_for(scene)
    surf, edge = halves(scene)
    hyp = hypotheses(scene)
    two = loam.RelocaliseStaged(surf, edge, hyp, (1, 2, 3), (16, 4), want_all=True)
    s = torch.cuda.Stream()
    loam.surf.set_stream(s.cuda_stream)
    loam.edge.set_stream(s.cuda_stream)
    try:
        one = loam.RelocaliseStaged(surf, edge, hyp, (1, 2, 3), (16, 4), want_all=True)
    finally:
        loam.surf.set_stream(0)
        loam.edge.set_stream(0)
    assert one[1:3] == two[1:3] and np.array_equal(one[0], two[0])
    for a, b in zip(one[3:], two[3:]):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("symbol", ["locreg_relocalise_loam_staged", "locreg_relocalise_loam_staged_sharded"])
def test_argument_errors(scene, symbol):
    import loc_lib_b200 as L
    from loc_lib_b200 import _lib
    a = np.ascontiguousarray(scene.scan[:1024], np.float32)
    hyp = np.stack([IDENTITY, IDENTITY, IDENTITY])
    bp, bs = np.zeros(7), np.zeros(1)
    bi = np.zeros(1, np.int64)
    t3 = np.array([1, 1, 1], np.int32)
    k2 = np.array([2, 1], np.int64)
    ptr = lambda x: None if x is None else x.ctypes.data  # noqa: E731
    h = lambda r: None if r is None else r._h  # noqa: E731

    def call(s, e, surf_xyz=a, n_surf=1024, edge_xyz=a, stride=16, pin=hyp, n_hyp=3, trips=t3, keep=k2, n_rounds=3):
        rc = getattr(_lib.lib(), symbol)(h(s), h(e), ptr(surf_xyz), n_surf, ptr(edge_xyz), 1024, stride, ptr(pin), n_hyp,
                                         ptr(trips), ptr(keep), n_rounds, 0.0, ptr(bp), ptr(bi), ptr(bs), None, None, None)
        return rc, _lib.lib().locreg_last_error()

    plane = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE))
    line = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2LINE))
    p2p = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2P))
    ndt = L.NdtRegistration(L.NdtOptions())
    p2p.SetInputTarget(scene.map)
    ndt.SetInputTarget(scene.map)
    rc, err = call(plane, line)
    assert rc == -3 and b"surf handle" in err  # no target yet
    plane.SetInputTarget(scene.map)
    rc, err = call(plane, line)
    assert rc == -3 and b"edge handle" in err
    line.SetInputTarget(scene.map)
    assert call(plane, line)[0] == 0
    assert call(None, line) == (-1, b"null handle") and call(plane, None) == (-1, b"null handle")
    for s, e in ((plane, plane), (line, line), (line, plane), (p2p, line), (plane, p2p), (plane, ndt), (ndt, line)):
        assert call(s, e)[0] == -1
    if GPU_COUNT > 1:
        other = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2LINE), device=1)
        other.SetInputTarget(scene.map)
        rc, err = call(plane, other)
        assert rc == -1 and b"different devices" in err
        other.close()
    assert call(plane, line, stride=8)[0] == -1 and call(plane, line, stride=18)[0] == -1
    assert call(plane, line, surf_xyz=None)[0] == -1 and call(plane, line, edge_xyz=None)[0] == -1
    for bad in ({"pin": None}, {"n_hyp": 0}, {"n_hyp": 1 << 31}):
        rc, err = call(plane, line, **bad)
        assert rc == -1 and b"invalid hypotheses" in err, bad
    for n_rounds in (0, -1, 33):
        rc, err = call(plane, line, n_rounds=n_rounds)
        assert rc == -1 and b"n_rounds" in err, n_rounds
    for bad in ({"trips": None}, {"trips": np.array([1, -2, 1], np.int32)}):
        rc, err = call(plane, line, **bad)
        assert rc == -1 and b"trips" in err, bad
    for bad in ({"keep": None}, {"keep": np.array([0, 1], np.int64)}, {"keep": np.array([2, -1], np.int64)}):
        rc, err = call(plane, line, **bad)
        assert rc == -1 and b"keep" in err, bad
    # valid: one round without keep, an empty cloud as a null pointer, score-only rounds and a keep beyond the alive set
    assert call(plane, line, keep=None, n_rounds=1)[0] == 0
    assert call(plane, line, surf_xyz=None, n_surf=0)[0] == 0
    assert call(plane, line, trips=np.array([0, 0, 0], np.int32), keep=np.array([1 << 40, 1], np.int64))[0] == 0
    # the refusals changed nothing on the device: the handles still work
    assert call(plane, line)[0] == 0
    for reg in (plane, line, p2p, ndt):
        reg.close()


def test_the_handles_are_unchanged_afterwards(scene):
    loam = loam_for(scene)
    surf, edge = halves(scene)
    hyp = hypotheses(scene)
    init = scene.init[0]

    def everything():
        return (loam.Relocalise(surf, edge, hyp, want_all=True), loam.ScanMatch(surf, edge, init)[0],
                loam.surf.ScanMatch(surf, init, want_cloud=False)[2], loam.edge.ScanMatch(edge, init, want_cloud=False)[2],
                loam.surf.Relocalise(surf, hyp, want_all=True), loam.edge.Relocalise(edge, hyp, want_all=True))

    def flat(x):
        return [y for z in x for y in (flat(z) if isinstance(z, tuple) else [z])]

    before = flat(everything())
    loam.RelocaliseStaged(surf, edge, hyp, (0, 2, 9), (20, 5))
    ms, launches = loam.last_timing()
    assert ms > 0 and launches > 10
    loam.RelocaliseStagedSharded(surf, edge, hyp, (0, 2, 9), (20, 5))
    after = flat(everything())
    assert loam.max_iteration == OWN_MAX_ITERATION
    for x, y in zip(before, after):
        assert (np.array_equal(x, y) if isinstance(x, np.ndarray) else x == y)


def assert_same(got, want, what):
    bp, bi, bs, scores, poses, rounds = got
    wbp, wbi, wbs, wscores, wposes, wrounds = want
    assert bi == wbi and np.array_equal(np.float64(bs), np.float64(wbs)), (what, bi, wbi, bs, wbs)
    assert np.array_equal(bp, wbp), what
    assert np.array_equal(rounds, wrounds), what
    assert np.array_equal(scores, wscores), (what, np.flatnonzero(scores != wscores))
    assert np.array_equal(poses, wposes), (what, np.flatnonzero((poses != wposes).any(axis=1)))


def test_world_of_one_is_the_single_gpu_call(scene):
    loam = loam_for(scene)
    surf, edge = halves(scene)
    hyp = hypotheses(scene)
    schedules = [((1, 2, 3), (16, 4)), ((2, 3), (len(hyp),)), ((0, 2), (8,))]  # cuts, no cut, a score-only round
    for comm in (False, True):
        if comm:
            loam.CommInit(loam.CommUniqueId(), 0, 1)
            assert loam.CommInfo()[:2] == (0, 1)
        try:
            for trips, keep in schedules:
                want = loam.RelocaliseStaged(surf, edge, hyp, trips, keep, want_all=True)
                launches = loam.last_timing()[1]
                got = loam.RelocaliseStagedSharded(surf, edge, hyp, trips, keep, want_all=True)
                assert_same(got, want, (comm, trips, keep))
                assert loam.last_timing()[1] == launches  # the same launch sequence: no deal, pack or unpack
                bp, bi, bs, scores, _, _ = loam.RelocaliseStagedSharded(surf, edge, hyp, trips, keep)
                assert scores is None and bi == want[1] and bs == want[2] and np.array_equal(bp, want[0])
        finally:
            if comm:
                loam.CommDestroy()


# Ranks that share one GPU: NCCL refuses two ranks of one host on one device, so each rank names a host of its own
# (NCCL_HOSTID) and the ranks talk over loopback sockets (as tests/test_gpu_reloc_staged_sharded.py does).
def _shared_gpu_env(rank):
    return {"NCCL_HOSTID": "locreg-test-rank-%d" % rank, "NCCL_SOCKET_IFNAME": "lo", "NCCL_NET": "Socket",
            "NCCL_IB_DISABLE": "1", "NCCL_MNNVL_ENABLE": "0"}


# (name, hypotheses (slice of hypotheses()), surf / edge halves present, trips, keep)
TWO_RANK_CASES = [
    ("cuts", slice(None), (True, True), (1, 2, 3), (16, 4)),
    ("odd survivors", slice(None), (True, True), (1, 2), (7,)),
    ("last round below the ranks", slice(None), (True, True), (1, 2, 2), (5, 1)),
    ("one hypothesis", slice(17, 18), (True, True), (1, 2, 3), (4, 4)),
    ("no edge half", slice(None), (True, False), (1, 2), (8,)),
]
# 64 -> 13 -> 6 -> 3 alive: m mod 4 = 0, 1, 2, 3; on 8 ranks rounds with more, and with fewer, alive than ranks
MANY_RANK_CASES = [("every remainder", slice(None), (True, True), (1, 1, 1, 1), (13, 6, 3)),
                   ("score-only round", slice(None), (True, True), (0, 2), (5,))]


def case_clouds(scene, present):
    surf, edge = halves(scene)
    return surf if present[0] else EMPTY, edge if present[1] else EMPTY


def _rank_main(rank, world, shared, cases, uid_q, q):
    sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
    if shared:
        os.environ.update(_shared_gpu_env(rank))  # before the first NCCL call of this process
    try:
        import loc_lib_b200 as L
        from conftest import Scene
        if rank == 0:
            uid = L.LoamRegistration.CommUniqueId()
            for _ in range(world - 1):
                uid_q.put(uid)
        else:
            uid = uid_q.get(timeout=300)
        scene = Scene()
        loam = make(device=0 if shared else rank)
        loam.SetInputTarget(scene.map, scene.map)
        loam.CommInit(uid, rank, world)
        assert loam.CommInfo()[:2] == (rank, world)
        outs = []
        for name, sl, present, trips, keep in cases:
            surf, edge = case_clouds(scene, present)
            outs.append(loam.RelocaliseStagedSharded(surf, edge, hypotheses(scene)[sl], trips, keep, want_all=True))
        # the handles afterwards: the exhaustive LOAM call as on a fresh pair
        surf, edge = halves(scene)
        after = loam.Relocalise(surf, edge, hypotheses(scene))[:3]
        loam.CommDestroy()
        loam.close()
        q.put((rank, outs, after, None))
    except Exception as e:  # noqa: BLE001 - reported to the parent, which fails the test with it
        q.put((rank, None, None, repr(e)))


def run_ranks(scene, world, cases, shared=False):
    """Every case on `world` spawned ranks (one GPU each, or all on GPU 0 with `shared`); every rank's outputs must
    equal the single-GPU staged call."""
    loam = loam_for(scene)
    want = []
    for name, sl, present, trips, keep in cases:
        surf, edge = case_clouds(scene, present)
        want.append(loam.RelocaliseStaged(surf, edge, hypotheses(scene)[sl], trips, keep, want_all=True))
    fresh = make()
    fresh.SetInputTarget(scene.map, scene.map)
    fresh_single = fresh.Relocalise(*halves(scene), hypotheses(scene))[:3]
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
        p1, i1, s1 = after
        assert (i1, s1) == fresh_single[1:] and np.array_equal(p1, fresh_single[0]), rank
    return want


def check_two_rank_cases(want):
    """The two-rank cases cover what they are named for."""
    rounds = {c[0]: w[5] for c, w in zip(TWO_RANK_CASES, want)}
    assert int((rounds["odd survivors"] == 2).sum()) == 7
    assert int((rounds["last round below the ranks"] == 3).sum()) == 1
    assert rounds["one hypothesis"].tolist() == [3]


def check_many_rank_cases(want):
    alive = [int((want[0][5] > r).sum()) for r in range(4)]
    assert alive == [64, 13, 6, 3] and {a % 4 for a in alive} == {0, 1, 2, 3}


def test_two_ranks_sharing_one_gpu_agree_with_one_gpu(scene):
    check_two_rank_cases(run_ranks(scene, 2, TWO_RANK_CASES, shared=True))


def test_four_ranks_sharing_one_gpu_agree_with_one_gpu(scene):
    check_many_rank_cases(run_ranks(scene, 4, MANY_RANK_CASES, shared=True))


def test_eight_ranks_sharing_one_gpu_agree_with_one_gpu(scene):
    check_many_rank_cases(run_ranks(scene, 8, MANY_RANK_CASES, shared=True))


@pytest.mark.skipif(GPU_COUNT < 2, reason="needs two GPUs")
def test_two_ranks_agree_with_one_gpu(scene):
    check_two_rank_cases(run_ranks(scene, 2, TWO_RANK_CASES))


@pytest.mark.skipif(GPU_COUNT < 4, reason="needs four GPUs")
def test_four_ranks_agree_with_one_gpu(scene):
    check_many_rank_cases(run_ranks(scene, 4, MANY_RANK_CASES))
