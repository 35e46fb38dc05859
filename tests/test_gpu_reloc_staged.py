"""GPU tests of locreg_relocalise_staged / RelocaliseStaged against its contract: a staged call equals the host chain of
locreg_relocalise calls (handles with max_iteration = trips[r], each round fed the previous round's poses, the cut by
reloc_staged_cases.survivors) bit for bit - poses, scores, rounds and the winner - with and without cuts, at ties, for
all-+inf rounds, in waves; argument errors; the handle unchanged afterwards; and the winner on the scene."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, pose_delta
from reloc_staged_cases import chain

pytestmark = pytest.mark.gpu

IDENTITY = np.array([0, 0, 0, 1, 0, 0, 0], np.float64)
P2PLANE, P2P, NDT = "p2plane", "p2p", "ndt"


def make(method, max_iteration, eps=0.0, zero_t=False):
    import loc_lib_b200 as L
    if method == NDT:
        return L.NdtRegistration(L.NdtOptions(max_iteration_=max_iteration, eps_=eps, remove_centroid_=zero_t))
    m = L.IcpMethod.P2PLANE if method == P2PLANE else L.IcpMethod.P2P
    return L.IcpRegistration(L.IcpOptions(method_=m, max_iteration_=max_iteration, eps_=eps, use_initial_translation_=not zero_t))


_HANDLES = {}


@pytest.fixture(scope="module", autouse=True)
def _close_handles():
    yield
    for reg in _HANDLES.values():
        reg.close()
    _HANDLES.clear()


def handle(scene, method, max_iteration, eps=0.0, zero_t=False):
    """One handle with its target per (method, max_iteration, eps, zero_t), kept for the module."""
    key = (method, max_iteration, eps, zero_t)
    if key not in _HANDLES:
        _HANDLES[key] = make(method, max_iteration, eps, zero_t)
        _HANDLES[key].SetInputTarget(scene.map)
    return _HANDLES[key]


def hypotheses(scene, n_far=16):
    """test_parity.py::test_relocalise's 48 hypotheses, then n_far far-off ones (up to 15 m and 60 degrees away)."""
    from loc_lib_b200 import synth
    hyp = [synth.perturb_pose(scene.gt[0], 1000 + i, 1.5, 6.0) for i in range(48)]
    hyp[17] = scene.init[0]
    hyp += [synth.perturb_pose(scene.gt[0], 3000 + i, 15.0, 60.0) for i in range(n_far)]
    return np.stack(hyp)


def assert_equals_chain(scene, method, trips, keep, hyp=None, eps=0.0, staged_max_iteration=7):
    """The staged call on a handle whose own max_iteration is not any trips[r] equals the host chain bit for bit."""
    hyp = hypotheses(scene) if hyp is None else hyp
    reg = handle(scene, method, staged_max_iteration, eps)
    bp, bi, bs, scores, poses, rounds = reg.RelocaliseStaged(scene.scan, hyp, trips, keep, want_all=True)
    cbest, cscores, cposes, crounds, history = chain(lambda t: handle(scene, method, t, eps), scene.scan, hyp, trips, keep)
    assert np.array_equal(rounds, crounds), (rounds, crounds)
    for r in range(1, len(trips)):  # the survivors of every cut, as rounds_out shows them
        assert np.array_equal(np.flatnonzero(rounds > r), history[r]), r
    assert np.array_equal(scores, cscores), np.flatnonzero(scores != cscores)
    assert np.array_equal(poses, cposes), np.flatnonzero((poses != cposes).any(axis=1))
    assert bi == cbest and bs == scores[bi] and np.array_equal(bp, poses[bi])
    assert rounds[bi] == len(trips)
    return bp, bi, bs, scores, poses, rounds


@pytest.mark.parametrize("method", [P2PLANE, P2P, NDT])
def test_one_round_equals_relocalise(scene, method):
    hyp = hypotheses(scene)
    reg = handle(scene, method, 4)
    bp, bi, bs, scores, poses = reg.Relocalise(scene.scan, hyp, want_all=True)
    sp, si, ss, sscores, sposes, rounds = reg.RelocaliseStaged(scene.scan, hyp, (4,), None, want_all=True)
    assert np.array_equal(sscores, scores) and np.array_equal(sposes, poses)
    assert (si, ss) == (bi, bs) and np.array_equal(sp, bp)
    assert np.all(rounds == 1)
    assert np.isfinite(scores).any()


@pytest.mark.parametrize("eps", [0.0, 1e-2])
def test_no_cut_equals_the_chain(scene, eps):
    n = len(hypotheses(scene))
    _, _, _, _, _, rounds = assert_equals_chain(scene, P2PLANE, (2, 3, 5), (n, 10 * n), eps=eps)
    assert np.all(rounds == 3)


@pytest.mark.parametrize("method", [P2PLANE, NDT])
def test_cuts_equal_the_chain(scene, method):
    _, _, _, scores, _, rounds = assert_equals_chain(scene, method, (1, 2, 3), (16, 4))
    assert [int((rounds == r).sum()) for r in (1, 2, 3)] == [len(rounds) - 16, 12, 4]


def test_zero_initial_translation_applies_in_round_0_only(scene):
    hyp = hypotheses(scene)[:24]
    reg = handle(scene, P2PLANE, 9, zero_t=True)
    _, bi, _, scores, poses, rounds = reg.RelocaliseStaged(scene.scan, hyp, (2, 3), (6,), want_all=True)
    # round 0 on a handle with the flag, round 1 on one without it
    cbest, cscores, cposes, crounds, _ = chain(lambda t: handle(scene, P2PLANE, t, zero_t=(t == 2)), scene.scan, hyp, (2, 3), (6,))
    assert np.array_equal(rounds, crounds) and np.array_equal(scores, cscores) and np.array_equal(poses, cposes)
    assert bi == cbest


def test_a_tie_at_the_cut_goes_to_the_lower_index(scene):
    hyp = hypotheses(scene)
    _, _, _, s0, _ = handle(scene, P2PLANE, 1).Relocalise(scene.scan, hyp, want_all=True)
    keep = 10
    order = np.lexsort((np.arange(len(hyp)), np.float32(s0)))
    last_in = int(order[keep - 1])  # the last survivor of a cut at `keep`
    assert np.float32(s0[order[keep - 1]]) != np.float32(s0[order[keep]])
    dup = np.concatenate([hyp, hyp[last_in][None]])  # the same hypothesis at the highest index straddles the cut
    _, _, _, scores, _, rounds = assert_equals_chain(scene, P2PLANE, (1, 2), (keep,), hyp=dup)
    assert scores[-1] == s0[last_in] and rounds[last_in] == 2 and rounds[-1] == 1


def test_an_all_inf_round_keeps_the_lowest_indices(scene):
    hyp = hypotheses(scene)[:20].copy()
    hyp[:, 4:] += 1000.0  # every hypothesis outside the map: no inlier anywhere
    bp, bi, bs, scores, poses, rounds = assert_equals_chain(scene, P2PLANE, (1, 1), (5,), hyp=hyp)
    assert np.all(np.isinf(scores))
    assert np.array_equal(np.flatnonzero(rounds == 2), np.arange(5))
    assert bi == 0 and bs == np.inf


def test_edge_cases(scene):
    hyp = hypotheses(scene)
    # one round without keep
    assert_equals_chain(scene, P2PLANE, (3,), None)
    # keep == 1: a single finalist, which wins
    _, bi, _, _, _, rounds = assert_equals_chain(scene, P2PLANE, (1, 2), (1,))
    assert np.flatnonzero(rounds == 2).tolist() == [bi]
    # a score-only round first, and a score-only last round
    assert_equals_chain(scene, P2PLANE, (0, 2), (8,))
    assert_equals_chain(scene, P2PLANE, (2, 0), (8,))
    # a single hypothesis runs every round
    _, bi, _, _, _, rounds = assert_equals_chain(scene, P2PLANE, (1, 2, 3), (4, 4), hyp=hyp[17:18])
    assert bi == 0 and rounds.tolist() == [3]
    # keep larger than the alive set
    _, _, _, _, _, rounds = assert_equals_chain(scene, P2PLANE, (1, 1, 1), (100, 3))
    assert int((rounds == 3).sum()) == 3 and int((rounds == 2).sum()) == len(hyp) - 3


_WAVES = r"""
import sys
import numpy as np
sys.path[:0] = [{root!r}, {tests!r}]
from conftest import Scene
from test_gpu_reloc_staged import handle, hypotheses
scene = Scene()
reg = handle(scene, "p2plane", 7)
bp, bi, bs, scores, poses, rounds = reg.RelocaliseStaged(scene.scan, hypotheses(scene), (1, 2, 3), (16, 4), want_all=True)
np.savez({out!r}, bp=bp, bi=bi, bs=bs, scores=scores, poses=poses, rounds=rounds, launches=reg.last_timing()[1])
reg.close()
"""


def test_waves_agree_bit_for_bit(scene, tmp_path):
    """LOCREG_RELOC_WAVE_GIB is read once per process: a subprocess runs every round in waves of a few hypotheses."""
    reg = handle(scene, P2PLANE, 7)
    bp, bi, bs, scores, poses, rounds = reg.RelocaliseStaged(scene.scan, hypotheses(scene), (1, 2, 3), (16, 4), want_all=True)
    launches = reg.last_timing()[1]
    out = str(tmp_path / "waves.npz")
    env = dict(os.environ, LOCREG_RELOC_WAVE_GIB="0.0005")
    code = _WAVES.format(root=ROOT, tests=os.path.join(ROOT, "tests"), out=out)
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    w = np.load(out)
    assert int(w["bi"]) == bi and float(w["bs"]) == bs and np.array_equal(w["bp"], bp)
    assert np.array_equal(w["scores"], scores) and np.array_equal(w["poses"], poses) and np.array_equal(w["rounds"], rounds)
    assert int(w["launches"]) > 2 * launches  # several waves per round really ran


def test_argument_errors(scene):
    import loc_lib_b200 as L
    from loc_lib_b200 import _lib
    a = np.ascontiguousarray(scene.scan[:1024, :4], np.float32)
    hyp = np.stack([IDENTITY, IDENTITY, IDENTITY])
    bp, bs = np.zeros(7), np.zeros(1)
    bi = np.zeros(1, np.int64)
    t3 = np.array([1, 1, 1], np.int32)
    k2 = np.array([2, 1], np.int64)
    ptr = lambda x: None if x is None else x.ctypes.data  # noqa: E731

    def call(reg, src=a, n=1024, stride=16, pin=hyp, n_hyp=3, trips=t3, keep=k2, n_rounds=3):
        rc = _lib.lib().locreg_relocalise_staged(None if reg is None else reg._h, ptr(src), n, stride, ptr(pin), n_hyp,
                                                 ptr(trips), ptr(keep), n_rounds, ptr(bp), ptr(bi), ptr(bs), None, None, None)
        return rc, _lib.lib().locreg_last_error()

    fresh = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE))
    rc, err = call(fresh)
    assert rc == -3 and b"SetInputTarget" in err
    reg = handle(scene, P2PLANE, 3)
    assert call(reg)[0] == 0
    assert call(None) == (-1, b"null handle")
    assert call(reg, src=None)[0] == -1 and call(reg, stride=8)[0] == -1 and call(reg, stride=18)[0] == -1
    assert call(reg, src=None, n=0)[0] == 0  # an empty scan may come as a null pointer
    for bad in ({"pin": None}, {"n_hyp": 0}, {"n_hyp": 1 << 31}):
        rc, err = call(reg, **bad)
        assert rc == -1 and b"invalid hypotheses" in err, bad
    for n_rounds in (0, 33):
        rc, err = call(reg, n_rounds=n_rounds)
        assert rc == -1 and b"n_rounds" in err
    for bad in ({"trips": None}, {"trips": np.array([1, -2, 1], np.int32)}):
        rc, err = call(reg, **bad)
        assert rc == -1 and b"trips" in err, bad
    for bad in ({"keep": None}, {"keep": np.array([0, 1], np.int64)}, {"keep": np.array([2, -1], np.int64)}):
        rc, err = call(reg, **bad)
        assert rc == -1 and b"keep" in err, bad
    assert call(reg, keep=None, n_rounds=1)[0] == 0
    # the refusals changed nothing on the device: the handle still works
    assert call(reg)[0] == 0


def test_the_handle_is_unchanged_afterwards(scene):
    hyp = hypotheses(scene)
    for zero_t in (False, True):
        reg = handle(scene, P2PLANE, 5, zero_t=zero_t)
        before = reg.Relocalise(scene.scan, hyp, want_all=True)
        single = reg.ScanMatch(scene.scan, scene.init[0], want_cloud=False)[2]
        reg.RelocaliseStaged(scene.scan, hyp, (0, 2, 9), (20, 5))
        after = reg.Relocalise(scene.scan, hyp, want_all=True)
        assert before[1:3] == after[1:3] and np.array_equal(before[0], after[0])
        assert np.array_equal(before[3], after[3]) and np.array_equal(before[4], after[4])
        assert np.array_equal(single, reg.ScanMatch(scene.scan, scene.init[0], want_cloud=False)[2])
        ms, launches = reg.last_timing()
        assert ms > 0 and launches > 0


def test_a_cut_schedule_reaches_the_truth_as_the_exhaustive_run_does(scene):
    """The staged winner, like the exhaustive one with 10 trips, is at the truth within test_relocalise's tolerance.
    Several hypotheses of this scene converge onto the truth, so which of them wins can differ between the two (each
    round restarts its loop unseeded): the winners are compared as places, not as indices."""
    hyp = hypotheses(scene)
    ebp, ebi, ebs, _, _ = handle(scene, P2PLANE, 10).Relocalise(scene.scan, hyp)
    bp, bi, bs, _, _, rounds = handle(scene, P2PLANE, 7).RelocaliseStaged(scene.scan, hyp, (2, 3, 5), (16, 4), want_all=True)
    assert rounds[bi] == 3 and np.isfinite(bs)
    for pose in (bp, ebp):
        dr, dt = pose_delta(pose, scene.gt[0])
        assert dr < 5e-3 and dt < 0.05, (bi, ebi, dr, dt)
