"""CPU tests of the LOAM loop (LoamRegistration::ScanMatch, SURVEY.md 3.3): the contract over the oracle, and the C ABI /
Python / C++ entry points failing loudly without a GPU."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle_py as O
from conftest import HAS_GPU, ROOT, pose_delta
from loam_cases import KatScene, oracle_loam_align, xyz


def oracles(max_line_distance=0.5):
    surf = O.OracleIcp(method=O.P2PLANE, nn_mode=O.NN_EXACT_TIEBREAK, skip_nonfinite=1)
    edge = O.OracleIcp(method=O.P2LINE, nn_mode=O.NN_EXACT_TIEBREAK, skip_nonfinite=1, max_line_distance=max_line_distance)
    return surf, edge


def rank(H):
    s = np.linalg.svd(H, compute_uv=False)
    return int(np.sum(s > 1e-9 * s.max()))


def test_kat_neither_half_alone_the_sum_recovers_the_pose():
    k = KatScene()
    surf, edge = oracles()
    surf.set_target(k.surf_map)
    edge.set_target(k.edge_map)
    _, Hs, _, rs, _, _ = surf.compute_hb(xyz(k.surf), k.truth, False, False)
    _, He, _, re, _, _ = edge.compute_hb(xyz(k.edge), k.truth, False, False)
    assert rs["n_inlier"] > 100 and re["n_inlier"] > 50
    assert rank(Hs) < 6 and rank(He) < 6
    assert np.linalg.matrix_rank(Hs + He) == 6
    pose, (r0, r1) = oracle_loam_align(surf, edge, k.surf, k.edge, k.init, 10, 1e-8)
    dr, dt = pose_delta(pose, k.truth)
    assert dr < 1e-3 and dt < 1e-3, (dr, dt, r0)
    assert r0["updates"] >= 2 and (r0["iters"], r0["updates"], r0["converged"]) == (r1["iters"], r1["updates"], r1["converged"])


def test_empty_edge_half_is_the_p2plane_loop_bit_for_bit(scene):
    for max_iteration, eps in ((10, 0.0), (20, 1e-2)):
        surf, edge = oracles()
        ref = O.OracleIcp(method=O.P2PLANE, nn_mode=O.NN_EXACT_TIEBREAK, skip_nonfinite=1, max_iteration=max_iteration,
                          eps=eps)
        for o in (surf, edge, ref):
            o.set_target(scene.map)
        pose, (r0, r1) = oracle_loam_align(surf, edge, scene.scan, np.zeros((0, 3), np.float32), scene.init[0],
                                           max_iteration, eps)
        rpose, _, rres, _ = ref.align(xyz(scene.scan), scene.init[0], want_cloud=False)
        assert rres["degenerate"] == 0 and rres["n_effective"] >= ref.opt.min_effective_pts
        assert np.array_equal(pose, rpose)
        assert (r0["iters"], r0["updates"], r0["converged"]) == (rres["iters"], rres["updates"], rres["converged"])
        assert (r0["n_effective"], r0["n_inlier"]) == (rres["n_effective"], rres["n_inlier"])
        assert (r1["n_effective"], r1["n_inlier"]) == (0, 0)


def test_both_halves_empty_and_zero_iterations():
    k = KatScene()
    surf, edge = oracles()
    surf.set_target(k.surf_map)
    edge.set_target(k.edge_map)
    empty = np.zeros((0, 3), np.float32)
    pose, (r0, _) = oracle_loam_align(surf, edge, empty, empty, k.truth, 5, 0.0)
    assert np.array_equal(pose, k.truth) and (r0["iters"], r0["updates"]) == (5, 0)
    pose, (r0, _) = oracle_loam_align(surf, edge, k.surf, k.edge, k.truth, 0, 0.0)
    assert np.array_equal(pose, k.truth) and r0["iters"] == 0


@pytest.mark.skipif(HAS_GPU, reason="checks the no-device behaviour")
def test_entry_points_fail_loudly_without_a_device():
    from loc_lib_b200 import _lib
    import loc_lib_b200 as L
    p = np.array([0, 0, 0, 1, 0, 0, 0], np.float64)
    out = np.zeros(7)
    assert _lib.lib().locreg_align_loam(None, None, None, 0, None, 0, 16, p.ctypes.data, 10, 0.0, out.ctypes.data,
                                        None) == -1
    assert b"null handle" in _lib.lib().locreg_last_error()
    with pytest.raises(_lib.LocregError, match="no CPU fallback"):
        L.LoamRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE), L.IcpOptions(method_=L.IcpMethod.P2LINE))


def test_python_class_checks_the_halves_methods():
    from loc_lib_b200 import _lib
    import loc_lib_b200 as L
    with pytest.raises(_lib.LocregError, match="P2PLANE options for the surf half"):
        L.LoamRegistration(L.IcpOptions(method_=L.IcpMethod.P2LINE), L.IcpOptions(method_=L.IcpMethod.P2LINE))
    with pytest.raises(_lib.LocregError, match="P2LINE options for the edge half"):
        L.LoamRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE), L.IcpOptions(method_=L.IcpMethod.P2P))


def test_loam_standin_builds_and_links():
    exe = os.path.join(ROOT, "tests", "loam", "_build", "loam_standin")
    assert os.path.exists(exe)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == (0 if HAS_GPU else 3), r.stdout + r.stderr
