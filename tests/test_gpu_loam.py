"""GPU tests of locreg_align_loam / LoamRegistration: the LOAM loop against the oracle's loop, against the host loop it
replaces (two CaculateMatrixHAndB calls per trip), its edges, argument errors, and the two handles staying usable."""
import ctypes as C

import numpy as np
import pytest

import oracle_py as O
from conftest import pose_delta
from loam_cases import KatScene, host_loop, oracle_loam_align, rot_diff

pytestmark = pytest.mark.gpu


def make(max_iteration=10, eps=0.0, max_line_distance=0.5, loop_mode=None):
    import loc_lib_b200 as L
    kw = {} if loop_mode is None else {"loop_mode": loop_mode}
    so = L.IcpOptions(method_=L.IcpMethod.P2PLANE, max_iteration_=max_iteration, eps_=eps, **kw)
    eo = L.IcpOptions(method_=L.IcpMethod.P2LINE, max_iteration_=max_iteration, eps_=eps,
                      max_line_distance_=max_line_distance, **kw)
    return L.LoamRegistration(so, eo, max_iteration=max_iteration, eps=eps)


def oracle_pair(surf_map, edge_map, max_line_distance=0.5):
    surf = O.OracleIcp(method=O.P2PLANE, nn_mode=O.NN_EXACT_TIEBREAK, skip_nonfinite=1)
    edge = O.OracleIcp(method=O.P2LINE, nn_mode=O.NN_EXACT_TIEBREAK, skip_nonfinite=1, max_line_distance=max_line_distance)
    surf.set_target(surf_map)
    edge.set_target(edge_map)
    return surf, edge


def scene_case(scene):
    return scene.map, scene.map, scene.scan[0::2], scene.scan[1::2], scene.init[0]


def kat_case():
    k = KatScene()
    return k.surf_map, k.edge_map, k.surf, k.edge, k.init


@pytest.mark.parametrize("case", ["scene", "kat"])
def test_parity_with_the_oracle(scene, case):
    surf_map, edge_map, surf, edge, init = scene_case(scene) if case == "scene" else kat_case()
    loam = make()
    loam.SetInputTarget(surf_map, edge_map)
    pose, (g0, g1) = loam.ScanMatch(surf, edge, init)
    rpose, (r0, r1) = oracle_loam_align(*oracle_pair(surf_map, edge_map), surf, edge, init, 10, 0.0)
    assert r0["n_inlier"] > 0 and r1["n_inlier"] > 0
    assert (g0["iters"], g0["updates"]) == (r0["iters"], r0["updates"]) == (g1["iters"], g1["updates"])
    for g, r in ((g0, r0), (g1, r1)):
        assert (g["n_inlier"], g["n_effective"], g["degenerate"]) == (r["n_inlier"], r["n_effective"], r["degenerate"])
    dr, dt = pose_delta(pose, rpose)
    assert dr < 1e-5 and dt < 1e-4, (dr, dt)
    ms, launches = loam.last_timing()
    assert ms > 0 and launches > 10


@pytest.mark.parametrize("eps", [0.0, 1e-3])
def test_equals_the_host_loop_over_compute_hb(scene, eps):
    loam = make(eps=eps)
    loam.SetInputTarget(scene.map, scene.map)
    surf, edge, init = scene.scan[0::2], scene.scan[1::2], scene.init[0]
    pose, (g0, _) = loam.ScanMatch(surf, edge, init)
    hpose, h = host_loop(loam.surf, loam.edge, surf, edge, init, 10, eps)
    assert (g0["iters"], g0["updates"], g0["converged"]) == (h["iters"], h["updates"], h["converged"])
    assert rot_diff(pose, hpose) < 1e-9 and np.linalg.norm(pose[4:] - hpose[4:]) < 1e-8


def test_loop_edges(scene):
    import loc_lib_b200 as L
    surf, edge, init = scene.scan[0::2], scene.scan[1::2], scene.init[0]
    empty = np.zeros((0, 4), np.float32)
    loam = make()
    loam.SetInputTarget(scene.map, scene.map)
    loam.max_iteration = 0
    pose, (g0, _) = loam.ScanMatch(surf, edge, init)
    assert np.array_equal(pose, init) and g0["iters"] == 0 and g0["pose_written"] == 1
    loam.max_iteration, loam.eps = 10, 1e3
    _, (g0, g1) = loam.ScanMatch(surf, edge, init)
    assert g0["converged"] == 1 and g0["iters"] < 10 and g1["converged"] == 1
    loam.eps = 0.0
    pose, (g0, _) = loam.ScanMatch(empty, empty, init)
    assert g0["updates"] == 0 and g0["iters"] == 10 and np.array_equal(pose, init)
    # an empty edge half: the P2Plane ScanMatch of the surf cloud on its own
    pose, (g0, g1) = loam.ScanMatch(surf, empty, init)
    assert (g1["n_effective"], g1["n_inlier"], g1["degenerate"]) == (0, 0, 1)
    icp = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE, max_iteration_=10, eps_=0.0, loop_mode=L.LOOP_GRAPH))
    icp.SetInputTarget(scene.map)
    _, _, ipose = icp.ScanMatch(surf, init, want_cloud=False)
    assert rot_diff(pose, ipose) < 1e-9 and np.linalg.norm(pose[4:] - ipose[4:]) < 1e-9
    assert (g0["iters"], g0["updates"]) == (icp.last_result["iters"], icp.last_result["updates"])


def test_argument_errors(scene):
    import loc_lib_b200 as L
    from loc_lib_b200 import _lib
    a = np.ascontiguousarray(scene.scan[:512], np.float32)
    p = np.array([0, 0, 0, 1, 0, 0, 0], np.float64)
    out = np.zeros(7)

    def call(s, e):
        return _lib.lib().locreg_align_loam(s._h, e._h, a.ctypes.data, a.shape[0], a.ctypes.data, a.shape[0],
                                            a.shape[1] * 4, p.ctypes.data, 5, 0.0, out.ctypes.data, None)

    plane = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE))
    line = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2LINE))
    assert call(plane, line) == -3  # no target yet
    assert b"surf handle" in _lib.lib().locreg_last_error()
    plane.SetInputTarget(scene.map)
    assert call(plane, line) == -3
    assert b"edge handle" in _lib.lib().locreg_last_error()
    line.SetInputTarget(scene.map)
    assert call(plane, line) == 0
    assert call(plane, plane) == -1 and call(line, line) == -1
    assert call(line, plane) == -1
    p2p = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2P))
    ndt = L.NdtRegistration(L.NdtOptions())
    p2p.SetInputTarget(scene.map)
    ndt.SetInputTarget(scene.map)
    assert call(p2p, line) == -1 and call(plane, p2p) == -1 and call(plane, ndt) == -1 and call(ndt, line) == -1
    assert _lib.lib().locreg_align_loam(plane._h, line._h, a.ctypes.data, a.shape[0], a.ctypes.data, a.shape[0], 8,
                                        p.ctypes.data, 5, 0.0, out.ctypes.data, None) == -1  # stride < 12
    assert _lib.lib().locreg_align_loam(plane._h, line._h, a.ctypes.data, a.shape[0], a.ctypes.data, a.shape[0], 16,
                                        None, 5, 0.0, out.ctypes.data, None) == -1


def test_handles_stay_usable(scene):
    loam = make()
    loam.SetInputTarget(scene.map, scene.map)
    surf, edge, init = scene.scan[0::2], scene.scan[1::2], scene.init[0]
    before = [loam.surf.ScanMatch(surf, init)[2], loam.edge.ScanMatch(edge, init)[2]]
    loam.ScanMatch(surf, edge, init)
    after = [loam.surf.ScanMatch(surf, init)[2], loam.edge.ScanMatch(edge, init)[2]]
    assert np.array_equal(before[0], after[0]) and np.array_equal(before[1], after[1])
    # and a LOAM call after them is what it was
    p1, _ = loam.ScanMatch(surf, edge, init)
    p2, _ = loam.ScanMatch(surf, edge, init)
    assert np.array_equal(p1, p2)


def test_one_caller_stream_equals_two_streams(scene):
    import torch
    loam = make()
    loam.SetInputTarget(scene.map, scene.map)
    surf, edge, init = scene.scan[0::2], scene.scan[1::2], scene.init[0]
    p_two, r_two = loam.ScanMatch(surf, edge, init)
    s = torch.cuda.Stream()
    loam.surf.set_stream(s.cuda_stream)
    loam.edge.set_stream(s.cuda_stream)
    p_one, r_one = loam.ScanMatch(surf, edge, init)
    loam.surf.set_stream(0)
    loam.edge.set_stream(0)
    assert np.array_equal(p_one, p_two) and r_one == r_two
