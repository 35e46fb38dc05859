"""GPU tests of locreg_align_loam_batch / LoamRegistration.ScanMatchBatch: every scan of a batch bit for bit what its own
ScanMatch call gives (small and large jobs, mixed and empty halves, early stops), parity with the oracle's LOAM loop,
argument errors, the handles staying usable, and one caller stream for both handles."""
import numpy as np
import pytest

import oracle_py as O
from conftest import GPU_COUNT, pose_delta
from loam_cases import KatScene, oracle_loam_align, pose_from_rpy_t

pytestmark = pytest.mark.gpu

IDENTITY = np.array([0, 0, 0, 1, 0, 0, 0], np.float64)


def make(max_iteration=10, eps=0.0, device=0):
    import loc_lib_b200 as L
    so = L.IcpOptions(method_=L.IcpMethod.P2PLANE, max_iteration_=max_iteration, eps_=eps)
    eo = L.IcpOptions(method_=L.IcpMethod.P2LINE, max_iteration_=max_iteration, eps_=eps, max_line_distance_=0.5)
    return L.LoamRegistration(so, eo, max_iteration=max_iteration, eps=eps, device=device)


def concat(clouds):
    """(cloud, offsets) of a list of (n, 4) clouds."""
    offs = np.concatenate([[0], np.cumsum([c.shape[0] for c in clouds])]).astype(np.int64)
    cloud = np.concatenate(clouds) if clouds else np.zeros((0, 4), np.float32)
    return np.ascontiguousarray(cloud, np.float32), offs


def run_batch(loam, pairs, inits):
    surf, so = concat([p[0] for p in pairs])
    edge, eo = concat([p[1] for p in pairs])
    return loam.ScanMatchBatch(surf, so, edge, eo, np.asarray(inits))


def assert_equals_single_calls(loam, pairs, inits):
    poses, res = run_batch(loam, pairs, inits)
    assert poses.shape == (len(pairs), 7) and len(res) == len(pairs)
    for s, ((a, b), init) in enumerate(zip(pairs, inits)):
        pose, r = loam.ScanMatch(a, b, init)
        assert np.array_equal(poses[s], pose), (s, poses[s], pose)
        assert res[s] == r, (s, res[s], r)
    return poses, res


def scene_pairs(scene):
    return [(sc[0::2], sc[1::2]) for sc in scene.scans]


def num_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def test_equal_to_single_calls_small_and_large_jobs(scene):
    from loc_lib_b200 import synth
    loam = make()
    loam.SetInputTarget(scene.map, scene.map)
    assert_equals_single_calls(loam, scene_pairs(scene), scene.init)
    ms, launches = loam.last_timing()
    assert ms > 0 and launches > 10
    # 32 scans: the surf half is a large job (more than 2 x SM-count tiles of 256 points)
    pairs = [scene_pairs(scene)[i % 4] for i in range(32)]
    inits = [synth.perturb_pose(scene.gt[i % 4], 1000 + i) for i in range(32)]
    assert sum(p[0].shape[0] for p in pairs) > 2 * num_sms() * 256
    _, res = assert_equals_single_calls(loam, pairs, inits)
    assert all(r[0]["n_inlier"] > 0 and r[1]["n_inlier"] > 0 for r in res)


def oracle_pair(surf_map, edge_map):
    surf = O.OracleIcp(method=O.P2PLANE, nn_mode=O.NN_EXACT_TIEBREAK, skip_nonfinite=1)
    edge = O.OracleIcp(method=O.P2LINE, nn_mode=O.NN_EXACT_TIEBREAK, skip_nonfinite=1, max_line_distance=0.5)
    surf.set_target(surf_map)
    edge.set_target(edge_map)
    return surf, edge


def assert_oracle_parity(surf_map, edge_map, pairs, inits, poses, res):
    surf, edge = oracle_pair(surf_map, edge_map)
    for (a, b), init, pose, (g0, g1) in zip(pairs, inits, poses, res):
        rpose, (r0, r1) = oracle_loam_align(surf, edge, a, b, init, 10, 0.0)
        assert r0["n_inlier"] > 0 and r1["n_inlier"] > 0
        assert (g0["iters"], g0["updates"]) == (r0["iters"], r0["updates"]) == (g1["iters"], g1["updates"])
        for g, r in ((g0, r0), (g1, r1)):
            assert (g["n_inlier"], g["n_effective"], g["degenerate"]) == (r["n_inlier"], r["n_effective"], r["degenerate"])
        dr, dt = pose_delta(pose, rpose)
        assert dr < 1e-5 and dt < 1e-4, (dr, dt)


def test_parity_with_the_oracle_loop(scene):
    loam = make()
    loam.SetInputTarget(scene.map, scene.map)
    pairs = scene_pairs(scene)
    poses, res = run_batch(loam, pairs, scene.init)
    assert_oracle_parity(scene.map, scene.map, pairs, scene.init, poses, res)
    # KatScene has its own surf and edge targets: its scan from two initial poses
    k = KatScene()
    kat = make()
    kat.SetInputTarget(k.surf_map, k.edge_map)
    pairs = [(k.surf, k.edge)] * 2
    inits = [k.init, pose_from_rpy_t([0.005, 0.0, -0.01], [0.02, 0.01, 0.0])]
    poses, res = run_batch(kat, pairs, inits)
    assert_oracle_parity(k.surf_map, k.edge_map, pairs, inits, poses, res)


def test_mixed_batch_empty_halves_and_early_stops(scene):
    empty = np.zeros((0, 4), np.float32)
    loam = make(eps=1e-2)
    loam.SetInputTarget(scene.map, scene.map)
    sp = scene_pairs(scene)
    pairs = [sp[0], (sp[1][0], empty), sp[2], (empty, sp[3][1]), (empty, empty), sp[3]]
    inits = [scene.init[0], scene.init[1], scene.init[2], scene.init[3], scene.init[0], scene.init[3]]
    poses, res = assert_equals_single_calls(loam, pairs, inits)
    iters = [r[0]["iters"] for r in res]
    assert len(set(iters)) > 1, iters  # the scans stop at different trips
    assert np.array_equal(poses[4], inits[4]) and res[4][0]["updates"] == 0 and res[4][0]["iters"] == 10
    assert (res[1][1]["n_effective"], res[1][1]["n_inlier"], res[1][1]["degenerate"]) == (0, 0, 1)
    assert (res[3][0]["n_effective"], res[3][0]["n_inlier"], res[3][0]["degenerate"]) == (0, 0, 1)
    # no edge point in the whole batch
    assert_equals_single_calls(loam, [(p[0], empty) for p in sp], scene.init)
    # nor any surf point
    assert_equals_single_calls(loam, [(empty, p[1]) for p in sp], scene.init)
    # max_iteration = 0: the poses come back as given
    loam.max_iteration = 0
    poses, res = assert_equals_single_calls(loam, sp, scene.init)
    assert np.array_equal(poses, np.asarray(scene.init))
    assert all(r[0]["iters"] == 0 and r[0]["pose_written"] == 1 for r in res)


def test_argument_errors(scene):
    import loc_lib_b200 as L
    from loc_lib_b200 import _lib
    a = np.ascontiguousarray(scene.scan[:1024], np.float32)
    offs = np.array([0, 512, 1024], np.int64)
    p = np.stack([IDENTITY, IDENTITY])
    out = np.zeros((2, 7))

    def call(s, e, S=2, so=offs, eo=offs, stride=16, surf_xyz=a, edge_xyz=a, pin=p, pout=out):
        ptr = lambda x: None if x is None else x.ctypes.data  # noqa: E731
        h = lambda r: None if r is None else r._h  # noqa: E731
        return _lib.lib().locreg_align_loam_batch(h(s), h(e), ptr(surf_xyz), ptr(so), ptr(edge_xyz), ptr(eo), stride, ptr(pin),
                                                  S, 5, 0.0, ptr(pout), None)

    def err():
        return _lib.lib().locreg_last_error()

    plane = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE))
    line = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2LINE))
    assert call(plane, line) == -3 and b"surf handle" in err()  # no target yet
    plane.SetInputTarget(scene.map)
    assert call(plane, line) == -3 and b"edge handle" in err()
    line.SetInputTarget(scene.map)
    assert call(plane, line) == 0
    assert call(None, line) == -1 and b"null handle" in err()
    assert call(plane, None) == -1 and b"null handle" in err()
    assert call(plane, plane) == -1 and call(line, line) == -1
    assert call(line, plane) == -1
    p2p = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2P))
    ndt = L.NdtRegistration(L.NdtOptions())
    p2p.SetInputTarget(scene.map)
    ndt.SetInputTarget(scene.map)
    assert call(p2p, line) == -1 and call(plane, p2p) == -1 and call(plane, ndt) == -1 and call(ndt, line) == -1
    if GPU_COUNT > 1:
        other = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2LINE), device=1)
        other.SetInputTarget(scene.map)
        assert call(plane, other) == -1 and b"different devices" in err()
    for half in ("surf", "edge"):
        for bad in ([-1, 512, 1024], [0, 600, 512]):
            kw = {"so" if half == "surf" else "eo": np.array(bad, np.int64)}
            assert call(plane, line, **kw) == -1, (half, bad)
            assert f"{half} offsets".encode() in err()
        assert call(plane, line, **{"so" if half == "surf" else "eo": None}) == -1
        assert call(plane, line, **{"surf_xyz" if half == "surf" else "edge_xyz": None}) == -1
    assert call(plane, line, stride=8) == -1 and call(plane, line, stride=18) == -1
    assert call(plane, line, pin=None) == -1 and call(plane, line, pout=None) == -1
    assert call(plane, line, S=1 << 31) == -1 and b"too many scans" in err()
    # S == 0: nothing happens, poses_out stays as it was
    sentinel = np.full((2, 7), 7.0)
    assert call(plane, line, S=0, pout=sentinel) == 0 and np.all(sentinel == 7.0)
    # an empty cloud may come as a null pointer
    z = np.zeros(3, np.int64)
    assert call(plane, line, eo=z, edge_xyz=None) == 0


def test_handles_stay_usable(scene):
    loam = make()
    loam.SetInputTarget(scene.map, scene.map)
    surf, edge, init = scene.scan[0::2], scene.scan[1::2], scene.init[0]

    def singles():
        return [loam.ScanMatch(surf, edge, init), loam.surf.ScanMatch(surf, init)[2], loam.edge.ScanMatch(edge, init)[2]]

    before = singles()
    b1 = run_batch(loam, scene_pairs(scene), scene.init)
    after = singles()
    assert np.array_equal(before[0][0], after[0][0]) and before[0][1] == after[0][1]
    assert np.array_equal(before[1], after[1]) and np.array_equal(before[2], after[2])
    b2 = run_batch(loam, scene_pairs(scene), scene.init)
    assert np.array_equal(b1[0], b2[0]) and b1[1] == b2[1]


def test_one_caller_stream_equals_two_streams(scene):
    import torch
    loam = make()
    loam.SetInputTarget(scene.map, scene.map)
    two = run_batch(loam, scene_pairs(scene), scene.init)
    s = torch.cuda.Stream()
    loam.surf.set_stream(s.cuda_stream)
    loam.edge.set_stream(s.cuda_stream)
    one = run_batch(loam, scene_pairs(scene), scene.init)
    loam.surf.set_stream(0)
    loam.edge.set_stream(0)
    assert np.array_equal(one[0], two[0]) and one[1] == two[1]
