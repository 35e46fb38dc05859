"""GPU tests of locreg_align_loam_batch_sharded / LoamRegistration.ScanMatchBatchSharded against their contract: every
rank's poses and results are bit for bit what ScanMatchBatch of the whole batch returns on one GPU.  Covers a world of
one (without a communicator and with a one-rank one: the same launches as ScanMatchBatch), a batch that mixes empty
surf halves, empty edge halves and early stops, every argument error (nothing written, the handles unchanged), ranks
with no scan (ragged blocks, S_global < world) on 2, 4 and 8 ranks sharing one GPU or on one GPU each, and the plain
C++ host of tests/cpp/loam_sharded_host.cpp."""
import multiprocessing as mp
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import GPU_COUNT, ROOT

pytestmark = pytest.mark.gpu

IDENTITY = np.array([0, 0, 0, 1, 0, 0, 0], np.float64)
EMPTY = np.zeros((0, 4), np.float32)
MIXED_SCAN = [0, 1, 2, 3, 0, 3]  # the scene scan each entry of mixed_batch cuts


@pytest.fixture(scope="module", autouse=True)
def _torch_first():
    """torch is imported before the first sharded call loads NCCL: liblocreg.so then binds the NCCL torch brought
    (nccl_dyn.h), which a later torch import needs, instead of the system's."""
    import torch  # noqa: F401


def make(max_iteration=10, eps=1e-2, device=0):
    import loc_lib_b200 as L
    so = L.IcpOptions(method_=L.IcpMethod.P2PLANE, max_iteration_=max_iteration, eps_=eps)
    eo = L.IcpOptions(method_=L.IcpMethod.P2LINE, max_iteration_=max_iteration, eps_=eps, max_line_distance_=0.5)
    return L.LoamRegistration(so, eo, max_iteration=max_iteration, eps=eps, device=device)


def concat(clouds):
    """(cloud, offsets) of a list of (n, 4) clouds."""
    offs = np.concatenate([[0], np.cumsum([c.shape[0] for c in clouds])]).astype(np.int64)
    cloud = np.concatenate(clouds) if clouds else np.zeros((0, 4), np.float32)
    return np.ascontiguousarray(cloud, np.float32), offs


def mixed_batch(scene, S=6):
    """S scans cycling through test_gpu_loam_batch's mixed batch: both halves, no edge half, both, no surf half, no
    point at all, both; with eps = 1e-2 the scans stop at different trips.  Entries past the sixth start from poses of
    their own."""
    from loc_lib_b200 import synth
    sp = [(sc[0::2], sc[1::2]) for sc in scene.scans]
    pattern = [sp[0], (sp[1][0], EMPTY), sp[2], (EMPTY, sp[3][1]), (EMPTY, EMPTY), sp[3]]
    pairs = [pattern[i % 6] for i in range(S)]
    inits = [scene.init[MIXED_SCAN[i]] if i < 6 else synth.perturb_pose(scene.gt[MIXED_SCAN[i % 6]], 2000 + i) for i in range(S)]
    return pairs, np.stack(inits)


def block(pairs, inits, rank, world):
    """This rank's block of a batch: (surf, surf offsets, edge, edge offsets, poses), offsets relative to its clouds."""
    from loc_lib_b200.dist import shard_range
    lo, hi = shard_range(len(pairs), rank, world)
    surf, so = concat([p[0] for p in pairs[lo:hi]])
    edge, eo = concat([p[1] for p in pairs[lo:hi]])
    return surf, so, edge, eo, inits[lo:hi]


def whole_batch(loam, pairs, inits):
    surf, so = concat([p[0] for p in pairs])
    edge, eo = concat([p[1] for p in pairs])
    return loam.ScanMatchBatch(surf, so, edge, eo, inits)


def assert_same(got, want, what):
    poses, res = got
    wposes, wres = want
    assert poses.shape == wposes.shape and np.array_equal(poses, wposes), (what, np.flatnonzero((poses != wposes).any(axis=1)))
    assert res == wres, what


def test_world_of_one_is_scan_match_batch(scene):
    loam = make()
    loam.SetInputTarget(scene.map, scene.map)
    pairs, inits = mixed_batch(scene)
    want = whole_batch(loam, pairs, inits)
    launches = loam.last_timing()[1]
    iters = [r[0]["iters"] for r in want[1]]
    assert len(set(iters)) > 1, iters  # early stops
    assert want[1][1][1]["n_effective"] == 0 and want[1][3][0]["n_effective"] == 0  # empty edge half, empty surf half
    surf, so, edge, eo, pin = block(pairs, inits, 0, 1)
    for comm in (False, True):
        if comm:
            loam.CommInit(loam.CommUniqueId(), 0, 1)
            assert loam.CommInfo()[:2] == (0, 1)
        try:
            got = loam.ScanMatchBatchSharded(surf, so, edge, eo, pin, len(pairs))
            assert_same(got, want, comm)
            ms, n = loam.last_timing()
            assert ms > 0 and n == launches, (comm, n, launches)  # the same launch sequence, no exchange
        finally:
            if comm:
                loam.CommDestroy()
    # eps = 0: every scan runs every trip
    loam.eps = 0.0
    assert_same(loam.ScanMatchBatchSharded(surf, so, edge, eo, pin, len(pairs)), whole_batch(loam, pairs, inits), "eps 0")
    loam.close()


def test_argument_errors_write_nothing_and_leave_the_handles_as_they_were(scene):
    import loc_lib_b200 as L
    from loc_lib_b200 import _lib
    lib = _lib.lib()
    a = np.ascontiguousarray(scene.scan[:1024], np.float32)
    offs = np.array([0, 512, 1024], np.int64)
    p = np.stack([IDENTITY, IDENTITY])
    ptr = lambda x: None if x is None else x.ctypes.data  # noqa: E731
    h = lambda r: None if r is None else r._h  # noqa: E731

    def call(s, e, S_local=2, S_global=2, so=offs, eo=offs, surf_xyz=a, edge_xyz=a, stride=16, pin=p, null_pout=False):
        """(return code, last error, poses_out untouched)"""
        out = np.full((2, 7), 7.0)
        rc = lib.locreg_align_loam_batch_sharded(h(s), h(e), ptr(surf_xyz), ptr(so), ptr(edge_xyz), ptr(eo), stride, ptr(pin),
                                                 S_local, S_global, 5, 0.0, None if null_pout else out.ctypes.data, None)
        return rc, lib.locreg_last_error(), bool(np.all(out == 7.0))

    plane = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE))
    line = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2LINE))
    rc, err, untouched = call(plane, line)
    assert rc == -3 and b"surf handle" in err and untouched  # no target yet
    plane.SetInputTarget(scene.map)
    rc, err, untouched = call(plane, line)
    assert rc == -3 and b"edge handle" in err and untouched
    plane.close()
    line.close()

    loam = make()
    loam.SetInputTarget(scene.map, scene.map)
    surf, edge, init = scene.scan[0::2], scene.scan[1::2], scene.init[0]
    before = loam.ScanMatch(surf, edge, init)
    s, e = loam.surf, loam.edge
    p2p = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2P))
    ndt = L.NdtRegistration(L.NdtOptions())
    p2p.SetInputTarget(scene.map)
    ndt.SetInputTarget(scene.map)
    bad = [((None, e), {}, b"null handle"), ((s, None), {}, b"null handle"),
           ((s, s), {}, b"two distinct handles"), ((e, e), {}, b"two distinct handles"),
           ((e, s), {}, b"P2PLANE surf"), ((p2p, e), {}, b"P2PLANE surf"), ((s, p2p), {}, b"P2PLANE surf"),
           ((s, ndt), {}, b"P2PLANE surf"), ((ndt, e), {}, b"P2PLANE surf"),
           ((s, e), {"S_local": 1}, b"S_local"), ((s, e), {"S_local": 3}, b"S_local"),
           ((s, e), {"S_global": 0}, b"S_local"), ((s, e), {"S_global": 1 << 31}, b"too many scans"),
           ((s, e), {"so": np.array([-1, 512, 1024], np.int64)}, b"surf offsets"),
           ((s, e), {"so": np.array([0, 600, 512], np.int64)}, b"surf offsets"),
           ((s, e), {"eo": np.array([-1, 512, 1024], np.int64)}, b"edge offsets"),
           ((s, e), {"eo": np.array([0, 600, 512], np.int64)}, b"edge offsets"),
           ((s, e), {"so": None}, b"null argument"), ((s, e), {"eo": None}, b"null argument"),
           ((s, e), {"surf_xyz": None}, b"invalid cloud"), ((s, e), {"edge_xyz": None}, b"invalid cloud"),
           ((s, e), {"stride": 8}, b"invalid cloud"), ((s, e), {"stride": 18}, b"invalid cloud"),
           ((s, e), {"pin": None}, b"null pose"), ((s, e), {"null_pout": True}, b"null pose")]
    for (hs, he), kw, msg in bad:
        rc, err, untouched = call(hs, he, **kw)
        assert rc == -1 and msg in err and untouched, (kw, rc, err)
    # S_global == 0: nothing happens, whatever the block's pointers
    for kw in ({}, {"so": None, "eo": None, "surf_xyz": None, "edge_xyz": None, "pin": None}):
        rc, _, untouched = call(s, e, S_local=0, S_global=0, **kw)
        assert rc == 0 and untouched, kw
    # the refusals changed nothing on the device: the pair gives the same ScanMatch, and a valid call works
    after = loam.ScanMatch(surf, edge, init)
    assert np.array_equal(before[0], after[0]) and before[1] == after[1]
    rc, _, untouched = call(s, e)
    assert rc == 0 and not untouched
    for reg in (p2p, ndt, loam):
        reg.close()


# Ranks that share one GPU: NCCL refuses two ranks of one host on one device, so each rank names a host of its own
# (NCCL_HOSTID) and the ranks talk over loopback sockets (as tests/test_gpu_loam_reloc_staged.py does).
def _shared_gpu_env(rank):
    return {"NCCL_HOSTID": "locreg-test-rank-%d" % rank, "NCCL_SOCKET_IFNAME": "lo", "NCCL_NET": "Socket",
            "NCCL_IB_DISABLE": "1", "NCCL_MNNVL_ENABLE": "0"}


# (S_global, eps) per case: every S_global leaves the blocks ragged, and those below the number of ranks leave ranks
# with no scan
TWO_RANK_CASES = [(7, 1e-2), (1, 1e-2), (5, 0.0)]
FOUR_RANK_CASES = [(13, 1e-2), (3, 1e-2)]
EIGHT_RANK_CASES = [(5, 1e-2), (13, 1e-2)]


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
        for S, eps in cases:
            pairs, inits = mixed_batch(scene, S)
            loam.eps = eps
            surf, so, edge, eo, pin = block(pairs, inits, rank, world)
            outs.append(loam.ScanMatchBatchSharded(surf, so, edge, eo, pin, S))
        loam.CommDestroy()
        loam.close()
        q.put((rank, outs, None))
    except Exception as e:  # noqa: BLE001 - reported to the parent, which fails the test with it
        q.put((rank, None, repr(e)))


def run_ranks(scene, world, cases, shared=False):
    """Every case on `world` spawned ranks (one GPU each, or all on GPU 0 with `shared`); every rank's poses and results
    must equal ScanMatchBatch of the whole batch on one GPU."""
    loam = make()
    loam.SetInputTarget(scene.map, scene.map)
    want = []
    for S, eps in cases:
        loam.eps = eps
        want.append(whole_batch(loam, *mixed_batch(scene, S)))
    loam.close()
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
    for rank, got, err in outs:
        assert err is None, (rank, err)
        for case, g, w in zip(cases, got, want):
            assert_same(g, w, (rank, case))
    return want


def test_two_ranks_sharing_one_gpu_agree_with_one_gpu(scene):
    want = run_ranks(scene, 2, TWO_RANK_CASES, shared=True)
    assert len({r[0]["iters"] for r in want[0][1]}) > 1  # early stops in the batch


def test_four_ranks_sharing_one_gpu_agree_with_one_gpu(scene):
    run_ranks(scene, 4, FOUR_RANK_CASES, shared=True)


def test_eight_ranks_sharing_one_gpu_agree_with_one_gpu(scene):
    run_ranks(scene, 8, EIGHT_RANK_CASES, shared=True)


@pytest.mark.skipif(GPU_COUNT < 2, reason="needs two GPUs")
def test_two_ranks_agree_with_one_gpu(scene):
    run_ranks(scene, 2, TWO_RANK_CASES)


@pytest.mark.skipif(GPU_COUNT < 4, reason="needs four GPUs")
def test_four_ranks_agree_with_one_gpu(scene):
    run_ranks(scene, 4, FOUR_RANK_CASES)


def test_cpp_host_runs_the_sharded_loam_batch(tmp_path):
    """tests/cpp/loam_sharded_host.cpp: one host thread per GPU, no Python / torch in the process.  Built by its own
    makefile into a temporary directory."""
    subprocess.check_call(["make", "-s", "-f", os.path.join(ROOT, "tests", "cpp", "loam_sharded_host.mk"), "OUT=%s" % tmp_path])
    r = subprocess.run([str(tmp_path / "loam_sharded_host"), str(min(GPU_COUNT, 4))],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert ": ok" in r.stdout, r.stdout
