"""GPU tests of the batch pre-filters (locreg_filter_remove_nan_batch / locreg_filter_voxel_grid_batch) and of batch
ScanMatch from raw scans (locreg_align_batch_filtered): every segment byte for byte the single-cloud filter and the
oracle, waves that change nothing, launches that do not grow with the batch, bit-identical registration of the
filtered batch, and argument errors that write nothing."""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_py as O

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LEAVES = (0.5, 1.0)


def concat(clouds, width):
    offs = np.concatenate([[0], np.cumsum([len(c) for c in clouds])]).astype(np.int64)
    cloud = np.concatenate(clouds) if clouds else np.zeros((0, width), np.float32)
    return np.ascontiguousarray(cloud, np.float32), offs


def widen(xyzt, width, rng):
    """(n, width) float32 cloud: x, y, z, then every other word filled (PointXYZI is 32 B: x y z pad i pad pad pad)."""
    out = np.zeros((len(xyzt), width), np.float32)
    out[:, :3] = xyzt[:, :3]
    out[:, 3:] = rng.random((len(xyzt), width - 3), dtype=np.float32) * 100
    return out


def mixed_scans(scene, width):
    """About a dozen scans: the scene's scans and subsamples with NaN / inf sprinkled in, an empty scan, an all-NaN scan,
    a scan with a far outlier (~3e8 voxels at 0.5 m), one whose int voxel index would overflow, one with exact
    duplicate points."""
    rng = np.random.default_rng(31 + width)
    base = [scene.scans[0], scene.scans[1], scene.scans[2][::3], scene.scans[3][1::2], scene.scans[1][::5]]
    scans = []
    for sc in base:
        c = widen(sc, width, rng)
        c[rng.integers(0, len(c), len(c) // 40), 1] = np.nan
        c[rng.integers(0, len(c), 3), 0] = np.inf
        c[rng.integers(0, len(c), 3), 2] = -np.inf
        scans.append(c)
    scans.insert(2, np.zeros((0, width), np.float32))
    all_nan = widen(scene.scans[2][:50], width, rng)
    all_nan[:, 0] = np.nan
    scans.insert(4, all_nan)
    far = widen(scene.scans[0][::2], width, rng)
    far[7, :3] = [600.0, -550.0, 40.0]
    scans.append(far)
    over = widen(scene.scans[3][::4], width, rng)
    over[3, :3] = [9000.0, -9000.0, 900.0]
    over[11, 1] = np.nan  # the unfiltered cloud comes back with its NaN
    scans.append(over)
    dup = widen(scene.scans[1][:1500], width, rng)
    scans.append(np.concatenate([dup, dup[::-1], dup[:300]]))
    scans.append(widen(scene.scans[2][::7], width, rng))
    return scans


@pytest.fixture(scope="module")
def icp(scene):
    import loc_lib_b200 as L
    reg = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE, max_iteration_=6, eps_=0.0))
    reg.SetInputTarget(scene.map)
    return reg


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def check_segments(out, offs, expected):
    lens = [len(e) for e in expected]
    assert np.array_equal(offs, np.concatenate([[0], np.cumsum(lens)])), (offs, lens)
    assert len(out) == offs[-1]
    for s, e in enumerate(expected):
        seg = out[offs[s]:offs[s + 1]]
        assert seg.shape == e.shape and np.array_equal(bits(seg), bits(e)), s


@pytest.mark.parametrize("width", [8, 4])
def test_batch_segments_equal_single_calls_and_oracle(scene, icp, width):
    scans = mixed_scans(scene, width)
    cloud, offs = concat(scans, width)
    # RemoveNanPoint
    out, oo = icp.RemoveNanPointBatch(cloud, offs)
    single = [icp.RemoveNanPoint(s) for s in scans]
    for s, sc in enumerate(scans):
        if len(sc):
            assert np.array_equal(bits(single[s]), bits(O.filter_remove_nan(sc))), s
    check_segments(out, oo, single)
    # VoxelFilter
    for leaf in LEAVES:
        out, oo = icp.VoxelFilterBatch(cloud, offs, leaf)
        single = [icp.VoxelFilter(s, leaf) for s in scans]
        for s, sc in enumerate(scans):
            if len(sc):
                assert np.array_equal(bits(single[s]), bits(O.filter_voxel_grid(sc, leaf))), (leaf, s)
        assert len(single[-3]) == len(scans[-3])  # the overflow scan comes back unfiltered
        assert len(single[4]) == 0 and len(single[2]) == 0
        check_segments(out, oo, single)
    # a batch of one scan, and offsets that do not start at the cloud's first point
    for sc in (scans[0], scans[-2]):
        out, oo = icp.VoxelFilterBatch(sc, [0, len(sc)], 1.0)
        check_segments(out, oo, [icp.VoxelFilter(sc, 1.0)])
        out, oo = icp.RemoveNanPointBatch(sc, [0, len(sc)])
        check_segments(out, oo, [icp.RemoveNanPoint(sc)])
    pre = np.concatenate([np.full((5, width), 123.0, np.float32), cloud])
    out, oo = icp.VoxelFilterBatch(pre, offs + 5, 0.5)
    check_segments(out, oo, [icp.VoxelFilter(s, 0.5) for s in scans])
    # only empty scans
    out, oo = icp.VoxelFilterBatch(np.zeros((0, width), np.float32), [0, 0, 0], 1.0)
    assert len(out) == 0 and np.array_equal(oo, [0, 0, 0])


_WAVES = r"""
import sys
import numpy as np
sys.path[:0] = [{root!r}, {tests!r}]
import loc_lib_b200 as L
reg = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE))
d = np.load({inp!r})
res = {{}}
for leaf in (0.5, 1.0):
    out, oo = reg.VoxelFilterBatch(d["cloud"], d["offs"], leaf)
    res["out%g" % leaf], res["oo%g" % leaf] = out, oo
res["launches"] = reg.last_timing()[1]
np.savez({out!r}, **res)
reg.close()
"""


def test_waves_change_nothing(scene, icp, tmp_path):
    """LOCREG_FILTER_WAVE_MIB is read once per process: a subprocess at its minimum runs every scan in a wave of its own."""
    scans = mixed_scans(scene, 8)
    cloud, offs = concat(scans, 8)
    inp, outp = str(tmp_path / "batch.npz"), str(tmp_path / "waves.npz")
    np.savez(inp, cloud=cloud, offs=offs)
    ref = {leaf: icp.VoxelFilterBatch(cloud, offs, leaf) for leaf in LEAVES}
    launches = icp.last_timing()[1]
    env = dict(os.environ, LOCREG_FILTER_WAVE_MIB="0")
    code = _WAVES.format(root=ROOT, tests=os.path.join(ROOT, "tests"), inp=inp, out=outp)
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    w = np.load(outp)
    for leaf in LEAVES:
        out, oo = ref[leaf]
        assert np.array_equal(w["oo%g" % leaf], oo)
        assert np.array_equal(bits(w["out%g" % leaf]), bits(out))
    assert int(w["launches"]) > launches  # it did run in more than one wave


def test_launches_do_not_grow_with_the_batch(scene, icp):
    """S = 8 and S = 256 copies of the same scans (one wave each): the same kernels, launched the same number of times."""
    rng = np.random.default_rng(3)
    base = [widen(s, 8, rng) for s in scene.scans]
    for s in base:
        s[::29, 2] = np.nan
    counts = {}
    for S in (8, 256):
        cloud, offs = concat([base[i % len(base)] for i in range(S)], 8)
        _, oo = icp.VoxelFilterBatch(cloud, offs, 1.0)
        vg = icp.last_timing()[1]
        _, on = icp.RemoveNanPointBatch(cloud, offs)
        counts[S] = (vg, icp.last_timing()[1])
        assert len(oo) == S + 1 and len(on) == S + 1
    assert counts[8] == counts[256], counts


def chain_batch(scene):
    """Raw PointXYZI scans with NaN rows, among them an all-NaN scan and one whose voxel index would overflow."""
    rng = np.random.default_rng(17)
    scans = []
    for i, sc in enumerate(scene.scans):
        c = widen(sc, 8, rng)
        c[rng.choice(len(c), len(c) // 10, replace=False), rng.integers(0, 3)] = np.nan
        scans.append(c)
    all_nan = widen(scene.scans[1][:64], 8, rng)
    all_nan[:, 2] = np.nan
    over = widen(scene.scans[2], 8, rng)
    over[5, :3] = [9000.0, -9000.0, 900.0]
    over[9, 0] = np.nan
    scans[1:1] = [all_nan]
    scans.append(over)
    poses = np.concatenate([scene.init, scene.init[:2]])
    return scans, poses


@pytest.mark.parametrize("method", ["p2plane", "p2p", "ndt"])
def test_scan_match_batch_filtered_equals_filter_then_batch(scene, method):
    import loc_lib_b200 as L
    if method == "ndt":
        reg = L.NdtRegistration(L.NdtOptions(max_iteration_=5, eps_=0.0))
    else:
        m = L.IcpMethod.P2PLANE if method == "p2plane" else L.IcpMethod.P2P
        reg = L.IcpRegistration(L.IcpOptions(method_=m, max_iteration_=6, eps_=0.0))
    reg.SetInputTarget(scene.map)
    scans, poses = chain_batch(scene)
    leaf = 1.0
    filtered = [reg.VoxelFilter(reg.RemoveNanPoint(s), leaf) for s in scans]
    fc, fo = concat(filtered, 8)
    ref_poses, ref_res = reg.ScanMatchBatch(fc, fo, poses)
    cloud, offs = concat(scans, 8)
    got_poses, got_res, n_filtered = reg.ScanMatchBatchFiltered(cloud, offs, poses, leaf)
    assert np.array_equal(n_filtered, [len(f) for f in filtered])
    assert n_filtered[1] == 0 and n_filtered[-1] == np.isfinite(scans[-1][:, :3]).all(1).sum()
    assert np.array_equal(got_poses, ref_poses)
    assert got_res == ref_res
    ms, launches = reg.last_timing()
    assert ms > 0 and launches > 0
    reg.close()


def test_argument_errors_write_nothing(scene, icp):
    import ctypes as C
    from loc_lib_b200 import _lib
    L = _lib.lib()
    h = icp._h
    scans, poses = chain_batch(scene)
    cloud, offs = concat(scans, 8)
    S = len(scans)
    bad = offs.copy()
    bad[2], bad[3] = bad[3], bad[2]
    out = np.full_like(cloud, 7.0)
    oo = np.full(S + 1, -5, np.int64)
    pout = np.full((S, 7), 3.0)
    nf = np.full(S, -9, np.int64)

    def unchanged():
        return np.all(out == 7.0) and np.all(oo == -5) and np.all(pout == 3.0) and np.all(nf == -9)

    p = cloud.ctypes.data
    for offsets, leaf, o, ooff in ((offs, 1.0, None, oo.ctypes.data), (offs, 1.0, out.ctypes.data, None),
                                   (bad, 1.0, out.ctypes.data, oo.ctypes.data), (offs, 0.0, out.ctypes.data, oo.ctypes.data),
                                   (offs, -1.0, out.ctypes.data, oo.ctypes.data)):
        assert L.locreg_filter_voxel_grid_batch(h, p, offsets.ctypes.data, S, 32, C.c_float(leaf), o, ooff) == -1
        if leaf > 0:
            assert L.locreg_filter_remove_nan_batch(h, p, offsets.ctypes.data, S, 32, o, ooff) == -1
        assert unchanged()
    pin = np.ascontiguousarray(poses)
    for offsets, leaf, po in ((offs, 1.0, None), (bad, 1.0, pout.ctypes.data), (offs, 0.0, pout.ctypes.data),
                              (offs, -2.0, pout.ctypes.data)):
        assert L.locreg_align_batch_filtered(h, p, offsets.ctypes.data, 32, pin.ctypes.data, S, C.c_float(leaf), po, None,
                                             nf.ctypes.data) == -1
        assert unchanged()
    assert L.locreg_align_batch_filtered(h, p, offs.ctypes.data, 32, None, S, C.c_float(1.0), pout.ctypes.data, None,
                                         nf.ctypes.data) == -1
    assert unchanged()
    # the handle still works
    _, oo2 = icp.VoxelFilterBatch(cloud, offs, 1.0)
    assert oo2[-1] > 0
