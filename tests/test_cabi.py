"""CPU tests of the drop-in boundary: liblocreg.so loads, exports every symbol include/locreg.h declares, mirrors the
reference's option defaults, validates arguments, and FAILS LOUDLY without a GPU (no CPU fallback).  No compute calls."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from conftest import HAS_GPU, ROOT

HEADER = os.path.join(ROOT, "include", "locreg.h")


def declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(locreg_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_exported():
    from loc_lib_b200 import _lib
    L = _lib.lib()
    names = declared_symbols()
    assert len(names) >= 20
    for n in names:
        assert hasattr(L, n), f"liblocreg.so does not export {n}"
    assert sorted(_lib.SYMBOLS) == names  # the ctypes binding covers the whole header
    out = subprocess.run(["nm", "-D", "--defined-only", os.path.join(ROOT, "loc_lib_b200", "liblocreg.so")],
                         capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (locreg_\w+)", out))
    assert exported == set(names)  # nothing undeclared leaks out of the C ABI either


def test_library_is_sm100a_and_self_contained():
    so = os.path.join(ROOT, "loc_lib_b200", "liblocreg.so")
    # the CUDA tools need not be on PATH: fall back to the toolkit of the nvcc csrc/Makefile builds with
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cuobjdump = shutil.which("cuobjdump") or os.path.join(os.path.dirname(nvcc), "cuobjdump")
    out = subprocess.run([cuobjdump, "-lelf", so], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    needed = subprocess.run(["readelf", "-d", so], capture_output=True, text=True).stdout
    assert "liboracle" not in needed and "hostsim" not in needed  # the product never links test infrastructure
    assert "libtorch" not in needed  # plain C ABI: no torch types behind the boundary


def test_struct_layouts_match_header():
    from loc_lib_b200 import _lib
    # locreg_options: 4 x i32, 6 x f64, 2 x i32, f64, 4 x i32 ; locreg_result: 48 bytes (kernels write it verbatim)
    assert C.sizeof(_lib.Options) == 16 + 48 + 8 + 8 + 8 + 8
    assert C.sizeof(_lib.Result) == 48
    assert _lib.Options.eps.offset == 16 and _lib.Options.knn_cell_size.offset == 72
    assert _lib.Result.n_effective.offset == 16 and _lib.Result.pose_written.offset == 40


def test_default_options_mirror_reference():
    """IcpOptions (icp_registration.hpp:22-39) and NdtOptions (ndt_registration.hpp:27-42) defaults."""
    from loc_lib_b200 import _lib
    import loc_lib_b200 as L
    o = _lib.Options()
    assert _lib.lib().locreg_default_options(C.byref(o), _lib.ICP_P2PLANE) == 0
    assert (o.max_iteration, o.min_effective_pts, o.eps) == (20, 10, 1e-2)
    assert (o.max_nn_distance, o.max_plane_distance, o.max_line_distance) == (1.0, 0.1, 0.5)
    assert (o.voxel_size, o.res_outlier_th, o.min_pts_in_voxel, o.nearby_type) == (1.0, 20.0, 3, _lib.NEARBY6)
    assert _lib.lib().locreg_default_options(None, 0) == -1
    i, n = L.IcpOptions(), L.NdtOptions()
    assert (i.max_iteration_, i.max_nn_distance_, i.max_plane_distance_, i.min_effective_pts_, i.eps_, i.use_ann) == \
        (20, 1.0, 0.1, 10, 1e-2, False)
    assert i.method_ == L.IcpMethod.P2P  # the reference's default method (icp_registration.hpp:38)
    assert (n.max_iteration_, n.voxel_size_, n.min_pts_in_voxel_, n.res_outlier_th_, n.nearby_type_) == \
        (20, 1.0, 3, 20.0, L.NdtNearbyType.NEARBY6)
    assert (L.IcpMethod.P2P, L.IcpMethod.P2LINE, L.IcpMethod.P2PLANE, L.IcpMethod.PCLICP) == (0, 1, 2, 3)


def test_pack_score_orders_like_score_then_index():
    from loc_lib_b200 import _lib
    from loc_lib_b200 import dist
    f = _lib.lib().locreg_pack_score
    rng = np.random.default_rng(0)
    sc = np.concatenate([rng.uniform(0, 10, 200), [0.0, 1.0, 1.0, np.inf, np.nan, -1.0]])
    idx = rng.integers(0, 2 ** 32 - 1, len(sc))
    keys = [f(float(s), int(i)) for s, i in zip(sc, idx)]
    assert keys == [dist.pack_score(s, i) for s, i in zip(sc, idx)]  # host-side helper is bit-identical
    clean = [np.float32(s) if (s == s and s >= 0) else np.float32(np.inf) for s in sc]
    order = sorted(range(len(sc)), key=lambda j: (clean[j], idx[j]))
    assert sorted(range(len(sc)), key=lambda j: keys[j]) == order
    assert max(keys) < 2 ** 63  # fits the signed int64 that torch.distributed reduces
    s, i = dist.unpack_score(f(2.5, 77))
    assert (s, i) == (2.5, 77)


def test_argument_validation_needs_no_gpu():
    from loc_lib_b200 import _lib
    L = _lib.lib()
    o = _lib.Options()
    L.locreg_default_options(C.byref(o), _lib.ICP_P2LINE)
    h = C.c_void_p()
    o.method = 17
    assert L.locreg_create(C.byref(o), 0, C.byref(h)) == -1
    assert L.locreg_create(None, 0, C.byref(h)) == -1
    assert L.locreg_align(None, None, 0, 16, None, None, None, None) == -1
    assert L.locreg_destroy(None) == 0
    assert L.locreg_version().startswith(b"locreg-b200")


@pytest.mark.skipif(HAS_GPU, reason="checks the behaviour of a box WITHOUT a CUDA device")
def test_no_cpu_fallback():
    """Every computing entry point needs a handle, and a handle cannot be created without a B200."""
    from loc_lib_b200 import _lib
    import loc_lib_b200 as L
    o = _lib.Options()
    _lib.lib().locreg_default_options(C.byref(o), _lib.ICP_P2PLANE)
    h = C.c_void_p()
    assert _lib.lib().locreg_create(C.byref(o), 0, C.byref(h)) == -2  # LOCREG_E_CUDA
    assert b"no CPU fallback" in _lib.lib().locreg_last_error()
    with pytest.raises(_lib.LocregError):
        L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE))
    with pytest.raises(_lib.LocregError):
        L.NdtRegistration()


def test_product_never_imports_oracle():
    """Only tests/, __graft_entry__.smoke() and bench.py's CPU legs may touch oracle/ or tests/hostsim."""
    pkg = os.path.join(ROOT, "loc_lib_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h", "Makefile")):
                text = open(os.path.join(dirpath, f), errors="replace").read()
                assert "oracle_py" not in text and "liboracle" not in text and "hostsim_py" not in text, f
                assert not re.search(r'#include\s+"[^"]*oracle', text), f


def _run_adapter():
    exe = os.path.join(ROOT, "tests", "cpp", "_build", "adapter_standin")
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "tests", "cpp")])
    return subprocess.run([exe], capture_output=True, text=True)


@pytest.mark.skipif(HAS_GPU, reason="checks the behaviour of a box WITHOUT a CUDA device")
def test_cpp_adapter_compiles_and_refuses_without_gpu():
    """include/locreg_adapter.hpp (the MatchingInterface drop-in) builds against stand-in PCL/Sophus types and,
    without a GPU, raises instead of computing on the CPU."""
    r = _run_adapter()
    assert r.returncode == 3, r.stdout + r.stderr
    assert "no CPU fallback" in r.stdout


@pytest.mark.gpu
def test_cpp_adapter_scan_match_on_gpu():
    """The same binary on the B200: SetInputTarget + ScanMatch through the virtual interface recover a known shift."""
    r = _run_adapter()
    assert r.returncode == 0, r.stdout + r.stderr


def test_se3_helpers_of_the_loc_slice():
    """predict = result * last^-1 * result (loc.cpp:232) on 7-double poses, against 4x4 matrices."""
    import loc_lib_b200 as L
    import oracle_py as O
    rng = np.random.default_rng(0)

    def rand_pose():
        q = rng.normal(size=4)
        return np.concatenate([q / np.linalg.norm(q), rng.uniform(-5, 5, 3)])

    def mat(p):
        T = np.eye(4)
        T[:3, :3] = O.pose_matrix(p)
        T[:3, 3] = p[4:]
        return T

    for _ in range(20):
        a, b = rand_pose(), rand_pose()
        assert np.allclose(mat(L.se3_mul(a, b)), mat(a) @ mat(b), atol=1e-13)
        assert np.allclose(mat(L.se3_inv(a)), np.linalg.inv(mat(a)), atol=1e-13)
        pred = L.se3_mul(L.se3_mul(a, L.se3_inv(b)), a)
        assert np.allclose(mat(pred), mat(a) @ np.linalg.inv(mat(b)) @ mat(a), atol=1e-12)


def test_lio_keyframe_criterion():
    """Lio::IsKeyframe (lio.cpp:616-623): |t| of last_kf^-1 * pose above kf_distance, or |log R| above kf_angle_deg."""
    import loc_lib_b200 as L
    from loc_lib_b200.registration import LioTracker, se3_log_angle

    class NoDevice:  # IsKeyframe touches no registration call
        def ClearLocalMap(self):
            pass

    def rot_z(deg, t=(0.0, 0.0, 0.0)):
        h = np.deg2rad(deg) / 2
        return np.array([0, 0, np.sin(h), np.cos(h), *t], np.float64)

    for deg in (0.0, 3.0, 9.9, 45.0, 179.0, -30.0):
        assert abs(se3_log_angle(rot_z(deg)) - abs(np.deg2rad(deg))) < 1e-12
    q = rot_z(30.0)
    assert abs(se3_log_angle(-q) - np.deg2rad(30.0)) < 1e-12  # q and -q are the same rotation
    base = rot_z(40.0, (10.0, -3.0, 1.0))
    trk = LioTracker(NoDevice(), init_pose=base, kf_distance=1.0, kf_angle_deg=10.0)
    assert not trk.IsKeyframe(base)
    assert not trk.IsKeyframe(L.se3_mul(base, rot_z(9.0, (0.9, 0.0, 0.0))))
    assert trk.IsKeyframe(L.se3_mul(base, rot_z(0.0, (0.8, 0.7, 0.0))))   # 1.06 m
    assert trk.IsKeyframe(L.se3_mul(base, rot_z(11.0)))                   # 11 degrees on the spot
