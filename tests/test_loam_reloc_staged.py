"""CPU tests of locreg_relocalise_loam_staged[_sharded] / LoamRegistration.RelocaliseStaged[Sharded]: the symbols are
bound, the null-handle and argument refusals run before any device work (with the messages of locreg_relocalise_loam
and locreg_relocalise_staged), and the entry points fail loudly without a device."""
import numpy as np
import pytest

from conftest import HAS_GPU

IDENTITY = np.array([0, 0, 0, 1, 0, 0, 0], np.float64)
SYMBOLS = ("locreg_relocalise_loam_staged", "locreg_relocalise_loam_staged_sharded")


def call(symbol, surf=None, edge=None, surf_xyz=None, n_surf=0, edge_xyz=None, n_edge=0, stride=16, pin=None, n_hyp=1,
         trips=None, keep=None, n_rounds=1, eps=0.0):
    from loc_lib_b200 import _lib
    ptr = lambda x: None if x is None else x.ctypes.data  # noqa: E731
    bp, bs = np.zeros(7), np.zeros(1)
    bi = np.zeros(1, np.int64)
    rc = getattr(_lib.lib(), symbol)(surf, edge, ptr(surf_xyz), n_surf, ptr(edge_xyz), n_edge, stride, ptr(pin), n_hyp,
                                     ptr(trips), ptr(keep), n_rounds, eps, ptr(bp), ptr(bi), ptr(bs), None, None, None)
    return rc, _lib.lib().locreg_last_error()


def test_symbols_are_bound():
    from loc_lib_b200 import _lib
    for s in SYMBOLS:
        assert s in _lib.SYMBOLS
        assert getattr(_lib.lib(), s).argtypes is not None


@pytest.mark.parametrize("symbol", SYMBOLS)
def test_null_handles_are_refused_before_any_device_work(symbol):
    trips = np.array([2, 3], np.int32)
    keep = np.array([4], np.int64)
    rc, err = call(symbol, pin=IDENTITY, trips=trips, keep=keep, n_rounds=2)
    assert rc == -1 and b"null handle" in err


@pytest.mark.parametrize("symbol", SYMBOLS)
def test_the_handle_check_comes_before_the_other_argument_checks(symbol):
    """Only the handle check is covered here: without a device no handle can be created, so every case has null
    handles, and whatever else is wrong the call refuses with "null handle" before any device work.  The cloud,
    hypothesis and schedule refusals and their messages are covered with real handles in
    test_gpu_loam_reloc_staged.py::test_argument_errors."""
    cloud = np.zeros((4, 4), np.float32)
    hyp = np.stack([IDENTITY] * 3)
    t3 = np.array([1, 2, 3], np.int32)
    k2 = np.array([2, 1], np.int64)
    ok = dict(surf_xyz=cloud, n_surf=4, edge_xyz=cloud, n_edge=4, pin=hyp, n_hyp=3, trips=t3, keep=k2, n_rounds=3)
    for bad in ({}, {"surf_xyz": None}, {"edge_xyz": None}, {"stride": 8}, {"pin": None}, {"n_hyp": 0},
                {"n_rounds": 0}, {"n_rounds": 33}, {"trips": None}, {"keep": None},
                {"keep": np.array([0, 1], np.int64)}):
        rc, err = call(symbol, **{**ok, **bad})
        assert rc == -1 and b"null handle" in err, bad


def test_python_checks_the_length_of_keep():
    import loc_lib_b200 as L
    loam = L.LoamRegistration.__new__(L.LoamRegistration)  # no handles: the length check comes first
    empty = np.zeros((4, 4), np.float32)
    for method in (loam.RelocaliseStaged, loam.RelocaliseStagedSharded):
        with pytest.raises(ValueError, match="keep"):
            method(empty, empty, IDENTITY, (2, 3), (4, 2))
        with pytest.raises(ValueError, match="keep"):
            method(empty, empty, IDENTITY, (2, 3), None)


@pytest.mark.skipif(HAS_GPU, reason="checks the no-device behaviour")
def test_relocalise_loam_staged_fails_loudly_without_a_device():
    from loc_lib_b200 import _lib
    import loc_lib_b200 as L
    empty = np.zeros((0, 4), np.float32)
    for staged in ("RelocaliseStaged", "RelocaliseStagedSharded"):
        with pytest.raises(_lib.LocregError, match=r"locreg error -2: .*no CPU fallback"):  # LOCREG_E_CUDA
            loam = L.LoamRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE), L.IcpOptions(method_=L.IcpMethod.P2LINE))
            getattr(loam, staged)(empty, empty, IDENTITY, (2,), None)
