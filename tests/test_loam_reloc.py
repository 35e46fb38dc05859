"""CPU tests of locreg_relocalise_loam / LoamRegistration.Relocalise: argument checks that need no device, and the
Python entry point failing loudly without one."""
import numpy as np
import pytest

from conftest import HAS_GPU


def test_null_handles_are_refused_before_any_device_work():
    from loc_lib_b200 import _lib
    hyp = np.array([0, 0, 0, 1, 0, 0, 0], np.float64)
    best_pose, best_score = np.zeros(7), np.zeros(1)
    best_idx = np.zeros(1, np.int64)
    args = [None, None, None, 0, None, 0, 16, hyp.ctypes.data, 1, 10, 0.0, best_pose.ctypes.data, best_idx.ctypes.data,
            best_score.ctypes.data]
    assert _lib.lib().locreg_relocalise_loam(*args, None, None) == -1
    assert b"null handle" in _lib.lib().locreg_last_error()
    assert _lib.lib().locreg_relocalise_loam_sharded(*args) == -1
    assert b"null handle" in _lib.lib().locreg_last_error()


@pytest.mark.skipif(HAS_GPU, reason="checks the no-device behaviour")
def test_relocalise_fails_loudly_without_a_device():
    from loc_lib_b200 import _lib
    import loc_lib_b200 as L
    empty = np.zeros((0, 4), np.float32)
    with pytest.raises(_lib.LocregError, match="no CPU fallback"):
        loam = L.LoamRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE), L.IcpOptions(method_=L.IcpMethod.P2LINE))
        loam.Relocalise(empty, empty, np.array([[0, 0, 0, 1, 0, 0, 0]], np.float64))
