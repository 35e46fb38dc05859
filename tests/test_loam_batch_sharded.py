"""CPU tests of locreg_align_loam_batch_sharded / LoamRegistration.ScanMatchBatchSharded: the null-handle refusal that
needs no device, and the Python entry point failing loudly without one."""
import numpy as np
import pytest

from conftest import HAS_GPU


def test_null_handles_are_refused_before_any_device_work():
    from loc_lib_b200 import _lib
    p = np.array([0, 0, 0, 1, 0, 0, 0], np.float64)
    out = np.full(7, 7.0)
    offs = np.zeros(2, np.int64)
    assert _lib.lib().locreg_align_loam_batch_sharded(None, None, None, offs.ctypes.data, None, offs.ctypes.data, 16,
                                                      p.ctypes.data, 1, 1, 10, 0.0, out.ctypes.data, None) == -1
    assert b"null handle" in _lib.lib().locreg_last_error()
    assert np.all(out == 7.0)


@pytest.mark.skipif(HAS_GPU, reason="checks the no-device behaviour")
def test_scan_match_batch_sharded_fails_loudly_without_a_device():
    from loc_lib_b200 import _lib
    import loc_lib_b200 as L
    empty = np.zeros((0, 4), np.float32)
    with pytest.raises(_lib.LocregError, match="no CPU fallback"):
        loam = L.LoamRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE), L.IcpOptions(method_=L.IcpMethod.P2LINE))
        loam.ScanMatchBatchSharded(empty, [0, 0], empty, [0, 0], np.array([[0, 0, 0, 1, 0, 0, 0]], np.float64), 1)
