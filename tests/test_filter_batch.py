"""CPU tests of the batch pre-filters and of batch ScanMatch from raw scans: the entry points are exported, a null
handle is refused before any device work, and without a device the calls fail loudly (there is no CPU fallback)."""
import ctypes as C

import numpy as np
import pytest

from conftest import HAS_GPU

NEW = ("locreg_filter_remove_nan_batch", "locreg_filter_voxel_grid_batch", "locreg_align_batch_filtered")


def test_new_symbols_are_exported_and_bound():
    from loc_lib_b200 import _lib
    for name in NEW:
        assert name in _lib.SYMBOLS
        assert getattr(_lib.lib(), name).argtypes is not None


def test_null_handle_is_refused_and_nothing_is_written():
    from loc_lib_b200 import _lib
    L = _lib.lib()
    cloud = np.zeros((6, 4), np.float32)
    offs = np.array([0, 2, 6], np.int64)
    out = np.full((6, 4), 7.0, np.float32)
    oo = np.full(3, -5, np.int64)
    assert L.locreg_filter_remove_nan_batch(None, cloud.ctypes.data, offs.ctypes.data, 2, 16, out.ctypes.data, oo.ctypes.data) == -1
    assert b"null handle" in L.locreg_last_error()
    assert L.locreg_filter_voxel_grid_batch(None, cloud.ctypes.data, offs.ctypes.data, 2, 16, C.c_float(1.0), out.ctypes.data,
                                            oo.ctypes.data) == -1
    assert b"null handle" in L.locreg_last_error()
    pin = np.tile(np.array([0, 0, 0, 1, 0, 0, 0], np.float64), (2, 1))
    pout = np.full((2, 7), 3.0)
    nf = np.full(2, -9, np.int64)
    assert L.locreg_align_batch_filtered(None, cloud.ctypes.data, offs.ctypes.data, 16, pin.ctypes.data, 2, C.c_float(1.0),
                                         pout.ctypes.data, None, nf.ctypes.data) == -1
    assert b"null handle" in L.locreg_last_error()
    assert np.all(out == 7.0) and np.all(oo == -5) and np.all(pout == 3.0) and np.all(nf == -9)


def test_argument_errors_come_before_the_handle():
    from loc_lib_b200 import _lib
    L = _lib.lib()
    cloud = np.zeros((6, 4), np.float32)
    bad = np.array([0, 4, 2], np.int64)
    oo = np.zeros(3, np.int64)
    assert L.locreg_filter_voxel_grid_batch(None, cloud.ctypes.data, bad.ctypes.data, 2, 16, C.c_float(1.0), cloud.ctypes.data,
                                            oo.ctypes.data) == -1
    assert b"non-decreasing" in L.locreg_last_error()
    good = np.array([0, 2, 6], np.int64)
    assert L.locreg_filter_voxel_grid_batch(None, cloud.ctypes.data, good.ctypes.data, 2, 16, C.c_float(0.0), cloud.ctypes.data,
                                            oo.ctypes.data) == -1
    assert b"leaf" in L.locreg_last_error()


@pytest.mark.skipif(HAS_GPU, reason="checks the no-device behaviour")
def test_batch_filters_fail_loudly_without_a_device():
    from loc_lib_b200 import _lib
    import loc_lib_b200 as L
    cloud = np.zeros((4, 4), np.float32)
    with pytest.raises(_lib.LocregError):
        reg = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE))
        reg.VoxelFilterBatch(cloud, [0, 4], 1.0)
    with pytest.raises(_lib.LocregError):
        reg = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE))
        reg.ScanMatchBatchFiltered(cloud, [0, 4], np.array([[0, 0, 0, 1, 0, 0, 0]], np.float64), 1.0)
