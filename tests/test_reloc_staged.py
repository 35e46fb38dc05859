"""CPU tests of locreg_relocalise_staged / RelocaliseStaged: the null-handle refusal, the argument checks that run before
any device work, the Python entry point failing loudly without a device, and the selection rule of the cut that the GPU
tests hold the device to."""
import numpy as np
import pytest

from conftest import HAS_GPU
from reloc_staged_cases import pack_order_scores, survivors

IDENTITY = np.array([0, 0, 0, 1, 0, 0, 0], np.float64)


def staged(h=None, src=None, n=0, stride=16, pin=None, n_hyp=1, trips=None, keep=None, n_rounds=1):
    from loc_lib_b200 import _lib
    ptr = lambda x: None if x is None else x.ctypes.data  # noqa: E731
    bp, bs = np.zeros(7), np.zeros(1)
    bi = np.zeros(1, np.int64)
    rc = _lib.lib().locreg_relocalise_staged(h, ptr(src), n, stride, ptr(pin), n_hyp, ptr(trips), ptr(keep), n_rounds,
                                             ptr(bp), ptr(bi), ptr(bs), None, None, None)
    return rc, _lib.lib().locreg_last_error()


def test_null_handle_is_refused_before_any_device_work():
    trips = np.array([2, 3], np.int32)
    keep = np.array([4], np.int64)
    rc, err = staged(pin=IDENTITY, trips=trips, keep=keep, n_rounds=2)
    assert rc == -1 and b"null handle" in err


def test_argument_errors_need_no_device():
    cloud = np.zeros((4, 4), np.float32)
    hyp = np.stack([IDENTITY] * 3)
    t1 = np.array([2], np.int32)
    t3 = np.array([1, 2, 3], np.int32)
    k2 = np.array([2, 1], np.int64)
    ok = dict(src=cloud, n=4, pin=hyp, n_hyp=3, trips=t3, keep=k2, n_rounds=3)
    rc, err = staged(**ok)  # every argument valid: only the handle is missing
    assert rc == -1 and b"null handle" in err
    rc, err = staged(**{**ok, "src": None})
    assert rc == -1 and b"cloud" in err
    assert staged(**{**ok, "stride": 8})[0] == -1 and staged(**{**ok, "stride": 18})[0] == -1
    for bad in ({"pin": None}, {"n_hyp": 0}, {"n_hyp": 1 << 31}):
        rc, err = staged(**{**ok, **bad})
        assert rc == -1 and b"invalid hypotheses" in err, bad
    for n_rounds in (0, -1, 33):
        rc, err = staged(**{**ok, "n_rounds": n_rounds})
        assert rc == -1 and b"n_rounds" in err, n_rounds
    rc, err = staged(**{**ok, "trips": None})
    assert rc == -1 and b"trips" in err
    rc, err = staged(**{**ok, "trips": np.array([1, -1, 3], np.int32)})
    assert rc == -1 and b"trips" in err
    rc, err = staged(**{**ok, "keep": None})
    assert rc == -1 and b"keep" in err
    for bad_keep in ([0, 1], [2, 0], [-5, 1]):
        rc, err = staged(**{**ok, "keep": np.array(bad_keep, np.int64)})
        assert rc == -1 and b"keep" in err, bad_keep
    # one round needs no keep; trips[r] == 0 and a keep beyond the alive set are valid
    rc, err = staged(**{**ok, "trips": t1, "keep": None, "n_rounds": 1})
    assert rc == -1 and b"null handle" in err
    rc, err = staged(**{**ok, "trips": np.array([0, 0, 0], np.int32), "keep": np.array([1 << 40, 1], np.int64)})
    assert rc == -1 and b"null handle" in err


def test_python_checks_the_length_of_keep():
    import loc_lib_b200 as L
    reg = L.IcpRegistration.__new__(L.IcpRegistration)  # no handle: the length check comes first
    reg._h = None
    with pytest.raises(ValueError, match="keep"):
        reg.RelocaliseStaged(np.zeros((4, 4), np.float32), IDENTITY, (2, 3), (4, 2))
    with pytest.raises(ValueError, match="keep"):
        reg.RelocaliseStaged(np.zeros((4, 4), np.float32), IDENTITY, (2, 3), None)


@pytest.mark.skipif(HAS_GPU, reason="checks the no-device behaviour")
def test_relocalise_staged_fails_loudly_without_a_device():
    from loc_lib_b200 import _lib
    import loc_lib_b200 as L
    with pytest.raises(_lib.LocregError, match="no CPU fallback"):
        reg = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE))
        reg.RelocaliseStaged(np.zeros((4, 4), np.float32), IDENTITY, (2,), None)


def test_selection_rule_orders_by_float32_score_then_index():
    inf = np.inf
    alive = np.array([2, 5, 7, 9, 11, 12])
    # 5 and 9 tie in float32 though not in double; 7 ties 12 exactly
    scores = np.array([0.30, 0.1, 0.2, 0.1 + 1e-12, 0.05, 0.2])
    assert list(survivors(scores, alive, 1)) == [11]
    assert list(survivors(scores, alive, 2)) == [5, 11]
    assert list(survivors(scores, alive, 3)) == [5, 9, 11]  # the tie goes to the lower index first
    assert list(survivors(scores, alive, 4)) == [5, 7, 9, 11]  # 7 before 12
    assert list(survivors(scores, alive, 100)) == list(alive)  # keep beyond the alive set
    # +inf, NaN and negative scores all rank as +inf, among themselves by index
    s = np.array([inf, np.nan, 0.5, -1.0, inf])
    assert list(survivors(s, np.arange(5), 1)) == [2]
    assert list(survivors(s, np.arange(5), 3)) == [0, 1, 2]
    assert list(survivors(np.full(6, inf), np.arange(10, 16), 2)) == [10, 11]
    assert pack_order_scores([np.nan, -0.5, 2.0])[:2].tolist() == [inf, inf]


def test_selection_rule_matches_locreg_pack_score():
    from loc_lib_b200 import _lib
    rng = np.random.default_rng(3)
    scores = np.concatenate([rng.choice([0.25, 0.5, 1.0], 20), rng.random(20), [np.inf] * 5, [np.nan, -1.0]])
    alive = np.sort(rng.choice(1000, len(scores), replace=False))
    keys = [_lib.lib().locreg_pack_score(float(s), int(i)) for s, i in zip(scores, alive)]
    for k in (1, 7, 20, 45, len(scores)):
        by_key = np.sort(alive[np.argsort(keys, kind="stable")[:k]])
        assert np.array_equal(survivors(scores, alive, k), by_key), k
