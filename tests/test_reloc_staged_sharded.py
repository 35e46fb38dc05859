"""CPU tests of locreg_relocalise_staged_sharded / RelocaliseStagedSharded: the null-handle refusal, the argument checks
(the same codes and messages as locreg_relocalise_staged, before any device work), the Python entry point failing
loudly without a device, and the deal / exchange maps of a round across ranks."""
import numpy as np
import pytest

from conftest import HAS_GPU

IDENTITY = np.array([0, 0, 0, 1, 0, 0, 0], np.float64)


def call(symbol, h=None, src=None, n=0, stride=16, pin=None, n_hyp=1, trips=None, keep=None, n_rounds=1):
    from loc_lib_b200 import _lib
    ptr = lambda x: None if x is None else x.ctypes.data  # noqa: E731
    bp, bs = np.zeros(7), np.zeros(1)
    bi = np.zeros(1, np.int64)
    rc = getattr(_lib.lib(), symbol)(h, ptr(src), n, stride, ptr(pin), n_hyp, ptr(trips), ptr(keep), n_rounds,
                                     ptr(bp), ptr(bi), ptr(bs), None, None, None)
    return rc, _lib.lib().locreg_last_error()


def sharded(**kw):
    return call("locreg_relocalise_staged_sharded", **kw)


def single(**kw):
    return call("locreg_relocalise_staged", **kw)


def test_null_handle_is_refused_before_any_device_work():
    rc, err = sharded(pin=IDENTITY, trips=np.array([2, 3], np.int32), keep=np.array([4], np.int64), n_rounds=2)
    assert rc == -1 and b"null handle" in err


def test_argument_errors_are_those_of_the_single_gpu_call():
    cloud = np.zeros((4, 4), np.float32)
    hyp = np.stack([IDENTITY] * 3)
    t3 = np.array([1, 2, 3], np.int32)
    k2 = np.array([2, 1], np.int64)
    ok = dict(src=cloud, n=4, pin=hyp, n_hyp=3, trips=t3, keep=k2, n_rounds=3)
    cases = [({}, b"null handle"), ({"src": None}, b"cloud"), ({"stride": 8}, None), ({"stride": 18}, None),
             ({"pin": None}, b"invalid hypotheses"), ({"n_hyp": 0}, b"invalid hypotheses"),
             ({"n_hyp": 1 << 31}, b"invalid hypotheses"),
             ({"n_rounds": 0}, b"n_rounds"), ({"n_rounds": -1}, b"n_rounds"), ({"n_rounds": 33}, b"n_rounds"),
             ({"trips": None}, b"trips"), ({"trips": np.array([1, -1, 3], np.int32)}, b"trips"),
             ({"keep": None}, b"keep"), ({"keep": np.array([0, 1], np.int64)}, b"keep"),
             ({"keep": np.array([2, 0], np.int64)}, b"keep"), ({"keep": np.array([-5, 1], np.int64)}, b"keep"),
             # valid: one round without keep, score-only rounds, keep beyond the alive set (only the handle is missing)
             ({"trips": np.array([2], np.int32), "keep": None, "n_rounds": 1}, b"null handle"),
             ({"trips": np.array([0, 0, 0], np.int32), "keep": np.array([1 << 40, 1], np.int64)}, b"null handle")]
    for bad, word in cases:
        rc, err = sharded(**{**ok, **bad})
        assert (rc, err) == single(**{**ok, **bad}), bad
        assert rc == -1, bad
        if word is not None:
            assert word in err, (bad, err)


def test_python_checks_the_length_of_keep():
    import loc_lib_b200 as L
    reg = L.IcpRegistration.__new__(L.IcpRegistration)  # no handle: the length check comes first
    reg._h = None
    with pytest.raises(ValueError, match="keep"):
        reg.RelocaliseStagedSharded(np.zeros((4, 4), np.float32), IDENTITY, (2, 3), (4, 2))


@pytest.mark.skipif(HAS_GPU, reason="checks the no-device behaviour")
def test_relocalise_staged_sharded_fails_loudly_without_a_device():
    from loc_lib_b200 import _lib
    import loc_lib_b200 as L
    with pytest.raises(_lib.LocregError, match="no CPU fallback"):
        reg = L.IcpRegistration(L.IcpOptions(method_=L.IcpMethod.P2PLANE))
        reg.RelocaliseStagedSharded(np.zeros((4, 4), np.float32), IDENTITY, (2,), None)


def test_the_python_method_goes_to_the_library_and_raises():
    """Valid arguments on a registration without a handle (as one whose construction failed): the method has no
    Python-side path of its own, so the library's refusal comes back as an exception."""
    from loc_lib_b200 import _lib
    import loc_lib_b200 as L
    reg = L.IcpRegistration.__new__(L.IcpRegistration)
    reg._h = None
    for want_all in (False, True):
        with pytest.raises(_lib.LocregError, match="null handle"):
            reg.RelocaliseStagedSharded(np.zeros((4, 4), np.float32), np.stack([IDENTITY] * 3), (2, 3), (2,), want_all)


def deal(m, rank, world):
    """The positions rank `rank` runs in a round of m alive hypotheses (k_reloc_deal): rank, rank + world, ..."""
    m_q = -(-(m - rank) // world) if m > rank else 0
    return rank + np.arange(m_q) * world


def exchange(m, world):
    """Every rank packs its results into slab `rank` of ceil(m / world) records (k_reloc_pack), the all-gather puts
    the slabs side by side, and k_reloc_unpack reads position p from slab p % world, record p // world.  Returns the
    position each unpacked entry came from (-1: a record no rank wrote)."""
    c = -(-m // world)
    gather = np.full(world * c, -1)
    for q in range(world):
        mine = deal(m, q, world)
        assert len(mine) <= c
        gather[q * c:q * c + len(mine)] = mine
    p = np.arange(m)
    return gather[(p % world) * c + p // world]


@pytest.mark.parametrize("world", range(1, 9))
def test_deal_then_unpack_returns_every_position_once(world):
    for m in sorted({1, 2, 3, world - 1, world, world + 1, 2 * world - 1, 2 * world + 3, 7 * world + 5, 64, 257} - {0}):
        shares = [deal(m, q, world) for q in range(world)]
        got = np.concatenate(shares)
        assert np.array_equal(np.sort(got), np.arange(m)), (m, world)  # every position runs on exactly one rank
        sizes = [len(s) for s in shares]
        assert max(sizes) - min(sizes) <= 1 and sizes == sorted(sizes, reverse=True), (m, world, sizes)
        assert np.array_equal(exchange(m, world), np.arange(m)), (m, world)
    # round 0 is locreg_relocalise_sharded's deal: rank q registers q, q + world, ...
    assert deal(10, 2, 4).tolist() == [2, 6] and deal(3, 5, 8).tolist() == []
