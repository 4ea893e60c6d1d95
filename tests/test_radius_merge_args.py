"""CPU-only: pn_merge_radius_dev and pn_multi_balltree_query_radius_f32 reject null and out-of-range arguments with
PN_BAD_ARG before they touch a device (the pointers below are never dereferenced)."""
import ctypes as C
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ffi():
    import __graft_entry__ as g
    if not os.path.exists(os.path.join(ROOT, "petal-neighbors_b200", "lib", "libpetal_b200.so")):
        g.build()
    from petal_neighbors_b200 import _ffi
    return _ffi


FAKE = 4096   # a non-null device pointer that must not be used


@pytest.mark.parametrize("args,msg", [
    ((0, None, FAKE, 2, 10, FAKE, FAKE), "null pointer"),
    ((0, FAKE, None, 2, 10, FAKE, FAKE), "null pointer"),
    ((0, FAKE, FAKE, 2, 10, None, FAKE), "null pointer"),
    ((0, FAKE, FAKE, 2, 10, FAKE, None), "null pointer"),
    ((0, FAKE, FAKE, 0, 10, FAKE, FAKE), "n_lists must be in 1..256"),
    ((0, FAKE, FAKE, 257, 10, FAKE, FAKE), "n_lists must be in 1..256"),
    ((0, FAKE, FAKE, 2, 1 << 32, FAKE, FAKE), "nq must be < 2^32"),
])
def test_merge_radius_dev_bad_args(ffi, args, msg):
    L = ffi.lib()
    assert L.pn_merge_radius_dev(*args, None, 1) == ffi.PN_BAD_ARG
    assert ffi.last_error() == msg


def test_multi_query_radius_bad_args(ffi):
    L = ffi.lib()
    q = (C.c_float * 6)()
    po, pi = C.POINTER(C.c_uint64)(), C.POINTER(C.c_uint64)()
    fn = L.pn_multi_balltree_query_radius_f32
    cases = [
        ((None, q, 2, 3, 0.5, None, C.byref(pi)), "output pointer is null"),
        ((None, q, 2, 3, 0.5, C.byref(po), None), "output pointer is null"),
        ((None, None, 2, 3, 0.5, C.byref(po), C.byref(pi)), "queries is null"),
        ((None, q, 1 << 32, 3, 0.5, C.byref(po), C.byref(pi)), "nq must be < 2^32 per call"),
        ((None, q, 2, 3, 0.5, C.byref(po), C.byref(pi)), "handle is null"),
        ((None, None, 0, 3, 0.5, C.byref(po), C.byref(pi)), "handle is null"),
    ]
    for args, msg in cases:
        assert fn(*args) == ffi.PN_BAD_ARG, msg
        assert ffi.last_error() == msg
    assert not po and not pi   # nothing was allocated
