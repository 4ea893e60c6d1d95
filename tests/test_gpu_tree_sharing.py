"""One device tree shared by a handle and its sessions: a vantage-point tree whose ball companion is built on the first
radius call (f64 here) builds it once, for every handle of the tree, and the handle that built the tree accounts for it."""
import threading

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

N, D, R = 20000, 3, 0.05


@pytest.fixture(scope="module")
def pn():
    import petal_neighbors_b200 as pn
    return pn


def points(seed):
    from petal_neighbors_b200 import synth
    return synth.uniform(N, D, seed, np.float64)


def assert_radius_equal(got, want):
    assert np.array_equal(got[0], want[0].astype(np.uint64)) and np.array_equal(got[1], want[1].astype(np.uint64))


def test_lazy_companion_shared_by_sessions(pn, oracle):
    from petal_neighbors_b200 import synth
    pts = points(91)
    Q = synth.uniform(500, D, 92, np.float64)
    want = oracle.brute_radius(pts, Q, R)
    tree = pn.VantagePointTree.euclidean(pts)
    s1 = tree.session()
    b0 = tree.info()["device_bytes"]
    assert_radius_equal(s1.query_radius_batch(Q, R), want)
    assert s1.info()["device_bytes"] == 0
    b1 = tree.info()["device_bytes"]
    assert b1 > b0   # the companion S1 built belongs to the tree
    s2 = s1.session()
    assert_radius_equal(s2.query_radius_batch(Q, R), want)
    assert tree.info()["device_bytes"] == b1   # built once
    tree.close()
    s1.close()   # S2 alone keeps the tree and its companion alive
    assert_radius_equal(s2.query_radius_batch(Q, R), want)
    ni, nd = s2.query_nearest_batch(Q)
    oi, od = oracle.brute_knn(pts, Q, 1)
    assert np.array_equal(ni, oi[:, 0].astype(np.uint64)) and np.array_equal(nd.view(np.uint64), od[:, 0].view(np.uint64))
    s2.close()


def test_lazy_companion_concurrent_first_calls(pn, oracle):
    from petal_neighbors_b200 import synth
    pts = points(93)
    # the companion's size, from a tree of the same shape with a single caller
    single = pn.VantagePointTree.euclidean(points(94))
    b0 = single.info()["device_bytes"]
    single.query_radius_batch(synth.uniform(8, D, 95, np.float64), R)
    grown = single.info()["device_bytes"] - b0
    single.close()
    assert grown > 0

    tree = pn.VantagePointTree.euclidean(pts)
    b0 = tree.info()["device_bytes"]
    Qs = [synth.uniform(500, D, 96 + t, np.float64) for t in range(4)]
    sessions = [tree.session() for _ in Qs]
    out = [None] * len(Qs)
    start = threading.Barrier(len(Qs))

    def work(t):
        start.wait()
        out[t] = sessions[t].query_radius_batch(Qs[t], R)

    th = [threading.Thread(target=work, args=(t,)) for t in range(len(Qs))]
    [x.start() for x in th]
    [x.join() for x in th]
    for t, Q in enumerate(Qs):
        assert_radius_equal(out[t], oracle.brute_radius(pts, Q, R))
    assert tree.info()["device_bytes"] - b0 == grown
    for s in sessions:
        s.close()
    tree.close()
