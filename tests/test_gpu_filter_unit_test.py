"""The narrow-row tensor filter tests each 64-column accumulator unit with one minimum and searches the columns only
when some lane has a hit (csrc/tc_filter.cuh).  Self-queries over every point make every stored position the exact
nearest neighbour (distance 0) of some query: the last column of each unit, the last rows of a partly filled last tile,
and the zero-filled rows past it, which must never be returned.  Results must match the oracle bit for bit."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pn():
    import petal_neighbors_b200 as pn
    return pn


# n = 39 tiles of 128 + 100 rows: the last tile's second unit holds 36 points (its last group 4); n = 4160: the last
# tile holds 64 points, a full first unit and an empty second one
@pytest.mark.parametrize("n", [5092, 4160])
@pytest.mark.parametrize("k", [1, 10])
def test_self_queries_reach_every_column(pn, oracle, n, k):
    from petal_neighbors_b200 import synth
    pts = synth.uniform(n, 16, 70 + n, np.float32)
    bt = pn.BallTree.euclidean(pts, algo=pn.PN_ALGO_TENSOR)
    idx, dist = bt.query_batch(pts, k)
    assert 0 < bt.counters()["filter_pairs"] <= n * n      # the tensor path ran (pruning may skip tiles)
    oi, od = oracle.brute_knn(pts, pts, k)
    assert np.array_equal(idx, oi.astype(np.uint64))
    assert np.array_equal(dist.view(np.uint32), od.view(np.uint32))
    assert np.array_equal(idx[:, 0], np.arange(n, dtype=np.uint64)) and not dist[:, 0].any()


def test_duplicated_points_tie_at_the_kth_distance(pn, oracle):
    """Every point twice: the two copies of a neighbour give the same accumulator value, so a query's k-th distance is
    always tied and the copy with the larger index must still pass the threshold; ties resolve by index."""
    from petal_neighbors_b200 import synth
    base = synth.uniform(2600, 16, 91, np.float32)
    pts = np.concatenate([base, base])
    Q = synth.uniform(2048, 16, 92, np.float32)
    bt = pn.BallTree.euclidean(pts, algo=pn.PN_ALGO_TENSOR)
    for k in (2, 10):
        idx, dist = bt.query_batch(Q, k)
        assert 0 < bt.counters()["filter_pairs"] <= pts.shape[0] * Q.shape[0]
        oi, od = oracle.brute_knn(pts, Q, k)
        assert np.array_equal(idx, oi.astype(np.uint64))
        assert np.array_equal(dist.view(np.uint32), od.view(np.uint32))
