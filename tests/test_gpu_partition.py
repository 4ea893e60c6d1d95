"""The two-means partition behind the pruned tensor scan (csrc/gpu_build.cu rule 1, DeviceTree::two_means_partition).

A handle on clustered data keeps a second ball tree over the same rows whose splits follow 2-means directions and whose
nodes start on tile boundaries; k-NN batches are answered from it.  The reference's pruning rule is the same
(src/ball_tree.rs:211-214, 230-238), the partition is not the reference's -- so everything here is about the one thing
that must not change: indices identical and distances bit-identical to the oracle, whatever the partition."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pn():
    import petal_neighbors_b200 as pn
    return pn


def bits(a):
    return a.view(np.uint32)


def check_knn(oracle, tree, pts, Q, k):
    idx, dist = tree.query_batch(Q, k)
    oi, od = oracle.brute_knn(pts, Q, k)
    bad = np.argwhere(idx != oi.astype(np.uint64))
    assert bad.size == 0, f"index mismatch at {bad[:5]}"
    assert np.array_equal(bits(dist), bits(od))
    return tree.counters()


@pytest.mark.parametrize("n,d,nq,k,centers,sigma", [
    (60000, 64, 3000, 1, 64, 0.05), (60000, 64, 3000, 10, 64, 0.05), (50001, 16, 20000, 10, 64, 0.004),
    (40000, 32, 700, 16, 32, 0.03), (30000, 128, 1500, 10, 16, 0.05), (20000, 20, 1, 5, 8, 0.02),
    (1024, 16, 300, 3, 4, 0.01), (5000, 100, 513, 2, 8, 0.05), (33000, 370, 600, 4, 8, 0.05),
])
def test_two_means_partition_forced(pn, oracle, n, d, nq, k, centers, sigma):
    """Forced on ball and VP handles, with the tile bitmaps forced on and in AUTO: exact, and the handle says which partition
    its k-NN batches scan.  Self-queries, radius queries and the layout of a ball handle stay on the reference partition."""
    from petal_neighbors_b200 import synth
    pts = synth.gaussian_mixture(n, d, 5, n_centers=centers, sigma=sigma)
    Q = synth.gaussian_mixture(nq, d, 6, n_centers=centers, sigma=sigma)
    for prune in (pn.PN_PRUNE_ON, pn.PN_PRUNE_AUTO):
        bt = pn.BallTree.euclidean(pts, prune=prune, partition=pn.PN_PARTITION_TWO_MEANS)
        assert bt.info()["tensor_partition"] == 1
        c = check_knn(oracle, bt, pts, Q, k)
        assert 0 < c["filter_pairs"] <= n * nq and c["pairs"] <= n * nq
    ref = pn.BallTree.euclidean(pts, partition=pn.PN_PARTITION_REFERENCE)
    assert ref.info()["tensor_partition"] == 0
    check_knn(oracle, ref, pts, Q, k)
    # the other entry points of the handle that keeps the second partition
    r = np.float32(np.median(oracle.brute_knn(pts, Q[:64], min(k + 3, n))[1][:, -1]))
    offs, ind = bt.query_radius_batch(Q[:200], r)
    boffs, bind = oracle.brute_radius(pts, Q[:200], r)
    assert np.array_equal(offs, boffs.astype(np.uint64)) and np.array_equal(ind, bind.astype(np.uint64))
    lay = bt.layout()
    assert np.array_equal(np.sort(lay["ids"]), np.arange(n, dtype=np.uint32))
    assert np.array_equal(lay["points"][:, :d], pts[lay["ids"]])
    vp = pn.VantagePointTree.euclidean(pts, prune=pn.PN_PRUNE_ON, partition=pn.PN_PARTITION_TWO_MEANS)
    assert vp.info()["tensor_partition"] == 1
    vi, vd = vp.query_nearest_batch(Q)
    oi, od = oracle.brute_knn(pts, Q, 1)
    assert np.array_equal(vi, oi[:, 0].astype(np.uint64)) and np.array_equal(bits(vd), bits(od[:, 0]))
    check_knn(oracle, vp, pts, Q, k)                       # VP k-NN extension
    offs, ind = vp.query_radius_batch(Q[:200], r)          # VP radius extension: the SIMT traversal of the two-means TREE
    assert np.array_equal(offs, boffs.astype(np.uint64)) and np.array_equal(ind, bind.astype(np.uint64))


def test_two_means_partition_prunes_where_the_reference_partition_cannot(pn, oracle):
    """A scaled-down BASELINE config 3 (d = 64 mixture, sigma 0.05): with the reference partition most 128-row tiles mix
    fragments of several clusters and the bitmaps keep ~90 % of the pairs; the two-means partition must get well below that,
    and AUTO must get there by itself."""
    from petal_neighbors_b200 import synth
    n, nq, d = 130000, 65536, 64
    pts = synth.gaussian_mixture(n, d, 5, n_centers=128, sigma=0.05)
    Q = synth.gaussian_mixture(nq, d, 6, n_centers=128, sigma=0.05)
    sample = np.arange(0, nq, nq // 500)[:500]
    oi, od = oracle.brute_knn(pts, Q[sample], 10)
    frac = {}
    for name, opts in (("reference", dict(prune=pn.PN_PRUNE_ON, partition=pn.PN_PARTITION_REFERENCE)),
                       ("two_means", dict(prune=pn.PN_PRUNE_ON, partition=pn.PN_PARTITION_TWO_MEANS)),
                       ("auto", dict())):
        bt = pn.BallTree.euclidean(pts, **opts)
        idx, dist = bt.query_batch(Q, 10)
        assert np.array_equal(idx[sample], oi.astype(np.uint64)) and np.array_equal(bits(dist[sample]), bits(od)), name
        frac[name] = bt.counters()["pairs"] / (float(n) * nq)
        if name == "auto":
            inf = bt.info()
            assert inf["prune_tiles"] == 1, inf
    assert frac["two_means"] < 0.6 and frac["two_means"] < 0.8 * frac["reference"], frac
    assert frac["auto"] < 0.6, frac
    vp = pn.VantagePointTree.euclidean(pts)
    vi, vd = vp.query_nearest_batch(Q)
    assert np.array_equal(vi[sample], oi[:, 0].astype(np.uint64)) and np.array_equal(bits(vd[sample]), bits(od[:, 0]))
    assert vp.counters()["pairs"] < 0.6 * float(n) * nq


def test_two_means_partition_degenerate_inputs(pn, oracle):
    """Identical points (no direction to split along: every key ties, the index decides), lattices of ties, a few points far
    away from everything, uniform data, sessions on a handle that keeps the second partition."""
    rng = np.random.default_rng(11)
    same = np.tile(rng.random((1, 24), np.float32), (3000, 1))
    base = rng.integers(0, 4, size=(40, 24)).astype(np.float32) * 10
    lattice = np.repeat(base, 250, axis=0) + rng.integers(0, 2, size=(10000, 24)).astype(np.float32)
    far = (rng.random((5, 24), np.float32) * 1e4).astype(np.float32)
    pts = np.concatenate([same, lattice, far]).astype(np.float32)
    rng.shuffle(pts)
    Q = np.concatenate([pts[:700] + 0.5, same[:50], rng.random((100, 24), np.float32) * 50.0]).astype(np.float32)
    for prune in (pn.PN_PRUNE_ON, pn.PN_PRUNE_AUTO):
        bt = pn.BallTree.euclidean(pts, prune=prune, partition=pn.PN_PARTITION_TWO_MEANS, algo=pn.PN_ALGO_TENSOR)
        assert bt.info()["tensor_partition"] == 1
        for k in (1, 10, 16, 20):
            check_knn(oracle, bt, pts, Q, k)
    idx, dist = bt.query_self(8)
    oi, od = oracle.brute_knn(pts, pts, 8)
    assert np.array_equal(idx, oi.astype(np.uint64)) and np.array_equal(bits(dist), bits(od))
    s = bt.session()
    check_knn(oracle, s, pts, Q, 10)
    s.close()
    from petal_neighbors_b200 import synth
    u = synth.uniform(20000, 16, 77, np.float32)
    uq = synth.uniform(1500, 16, 78, np.float32)
    bu = pn.BallTree.euclidean(u, partition=pn.PN_PARTITION_TWO_MEANS, bucket_size=64)   # bucket below a tile: the plain shape
    check_knn(oracle, bu, u, uq, 10)
    auto = pn.BallTree.euclidean(u)                       # uniform data: AUTO never builds the second partition
    assert auto.info()["tensor_partition"] == 0
