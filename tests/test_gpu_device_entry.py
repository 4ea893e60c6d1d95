"""The device-pointer entry points -- pn_tree_query_knn_dev (the call bench.py times) and pn_tree_query_self_dev -- on every
scan engine, against the oracle: indices identical (ties by index), distances bit-identical.

The host-buffer calls pack the queries to row stride d before any kernel runs; only the device calls hand a caller's
row stride to the staging kernels, and only they run a whole batch as one launch plan (full waves plus a split tail).
So the queries here sit in a NaN-filled buffer at a misaligned base with a row stride wider than d -- a kernel that reads
a padding element gets a NaN distance -- and every output buffer has a sentinel row before and after the rows the call
may write.  Every case also asserts which engine answered it, so that a change of the selection heuristics cannot move a
case onto another engine unnoticed."""
import threading

import numpy as np
import pytest

from petal_neighbors_b200 import (PN_ALGO_AUTO, PN_ALGO_SIMT, PN_ALGO_TENSOR, PN_PARTITION_TWO_MEANS, PN_PRUNE_OFF,
                                  PN_PRUNE_ON)

pytestmark = pytest.mark.gpu

KS = (1, 10, 16, 17, 32, 33)
PADS = (1, 3, 13)
SENT_I = 0x5A5A5A5A5A5A5A5A
NO_ID = np.iinfo(np.uint64).max


@pytest.fixture(scope="module")
def pn():
    import petal_neighbors_b200 as pn
    return pn


@pytest.fixture(scope="module")
def torch():
    import torch
    return torch


def bits(a):
    return a.view(np.uint32 if a.dtype == np.float32 else np.uint64)


def assert_knn_equal(idx, dist, oi, od, tag=""):
    bad = np.argwhere(idx != oi.astype(np.uint64))
    assert bad.size == 0, f"{tag}: index mismatch at {bad[:5].tolist()} got {idx[tuple(bad[0])]} want {oi[tuple(bad[0])]}"
    bad = np.argwhere(bits(dist) != bits(od))
    assert bad.size == 0, f"{tag}: distances not bit-identical at {bad[:5].tolist()}"


def tdtype(torch, dtype):
    return torch.float32 if dtype == np.float32 else torch.float64


def poisoned_queries(torch, Q, pad, stride=None):
    """Q (nq x d) in a NaN-filled device buffer with row stride d + pad (or `stride`), starting at an odd element offset
    past a whole NaN row: the base pointer is not 16-byte aligned and every element between rows is NaN.  Returns
    (buffer, pointer of row 0, row stride)."""
    nq, d = Q.shape
    s = d + pad if stride is None else stride
    s_rows = max(s, d)
    base = s_rows + (1 if s_rows % 2 == 0 else 2)          # odd: never 16-byte aligned for f32 or f64
    buf = torch.full(((nq + 2) * s_rows + 4,), float("nan"), dtype=tdtype(torch, Q.dtype), device="cuda")
    buf.as_strided((nq, d), (s_rows, 1), base).copy_(torch.from_numpy(np.ascontiguousarray(Q)))
    assert (buf.data_ptr() + base * Q.itemsize) % 16 != 0
    return buf, buf.data_ptr() + base * Q.itemsize, s


class Guarded:
    """(rows + 2) x k outputs filled with a sentinel (index 0x5a5a..., distance -1); the call gets the pointers of row 1."""

    def __init__(self, torch, rows, k, dtype):
        self.rows, self.k = rows, k
        self.i = torch.full(((rows + 2) * k,), SENT_I, dtype=torch.int64, device="cuda")
        self.d = torch.full(((rows + 2) * k,), -1.0, dtype=tdtype(torch, dtype), device="cuda")
        self.ip = self.i.data_ptr() + k * 8
        self.dp = self.d.data_ptr() + k * self.d.element_size()

    def result(self):
        """(idx[rows, k] u64, dist[rows, k]) after checking that the guard rows are untouched."""
        i = self.i.cpu().numpy().view(np.uint64).reshape(self.rows + 2, self.k)
        d = self.d.cpu().numpy().reshape(self.rows + 2, self.k)
        for g in (0, self.rows + 1):
            assert np.all(i[g] == SENT_I) and np.all(d[g] == -1), f"guard row {g} was written"
        return i[1:-1], d[1:-1]

    def untouched(self):
        i = self.i.cpu().numpy().view(np.uint64)
        d = self.d.cpu().numpy()
        return bool(np.all(i == SENT_I) and np.all(d == -1))


def knn_dev(pn, torch, tree, Q, k, pad, stride=None, stream=0, sync=True):
    """One query_knn_dev call over poisoned strided queries into guarded outputs; returns (idx, dist)."""
    buf, qp, s = poisoned_queries(torch, Q, pad, stride)
    out = Guarded(torch, Q.shape[0], k, Q.dtype)
    torch.cuda.synchronize()
    tree.query_knn_dev(qp, Q.shape[0], s, k, out.ip, out.dp, stream=stream, sync=sync)
    torch.cuda.synchronize()
    return out.result()


# ------------------------------------------------------------------ data
def lattice(rng, n, d, dtype, hi=4):
    return rng.integers(0, hi, size=(n, d)).astype(dtype)


def cluster_lattice(rng, n, d):
    """tight clusters of lattice points (as in test_gpu_prune): tile balls that prune, and masses of exact ties"""
    base = rng.integers(0, 4, size=(64, d)).astype(np.float32) * 10
    pts = base[rng.integers(0, 64, size=n)] + rng.integers(0, 2, size=(n, d)).astype(np.float32)
    return pts.astype(np.float32)


def make_data(kind, data, n, d, dtype, seed):
    from petal_neighbors_b200 import synth
    rng = np.random.default_rng(seed)
    if kind == "clusters":
        if data == "lattice":
            pts = cluster_lattice(rng, n, d)
            Q = pts[rng.integers(0, n, size=129)] + np.float32(0.5) * rng.integers(0, 2, size=(129, d)).astype(np.float32)
            return pts, Q.astype(np.float32)
        return (synth.gaussian_mixture(n, d, 5, n_centers=64, sigma=0.004),
                synth.gaussian_mixture(129, d, 6, n_centers=64, sigma=0.004))
    if data == "lattice":
        return lattice(rng, n, d, dtype), lattice(rng, 129, d, dtype)
    return synth.uniform(n, d, seed, dtype), synth.uniform(129, d, seed + 1, dtype)


# engine -> (tree class, dtype, n, d, data kind, build options, engine check)
def _simt(inf, c):
    return c["filter_pairs"] == 0


def _dense(inf, c):
    return c["filter_pairs"] > 0 and not inf["prune_seeded"] and not inf["prune_tiles"]


def _seeded(inf, c):
    return c["filter_pairs"] > 0 and inf["prune_seeded"] and not inf["prune_tiles"]


def _tiles(inf, c):
    return c["filter_pairs"] > 0 and inf["prune_seeded"] and inf["prune_tiles"] and inf["tensor_partition"] == 0


def _two_means(inf, c):
    return c["filter_pairs"] > 0 and inf["tensor_partition"] == 1


def _tensor(inf, c):
    return c["filter_pairs"] > 0


ENGINES = {
    "warp_f32_d5": ("ball", np.float32, 4000, 5, "plain", {}, _simt),
    "warp_f64_d3": ("ball", np.float64, 4000, 3, "plain", {}, _simt),
    "tile_f64_d12": ("ball", np.float64, 4000, 12, "plain", {}, _simt),
    "tile_f32_d12": ("ball", np.float32, 4000, 12, "plain", {"algo": PN_ALGO_SIMT}, _simt),
    "vp_simt_d24": ("vp", np.float32, 6000, 24, "plain", {"algo": PN_ALGO_SIMT}, _simt),
    "dense_d16": ("ball", np.float32, 20000, 16, "plain", {"prune": PN_PRUNE_OFF}, _dense),
    "dense_d20": ("ball", np.float32, 20000, 20, "plain", {"prune": PN_PRUNE_OFF}, _dense),
    "tiles_d16": ("ball", np.float32, 50000, 16, "clusters", {"prune": PN_PRUNE_ON}, _tiles),
    "two_means_d16": ("ball", np.float32, 50001, 16, "clusters", {"prune": PN_PRUNE_ON, "partition": PN_PARTITION_TWO_MEANS},
                      _two_means),
    "wide_d300": ("ball", np.float32, 1500, 300, "plain", {}, _tensor),
    "wide_d500": ("ball", np.float32, 800, 500, "plain", {}, _simt),
    "vp_tensor_d24": ("vp", np.float32, 20000, 24, "plain", {}, _tensor),
}


@pytest.mark.parametrize("data", ["random", "lattice"])
@pytest.mark.parametrize("engine", list(ENGINES))
def test_knn_dev_engines(pn, torch, oracle, engine, data):
    """Every k of KS (k = 16 | 17 and 32 | 33 are the pass boundaries of the tensor and warp scans) for 129 queries, and
    single queries with a row stride and with stride 0, through strided NaN-poisoned queries into guarded outputs."""
    kind, dtype, n, d, shape, opts, is_engine = ENGINES[engine]
    pts, Q = make_data(shape, data, n, d, dtype, 100 + d)
    cls = pn.BallTree if kind == "ball" else pn.VantagePointTree
    tree = cls.euclidean(pts, **opts)
    inf = tree.info()
    oi, od = oracle.brute_knn(pts, Q, max(KS))
    for j, k in enumerate(KS):
        tag = f"{engine} {data} k={k}"
        idx, dist = knn_dev(pn, torch, tree, Q, k, PADS[j % 3])
        c = tree.counters()
        assert is_engine(inf, c), f"{tag}: ran on another engine: {inf} {c}"
        assert c["queries"] == 129 and c["h2d_bytes"] == 0 and c["d2h_bytes"] == 0, f"{tag}: {c}"
        assert_knn_equal(idx, dist, oi[:, :k], od[:, :k], tag)
    for k in (10, 33):
        for j, stride in enumerate((None, 0)):
            idx, dist = knn_dev(pn, torch, tree, Q[5:6], k, PADS[j + 1], stride=stride)
            assert is_engine(inf, tree.counters()), f"{engine} {data}: single query ran on another engine"
            assert_knn_equal(idx, dist, oi[5:6, :k], od[5:6, :k], f"{engine} {data} single query k={k} stride={stride}")


# A tree the AUTO estimates put on the seeded d = 16 scan without tile bitmaps: the engine of the benchmark's C2 shape.
# (PN_PRUNE_ON cannot select it: forcing pruning on builds the tile bitmaps too.)
SEEDED_N = 200_000
SEEDED_HI = 4      # lattice coordinates in [0, SEEDED_HI)


@pytest.mark.parametrize("data", ["random", "lattice"])
def test_knn_dev_seeded_scan(pn, torch, oracle, data):
    """Uniform data, and a lattice whose 16th / 17th and 32nd / 33rd neighbours are tied for most queries."""
    from petal_neighbors_b200 import synth
    if data == "lattice":
        rng = np.random.default_rng(23)
        pts, Q = lattice(rng, SEEDED_N, 16, np.float32, SEEDED_HI), lattice(rng, 1000, 16, np.float32, SEEDED_HI)
    else:
        pts = synth.uniform(SEEDED_N, 16, 23, np.float32)
        Q = synth.uniform(1000, 16, 24, np.float32)
    Q[7] = pts[SEEDED_N // 3]                                  # a query at distance 0
    tree = pn.BallTree.euclidean(pts)
    inf = tree.info()
    oi, od = oracle.brute_knn(pts, Q, max(KS))
    for j, k in enumerate(KS):
        idx, dist = knn_dev(pn, torch, tree, Q, k, PADS[j % 3])
        c = tree.counters()
        assert _seeded(inf, c), f"k={k}: {inf} {c}"
        assert_knn_equal(idx, dist, oi[:, :k], od[:, :k], f"seeded {data} k={k}")
    idx, dist = knn_dev(pn, torch, tree, Q[7:8], 10, 3, stride=0)
    assert_knn_equal(idx, dist, oi[7:8, :10], od[7:8, :10], "seeded single query")


@pytest.mark.parametrize("engine", ["warp_f32_d5", "tile_f64_d12", "vp_simt_d24", "dense_d16", "wide_d300", "vp_tensor_d24"])
def test_knn_dev_k_beyond_n(pn, torch, oracle, engine):
    """k > n: the columns past n are (2^64 - 1, +inf), inside each row (the guard rows stay untouched)."""
    kind, dtype, _, d, _, opts, _ = ENGINES[engine]
    n = 1100 if engine == "vp_tensor_d24" else 40           # a VP handle keeps its ball partition from 1024 points on
    rng = np.random.default_rng(d)
    pts, Q = lattice(rng, n, d, dtype), lattice(rng, 129, d, dtype)
    cls = pn.BallTree if kind == "ball" else pn.VantagePointTree
    tensor = engine in ("dense_d16", "wide_d300")               # at n = 40 only a forced tensor path scans with the filter
    tree = cls.euclidean(pts, **dict(opts, algo=opts.get("algo", PN_ALGO_TENSOR if tensor else PN_ALGO_AUTO)))
    k = n + 7
    oi, od = oracle.brute_knn(pts, Q, k)
    idx, dist = knn_dev(pn, torch, tree, Q, k, 3)
    assert (tree.counters()["filter_pairs"] > 0) == (engine in ("dense_d16", "wide_d300", "vp_tensor_d24")), engine
    assert_knn_equal(idx, dist, oi, od, engine)
    assert np.all(idx[:, n:] == NO_ID) and np.all(np.isinf(dist[:, n:])) and np.all(idx[:, :n] < n)


def test_knn_dev_waves_and_tail(pn, torch, oracle):
    """More than one wave of query tiles plus a partial one (148 x 512 + 224 queries at d = 16): the main launch and the
    split-stream tail launch, with one and with two passes."""
    from petal_neighbors_b200 import synth
    n, d, nq = 20000, 16, 76000
    pts = synth.uniform(n, d, 61, np.float32)
    pts[n // 2] = pts[n // 3]
    Q = synth.uniform(nq, d, 62, np.float32)
    Q[0] = Q[nq - 1] = pts[n // 3]
    tree = pn.BallTree.euclidean(pts, prune=pn.PN_PRUNE_OFF)
    oi, od = oracle.brute_knn(pts, Q, 17)
    for k, pad in ((10, 13), (17, 1)):
        idx, dist = knn_dev(pn, torch, tree, Q, k, pad)
        c = tree.counters()
        assert c["filter_pairs"] == n * nq * (-(-k // 16)) and c["queries"] == nq
        assert_knn_equal(idx, dist, oi[:, :k], od[:, :k], f"waves k={k}")


# ------------------------------------------------------------------ self-queries through device pointers
def self_dev(pn, torch, tree, n, k, dtype, stream=0, sync=True):
    out = Guarded(torch, n, k, dtype)
    torch.cuda.synchronize()
    tree.query_self_dev(k, out.ip, out.dp, stream=stream, sync=sync)
    torch.cuda.synchronize()
    return out.result()


def dup_lattice(n, d, dtype, hi, seed):
    """lattice points with exact duplicates (distance-0 ties) and tied neighbours at every pass boundary"""
    rng = np.random.default_rng(seed)
    pts = lattice(rng, n, d, dtype, hi)
    pts[n // 2] = pts[n // 3]
    pts[n - 1] = pts[0]
    return pts


def check_self(pn, torch, tree, pts, ks, oi, od, tag, is_engine, host=True):
    n = pts.shape[0]
    for k in ks:
        idx, dist = self_dev(pn, torch, tree, n, k, pts.dtype)
        c = tree.counters()
        assert is_engine(tree.info(), c, k), f"{tag} k={k}: self_dev ran on another engine: {c}"
        assert c["queries"] == n and c["h2d_bytes"] == 0 and c["d2h_bytes"] == 0, f"{tag} k={k}: {c}"
        assert_knn_equal(idx, dist, oi[:, :k], od[:, :k], f"{tag} self_dev k={k}")
        assert np.all(dist[:, 0] == 0)
        if host:
            hi, hd = tree.query_self(k)
            assert_knn_equal(hi, hd, oi[:, :k], od[:, :k], f"{tag} query_self k={k}")
    return c


def test_self_dev_tensor_main_and_tail(pn, torch, oracle):
    """n = 76 000 stored points at d = 16: a main launch of whole waves and a split tail, one to three passes (the floors
    of pass p + 1 are indexed by stored slot while the results go to the original rows), binary lattice: every pass
    boundary falls inside a run of tied distances.  A session of the same tree answers the same."""
    n, d = 76000, 16
    pts = dup_lattice(n, d, np.float32, 2, 5)
    tree = pn.BallTree.euclidean(pts, algo=pn.PN_ALGO_TENSOR, prune=pn.PN_PRUNE_OFF)
    oi, od = oracle.brute_knn(pts, pts, 33)
    check_self(pn, torch, tree, pts, (10, 17, 33), oi, od, "tensor",
               lambda inf, c, k: _dense(inf, c) and c["filter_pairs"] == n * n * -(-k // 16))
    s = tree.session()
    idx, dist = self_dev(pn, torch, s, n, 17, np.float32)
    assert s.counters()["filter_pairs"] == n * n * 2
    assert_knn_equal(idx, dist, oi[:, :17], od[:, :17], "session self_dev k=17")


@pytest.mark.parametrize("engine,n,ks", [("warp_f32_d5", 6000, (40, 17, 33)), ("tile_f64_d12", 5000, (20, 17, 33)),
                                         ("dense_d16", 3000, (10, 17, 33)), ("vp_simt_d24", 4000, (10, 17, 33)),
                                         ("vp_tensor_d24", 4000, (10, 17, 33))])
def test_self_dev_engines(pn, torch, oracle, engine, n, ks):
    """Multi-pass self-queries on the SIMT kernels, the dense tensor scan and both engines of a VP handle."""
    kind, dtype, _, d, _, opts, is_engine = ENGINES[engine]
    pts = dup_lattice(n, d, dtype, 3 if d <= 5 else 2, d)
    cls = pn.BallTree if kind == "ball" else pn.VantagePointTree
    tree = cls.euclidean(pts, **opts)
    oi, od = oracle.brute_knn(pts, pts, max(ks))
    check_self(pn, torch, tree, pts, ks, oi, od, engine, lambda inf, c, k: is_engine(inf, c), host=kind == "ball")
    s = tree.session()
    idx, dist = self_dev(pn, torch, s, n, ks[-1], dtype)
    assert is_engine(tree.info(), s.counters()), f"{engine} session"
    assert_knn_equal(idx, dist, oi[:, :ks[-1]], od[:, :ks[-1]], f"{engine} session")


def test_self_dev_shard_is_rejected(pn, torch):
    from petal_neighbors_b200 import synth
    pts = synth.uniform(5000, 8, 3, np.float32)
    shard = pn.BallTree.euclidean(pts, shard_depth=1, shard_index=0)
    out = Guarded(torch, 5000, 5, np.float32)
    with pytest.raises(pn.EngineError) as e:
        shard.query_self_dev(5, out.ip, out.dp)
    assert e.value.status == 3   # PN_BAD_ARG
    torch.cuda.synchronize()
    assert out.untouched()


# ------------------------------------------------------------------ streams, asynchronous calls, no-ops and errors
@pytest.fixture(scope="module")
def d16(pn, oracle):
    from petal_neighbors_b200 import synth
    pts = synth.uniform(20000, 16, 71, np.float32)
    Qs = [synth.uniform(nq, 16, 72 + nq, np.float32) for nq in (129, 5000, 3000, 60000)]
    return pts, Qs, [oracle.brute_knn(pts, Q, 33) for Q in Qs]


def enqueue(torch, tree, calls):
    """query_knn_dev(sync=False) for each (Q, k, pad, stream) of `calls`, back to back.  Every buffer is allocated and
    filled first (an allocation could synchronise the device); then each stream waits for the fills on torch's current
    stream -- and for nothing else -- and the calls are issued.  Returns the Guarded outputs (the query buffers live in
    their closure until the caller has synchronised)."""
    prep = [(poisoned_queries(torch, Q, pad), Guarded(torch, Q.shape[0], k, Q.dtype)) for Q, k, pad, _ in calls]
    for _, _, _, stream in calls:
        stream.wait_stream(torch.cuda.current_stream())
    outs = []
    for ((buf, qp, s), out), (Q, k, _, stream) in zip(prep, calls):
        tree.query_knn_dev(qp, Q.shape[0], s, k, out.ip, out.dp, stream=stream.cuda_stream, sync=False)
        assert tree.counters()["queries"] == Q.shape[0]
        out.keep = buf
        outs.append(out)
    return outs


def test_async_calls_grow_workspaces(pn, torch, d16):
    """Two unsynchronised calls on one handle and one stream, the second with more queries and a larger k: the
    workspaces grow while the first call may still run."""
    pts, Qs, ref = d16
    tree = pn.BallTree.euclidean(pts, prune=PN_PRUNE_OFF)
    st = torch.cuda.Stream()
    a, b = enqueue(torch, tree, [(Qs[1], 10, 3, st), (Qs[3], 33, 13, st)])
    st.synchronize()
    for out, (oi, od), k in ((a, ref[1], 10), (b, ref[3], 33)):
        idx, dist = out.result()
        assert_knn_equal(idx, dist, oi[:, :k], od[:, :k], f"async k={k}")


def test_async_calls_on_two_streams_then_host_call(pn, torch, d16):
    """sync=False on stream A (60 000 queries, three passes: still running when the next call is issued), then on
    stream B with smaller workspaces than A's (so no allocation synchronises the device): the handle must wait for A
    before B reuses A's workspaces.  Then again on A, and a host-buffer query_batch right after that unsynchronised
    call."""
    pts, Qs, ref = d16
    tree = pn.BallTree.euclidean(pts, prune=PN_PRUNE_OFF)
    sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
    a, b, c = enqueue(torch, tree, [(Qs[3], 33, 1, sa), (Qs[1], 17, 3, sb), (Qs[2], 10, 13, sa)])
    hi, hd = tree.query_batch(Qs[1], 16)
    sa.synchronize()
    sb.synchronize()
    for out, (oi, od), tag in ((a, ref[3], "A k=33"), (b, ref[1], "B k=17"), (c, ref[2], "A again k=10")):
        idx, dist = out.result()
        assert_knn_equal(idx, dist, oi[:, :out.k], od[:, :out.k], f"two streams, call {tag}")
    assert_knn_equal(hi, hd, ref[1][0][:, :16], ref[1][1][:, :16], "host call after async")


def test_sessions_on_own_streams_and_threads(pn, torch, d16):
    pts, Qs, ref = d16
    tree = pn.BallTree.euclidean(pts)
    sessions = [tree.session(), tree.session()]
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    bufs = [poisoned_queries(torch, Qs[t + 1], 3) for t in range(2)]
    outs = [Guarded(torch, Qs[t + 1].shape[0], 17, np.float32) for t in range(2)]
    torch.cuda.synchronize()
    errors = []

    def work(t):
        try:
            for _ in range(3):
                sessions[t].query_knn_dev(bufs[t][1], Qs[t + 1].shape[0], bufs[t][2], 17, outs[t].ip, outs[t].dp,
                                          stream=streams[t].cuda_stream, sync=False)
            streams[t].synchronize()
        except Exception as e:  # surfaced below: a failing thread must fail the test
            errors.append(e)

    th = [threading.Thread(target=work, args=(t,)) for t in range(2)]
    [x.start() for x in th]
    [x.join() for x in th]
    assert not errors, errors
    for t in range(2):
        idx, dist = outs[t].result()
        assert_knn_equal(idx, dist, ref[t + 1][0][:, :17], ref[t + 1][1][:, :17], f"session {t}")
        assert sessions[t].counters()["queries"] == Qs[t + 1].shape[0]


@pytest.mark.parametrize("engine", ["warp_f32_d5", "dense_d16"])
def test_noops_and_bad_stride(pn, torch, engine):
    kind, dtype, _, d, _, opts, _ = ENGINES[engine]
    rng = np.random.default_rng(1)
    pts, Q = rng.random((3000, d)).astype(dtype), rng.random((50, d)).astype(dtype)
    tree = pn.BallTree.euclidean(pts, **opts)
    buf, qp, s = poisoned_queries(torch, Q, 3)
    out = Guarded(torch, 50, 10, dtype)
    torch.cuda.synchronize()
    tree.query_knn_dev(qp, 0, s, 10, out.ip, out.dp)
    tree.query_knn_dev(qp, 50, s, 0, out.ip, out.dp)
    tree.query_self_dev(0, out.ip, out.dp)
    torch.cuda.synchronize()
    assert out.untouched()
    with pytest.raises(pn.EngineError) as e:
        tree.query_knn_dev(qp, 50, d - 1, 10, out.ip, out.dp)
    assert e.value.status == 3   # PN_BAD_ARG
    torch.cuda.synchronize()
    assert out.untouched()


# ------------------------------------------------------------------ the benchmarked call at full size
def test_c2_one_async_call_full_size(pn, torch, oracle):
    """BASELINE config 2 as bench.py runs it: 1M x 16 f32 points, 1M queries, k = 10, ONE query_knn_dev(sync=False) on
    a user stream -- the seeded d = 16 scan over many waves and a split tail.  Bit-identical to the host-buffer call on
    every row, distances that recompute with the sequential f32 fold, exact against the oracle on samples and on the
    last 64 rows (the tail launch)."""
    from petal_neighbors_b200 import synth
    n = nq = 1_000_000
    d, k = 16, 10
    pts = synth.uniform(n, d, 2, np.float32)
    Q = synth.uniform(nq, d, 3, np.float32)
    tree = pn.BallTree.euclidean(pts)
    assert tree.info()["prune_seeded"] == 1, tree.info()
    st = torch.cuda.Stream()
    qd = torch.from_numpy(Q).cuda()
    idx_d = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    dist_d = torch.empty((nq, k), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    tree.query_knn_dev(qd.data_ptr(), nq, d, k, idx_d.data_ptr(), dist_d.data_ptr(), stream=st.cuda_stream, sync=False)
    assert tree.counters()["queries"] == nq
    st.synchronize()
    idx, dist = idx_d.cpu().numpy().view(np.uint64), dist_d.cpu().numpy()
    hi, hd = tree.query_batch(Q, k)
    assert np.array_equal(idx, hi) and np.array_equal(bits(dist), bits(hd))
    rows = np.arange(0, nq, 37)
    acc = np.zeros((rows.size, k), np.float32)
    for j in range(d):
        diff = Q[rows, j][:, None] - pts[idx[rows].astype(np.int64), j]
        acc = acc + diff * diff
    assert np.array_equal(bits(np.sqrt(acc)), bits(dist[rows]))
    sample = np.concatenate([np.arange(0, nq, 2503)[:400], np.arange(nq - 64, nq)])
    oi, od = oracle.brute_knn(pts, Q[sample], k)
    assert_knn_equal(idx[sample], dist[sample], oi, od, "c2 sample")
