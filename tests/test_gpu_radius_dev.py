"""pn_tree_query_radius_dev (radius search from and into device memory) and the CUDA-tensor paths of query_batch /
query_nearest_batch / query_radius_batch.

Offsets and indices must be identical to the host-buffer call (pn_*_query_radius_*), which is itself checked against the
oracle on a sample.  As in test_gpu_device_entry.py, the queries sit in a NaN-filled buffer at a misaligned base with a
row stride wider than d, and the outputs have sentinel regions: before the offsets and after offsets[nq], before the
indices and after `capacity`.  With a capacity below the total, exactly the queries whose segment ends at or below it
must be written, and nothing else."""
import threading

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SENT = 0x5A5A5A5A5A5A5A5A
G = 16   # sentinel entries on each side of an output


@pytest.fixture(scope="module")
def pn():
    import petal_neighbors_b200 as pn
    return pn


@pytest.fixture(scope="module")
def torch():
    import torch
    return torch


def tdtype(torch, dtype):
    return torch.float32 if dtype == np.float32 else torch.float64


def poisoned_queries(torch, Q, pad, stride=None):
    """Q in a NaN-filled device buffer, row stride d + pad (or `stride`), base not 16-byte aligned.  Returns (buffer,
    pointer of row 0, row stride)."""
    nq, d = Q.shape
    s = d + pad if stride is None else stride
    s_rows = max(s, d)
    base = s_rows + (1 if s_rows % 2 == 0 else 2)
    buf = torch.full(((nq + 2) * s_rows + 4,), float("nan"), dtype=tdtype(torch, Q.dtype), device="cuda")
    if nq:
        buf.as_strided((nq, d), (s_rows, 1), base).copy_(torch.from_numpy(np.ascontiguousarray(Q)))
    return buf, buf.data_ptr() + base * Q.itemsize, s


class GuardedCSR:
    """offsets[nq + 1] and indices[capacity] between G sentinel entries on each side."""

    def __init__(self, torch, nq, capacity):
        self.nq, self.cap = nq, capacity
        self.o = torch.full((nq + 1 + 2 * G,), SENT, dtype=torch.int64, device="cuda")
        self.i = torch.full((capacity + 2 * G,), SENT, dtype=torch.int64, device="cuda")
        self.op = self.o.data_ptr() + G * 8
        self.ip = self.i.data_ptr() + G * 8

    def result(self):
        """(offsets u64, indices[capacity] u64) after checking the guards"""
        o = self.o.cpu().numpy().view(np.uint64)
        i = self.i.cpu().numpy().view(np.uint64)
        assert np.all(o[:G] == SENT) and np.all(o[G + self.nq + 1:] == SENT), "offsets guard written"
        assert np.all(i[:G] == SENT) and np.all(i[G + self.cap:] == SENT), "indices guard written"
        return o[G:G + self.nq + 1], i[G:G + self.cap]

    def untouched(self):
        return bool(np.all(self.o.cpu().numpy().view(np.uint64) == SENT) and np.all(self.i.cpu().numpy().view(np.uint64) == SENT))


def radius_dev(torch, tree, Q, r, capacity=None, pad=3, stride=None, null_indices=False, stream=0, sync=True):
    """One query_radius_dev over poisoned queries into guarded outputs; capacity None = the host call's total."""
    if capacity is None:
        capacity = int(tree.query_radius_batch(Q, r)[0][-1])
    buf, qp, s = poisoned_queries(torch, Q, pad, stride)
    out = GuardedCSR(torch, Q.shape[0], capacity)
    torch.cuda.synchronize()
    tree.query_radius_dev(qp, Q.shape[0], s, r, out.op, 0 if null_indices else out.ip, capacity, stream=stream, sync=sync)
    torch.cuda.synchronize()
    return out.result()


def check_against_host(tree, Q, r, offs, ind, capacity=None, tag=""):
    """offsets equal the host call's; exactly the prefix of queries ending at or below capacity is written and equals the
    host result; everything between that prefix and capacity is untouched.  Returns the host result."""
    ho, hi = tree.query_radius_batch(Q, r)
    assert np.array_equal(offs, ho), f"{tag}: offsets differ from the host call"
    cap = int(ho[-1]) if capacity is None else capacity
    done = int(np.searchsorted(ho[1:], cap, side="right"))
    end = int(ho[done])
    assert np.array_equal(ind[:end], hi[:end]), f"{tag}: indices of the written prefix differ from the host call"
    assert np.all(ind[end:cap] == SENT), f"{tag}: entries past the written prefix ({end}) and below capacity were written"
    return ho, hi


def check_oracle(oracle, pts, Q, r, ho, hi, rows):
    bo, bi = oracle.brute_radius(pts, Q[rows], r)
    for j, q in enumerate(rows):
        assert np.array_equal(hi[ho[q]:ho[q + 1]], bi[bo[j]:bo[j + 1]].astype(np.uint64)), f"query {q} differs from the oracle"


def radius_for_hits(pts, Q, k):
    """a radius around which the first queries have about k hits"""
    d2 = ((Q[:8, None, :].astype(np.float64) - pts[None, :, :].astype(np.float64)) ** 2).sum(-1)
    return float(np.median(np.sqrt(np.partition(d2, k, axis=1)[:, k])))


def data(kind, n, nq, d, dtype, seed):
    from petal_neighbors_b200 import synth
    if kind == "clustered":
        return (synth.gaussian_mixture(n, d, seed, n_centers=64, sigma=0.01).astype(dtype),
                synth.gaussian_mixture(nq, d, seed + 1, n_centers=64, sigma=0.01).astype(dtype))
    return synth.uniform(n, d, seed, dtype), synth.uniform(nq, d, seed + 1, dtype)


# ------------------------------------------------------------------ parity with the host call
@pytest.mark.parametrize("kind", ["uniform", "clustered"])
@pytest.mark.parametrize("d", [3, 16, 64])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("cls", ["BallTree", "VantagePointTree"])
def test_parity(pn, torch, oracle, cls, dtype, d, kind):
    pts, Q = data(kind, 12000, 301, d, dtype, 11 + d)
    tree = getattr(pn, cls).euclidean(pts)
    r = radius_for_hits(pts, Q, 80)
    offs, ind = radius_dev(torch, tree, Q, r)
    ho, hi = check_against_host(tree, Q, r, offs, ind, tag=f"{cls} {np.dtype(dtype)} d={d} {kind}")
    assert np.diff(ho).max() > 64, "no query reached the second traversal"
    check_oracle(oracle, pts, Q, dtype(r), ho, hi, np.arange(0, 301, 10))


def test_session_and_shard(pn, torch, oracle):
    pts, Q = data("uniform", 20000, 500, 8, np.float32, 5)
    r = radius_for_hits(pts, Q, 100)
    tree = pn.BallTree.euclidean(pts)
    sess = tree.session()
    offs, ind = radius_dev(torch, sess, Q, r)
    ho, hi = check_against_host(tree, Q, r, offs, ind, tag="session")
    check_oracle(oracle, pts, Q, np.float32(r), ho, hi, np.arange(0, 500, 25))
    bo, bi = oracle.brute_radius(pts, Q, np.float32(r))
    shard_total = 0
    for s in range(4):
        shard = pn.BallTree.euclidean(pts, shard_depth=2, shard_index=s)
        so, si = radius_dev(torch, shard, Q, r)
        sho, shi = check_against_host(shard, Q, r, so, si, tag=f"shard {s}")
        for q in range(0, 500, 7):   # global indices: a subset of the whole tree's hits
            assert np.all(np.isin(shi[sho[q]:sho[q + 1]], bi[bo[q]:bo[q + 1]].astype(np.uint64)))
        shard_total += int(sho[-1])
    assert shard_total == int(bo[-1])


# ------------------------------------------------------------------ hit regimes and batch sizes
@pytest.fixture(scope="module")
def d3(pn):
    """uniform d = 3 points plus a dense clump (queries inside it have thousands of hits), and a far-away query"""
    from petal_neighbors_b200 import synth
    pts = synth.uniform(60000, 3, 21, np.float32)
    pts[:4000] = np.float32(0.5) + np.float32(0.002) * synth.uniform(4000, 3, 22, np.float32)
    Q = synth.uniform(999, 3, 23, np.float32)
    Q[::50] = np.float32(0.501)
    Q[7] = np.float32(1000.0)
    return pts, Q, pn.BallTree.euclidean(pts)


@pytest.mark.parametrize("regime,r,lo,hi", [("zero", 0.0, 0, 0), ("slab", 0.03, 1, 64), ("overflow", 0.08, 65, 1024),
                                            ("large", 0.2, 1025, None)])
def test_hit_regimes(torch, oracle, d3, regime, r, lo, hi):
    """r = 0 and the far query: no hits; some uniform queries at the given radius land in the named regime (slab only,
    second traversal, block sort); the clump queries have thousands of hits from whole nodes inside the ball."""
    pts, Q, tree = d3
    offs, ind = radius_dev(torch, tree, Q, r)
    ho, hi_ = check_against_host(tree, Q, r, offs, ind, tag=regime)
    cnt = np.diff(ho.astype(np.int64))
    assert cnt[7] == 0
    uni = np.ones(Q.shape[0], bool)
    uni[::50] = False
    uni[7] = False
    if hi == 0:
        assert ho[-1] == 0
    else:
        c = cnt[uni]
        assert np.any((c >= lo) & (c <= (hi or c.max()))), f"{regime}: no uniform query with {lo}..{hi} hits"
        assert cnt[::50].min() > 1024
    check_oracle(oracle, pts, Q, np.float32(r), ho, hi_, np.concatenate([np.arange(0, 999, 37), [7, 50, 100]]))


@pytest.mark.parametrize("nq", [0, 1, 777, (1 << 18) + (1 << 17) + 123])
def test_batch_sizes(pn, torch, oracle, nq):
    from petal_neighbors_b200 import synth
    pts = synth.uniform(100000, 3, 31, np.float32)
    tree = pn.BallTree.euclidean(pts)
    Q = synth.uniform(nq, 3, 32, np.float32)
    r = 0.025
    offs, ind = radius_dev(torch, tree, Q, r, stride=0 if nq == 1 else None)
    ho, hi = check_against_host(tree, Q, r, offs, ind, tag=f"nq={nq}")
    assert offs[0] == 0 and offs.size == nq + 1
    if nq > (1 << 18):
        for c in range(4):   # every chunk of 2^17 queries has hits
            q0 = c << 17
            assert ho[min(q0 + (1 << 17), nq)] > ho[q0]
        rows = np.concatenate([np.arange(c << 17, (c << 17) + 8) for c in range(4)] + [np.arange(nq - 8, nq)])
        check_oracle(oracle, pts, Q, np.float32(r), ho, hi, rows)
    elif nq:
        check_oracle(oracle, pts, Q, np.float32(r), ho, hi, np.arange(0, nq, max(1, nq // 40)))


# ------------------------------------------------------------------ capacity
@pytest.mark.parametrize("which", ["total", "total-1", "mid", "zero-null"])
def test_capacity(pn, torch, d3, which):
    """Several chunks (nq > 2^18) with clump queries (block sort) and overflowing queries in each"""
    from petal_neighbors_b200 import synth
    pts, _, tree = d3
    nq = (1 << 18) + 5000
    Q = synth.uniform(nq, 3, 41, np.float32)
    Q[::997] = np.float32(0.501)
    r = 0.03
    ho, _ = tree.query_radius_batch(Q, r)
    total = int(ho[-1])
    cap = {"total": total, "total-1": total - 1, "mid": int(ho[(1 << 17) + 1234]) + 17, "zero-null": 0}[which]
    offs, ind = radius_dev(torch, tree, Q, r, capacity=cap, null_indices=which == "zero-null")
    check_against_host(tree, Q, r, offs, ind, capacity=cap, tag=which)


# ------------------------------------------------------------------ streams and sessions
def test_no_synchronisation(pn, torch, d3):
    """A sync=0 call enqueued behind half a second of spinning on its stream returns while the stream is still busy"""
    pts, Q, tree = d3
    r = 0.03
    buf, qp, s = poisoned_queries(torch, Q, 3)
    total = int(tree.query_radius_batch(Q, r)[0][-1])
    out = GuardedCSR(torch, Q.shape[0], total)
    st = torch.cuda.Stream()
    torch.cuda.synchronize()
    tree.query_radius_dev(qp, Q.shape[0], s, r, out.op, out.ip, total, stream=st.cuda_stream, sync=False)   # warm-up
    st.synchronize()
    out.o.fill_(SENT)
    out.i.fill_(SENT)
    torch.cuda.synchronize()
    with torch.cuda.stream(st):
        torch.cuda._sleep(1_000_000_000)   # about half a second at the B200's clocks
    tree.query_radius_dev(qp, Q.shape[0], s, r, out.op, out.ip, total, stream=st.cuda_stream, sync=False)
    assert not st.query(), "the call waited for its stream"
    st.synchronize()
    offs, ind = out.result()
    check_against_host(tree, Q, r, offs, ind, tag="no sync")


def test_sessions_on_threads(pn, torch, d3):
    pts, Q, tree = d3
    radii = (0.02, 0.04)
    sessions = [tree.session(), tree.session()]
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    totals = [int(tree.query_radius_batch(Q, r)[0][-1]) for r in radii]
    bufs = [poisoned_queries(torch, Q, 5) for _ in range(2)]
    outs = [GuardedCSR(torch, Q.shape[0], totals[t]) for t in range(2)]
    torch.cuda.synchronize()
    errors = []

    def work(t):
        try:
            for _ in range(3):
                sessions[t].query_radius_dev(bufs[t][1], Q.shape[0], bufs[t][2], radii[t], outs[t].op, outs[t].ip,
                                             totals[t], stream=streams[t].cuda_stream, sync=False)
            streams[t].synchronize()
        except Exception as e:  # surfaced below: a failing thread must fail the test
            errors.append(e)

    th = [threading.Thread(target=work, args=(t,)) for t in range(2)]
    [x.start() for x in th]
    [x.join() for x in th]
    assert not errors, errors
    for t in range(2):
        offs, ind = outs[t].result()
        check_against_host(tree, Q, radii[t], offs, ind, tag=f"session {t}")


def test_errors(pn, torch):
    pts = np.random.default_rng(3).random((3000, 4)).astype(np.float32)
    Q = np.random.default_rng(4).random((50, 4)).astype(np.float32)
    tree = pn.BallTree.euclidean(pts)
    buf, qp, s = poisoned_queries(torch, Q, 3)
    out = GuardedCSR(torch, 50, 100)
    torch.cuda.synchronize()
    for args, status in (((qp, 50, s, 0.1, 0, out.ip, 100), 3),          # NULL offsets
                         ((qp, 50, s, 0.1, out.op, 0, 100), 3),          # NULL indices with capacity > 0
                         ((qp, 50, 3, 0.1, out.op, out.ip, 100), 3)):    # stride < d
        with pytest.raises(pn.EngineError) as e:
            tree.query_radius_dev(*args)
        assert e.value.status == status
    host = pn.BallTree.euclidean(pts, host_only=True)
    with pytest.raises(pn.EngineError) as e:
        host.query_radius_dev(qp, 50, s, 0.1, out.op, out.ip, 100)
    assert e.value.status == 4   # PN_CUDA
    torch.cuda.synchronize()
    assert out.untouched()


# ------------------------------------------------------------------ CUDA-tensor queries through the Python trees
@pytest.mark.parametrize("cls", ["BallTree", "VantagePointTree"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_tensor_path(pn, torch, cls, dtype):
    pts, Q = data("uniform", 20000, 2100, 16, dtype, 51)
    tree = getattr(pn, cls).euclidean(pts)
    Qt = torch.from_numpy(Q).cuda()
    for k in (1, 10, 33):
        ti, td = tree.query_batch(Qt, k)
        hi, hd = tree.query_batch(Q, k)
        assert ti.is_cuda and ti.dtype == torch.int64 and td.dtype == tdtype(torch, dtype)
        assert np.array_equal(ti.cpu().numpy().view(np.uint64), hi) and np.array_equal(td.cpu().numpy(), hd)
    ti, td = tree.query_nearest_batch(Qt)
    hi, hd = tree.query_nearest_batch(Q)
    assert np.array_equal(ti.cpu().numpy().view(np.uint64), hi) and np.array_equal(td.cpu().numpy(), hd)
    r = radius_for_hits(pts, Q, 50)
    to, tx = tree.query_radius_batch(Qt, r)
    ho, hx = tree.query_radius_batch(Q, r)
    assert to.dtype == torch.int64 and tx.dtype == torch.int64
    assert np.array_equal(to.cpu().numpy().view(np.uint64), ho) and np.array_equal(tx.cpu().numpy().view(np.uint64), hx)
    # other element type and non-contiguous rows: converted as the numpy path converts
    other = np.float64 if dtype == np.float32 else np.float32
    wide = torch.from_numpy(np.repeat(Q.astype(other), 2, axis=1)).cuda()[:, ::2]
    assert not wide.is_contiguous()
    ti, td = tree.query_batch(wide, 10)
    hi, hd = tree.query_batch(Q.astype(other), 10)
    assert np.array_equal(ti.cpu().numpy().view(np.uint64), hi) and np.array_equal(td.cpu().numpy(), hd)
    to, tx = tree.query_radius_batch(wide.t().contiguous().t(), r)
    ho, hx = tree.query_radius_batch(Q.astype(other), r)
    assert np.array_equal(to.cpu().numpy().view(np.uint64), ho) and np.array_equal(tx.cpu().numpy().view(np.uint64), hx)
    # k > n: -1 where the host path pads with 2^64 - 1
    small = getattr(pn, cls).euclidean(pts[:5])
    ti, td = small.query_batch(Qt[:9], 8)
    hi, hd = small.query_batch(Q[:9], 8)
    assert np.all(ti[:, 5:].cpu().numpy() == -1) and np.array_equal(ti.cpu().numpy().view(np.uint64), hi)
    assert np.array_equal(td.cpu().numpy(), hd)


@pytest.mark.parametrize("side", [False, True], ids=["default_stream", "side_stream"])
def test_tensor_radius_small_capacity_guess(pn, torch, d3, side):
    """After a call without hits the capacity guess is tiny (1024 entries): the queries that did not fit are issued
    again.  The batch starts with uniform queries, so that a prefix fits.  On a side stream, the calls, the torch ops
    between them (searchsorted, the copy of the prefix, the rebasing of the offsets) and k-NN must all run on the current
    stream, behind a spin kernel already queued there."""
    pts, Q, tree = d3
    Q = Q[1:]
    Qt = torch.from_numpy(Q).cuda()
    s = torch.cuda.Stream() if side else torch.cuda.current_stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        to, tx = tree.query_radius_batch(Qt, 0.0)
        assert int(to[-1]) == 0 and tx.numel() == 0
        if side:
            torch.cuda._sleep(50_000_000)   # a few tens of milliseconds of work ahead of the call on its stream
        to, tx = tree.query_radius_batch(Qt, 0.06)
        assert 0 < tree.counters()["queries"] < Q.shape[0], "the second call was not issued for a suffix of the batch"
        if side:
            torch.cuda._sleep(50_000_000)
        ti, td = tree.query_batch(Qt, 10)
    s.synchronize()
    ho, hx = tree.query_radius_batch(Q, 0.06)
    assert np.array_equal(to.cpu().numpy().view(np.uint64), ho) and np.array_equal(tx.cpu().numpy().view(np.uint64), hx)
    hi, hd = tree.query_batch(Q, 10)
    assert np.array_equal(ti.cpu().numpy().view(np.uint64), hi) and np.array_equal(td.cpu().numpy(), hd)


def test_tensor_radius_guess_bounded(pn, torch, d3):
    """A dense call followed by a large, sparse batch on the same handle: the first index buffer is bounded (1 GiB of
    int64, where the previous density would ask for tens of GB), and the result comes back in a buffer of its own size"""
    from petal_neighbors_b200 import synth
    pts, Q, tree = d3
    sess = tree.session()   # a handle of its own: its density history starts here
    to, _ = sess.query_radius_batch(torch.from_numpy(Q).cuda(), 0.3)
    assert int(to[-1]) > 1000 * Q.shape[0]   # the unclamped guess for the next call would be several GB
    big = synth.uniform(400_000, 3, 61, np.float32)
    bt = torch.from_numpy(big).cuda()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    before = torch.cuda.memory_allocated()
    to, tx = sess.query_radius_batch(bt, 0.005)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - before
    assert peak <= (1 << 30) + (64 << 20), f"{peak} bytes for the first index buffer"
    assert tx.untyped_storage().nbytes() == int(to[-1]) * 8, "the result keeps the oversized guess alive"
    ho, hx = sess.query_radius_batch(big, 0.005)
    assert np.array_equal(to.cpu().numpy().view(np.uint64), ho) and np.array_equal(tx.cpu().numpy().view(np.uint64), hx)


@pytest.mark.parametrize("cls", ["BallTree", "VantagePointTree"])
def test_tensor_empty_batch(pn, torch, cls):
    pts = np.random.default_rng(2).random((3000, 3)).astype(np.float32)
    tree = getattr(pn, cls).euclidean(pts)
    Qt = torch.empty((0, 3), device="cuda")
    to, tx = tree.query_radius_batch(Qt, 0.1)
    assert to.tolist() == [0] and tx.numel() == 0 and to.dtype == tx.dtype == torch.int64
    ti, td = tree.query_batch(Qt, 5)
    assert ti.shape == (0, 5) and td.shape == (0, 5) and ti.dtype == torch.int64
    ni, nd = tree.query_nearest_batch(Qt)
    assert ni.shape == (0,) and nd.shape == (0,)


def test_tensor_on_other_device(pn, torch):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    pts = np.random.default_rng(1).random((2000, 4)).astype(np.float32)
    tree = pn.BallTree.euclidean(pts, device=0)
    Qt = torch.rand((10, 4), device="cuda:1")
    for call in (lambda: tree.query_batch(Qt, 3), lambda: tree.query_nearest_batch(Qt), lambda: tree.query_radius_batch(Qt, 0.1)):
        with pytest.raises(ValueError):
            call()
