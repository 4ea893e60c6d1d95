"""Radius search above one GPU: pn_merge_radius_dev (the merge of per-shard CSR hit lists) and
MultiGpuBallTree.query_radius_batch (pn_multi_balltree_query_radius_f32) in both shard modes.  Every result must be
bit-identical to one BallTree over all the points.  The merge is checked on one device with several shard trees; the
multi-GPU handle runs on the largest power of two <= 8 of the box's devices (one device: a single rank)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pn():
    import petal_neighbors_b200 as pn
    return pn


def radius_for(pts, q, m):
    """a radius that gives query q about m hits"""
    dd = np.sort(np.sqrt(((pts.astype(np.float64) - q.astype(np.float64)) ** 2).sum(1)))
    return np.float32(dd[min(m, len(dd) - 1)])


def merged_on_device(pn, lists, nq, gap=0):
    """concatenate per-list CSR results (optionally `gap` unused entries before each list) and merge them on cuda:0"""
    import torch
    offs, chunks, pos = [], [], 0
    for o, ind in lists:
        pos += gap
        chunks.append(np.zeros(gap, np.uint64))
        offs.append(o.astype(np.uint64) - o[0] + np.uint64(pos))
        chunks.append(ind.astype(np.uint64))
        pos += len(ind)
    cat = np.concatenate(chunks + [np.zeros(1, np.uint64)])
    total = sum(len(ind) for _, ind in lists)
    d_offs = torch.from_numpy(np.stack(offs).view(np.int64)).cuda(0)
    d_ind = torch.from_numpy(cat.view(np.int64)).cuda(0)
    o_offs = torch.full((nq + 1,), -1, dtype=torch.int64, device="cuda:0")
    o_ind = torch.full((max(total, 1),), -1, dtype=torch.int64, device="cuda:0")
    pn.merge_radius_dev(0, d_offs.data_ptr(), d_ind.data_ptr(), len(lists), nq, o_offs.data_ptr(), o_ind.data_ptr())
    return o_offs.cpu().numpy().view(np.uint64), o_ind.cpu().numpy().view(np.uint64)[:total]


def check_against_oracle(oracle, pts, Q, r, offs, ind, n_sample=40):
    sample = np.unique(np.linspace(0, len(Q) - 1, min(n_sample, len(Q))).astype(int))
    bo, bi = oracle.brute_radius(pts, Q[sample], r)
    for j, qi in enumerate(sample):
        assert np.array_equal(ind[offs[qi]:offs[qi + 1]], bi[bo[j]:bo[j + 1]].astype(np.uint64)), f"query {qi}"


@pytest.mark.parametrize("depth,data", [(2, "uniform"), (3, "clustered")])
def test_merge_of_shard_lists(pn, oracle, depth, data):
    from petal_neighbors_b200 import synth
    n = 150000
    if data == "uniform":
        pts = synth.uniform(n, 3, 81, np.float32)
        Q = synth.uniform(3000, 3, 82, np.float32)
    else:
        pts = synth.gaussian_mixture(n, 16, 83, n_centers=64, sigma=0.02)
        Q = synth.gaussian_mixture(3000, 16, 84, n_centers=64, sigma=0.02)
    Q[-1] = 10.0                                     # far from every point: no hits in any shard
    full = pn.BallTree.euclidean(pts, device=0)
    shards = [pn.BallTree.euclidean(pts, device=0, shard_depth=depth, shard_index=i) for i in range(1 << depth)]
    centre = pts.mean(0, keepdims=True).astype(np.float32)
    cases = [
        (Q, radius_for(pts, Q[0], 30)),                                # most queries hit one or two shards only
        (Q[:60], radius_for(pts, Q[0], 3000)),                         # > 1024 hits, whole nodes inside the ball
        (np.concatenate([centre, Q[:3]]), radius_for(pts, centre[0], 120000)),   # > 10^5 hits for one query
        (Q[5:6], radius_for(pts, Q[5], 500)),                          # nq = 1
    ]
    for Qc, r in cases:
        nq = len(Qc)
        ro, ri = full.query_radius_batch(Qc, r)
        lists = [s.query_radius_batch(Qc, r) for s in shards]
        for gap in (0, 3):
            mo, mi = merged_on_device(pn, lists, nq, gap)
            assert np.array_equal(mo, ro) and np.array_equal(mi, ri), (nq, r, gap)
        check_against_oracle(oracle, pts, Qc, r, ro, ri)
        if nq == 4:
            assert np.diff(ro)[0] > 100000
        elif nq == 60:
            assert np.diff(ro).max() > 1024
        elif nq == 3000:
            assert ro[-1] == ro[-2]
            hit = np.diff(ro) > 0
            assert any(((np.diff(o) == 0) & hit).any() for o, _ in lists)   # hits in some shards only


def test_merge_keeps_duplicates_in_list_order(pn):
    """hand-made lists: equal values in several lists are all kept; u64 values; empty lists and segments"""
    big = np.uint64(1) << np.uint64(40)
    nq = 4
    raw = [
        [[1, 5, 5, 9], [], [big], [2]],
        [[5, 9, 9], [7], [], [2, 2]],
        [[], [], [], []],
        [[0, 5, 10], [7, 7], [big, big + np.uint64(1)], []],
    ]
    lists = []
    for segs in raw:
        ind = np.array([v for s in segs for v in s], np.uint64)
        o = np.concatenate([[0], np.cumsum([len(s) for s in segs])]).astype(np.uint64)
        lists.append((o, ind))
    for gap in (0, 2):
        mo, mi = merged_on_device(pn, lists, nq, gap)
        want = [np.sort(np.array([v for segs in raw for v in segs[q]], np.uint64), kind="stable") for q in range(nq)]
        assert np.array_equal(mo, np.concatenate([[0], np.cumsum([len(w) for w in want])]).astype(np.uint64))
        assert np.array_equal(mi, np.concatenate(want))
    # nq = 0 writes the single offset 0
    mo, mi = merged_on_device(pn, [(np.zeros(1, np.uint64), np.zeros(0, np.uint64))], 0)
    assert mo.tolist() == [0] and len(mi) == 0


def test_merge_with_decreasing_offsets_stays_in_bounds(pn):
    """malformed input (offsets that decrease) may give a wrong result but writes nothing past the documented capacity"""
    import torch
    offs = torch.tensor([[0, 2, 1, 8]], dtype=torch.int64, device="cuda:0")
    ind = torch.arange(8, dtype=torch.int64, device="cuda:0")
    o_offs = torch.zeros(4, dtype=torch.int64, device="cuda:0")
    o_ind = torch.full((8 + 16,), -7, dtype=torch.int64, device="cuda:0")   # capacity 8, then a guard region
    pn.merge_radius_dev(0, offs.data_ptr(), ind.data_ptr(), 1, 3, o_offs.data_ptr(), o_ind.data_ptr())
    assert (o_ind[8:].cpu().numpy() == -7).all()


@pytest.mark.parametrize("mode", [0, 1])
def test_multi_gpu_radius(pn, oracle, mode):
    import torch
    from petal_neighbors_b200 import parallel, synth
    ng = torch.cuda.device_count()
    world = 1 << (min(ng, 8).bit_length() - 1)
    n, d = 120000, 24
    pts = synth.fast_gaussian_mixture(n, d, 91, n_centers=128, sigma=0.05)
    Q = synth.fast_gaussian_mixture(90000, d, 92, n_centers=128, sigma=0.05)
    full = pn.BallTree.euclidean(pts, device=0)
    m = parallel.MultiGpuBallTree(pts, list(range(world)), mode=mode)
    kq = Q[:2000]
    k_before = m.query_batch(kq, 10)
    _, nd = full.query_batch(Q[:200], 50)
    r50 = np.float32(np.median(nd[:, -1]))                       # about 50 hits per query
    r_big = radius_for(pts, Q[0], 3000)                          # overflows the slab and the warp sort
    r_none = np.float32(full.query_batch(Q[:2000], 1)[1].min() * 0.5)
    cases = [(Q[:0], r50), (Q[:1], r50), (Q[:3], r50), (Q, r50), (Q[:300], r_big), (Q[:1000], np.float32(0)), (Q[:1000], r_none)]
    for Qc, r in cases:
        nq = len(Qc)
        offs, ind = m.query_radius_batch(Qc, r)
        ro, ri = full.query_radius_batch(Qc, r)
        assert offs.dtype == np.uint64 and ind.dtype == np.uint64
        assert np.array_equal(offs, ro) and np.array_equal(ind, ri), (mode, nq, r)
        if r in (0, r_none):
            assert not offs.any() and len(ind) == 0
        if nq == 300:
            assert np.diff(offs).max() > 1024 and (np.diff(offs) > 64).sum() > 10
        if nq == 90000:
            check_against_oracle(oracle, pts, Qc, r, offs, ind)
        if nq:
            st = m.stats()
            assert sum(s["rows_out"] for s in st) == nq
            assert all(s["nccl_calls"] == 0 and s["nccl_bytes_sent"] == 0 for s in st)
            if mode == 1 and world > 1 and nq == 90000:
                assert all(s["peer_mib"] > 0 for s in st)
    k_after = m.query_batch(kq, 10)
    assert np.array_equal(k_before[0], k_after[0]) and np.array_equal(k_before[1].view(np.uint32), k_after[1].view(np.uint32))
    m.close()
