"""petal_neighbors_b200 -- host-side mirror of the petal-neighbors API over libpetal_b200.so.

The reference is a Rust crate (petabi/petal-neighbors v0.18.0); no Rust toolchain exists in this
image, so this Python module is the tested host binding of the C ABI (include/petal_b200.h) and
mirrors the reference's public surface name for name:

    petal_neighbors::BallTree::{euclidean, new, query, query_nearest, query_radius,
                                num_points}                       src/ball_tree.rs:26-142, 351-373
    petal_neighbors::VantagePointTree::{euclidean, new, query_nearest}
                                                                  src/vantage_point_tree.rs:21-98
    petal_neighbors::ArrayError::{Empty, NotContiguous}           src/lib.rs:9-16
    petal_neighbors::distance::{Metric, Euclidean}                src/distance.rs:9-55

plus the batched additions (`query_batch`, `query_nearest_batch`, `query_radius_batch`) that a
GPU engine needs; the single-point methods are batches of one.  The batched calls also take a torch CUDA tensor of
queries on the tree's device: they then run on torch's current stream and return CUDA tensors (int64 indices, -1 where
the host path pads with 2^64 - 1; distances in the tree's dtype; radius search: int64 offsets and indices).  All compute happens in the CUDA
library; nothing here falls back to the CPU.  (The Rust crate that binds the same ABI is under
rust/petal-neighbors-b200/, see INTEGRATION.md.)
"""
from __future__ import annotations

import ctypes as C
import weakref

import numpy as np

from . import _ffi
from . import distance
from ._ffi import (PN_ALGO_AUTO, PN_ALGO_SIMT, PN_ALGO_TENSOR, PN_BUILDER_AUTO, PN_BUILDER_HOST, PN_BUILDER_DEVICE,
                   PN_PRUNE_AUTO, PN_PRUNE_ON, PN_PRUNE_OFF,
                   PN_PARTITION_AUTO, PN_PARTITION_REFERENCE, PN_PARTITION_TWO_MEANS)

__all__ = ["BallTree", "VantagePointTree", "ArrayError", "EngineError", "distance", "merge_topk_dev", "merge_radius_dev",
           "PN_ALGO_AUTO", "PN_ALGO_SIMT", "PN_ALGO_TENSOR", "PN_BUILDER_AUTO", "PN_BUILDER_HOST", "PN_BUILDER_DEVICE", "PN_PRUNE_AUTO", "PN_PRUNE_ON", "PN_PRUNE_OFF",
           "PN_PARTITION_AUTO", "PN_PARTITION_REFERENCE", "PN_PARTITION_TWO_MEANS"]


class ArrayError(Exception):
    """The error type for input arrays (src/lib.rs:9-16)."""
    Empty = "Empty"
    NotContiguous = "NotContiguous"

    def __init__(self, kind: str):
        self.kind = kind
        super().__init__("array is empty" if kind == ArrayError.Empty else "array is not contiguous in memory")


class EngineError(RuntimeError):
    """Any non-ArrayError status of the C ABI (the Rust shim panics on these)."""

    def __init__(self, status: int, message: str):
        self.status = status
        super().__init__(f"petal_b200 status {status}: {message}")


def _check(status: int):
    if status == _ffi.PN_OK:
        return
    if status == _ffi.PN_EMPTY:
        raise ArrayError(ArrayError.Empty)
    if status == _ffi.PN_NOT_CONTIGUOUS:
        raise ArrayError(ArrayError.NotContiguous)
    raise EngineError(status, _ffi.last_error())


def _sfx(dtype):
    if dtype == np.float32:
        return "f32"
    if dtype == np.float64:
        return "f64"
    raise TypeError(f"A must be f32 or f64 (got {dtype})")


def _strides(a):
    it = a.dtype.itemsize
    rs = a.strides[0] // it if a.shape[0] > 1 else max(a.shape[1], 1)
    cs = a.strides[1] // it if a.shape[1] > 1 else 1
    return rs, cs


_CUDA_STREAM_LEGACY = 1   # cudaStreamLegacy
# the largest first index buffer of a CUDA-tensor radius search (1 GiB of int64): a larger result is completed by
# re-issuing the queries that did not fit, so the cap bounds memory, not the result
_RADIUS_GUESS_MAX = 1 << 27


def _is_cuda_tensor(x):
    return hasattr(x, "data_ptr") and getattr(x, "is_cuda", False)


def _csr_arrays(offs_p, idx_p, nq):
    """The engine-allocated CSR result of a radius call as numpy arrays (offsets[nq + 1], indices), zero-copy: the buffers
    back the arrays and are released with pn_free when the arrays are garbage-collected (the Rust shim's
    Vec::from_raw_parts equivalent)."""
    L = _ffi.lib()
    offsets = np.ctypeslib.as_array(offs_p, shape=(nq + 1,))
    weakref.finalize(offsets, L.pn_free, C.cast(offs_p, C.c_void_p))
    total = int(offsets[-1])
    if total:
        indices = np.ctypeslib.as_array(idx_p, shape=(total,))
        weakref.finalize(indices, L.pn_free, C.cast(idx_p, C.c_void_p))
    else:
        indices = np.empty(0, np.uint64)
        L.pn_free(idx_p)
    return offsets, indices


class _Tree:
    _kind = "balltree"

    def __init__(self, points, metric=None, *, device=-1, bucket_size=0, algo=PN_ALGO_AUTO, host_threads=0,
                 host_only=False, shard_depth=0, shard_index=0, builder=PN_BUILDER_AUTO, prune=PN_PRUNE_AUTO,
                 partition=PN_PARTITION_AUTO):
        if metric is not None and not isinstance(metric, distance.Euclidean):
            raise TypeError("only distance.Euclidean is offered by the B200 engine (Cosine is not a metric; "
                            "there is no CPU fallback)")
        opts = _ffi.BuildOpts()
        opts.struct_size = C.sizeof(_ffi.BuildOpts)
        opts.device = device
        opts.bucket_size = bucket_size
        opts.algo = algo
        opts.host_threads = host_threads
        opts.flags = _ffi.PN_FLAG_HOST_ONLY if host_only else 0
        opts.shard_depth = shard_depth
        opts.shard_index = shard_index
        opts.builder = builder
        opts.prune = prune
        opts.partition = partition
        self._h = C.c_void_p()
        self.metric = metric if metric is not None else distance.Euclidean()
        if hasattr(points, "data_ptr") and getattr(points, "is_cuda", False):
            # a CUDA tensor (torch): the points stay on the device and the tree is built there
            if self._kind != "balltree":
                raise TypeError("device-resident construction is a BallTree feature")
            if points.dim() != 2 or (points.shape[1] > 1 and points.stride(1) != 1):
                raise ValueError("points must be a 2-D tensor with unit column stride")
            self.dtype = np.dtype(str(points.dtype).replace("torch.", ""))
            self._sfx = _sfx(self.dtype)
            n, d = int(points.shape[0]), int(points.shape[1])
            if opts.device < 0:
                opts.device = points.device.index
            fn = getattr(_ffi.lib(), f"pn_balltree_create_dev_{self._sfx}")
            _check(fn(points.data_ptr(), n, d, int(points.stride(0)) if n > 1 else max(d, 1), C.byref(opts), C.byref(self._h)))
            self.dim = d
            return
        points = np.asarray(points)
        if points.ndim != 2:
            raise ValueError("points must be a 2-D array")
        self.dtype = points.dtype
        self._sfx = _sfx(points.dtype)
        n, d = points.shape
        if n and d and (points.strides[0] < 0 or points.strides[1] < 0):
            points = np.ascontiguousarray(points)
        rs, cs = _strides(points) if n else (d, 1)
        L = _ffi.lib()
        fn = getattr(L, f"pn_{self._kind}_create_{self._sfx}")
        _check(fn(points.ctypes.data if n else None, n, d, rs, cs, C.byref(opts), C.byref(self._h)))
        self.dim = d

    # BallTree::euclidean src/ball_tree.rs:367-373 / VantagePointTree::euclidean src/vantage_point_tree.rs:31-36
    @classmethod
    def euclidean(cls, points, **opts):
        return cls(points, distance.Euclidean(), **opts)

    # BallTree::new src/ball_tree.rs:38 / VantagePointTree::new src/vantage_point_tree.rs:51
    @classmethod
    def new(cls, points, metric, **opts):
        return cls(points, metric, **opts)

    def session(self):
        """pn_tree_session: a second handle onto the same device-resident tree with its own stream and workspaces, for
        a concurrent caller (the reference's `&self` queries from several threads).  Nothing of the tree is copied."""
        other = object.__new__(type(self))
        other._h = C.c_void_p()
        other.metric, other.dtype, other._sfx, other.dim = self.metric, self.dtype, self._sfx, self.dim
        _check(_ffi.lib().pn_tree_session(self._h, C.byref(other._h)))
        return other

    def close(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            _ffi.lib().pn_tree_destroy(h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def info(self) -> dict:
        s = _ffi.TreeInfo()
        _check(_ffi.lib().pn_tree_get_info(self._h, C.byref(s)))
        return _ffi._struct_dict(s)

    def counters(self) -> dict:
        s = _ffi.Counters()
        _check(_ffi.lib().pn_tree_get_counters(self._h, C.byref(s)))
        return _ffi._struct_dict(s)

    def num_points(self) -> int:  # src/ball_tree.rs:351-353
        return int(self.info()["n_points_total"])

    def layout(self) -> dict:
        """Copy of the flattened GPU layout (builder tests)."""
        inf = self.info()
        n, nb, nn, dp = inf["n_points"], inf["n_buckets"], inf["n_nodes"], inf["dim_padded"]
        ids = np.empty(n, np.uint32)
        blo = np.empty(nb, np.uint32)
        bhi = np.empty(nb, np.uint32)
        rad = np.empty(nn, self.dtype)
        cen = np.empty((nn, dp), self.dtype)
        pts = np.empty((n, dp), self.dtype)
        _check(_ffi.lib().pn_tree_get_layout(self._h, ids.ctypes.data, blo.ctypes.data, bhi.ctypes.data,
                                             rad.ctypes.data, cen.ctypes.data, pts.ctypes.data))
        return dict(ids=ids, bucket_lo=blo, bucket_hi=bhi, node_radius=rad, node_center=cen, points=pts, **inf)

    def _queries(self, Q):
        Q = np.asarray(Q, dtype=self.dtype)
        if Q.ndim != 2:
            raise ValueError("queries must be 2-D (nq x d)")
        if Q.shape[1] != self.dim:
            raise ValueError(f"query dimension {Q.shape[1]} != tree dimension {self.dim}")
        if Q.shape[0] and (Q.strides[1] != Q.dtype.itemsize and Q.shape[1] > 1 or Q.strides[0] < 0):
            Q = np.ascontiguousarray(Q)
        return Q, (Q.strides[0] // Q.dtype.itemsize if Q.shape[0] > 1 else max(Q.shape[1], 1))

    def _tensor_queries(self, Q):
        """A CUDA tensor of queries on the tree's device, in the tree's dtype and with unit column stride (copied only if
        needed), its row stride, and the handle of the current torch stream of that device.  Torch's default stream is the
        legacy NULL stream, handle 0, which the C API reads as the tree handle's own stream: it is passed as
        cudaStreamLegacy."""
        import torch
        dev = self.info()["device"]
        if Q.device.index != dev:
            raise ValueError(f"queries are on {Q.device}, the tree on cuda:{dev}")
        if Q.dim() != 2:
            raise ValueError("queries must be 2-D (nq x d)")
        if Q.shape[1] != self.dim:
            raise ValueError(f"query dimension {Q.shape[1]} != tree dimension {self.dim}")
        Q = Q.to(torch.float32 if self.dtype == np.float32 else torch.float64)
        nq, d = Q.shape
        if (d > 1 and Q.stride(1) != 1) or (nq > 1 and Q.stride(0) < d):
            Q = Q.contiguous()
        return Q, (Q.stride(0) if nq > 1 else max(d, 1)), torch.cuda.current_stream(Q.device).cuda_stream or _CUDA_STREAM_LEGACY

    def _knn_tensor(self, Q, k):
        """k-NN of CUDA-tensor queries on the current stream, without synchronising: (indices[nq, k] int64, -1 where
        k > n; distances[nq, k] in the tree's dtype)."""
        import torch
        Q, qs, st = self._tensor_queries(Q)
        nq = Q.shape[0]
        idx = torch.empty((nq, k), dtype=torch.int64, device=Q.device)
        dist = torch.empty((nq, k), dtype=Q.dtype, device=Q.device)
        if nq and k:
            self.query_knn_dev(Q.data_ptr(), nq, qs, k, idx.data_ptr(), dist.data_ptr(), stream=st, sync=False)
        return idx, dist

    def _radius_tensor(self, Q, radius):
        """Radius search of CUDA-tensor queries on the current stream: (offsets[nq + 1], indices) int64 CUDA tensors.  The
        indices first go to a buffer sized from the density of this handle's previous tensor call, but never larger than
        nq x (points of the handle) or _RADIUS_GUESS_MAX entries; the one synchronisation reads the total.  If the buffer
        was too small, only the queries that did not fit are issued again, into the exact-size remainder; if it was much
        too large, the indices are returned in a copy of their own size."""
        import torch
        Q, qs, st = self._tensor_queries(Q)
        nq = Q.shape[0]
        offs = torch.empty(nq + 1, dtype=torch.int64, device=Q.device)
        guess = int(nq * getattr(self, "_radius_density", 8.0) * 1.12) + 1024
        cap = min(guess, nq * int(self.info()["n_points"]), _RADIUS_GUESS_MAX)
        idx = torch.empty(cap, dtype=torch.int64, device=Q.device)
        self.query_radius_dev(Q.data_ptr(), nq, qs, radius, offs.data_ptr(), idx.data_ptr(), cap, stream=st,
                              sync=False)
        # the queries written: those whose segment ends at or below cap (a prefix); their end is where the rest goes
        done = torch.searchsorted(offs[1:], cap, right=True).view(1)
        total, done, base = torch.cat([offs[-1:], done, offs.index_select(0, done)]).tolist()
        self._radius_density = total / max(nq, 1)
        if total <= cap:   # a view would keep the whole guess alive as long as the result
            return offs, (idx[:total] if cap - total <= total // 4 else idx[:total].clone())
        out = torch.empty(total, dtype=torch.int64, device=Q.device)
        out[:base] = idx[:base]
        rest = Q[done:]
        self.query_radius_dev(rest.data_ptr(), nq - done, qs, radius, offs[done:].data_ptr(), out[base:].data_ptr(),
                              total - base, stream=st, sync=False)
        offs[done:] += base
        return offs, out

    def _knn(self, fname, Q, k):
        if _is_cuda_tensor(Q):
            return self._knn_tensor(Q, k)
        Q, qs = self._queries(Q)
        nq = Q.shape[0]
        idx = np.empty((nq, k), np.uint64)
        dist = np.empty((nq, k), self.dtype)
        if nq and k:
            fn = getattr(_ffi.lib(), f"{fname}_{self._sfx}")
            if fname.endswith("query"):
                _check(fn(self._h, Q.ctypes.data, nq, qs, k, idx.ctypes.data, dist.ctypes.data))
            else:
                _check(fn(self._h, Q.ctypes.data, nq, qs, idx.ctypes.data, dist.ctypes.data))
        return idx, dist

    def _radius(self, Q, radius):
        if _is_cuda_tensor(Q):
            return self._radius_tensor(Q, radius)
        Q, qs = self._queries(Q)
        nq = Q.shape[0]
        L = _ffi.lib()
        offs_p = C.POINTER(C.c_uint64)()
        idx_p = C.POINTER(C.c_uint64)()
        fn = getattr(L, f"pn_{self._kind}_query_radius_{self._sfx}")
        _check(fn(self._h, Q.ctypes.data if nq else None, nq, qs, self.dtype.type(radius), C.byref(offs_p), C.byref(idx_p)))
        return _csr_arrays(offs_p, idx_p, nq)

    def query_knn_dev(self, q_ptr: int, nq: int, q_row_stride: int, k: int, idx_ptr: int, dist_ptr: int,
                      stream: int = 0, sync: bool = True):
        """Device-pointer k-NN (pn_tree_query_knn_dev): queries/outputs already in HBM."""
        _check(_ffi.lib().pn_tree_query_knn_dev(self._h, q_ptr, nq, q_row_stride, k, idx_ptr, dist_ptr, stream,
                                                1 if sync else 0))

    def query_radius_dev(self, q_ptr: int, nq: int, q_row_stride: int, radius, offsets_ptr: int, indices_ptr: int,
                         capacity: int, stream: int = 0, sync: bool = True):
        """Device-pointer radius search (pn_tree_query_radius_dev): queries and the CSR outputs in HBM.  offsets[nq + 1]
        is always written; query q's indices are written only if offsets[q + 1] <= capacity (a prefix of the batch)."""
        _check(_ffi.lib().pn_tree_query_radius_dev(self._h, q_ptr, nq, q_row_stride, float(self.dtype.type(radius)),
                                                   offsets_ptr, indices_ptr, capacity, stream, 1 if sync else 0))

    def query_self_dev(self, k: int, idx_ptr: int, dist_ptr: int, stream: int = 0, sync: bool = True):
        """Device-pointer self-query (pn_tree_query_self_dev): every stored point is a query, row i of the n x k
        outputs (already in HBM) is the answer for points[i]."""
        _check(_ffi.lib().pn_tree_query_self_dev(self._h, k, idx_ptr, dist_ptr, stream, 1 if sync else 0))


class BallTree(_Tree):
    """petal_neighbors::BallTree<A, Euclidean> on the GPU (src/ball_tree.rs:15-24)."""
    _kind = "balltree"

    def query_batch(self, Q, k: int):
        """Batched BallTree::query: (indices[nq, k] u64, distances[nq, k]); rows padded with
        (2^64-1, +inf) when k > n.
        CUDA-tensor queries (on the tree's device, any float dtype and strides): CUDA tensors on torch's current stream,
        without synchronising; indices int64, -1 where k > n pads; distances in the tree's dtype."""
        return self._knn("pn_balltree_query", Q, int(k))

    def query(self, point, k: int):
        """BallTree::query src/ball_tree.rs:102-121: (indices, distances), ascending, len min(k, n)."""
        idx, dist = self.query_batch(np.asarray(point, dtype=self.dtype)[None, :], k)
        m = min(int(k), self.num_points())
        return idx[0, :m].astype(np.uintp), dist[0, :m]

    def query_self(self, k: int):
        """Every stored point as a query (benches/ball_tree.rs:53-59): (indices[n, k], distances[n, k])."""
        n = self.num_points()
        idx = np.empty((n, k), np.uint64)
        dist = np.empty((n, k), self.dtype)
        if k:
            fn = getattr(_ffi.lib(), f"pn_balltree_query_self_{self._sfx}")
            _check(fn(self._h, k, idx.ctypes.data, dist.ctypes.data))
        return idx, dist

    def query_nearest_batch(self, Q):
        """Batched BallTree::query_nearest: (indices[nq] u64, distances[nq]).  CUDA-tensor queries (on the tree's device): CUDA tensors on torch's current stream, without synchronising;
        indices int64, distances in the tree's dtype."""
        idx, dist = self._knn("pn_balltree_query_nearest", Q, 1)
        return idx[:, 0], dist[:, 0]

    def query_nearest(self, point):
        """BallTree::query_nearest src/ball_tree.rs:80-86: (index, distance)."""
        idx, dist = self.query_nearest_batch(np.asarray(point, dtype=self.dtype)[None, :])
        return int(idx[0]), dist[0]

    def query_radius_batch(self, Q, radius):
        """Batched BallTree::query_radius: CSR (offsets[nq+1], indices), each query's indices
        ascending; strict `distance < radius` (src/ball_tree.rs:277).  Numpy queries: u64 numpy arrays.
        CUDA-tensor queries (on the tree's device): int64 CUDA tensors on torch's current stream; the call
        synchronises once, to read the total."""
        return self._radius(Q, radius)

    def query_radius(self, point, radius):
        """BallTree::query_radius src/ball_tree.rs:137-142 (indices ascending)."""
        _, indices = self.query_radius_batch(np.asarray(point, dtype=self.dtype)[None, :], radius)
        return indices.astype(np.uintp)


class VantagePointTree(_Tree):
    """petal_neighbors::VantagePointTree<A, Euclidean> on the GPU (src/vantage_point_tree.rs:13-18)."""
    _kind = "vptree"

    def query_nearest_batch(self, Q):
        """Batched VantagePointTree::query_nearest: (indices[nq] u64, distances[nq]).  CUDA-tensor queries (on the tree's device): CUDA tensors on torch's current stream, without synchronising;
        indices int64, distances in the tree's dtype."""
        idx, dist = self._knn("pn_vptree_query_nearest", Q, 1)
        return idx[:, 0], dist[:, 0]

    def query_nearest(self, needle):
        """VantagePointTree::query_nearest src/vantage_point_tree.rs:88-98: (index, distance)."""
        idx, dist = self.query_nearest_batch(np.asarray(needle, dtype=self.dtype)[None, :])
        return int(idx[0]), dist[0]

    # Extensions (the reference VP tree has query_nearest only): the answers BallTree gives for the same points.
    def query_batch(self, Q, k: int):
        """k-NN on the vantage-point handle: (indices[nq, k] u64, distances[nq, k]), (distance, index) ascending; rows
        padded with (2^64-1, +inf) when k > n.
        CUDA-tensor queries (on the tree's device, any float dtype and strides): CUDA tensors on torch's current stream,
        without synchronising; indices int64, -1 where k > n pads; distances in the tree's dtype."""
        return self._knn("pn_vptree_query", Q, int(k))

    def query(self, point, k: int):
        idx, dist = self.query_batch(np.asarray(point, dtype=self.dtype)[None, :], k)
        m = min(int(k), self.num_points())
        return idx[0, :m].astype(np.uintp), dist[0, :m]

    def query_radius_batch(self, Q, radius):
        """Radius search on the vantage-point handle: CSR (offsets[nq+1], indices), strict `distance < radius`.  Numpy
        queries: u64 numpy arrays.
        CUDA-tensor queries (on the tree's device): int64 CUDA tensors on torch's current stream; the call
        synchronises once, to read the total."""
        return self._radius(Q, radius)

    def query_radius(self, point, radius):
        _, indices = self.query_radius_batch(np.asarray(point, dtype=self.dtype)[None, :], radius)
        return indices.astype(np.uintp)


def merge_topk_dev(dtype, device: int, idx_lists_ptr: int, dist_lists_ptr: int, n_lists: int, nq: int, k: int,
                   idx_out_ptr: int, dist_out_ptr: int, stream: int = 0, sync: bool = True):
    """pn_merge_topk_dev: k-way merge of per-shard sorted top-k lists (after the all-gather)."""
    code = _ffi.PN_F32 if np.dtype(dtype) == np.float32 else _ffi.PN_F64
    _check(_ffi.lib().pn_merge_topk_dev(code, device, idx_lists_ptr, dist_lists_ptr, n_lists, nq, k, idx_out_ptr,
                                        dist_out_ptr, stream, 1 if sync else 0))


def merge_radius_dev(device: int, offsets_ptr: int, indices_ptr: int, n_lists: int, nq: int, out_offsets_ptr: int,
                     out_indices_ptr: int, stream: int = 0, sync: bool = True):
    """pn_merge_radius_dev: merge of n_lists CSR radius results over the same nq queries (device pointers, u64).
    offsets[n_lists][nq + 1] are absolute positions into the indices; each list's segment of a query is ascending.  The
    merged CSR has each query's indices ascending; equal indices from different lists are all kept, in list order."""
    _check(_ffi.lib().pn_merge_radius_dev(device, offsets_ptr, indices_ptr, n_lists, nq, out_offsets_ptr, out_indices_ptr,
                                          stream, 1 if sync else 0))
