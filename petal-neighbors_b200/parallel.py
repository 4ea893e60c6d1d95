"""Multi-GPU drivers: one process per GPU (SURVEY.md 8e).  The collectives run INSIDE the library over NCCL
(include/petal_b200.h: pn_comm_*, pn_sharded_query_knn_dev, pn_tree_replicate); torch.distributed is only the
out-of-band channel that ships the 128-byte NCCL unique id from rank 0 to the other ranks.

* Query sharding (default whenever the flattened tree fits one GPU): the tree is replicated -- built once and sent with
  ncclBroadcast (`replicate`) or rebuilt per rank -- the queries are split into contiguous slices, and there is NO
  data-path collective.
* Point sharding by subtree ("points larger than one GPU's HBM"): rank r keeps subtree r at depth log2(world) of the
  ball tree (pn_build_opts.shard_depth / shard_index, the reference's mid = (start+end)/2 split,
  src/ball_tree.rs:535-537); every rank scans ALL queries on its shard in chunks, the per-shard sorted lists of chunk i
  cross NVLink (ncclAllGather, or grouped ncclSend/ncclRecv towards the owner of each query slice) while chunk i+1 is
  scanned, and a k-way merge kernel produces the final rows.

Nothing here computes distances or selections on the CPU.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch
import torch.distributed as dist

from . import BallTree, _Tree, _check, _csr_arrays, _ffi, merge_radius_dev, merge_topk_dev  # noqa: F401
from ._ffi import PN_EXCHANGE_ALLGATHER, PN_EXCHANGE_PEER, PN_EXCHANGE_SLICE, PN_SHARD_BY_SUBTREE, PN_SHARD_REPLICATE


def query_slice(n_queries: int, rank: int, world: int):
    """Contiguous slice [lo, hi) of the query batch owned by `rank` (sizes differ by at most 1); pn_query_slice."""
    base, rem = divmod(n_queries, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def shard_depth(world: int) -> int:
    d = world.bit_length() - 1
    if world < 1 or (1 << d) != world:
        raise ValueError("point sharding by subtree needs a power-of-two number of ranks")
    return d


def allgather_lists(local_idx: torch.Tensor, local_dist: torch.Tensor, group=None):
    """The exchange step through torch.distributed: every rank contributes its [nq, k] sorted lists, every rank receives
    [world, nq, k].  Used by the host-logic tests over gloo on the CPU; the product path is Comm / ShardedBallTree."""
    world = dist.get_world_size(group)
    nq = local_idx.shape[0]
    rest = tuple(local_idx.shape[1:])
    gi = torch.empty((world * nq,) + rest, dtype=local_idx.dtype, device=local_idx.device)  # concatenation along dim 0
    gd = torch.empty((world * nq,) + rest, dtype=local_dist.dtype, device=local_dist.device)
    dist.all_gather_into_tensor(gi, local_idx.contiguous(), group=group)
    dist.all_gather_into_tensor(gd, local_dist.contiguous(), group=group)
    return gi.view((world, nq) + rest), gd.view((world, nq) + rest)


class Comm:
    """One rank of the library's NCCL communicator (pn_comm).  `Comm.from_torch()` takes rank / world from the default
    torch.distributed group and uses it to ship the unique id."""

    def __init__(self, unique_id: bytes, world: int, rank: int, device: int):
        self.world, self.rank, self.device = world, rank, device
        self._h = C.c_void_p()
        buf = (C.c_char * _ffi.PN_UNIQUE_ID_BYTES).from_buffer_copy(unique_id)
        _check(_ffi.lib().pn_comm_create(buf, world, rank, device, C.byref(self._h)))

    @staticmethod
    def unique_id() -> bytes:
        buf = (C.c_char * _ffi.PN_UNIQUE_ID_BYTES)()
        _check(_ffi.lib().pn_comm_unique_id(buf))
        return bytes(buf)

    @classmethod
    def create_all(cls, devices):
        """pn_comm_create_all: every rank of a communicator over `devices` in THIS process (ncclCommInitAll); calls that
        communicate must then be made from one host thread per rank."""
        n = len(devices)
        arr = (C.c_int32 * n)(*devices)
        outs = (C.c_void_p * n)()
        _check(_ffi.lib().pn_comm_create_all(arr, n, outs))
        comms = []
        for r in range(n):
            c = cls.__new__(cls)
            c.world, c.rank, c.device = n, r, int(devices[r])
            c._h = C.c_void_p(outs[r])
            comms.append(c)
        return comms

    @classmethod
    def from_torch(cls, device=None, group=None):
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        device = torch.cuda.current_device() if device is None else device
        box = [cls.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0, group=group)
        return cls(box[0], world, rank, device)

    def close(self):
        if self._h is not None and self._h.value:
            _ffi.lib().pn_comm_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def replicate(tree, comm: Comm, root: int = 0, cls=BallTree):
    """pn_tree_replicate: the root's flattened tree (device arrays) is broadcast over NCCL; every other rank gets a new
    handle without building anything.  `tree` is None on the non-root ranks."""
    out = C.c_void_p()
    _check(_ffi.lib().pn_tree_replicate(tree._h if tree is not None else None, comm._h, root, C.byref(out)))
    if comm.rank == root:
        return tree
    t = cls.__new__(cls)
    t._h = out
    s = _ffi.TreeInfo()
    _check(_ffi.lib().pn_tree_get_info(out, C.byref(s)))
    t.dtype = np.dtype(np.float32 if s.dtype == _ffi.PN_F32 else np.float64)
    t._sfx = "f32" if s.dtype == _ffi.PN_F32 else "f64"
    t.dim = int(s.dim)
    from . import distance
    t.metric = distance.Euclidean()
    return t


class ShardedBallTree:
    """Ball tree whose points are sharded by subtree over the ranks of a Comm."""

    def __init__(self, points, comm: Comm, **opts):
        self.comm = comm
        self.rank, self.world, self.device = comm.rank, comm.world, comm.device
        self.tree = BallTree.euclidean(points, device=self.device, shard_depth=shard_depth(self.world), shard_index=self.rank, **opts)
        self.dtype = self.tree.dtype
        self.dim = self.tree.dim
        self.stats = {}

    def query_batch_dev(self, q_dev: torch.Tensor, k: int, exchange: int = PN_EXCHANGE_ALLGATHER):
        """q_dev: [nq, d] CUDA tensor holding ALL queries (identical on every rank).  Returns (idx int64, dist) CUDA
        tensors: all nq rows (ALLGATHER) or the rows of this rank's slice query_slice(nq, rank, world) (SLICE)."""
        nq = q_dev.shape[0]
        rows = nq
        if exchange == PN_EXCHANGE_SLICE:
            lo, hi = query_slice(nq, self.rank, self.world)
            rows = hi - lo
        oi = torch.empty((rows, k), dtype=torch.int64, device=q_dev.device)
        od = torch.empty((rows, k), dtype=q_dev.dtype, device=q_dev.device)
        st = _ffi.ShardStats()
        stream = torch.cuda.current_stream().cuda_stream
        _check(_ffi.lib().pn_sharded_query_knn_dev(self.tree._h, self.comm._h, q_dev.data_ptr(), nq, q_dev.stride(0) if nq > 1 else q_dev.shape[1],
                                                   k, exchange, oi.data_ptr(), od.data_ptr(), stream, C.byref(st)))
        self.stats = _ffi._struct_dict(st)
        return oi, od

    def query_batch(self, Q, k: int):
        q_dev = torch.from_numpy(np.ascontiguousarray(Q, dtype=self.dtype)).cuda(self.device)
        oi, od = self.query_batch_dev(q_dev, k)
        return oi.cpu().numpy().astype(np.uint64), od.cpu().numpy()


class MultiGpuBallTree:
    """pn_multi_*: ONE process driving several GPUs through the C ABI -- one rank and one host thread per device inside
    the library (ncclCommInitAll), tree replicated over ncclBroadcast or sharded by subtree.  Host buffers in and out."""

    def __init__(self, points, devices, mode=PN_SHARD_REPLICATE, **opts):
        points = np.ascontiguousarray(points, dtype=np.float32)
        self.dim = points.shape[1]
        self.devices = list(devices)
        o = _ffi.BuildOpts()
        o.struct_size = C.sizeof(_ffi.BuildOpts)
        o.device = -1
        for key, val in opts.items():
            setattr(o, key, val)
        arr = (C.c_int32 * len(self.devices))(*self.devices)
        self._h = C.c_void_p()
        _check(_ffi.lib().pn_multi_balltree_create_f32(arr, len(self.devices), mode, points.ctypes.data, points.shape[0], self.dim, self.dim,
                                                      C.byref(o), C.byref(self._h)))

    def query_batch(self, Q, k: int):
        Q = np.ascontiguousarray(Q, dtype=np.float32)
        if Q.ndim != 2 or Q.shape[1] != self.dim:
            raise ValueError("queries must be nq x d")
        nq = Q.shape[0]
        idx = np.empty((nq, k), np.uint64)
        dist = np.empty((nq, k), np.float32)
        _check(_ffi.lib().pn_multi_balltree_query_f32(self._h, Q.ctypes.data, nq, self.dim, k, idx.ctypes.data, dist.ctypes.data))
        return idx, dist

    def query_radius_batch(self, Q, radius):
        """pn_multi_balltree_query_radius_f32: CSR (offsets[nq+1], indices), as BallTree.query_radius_batch returns it
        for a tree of all the points (strict `distance < radius`, each query's indices ascending).  BY_SUBTREE handles pull
        the per-shard hit lists with peer copies and merge them on the device; no NCCL, whatever set_exchange chose."""
        Q = np.ascontiguousarray(Q, dtype=np.float32)
        if Q.ndim != 2 or Q.shape[1] != self.dim:
            raise ValueError("queries must be nq x d")
        nq = Q.shape[0]
        offs_p = C.POINTER(C.c_uint64)()
        idx_p = C.POINTER(C.c_uint64)()
        _check(_ffi.lib().pn_multi_balltree_query_radius_f32(self._h, Q.ctypes.data if nq else None, nq, self.dim, np.float32(radius),
                                                            C.byref(offs_p), C.byref(idx_p)))
        return _csr_arrays(offs_p, idx_p, nq)

    def set_exchange(self, exchange: int):
        """BY_SUBTREE handles: PN_EXCHANGE_PEER (merge kernels read the other devices' lists over NVLink, no collective; the
        default when every pair of devices has peer access) or PN_EXCHANGE_SLICE (grouped ncclSend / ncclRecv)."""
        _check(_ffi.lib().pn_multi_set_exchange(self._h, exchange))

    def stats(self):
        arr = (_ffi.ShardStats * len(self.devices))()
        _check(_ffi.lib().pn_multi_get_stats(self._h, arr, len(self.devices)))
        return [_ffi._struct_dict(x) for x in arr]

    def close(self):
        if self._h is not None and self._h.value:
            _ffi.lib().pn_multi_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
