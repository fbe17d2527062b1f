# -*- coding: utf-8 -*-
"""
Multi-GPU HODLR: one process per GPU, the tree sharded by top-level sub-tree (SURVEY.md §8e).

The reference has no distributed code; what shards is the algorithmic independence of HODLR sub-trees
(``hodlr.h:58-61,78-79``): below depth ``log2(P)`` the ``P`` sub-trees of ``~N/P`` points never touch each other's rows
(``hodlr.h:95-102,240-253``).  Each rank

1. factors its own sub-tree (leaves, ACAs, up-sweep) and applies it to ITS rows of the ``log2(P)`` top-level factor
   panels (whose ACAs every rank recomputes redundantly from the replicated coordinates — no communication);
2. takes part in ONE all-gather of those locally-solved row slices — the only data-path collective of ``compute`` —
   issued by the library itself on the solver's stream (``csrc/comm.cu``: pack kernel -> ``ncclAllGather`` -> unpack
   kernels, no host round trip);
3. finishes the ``P - 1`` top nodes redundantly (Gram, 2r x 2r LU, log-det, update).

``log|K|`` is an all-reduce of one double; a solve is: local sub-tree solve on the owned slice, one all-gather of the
vector, top nodes redundantly.  ``torch.distributed`` is plumbing only: it broadcasts the 128-byte NCCL unique id with
which every rank initialises the library's communicator (``ensure_device_comm``).  All arithmetic and all data-path
collectives are in ``csrc/hodlr.cu`` / ``csrc/comm.cu``.
"""

import ctypes as C

import numpy as np

from . import _lib
from ._spec import flatten

__all__ = ["ShardedHODLRSolver", "shard_ranges"]


def shard_ranges(n, shard_count, min_size):
    """Row ranges ``[(start, size), ...]`` of the depth-``log2(shard_count)`` nodes of the reference tree
    (``hodlr.h:48-61``: ``half = size // 2``; a node splits iff ``half >= min_size``), or ``None`` when the tree is
    too shallow to be cut that many ways."""
    if shard_count < 1 or shard_count & (shard_count - 1):
        raise ValueError("shard_count must be a power of two")
    level = [(0, int(n))]
    cut = shard_count.bit_length() - 1
    for _ in range(cut):
        nxt = []
        for start, size in level:
            half = size // 2
            if half < min_size:
                return None
            nxt.append((start, half))
            nxt.append((start + half, size - half))
        level = nxt
    return level


_COMM_WORLD = 0


def ensure_device_comm(group=None):
    """Create (once) the NCCL communicator libbgp_b200 issues its data-path collectives on (``csrc/comm.cu``): rank 0
    makes the unique id, it is broadcast over the host's process group, every rank initialises.  Returns the world size."""
    global _COMM_WORLD
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)
    if world == 1 or _COMM_WORLD == world:
        return world
    lib = _lib.load()
    rank = dist.get_rank(group)
    buf = (C.c_ubyte * 128)()
    path = None
    try:
        import nvidia.nccl
        import glob
        import os
        hits = glob.glob(os.path.join(os.path.dirname(nvidia.nccl.__file__), "lib", "libnccl.so*"))
        path = hits[0].encode() if hits else None
    except Exception:
        path = None
    if rank == 0:
        _lib.check(lib.bgp_comm_unique_id(buf, path))
    dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend(group) == "nccl" else torch.device("cpu")
    t = torch.tensor(list(bytes(buf)), dtype=torch.uint8, device=dev)
    dist.broadcast(t, src=0, group=group)
    ident = (C.c_ubyte * 128)(*t.cpu().tolist())
    _lib.check(lib.bgp_comm_init(ident, rank, world, path))
    _COMM_WORLD = world
    return world


class ShardedHODLRSolver(object):
    """Solver plugin with the ``HODLRSolver`` surface whose ``compute``/``dot_solve`` are collective over a
    ``torch.distributed`` process group (one rank per GPU).  ``x``, ``yerr`` and ``y`` are replicated on every rank."""

    def __init__(self, kernel, min_size=100, tol=0.1, seed=42, rank_capacity=0, exhaust="dense", group=None):
        self.kernel = kernel
        self.min_size, self.tol, self.seed = min_size, tol, seed
        self.rank_capacity, self.exhaust, self.group = rank_capacity, exhaust, group
        self._computed = False
        self._log_det = None
        self.solver = None

    @property
    def computed(self):
        return self._computed

    @property
    def log_determinant(self):
        return self._log_det

    def compute(self, x, yerr):
        import torch.distributed as dist
        from .solvers._hodlr import HODLRSolver as Native
        rank, world = dist.get_rank(self.group), dist.get_world_size(self.group)
        x = np.ascontiguousarray(x, dtype=np.float64)
        if x.ndim == 1:
            x = x[:, None]
        yerr = np.ascontiguousarray(yerr, dtype=np.float64)
        self._n = x.shape[0]
        self._ranges = shard_ranges(self._n, world, self.min_size)
        if self._ranges is None:
            raise ValueError("the HODLR tree (N={0}, min_size={1}) is too shallow to shard {2} ways".format(
                self._n, self.min_size, world))
        if ensure_device_comm(self.group) != world:
            raise RuntimeError("the library's NCCL communicator does not span the process group")
        if self.solver is None:
            self.solver = Native()  # one handle for the life of the solver: buffers and rank capacities are reused
        # collective: local sub-tree, all-gather of the top panel rows, top nodes, log-det all-reduce (csrc/hodlr.cu)
        self.solver.compute(self.kernel, x, yerr, self.min_size, self.tol, self.seed, rank_capacity=self.rank_capacity,
                            shard_rank=rank, shard_count=world, exhaust=self.exhaust)
        self._log_det = self.solver.log_determinant
        self._computed = True

    def apply_inverse(self, y, in_place=False):
        """Collective; ``y`` replicated on every rank."""
        return self.solver.apply_inverse(y, in_place=in_place)

    def dot_solve(self, y):
        """Collective; ``y`` replicated on every rank."""
        return self.solver.dot_solve(y)

    def apply_sqrt(self, r):
        raise NotImplementedError("apply_sqrt is not implemented for the HODLRSolver")

    def get_inverse(self):
        return self.solver.get_inverse()
