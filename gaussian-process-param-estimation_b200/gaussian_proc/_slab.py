"""
Row-slab sparse engine: ONE sparse likelihood evaluation (n = 2^20 in BASELINE configs[3]) on several GPUs.

The reference evaluates it on one host through imate SLQ and scipy CG over the whole matrix
(/root/reference/gaussian_proc/_mixed_correlation/mixed_correlation.py:193-209, 263-299). Here the rows of the spatially
ordered operator (Hilbert / Z-order, the order SparseEngine uses anyway) are cut into `world` contiguous slabs of 16-row
blocks, one per GPU (one process per GPU). Every n-vector of the Krylov iterations exists only as slabs; what crosses
GPUs is

* the HALO rows of the SpMM input: a block-column index carries (owner rank, row in the owner's slab) and the kernel
  loads the row from the owner's memory over NVLink (the peers' arenas are mapped through CUDA IPC, csrc/gp_peer.cu) -
  the spatial order keeps most columns of a slab inside the slab;
* the column reductions (Lanczos alpha / beta, CG p^T A p / r^T r, dots, Gram blocks): pushed into every rank's mailbox
  and added in rank order inside the reduction kernel itself (csrc/gp_peer.cuh) - bit-identical on every rank, so the
  ranks run the same recurrences, take the same stopping decisions and return the same numbers.

torch.distributed is used for the set-up (exchange of 64-byte IPC handles, one barrier) and for the host API's
all-gather of a solution; nothing on the evaluation path calls a library collective.
"""

import ctypes

import numpy

from . import _device as dev
from ._sparse import SparseEngine, DeviceCSR, DeviceRowBlocks, check, _p

lib = dev.lib

__all__ = ['SlabSparseEngine', 'slab_geometry', 'PeerArena']


def slab_geometry(n, world, rank):
    """(slab, first, last): uniform slabs of `slab` rows (a multiple of the 16-row block height), this rank's rows are
    [first, last) of the ordered operator. The last slab may be short."""
    per = (n + world - 1) // world
    slab = (per + 15) // 16 * 16
    first = min(n, rank * slab)
    return slab, first, min(n, first + slab)


class PeerArena(object):
    """This rank's arena + the mapped arenas of the peers (see csrc/gp_peer.cu). One per process and slab size, reused by
    every engine (an optimiser builds a new operator per rho)."""

    _cache = {}

    def __init__(self, rank, world, nloc_max):
        torch = dev.require_cuda()
        self.rank, self.world, self.nloc_max = int(rank), int(world), int(nloc_max)
        self.ctx = lib.gp_peer_create(self.rank, self.world, self.nloc_max)
        if not self.ctx:
            raise MemoryError('gp_peer_create failed (arena for slabs of %d rows)' % nloc_max)
        hb = int(lib.gp_peer_handle_bytes())
        mine = numpy.zeros(hb, dtype=numpy.uint8)
        check(lib.gp_peer_handle(self.ctx, dev.host_ptr(mine)), 'gp_peer_handle')
        if self.world > 1:
            import torch.distributed as dist
            d = torch.device('cuda', torch.cuda.current_device()) if dist.get_backend() == 'nccl' else torch.device('cpu')
            t = torch.from_numpy(mine).to(d)
            bufs = [torch.empty_like(t) for _ in range(self.world)]
            dist.all_gather(bufs, t)
            handles = numpy.ascontiguousarray(numpy.stack([b.cpu().numpy() for b in bufs]))
            check(lib.gp_peer_connect(self.ctx, dev.host_ptr(handles)), 'gp_peer_connect (CUDA IPC)')
            dist.barrier()        # every arena is zeroed and mapped everywhere before the first kernel touches one
        else:
            check(lib.gp_peer_connect(self.ctx, None), 'gp_peer_connect')

    @classmethod
    def get(cls, rank, world, nloc_max, tag='main'):
        key = (int(rank), int(world), tag)
        cur = cls._cache.get(key)
        if cur is None or cur.nloc_max < nloc_max:
            # (a larger arena replaces the old one on every rank at the same call: nloc_max depends on n and world only)
            if cur is not None:
                cur.close()
            cur = cls(rank, world, nloc_max)
            cls._cache[key] = cur
        return cur

    def vec(self, k, rows, B):
        """exchange vector k of this rank as an address (rows x B doubles live there)"""
        if rows > self.nloc_max or B > 32:
            raise ValueError('exchange vector too small')
        return ctypes.c_void_p(lib.gp_peer_vec(self.ctx, k))

    def barrier(self):
        check(lib.gp_peer_barrier(self.ctx, dev.stream_ptr()), 'gp_peer_barrier')

    def check_error(self):
        if lib.gp_peer_error(self.ctx, dev.stream_ptr()) != 0:
            raise RuntimeError('row-slab engine: a peer exchange timed out (the ranks issued different kernel sequences)')

    def close(self):
        """collective: every rank closes its arena at the same point (nobody may still gather from it)"""
        if self.ctx:
            if self.world > 1:
                import torch.distributed as dist
                dev.torch.cuda.synchronize()
                dist.barrier()
            lib.gp_peer_destroy(self.ctx)
            self.ctx = None
            if self.world > 1:
                dist.barrier()


class SlabSparseEngine(SparseEngine):
    """SparseEngine on this rank's slab of rows, with the peer arenas that carry the halo rows and the reductions. Same
    interface and - to rounding of the reordered sums - the same numbers as SparseEngine on one GPU; every rank of the
    group must make the same calls in the same order."""

    def __init__(self, K, imate_method='slq', imate_options=None, rank=None, world=None):
        from ._distributed import rank_world
        r, w = rank_world()
        self.rank = int(r if rank is None else rank)
        self.world = int(w if world is None else world)
        if not isinstance(K, (DeviceCSR, DeviceRowBlocks)) or K.order is None:
            raise ValueError('the row-slab engine needs a device handle from generate_sparse_operator / '
                             'generate_sparse_correlation(..., device=True).')
        opts = dict(imate_options or {})
        self.slab, self.first_row, self.last_row = slab_geometry(K.n, self.world, self.rank)
        if self.last_row <= self.first_row:
            raise ValueError('n = %d is too small for %d slabs of 16-row blocks.' % (K.n, self.world))
        part = getattr(K, 'row_slab', None)         # a handle generated with row_slab=(rank, world) holds only this slab
        if part is not None and part != (self.rank, self.world, self.first_row, self.last_row):
            raise ValueError('this handle holds the rows of slab %r, not those of rank %d of %d.'
                             % (part, self.rank, self.world))
        if isinstance(K, DeviceRowBlocks) and (K.first_row, K.last_row) != (self.first_row, self.last_row):
            raise ValueError('a directly generated operator must be generated for this slab (row_slab=(rank, world)).')
        self.peer = PeerArena.get(self.rank, self.world, self.slab)
        # the first SLQ block runs on a side stream next to the CG for [X z] (SparseEngine.prefetch_slq): its exchanges go
        # through a second arena - mailboxes and exchange vectors of two concurrent Krylov runs must not mix
        self.peer_side = (PeerArena.get(self.rank, self.world, self.slab, tag='side')
                          if bool(opts.get('overlap', True)) else None)
        SparseEngine.__init__(self, K, imate_method, opts, probe_range=None)

    # ---- operator -------------------------------------------------------------------------------------------------
    def from_op(self, X_dev):
        """the FULL (n x B) block in the caller's row order from the ranks' slabs (host API only: all-gather)"""
        torch = dev.torch
        B = X_dev.shape[1]
        pad = torch.zeros((self.slab, B), dtype=torch.float64, device='cuda')
        pad[:self.rows].copy_(X_dev)
        if self.world > 1:
            import torch.distributed as dist
            full = torch.empty((self.world * self.slab, B), dtype=torch.float64, device='cuda')
            dist.all_gather_into_tensor(full, pad)
        else:
            full = pad
        Y = torch.empty((self.n, B), dtype=torch.float64, device='cuda')
        check(lib.gp_gather_rows(_p(full), _p(self.inv_order), self.n, B, _p(Y), dev.stream_ptr()), 'gp_gather_rows')
        return Y

    def fused(self, eta, X, z, traceinv=True, drho=True, cubic=False):
        out = SparseEngine.fused(self, eta, X, z, traceinv=traceinv, drho=drho, cubic=cubic)
        self.peer.check_error()
        if self.peer_side is not None:
            self.peer_side.check_error()
        return out

    def trace_K(self):
        raise NotImplementedError('trace_K is a host reduction of the single-GPU engine.')
