"""Sample-sharded engine: one process per GPU.

Each rank owns a contiguous chunk of the samples (x, y and the latent buffers never leave the GPU); after each
streaming phase the per-region sufficient statistics (<= R x 60 doubles per layer) are summed over the ranks,
and the small-matrix steps are replicated (identical inputs -> identical state on every rank, no broadcast).
SURVEY.md §8e.

The sums go through the library's own exchange over peer memory (NVLink / NVSwitch): torch.distributed is used
once, to all-gather the 128-byte arena descriptions, and at the barrier of close(); a sweep is one CUDA graph of
the library's kernels, exchanges included (include/cimrgp.h, "sample sharding").
"""
import ctypes as C

import numpy as np

from . import _lib
from .engine import Engine


def chunk_bounds(n_samples, world_size, rank):
    """Contiguous, 32-aligned split of [0, n_samples): the same chunking for every layer."""
    per = -(-n_samples // world_size)
    per = -(-per // 32) * 32
    lo = min(n_samples, rank * per)
    hi = min(n_samples, lo + per)
    return lo, hi


class TorchComm(object):
    """All-gather and barrier over a torch.distributed process group."""

    def __init__(self, group=None):
        import torch.distributed as dist
        self.dist, self.group = dist, group

    def all_gather_bytes(self, payload):
        out = [None] * self.dist.get_world_size(self.group)
        self.dist.all_gather_object(out, bytes(payload), group=self.group)
        return out

    def sync(self):
        self.dist.barrier(group=self.group)


class ShardedEngine(Engine):
    def __init__(self, x_norm, y, offsets, n_basis, rank, world_size, comm=None, **kw):
        self.comm = comm if comm is not None else TorchComm()
        self.rank, self.world_size = rank, world_size
        n_total = int(offsets[0][-1])
        # the same deterministic check on every rank, BEFORE any collective: either all ranks raise or none does
        empty = [q for q in range(world_size) if chunk_bounds(n_total, world_size, q)[1] <= chunk_bounds(n_total, world_size, q)[0]]
        if empty:
            raise ValueError('%d samples over %d ranks in 32-aligned chunks leave rank(s) %s without samples: use at '
                             'most %d ranks' % (n_total, world_size, empty, max(1, -(-n_total // 32))))
        lo, hi = chunk_bounds(n_total, world_size, rank)
        Engine.__init__(self, x_norm[lo:hi], y[lo:hi], offsets, n_basis, chunk=(lo, hi), defer_build=True, **kw)
        blob = C.create_string_buffer(_lib.COMM_BLOB_BYTES)
        self._ck(self.lib.mrgp_comm_export(self.handle, blob))
        blobs = b''.join(self.comm.all_gather_bytes(blob.raw))
        bounds = (C.c_int64 * (world_size + 1))(*([chunk_bounds(n_total, world_size, q)[0] for q in range(world_size)]
                                                  + [n_total]))
        self._ck(self.lib.mrgp_comm_bind(self.handle, rank, world_size, blobs, bounds))
        if self.mode == 'ci' and self.J > 1:
            # inputs of all ranks (x only, 8 B per sample): the closed-form statistics of the upper layers
            xa = np.ascontiguousarray(x_norm, dtype=np.float64)
            self._ck(self.lib.mrgp_set_all_inputs_host(self.handle, _lib._dptr(xa) if hasattr(_lib, '_dptr') else
                                                       xa.ctypes.data_as(C.POINTER(C.c_double))))
            self.synchronize()
        for j in range(self.J):
            self._ck(self.lib.mrgp_build_basis(self.handle, j, float(self._interval_factor[j]), None))
        self._ck(self.lib.mrgp_init_state(self.handle, *self._init_args))
        self.synchronize()
        self.comm.sync()

    def close(self):
        """Collective: no rank may free its arena while a peer can still read it."""
        if self.handle is not None:
            try:
                self.synchronize()
                self.comm.sync()
            except Exception:
                pass
        Engine.close(self)

    def __del__(self):
        # Never a collective from the garbage collector.  Call close() explicitly on every rank (it synchronises and
        # meets the peers at a barrier before the arena is freed): a rank that is merely garbage-collected frees its
        # arena while peers may still read it.
        try:
            Engine.close(self)
        except Exception:
            pass

    def sweep_stepwise(self):
        lib, h = self.lib, self.handle
        for j in range(self.J):
            self._ck(lib.mrgp_phase_a(h, j))
            self._ck(lib.mrgp_exchange(h, j, 0))
            self._ck(lib.mrgp_axis_update(h, j))
            self._ck(lib.mrgp_phase_b(h, j))
            self._ck(lib.mrgp_exchange(h, j, 1))
            self._ck(lib.mrgp_bias_noise(h, j))

    def sweep(self, n_iter=1, use_graph=True):
        """n_iter sweeps: one captured CUDA graph each, or (use_graph=False) phase by phase through mrgp_exchange."""
        if n_iter <= 0:
            return
        if use_graph:
            self._ck(self.lib.mrgp_sweep(self.handle, int(n_iter)))
        else:
            for _ in range(n_iter):
                self.sweep_stepwise()

    def latent(self, j):
        raise NotImplementedError('latent export is not available on a sharded engine')

    def state(self, latent=False):
        return Engine.state(self, latent=False)
