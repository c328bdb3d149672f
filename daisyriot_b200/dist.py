"""Row-sharded form factors + gather across the GPUs of one box (one process per GPU, torch.distributed / NCCL).

Each rank builds rows ``[rank*n, (rank+1)*n)`` of F against a replicated LBVH and owns that slice of B.  One gather
pass is: local kernel -> in-place all-gather of this rank's residual block (``K x n`` floats + ``K`` partial band
sums) over NVLink -> every rank totals the band sums in rank order, so all ranks take identical stop decisions
with a single collective per pass (reference loop: ``visual studio/Lightning.h:145-151, 196-226``).

The exchange itself is backend-agnostic (``exchange_pass``) so the host logic is testable on CPU with gloo."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib


def partition(N: int, rank: int, nranks: int):
    """(row0, row1, rows_per_rank) -- must match ``set_partition`` in csrc/api.cu."""
    n = (N + nranks - 1) // nranks
    # one block: multiple of 4 floats (16-byte TMA alignment); several: multiple of 256 so that a 256-column TMA
    # tile of the residual never straddles two ranks' blocks
    n = max(4, (n + 255) // 256 * 256 if nranks > 1 else (n + 3) // 4 * 4)
    return min(N, rank * n), min(N, (rank + 1) * n), n


def block_layout(K_padded: int, n: int):
    """(floats per exchange block, float offset of the K band-sum doubles) -- matches gather.cu."""
    body = K_padded * n
    return (body + 2 * K_padded + 3) // 4 * 4, body


def padded_K(K: int) -> int:
    return 1 if K <= 1 else 3 if K <= 3 else 9 if K <= 9 else 16 if K <= 16 else 32 if K <= 32 else 64


def exchange_pass(step_local, next_buffer, rank: int, nranks: int, group=None):
    """One pass of the exchange protocol on any backend.

    ``step_local()`` fills block ``rank`` of ``next_buffer`` (a 1-D tensor of ``nranks`` equal blocks); the in-place
    all-gather then completes the buffer on every rank."""
    import torch.distributed as dist
    step_local()
    if nranks > 1:
        blk = next_buffer.numel() // nranks
        dist.all_gather_into_tensor(next_buffer, next_buffer[rank * blk:(rank + 1) * blk], group=group)


def total_band_sums(buffer_f32, K: int, K_padded: int, n: int, nranks: int) -> np.ndarray:
    """Sum the per-rank partial band sums (doubles in each block's tail) in rank order."""
    bstride, off = block_layout(K_padded, n)
    host = buffer_f32.detach().cpu().numpy() if hasattr(buffer_f32, "detach") else np.asarray(buffer_f32)
    out = np.zeros(K, np.float64)
    for g in range(nranks):
        tail = host[g * bstride + off: g * bstride + off + 2 * K_padded].view(np.float64)
        out += tail[:K]
    return out


def build_formfactors_sharded(optixP, variant: int = _lib.FF_DEVICE, group=None, peer_tiles: bool = True):
    """Row-sharded form-factor build on every rank of ``group``.

    ``peer_tiles=True``: CUDA-IPC handles of every rank's matrix are exchanged once, each upper-triangle tile is then
    traced by exactly one rank and its mirror is stored into the peer's matrix over NVLink (no ray is traced twice).
    ``peer_tiles=False``: no exchange at all; each rank traces every tile touching its rows."""
    import torch
    import torch.distributed as tdist
    L = _lib.lib()
    world = optixP.nranks
    if world > 1 and peer_tiles:
        _lib.check(L.daisy_formfactors_alloc(optixP._ctx), "formfactors_alloc")
        h = C.create_string_buffer(64)
        _lib.check(L.daisy_formfactors_ipc_handle(optixP._ctx, h), "formfactors_ipc_handle")
        handles = [None] * world
        tdist.all_gather_object(handles, bytes(h.raw), group=group)
        blob = C.create_string_buffer(b"".join(handles), 64 * world)
        _lib.check(L.daisy_formfactors_set_peers(optixP._ctx, blob, world), "formfactors_set_peers")
    _lib.check(L.daisy_formfactors_build(optixP._ctx, variant), "formfactors_build")
    if world > 1:
        torch.cuda.synchronize()
        tdist.barrier(group=group)  # peers have finished writing into this rank's rows


def update_formfactors_sharded(optixP, variant: int = _lib.FF_DEVICE, group=None):
    """Row-sharded matrix update after ``optixP.updateGeometry`` (called with identical arrays on every rank): each rank
    re-traces its share of the tiles the change can reach -- with the peer mappings of an earlier
    :func:`build_formfactors_sharded`, each such tile on exactly one rank -- then all ranks barrier as after the build."""
    import torch
    import torch.distributed as tdist
    _lib.check(_lib.lib().daisy_formfactors_update(optixP._ctx, variant), "formfactors_update")
    if optixP.nranks > 1:
        torch.cuda.synchronize()
        tdist.barrier(group=group)  # peers have finished writing into this rank's rows


class _DevMem:
    """Exposes a raw device pointer through __cuda_array_interface__ so torch can alias it without a copy."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (nbytes // 4,), "typestr": "<f4", "data": (ptr, False), "version": 2}


class PartitionedSolver:
    """A ``daisy_solver`` driven through the multi-GPU entry points with torch.distributed doing the exchange."""

    def __init__(self, optixP, K, E, M, mat_idx, group=None, fused: bool = True):
        """``fused=True`` (default with more than one rank): the exchange is done by the epilogue kernel itself -- it
        stores this rank's block into every rank's next buffer through CUDA-IPC mappings over NVLink and raises
        per-rank flags the next pass waits on (``daisy_solver_step_fused``).  ``fused=False``: local kernels + one
        in-place NCCL all-gather per pass (``exchange_pass``)."""
        import torch
        self.torch = torch
        self.p = optixP
        self.K, self.rank, self.nranks, self.group = K, optixP.rank, optixP.nranks, group
        L = _lib.lib()
        self._s = C.c_void_p()
        E = np.ascontiguousarray(E, np.float32)
        M = np.ascontiguousarray(M, np.float32)
        mat = np.ascontiguousarray(mat_idx, np.int32)
        _lib.check(L.daisy_solver_create(optixP._ctx, K, _lib.fptr(E), _lib.fptr(M), M.shape[0], _lib.iptr(mat), C.byref(self._s)),
                   "solver_create")
        self._views = {}
        self.fused = bool(fused) and self.nranks > 1
        if self.fused:
            import torch.distributed as tdist
            h = C.create_string_buffer(192)
            _lib.check(L.daisy_solver_ipc_handles(self._s, h), "solver_ipc_handles")
            handles = [None] * self.nranks
            tdist.all_gather_object(handles, bytes(h.raw), group=group)
            blob = C.create_string_buffer(b"".join(handles), 192 * self.nranks)
            _lib.check(L.daisy_solver_set_peers(self._s, blob, self.nranks), "solver_set_peers")
            tdist.barrier(group=group)  # every rank has mapped every buffer before the first remote store

    def _next_view(self):
        L = _lib.lib()
        ptr, blk, tot = C.c_void_p(), C.c_int64(), C.c_int64()
        _lib.check(L.daisy_solver_exchange_info(self._s, C.byref(ptr), C.byref(blk), C.byref(tot)))
        if ptr.value not in self._views:
            self._views[ptr.value] = self.torch.as_tensor(_DevMem(ptr.value, tot.value), device="cuda")
        return self._views[ptr.value]

    def step(self, want_sums: bool = False):
        L = _lib.lib()
        if self.fused:
            if want_sums:
                sums = np.zeros(self.K, np.float64)
                _lib.check(L.daisy_solver_step_fused(self._s, sums.ctypes.data_as(C.POINTER(C.c_double))), "step_fused")
                return sums
            _lib.check(L.daisy_solver_step_fused(self._s, None), "step_fused")
            return None
        buf = self._next_view()
        exchange_pass(lambda: _lib.check(L.daisy_solver_step_local(self._s), "step_local"), buf, self.rank, self.nranks, self.group)
        if want_sums:
            self.torch.cuda.current_stream().synchronize()
            sums = np.zeros(self.K, np.float64)
            _lib.check(L.daisy_solver_step_finish(self._s, sums.ctypes.data_as(C.POINTER(C.c_double))), "step_finish")
            return sums
        _lib.check(L.daisy_solver_step_finish(self._s, None), "step_finish")
        return None

    def band_sums(self):
        sums = np.zeros(self.K, np.float64)
        self.torch.cuda.current_stream().synchronize()
        _lib.check(_lib.lib().daisy_solver_band_sums(self._s, sums.ctypes.data_as(C.POINTER(C.c_double))))
        return sums

    def reset(self):
        _lib.check(_lib.lib().daisy_solver_reset(self._s))

    def converge(self, threshold: float, per_band: bool, max_passes: int = 0, on_device: bool = False) -> int:
        """Passes run by this call.  ``on_device=True`` (fused exchange, or a single rank): every rank calls
        ``daisy_solver_converge_device`` with the same arguments; the pass kernels apply the stop rule themselves, all ranks
        stop at the same pass, and no pass waits for the host."""
        if on_device:
            if self.nranks > 1 and not self.fused:
                raise _lib.DaisyError("PartitionedSolver.converge(on_device=True) needs the fused exchange; this solver exchanges through NCCL")
            L = _lib.lib()
            before = int(L.daisy_solver_numpasses(self._s))
            out = C.c_int()
            _lib.check(L.daisy_solver_converge_device(self._s, float(threshold), int(per_band), int(max_passes), C.byref(out)), "solver_converge_device")
            return out.value - before
        passes = 0
        sums = self.band_sums()
        crit = (lambda s: (s > threshold).any()) if per_band else (lambda s: s.sum() > threshold)
        while crit(sums) and (max_passes <= 0 or passes < max_passes):
            sums = self.step(want_sums=True)
            passes += 1
        return passes

    def restart(self, B0_local=None):
        """``daisy_solver_restart`` on this rank (every rank calls it): ``B0_local`` holds this rank's K x (row1 - row0) rows
        of the B to restart from, ``None`` restarts from the current B.  Needs the fused exchange with more than one rank
        (a partition exchanged through NCCL gets DAISY_E_STATE).  Returns the band sums (sum of |residual|)."""
        b = None
        if B0_local is not None:
            r0, r1 = self.p.row_range
            b = np.ascontiguousarray(B0_local, np.float32)
            if b.shape != (self.K, r1 - r0):
                raise ValueError("restart: B0_local must be K x (row1 - row0), got %s" % (b.shape,))
        _lib.check(_lib.lib().daisy_solver_restart(self._s, None if b is None else _lib.fptr(b)), "solver_restart")
        return self.band_sums()

    def set_emission(self, E):
        """The whole scene's K x N emission (every rank passes the same); used at the next reset or restart."""
        E = np.ascontiguousarray(E, np.float32)
        _lib.check(_lib.lib().daisy_solver_set_emission(self._s, _lib.fptr(E)), "solver_set_emission")

    def set_materials(self, M, mat_idx):
        """nmat x K x K material matrices and the N material ids of the whole scene; used from the next pass."""
        M = np.ascontiguousarray(M, np.float32)
        mat = np.ascontiguousarray(mat_idx, np.int32)
        _lib.check(_lib.lib().daisy_solver_set_materials(self._s, _lib.fptr(M), M.shape[0], _lib.iptr(mat)), "solver_set_materials")

    def read_local(self):
        r0, r1 = self.p.row_range
        B = np.empty((self.K, r1 - r0), np.float32)
        R = np.empty((self.K, r1 - r0), np.float32)
        _lib.check(_lib.lib().daisy_solver_read(self._s, _lib.fptr(B), _lib.fptr(R)))
        return B, R

    def close(self):
        if self._s and self.fused:
            import torch.distributed as tdist
            self.torch.cuda.synchronize()
            tdist.barrier(group=self.group)  # no rank unmaps while a peer may still be storing into its buffers
        if self._s:
            _lib.lib().daisy_solver_destroy(self._s)
            self._s = None
