"""Multi-GPU plumbing of the pair-synthesis path: one process per GPU, units sharded by rank.

Granules and tiles are independent for the ortho and SRF kernels, so they are dealt round-robin
to ranks with NO data-path exchange.  The polynomial fit is the one global step: every rank
reduces its pixels to a ``[K, 3*deg+2]`` float64 moment matrix (768 B for K = 12, deg = 2) and a
single ``all_reduce(SUM)`` — NCCL over NVLink on GPUs, gloo in the CPU tests — makes the normal
equations global; every rank then solves redundantly and applies to its own shard.
(The reference is a single Python process: there is nothing to mirror here.)
"""
from __future__ import annotations

import os
from typing import List, Optional, Sequence

import torch
import torch.distributed as dist


def world() -> tuple:
    """(rank, world_size) of the default process group, (0, 1) when not initialised."""
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def group_size(group=None) -> int:
    """Processes in ``group`` (the default group when None); 1 when torch.distributed is not initialised."""
    if dist.is_available() and dist.is_initialized():
        return dist.get_world_size(group)
    return 1


def init_from_env(backend: Optional[str] = None) -> tuple:
    """Initialise torch.distributed from the torchrun environment (RANK / LOCAL_RANK / WORLD_SIZE /
    MASTER_ADDR / MASTER_PORT) and bind this process to its GPU.  Returns (rank, world_size, device)."""
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    use_cuda = torch.cuda.is_available()
    device = torch.device("cuda", local_rank) if use_cuda else torch.device("cpu")
    if use_cuda:
        torch.cuda.set_device(device)
    if world_size > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29511")
        kwargs = {}
        if use_cuda:
            kwargs["device_id"] = device
        dist.init_process_group(backend or ("nccl" if use_cuda else "gloo"), rank=rank, world_size=world_size,
                                **kwargs)
    return rank, world_size, device


def shard_units(n_units: int, rank: Optional[int] = None, world_size: Optional[int] = None) -> List[int]:
    """Indices of the units (granules, tiles) this rank owns: round-robin, so ranks differ by at most one unit."""
    if rank is None or world_size is None:
        rank, world_size = world()
    if not (0 <= rank < world_size):
        raise ValueError(f"rank {rank} outside world of {world_size}")
    return list(range(rank, int(n_units), world_size))


def shard_rows(n_rows: int, rank: Optional[int] = None, world_size: Optional[int] = None, align: int = 1,
               weights=None) -> tuple:
    """Contiguous [row0, row1) slab of an ortho grid for this rank (mosaic config): slabs are
    ``align``-row multiples except the last.  ``weights`` (one non-negative number per row, e.g. the bytes the row
    costs: valid pixels x spectrum + outputs) balances the WORK instead of the row count — the rows of a rotated
    swath hold very different numbers of valid pixels, and the step waits for the slowest slab."""
    if rank is None or world_size is None:
        rank, world_size = world()
    n_rows = int(n_rows)
    if weights is None:
        per = -(-n_rows // world_size)
        per = -(-per // align) * align
        r0 = min(n_rows, rank * per)
        r1 = min(n_rows, r0 + per)
        return r0, r1
    import numpy as np

    w = np.asarray(weights, dtype=np.float64).reshape(-1)
    if w.size != n_rows or (w < 0).any():
        raise ValueError("weights must hold one non-negative number per row")
    cum = np.concatenate([[0.0], np.cumsum(w)])
    total = cum[-1]
    if total <= 0:
        return shard_rows(n_rows, rank, world_size, align)
    # boundary b_i = first row (a multiple of align) whose cumulative weight reaches i / world of the total
    bounds = [0]
    for i in range(1, world_size):
        b = int(np.searchsorted(cum, total * i / world_size, side="left"))
        b = min(n_rows, -(-b // align) * align)
        bounds.append(max(b, bounds[-1]))
    bounds.append(n_rows)
    return bounds[rank], bounds[rank + 1]


def allreduce_moments(moments: torch.Tensor, group=None) -> torch.Tensor:
    """In-place SUM all-reduce of the float64 moment matrix; a no-op for a single process."""
    if moments.dtype != torch.float64:
        raise TypeError("moments must be float64")
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(moments, op=dist.ReduceOp.SUM, group=group)
    return moments


class PeerExchangeUnavailable(RuntimeError):
    """The peer blocks could not be set up on every rank (raised on ALL ranks: fall back to ``allreduce_moments``)."""


class PeerExchange:
    """The global-fit "all-reduce" as peer-memory traffic fused into the kernels either side of it.

    Every rank owns a small peer block in device memory; the blocks are mapped into every process of the node by
    CUDA IPC (handles travel through ``torch.distributed.all_gather_object``).  ``kernels.fit_moments(...,
    exchange=px.next())`` makes the finalize kernel store this rank's moment sums into every rank's block over
    NVLink / NVSwitch and raise a flag; ``kernels.poly_solve_apply(..., exchange=<same struct>)`` polls the local
    block, adds the slots in rank order and solves — no collective call, no extra launch, 10-15 us per step
    (measured, N = 2 / 4; 12-17 us for a 768-byte NCCL all-reduce), and bit-identical sums on every rank.
    One node only (CUDA IPC); ``hsr_b200.dist.allreduce_moments`` (NCCL / gloo) remains for everything else.

    Contract (checked on the host where it can be, bounded on the device where it cannot):
    * descriptors are used in strict fit -> solve/apply pairs on one stream: ``next()`` raises if the previous
      descriptor has not been through both kernels;
    * every rank performs the same number of exchanges.  A rank that is missing (it died, raised before its fit, or
      was dealt fewer units) cannot hang the others: the solve/apply kernel waits ``timeout_ms`` for the peers'
      flags, then writes NaN coefficients and sets a sticky status word — :meth:`check` raises ``HsrError`` from then
      on.  Deal uneven unit counts with ``synthesize_sharded`` (local sum + one all-reduce) instead.
    """

    def __init__(self, group=None, device=None, timeout_ms: int = 0):
        import ctypes

        from . import _lib

        self._lib = _lib
        self.rank, self.world = (dist.get_rank(group), dist.get_world_size(group)) if dist.is_initialized() else (0, 1)
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.epoch = 0
        self.timeout_ms = int(timeout_ms)
        self._last = None
        self._imported = []
        self._block = None
        lib = _lib.lib()
        failure = None
        with torch.cuda.device(self.device):
            handle = (ctypes.c_ubyte * 64)()
            try:
                blk = ctypes.c_void_p()
                _lib.check(lib.hsr_peer_alloc(ctypes.byref(blk)))
                self._block = blk.value
                _lib.check(lib.hsr_ipc_export(self._block, handle))
                if os.environ.get("HSR_PEER_FAIL_RANK") == str(self.rank):      # fault injection for the fallback test
                    raise RuntimeError("injected failure (HSR_PEER_FAIL_RANK)")
            except Exception as e:  # noqa: BLE001 - any failure must reach the collective agreement below
                failure = e
            handles = [None] * self.world
            if self.world > 1:
                dist.all_gather_object(handles, None if failure is not None else bytes(handle), group=group)
            ptrs = []
            if failure is None and all(h is not None for q, h in enumerate(handles) if q != self.rank):
                try:
                    for q in range(self.world):
                        if q == self.rank:
                            ptrs.append(self._block)
                            continue
                        buf = (ctypes.c_ubyte * 64).from_buffer_copy(handles[q])
                        out = ctypes.c_void_p()
                        _lib.check(lib.hsr_ipc_import(buf, ctypes.byref(out)))
                        self._imported.append(out.value)
                        ptrs.append(out.value)
                except Exception as e:  # noqa: BLE001
                    failure = e
            elif failure is None:
                failure = RuntimeError("a peer could not export its block")
            # every rank must reach the same verdict (a rank that raised alone would leave the others in the barrier)
            if self.world > 1:
                verdicts = [None] * self.world
                dist.all_gather_object(verdicts, failure is None, group=group)
                if not all(verdicts):
                    self.close()
                    bad = [q for q, v in enumerate(verdicts) if not v]
                    raise PeerExchangeUnavailable(f"CUDA IPC peer blocks unavailable on rank(s) {bad}: {failure}")
            elif failure is not None:
                self.close()
                raise PeerExchangeUnavailable(str(failure))
            self.peer_ptrs = torch.tensor(ptrs, dtype=torch.int64, device=self.device)
            torch.cuda.synchronize(self.device)
        if self.world > 1:
            dist.barrier(group=group)          # every block is mapped everywhere before anyone writes

    def next(self):
        """The exchange descriptor (pass the same object to fit_moments and poly_solve_apply).  The kernels number
        the exchanges themselves (epoch 0 = device-side counter), so consecutive descriptors are identical and a
        step that contains an exchange can be captured into a CUDA graph and replayed."""
        if self._last is not None and getattr(self._last, "_stage", 2) != 2:
            raise RuntimeError("PeerExchange: the previous descriptor was not used by both fit_moments and "
                               "poly_solve_apply (exchanges must strictly alternate fit -> solve/apply)")
        self.epoch += 1
        ex = self._lib.Exchange(self.peer_ptrs.data_ptr(), self._block, self.world, self.rank, 0, self.timeout_ms, 0)
        ex._stage = 0              # 0: fresh, 1: published by fit_moments, 2: consumed by poly_solve_apply
        self._last = ex
        return ex

    def check(self, stream=None) -> None:
        """Synchronise ``stream`` (default: the current one) and raise ``HsrError`` if any solve/apply kernel of this
        rank gave up waiting for a peer (its coefficients are NaN).  Call it before trusting a batch of results."""
        import ctypes

        if self._block is None:
            return
        with torch.cuda.device(self.device):
            st = stream if stream is not None else torch.cuda.current_stream(self.device)
            word = ctypes.c_uint(0)
            self._lib.check(self._lib.lib().hsr_peer_status(self._block, ctypes.byref(word), st.cuda_stream))

    def close(self):
        lib = self._lib.lib()
        for p in self._imported:
            lib.hsr_ipc_close(p)
        self._imported = []
        if self._block is not None:
            lib.hsr_peer_free(self._block)
            self._block = None


class RawNcclComm:
    """An ``ncclComm_t`` created without torch.distributed — what a non-torch host hands to
    ``hsr_allreduce_moments`` (include/hsr_b200.h).  ``RawNcclComm.unique_id()`` on one rank, ship the 128 bytes
    to the others by any means, then ``RawNcclComm(uid, nranks, rank)`` on every rank (collective)."""

    _ID_BYTES = 128

    @staticmethod
    def _nccl():
        import ctypes

        for name in ("libnccl.so.2", "libnccl.so"):
            try:
                return ctypes.CDLL(name, mode=ctypes.RTLD_GLOBAL)
            except OSError:
                continue
        raise RuntimeError("libnccl.so.2 not found")

    @classmethod
    def unique_id(cls) -> bytes:
        import ctypes

        buf = (ctypes.c_ubyte * cls._ID_BYTES)()
        rc = cls._nccl().ncclGetUniqueId(buf)
        if rc != 0:
            raise RuntimeError(f"ncclGetUniqueId failed: {rc}")
        return bytes(buf)

    def __init__(self, uid: bytes, nranks: int, rank: int, device=None):
        import ctypes

        class _Uid(ctypes.Structure):
            _fields_ = [("internal", ctypes.c_ubyte * self._ID_BYTES)]

        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self._lib = self._nccl()
        self._lib.ncclCommInitRank.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.c_int, _Uid, ctypes.c_int]
        self.comm = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            rc = self._lib.ncclCommInitRank(ctypes.byref(self.comm), int(nranks), _Uid.from_buffer_copy(uid), int(rank))
        if rc != 0:
            raise RuntimeError(f"ncclCommInitRank failed: {rc}")

    def allreduce_moments(self, moments: torch.Tensor) -> torch.Tensor:
        """In-place SUM of a float64 CUDA tensor over the communicator, on the current stream (hsr_allreduce_moments)."""
        from . import _lib

        if moments.dtype != torch.float64 or not moments.is_cuda or not moments.is_contiguous():
            raise TypeError("moments must be a contiguous float64 CUDA tensor")
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().hsr_allreduce_moments(moments.data_ptr(), moments.numel(), self.comm,
                                                        torch.cuda.current_stream().cuda_stream))
        return moments

    def close(self):
        import ctypes

        if self.comm:
            self._lib.ncclCommDestroy.argtypes = [ctypes.c_void_p]
            self._lib.ncclCommDestroy(self.comm)
            self.comm = ctypes.c_void_p()


def sum_moments(per_unit: Sequence[torch.Tensor]) -> torch.Tensor:
    """Fixed-order float64 sum of the moment matrices of this rank's units."""
    total = per_unit[0].clone()
    for m in per_unit[1:]:
        total += m
    return total
