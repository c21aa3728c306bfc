"""Peer-memory (NVLink / NVSwitch) all-reduce for the dialogue-sharded train step -- host side of csrc/p2p.cu.

The reference reaches NCCL through accelerate / DDP (lumo/trainer/trainer.py:62-64,315-327).  What the COGMEN step exchanges is
small and latency-bound (BatchNorm statistics, their backward sums, 1.1 MB of gradients), so on ONE node it goes through
``ercg_p2p_allreduce``: a one-shot exchange over peer memory, one ordinary kernel launch per collective (capturable in the
step's CUDA graph), bit-identical on every rank.  ``PeerComm`` owns the set-up: one region per rank (cudaMalloc), its CUDA IPC
handle sent to the peers over any torch.distributed group (gloo or NCCL -- set-up only), every peer's region opened here.

A communicator serialises its calls on ONE stream; ``CogmenTrainStep`` therefore keeps two (main stream, side stream of the
early gradient bucket).  ``torch.distributed`` stays the transport for CPU tensors (the gloo tests of the host logic) and the
fallback when peer access is not available (``PeerComm.create`` returns None on every rank in that case).
"""
import ctypes
import os

import torch
import torch.distributed as dist

from ._lib import ErcgError, check, lib

HANDLE_BYTES = 64


class PeerComm:
    def __init__(self, group, device, max_bytes=4 << 20):
        """Collective over ``group`` (every rank calls it); raises on the ranks where the set-up fails."""
        self.group, self.device = group, torch.device(device)
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.max_bytes = int(max_bytes)
        self._own = None
        self._peers = []
        L = lib()
        nbytes = L.ercg_p2p_region_bytes(self.max_bytes)
        with torch.cuda.device(self.device):
            ptr = ctypes.c_void_p()
            handle = (ctypes.c_ubyte * HANDLE_BYTES)()
            check(L.ercg_p2p_alloc(nbytes, ctypes.byref(ptr), handle), "ercg_p2p_alloc")
            self._own = ptr.value
            handles = [None] * self.world
            dist.all_gather_object(handles, bytes(handle), group=group)
            bases = []
            for r, h in enumerate(handles):
                if r == self.rank:
                    bases.append(self._own)
                    continue
                peer = ctypes.c_void_p()
                buf = (ctypes.c_ubyte * HANDLE_BYTES).from_buffer_copy(h)
                check(L.ercg_p2p_open(buf, ctypes.byref(peer)), "ercg_p2p_open (rank %d)" % r)
                self._peers.append(peer.value)
                bases.append(peer.value)
            self.regions = torch.tensor(bases, dtype=torch.int64).to(self.device)
            torch.cuda.synchronize(self.device)

    @classmethod
    def simulate(cls, world, device, max_bytes=4 << 20):
        """``world`` communicator endpoints inside ONE process on ONE device (their regions are plain allocations of this
        process, no IPC): rank r's collective is launched on its own stream and the kernels meet through the same flag
        protocol as across GPUs.  For tests of every world size on a one-GPU box; not a transport."""
        device = torch.device(device)
        L = lib()
        nbytes = L.ercg_p2p_region_bytes(int(max_bytes))
        bases = []
        with torch.cuda.device(device):
            for _ in range(world):
                ptr = ctypes.c_void_p()
                handle = (ctypes.c_ubyte * HANDLE_BYTES)()
                check(L.ercg_p2p_alloc(nbytes, ctypes.byref(ptr), handle), "ercg_p2p_alloc")
                bases.append(ptr.value)
            regions = torch.tensor(bases, dtype=torch.int64).to(device)
            torch.cuda.synchronize(device)
        out = []
        for r in range(world):
            c = cls.__new__(cls)
            c.group, c.device, c.rank, c.world, c.max_bytes = None, device, r, world, int(max_bytes)
            c._own, c._peers, c.regions = bases[r], [], regions
            out.append(c)
        return out

    @classmethod
    def create(cls, group, device, max_bytes=4 << 20, n=1):
        """``n`` communicators, or None on EVERY rank if any rank could not set one up (no peer access, IPC refused, more than
        16 ranks, ERCG_P2P=0): the caller then stays on torch.distributed.  Collective."""
        ok, comms = 1, []
        if os.environ.get("ERCG_P2P", "1") == "0" or dist.get_world_size(group) > 16:
            ok = 0
        else:
            try:
                comms = [cls(group, device, max_bytes) for _ in range(n)]
            except (ErcgError, RuntimeError, OSError):
                ok = 0
        votes = [None] * dist.get_world_size(group)
        dist.all_gather_object(votes, ok, group=group)         # also the barrier behind which every region is zeroed and opened
        if not all(votes):
            for c in comms:
                c.close()
            return None
        return comms

    def all_reduce(self, t):
        """In-place sum over the ranks of a contiguous fp32 / fp64 CUDA tensor, on the current stream."""
        assert t.is_cuda and t.is_contiguous() and t.dtype in (torch.float32, torch.float64), (t.dtype, t.device)
        from .ops import _stream
        check(lib().ercg_p2p_allreduce(self.regions.data_ptr(), self.rank, self.world, t.data_ptr(), t.data_ptr(), t.numel(),
                                       0 if t.dtype == torch.float32 else 1, self.max_bytes, _stream()), "ercg_p2p_allreduce")
        return t

    def status(self):
        """0, or ERCG_P2P_ETIMEOUT if a peer failed to arrive at some collective (synchronises the device)."""
        st = ctypes.c_int(0)
        torch.cuda.synchronize(self.device)
        check(lib().ercg_p2p_status(self._own, ctypes.byref(st)), "ercg_p2p_status")
        return st.value

    def status_word(self):
        """Device address of this rank's sticky status word (for FlatAdam.skip_if_nonzero / ercg_adam_step_guarded)."""
        ptr = ctypes.c_void_p()
        check(lib().ercg_p2p_status_word(self._own, ctypes.byref(ptr)), "ercg_p2p_status_word")
        return ptr.value

    def check(self):
        st = self.status()
        if st != 0:
            raise ErcgError("peer-memory all-reduce: %s (%d)" % (lib().ercg_strerror(st).decode(), st))

    def close(self):
        L = lib()
        for p in self._peers:
            L.ercg_p2p_close(p)
        self._peers = []
        if self._own is not None:
            L.ercg_p2p_free(self._own)
            self._own = None


class Reducer:
    """``reducer(t)``: in-place all-reduce(sum) of ``t`` through a PeerComm when there is one (CUDA tensors), else through
    torch.distributed on ``group``."""

    def __init__(self, group=None, comm=None):
        self.group, self.comm = group, comm

    def __call__(self, t):
        if self.comm is not None and t.is_cuda:
            return self.comm.all_reduce(t)
        dist.all_reduce(t, group=self.group)
        return t

    @property
    def transport(self):
        return "peer memory (ercg_p2p_allreduce)" if self.comm is not None else "torch.distributed"
