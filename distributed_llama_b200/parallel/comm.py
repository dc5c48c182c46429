"""One-process-per-GPU communicator: torch.distributed (NCCL) for bootstrap and the baseline collectives, plus a
symmetric peer-memory arena that the fused kernels write into directly over NVLink.

Reference component replaced: NnNetwork::serve/connect + NnNetworkNodeSynchronizer (src/nn/nn-network.cpp:295-632):
root/worker TCP mesh bootstrap and the per-segment sync steps. Here rank 0 is the root, ranks 1..n-1 are the workers.
"""
from __future__ import annotations

import ctypes as C
from typing import List

import torch
import torch.distributed as dist

from ..ops import cuda_lib as cl

class Communicator:
    """Wraps the default process group. `alloc_arena` creates the symmetric buffer and maps every peer's copy."""

    def __init__(self):
        if not dist.is_initialized():
            raise RuntimeError("torch.distributed must be initialised (one rank per GPU, backend nccl)")
        self.rank = dist.get_rank()
        self.world_size = dist.get_world_size()
        self.device = torch.device("cuda", torch.cuda.current_device())
        self._lib = cl.lib()
        self.arena_ptrs: List[int] = []
        self.mc_ptr: int = 0             # NVLS multicast mapping of the arena (0: not available, kernels use unicast peer stores)
        self.arena_kind = "none"         # "vmm" (cuMem* + multicast) or "ipc" (cudaMalloc + CUDA IPC)
        self._local = None
        self._vmm = None
        # Peer-memory (CUDA IPC over NVLink) collectives need every rank on one host; otherwise the engine falls back to NCCL.
        import socket
        hosts = [None] * self.world_size
        dist.all_gather_object(hosts, socket.gethostname())
        self.single_node = len(set(hosts)) == 1

    @property
    def is_root(self) -> bool:
        return self.rank == 0

    _arena_seq = 0

    def alloc_arena(self, nbytes: int) -> None:
        """Creates the symmetric arena of `nbytes` per rank. Preferred: CUDA VMM allocation shared through POSIX descriptors with
        an NVLS multicast mapping (csrc/cuda/comm_vmm.cu); fallback: cudaMalloc + CUDA IPC handles (no multicast)."""
        import os
        if os.environ.get("DL_NO_VMM") is None and self.single_node and self._alloc_vmm(nbytes):
            return
        self._alloc_ipc(nbytes)

    def alloc_shared(self, nbytes: int):
        """A second symmetric allocation (no multicast mapping): returns the list of per-rank device pointers, or None when the VMM
        path is unavailable. Used for the vocabulary-sharded embedding table."""
        import os
        if os.environ.get("DL_NO_VMM") is not None or not self.single_node:
            return None
        res = self._vmm_bootstrap(nbytes, want_mc=0)
        if res is None:
            return None
        h, ptrs, _mc = res
        self._shared_handles = getattr(self, "_shared_handles", []) + [h]
        return ptrs

    def _alloc_vmm(self, nbytes: int) -> bool:
        res = self._vmm_bootstrap(nbytes, want_mc=0 if __import__("os").environ.get("DL_NO_MULTICAST") is not None else 1)
        if res is None:
            return False
        self._vmm, self.arena_ptrs, self.mc_ptr = res
        self._local = self.arena_ptrs[self.rank]
        self.arena_kind = "vmm"
        return True

    def _vmm_bootstrap(self, total: int, want_mc: int):
        import os
        lib = self._lib
        flags = C.c_int(0)
        if lib.dl_vmm_supported(C.byref(flags)) != 0:
            flags.value = 0
        ok = torch.tensor([1 if (flags.value & 1) else 0], dtype=torch.int32, device=self.device)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:
            return None
        Communicator._arena_seq += 1
        nonce = [None]
        if self.rank == 0:
            nonce[0] = f"{os.getpid()}-{Communicator._arena_seq}-{int.from_bytes(os.urandom(4), 'little')}"
        dist.broadcast_object_list(nonce, src=0)
        h = lib.dl_vmm_create(self.rank, self.world_size, total, nonce[0].encode(), want_mc)
        ok = torch.tensor([1 if h else 0], dtype=torch.int32, device=self.device)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:
            if h:
                lib.dl_vmm_destroy(h)
            return None
        rc = lib.dl_vmm_connect(h)
        ok = torch.tensor([1 if rc == 0 else 0], dtype=torch.int32, device=self.device)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:
            raise RuntimeError(f"rank {self.rank}: VMM arena bootstrap failed (code {rc}); set DL_NO_VMM=1 to use the CUDA IPC arena")
        ptrs = [int(lib.dl_vmm_ptr(h, r)) for r in range(self.world_size)]
        mc = lib.dl_vmm_mc_ptr(h)
        # the multicast mapping is used only if every rank has it
        have = torch.tensor([1 if mc else 0], dtype=torch.int32, device=self.device)
        dist.all_reduce(have, op=dist.ReduceOp.MIN)
        mc_ptr = int(mc) if (mc and int(have.item()) == 1) else 0
        dist.barrier()
        return h, ptrs, mc_ptr

    def _alloc_ipc(self, nbytes: int) -> None:
        ptr = C.c_void_p()
        cl.check(self._lib.dl_comm_alloc(nbytes, C.byref(ptr)), "comm_alloc")
        self._local = ptr.value
        handle = (C.c_ubyte * 64)()
        cl.check(self._lib.dl_comm_ipc_handle(ptr, handle), "comm_ipc_handle")
        mine = (bytes(handle), torch.cuda.current_device())
        gathered = [None] * self.world_size
        dist.all_gather_object(gathered, mine)
        self.arena_ptrs = []
        for r, (h, _dev) in enumerate(gathered):
            if r == self.rank:
                self.arena_ptrs.append(self._local)
            else:
                buf = (C.c_ubyte * 64).from_buffer_copy(h)
                out = C.c_void_p()
                cl.check(self._lib.dl_comm_ipc_open(buf, C.byref(out)), "comm_ipc_open")
                self.arena_ptrs.append(out.value)
        self.mc_ptr = 0
        self.arena_kind = "ipc"
        dist.barrier()

    # ---- baseline collectives (NCCL) ----
    def all_reduce(self, t: torch.Tensor) -> torch.Tensor:
        dist.all_reduce(t)
        return t

    def all_gather_cat(self, t: torch.Tensor, dim: int = -1) -> torch.Tensor:
        parts = [torch.empty_like(t) for _ in range(self.world_size)]
        dist.all_gather(parts, t.contiguous())
        return torch.cat(parts, dim=dim)

    def broadcast_int(self, value: int, src: int = 0) -> int:
        t = torch.tensor([value], dtype=torch.int64, device=self.device)
        dist.broadcast(t, src)
        return int(t.item())

    def barrier(self):
        dist.barrier()
