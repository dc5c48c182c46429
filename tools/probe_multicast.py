"""Probe of the symmetric VMM arena + NVLS multicast mapping (run with torchrun on >= 2 GPUs).

Checks, on every rank: unicast peer stores land in every arena; `multimem.red.add` on the multicast mapping is applied to every
replica; `multimem.ld_reduce` returns the switch-side sum. Prints one PROBE line per rank and `PROBE PASS` / `PROBE FAIL`.
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist

from distributed_llama_b200.ops import cuda_lib as cl
from distributed_llama_b200.parallel.comm import Communicator

rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
comm = Communicator()
n = 4096
W = comm.world_size
total = (4 + W) * n * 4 + 4096
comm.alloc_arena(total)
lib = cl.lib()
print(f"PROBE rank {rank}: arena kind={comm.arena_kind} mc_ptr={'0x%x' % comm.mc_ptr if comm.mc_ptr else 0} "
      f"uc={[hex(p) for p in comm.arena_ptrs]}", flush=True)
ok = True
if comm.arena_kind == "vmm":
    arena = cl.device_view(comm.arena_ptrs[rank], ((4 + W) * n,), torch.float32, device=f"cuda:{local}")
    # region 2+W: every rank writes its own value, later summed by multimem.ld_reduce
    arena[(2 + W) * n:(3 + W) * n] = float(10 * (rank + 1))
    torch.cuda.synchronize()
    dist.barrier()
    cl.check(lib.dl_vmm_selftest_kernel(comm._vmm, n, 0, cl.stream_ptr()), "selftest phase 0")
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    idx = torch.arange(n, device=arena.device, dtype=torch.float32)
    for r in range(W):
        got = arena[(1 + r) * n:(2 + r) * n]
        if not torch.equal(got, r * 1000 + idx):
            ok = False
            print(f"PROBE rank {rank}: unicast slot of rank {r} wrong: {got[:4].tolist()}", flush=True)
    if comm.mc_ptr:
        want = float(sum(range(1, W + 1)))
        got = arena[:n]
        if not torch.all(got == want):
            ok = False
            print(f"PROBE rank {rank}: multimem.red result {got[:4].tolist()} != {want}", flush=True)
        cl.check(lib.dl_vmm_selftest_kernel(comm._vmm, n, 1, cl.stream_ptr()), "selftest phase 1")
        torch.cuda.synchronize()
        got = arena[(3 + W) * n:(4 + W) * n]
        want = float(sum(10 * (r + 1) for r in range(W)))
        if not torch.all(got == want):
            ok = False
            print(f"PROBE rank {rank}: multimem.ld_reduce result {got[:4].tolist()} != {want}", flush=True)
    print(f"PROBE rank {rank}: multicast={'yes' if comm.mc_ptr else 'NO'} checks={'ok' if ok else 'BAD'}", flush=True)
t = torch.tensor([1 if ok else 0], device="cuda", dtype=torch.int32)
dist.all_reduce(t, op=dist.ReduceOp.MIN)
if rank == 0:
    print("PROBE PASS" if int(t.item()) == 1 else "PROBE FAIL", f"kind={comm.arena_kind} multicast={'yes' if comm.mc_ptr else 'no'}", flush=True)
dist.barrier()
dist.destroy_process_group()
