"""Tensor-parallel scoring check, run under torchrun (one rank per GPU): Engine.score at TP=N (records exchanged over the peer
arena) must give bit-identical results on every rank and match the TP=1 engine within 0.25 per token (twice the 0.12
prefill-logits tolerance of tools/tp_check.py; scores carry the logits error of the target and of the normaliser).

    python -m torch.distributed.run --nproc-per-node=2 tools/score_check.py tiny-qwen3-moe
"""
import os
import shutil
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist

from distributed_llama_b200.formats import ModelFile
from distributed_llama_b200.models.config import get_config
from distributed_llama_b200.models.loader import load_device_weights
from distributed_llama_b200.models.synthetic import write_synthetic_model
from distributed_llama_b200.parallel.comm import Communicator
from distributed_llama_b200.runtime import Engine


def main():
    name = sys.argv[1] if len(sys.argv) > 1 else "tiny-llama31"
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    comm = Communicator()
    d = [tempfile.mkdtemp(prefix="score_check_") if comm.rank == 0 else None]
    dist.broadcast_object_list(d, src=0)
    path = os.path.join(d[0], f"{name}.m")
    if comm.rank == 0:
        write_synthetic_model(path, get_config(name), seed=11)
    dist.barrier()
    mf = ModelFile(path)
    n_tok = min(mf.header.seq_len, 240)
    toks = [(11 * i + 5) % 500 + 1 for i in range(n_tok)]
    eng = Engine(load_device_weights(mf, comm.rank, comm.world_size, comm=comm), comm=comm)
    cap = eng.score_max_tokens
    res = eng.score(toks, 0)
    flat = torch.cat([res.logprobs, res.top_ids.float(), res.top_logprobs]).cuda()
    gathered = [torch.empty_like(flat) for _ in range(comm.world_size)]
    dist.all_gather(gathered, flat)
    # bitwise comparison (NaN-free: every row but the last has a target, and the last has no logprob entry)
    same = all(torch.equal(g.view(torch.int32), flat.view(torch.int32)) for g in gathered)
    ok = True
    if comm.rank == 0:
        ref = Engine(load_device_weights(mf, 0, 1)).score(toks, 0)
        err = (res.logprobs - ref.logprobs).abs().max().item()
        err_top = (res.top_logprobs - ref.top_logprobs).abs().max().item()
        chunks = (n_tok + cap - 1) // cap
        print(f"model={name} tp={comm.world_size} tokens={n_tok} chunk cap={cap} chunks={chunks} max|tp - tp1| logprob={err:.4g} "
              f"top logprob={err_top:.4g} ranks bit-identical {same}")
        ok = same and err < 0.25 and err_top < 0.25
        print("SCORE_CHECK", "PASS" if ok else "FAIL")
    dist.barrier()
    if comm.rank == 0:
        shutil.rmtree(d[0], ignore_errors=True)
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
