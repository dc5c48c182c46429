"""Size of the tensor-parallel peer arena as the engine lays it out (a host function: no GPU needed)."""
import ctypes as C

import pytest


@pytest.fixture(scope="module")
def lib():
    from distributed_llama_b200.ops import cuda_lib as cl
    try:
        return cl.lib()
    except Exception as e:   # no nvcc, or a CUDA runtime that cannot be loaded
        pytest.skip(f"CUDA library unavailable: {e}")


# Totals of the layout the Python and native front ends computed before the engine owned it: LL slots of the decode and
# prefill all-reduces, logits-gather counters, arg-max candidates and gathered logits, each region 256-byte aligned.
@pytest.mark.parametrize("n_ranks,max_batch,n_experts,dim,vocab_full,max_prefill,nbytes", [
    (2, 8, 0, 4096, 128256, 192, 30322944),      # llama-3.1-8b shape
    (8, 8, 0, 4096, 128256, 192, 108978432),
    (4, 8, 128, 2048, 151936, 192, 25913088),    # qwen3-30b-a3b shape: mixture of experts runs one token per forward
])
def test_arena_bytes(lib, n_ranks, max_batch, n_experts, dim, vocab_full, max_prefill, nbytes):
    from distributed_llama_b200.ops import cuda_lib as cl
    cfg = cl.EngineConfig(dim=dim, nRanks=n_ranks, maxBatch=max_batch, nExperts=n_experts, nActiveExperts=8 if n_experts else 0,
                          vocabFull=vocab_full, maxPrefill=max_prefill)
    assert lib.dl_engine_arena_bytes(C.byref(cfg)) == nbytes
