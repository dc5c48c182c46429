"""Workload for compute-sanitizer (tools/sanitize.sh): tiny synthetic models through every kernel family — tcgen05 prefill,
persistent decode kernel, multi-kernel PDL decode path, MoE router + routed GEMVs, dense f32 weights, prompt scoring."""
import os
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from distributed_llama_b200.formats import ModelFile, quants
from distributed_llama_b200.models.config import get_config
from distributed_llama_b200.models.loader import load_device_weights
from distributed_llama_b200.models.synthetic import write_synthetic_model
from distributed_llama_b200.runtime import Engine

which = sys.argv[1:] or ["tiny-llama31", "tiny-qwen3", "tiny-qwen3-moe", "tiny-llama31:f32"]
with tempfile.TemporaryDirectory() as d:
    for spec in which:
        name, _, wt = spec.partition(":")
        path = os.path.join(d, spec.replace(":", "_") + ".m")
        write_synthetic_model(path, get_config(name), weights_float_type=quants.parse_float_type(wt or "q40"), seed=3)
        mf = ModelFile(path)
        for mega in (True, False):
            eng = Engine(load_device_weights(mf))
            if eng.mega != mega:
                if mega:
                    continue
                eng.enable_mega(False)
            prompt = [(5 * i + 2) % 500 + 1 for i in range(21)]
            eng.prefill(prompt[:-1], 0, want_logits=False)
            toks = eng.decode_greedy(prompt[-1], len(prompt) - 1, 6, use_graph=False)
            eng.step(toks[-1], len(prompt) + 5)
            torch.cuda.synchronize()
            print(spec, "mega" if eng.mega else "multi-kernel", toks)
        # prompt scoring: prefill chain + logits GEMM + score kernel in chunks of 64 (dense files: the GEMV fallback)
        res = Engine(load_device_weights(mf), max_prefill=64).score([(3 * i + 1) % 500 + 1 for i in range(150)], 0)
        torch.cuda.synchronize()
        print(spec, "score", res.top_ids[:6].tolist())
print("SANITIZE_TARGET_DONE")
