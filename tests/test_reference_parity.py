"""Cross-check against the unmodified reference binary (CPU): the reference's `dllama perplexity` on our synthetic `.m`/`.t`
files must report the same per-token probabilities as the PyTorch oracle (which the CUDA engine is tested against).
This pins down file formats, tokenizer encoding, RoPE/QK-norm conventions and the MoE routing for all three families.
The reference's output is stored in tests/golden/reference_parity.json (oracle/golden_reference_parity.py regenerates it)."""
import hashlib
import json
import os

import numpy as np
import pytest
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_parity.json")


def _sha256(path):
    with open(path, "rb") as f:
        return hashlib.sha256(f.read()).hexdigest()


@pytest.mark.parametrize("name", ["tiny-llama", "tiny-llama31", "tiny-qwen3", "tiny-qwen3-moe"])
def test_reference_binary_agrees_with_oracle(tmp_models, name):
    from distributed_llama_b200 import host
    from distributed_llama_b200.formats import ModelFile
    from distributed_llama_b200.models.reference import OracleModel
    with open(GOLDEN) as f:
        golden = json.load(f)
    ref = golden["models"][name]
    m, t = tmp_models[name]
    # the stored probabilities belong to these exact files; a generator that writes other bytes needs the golden data regenerated
    assert _sha256(m) == ref["model_sha256"] and _sha256(t) == ref["tokenizer_sha256"]
    prompt = golden["prompt"]
    ref_probs = ref["probs"]
    tok = host().Tokenizer(t)
    ids = tok.encode(prompt, True, True)
    assert len(ref_probs) == len(ids) - 1          # same tokenisation length as the reference
    oracle = OracleModel(ModelFile(m), act_quant="q80")
    logits = oracle.forward(ids[:-1], 0)
    probs = torch.softmax(logits, dim=-1)
    ours = [float(probs[i, ids[i + 1]]) for i in range(len(ids) - 1)]
    np.testing.assert_allclose(ours, ref_probs, rtol=0.08, atol=2e-5)
    ppl = float(np.exp(-np.mean(np.log(np.maximum(ours, 1e-30)))))
    assert abs(ppl - ref["perplexity"]) / ref["perplexity"] < 0.05
