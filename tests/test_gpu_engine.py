"""End-to-end: native engine vs the PyTorch oracle on synthetic models."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _setup(tmp_models, name, **kw):
    from distributed_llama_b200.formats import ModelFile
    from distributed_llama_b200.models.loader import load_device_weights
    from distributed_llama_b200.models.reference import OracleModel
    from distributed_llama_b200.runtime import Engine
    mf = ModelFile(tmp_models[name][0])
    eng = Engine(load_device_weights(mf), **kw)
    oracle = OracleModel(mf, act_quant="q80", device="cuda")
    return mf, eng, oracle


@pytest.mark.parametrize("name", ["tiny-llama", "tiny-llama31", "tiny-qwen3", "tiny-qwen3-moe"])
def test_engine_matches_oracle(tmp_models, name):
    mf, eng, oracle = _setup(tmp_models, name)
    toks = [3, 17, 250, 9, 44, 101, 7, 300, 12, 5, 77]
    ref = oracle.forward(toks, 0)
    # token by token
    for i, t in enumerate(toks):
        lg = eng.step(t, i)
        err = (lg - ref[i]).abs().max().item()
        assert err < 0.06, f"pos {i}: {err}"
    # batched prefill path (8 + 2 + 1) must agree with the sequential one
    eng2 = _setup(tmp_models, name)[1]
    eng2.use_tc_prefill = False
    lg = eng2.prefill(toks, 0)
    assert (lg - ref[-1]).abs().max().item() < 0.06
    if "moe" in name:
        return
    # all-token logits of a batch
    eng3 = _setup(tmp_models, name)[1]
    la = eng3.logits_all(toks[:8], 0)
    assert (la - ref[:8]).abs().max().item() < 0.06


def test_graph_decode_equals_eager(tmp_models):
    mf, eng, oracle = _setup(tmp_models, "tiny-llama")
    prompt = [3, 17, 250, 9]
    eng.prefill(prompt[:-1], 0, want_logits=False)
    a = eng.decode_greedy(prompt[-1], len(prompt) - 1, 24, use_graph=False)
    eng_b = _setup(tmp_models, "tiny-llama")[1]
    eng_b.prefill(prompt[:-1], 0, want_logits=False)
    b = eng_b.decode_greedy(prompt[-1], len(prompt) - 1, 24, use_graph=True)
    assert a == b
    # oracle greedy continuation (f32) should agree on at least the first tokens
    oracle.forward(prompt[:-1], 0)
    tok, pos, ref = prompt[-1], len(prompt) - 1, []
    for _ in range(8):
        tok = int(oracle.forward([tok], pos)[0].argmax())
        ref.append(tok)
        pos += 1
    assert a[:4] == ref[:4]


@pytest.mark.parametrize("name", ["tiny-llama31", "tiny-qwen3", "tiny-qwen3-moe"])
def test_tensor_core_prefill_matches_oracle(tmp_models, name):
    """Prompt chunks > 8 tokens run on the tcgen05 GEMM path (bf16 activations); later decode steps read its KV cache."""
    mf, eng, oracle = _setup(tmp_models, name)
    toks = [(7 * i + 3) % 500 + 1 for i in range(45)]
    ref = oracle.forward(toks, 0)
    lg = eng.prefill(toks, 0).clone()   # the engine returns a view of its logits buffer
    assert (lg - ref[-1]).abs().max().item() < 0.12
    # continue decoding on top of the tensor-core-written KV cache
    nxt = eng.step(11, len(toks))
    ref2 = oracle.forward([11], len(toks))
    assert (nxt - ref2[0]).abs().max().item() < 0.12
    # and the GEMV-path prefill gives (nearly) the same logits
    eng_b = _setup(tmp_models, name)[1]
    eng_b.use_tc_prefill = False
    lg_b = eng_b.prefill(toks, 0)
    assert (lg - lg_b).abs().max().item() < 0.12


def test_views_outlive_engine(tmp_models):
    """`logits` is a view of engine-owned memory: it keeps the engine alive after the Engine object is dropped."""
    import gc
    eng = _setup(tmp_models, "tiny-llama31")[1]
    eng.step(3, 0)
    logits, want = eng.logits, eng.logits.clone()
    del eng
    gc.collect()
    other = _setup(tmp_models, "tiny-llama31")[1]   # would be handed the freed memory if the view did not hold it
    torch.cuda.synchronize()
    assert torch.equal(logits.clone(), want) and other.logits.data_ptr() != logits.data_ptr()


@pytest.mark.parametrize("name", ["tiny-llama31", "tiny-qwen3"])
def test_persistent_decode_kernel(tmp_models, name):
    """The one-launch-per-token megakernel must reproduce the multi-kernel path (logits close, greedy tokens equal)."""
    mf, eng, oracle = _setup(tmp_models, name)
    eng.enable_mega(False)          # reference: the multi-kernel PDL chain
    prompt = [3, 17, 250, 9, 44, 101, 7]
    eng.prefill(prompt[:-1], 0, want_logits=False)
    ref_toks = eng.decode_greedy(prompt[-1], len(prompt) - 1, 40)
    eng_m = _setup(tmp_models, name)[1]
    eng_m.enable_mega()
    eng_m.prefill(prompt[:-1], 0, want_logits=False)
    lg_m = eng_m.step(prompt[-1], len(prompt) - 1).clone()
    eng_c = _setup(tmp_models, name)[1]
    eng_c.enable_mega(False)
    eng_c.prefill(prompt[:-1], 0, want_logits=False)
    lg_c = eng_c.step(prompt[-1], len(prompt) - 1).clone()
    assert (lg_m - lg_c).abs().max().item() < 2e-3
    for use_graph in (False, True):
        e = _setup(tmp_models, name)[1]
        e.enable_mega()
        e.prefill(prompt[:-1], 0, want_logits=False)
        toks = e.decode_greedy(prompt[-1], len(prompt) - 1, 40, use_graph=use_graph)
        agree = sum(a == b for a, b in zip(toks, ref_toks))
        assert agree >= 36, (toks, ref_toks)


@pytest.mark.parametrize("name,tol", [("tiny-llama31-f32", 2e-2), ("tiny-qwen3-f16", 2e-2), ("tiny-llama-q80", 2e-2)])
def test_dense_weight_files(tmp_models, name, tol):
    """f32 / f16 / q80 weight files run on the dense GEMV kernels with f32 activations (reference: F32_F32_F32 matmul with
    --buffer-float-type f32); compared with the oracle without activation quantisation (tolerance = the bf16 KV cache; the oracle keeps f32 KV)."""
    from distributed_llama_b200.formats import ModelFile
    from distributed_llama_b200.models.loader import load_device_weights
    from distributed_llama_b200.models.reference import OracleModel
    from distributed_llama_b200.runtime import Engine
    mf = ModelFile(tmp_models[name][0])
    eng = Engine(load_device_weights(mf))
    assert eng.dense and not eng.mega
    oracle = OracleModel(mf, act_quant="none", device="cuda")
    toks = [3, 17, 250, 9, 44, 101, 7, 300, 12, 5, 77]
    ref = oracle.forward(toks, 0)
    lg = eng.prefill(toks[:8], 0).clone()                  # one 8-token batch
    assert (lg - ref[7]).abs().max().item() < tol
    for i in range(8, len(toks)):                          # then token by token
        lg = eng.step(toks[i], i)
        assert (lg - ref[i]).abs().max().item() < tol, i
    # device-resident greedy loop (logits kernel + arg-max/advance kernel, graph replay) follows the oracle's arg-max
    out = eng.decode_greedy(toks[-1], len(toks) - 1, 6)
    tok, pos, want = toks[-1], len(toks) - 1, []
    for _ in range(3):
        tok = int(oracle.forward([tok], pos)[0].argmax())
        want.append(tok)
        pos += 1
    assert out[:3] == want
