"""Prompt scoring on the device: the score kernel (csrc/cuda/score.cu), Engine.score against the PyTorch oracle, its invariants,
the tensor-parallel record exchange and POST /v1/completions of dllama-api."""
import http.client
import json
import math
import os
import socket
import subprocess
import sys
import time

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _score_rows(logits, targets, limit=0):
    from distributed_llama_b200.ops import cuda_lib as cl
    T, ld = logits.shape[0], logits.stride(0)
    vocab = logits.shape[1]
    tg = torch.tensor(targets, dtype=torch.int32, device="cuda")
    lp = torch.empty(T, dtype=torch.float32, device="cuda")
    ids = torch.empty(T, dtype=torch.int32, device="cuda")
    top = torch.empty(T, dtype=torch.float32, device="cuda")
    cl.check(cl.lib().dl_score_rows(logits.data_ptr(), T, vocab, ld, tg.data_ptr(), limit, lp.data_ptr(), ids.data_ptr(), top.data_ptr(),
                                    cl.stream_ptr()), "score_rows")
    torch.cuda.synchronize()
    return lp.cpu(), ids.cpu(), top.cpu()


@pytest.mark.parametrize("vocab,ld,limit", [(512, 512, 0), (1003, 1003, 0), (4099, 4104, 4000), (128256, 128256, 128000)])
def test_score_kernel_matches_log_softmax(vocab, ld, limit):
    """Vocabularies that are not a multiple of the block size, padded row strides (vector and scalar loads), a top-1 limit below
    the vocabulary, exact ties (the lowest index wins) and rows without a target."""
    g = torch.Generator(device="cuda").manual_seed(vocab)
    T = 37
    buf = torch.randn(T, ld, generator=g, device="cuda") * 4
    x = buf[:, :vocab]
    x[3, 10] = x[3, 700 % vocab] = x[3].max() + 1.0           # tie: index 10 must win
    x[4, vocab - 1] = x[4].max() + 5.0                        # the largest logit lies beyond the limit when one is set
    x[5, :] = 0.25                                            # all equal: index 0
    targets = [(7 * t + 1) % vocab for t in range(T)]
    targets[2] = targets[9] = -1
    targets[4] = vocab - 1
    lp, ids, top = _score_rows(x, targets, limit)
    lsm = torch.log_softmax(x.double(), dim=-1).cpu()
    lim = limit or vocab
    want_ids = lsm[:, :lim].argmax(dim=-1)
    assert torch.equal(ids.long(), want_ids), (ids[:8], want_ids[:8])
    assert ids[3] == 10 and ids[5] == 0
    assert (top.double() - lsm.gather(1, want_ids[:, None])[:, 0]).abs().max().item() < 1e-5
    for t in range(T):
        if targets[t] < 0:
            assert math.isnan(lp[t].item())
        else:
            assert abs(lp[t].item() - lsm[t, targets[t]].item()) < 1e-5, t
    again = _score_rows(x, targets, limit)
    assert all(torch.equal(a.view(torch.int32), b.view(torch.int32)) for a, b in zip((lp, ids, top), again))


def _engine(path, **kw):
    from distributed_llama_b200.formats import ModelFile
    from distributed_llama_b200.models.loader import load_device_weights
    from distributed_llama_b200.runtime import Engine
    return Engine(load_device_weights(ModelFile(path)), **kw)


def _text(n, mul=7, add=3):
    return [(mul * i + add) % 500 + 1 for i in range(n)]


def _oracle_scores(path, toks, act_quant="q80"):
    from distributed_llama_b200.formats import ModelFile
    from distributed_llama_b200.models.reference import OracleModel
    ref = OracleModel(ModelFile(path), act_quant=act_quant, device="cuda").forward(toks, 0)
    lsm = torch.log_softmax(ref.double(), dim=-1).cpu()
    tg = torch.tensor(toks[1:])
    return lsm[:-1].gather(1, tg[:, None])[:, 0], lsm.max(dim=-1).values


# Mean |engine - oracle| per token over the text: half the 0.12 per-logit tolerance of test_tensor_core_prefill_matches_oracle.
# Rounding errors of the bf16 prefill do not sit at that bound for every token, so a mean above it points at a systematic offset,
# such as a wrong normaliser or a target shifted by one row, that the per-token bound alone would let through.
MEAN_BOUND = 0.06


@pytest.mark.parametrize("name", ["tiny-llama", "tiny-llama31", "tiny-qwen3", "tiny-qwen3-moe"])
def test_engine_score_matches_oracle(tmp_models, name):
    path = tmp_models[name][0]
    eng = _engine(path)
    n = min(eng.seq_len, 450)        # tiny-llama31: 450 tokens = 3 chunks; the others fill their 256-token context (2 chunks)
    toks = _text(n)
    assert n > eng.score_max_tokens  # cross-chunk targets are exercised
    res = eng.score(toks, 0)
    assert res.logprobs.shape == (n - 1,) and res.top_ids.shape == (n,) and res.top_logprobs.shape == (n,)
    assert res.logprobs.dtype == torch.float32 and res.top_ids.dtype == torch.int32
    want, want_top = _oracle_scores(path, toks)
    err = (res.logprobs.double() - want).abs()
    err_top = (res.top_logprobs.double() - want_top).abs()
    print(f"{name}: max {err.max().item():.4g} mean {err.mean().item():.4g} top max {err_top.max().item():.4g}")
    assert err.max().item() < 0.25 and err_top.max().item() < 0.25
    assert err.mean().item() < MEAN_BOUND


def test_engine_score_invariants(tmp_models):
    path = tmp_models["tiny-llama31"][0]
    toks = _text(420, 13, 5)
    a = _engine(path).score(toks, 0)
    b = _engine(path).score(toks, 0)
    assert all(torch.equal(x.view(torch.int32), y.view(torch.int32)) for x, y in
               zip((a.logprobs, a.top_ids, a.top_logprobs), (b.logprobs, b.top_ids, b.top_logprobs)))
    small = _engine(path, max_prefill=64)
    assert small.score_max_tokens == 64
    c = small.score(toks, 0)
    assert (a.logprobs - c.logprobs).abs().max().item() < 2e-3
    assert (a.top_logprobs - c.top_logprobs).abs().max().item() < 2e-3


@pytest.mark.parametrize("name", ["tiny-llama31", "tiny-qwen3-moe"])
def test_score_then_decode_equals_prefill_then_decode(tmp_models, name):
    """score(p) writes the same KV rows as prefill(p[:-1]) (plus the row of p[-1], which the next decode step rewrites)."""
    path = tmp_models[name][0]
    p = _text(100, 3, 1)              # one chunk on the tensor-core path for both calls
    e1 = _engine(path)
    e1.prefill(p[:-1], 0, want_logits=False)
    want = e1.decode_greedy(p[-1], len(p) - 1, 16)
    e2 = _engine(path)
    e2.score(p, 0)
    assert e2.decode_greedy(p[-1], len(p) - 1, 16) == want


def test_session_score_advances_like_prefill(tmp_models):
    from distributed_llama_b200.api import InferenceSession
    m, t = tmp_models["tiny-llama31"]
    s = InferenceSession(m, t)
    p = _text(40)
    res = s.score(p)
    assert s.pos == len(p) - 1 and res.logprobs.shape == (len(p) - 1,)
    nxt = s.next_token(p[-1])
    s2 = InferenceSession(m, t)
    s2.prefill(p[:-1])
    assert s2.next_token(p[-1]) == nxt


def test_dense_fallback_matches_oracle(tmp_models):
    """Dense weight files have no tensor-core path: GEMV logits batches + torch.log_softmax on the device."""
    path = tmp_models["tiny-llama31-f32"][0]
    eng = _engine(path)
    assert not eng._tc_prefill_ok()
    toks = _text(60)
    res = eng.score(toks, 0)
    want, want_top = _oracle_scores(path, toks, act_quant="none")
    # the dense logits test accepts 2e-2 (bf16 KV cache); a log-probability carries the error of two logits
    assert (res.logprobs.double() - want).abs().max().item() < 4e-2
    assert (res.top_logprobs.double() - want_top).abs().max().item() < 4e-2
    assert res.top_ids.shape == (60,)


@pytest.mark.parametrize("name", ["tiny-llama31", "tiny-qwen3-moe"])
def test_tensor_parallel_score(name):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29677", os.path.join(ROOT, "tools", "score_check.py"), name]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert "SCORE_CHECK PASS" in r.stdout, r.stdout[-3000:]
    if "moe" in name:
        assert "chunks=1 " not in r.stdout, r.stdout[-3000:]   # the exchange capacity caps the chunks of this model


def _post(port, path, body, timeout=120):
    c = http.client.HTTPConnection("127.0.0.1", port, timeout=timeout)
    c.request("POST", path, json.dumps(body), {"Content-Type": "application/json"})
    r = c.getresponse()
    data = r.read()
    c.close()
    return r.status, json.loads(data)


def test_completions_endpoint(tmp_models):
    from distributed_llama_b200 import host
    from distributed_llama_b200.api import InferenceSession
    m, t = tmp_models["tiny-llama31"]
    port = 20990 + os.getpid() % 1000
    p = subprocess.Popen([os.path.join(ROOT, "dllama-api"), "--model", m, "--tokenizer", t, "--port", str(port), "--host", "127.0.0.1",
                          "--temperature", "0"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    prompt = "Hello world, the llama runs on the device and scores its prompt"
    try:
        for _ in range(300):
            try:
                socket.create_connection(("127.0.0.1", port), timeout=0.2).close()
                break
            except OSError:
                time.sleep(0.2)
        hist = [{"role": "user", "content": "Hello"}]
        st, chat1 = _post(port, "/v1/chat/completions", {"messages": hist, "max_tokens": 6})
        assert st == 200
        st, r0 = _post(port, "/v1/completions", {"prompt": prompt, "echo": True, "logprobs": 1, "max_tokens": 0})
        assert st == 200 and r0["object"] == "text_completion"
        lp0 = r0["choices"][0]["logprobs"]
        assert r0["choices"][0]["finish_reason"] == "length" and r0["usage"]["completion_tokens"] == 0
        st, r4 = _post(port, "/v1/completions", {"prompt": prompt, "logprobs": 1, "max_tokens": 4, "temperature": 0})
        assert st == 200
        c4 = r4["choices"][0]
        assert 1 <= len(c4["logprobs"]["tokens"]) <= 4 and len(c4["logprobs"]["token_logprobs"]) == len(c4["logprobs"]["tokens"])
        assert all(v <= 0.0 for v in c4["logprobs"]["token_logprobs"])
        st, bad = _post(port, "/v1/completions", {"prompt": prompt, "logprobs": 5})
        assert st == 400 and "error" in bad
        # the completions request overwrote the KV rows of the chat turn: the follow-up must not reuse them
        hist2 = hist + [{"role": "assistant", "content": chat1["choices"][0]["message"]["content"]}, {"role": "user", "content": "more"}]
        st, _ = _post(port, "/v1/chat/completions", {"messages": hist2, "max_tokens": 4})
        assert st == 200
    finally:
        p.terminate()
        out = p.communicate(timeout=30)[0]
    assert "🐤 Found naive cache" not in out, out[-2000:]
    tok = host().Tokenizer(t)
    ids = list(tok.encode(prompt, True, True))
    assert len(lp0["tokens"]) == len(ids) and lp0["token_logprobs"][0] is None and lp0["top_logprobs"][0] is None
    want = InferenceSession(m, t).score(ids).logprobs.tolist()
    assert max(abs(a - b) for a, b in zip(lp0["token_logprobs"][1:], want)) < 1e-6
