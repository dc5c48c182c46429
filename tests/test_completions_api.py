"""POST /v1/completions of the Python API server (apps/api_server.py) on the CPU, over a fake inference object with a `score` method:
the shape of the `logprobs` object, its null first entries, text offsets, finish reasons and the 400 responses."""
import http.client
import json
import socket
import threading
import time
from types import SimpleNamespace

import pytest
import torch


@pytest.fixture(scope="module")
def server(tmp_path_factory):
    from distributed_llama_b200 import host
    from distributed_llama_b200.apps import api_server as py_api
    from distributed_llama_b200.apps.args import parse_args
    from distributed_llama_b200.models.synthetic import write_synthetic_tokenizer
    from distributed_llama_b200.runtime.engine import ScoreResult

    tok_path = str(tmp_path_factory.mktemp("completions") / "t.t")
    write_synthetic_tokenizer(tok_path, 512, style="llama3")
    H = host()
    tok = H.Tokenizer(tok_path)
    regular, eos = tok.regular_vocab_size, list(tok.eos_ids)[0]

    class FakeInference:
        comm = None

        def __init__(self):
            self.calls = []
            self.eos_after = 3

        def prefill(self, tokens, pos):
            self.calls.append(("prefill", list(tokens), pos))
            self.produced = 0

        def next_token(self, token, pos, sampler):
            self.produced += 1
            return eos if self.produced > self.eos_after else (token * 7 + pos * 13 + 5) % regular

        def score(self, tokens, pos, next_token=None):
            self.calls.append(("score", list(tokens), pos, next_token))
            self.produced = 0
            n = len(tokens) - (0 if next_token is not None else 1)
            return ScoreResult(torch.tensor([-(pos + i + 1) / 8 for i in range(n)], dtype=torch.float32),
                               torch.tensor([(t + 1) % regular for t in tokens], dtype=torch.int32),
                               torch.full((len(tokens),), -0.5, dtype=torch.float32))

    port = _free_port()
    args = parse_args(["--model", "stub.m", "--tokenizer", tok_path, "--host", "127.0.0.1", "--port", str(port), "--temperature", "0"], False)
    inf = FakeInference()
    ctx = SimpleNamespace(args=args, sess=None, inference=inf, tokenizer=tok, sampler=H.Sampler(tok.vocab_size, 0.0, 0.9, 1),
                          header=SimpleNamespace(seq_len=64, vocab_size=tok.vocab_size))
    th = threading.Thread(target=py_api.serve, args=(ctx, 0), daemon=True)
    th.start()
    for _ in range(100):
        try:
            socket.create_connection(("127.0.0.1", port), timeout=0.2).close()
            break
        except OSError:
            time.sleep(0.05)
    return port, inf, tok


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _post(port, body):
    c = http.client.HTTPConnection("127.0.0.1", port, timeout=20)
    c.request("POST", "/v1/completions", json.dumps(body), {"Content-Type": "application/json"})
    r = c.getresponse()
    data = r.read()
    c.close()
    return r.status, r.getheader("Content-Type"), json.loads(data)


def test_echo_scores_the_prompt(server):
    port, inf, tok = server
    prompt = "the llama scores"
    ids = list(tok.encode(prompt, True, True))
    n = len(ids)
    inf.calls.clear()
    st, ctype, j = _post(port, {"prompt": prompt, "echo": True, "logprobs": 1, "max_tokens": 0})
    assert st == 200 and ctype.startswith("application/json") and j["object"] == "text_completion"
    assert inf.calls == [("score", ids, 0, None)]                 # the score pass is the prompt's prefill
    c = j["choices"][0]
    lp = c["logprobs"]
    assert set(lp) == {"tokens", "token_logprobs", "top_logprobs", "text_offset"}
    assert len(lp["tokens"]) == len(lp["token_logprobs"]) == len(lp["top_logprobs"]) == len(lp["text_offset"]) == n
    assert lp["token_logprobs"][0] is None and lp["top_logprobs"][0] is None
    assert lp["token_logprobs"][1:] == [-(i + 1) / 8 for i in range(n - 1)]
    assert all(len(d) == 1 and list(d.values()) == [-0.5] for d in lp["top_logprobs"][1:])
    assert c["text"] == "".join(lp["tokens"]) and c["text"].endswith(prompt)
    for tok_text, off in zip(lp["tokens"], lp["text_offset"]):
        assert c["text"][off:off + len(tok_text)] == tok_text
    assert c["finish_reason"] == "length" and j["usage"] == {"completion_tokens": 0, "prompt_tokens": n, "total_tokens": n}


def test_generated_tokens_get_logprobs(server):
    port, inf, tok = server
    prompt = "hello"
    ids = list(tok.encode(prompt, True, True))
    n = len(ids)
    inf.calls.clear()
    st, _, j = _post(port, {"prompt": prompt, "logprobs": 0, "max_tokens": 2})
    assert st == 200
    c = j["choices"][0]
    assert c["finish_reason"] == "length" and len(c["logprobs"]["tokens"]) == 2
    assert inf.calls[0] == ("prefill", ids[:-1], 0)
    kind, toks, pos, nxt = inf.calls[1]                             # one pass over the last prompt token + the completion
    assert kind == "score" and pos == n - 1 and toks[0] == ids[-1] and len(toks) == 2 and nxt is not None
    assert c["logprobs"]["token_logprobs"] == [-(n + i) / 8 for i in range(2)]
    assert c["logprobs"]["top_logprobs"] == [{}, {}]                # logprobs: 0 -> no alternatives
    assert c["logprobs"]["text_offset"][0] == 0 and c["text"] == "".join(c["logprobs"]["tokens"])
    # EOS ends the completion with finish_reason "stop"; without logprobs there is no score pass
    inf.calls.clear()
    st, _, j = _post(port, {"prompt": prompt, "max_tokens": 16})
    c = j["choices"][0]
    assert st == 200 and c["finish_reason"] == "stop" and c["logprobs"] is None and j["usage"]["completion_tokens"] == 3
    assert [k[0] for k in inf.calls] == ["prefill"]


@pytest.mark.parametrize("body", [{"prompt": "x", "logprobs": 2}, {"prompt": "x", "stream": True}, {"prompt": "x " * 200},
                                  {"prompt": ["x"]}, {"prompt": "x", "max_tokens": -1}])
def test_bad_requests_get_400(server, body):
    port, inf, _ = server
    st, ctype, j = _post(port, body)
    assert st == 400 and ctype.startswith("application/json") and "message" in j["error"]
    st, _, _ = _post(port, {"prompt": "still serving", "max_tokens": 1})
    assert st == 200
