"""`dllama-api`: OpenAI-style HTTP server (reference src/dllama-api.cpp:43-632, src/api-types.hpp).

Routes: POST /v1/chat/completions (JSON or SSE-chunked stream), POST /v1/completions (prompt log-probabilities and plain
completions, JSON only), GET /v1/models, OPTIONS * (CORS pre-flight), else 404.
Single request at a time over one global KV sequence, with the reference's NaiveCache prefix reuse: if the new message
history extends the cached one, generation restarts from the cached end position instead of 0.
Deliberate fixes over the reference (SURVEY A.2): request `temperature`/`top_p` are applied, `finish_reason` is "stop"
on non-stream responses.
"""
from __future__ import annotations

import json
import socket
import sys
import time
from typing import Dict, List, Optional, Tuple

from .. import host
from .args import AppArgs, parse_args
from .cli import make_chat_tools
from .runtime import AppContext, run_inference_app


class NaiveCache:
    """(endPos, message) per chat turn; reuse only if *all* cached messages are an exact prefix of the new history."""

    def __init__(self):
        self.items: List[Tuple[int, Tuple[str, str]]] = []

    def push(self, end_pos: int, msg: Tuple[str, str]):
        self.items.append((end_pos, msg))

    def clear(self):
        self.items.clear()

    def resolve_delta_prompt(self, messages: List[Tuple[str, str]]) -> Tuple[List[Tuple[str, str]], int]:
        n = len(self.items)
        if n == 0:
            return messages, 0
        if len(messages) > n and all(self.items[i][1] == messages[i] for i in range(n)):
            start = self.items[n - 1][0]
            print(f"🐤 Found naive cache for {n} messages, pos={start}")
            return messages[n:], start
        self.clear()
        return messages, 0


class HttpRequest:
    def __init__(self, conn: socket.socket):
        self.conn = conn
        self.method = "UNKNOWN"
        self.path = ""
        self.headers: Dict[str, str] = {}
        self.body = b""
        self.json = None

    @staticmethod
    def read(conn: socket.socket) -> "HttpRequest":
        req = HttpRequest(conn)
        data = b""
        while b"\r\n\r\n" not in data and b"\n\n" not in data:
            chunk = conn.recv(65536)
            if not chunk:
                raise ConnectionError("Error while reading headers from socket")
            data += chunk
        sep = b"\r\n\r\n" if b"\r\n\r\n" in data else b"\n\n"
        head, rest = data.split(sep, 1)
        lines = head.decode("latin-1").splitlines()
        parts = lines[0].split()
        if len(parts) >= 2:
            req.method, req.path = parts[0].upper(), parts[1]
        for ln in lines[1:]:
            if ":" in ln:
                k, v = ln.split(":", 1)
                req.headers[k.strip().lower()] = v.strip()
        length = int(req.headers.get("content-length", "0") or 0)
        if len(rest) > length > 0:
            raise ValueError("Received more body data than Content-Length header said")
        while len(rest) < length:
            chunk = conn.recv(length - len(rest))
            if not chunk:
                raise ConnectionError("Error while reading body from socket")
            rest += chunk
        req.body = rest
        if rest:
            req.json = json.loads(rest.decode("utf-8"))
        return req

    def _send(self, data: bytes):
        self.conn.sendall(data)

    def write_cors(self):
        self._send(b"HTTP/1.1 204 No Content\r\nAccess-Control-Allow-Origin: *\r\nAccess-Control-Allow-Methods: GET, POST, PUT, DELETE\r\n"
                   b"Access-Control-Allow-Headers: Content-Type, Authorization\r\nConnection: close\r\n\r\n")

    def write_not_found(self):
        self._send(b"HTTP/1.1 404 Not Found\r\nConnection: close\r\nContent-Length: 9\r\n\r\nNot Found")

    def write_json(self, text: str):
        body = text.encode("utf-8")
        self._send(b"HTTP/1.1 200 OK\r\nAccess-Control-Allow-Origin: *\r\nContent-Type: application/json; charset=utf-8\r\n"
                   b"Connection: close\r\nContent-Length: " + str(len(body)).encode() + b"\r\n\r\n" + body)

    def write_error(self, status: int, message: str):
        body = json.dumps({"error": {"message": message, "type": "invalid_request_error"}}).encode("utf-8")
        reason = {400: "Bad Request"}.get(status, "Error")
        self._send(f"HTTP/1.1 {status} {reason}\r\n".encode() + b"Access-Control-Allow-Origin: *\r\nContent-Type: application/json; charset=utf-8\r\n"
                   b"Connection: close\r\nContent-Length: " + str(len(body)).encode() + b"\r\n\r\n" + body)

    def write_stream_start(self):
        self._send(b"HTTP/1.1 200 OK\r\nAccess-Control-Allow-Origin: *\r\nContent-Type: text/event-stream; charset=utf-8\r\n"
                   b"Connection: close\r\nTransfer-Encoding: chunked\r\n\r\n")

    def write_stream_chunk(self, data: str):
        b = data.encode("utf-8")
        self._send(("%x" % len(b)).encode() + b"\r\n" + b + b"\r\n")

    def write_stream_end(self):
        self._send(b"0000\r\n\r\n")


def chunk_json(delta: Optional[str], stop: bool) -> str:
    choice = {"index": 0, "finish_reason": "stop" if stop else ""}
    if not stop:
        choice["delta"] = {"role": "assistant", "content": delta}
    return json.dumps({"id": "cmpl-c0", "object": "chat.completion", "created": int(time.time()), "model": "Distributed Model",
                       "choices": [choice]})


class ApiServer:
    def __init__(self, ctx: AppContext):
        self.ctx = ctx
        self.cache = NaiveCache()
        self.gen, self.det = make_chat_tools(ctx)
        self.H = host()

    def complete(self, req: HttpRequest):
        ctx, H = self.ctx, self.H
        tok, inf, h, smp = ctx.tokenizer, ctx.inference, ctx.header, ctx.sampler
        body = req.json or {}
        messages = [(m["role"], m["content"]) for m in body["messages"]]
        stream = bool(body.get("stream", False))
        max_tokens = int(body.get("max_tokens", -1))
        smp.set_temperature(float(body.get("temperature", ctx.args.temperature)))
        smp.set_topp(float(body.get("top_p", ctx.args.topp)))
        if "seed" in body:
            smp.set_seed(int(body["seed"]))
        delta_prompt, start_pos = self.cache.resolve_delta_prompt(list(messages))
        content, public = self.gen.generate(delta_prompt, True)
        print(f"🔹{content.decode('utf-8', errors='replace')}🔸", end="")
        tokens = tok.encode(content, start_pos == 0, True)
        n_prompt = len(tokens)
        prompt_end = min(start_pos + n_prompt - 1, h.seq_len)
        max_pred = min(prompt_end + max_tokens, h.seq_len) if max_tokens > 0 else h.seq_len
        for m in delta_prompt:
            self.cache.push(prompt_end, m)
        buffer = ""
        if stream:
            req.write_stream_start()
        if public:
            p = public.decode("utf-8", errors="replace")
            if stream:
                req.write_stream_chunk("data: " + chunk_json(p, False) + "\r\n\r\n")
            buffer += p
        pos = start_pos
        n = prompt_end - pos
        inf.prefill(tokens[:n], pos)
        pos += n
        token = tokens[n] if n < len(tokens) else tokens[-1]
        tok.reset_decoder()
        self.det.reset()
        greedy = smp.temperature == 0.0
        while pos < max_pred:
            token = inf.next_token(token, pos, smp)
            piece = tok.decode(token)
            kind = self.det.append(token, piece)
            if piece:
                print(piece.decode("utf-8", errors="replace"), end="", flush=True)
            if kind in (H.NOT_EOS, H.EOS):
                delta = self.det.get_delta()
                if delta:
                    d = delta.decode("utf-8", errors="replace")
                    if stream:
                        req.write_stream_chunk("data: " + chunk_json(d, False) + "\r\n\r\n")
                    buffer += d
                self.det.reset()
            pos += 1
            if kind == H.EOS:
                break
        if pos == h.seq_len:
            self.cache.clear()
        else:
            self.cache.push(pos, ("assistant", buffer))
        if stream:
            req.write_stream_chunk("data: " + chunk_json(None, True) + "\r\n\r\n")
            req.write_stream_chunk("data: [DONE]")
            req.write_stream_end()
        else:
            n_completion = pos - prompt_end
            req.write_json(json.dumps({
                "id": "cmpl-j0", "object": "chat.completion", "created": int(time.time()), "model": "Distributed Model",
                "usage": {"completion_tokens": n_completion, "prompt_tokens": n_prompt, "total_tokens": n_prompt + n_completion},
                "choices": [{"index": 0, "message": {"role": "assistant", "content": buffer}, "finish_reason": "stop"}]}))
        print("🔶")

    def text_completion(self, req: HttpRequest):
        """POST /v1/completions, the OpenAI legacy completions contract that evaluation harnesses use for log-likelihoods. The
        prompt is tokenized with BOS and no chat template. With `echo` and `logprobs`, the prompt is scored on the device
        (InferenceSession.score), which is also its prefill; generated tokens come from the decode loop, and with `logprobs` one
        score pass over the last prompt token and the completion gives their log-probabilities afterwards. `tokens[i]` is the text
        the tokenizer's decoder emits for token i, and `text_offset[i]` its character offset in `text`."""
        ctx = self.ctx
        tok, inf, h, smp = ctx.tokenizer, ctx.inference, ctx.header, ctx.sampler
        body = req.json if isinstance(req.json, dict) else {}
        prompt, logprobs, max_tokens = body.get("prompt"), body.get("logprobs"), body.get("max_tokens", 16)
        if body.get("stream"):
            return req.write_error(400, "stream is not supported on /v1/completions")
        if not isinstance(prompt, str):
            return req.write_error(400, "prompt must be a string")
        if logprobs is not None and (type(logprobs) is not int or not 0 <= logprobs <= 1):
            return req.write_error(400, "logprobs must be null, 0 or 1")
        if type(max_tokens) is not int or max_tokens < 0:
            return req.write_error(400, "max_tokens must be a non-negative integer")
        tokens = list(tok.encode(prompt, True, True))
        n = len(tokens)
        if n > h.seq_len:
            return req.write_error(400, f"the prompt has {n} tokens, more than the context length ({h.seq_len})")
        echo = bool(body.get("echo", False))
        smp.set_temperature(float(body.get("temperature", ctx.args.temperature)))
        smp.set_topp(float(body.get("top_p", ctx.args.topp)))
        if "seed" in body:
            smp.set_seed(int(body["seed"]))
        self.cache.clear()   # this request overwrites the KV rows the chat cache points at
        prompt_scores = None
        if echo and logprobs is not None:
            prompt_scores = inf.score(tokens, 0)
        else:
            inf.prefill(tokens[:-1], 0)
        pos, token, generated, finish = n - 1, tokens[-1], [], "length"
        while len(generated) < max_tokens and pos < h.seq_len:
            token = inf.next_token(token, pos, smp)
            pos += 1
            if tok.is_eos(token):
                finish = "stop"
                break
            generated.append(token)
        tok.reset_decoder()
        ids = (tokens if echo else []) + generated
        strs = [tok.decode(t).decode("utf-8", errors="replace") for t in ids]
        choice = {"index": 0, "text": "".join(strs), "logprobs": None, "finish_reason": finish}
        if logprobs is not None:
            def top(i, lp):
                return {tok.piece(i).decode("utf-8", errors="replace"): lp} if logprobs else {}
            token_lp, top_lp = [], []
            if echo:
                token_lp = [None] + prompt_scores.logprobs.tolist()
                top_lp = [None] + [top(i, lp) for i, lp in zip(prompt_scores.top_ids.tolist()[:n - 1], prompt_scores.top_logprobs.tolist())]
            if generated:
                s = inf.score([tokens[-1]] + generated[:-1], n - 1, next_token=generated[-1])
                token_lp += s.logprobs.tolist()
                top_lp += [top(i, lp) for i, lp in zip(s.top_ids.tolist(), s.top_logprobs.tolist())]
            offsets, off = [], 0
            for s_ in strs:
                offsets.append(off)
                off += len(s_)
            choice["logprobs"] = {"tokens": strs, "token_logprobs": token_lp, "top_logprobs": top_lp, "text_offset": offsets}
        n_completion = len(generated)
        req.write_json(json.dumps({
            "id": "cmpl-t0", "object": "text_completion", "created": int(time.time()), "model": "Distributed Model",
            "usage": {"completion_tokens": n_completion, "prompt_tokens": n, "total_tokens": n + n_completion},
            "choices": [choice]}))

    def models(self, req: HttpRequest):
        name = self.ctx.args.model.replace("\\", "/").split("/")[-1]
        req.write_json(json.dumps({"object": "list", "data": [{"id": name, "object": "model", "created": 0, "owned_by": "user"}]}))


def serve(ctx: AppContext, max_requests: int = 0) -> None:
    a = ctx.args
    srv = socket.socket(socket.AF_INET, socket.SOCK_STREAM)
    srv.setsockopt(socket.SOL_SOCKET, socket.SO_REUSEADDR, 1)
    srv.bind((a.host, a.port))
    srv.listen(8)
    api = ApiServer(ctx)
    if a.host in ("0.0.0.0", "127.0.0.1"):
        print(f"Server URL: http://localhost:{a.port}/v1/", flush=True)
    served = 0
    while max_requests == 0 or served < max_requests:
        conn, _ = srv.accept()
        try:
            req = HttpRequest.read(conn)
            print(f"🔷 {req.method} {req.path}")
            if req.method == "OPTIONS":
                req.write_cors()
            elif req.method == "POST" and req.path == "/v1/chat/completions":
                api.complete(req)
            elif req.method == "POST" and req.path == "/v1/completions":
                api.text_completion(req)
            elif req.method == "GET" and req.path == "/v1/models":
                api.models(req)
            else:
                req.write_not_found()
        except (ConnectionError, BrokenPipeError, ValueError, KeyError, json.JSONDecodeError) as e:
            print(f"Socket error: {e}")
        finally:
            conn.close()
            served += 1
    srv.close()


USAGE = """Usage: dllama-api {--model <path>} {--tokenizer <path>} [--host <addr>] [--port <p>]
        [--buffer-float-type {f32|f16|q40|q80}] [--max-seq-len <max>] [--gpus <n>] [--workers <ip:port> ...]
        [--temperature <temp>] [--topp <t>] [--seed <s>] [--chat-template {llama2|llama3|deepSeek3|chatml}]
"""


def main(argv=None) -> int:
    import os
    argv = list(sys.argv[1:] if argv is None else argv)
    args = parse_args(argv, False)
    if args.help:
        sys.stderr.write(USAGE)
        return 0
    if args.gpus > 1 and os.environ.get("DLLAMA_SPAWNED") != "1" and int(os.environ.get("WORLD_SIZE", "1")) == 1:
        # Supervisor of a tensor-parallel serving job: a rank that loses a peer (control-channel heartbeat, device-side wait timeout)
        # exits non-zero and torchrun tears the job down; the whole job is then started again after 3 s — the reference's root retry
        # loop + worker re-listen loop (dllama-api.cpp:616-628, app.cpp:306-365).
        import subprocess
        attempt = 0
        while True:
            port = 29500 + ((os.getpid() + 7 * attempt) % 2000)
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
                   "--master-port", str(port), "-m", "distributed_llama_b200.apps.api_server"] + argv
            try:
                rc = subprocess.call(cmd, env=dict(os.environ, DLLAMA_SPAWNED="1"))
            except KeyboardInterrupt:
                return 130
            if rc == 0 or rc < 0 or rc == 130:
                return rc
            print(f"🚨 Inference error: the tensor-parallel job exited with code {rc}\n🔄 Retrying in 3 seconds...", flush=True)
            time.sleep(3)
            attempt += 1
    # the reference retries runInferenceApp forever on connection / executor errors (dllama-api.cpp:616-628)
    while True:
        try:
            run_inference_app(args, serve)
            return 0
        except (ConnectionError, RuntimeError) as e:
            print(f"🚨 Inference error: {e}")
            if int(os.environ.get("WORLD_SIZE", "1")) > 1:
                return 1          # a lost rank cannot be re-joined from inside the job: the supervisor above restarts the whole job
            print("🔄 Retrying in 3 seconds...")
            time.sleep(3)
            args.info = False


if __name__ == "__main__":
    sys.exit(main())
