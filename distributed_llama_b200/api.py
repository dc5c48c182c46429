"""Public Python API: load a `.m`/`.t` pair and run inference on the local rank(s).

    from distributed_llama_b200.api import InferenceSession
    s = InferenceSession("model.m", "tokenizer.t")
    text = s.generate("Hello", steps=64)

This is the call path `dllama inference|chat|perplexity` and `dllama-api` sit on (reference: runInferenceApp,
src/app.cpp:232-304).
"""
from __future__ import annotations

import time
from dataclasses import dataclass
from typing import Callable, List, Optional, Sequence

import numpy as np
import torch

from . import host
from .formats.model_file import ModelFile


@dataclass
class GenerationStats:
    n_prompt_tokens: int = 0
    n_generated: int = 0
    prefill_ms: float = 0.0
    decode_ms: float = 0.0


class InferenceSession:
    def __init__(self, model_path: str, tokenizer_path: Optional[str] = None, max_seq_len: int = 0,
                 temperature: float = 0.0, topp: float = 0.9, seed: int = 12345, device: Optional[str] = None,
                 max_batch: int = 8, use_pdl: bool = True, comm=None, moe_mode: str = "auto"):
        from .models.loader import load_device_weights
        from .runtime.engine import Engine

        self.model_file = ModelFile(model_path, max_seq_len)
        self.header = self.model_file.header
        self.comm = comm
        rank = comm.rank if comm is not None else 0
        n_ranks = comm.world_size if comm is not None else 1
        if device is None:
            device = f"cuda:{torch.cuda.current_device()}"
        self.device = torch.device(device)
        self.weights = load_device_weights(self.model_file, rank, n_ranks, self.device, moe_mode=moe_mode, comm=comm)
        self.engine = Engine(self.weights, max_batch=max_batch, use_pdl=use_pdl, comm=comm)
        H = host()
        self.tokenizer = H.Tokenizer(tokenizer_path) if tokenizer_path else None
        vocab = self.tokenizer.vocab_size if self.tokenizer else self.header.vocab_size
        self.sampler = H.Sampler(vocab, temperature, topp, seed)
        if self.tokenizer and self.tokenizer.vocab_size < self.header.vocab_size:
            self.engine.set_vocab_limit(self.tokenizer.vocab_size)
        self.pos = 0
        self._dev_seeded = None
        self._pin_in = torch.zeros(2, dtype=torch.int32).pin_memory()
        self._pin_out = torch.zeros(1, dtype=torch.int32).pin_memory()

    # ---- token level ----
    def reset(self):
        self.pos = 0

    def prefill(self, tokens: Sequence[int]) -> None:
        """Evaluates tokens at positions pos..pos+n-1 without producing logits (prompt minus its last token)."""
        if tokens:
            self.engine.prefill(tokens, self.pos, want_logits=False)
            self.pos += len(tokens)

    def score(self, tokens: Sequence[int]):
        """Evaluates tokens at positions pos..pos+n-1 and returns their scores (runtime.engine.ScoreResult: log P(tokens[i+1] |
        tokens[..i]), top-1 ids and log-probabilities). Advances pos by n-1, like prefill(tokens[:-1]): feeding tokens[-1] to
        next_token continues the sequence."""
        res = self.engine.score(tokens, self.pos)
        self.pos += len(tokens) - 1
        return res

    def forward_logits(self, token: int) -> torch.Tensor:
        lg = self.engine.step(token, self.pos)
        self.pos += 1
        return lg

    def next_token(self, token: int) -> int:
        """One decode step with host-visible result: H2D (token,pos) from pinned memory, forward + sampling, D2H."""
        if self.sampler.temperature == 0.0:
            self._pin_in[0] = token
            self._pin_in[1] = self.pos
            eng = self.engine
            eng.tokens[:1].copy_(self._pin_in[:1], non_blocking=True)
            eng.pos[:1].copy_(self._pin_in[1:2], non_blocking=True)
            eng.run_decode_step()
            self._pin_out.copy_(eng.tokens[:1], non_blocking=True)
            torch.cuda.current_stream().synchronize()
            eng.check_abort()
            self.pos += 1
            return int(self._pin_out[0])
        eng = self.engine
        if self.device.type == "cuda" and not getattr(eng, "_parts", False):
            # temperature / top-p on the device (csrc/cuda/sampler.cu): only the sampled token crosses PCIe
            gen = (self.sampler.seed, self.sampler.seed_generation)
            if self._dev_seeded != gen:
                eng.seed_sampler(self.sampler.seed)
                self._dev_seeded = gen
            eng.step_sampled(token, self.pos, self.sampler.temperature, self.sampler.topp)
            self._pin_out.copy_(eng.tokens[:1], non_blocking=True)
            torch.cuda.current_stream().synchronize()
            eng.check_abort()
            self.pos += 1
            return int(self._pin_out[0])
        lg = self.forward_logits(token)
        return int(self.sampler.sample(lg.float().cpu().numpy()))

    # ---- text level ----
    def generate(self, prompt: str, steps: int, on_piece: Optional[Callable[[str], None]] = None) -> str:
        assert self.tokenizer is not None
        toks = self.tokenizer.encode(prompt, True, True)
        self.prefill(toks[:-1])
        tok = toks[-1]
        self.tokenizer.reset_decoder()
        out = []
        while self.pos < min(steps, self.header.seq_len):
            tok = self.next_token(tok)
            piece = self.tokenizer.decode(tok).decode("utf-8", errors="replace")
            out.append(piece)
            if on_piece:
                on_piece(piece)
            if self.tokenizer.is_eos(tok):
                break
        return "".join(out)
