"""Python handle of the native per-rank engine (csrc/cuda/engine.cu).

Hands the weight pointers to the C++ engine, which owns the KV cache and activation buffers (`tokens`, `logits`, `k_cache`,
... are torch views of its memory), and exposes the three calls the apps need: `prefill(tokens, pos)`, `step(token, pos)`
-> logits, and the device-resident greedy decode loop `decode_greedy(n)` that replays the captured CUDA graph.
Plays the role of the reference's RootLlmInference (src/app.cpp:168-208): setBatchSize/setPosition/setToken/forward.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np
import torch

from ..models.loader import DeviceWeights
from ..ops import cuda_lib as cl


@dataclass
class ScoreResult:
    """Scores of a token sequence t[0..n): `logprobs[i]` = log P(t[i+1] | t[..i]) (length n-1, or n when the following token was
    given), `top_ids[i]` / `top_logprobs[i]` = the most likely token after t[..i] and its log-probability (length n). CPU tensors."""
    logprobs: torch.Tensor       # float32
    top_ids: torch.Tensor        # int32
    top_logprobs: torch.Tensor   # float32

    @staticmethod
    def cat(parts: Sequence["ScoreResult"]) -> "ScoreResult":
        return ScoreResult(torch.cat([p.logprobs for p in parts]), torch.cat([p.top_ids for p in parts]),
                           torch.cat([p.top_logprobs for p in parts]))


def _p(t: Optional[torch.Tensor]):
    return t.data_ptr() if t is not None else None


def _ptrs8(ptrs):
    return (C.c_void_p * 8)(*ptrs, *([None] * (8 - len(ptrs))))


class _Handle:
    """Owns the native engine. The Engine and every view of engine memory hold it, so the memory outlives them all."""

    def __init__(self, lib, cfg):
        self.lib = lib
        self.h = lib.dl_engine_create(C.byref(cfg))
        if not self.h:
            raise RuntimeError("dl_engine_create failed: cannot allocate the engine's device memory")

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.lib.dl_engine_destroy(self.h)
        except Exception:
            pass


class Engine:
    def __init__(self, weights: DeviceWeights, max_batch: int = 8, n_splits: int = 0, use_pdl: bool = True,
                 seq_len: Optional[int] = None, comm=None, max_prefill: int = 192, collectives: str = "auto"):
        self.w = w = weights
        h = w.header
        dev = w.embedding.device
        self.device = dev
        self.seq_len = seq_len or h.seq_len
        self.dense = getattr(w, "weight_kind", 0) != 0
        if self.dense:
            # f32 activations of all tokens of a launch are staged in shared memory (gemv_dense.cu)
            widest = max(h.dim, w.ff_dim, w.n_heads * h.head_dim)
            cap = (200 * 1024) // (4 * widest)
            if cap < 1:
                raise ValueError("matrix rows too wide for the dense-weight kernels on one GPU; use more ranks")
            while max_batch > cap:
                max_batch //= 2
        cfg = cl.EngineConfig(dim=h.dim, nLayers=h.n_layers, nHeads=w.n_heads, nKvHeads=w.n_kv_heads, headDim=h.head_dim,
                              ffDim=w.ff_dim, vocab=w.vocab, seqLen=self.seq_len, nExperts=h.n_experts,
                              nActiveExperts=h.n_active_experts, maxBatch=max_batch, nSplits=max(0, n_splits), rank=w.rank,
                              nRanks=w.n_ranks, numSms=0, eps=h.norm_epsilon, usePdl=1 if use_pdl else 0,
                              moeFirstExpert=w.first_expert, moeNumLocal=w.n_local_experts,
                              wType=getattr(w, "weight_kind", 0),
                              hiddenAct=1 if int(h.hidden_act) == 0 else 0,   # header: ACT_GELU = 0, ACT_SILU = 1
                              vocabFull=h.vocab_size, maxPrefill=max_prefill)
        self._lib = cl.lib()
        with torch.cuda.device(dev):
            owner = _Handle(self._lib, cfg)
        self._owner, self._h = owner, owner.h
        cl.check(self._lib.dl_engine_get_config(self._h, C.byref(cfg)), "engine_get_config")
        mb, mp = cfg.maxBatch, cfg.maxPrefill   # the engine's limits applied
        self.max_batch, self.max_prefill, self.num_sms = mb, mp, cfg.numSms
        for l, L in enumerate(w.layers):
            lp = cl.LayerPtrs(qkvQs=_p(L.qkv.qs), qkvSc=_p(L.qkv.scales), woQs=_p(L.wo.qs), woSc=_p(L.wo.scales),
                              w13Qs=_p(L.w13.qs), w13Sc=_p(L.w13.scales), w2Qs=_p(L.w2.qs), w2Sc=_p(L.w2.scales),
                              norm0=_p(L.norm0), norm1=_p(L.norm1), qNorm=_p(L.q_norm), kNorm=_p(L.k_norm), moeGate=_p(L.moe_gate))
            cl.check(self._lib.dl_engine_set_layer(self._h, l, C.byref(lp)), "engine_set_layer")
        gp = cl.GlobalPtrs(embedding=_p(w.embedding), embeddingPeers=_ptrs8(w.embedding_ptrs or []), embRowsPerRank=w.embedding_rows or 0,
                           finalNorm=_p(w.final_norm), wclsQs=_p(w.wcls.qs), wclsSc=_p(w.wcls.scales), rope=_p(w.rope))
        cl.check(self._lib.dl_engine_set_globals(self._h, C.byref(gp)), "engine_set_globals")
        b = cl.EngineBuffers()
        cl.check(self._lib.dl_engine_buffers(self._h, C.byref(b)), "engine_buffers")

        def view(ptr, shape, dtype=torch.int32):
            return cl.device_view(ptr, shape, dtype, owner, dev)
        self.tokens, self.pos, self.history = view(b.tokens, (mb,)), view(b.pos, (mb,)), view(b.history, (self.seq_len + 1,))
        self.logits, self.x = view(b.logits, (mb, w.vocab), torch.float32), view(b.x, (mb, h.dim), torch.float32)
        self.p_tokens, self.p_pos = view(b.pTokens, (mp,)), view(b.pPos, (mp,))
        self.p_targets, self.p_top_id = view(b.pTargets, (mp,)), view(b.pTopId, (mp,))
        self.p_logprob, self.p_top_logprob = view(b.pLogprob, (mp,), torch.float32), view(b.pTopLogprob, (mp,), torch.float32)
        kv = (w.n_kv_heads, self.seq_len, h.head_dim)
        self.k_cache = [view(b.kCache[l], kv, torch.bfloat16) for l in range(h.n_layers)]
        self.v_cache = [view(b.vCache[l], kv, torch.bfloat16) for l in range(h.n_layers)]
        self.comm = comm
        tp = comm is not None and comm.world_size > 1
        # Collectives: "fused" = inside the kernels over NVLink peer memory (ranks of one node, q40 weights);
        # "nccl" = library all-reduce between kernel groups (ranks on several nodes, dense weight files, DL_COLLECTIVES=nccl).
        self.collectives = "fused"
        if tp and (collectives == "nccl" or os.environ.get("DL_COLLECTIVES") == "nccl" or self.dense
                   or not getattr(comm, "single_node", True)):
            self.collectives = "nccl"
        if tp and self.collectives == "fused":
            comm.alloc_arena(self._lib.dl_engine_arena_bytes(C.byref(cfg)))
            cp = cl.CommPtrs(arena=_ptrs8(comm.arena_ptrs), mcArena=comm.mc_ptr or None)
            cl.check(self._lib.dl_engine_set_comm(self._h, C.byref(cp)), "engine_set_comm")
        self._parts = tp and self.collectives == "nccl"
        self._ybuf = torch.zeros(mb, h.dim, dtype=torch.float32, device=dev)
        self.use_tc_prefill = not self.dense and not self._parts
        self.mega = False
        if h.n_experts == 0 and not self.dense and not self._parts and os.environ.get("DL_NO_MEGA") is None:
            self.enable_mega(True)     # persistent decode kernel by default; the engine falls back per call if a shape is unsupported
        self.tc_min_tokens = 9          # shorter chunks stay on the GEMV path
        self._vocab_limit = 0
        self._graph_ready = False
        self._stage_tok = torch.zeros(mb, dtype=torch.int32).pin_memory()
        self._stage_pos = torch.zeros(mb, dtype=torch.int32).pin_memory()

    def set_vocab_limit(self, limit: int):
        """Greedy arg-max on the device never returns ids >= limit (the tokenizer's vocabulary size: embeddings may be padded
        beyond it, reference src/app.cpp:243-246 builds its sampler on the tokenizer size too)."""
        cl.check(self._lib.dl_engine_set_vocab_limit(self._h, int(limit)), "engine_set_vocab_limit")
        self._vocab_limit = int(limit)
        self._graph_ready = False

    # -- device-side sampling --
    def seed_sampler(self, seed: int):
        """Seeds the device-resident generator (same xorshift* stream as the host Sampler). Every rank must use the same seed."""
        cl.check(self._lib.dl_engine_sampler_seed(self._h, int(seed) & 0xFFFFFFFFFFFFFFFF), "engine_sampler_seed")
        self._sampler_ready = True

    def step_sampled(self, token: int, pos: int, temperature: float, topp: float) -> None:
        """Forward of one token + temperature/top-p sampling on the device (csrc/cuda/sampler.cu); the sampled token lands in
        tokens[0] and history[pos + 1]. No logits leave the GPU; under tensor parallelism the vocabulary slices are exchanged
        through peer memory and every rank draws the same token."""
        if not getattr(self, "_sampler_ready", False):
            raise RuntimeError("seed_sampler() must be called first")
        self.forward_batch([token], pos, logits_mode=1)
        cl.check(self._lib.dl_engine_sample(self._h, float(temperature), float(topp), cl.stream_ptr()), "engine_sample")

    # -- traffic / synchronisation accounting (reference: NnNetwork::getStats + executor sync timers, src/dllama.cpp:59-66) --
    def sync_ns(self) -> int:
        """Cumulative ns the decode kernel waited for peer ranks inside its fused all-reduces (0 on one GPU)."""
        return int(self._lib.dl_engine_sync_ns(self._h))

    def link_bytes(self, n_tokens: int) -> tuple:
        """(sent, received) NVLink bytes of this rank for a forward over n_tokens tokens: 2 all-reduces per layer, every value
        travels as an 8-byte LL word; with the NVSwitch multicast mapping a value is sent once and replicated by the switch."""
        n = self.comm.world_size if (self.comm is not None and not self._parts) else 1
        if n <= 1:
            return 0, 0
        h = self.w.header
        per_ar = n_tokens * h.dim * 8
        mc = 1 if getattr(self.comm, "mc_ptr", 0) and n_tokens == 1 else (n - 1)
        return 2 * h.n_layers * per_ar * mc, 2 * h.n_layers * per_ar * (n - 1)

    @property
    def mega_active(self) -> bool:
        """True if the last single-token forward actually ran on the persistent kernel (it falls back per call when the shape or
        the co-residency check rules it out)."""
        return bool(self._lib.dl_engine_mega_active(self._h))

    def check_abort(self):
        """Raises if a device-side wait loop ran out of its spin budget (a peer rank died or a CTA never became resident): the
        kernels drain instead of hanging and flag the step as invalid (csrc/cuda/mega_decode.cu: SpinGuard)."""
        if self._lib.dl_engine_aborted(self._h):
            raise RuntimeError("device-side wait timed out: a tensor-parallel peer stopped responding (or the persistent kernel was not co-resident)")

    def enable_mega(self, enable: bool = True):
        """Single-token forwards through the persistent per-token kernel (dense models). Re-captures the decode graph."""
        cl.check(self._lib.dl_engine_enable_mega(self._h, 1 if enable else 0), "engine_enable_mega")
        self.mega = enable
        self._graph_ready = False

    # -- tracing --
    def enable_trace(self, cap_launches: int = 1024, all_ctas: bool = False):
        """Device-side timeline: every kernel stamps globaltimer at entry / dependency resolved / prologue done / exit.
        Must be enabled before the decode graph is captured. `all_ctas`: every CTA of the persistent kernel records its own
        phase stamps (row c of `trace_buf.view(num_sms, -1)`), for barrier-skew analysis."""
        if all_ctas:
            cap_launches = max(cap_launches, self.num_sms * 256)
        self.trace_buf = torch.zeros(cap_launches, 4, dtype=torch.int64, device=self.device)
        cl.check(self._lib.dl_engine_set_trace(self._h, self.trace_buf.data_ptr(), cap_launches), "engine_set_trace")
        cl.check(self._lib.dl_engine_set_trace_all(self._h, 1 if all_ctas else 0), "engine_set_trace_all")
        self.trace_stride = (cap_launches * 4) // self.num_sms if all_ctas else 0
        self._graph_ready = False

    def read_trace(self):
        t = self.trace_buf.cpu().numpy()
        return t[t[:, 0] != 0]

    # -- low level --
    def _set_inputs(self, tokens: Sequence[int], start_pos: int):
        # Pageable source tensors: the copy is staged before the call returns, so back-to-back chunks cannot
        # overwrite a host buffer that an earlier async copy has not consumed yet.
        n = len(tokens)
        self.tokens[:n].copy_(torch.tensor(list(tokens), dtype=torch.int32))
        self.pos[:n].copy_(torch.arange(start_pos, start_pos + n, dtype=torch.int32))

    def forward_batch(self, tokens: Sequence[int], start_pos: int, logits_mode: int = 1, greedy_advance: bool = False):
        """Runs one forward over len(tokens) in {1,2,4,8} tokens at consecutive positions."""
        n = len(tokens)
        if start_pos + n > self.seq_len:
            raise ValueError("position beyond the context length")
        self._set_inputs(tokens, start_pos)
        self._forward(n, logits_mode, greedy_advance)

    def _forward(self, n: int, logits_mode: int, greedy_advance: bool = False):
        if self._parts:
            self._forward_parts(n, logits_mode, greedy_advance)
        else:
            cl.check(self._lib.dl_engine_forward(self._h, n, logits_mode, 1 if greedy_advance else 0, cl.stream_ptr()), "engine_forward")

    def prefill(self, tokens: Sequence[int], start_pos: int = 0, want_logits: bool = True) -> Optional[torch.Tensor]:
        """Feeds a prompt; returns the logits row of its last token (device tensor). Single GPU: chunks of up to 256 tokens
        on the tcgen05 GEMM path. Tensor parallel: chunks of up to max_batch tokens on the GEMV path (fused all-reduce)."""
        tokens = list(tokens)
        if start_pos + len(tokens) > self.seq_len:
            raise ValueError("position beyond the context length")
        tc_path = self._tc_prefill_ok()
        i = 0
        while i < len(tokens):
            rem = len(tokens) - i
            if tc_path and rem >= self.tc_min_tokens:
                n = min(rem, self.max_prefill)
                last = i + n == len(tokens)
                self.p_tokens[:n].copy_(torch.tensor(tokens[i:i + n], dtype=torch.int32))
                self.p_pos[:n].copy_(torch.arange(start_pos + i, start_pos + i + n, dtype=torch.int32))
                cl.check(self._lib.dl_engine_prefill(self._h, n, start_pos + i, 1 if (last and want_logits) else 0, cl.stream_ptr()), "engine_prefill")
            else:
                n = 1
                while n * 2 <= min(rem, self.max_batch):
                    n *= 2
                last = i + n == len(tokens)
                self.forward_batch(tokens[i:i + n], start_pos + i, logits_mode=1 if (last and want_logits) else 0)
            i += n
        return self._full_logits(self.logits[0]) if want_logits else None

    def _tc_prefill_ok(self) -> bool:
        """Whether prompt chunks can take the tensor-core path (dl_engine_prefill / dl_engine_score) on this configuration."""
        hdr = self.w.header
        tp = self.comm is not None and self.comm.world_size > 1
        # tensor parallel: the fused GEMM + all-reduce kernel needs 256-wide K slices on every rank
        tp_ok = (not tp) or ((self.w.n_heads * hdr.head_dim) % 256 == 0 and self.w.ff_dim % 256 == 0 and hdr.dim % 256 == 0)
        # mixture of experts: the grouped tensor-core GEMMs need 256-wide K on both expert matrices
        moe_ok = hdr.n_experts == 0 or (hdr.dim % 256 == 0 and self.w.ff_dim % 256 == 0 and os.environ.get("DL_NO_MOE_PREFILL") is None)
        return tp_ok and moe_ok and self.use_tc_prefill

    @property
    def score_max_tokens(self) -> int:
        """Tokens per dl_engine_score call (prefill chunk limit; under tensor parallelism also the record-exchange capacity)."""
        return int(self._lib.dl_engine_score_max_tokens(self._h))

    def score(self, tokens: Sequence[int], start_pos: int = 0, next_token: Optional[int] = None) -> ScoreResult:
        """Evaluates tokens at positions start_pos.. (writing the same KV rows as `prefill`) and scores every next token on the
        device: see ScoreResult. `next_token`, the token that follows `tokens`, adds its log-probability as a last entry.
        Tensor-core path: chunks of `score_max_tokens`, logits of all tokens by one GEMM, log-softmax by csrc/cuda/score.cu; the
        target of a chunk's last row is the first token of the next chunk. Where that path does not run (dense weight files, the
        library-collective mode, shapes the tensor-core prefill does not cover) the logits come from the GEMV batches and are
        normalised with torch.log_softmax on the device. Under tensor parallelism every rank must make the same call."""
        tokens = [int(t) for t in tokens]
        n = len(tokens)
        if n == 0:
            raise ValueError("nothing to score")
        if start_pos + n > self.seq_len:
            raise ValueError("position beyond the context length")
        targets = tokens[1:] + [-1 if next_token is None else int(next_token)]
        lp, ids, top = [], [], []
        if self._tc_prefill_ok():
            cap = self.score_max_tokens
            for i in range(0, n, cap):
                m = min(cap, n - i)
                self.p_tokens[:m].copy_(torch.tensor(tokens[i:i + m], dtype=torch.int32))
                self.p_pos[:m].copy_(torch.arange(start_pos + i, start_pos + i + m, dtype=torch.int32))
                self.p_targets[:m].copy_(torch.tensor(targets[i:i + m], dtype=torch.int32))
                cl.check(self._lib.dl_engine_score(self._h, m, start_pos + i, cl.stream_ptr()), "engine_score")
                lp.append(self.p_logprob[:m].clone()); ids.append(self.p_top_id[:m].clone()); top.append(self.p_top_logprob[:m].clone())
        else:
            limit = self._vocab_limit
            i = 0
            while i < n:
                nb = 1
                while nb * 2 <= min(n - i, self.max_batch):
                    nb *= 2
                lsm = torch.log_softmax(self.logits_all(tokens[i:i + nb], start_pos + i).float(), dim=-1)
                tv = lsm[:, :limit] if 0 < limit < lsm.shape[1] else lsm
                best = tv.argmax(dim=-1)                       # first maximal index: the lowest id wins ties
                tg = torch.tensor(targets[i:i + nb], dtype=torch.int64, device=lsm.device)
                got = lsm.gather(1, tg.clamp(min=0)[:, None])[:, 0]
                lp.append(torch.where(tg >= 0, got, torch.full_like(got, float("nan"))))
                ids.append(best.to(torch.int32)); top.append(lsm.gather(1, best[:, None])[:, 0])
                i += nb
        n_lp = n if next_token is not None else n - 1
        return ScoreResult(torch.cat(lp)[:n_lp].cpu(), torch.cat(ids).cpu(), torch.cat(top).cpu())

    def step(self, token: int, pos: int) -> torch.Tensor:
        """Forward of one token; returns the full-vocabulary logits row (gathered over ranks under tensor parallelism)."""
        self.forward_batch([token], pos, logits_mode=1)
        return self._full_logits(self.logits[0])

    def _full_logits(self, local: torch.Tensor) -> torch.Tensor:
        if self.comm is None or self.comm.world_size == 1:
            return local
        return self.comm.all_gather_cat(local, dim=-1)

    def logits_all(self, tokens: Sequence[int], start_pos: int) -> torch.Tensor:
        """Logits for every token of a (<= max_batch, power of two) batch — used by perplexity and tests."""
        self.forward_batch(tokens, start_pos, logits_mode=2)
        return self._full_logits(self.logits[: len(tokens)])

    # -- library-collective path (tensor parallel): same kernels, all-reduce through torch.distributed between kernel groups --
    def _forward_parts(self, nb: int, logits_mode: int = 1, greedy_advance: bool = False) -> None:
        """One forward over the tokens staged in self.tokens/self.pos with per-layer NCCL all-reduces (the reference's K2/K3
        sync sites as library collectives, src/llm.cpp:397-403,548-554). Runs when the ranks do not share a peer-memory
        domain, for dense weight files, and as the baseline the fused kernels are measured against. Graph capturable."""
        import torch.distributed as dist
        y, sp, lib, h = self._ybuf, cl.stream_ptr(), self._lib, self._h
        tp = self.comm is not None and self.comm.world_size > 1
        cl.check(lib.dl_engine_forward_part(h, nb, 0, 0, y.data_ptr(), sp), "forward_part")
        for l in range(self.w.header.n_layers):
            for part in (1, 2):
                cl.check(lib.dl_engine_forward_part(h, nb, l, part, y.data_ptr(), sp), "forward_part")
                if tp:
                    dist.all_reduce(y[:nb])
                self.x[:nb].add_(y[:nb])
        if logits_mode:
            cl.check(lib.dl_engine_forward_part(h, nb, 0, 3 if logits_mode == 1 else 4, y.data_ptr(), sp), "forward_part")
        if greedy_advance:
            tok = self._full_logits(self.logits[0]).argmax().to(torch.int32).reshape(1)
            self.tokens[:1].copy_(tok)
            self.pos[:1].add_(1)
            self.history.index_copy_(0, self.pos[:1].long().clamp_(max=self.history.numel() - 1), tok)

    def forward_nccl_baseline(self, token_count: int = 1) -> torch.Tensor:
        """Library-collective forward of the staged tokens; returns the local logits slice (tools/bench_nccl_baseline.py)."""
        self._forward_parts(token_count, 1, False)
        return self.logits[0]

    # -- device-resident greedy decoding --
    def run_decode_step(self, use_graph: bool = True):
        """One greedy step on whatever (token, pos) currently sit in device memory; result lands in tokens[0]."""
        if self._parts:
            self._forward_parts(1, 1, True)
            return
        if use_graph:
            if not self._graph_ready:
                saved = (self.tokens.clone(), self.pos.clone())
                cl.check(self._lib.dl_engine_forward(self._h, 1, 1, 0, cl.stream_ptr()), "engine_forward")
                torch.cuda.current_stream().synchronize()
                self.capture_decode()
                self.tokens.copy_(saved[0]); self.pos.copy_(saved[1])
            cl.check(self._lib.dl_engine_decode_graph(self._h, 1, cl.stream_ptr()), "engine_decode_graph")
        else:
            cl.check(self._lib.dl_engine_forward(self._h, 1, 1, 1, cl.stream_ptr()), "engine_forward")

    @property
    def launches_per_decode_step(self) -> int:
        if self.mega and self.mega_active:
            return 1                # one persistent kernel per token (plus a 4-byte memset node)
        if self._parts:
            return self.w.header.n_layers * 7 + 2
        if self.w.header.n_experts > 0:
            return self.w.header.n_layers * 6 + 2
        return self.w.header.n_layers * 5 + 2   # embedding + 5 fused kernels per layer + logits/arg-max

    def capture_decode(self):
        cl.check(self._lib.dl_engine_capture_decode(self._h), "engine_capture_decode")
        self._graph_ready = True

    def decode_greedy(self, first_token: int, start_pos: int, n_steps: int, use_graph: bool = True) -> List[int]:
        """Generates n_steps tokens greedily: step i consumes the token at position start_pos+i and emits the next.
        The loop runs entirely on the device (token + position live in device memory)."""
        if start_pos + n_steps > self.seq_len:
            raise ValueError("decode would run past the context length")
        self._set_inputs([first_token], start_pos)
        if self._parts:
            for _ in range(n_steps):
                self._forward_parts(1, 1, True)
        elif use_graph:
            if not self._graph_ready:
                # warm-up run configures kernel attributes outside of capture
                cl.check(self._lib.dl_engine_forward(self._h, 1, 1, 0, cl.stream_ptr()), "engine_forward")
                torch.cuda.current_stream().synchronize()
                self.capture_decode()
            cl.check(self._lib.dl_engine_decode_graph(self._h, n_steps, cl.stream_ptr()), "engine_decode_graph")
        else:
            for _ in range(n_steps):
                cl.check(self._lib.dl_engine_forward(self._h, 1, 1, 1, cl.stream_ptr()), "engine_forward")
        out = self.history[start_pos + 1: start_pos + 1 + n_steps].cpu()
        self.check_abort()
        return out.tolist()
