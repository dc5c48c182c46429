"""Root/worker application runtime (reference: runInferenceApp / runWorkerApp, src/app.cpp:232-365).

Process model on the B200 box: one process per GPU. Rank 0 is the *root* (tokenizer, sampler, user I/O), ranks >= 1 are
*workers*: they hold their tensor-parallel weight slices and mirror every forward the root issues. Control flows as the
reference's 8-byte LlmControlPacket {position, batchSize} (src/app.hpp:46-49) — here extended with an opcode and passed through a
shared-memory channel with heartbeats (parallel/control.py; torch.distributed broadcasts only when the ranks span hosts);
op 0 is the stop signal. All activation traffic happens inside the kernels over NVLink.
"""
from __future__ import annotations

import os
import sys
from dataclasses import dataclass
from typing import Callable, List, Optional, Sequence

import numpy as np
import torch

from .. import host
from ..api import InferenceSession
from .args import AppArgs

OP_STOP, OP_PREFILL, OP_STEP_LOGITS, OP_STEP_GREEDY, OP_DECODE_N, OP_STEP_SAMPLE, OP_SEED, OP_SCORE = 0, 1, 2, 3, 4, 5, 6, 7


def world():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def init_distributed_from_env():
    """Initialises torch.distributed when launched by torchrun (RANK/WORLD_SIZE set). Returns (comm or None)."""
    ws = int(os.environ.get("WORLD_SIZE", "1"))
    if ws <= 1:
        if torch.cuda.is_available():
            torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
        return None
    import torch.distributed as dist
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    from ..parallel.comm import Communicator
    return Communicator()


def open_control_channel(comm):
    """Creates (rank 0) / attaches to (workers) the shared-memory control channel of the job. DL_CONTROL=nccl keeps the
    torch.distributed broadcasts (needed when the ranks do not share a host)."""
    if comm is None or os.environ.get("DL_CONTROL") == "nccl" or not getattr(comm, "single_node", True):
        return None
    import torch.distributed as dist
    from ..parallel.control import ControlChannel
    name = [None]
    chan = None
    if comm.rank == 0:
        chan = ControlChannel(0, comm.world_size)
        name[0] = chan.name
    dist.broadcast_object_list(name, src=0)
    if comm.rank != 0:
        chan = ControlChannel(comm.rank, comm.world_size, name=name[0])
    chan.start_heartbeat()
    dist.barrier()
    return chan


class RootInference:
    """Root-side handle (reference RootLlmInference, src/app.cpp:168-208): every call first tells the workers what to run.
    The packet travels through shared memory (parallel/control.py); the activations never leave the GPUs."""

    def __init__(self, sess: InferenceSession, comm, chan=None):
        self.sess = sess
        self.comm = comm
        self.chan = chan
        self.eng = sess.engine
        self.header = sess.header
        self.eval_ms = 0.0
        self._ctl = torch.zeros(4, dtype=torch.int64, device=sess.device) if (comm is not None and chan is None) else None
        on_gpu = sess.device.type == "cuda"
        self._pin_out = torch.zeros(1, dtype=torch.int32).pin_memory() if on_gpu else None
        self._pin_in = torch.zeros(2, dtype=torch.int32).pin_memory() if on_gpu else None

    def _send(self, op: int, pos: int, tokens: Sequence[int]):
        if self.comm is None:
            return
        if self.chan is not None:
            self.chan.send(op, pos, tokens)
            return
        import torch.distributed as dist
        n = len(tokens)
        self._ctl[0], self._ctl[1], self._ctl[2] = op, pos, n
        dist.broadcast(self._ctl, 0)
        if n:
            t = torch.tensor(list(tokens), dtype=torch.int64, device=self.sess.device)
            dist.broadcast(t, 0)

    def prefill(self, tokens: Sequence[int], pos: int) -> None:
        if tokens:
            self._send(OP_PREFILL, pos, tokens)
            self.eng.prefill(tokens, pos, want_logits=False)

    def score(self, tokens: Sequence[int], pos: int, next_token: Optional[int] = None):
        """Scores tokens at positions pos.. (Engine.score). One OP_SCORE packet per piece that fits a control packet: the piece,
        then the token that follows it (-1: none), so the pieces' scores join up exactly."""
        from ..parallel.control import MAX_TOKENS
        from ..runtime.engine import ScoreResult
        tokens = list(tokens)
        step = MAX_TOKENS - 1
        parts = []
        for i in range(0, len(tokens), step):
            piece = tokens[i:i + step]
            nxt = tokens[i + step] if i + step < len(tokens) else next_token
            self._send(OP_SCORE, pos + i, piece + [-1 if nxt is None else nxt])
            parts.append(self.eng.score(piece, pos + i, next_token=nxt))
        return ScoreResult.cat(parts)

    def forward_logits(self, token: int, pos: int) -> torch.Tensor:
        self._send(OP_STEP_LOGITS, pos, [token])
        return self.eng.step(token, pos)

    def forward_greedy(self, token: int, pos: int) -> int:
        self._send(OP_STEP_GREEDY, pos, [token])
        if self._pin_in is None:          # session on the CPU (protocol tests)
            self.eng._set_inputs([token], pos)
            self.eng.run_decode_step()
            return int(self.eng.tokens[0])
        # the root synchronises every step, so one pinned staging slot is enough (workers enqueue ahead: pageable staging)
        self._pin_in[0], self._pin_in[1] = token, pos
        self.eng.tokens[:1].copy_(self._pin_in[:1], non_blocking=True)
        self.eng.pos[:1].copy_(self._pin_in[1:2], non_blocking=True)
        self.eng.run_decode_step()
        self._pin_out.copy_(self.eng.tokens[:1], non_blocking=True)
        torch.cuda.current_stream().synchronize()
        self.eng.check_abort()
        return int(self._pin_out[0])

    # ---- sampling on the device: the logits never leave the GPUs (csrc/cuda/sampler.cu) ----
    @property
    def device_sampling(self) -> bool:
        return torch.cuda.is_available() and not getattr(self.eng, "_parts", False) and os.environ.get("DL_HOST_SAMPLER") is None

    def seed(self, seed: int) -> None:
        self._send(OP_SEED, 0, [seed & 0x7FFFFFFF, (seed >> 31) & 0x7FFFFFFF, (seed >> 62) & 0x3])
        self.eng.seed_sampler(seed)

    def forward_sampled(self, token: int, pos: int, temperature: float, topp: float) -> int:
        import struct
        t_bits, p_bits = struct.unpack("<ii", struct.pack("<ff", temperature, topp))
        self._send(OP_STEP_SAMPLE, pos, [token, t_bits, p_bits])
        self.eng.step_sampled(token, pos, temperature, topp)
        self._pin_out.copy_(self.eng.tokens[:1], non_blocking=True)
        torch.cuda.current_stream().synchronize()
        self.eng.check_abort()
        return int(self._pin_out[0])

    def next_token(self, token: int, pos: int, sampler) -> int:
        """One generated token with the sampler's settings: greedy and temperature/top-p both run on the device; the host sampler
        is only used with the library-collective (multi-node) mode or DL_HOST_SAMPLER=1."""
        if sampler.temperature == 0.0:
            return self.forward_greedy(token, pos)
        if self.device_sampling:
            if getattr(self, "_seeded", None) != (sampler.seed, sampler.seed_generation):
                self.seed(sampler.seed)
                self._seeded = (sampler.seed, sampler.seed_generation)
            return self.forward_sampled(token, pos, sampler.temperature, sampler.topp)
        return int(sampler.sample(self.forward_logits(token, pos).float().cpu().numpy()))

    def decode_greedy(self, token: int, pos: int, n_steps: int) -> List[int]:
        """n greedy steps with the token fed back on the device (no host round trip per step): one control packet for all."""
        self._send(OP_DECODE_N, pos, [token, n_steps])
        return self.eng.decode_greedy(token, pos, n_steps)

    def finish(self):
        try:
            self._send(OP_STOP, 0, [])
        finally:
            if self.chan is not None:
                self.chan.close()


def worker_loop(sess: InferenceSession, comm, chan=None) -> None:
    """Worker main loop (reference runWorkerApp, src/app.cpp:306-365): mirror the root's forwards until the stop packet."""
    import torch.distributed as dist
    ctl = torch.zeros(4, dtype=torch.int64, device=sess.device) if chan is None else None
    eng = sess.engine
    while True:
        if chan is not None:
            op, pos, toks = chan.recv()
        else:
            dist.broadcast(ctl, 0)
            op, pos, n = int(ctl[0]), int(ctl[1]), int(ctl[2])
            toks = []
            if op != OP_STOP and n:
                t = torch.zeros(n, dtype=torch.int64, device=sess.device)
                dist.broadcast(t, 0)
                toks = t.tolist()
        if op == OP_STOP:
            print("🛑 Stop signal")
            if chan is not None:
                chan.close()
            return
        if op == OP_PREFILL:
            eng.prefill(toks, pos, want_logits=False)
        elif op == OP_STEP_LOGITS:
            eng.step(toks[0], pos)
        elif op == OP_STEP_GREEDY:
            eng._set_inputs(toks, pos)
            eng.run_decode_step()
        elif op == OP_DECODE_N:
            eng.decode_greedy(toks[0], pos, toks[1])
        elif op == OP_SCORE:
            eng.score(toks[:-1], pos, next_token=None if toks[-1] < 0 else toks[-1])
        elif op == OP_SEED:
            eng.seed_sampler(toks[0] | (toks[1] << 31) | (toks[2] << 62))
        elif op == OP_STEP_SAMPLE:
            import struct
            temperature, topp = struct.unpack("<ff", struct.pack("<ii", toks[1], toks[2]))
            eng.step_sampled(toks[0], pos, temperature, topp)


@dataclass
class AppContext:
    args: AppArgs
    sess: InferenceSession
    inference: RootInference
    tokenizer: object
    sampler: object
    header: object


def run_inference_app(args: AppArgs, handler: Callable[[AppContext], None]) -> None:
    if args.model is None:
        raise RuntimeError("Model is required")
    if args.tokenizer is None:
        raise RuntimeError("Tokenizer is required")
    comm = init_distributed_from_env()
    rank = comm.rank if comm else 0
    H = host()
    header = H.load_model_header(args.model, args.max_seq_len)
    n_nodes = comm.world_size if comm else 1
    if header.weight_type == H.F_Q40 and args.buffer_float_type != "q80":
        raise RuntimeError("This version supports only Q40 weights with Q80 sync type")
    sess = InferenceSession(args.model, args.tokenizer, max_seq_len=args.max_seq_len, temperature=args.temperature,
                            topp=args.topp, seed=args.seed, comm=comm, moe_mode=getattr(args, "moe_mode", "auto") or "auto")
    chan = open_control_channel(comm)
    if rank != 0:
        worker_loop(sess, comm, chan)
        return
    tok = sess.tokenizer
    if args.info:
        if tok.vocab_size != header.vocab_size:
            print(f"Tokenizer vocab size ({tok.vocab_size}) does not match the model vocab size ({header.vocab_size})")
        print(tok.describe(), end="")
        print(header.describe(), end="")
        req = H.required_device_bytes(header, n_nodes, 2)
        print(f"📀 RequiredMemory: {req // (1024 * 1024)} MB")
        name = torch.cuda.get_device_name(sess.device)
        print(f"🧠 GPU: {name} x{n_nodes} (sm_100a kernels; tensor parallel over NVLink peer memory)")
        print("💿 Weights loaded")
    inf = RootInference(sess, comm, chan)
    ctx = AppContext(args=args, sess=sess, inference=inf, tokenizer=tok, sampler=sess.sampler, header=header)
    try:
        handler(ctx)
    finally:
        inf.finish()
