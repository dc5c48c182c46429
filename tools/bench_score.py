"""Prompt-scoring throughput (Engine.score, dl_engine_score) on one of the large configurations with random-init device weights
(models/loader.py synthetic_device_weights): scored tokens/s over a synthetic text, the device time of each stage of one chunk
(prefill chain, final norm + logits GEMM, score kernel; CUDA events), the score kernel's bytes over its time against the 7.7 TB/s
HBM3e figure of the B200 data sheet, and the token-by-token `forward_logits` + host softmax loop that scoring replaces. Prints one
JSON line. Run under torchrun for N > 1 (the per-stage kernel timings are taken at N = 1 only).

    python tools/bench_score.py [llama-3.1-8b] [--tokens 4096] [--loop-tokens 256]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

from distributed_llama_b200.models.config import get_config
from distributed_llama_b200.models.loader import synthetic_device_weights
from distributed_llama_b200.ops import cuda_lib as cl
from distributed_llama_b200.runtime import Engine

HBM_BYTES_PER_S = 7.7e12

ap = argparse.ArgumentParser()
ap.add_argument("model", nargs="?", default="llama-3.1-8b")
ap.add_argument("--tokens", type=int, default=4096, help="length of the scored text")
ap.add_argument("--loop-tokens", type=int, default=256, help="tokens of the text fed to the token-by-token comparison loop")
ap.add_argument("--reps", type=int, default=20, help="timed repetitions of each per-chunk stage")
args = ap.parse_args()
world, rank, local = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
torch.cuda.set_device(local)
comm = None
if world > 1:
    from distributed_llama_b200.parallel.comm import Communicator
    dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    comm = Communicator()
cfg = get_config(args.model)
W = synthetic_device_weights(cfg, rank, world, f"cuda:{local}", max_seq_len=args.tokens)
eng = Engine(W, comm=comm)
hdr, lib, h = W.header, eng._lib, eng._h
text = [(7919 * i + 13) % (hdr.vocab_size - 1) + 1 for i in range(args.tokens)]


def sync():
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def gpu_info():
    name = torch.cuda.get_device_name(local)
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


def events_ms(fn, reps):
    """Mean device time of fn() over reps launches (after one warm-up), CUDA events around the whole window."""
    fn()
    sync()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        fn()
    e.record()
    sync()
    return s.elapsed_time(e) / reps


# 1. whole text through Engine.score (warm-up on the same text: the first call allocates the logits scratch)
eng.score(text, 0)
sync()
t0 = time.perf_counter()
res = eng.score(text, 0)
sync()
score_s = time.perf_counter() - t0

# 2. one chunk, stage by stage (single rank: the stages are called directly with the engine's weights)
T = eng.score_max_tokens
stages = {}
if world == 1:
    sp = cl.stream_ptr()
    vocab, dim = W.vocab, hdr.dim
    eng.p_tokens[:T].copy_(torch.tensor(text[:T], dtype=torch.int32))
    eng.p_targets[:T].copy_(torch.tensor(text[1:T + 1], dtype=torch.int32))
    xs = torch.randn(T, dim, device="cuda")
    xn = torch.empty(T, dim, dtype=torch.bfloat16, device="cuda")
    lg = torch.empty(T, vocab, device="cuda")
    tg = torch.tensor(text[1:T + 1], dtype=torch.int32, device="cuda")
    out_f, out_i, out_t = torch.empty(T, device="cuda"), torch.empty(T, dtype=torch.int32, device="cuda"), torch.empty(T, device="cuda")
    for p0 in (0, args.tokens - T):
        eng.p_pos[:T].copy_(torch.arange(p0, p0 + T, dtype=torch.int32))

        def logits_gemm():
            cl.check(lib.dl_rmsnorm_bf16(xs.data_ptr(), dim, W.final_norm.data_ptr(), xn.data_ptr(), dim, dim, hdr.norm_epsilon, T, sp), "rmsnorm")
            cl.check(lib.dl_gemm_q40_tc(cl.GEPI_STORE_F32, W.wcls.qs.data_ptr(), W.wcls.scales.data_ptr(), vocab, dim, xn.data_ptr(), dim, T,
                                        lg.data_ptr(), vocab, eng.num_sms, sp, 0, 0), "logits gemm")

        def gemm_then_score():
            logits_gemm()
            cl.check(lib.dl_score_rows(lg.data_ptr(), T, vocab, vocab, tg.data_ptr(), 0, out_f.data_ptr(), out_i.data_ptr(), out_t.data_ptr(), sp),
                     "score rows")

        prefill_ms = events_ms(lambda: cl.check(lib.dl_engine_prefill(h, T, p0, 0, sp), "prefill"), args.reps)
        gemm_ms = events_ms(logits_gemm, args.reps)
        # the score kernel as it runs in dl_engine_score: right after the GEMM that wrote its input (partly still in L2)
        score_kernel_ms = events_ms(gemm_then_score, args.reps) - gemm_ms
        full_ms = events_ms(lambda: cl.check(lib.dl_engine_score(h, T, p0, sp), "engine score"), args.reps)
        rows_bytes = T * vocab * 4 + T * 16
        stages[f"p0={p0}"] = {"prefill_chain_ms": round(prefill_ms, 4), "norm_logits_gemm_ms": round(gemm_ms, 4),
                              "score_kernel_ms": round(score_kernel_ms, 4), "dl_engine_score_ms": round(full_ms, 4),
                              "score_kernel_GBps": round(rows_bytes / (score_kernel_ms * 1e-3) / 1e9, 1),
                              "score_kernel_share_of_hbm_peak": round(rows_bytes / (score_kernel_ms * 1e-3) / HBM_BYTES_PER_S, 3)}
    # the score kernel alone, input evicted from L2 between launches by a 256 MB write
    flush = torch.empty(64 << 20, device="cuda")

    def cold_score():
        flush.zero_()
        cl.check(lib.dl_score_rows(lg.data_ptr(), T, vocab, vocab, tg.data_ptr(), 0, out_f.data_ptr(), out_i.data_ptr(), out_t.data_ptr(), sp),
                 "score rows")
    cold_ms = events_ms(cold_score, args.reps) - events_ms(lambda: flush.zero_(), args.reps)
    stages["score_kernel_cold_l2_ms"] = round(cold_ms, 4)
    stages["score_kernel_cold_l2_GBps"] = round((T * vocab * 4 + T * 16) / (cold_ms * 1e-3) / 1e9, 1)

# 3. the token-by-token loop it replaces: one decode forward, a full logits row to the host and a host softmax per token
n_loop = min(args.loop_tokens, args.tokens - 1)
eng2 = Engine(W, comm=comm)
eng2.step(text[0], 0)
sync()
t0 = time.perf_counter()
loop_lp = []
for i in range(n_loop):
    row = eng2.step(text[i], i).float().cpu().numpy().astype(np.float64)
    m = row.max()
    loop_lp.append(row[text[i + 1]] - m - np.log(np.exp(row - m).sum()))
sync()
loop_s = time.perf_counter() - t0
agree = float(np.abs(np.array(loop_lp) - res.logprobs[:n_loop].double().numpy()).max())

if rank == 0:
    name, power = gpu_info()
    print(json.dumps({
        "model": args.model, "gpus": world, "gpu": name, "power_limit_and_max_sm_clock": power, "tokens": args.tokens, "chunk_tokens": T,
        "score_tokens_per_s": round(args.tokens / score_s, 1), "score_s": round(score_s, 4),
        "token_loop_tokens": n_loop, "token_loop_tokens_per_s": round(n_loop / loop_s, 1),
        "max_abs_logprob_diff_score_vs_loop": round(agree, 4), "chunk_stages": stages}))
if world > 1:
    dist.barrier()
    dist.destroy_process_group()
