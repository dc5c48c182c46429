#!/usr/bin/env python
"""Headline benchmark: batch-1 decode tokens/s (+ prefill TTFT) of Llama-3.1-8B q40, tensor-parallel over N B200s.

    python bench.py --gpus 1 --steps 64 --warmup 8
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 4 --master-addr 127.0.0.1 --master-port 29501 \
        bench.py --gpus 4 --steps 64 --warmup 8
    python bench.py --impl reference --gpus 1 --steps 32 --warmup 3     # unmodified reference (CPU build, TCP loopback)

Metric definition follows the reference's own benchmark mode (`dllama inference`, src/dllama.cpp:76-115): one "step"
is one generated token of a single sequence (forward of 1 token through all layers + sampling); `value` is the
whole-job tokens/s. The model is random-init in the real `.m` layout (no network for checkpoints); weights (4.5 GB) are
far larger than L2 (126 MB) so every step streams them from HBM — no L2 flush is needed between steps.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import re
import shutil
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# Published numbers of the reference (report/report.pdf, Llama 2 7B q40 on Raspberry Pi 4B, ms per token by device count).
PUBLISHED_MS_PER_TOKEN = {1: 1312.50, 2: 793.69, 4: 494.00, 8: 588.19}

CACHE_DIR = os.environ.get("DLLAMA_BENCH_DIR", "/tmp/dllama_bench")


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def ensure_model(name: str, max_seq_len_hint: int = 0):
    """Synthetic model + tokenizer in the real file formats (cached per box)."""
    from distributed_llama_b200.models.config import get_config
    from distributed_llama_b200.models.synthetic import write_synthetic_model, write_synthetic_tokenizer

    os.makedirs(CACHE_DIR, exist_ok=True)
    cfg = get_config(name)
    m = os.path.join(CACHE_DIR, f"dllama_model_{name}_q40.m")
    t = os.path.join(CACHE_DIR, f"dllama_tokenizer_{name}.t")
    if not os.path.exists(m):
        t0 = time.time()
        size = write_synthetic_model(m, cfg, seed=20240607)
        log(f"[bench] wrote {m} ({size / 1e9:.2f} GB) in {time.time() - t0:.1f}s")
    if not os.path.exists(t):
        write_synthetic_tokenizer(t, cfg.vocab_size, style="chatml" if name.startswith("qwen") else "llama3")
    return m, t


class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int = 0):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        exe = shutil.which("nvidia-smi")
        if not exe:
            return
        try:
            self.proc = subprocess.Popen([exe, f"--id={self.gpu}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        clocks, max_clock, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                clocks.append(float(parts[0]))
                max_clock = max(max_clock, float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        clocks.sort()
        # "under load" = upper half of the samples (the sampler also sees idle gaps before/after)
        load = clocks[len(clocks) // 2:] if clocks else []
        med = load[len(load) // 2] if load else None
        return {"sm_mhz": med, "sm_max_mhz": max_clock or None, "reasons": sorted(reasons), "samples": len(clocks)}


# ------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    os.environ["NCCL_DEBUG"] = "WARN"   # keep stdout to the single JSON line (NCCL prints its version banner on stdout)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("for --gpus N>1 launch with torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local_rank)
    comm = None
    if world > 1:
        from distributed_llama_b200.parallel.comm import Communicator
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
        comm = Communicator()

    if rank == 0:
        model_path, tok_path = ensure_model(args.model)
    if world > 1:
        dist.barrier()
    model_path, tok_path = ensure_model(args.model)

    from distributed_llama_b200.api import InferenceSession

    t0 = time.time()
    sess = InferenceSession(model_path, tok_path, max_seq_len=args.max_seq_len, temperature=0.0, comm=comm)
    eng = sess.engine
    if args.decode_path == "multi":
        eng.enable_mega(False)
    load_s = time.time() - t0
    log(f"[bench] rank {rank}: weights on device in {time.time() - t0:.1f}s ({sess.weights.bytes_uploaded / 1e9:.2f} GB uploaded)")

    steps, warmup = args.steps, max(args.warmup, 3)
    prompt = [(7 * i + 3) % 1000 + 1 for i in range(args.prompt_len)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- prefill (TTFT): prompt evaluated + first token sampled ----
    ttft = []
    for it in range(3):
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        eng.prefill(prompt[:-1], 0, want_logits=False)
        eng.decode_greedy(prompt[-1], len(prompt) - 1, 1)
        e.record()
        torch.cuda.synchronize()
        ttft.append(max_over_ranks(s.elapsed_time(e)))
    ttft_ms = min(ttft[1:])

    # ---- decode: device-timed, graph-replayed steps, no host involvement inside the region ----
    pos0 = len(prompt) - 1
    eng.decode_greedy(prompt[-1], pos0, warmup)            # warm-up (also captures the graph)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    barrier()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    toks = eng.decode_greedy(prompt[-1], pos0, steps)
    e.record()
    barrier()
    dev_ms = max_over_ranks(s.elapsed_time(e))
    if args.dump_outputs:
        # what the timed decode hands its caller (the greedy tokens) and the full-vocabulary logits row of its last step, read
        # before the decodes below overwrite the logits buffer
        logits = eng.logits[0] if world == 1 else comm.all_gather_cat(eng.logits[0], dim=-1)
        if rank == 0:
            import numpy as np
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "tokens.npy"), np.asarray(toks, dtype=np.float64))
            np.save(os.path.join(args.dump_outputs, "logits.npy"), logits.float().cpu().numpy())
    # long-context decode: the same step at position 2048 (the KV rows below it hold whatever the cache was initialised with —
    # only the attention cost over 2048 positions is of interest)
    extra = {}
    if args.max_seq_len >= 2048 + 40:
        eng.decode_greedy(prompt[-1], 2048, 4)
        barrier()
        s2, e2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s2.record()
        eng.decode_greedy(prompt[-1], 2048, 32)
        e2.record()
        barrier()
        extra["decode_at_pos2048_tok_s"] = round(32.0 / max_over_ranks(s2.elapsed_time(e2)) * 1e3, 1)
    # ---- end-to-end through the public API: per step H2D(token,pos) from pinned memory + D2H(token) ----
    # 1 GPU: InferenceSession.next_token. N GPUs: the product path of `dllama inference --gpus N` — the root sends one control packet
    # per token through the shared-memory channel (apps/runtime.py RootInference.forward_greedy), the workers mirror it in
    # worker_loop; the root copies the sampled token back to pinned host memory every step.
    from distributed_llama_b200.apps.runtime import RootInference, open_control_channel, worker_loop
    chan = open_control_channel(comm) if world > 1 else None
    e2e_tokens, e2e_ms = [], 0.0
    if world > 1 and rank != 0:
        worker_loop(sess, comm, chan)
    else:
        inf = RootInference(sess, comm, chan) if world > 1 else None

        def one(tok_, pos_):
            if inf is not None:
                return inf.forward_greedy(tok_, pos_)
            sess.pos = pos_
            return sess.next_token(tok_)
        tok, pos = prompt[-1], pos0
        for _ in range(warmup):
            tok = one(tok, pos); pos += 1
        tok, pos = prompt[-1], pos0
        torch.cuda.synchronize()
        t_start = time.perf_counter()
        for _ in range(steps):
            tok = one(tok, pos); pos += 1
            e2e_tokens.append(tok)
        torch.cuda.synchronize()
        e2e_ms = (time.perf_counter() - t_start) * 1e3      # root wall clock: every step ends with the token in host memory
        if inf is not None:
            inf.finish()
    barrier()
    clocks = sampler.stop() if rank == 0 else None

    if rank == 0:
        ms_per_step = dev_ms / steps
        value = 1000.0 / ms_per_step
        base = 1000.0 / PUBLISHED_MS_PER_TOKEN.get(args.gpus, PUBLISHED_MS_PER_TOKEN[1])
        h = sess.header
        weight_bytes = sum(L.qkv.qs.numel() * 4 + L.qkv.scales.numel() * 2 + L.wo.qs.numel() * 4 + L.wo.scales.numel() * 2 +
                           L.w13.qs.numel() * 4 + L.w13.scales.numel() * 2 + L.w2.qs.numel() * 4 + L.w2.scales.numel() * 2
                           for L in sess.weights.layers) + sess.weights.wcls.qs.numel() * 4 + sess.weights.wcls.scales.numel() * 2
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm = peaks.get("hbm_gbs", 6650.0)
        out = {
            "metric": "decode tokens/sec (batch-1 sequence, greedy) + prefill TTFT, Llama-3.1-8B q40" if args.model == "llama-3.1-8b"
                      else f"decode tokens/sec + prefill TTFT, {args.model} q40",
            "value": round(value, 2), "unit": "tokens/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
            "ms_per_step": round(ms_per_step, 4), "higher_is_better": True, "scaling": "strong",
            "vs_baseline": round(value / base, 2), "dtype": "q40 weights, q80 activations (int8 dp4a), bf16 KV, f32 accum",
            "data": "synthetic (random-init weights in .m layout, synthetic prompt)",
            "config": {"model": args.model, "global_batch": 1, "seq_len": args.prompt_len + steps, "prompt_len": args.prompt_len,
                       "parallelism": f"tp{args.gpus}", "decode_path": "persistent megakernel" if (eng.mega and eng.mega_active) else "multi-kernel PDL chain", "l2_policy": "weights per step (%.2f GB/GPU) >> 126 MB L2, no flush needed" % (weight_bytes / 1e9),
                       "baseline_ref": "reference published Llama-2-7B q40 ms/token on %d x RPi 4B (report.pdf)" % args.gpus},
            "ttft_ms": round(ttft_ms, 3), "prefill_tokens_per_s": round(args.prompt_len / ttft_ms * 1e3, 1),
            "e2e": {"value": round(steps / e2e_ms * 1e3, 2), "unit": "tokens/s", "h2d_bytes_per_step": 8, "d2h_bytes_per_step": 4},
            "gpu_launches": eng.launches_per_decode_step * steps,
            "hbm_roofline": {"weight_bytes_per_step_per_gpu": weight_bytes, "achieved_gbs": round(weight_bytes / ms_per_step / 1e6, 1),
                             "frac_of_measured_hbm": round(weight_bytes / ms_per_step / 1e6 / hbm, 3)},
            "clocks": clocks, "tokens_agree": e2e_tokens == toks, "impl": "ours",
            "tokens_sha": hashlib.sha1(",".join(map(str, toks[:16])).encode()).hexdigest()[:16],   # first 16 greedy tokens: TP=N must equal TP=1
            "load_s": round(load_s, 2), "bytes_uploaded_per_rank": int(sess.weights.bytes_uploaded),
            "extra": extra,
        }
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------------------
def ref_binary():
    """The reference tree that oracle/build_reference.sh put under oracle/_ref/, copied to the cache directory and built there
    (the repository may be read-only)."""
    tree = os.path.join(ROOT, "oracle", "_ref", "distributed-llama")
    if not os.path.isdir(tree):
        return None, "reference sources not present under oracle/_ref (oracle/build_reference.sh)"
    src = os.path.join(CACHE_DIR, "reference")
    exe = os.path.join(src, "dllama")
    if not os.path.isdir(src):
        shutil.copytree(tree, src)
        subprocess.run(["chmod", "-R", "u+w", src])
    # always (re)build on the box we run on: the reference Makefile uses -march=native
    stamp = os.path.join(src, ".built_on")
    host_id = open("/proc/cpuinfo").read().split("model name")[1].split("\n")[0] if os.path.exists("/proc/cpuinfo") else "?"
    if not os.path.exists(exe) or not os.path.exists(stamp) or open(stamp).read() != host_id:
        subprocess.run(["make", "clean"], cwd=src, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        r = subprocess.run(["make", "dllama", f"-j{os.cpu_count() or 4}"], cwd=src, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if r.returncode != 0 or not os.path.exists(exe):
            return None, "reference build failed: " + r.stdout[-300:].replace("\n", " ")
        open(stamp, "w").write(host_id)
    return exe, None


def _cpu_topology():
    """(logical CPUs this process may use, hardware threads per core) — the reference spins one busy thread per --nthreads."""
    try:
        cpus = sorted(os.sched_getaffinity(0))
    except Exception:
        cpus = list(range(os.cpu_count() or 8))
    tpc = 1
    try:
        sib = open(f"/sys/devices/system/cpu/cpu{cpus[0]}/topology/thread_siblings_list").read().strip()
        tpc = max(1, len([x for part in sib.split(",") for x in ([part] if "-" not in part else range(int(part.split("-")[0]), int(part.split("-")[1]) + 1))]))
    except Exception:
        pass
    return cpus, tpc


def _run_reference_once(exe, args, model_path, tok_path, n, threads, steps, warm, cpus, timeout):
    """One run of the stock reference CLI: root + (n-1) `dllama worker` processes on 127.0.0.1, each pinned to its own CPU set."""
    workers, ports = [], []
    per = max(1, len(cpus) // n)

    def pin(i):
        mine = cpus[i * per:(i + 1) * per] or cpus
        return lambda: os.sched_setaffinity(0, mine)
    try:
        for w in range(n - 1):
            port = 9999 - w
            ports.append(port)
            workers.append(subprocess.Popen([exe, "worker", "--port", str(port), "--nthreads", str(threads)],
                                            stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, preexec_fn=pin(w + 1)))
        if workers:
            time.sleep(2.0)
        prompt = " ".join(["hello"] * max(1, args.prompt_len - 1))
        total_steps = args.prompt_len + steps + warm + 8
        cmd = [exe, "inference", "--model", model_path, "--tokenizer", tok_path, "--buffer-float-type", "q80",
               "--prompt", prompt, "--steps", str(total_steps), "--nthreads", str(threads), "--temperature", "0",
               "--max-seq-len", str(max(args.max_seq_len, total_steps + 8))]
        if ports:
            cmd += ["--workers"] + [f"127.0.0.1:{p}" for p in ports]
        t0 = time.time()
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=timeout, preexec_fn=pin(0))
        wall = time.time() - t0
        text = r.stdout
        pred = [int(m.group(1)) + int(m.group(2)) for m in re.finditer(r"Pred\s*(\d+) ms Sync\s*(\d+) ms", text)]
        evals = [(int(m.group(1)) + int(m.group(2)), int(m.group(3))) for m in re.finditer(r"Eval\s*(\d+) ms Sync\s*(\d+) ms.*\((\d+) tokens\)", text)]
        m_pred = re.search(r"Prediction\s*\n\s*nTokens: (\d+)\s*\n\s*tokens/s: ([\d.]+) \(([\d.]+) ms/tok\)", text)
        if r.returncode != 0 or not m_pred:
            return {"error": "reference run failed: " + text[-300:].replace("\n", " ")}
        timed = pred[warm: warm + steps] if len(pred) >= warm + steps else pred[warm:]
        ms_per_step = sum(timed) / max(1, len(timed)) if timed else float(m_pred.group(3))
        if ms_per_step <= 0:     # ms granularity of the reference's printout; fall back to its own summary
            ms_per_step = float(m_pred.group(3))
        return {"ms_per_step": ms_per_step, "n_timed": len(timed) or int(m_pred.group(1)), "eval_ms": sum(e[0] for e in evals),
                "summary_tok_s": float(m_pred.group(2)), "wall": wall, "threads": threads}
    except subprocess.TimeoutExpired:
        return {"error": "reference run timed out"}
    finally:
        for p in workers:
            try:
                p.kill()
                p.wait(timeout=5)
            except Exception:
                pass


def run_reference(args):
    """Reference arm: the UNMODIFIED reference tree (oracle/_ref/distributed-llama), built with its own Makefile, driven through
    its own CLI. The only thing chosen here is how it is launched: `--nthreads` is swept over the power-of-two counts that fit the
    physical cores available to each of the n processes (short probe runs), processes are pinned to disjoint CPU sets, and the
    best configuration is then timed on the full step count."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        # ranks other than 0 only exist because the driver launches both arms the same way
        try:
            import torch.distributed as dist
            dist.init_process_group("gloo")
            dist.barrier()
            dist.destroy_process_group()
        except Exception:
            pass
        return

    def finish(payload):
        print(json.dumps(payload), flush=True)
        if int(os.environ.get("WORLD_SIZE", "1")) > 1:
            try:
                import torch.distributed as dist
                dist.init_process_group("gloo")
                dist.barrier()
                dist.destroy_process_group()
            except Exception:
                pass

    exe, err = ref_binary()
    if exe is None:
        return finish({"impl": "reference", "unavailable": err})
    model_path, tok_path = ensure_model(args.model)
    n = args.gpus
    cpus, tpc = _cpu_topology()
    phys_per_proc = max(1, len(cpus) // tpc // n)
    cands = sorted({t for t in (4, 8, 16, 32, 64) if t <= phys_per_proc} | {1 << (max(1, min(64, phys_per_proc)).bit_length() - 1)})
    warm = max(args.warmup, 3)
    deadline = time.time() + args.ref_timeout
    sweep = {}
    best_t = cands[-1]
    if len(cands) > 1:
        for t in cands:
            if time.time() > deadline - 0.6 * args.ref_timeout:
                break
            r = _run_reference_once(exe, args, model_path, tok_path, n, t, 8, 2, cpus, max(60, int(deadline - time.time())))
            if "error" not in r:
                sweep[t] = round(1000.0 / r["ms_per_step"], 3)
        if sweep:
            best_t = max(sweep, key=sweep.get)
    r = _run_reference_once(exe, args, model_path, tok_path, n, best_t, args.steps, warm, cpus, max(60, int(deadline - time.time())))
    if "error" in r:
        return finish({"impl": "reference", "unavailable": r["error"]})
    value = 1000.0 / r["ms_per_step"]
    base = 1000.0 / PUBLISHED_MS_PER_TOKEN.get(n, PUBLISHED_MS_PER_TOKEN[1])
    finish({"metric": "decode tokens/sec (batch-1 sequence, greedy) + prefill TTFT, Llama-3.1-8B q40" if args.model == "llama-3.1-8b"
                      else f"decode tokens/sec + prefill TTFT, {args.model} q40",
            "value": round(value, 3), "unit": "tokens/s", "n_gpus": n, "steps": r["n_timed"], "warmup": warm,
            "ms_per_step": round(r["ms_per_step"], 3), "higher_is_better": True, "scaling": "strong", "vs_baseline": round(value / base, 2),
            "dtype": "q40 weights, q80 activations (reference CPU build, AVX)", "data": "synthetic (same .m/.t files)",
            "config": {"model": args.model, "global_batch": 1, "seq_len": args.prompt_len + args.steps, "prompt_len": args.prompt_len,
                       "parallelism": f"tp{n}", "launch": f"root + {n - 1} TCP-loopback workers, pinned to disjoint CPU sets",
                       "nthreads_per_node": r["threads"], "nthreads_sweep_tok_s": sweep,
                       "note": "the reference has no CUDA path; its stock build runs on the host CPUs"},
            "ttft_ms": r["eval_ms"], "prefill_tokens_per_s": round(max(1, args.prompt_len - 1) / max(1e-3, r["eval_ms"]) * 1e3, 1),
            # end to end = the reference's own root-side wall clock per generated token (forward + host sampling + printing)
            "e2e": {"value": r["summary_tok_s"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                    "note": "reference summary line `Prediction tokens/s` (root wall clock, CPU only: no device copies)"},
            "gpu_launches": 0, "impl": "reference", "reference_summary_tokens_per_s": r["summary_tok_s"], "wall_s": round(r["wall"], 1)})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="llama-3.1-8b")
    ap.add_argument("--prompt-len", type=int, default=64)
    ap.add_argument("--max-seq-len", type=int, default=4096)
    ap.add_argument("--ref-timeout", type=int, default=1500)
    ap.add_argument("--decode-path", default="mega", choices=["multi", "mega"], help="multi-kernel PDL chain or persistent megakernel")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the timed decode's tokens and last-step logits as DIR/*.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
