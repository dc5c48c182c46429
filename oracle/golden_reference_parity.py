"""Regenerates tests/golden/reference_parity.json: what the original project's `dllama perplexity` reports on the tiny synthetic
models that tests/test_reference_parity.py compares the PyTorch oracle against.

    bash oracle/build_reference.sh <distributed-llama checkout>
    python oracle/golden_reference_parity.py

The models are written exactly as the `tmp_models` fixture of tests/conftest.py writes them; their SHA-256 is stored with the
reference's output so the test can tell when the generator no longer produces the files the reference read.
"""
import hashlib
import json
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

REF_EXE = os.path.join(ROOT, "oracle", "_ref", "distributed-llama", "dllama")
GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_parity.json")
PROMPT = "Hello world, the model is a llama and the token"
MODELS = ("tiny-llama", "tiny-llama31", "tiny-qwen3", "tiny-qwen3-moe")


def sha256(path: str) -> str:
    with open(path, "rb") as f:
        return hashlib.sha256(f.read()).hexdigest()


def main():
    from distributed_llama_b200.models.config import get_config
    from distributed_llama_b200.models.synthetic import write_synthetic_model, write_synthetic_tokenizer

    if not os.path.exists(REF_EXE):
        raise SystemExit(f"{REF_EXE} is missing: run oracle/build_reference.sh first")
    out = {"reference": "b4rtaz/distributed-llama @ 8d624a7b, CPU build: dllama perplexity --buffer-float-type q80 --nthreads 2",
           "prompt": PROMPT, "models": {}}
    with tempfile.TemporaryDirectory() as d:
        for name in MODELS:
            cfg = get_config(name)
            m, t = os.path.join(d, f"{name}.m"), os.path.join(d, f"{name}.t")
            write_synthetic_model(m, cfg, seed=7)
            write_synthetic_tokenizer(t, cfg.vocab_size, style="chatml" if "qwen" in name else "llama3")
            r = subprocess.run([REF_EXE, "perplexity", "--model", m, "--tokenizer", t, "--buffer-float-type", "q80", "--prompt", PROMPT,
                                "--nthreads", "2"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=300)
            if r.returncode != 0:
                raise SystemExit(f"reference failed on {name}:\n{r.stdout[-2000:]}")
            out["models"][name] = {"model_sha256": sha256(m), "tokenizer_sha256": sha256(t),
                                   "probs": [float(x) for x in re.findall(r"prob=([0-9.eE+-]+)", r.stdout)],
                                   "perplexity": float(re.search(r"perplexity: ([0-9.]+)", r.stdout).group(1))}
    os.makedirs(os.path.dirname(GOLDEN), exist_ok=True)
    with open(GOLDEN, "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print(f"wrote {GOLDEN}")


if __name__ == "__main__":
    main()
