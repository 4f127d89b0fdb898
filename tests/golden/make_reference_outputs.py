"""Writes tests/golden/reference_*.pt.gz: what the REAL reference (oracle/_ref, compiled by
oracle/build_ref.py from the reference's own sources) materialises for the programs the tests
compare against it -- the same programs, seeds and dtypes the tests run.  Format: oracle/golden.py.

    python tests/golden/make_reference_outputs.py [--only cpu_parity,differential,gpu_cases,t1_fullsize]

Needs the compiled reference; every run is a subprocess (the reference and torchdistx_b200 register
the same dispatch keys and cannot share a process).  Regenerate when a test's programs change.
"""
import argparse
import os
import subprocess
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import cases  # noqa: E402
from oracle import golden as G  # noqa: E402

# tests/test_parity_cpu_reference.py
PARITY_CASES = [
    ("linear128", "fp32"), ("init_zoo", "fp32"), ("init_zoo", "bf16"), ("mlp_stack", "fp32"),
    ("tiny_llama", "fp32"), ("tiny_llama", "bf16"), ("tiny_gpt2", "fp32"),
    ("torch_transformer", "fp32"), ("clones", "fp32"), ("cast_variant", "fp32"),
] + [(f"family_{name}", "fp32") for name in cases.FAMILIES] + [("family_llama", "bf16"), ("family_gpt2", "bf16")]
PARITY_SEED = 5
# tests/test_reference_differential_cpu.py
DIFFERENTIAL_SCRIPTS = 300
# tests/test_materialize_gpu.py (two seeds: tensors equal across them are deterministic programs)
GPU_CASES = [("init_zoo", "fp32"), ("init_zoo", "bf16"), ("tiny_llama", "fp32"), ("tiny_llama", "bf16"),
             ("tiny_gpt2", "fp32"), ("mlp_stack", "fp32"), ("torch_transformer", "fp32"), ("clones", "fp32"),
             ("cast_variant", "fp32")]
GPU_SEEDS = (5, 6)
GPU_QUANTILES = 512  # kept where those tests run a KS test: fp32 cases, tensors of >= 4096 elements
# tests/test_engine_round2_gpu.py: padding_idx embeddings, (weight, padded row)
PADDED_ROWS = (("torch_style", 3), ("hf_style", 0), ("last_row", 256))
# tests/test_t1_fullsize_gpu.py: (case, dtype the reference runs in, --round-to)
T1_SEED = 11
T1_RUNS = {
    "llama_bf16": ("llama8b_layer", "fp32", "bf16"),
    "llama_cast": ("llama8b_layer_cast", "fp32", ""),
    "big_fp32": ("big_inits", "fp32", ""),
    "big_bf16": ("big_inits", "fp32", "bf16"),
}
T1_QUANTILES = 4096

VIEW_WRITE = (
    "import sys, torch; sys.path.insert(0, %r)\n"
    "from torch import nn\n"
    "from oracle import ref_torchdistx as R\n"
    "def before():\n"
    "    t = torch.ones(4, 4); t[1].zero_(); return nn.ParameterList([nn.Parameter(t)])\n"
    "def after():\n"
    "    t = nn.Parameter(torch.ones(4, 4))\n"
    "    with torch.no_grad(): t[1].zero_()\n"
    "    return nn.ParameterList([t])\n"
    "for fn in (before, after):\n"
    "    m = R.deferred_init(fn); R.materialize_module(m); print(fn.__name__, m[0].detach()[1].tolist())\n" % ROOT)


def ref_driver(*args):
    subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "ref_driver.py"), *map(str, args)],
                   check=True, cwd=ROOT, timeout=1800)


def ref_cases(case_list, seed, tmp):
    out = os.path.join(tmp, f"cases{seed}")
    os.makedirs(out, exist_ok=True)
    ref_driver("--cases", ",".join(f"{c}:{d}" for c, d in case_list), "--seed", seed, "--outdir", out)
    return {(c, d): torch.load(os.path.join(out, f"{c}_{d}.pt")) for c, d in case_list}


def cpu_parity(tmp):
    ref = ref_cases(PARITY_CASES, PARITY_SEED, tmp)
    return {f"{c}_{d}": {k: {"dtype": str(t.dtype), "shape": tuple(t.shape), "digest": G.digest(t)}
                         for k, t in ref[(c, d)].items()} for c, d in PARITY_CASES}


def differential(tmp):
    out = os.path.join(tmp, "refdiff.pt")
    subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "ref_fuzz_driver.py"), "--lo", "0",
                    "--hi", str(DIFFERENTIAL_SCRIPTS), "--out", out], check=True, cwd=ROOT, timeout=1800)
    runs = torch.load(out)
    scripts = {seed: r if isinstance(r, str) else {k: G.value_digest(v) for k, v in r.items()}
               for seed, r in runs.items()}
    view_write = subprocess.run([sys.executable, "-c", VIEW_WRITE], check=True, capture_output=True, text=True,
                                cwd=ROOT, timeout=300).stdout
    return {"scripts": scripts, "view_write": view_write}


def gpu_cases(tmp):
    a, b = (ref_cases(GPU_CASES + [("padded_embeddings", "fp32")], s, tmp) for s in GPU_SEEDS)
    out = {}
    for key in GPU_CASES:
        out[f"{key[0]}_{key[1]}"] = {
            k: t if torch.equal(t, b[key][k]) else
            G.summary(t, GPU_QUANTILES if key[1] == "fp32" and t.numel() >= 4096 else 0)
            for k, t in a[key].items()}
    padded = a[("padded_embeddings", "fp32")]
    out["padded_embeddings_fp32"] = {
        f"{name}.weight": {"padded_row": padded[f"{name}.weight"][row].clone(),
                           "rest": G.summary(torch.cat([padded[f"{name}.weight"][:row],
                                                        padded[f"{name}.weight"][row + 1:]]))}
        for name, row in PADDED_ROWS}
    return out


def t1_fullsize(tmp):
    out = {}
    for key, (case, dtype, round_to) in T1_RUNS.items():
        p = os.path.join(tmp, f"{key}.pt")
        ref_driver("--case", case, "--dtype", dtype, "--seed", T1_SEED, "--stats", "--out", p,
                   *(["--round-to", round_to] if round_to else []))
        ref = torch.load(p)
        for k, r in ref.items():
            if isinstance(r, dict):  # the 2^20-element strided subsample -> its quantiles
                r["quantiles"] = G.quantiles(r.pop("sample"), T1_QUANTILES)
        out[key] = ref
        os.remove(p)
    return out


MAKERS = {"cpu_parity": cpu_parity, "differential": differential, "gpu_cases": gpu_cases,
          "t1_fullsize": t1_fullsize}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default=",".join(MAKERS))
    a = ap.parse_args()
    with tempfile.TemporaryDirectory() as tmp:
        for name in a.only.split(","):
            p = G.save(f"reference_{name}", MAKERS[name](tmp))
            print(p, os.path.getsize(p), "bytes", flush=True)


if __name__ == "__main__":
    main()
