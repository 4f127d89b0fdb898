"""bench.py -- params/s and HBM GB/s of `materialize_module` (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--model llama3-8b] [--impl reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

A "step" is one `materialize_module` of one freshly recorded (deferred_init, zero-storage) model:
every parameter and buffer written to HBM once.  Recording (Python module construction under
`deferred_init`) is outside the timed region -- the metric is named for materialize_module.

  value  : params/s with the descriptor plan already resident in HBM (tdx_plan_launch only:
           the kernels, nothing else), whole job (all ranks), max time over ranks.
  e2e    : the same metric through the public API `materialize_module(m, device=cuda[, shard=...])`
           -- planning, allocation, descriptor H2D copy, kernels, and a D2H read of 64 result bytes
           inside the timed region.
  N > 1  : one model, dim-0 sharded across the ranks (each rank writes only its rows; the
           unsharded tensors never exist) => "scaling": "strong".  The only collective is the
           16-byte seed/offset broadcast (torchdistx_b200.parallel.sync_rng), once per step inside
           the e2e timed region; there is none in or between the kernels.
  --impl reference : the reference's own CPU materialize (oracle/_ref = pytorch/torchdistx
           compiled from the reference's sources) on a bounded sample of the same model, on the host cores.
  --dump-outputs DIR : after the timed steps, every parameter and buffer of the model the `value`
           steps wrote, as DIR/<name>.npy (see dump_outputs), for comparing two builds output for
           output: the model, the seed and the step counts fix every value.
"""
from __future__ import annotations

import argparse
import ctypes
import gc
import json
import os
import statistics
import subprocess
import sys
import threading
import time
import zlib

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODELS = {
    # name: (family, kwargs, dtype)
    "llama3-8b": ("llama", dict(vocab_size=128256, hidden_size=4096, intermediate_size=14336,
                                num_hidden_layers=32, num_attention_heads=32, num_key_value_heads=8,
                                max_position_embeddings=8192, rope_theta=500000.0), "bf16"),
    "llama3-70b": ("llama", dict(vocab_size=128256, hidden_size=8192, intermediate_size=28672,
                                 num_hidden_layers=80, num_attention_heads=64, num_key_value_heads=8,
                                 max_position_embeddings=8192, rope_theta=500000.0), "bf16"),
    # SURVEY 8d cfg3 variant: constructed in fp32, converted with `.to(torch.bfloat16)` inside deferred_init
    "llama3-8b-cast": ("llama", dict(vocab_size=128256, hidden_size=4096, intermediate_size=14336,
                                     num_hidden_layers=32, num_attention_heads=32, num_key_value_heads=8,
                                     max_position_embeddings=8192, rope_theta=500000.0), "fp32->bf16"),
    "gpt2-xl": ("gpt2", dict(n_layer=48, n_embd=1600, n_head=25, vocab_size=50257, n_positions=1024), "fp32"),
    "llama-tiny": ("llama", dict(vocab_size=4096, hidden_size=512, intermediate_size=1024,
                                 num_hidden_layers=4, num_attention_heads=8, num_key_value_heads=2), "bf16"),
}


def build_model(name: str, layers: int | None = None, vocab: int | None = None):
    """Constructs the HF model (random init, no checkpoint); call under deferred_init."""
    import torch
    family, kw, dtype = MODELS[name]
    kw = dict(kw)
    if layers is not None:
        kw["num_hidden_layers" if family == "llama" else "n_layer"] = layers
    if vocab is not None:
        kw["vocab_size"] = vocab
    prev = torch.get_default_dtype()
    torch.set_default_dtype({"bf16": torch.bfloat16, "fp32": torch.float32, "fp32->bf16": torch.float32}[dtype])
    try:
        if family == "llama":
            from transformers import LlamaConfig, LlamaForCausalLM
            m = LlamaForCausalLM(LlamaConfig(**kw))
            return m.to(torch.bfloat16) if dtype == "fp32->bf16" else m
        from transformers import GPT2Config, GPT2LMHeadModel
        return GPT2LMHeadModel(GPT2Config(**kw))
    finally:
        torch.set_default_dtype(prev)


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int, period_ms: int = 100):
        # rank 0 samples every 100 ms (20 ms around the short kernels-only region); the other ranks every 500 ms (eight fast
        # nvidia-smi loops compete with the ranks' own driver calls inside the timed region)
        self.rows, self.proc, self.index, self.period_ms = [], None, index, period_ms

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", str(self.period_ms)],
                                         stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            # the timed regions are short (the kernels-only one is ~35 ms): do not start them before the
            # sampler has delivered its first row, or every sample could fall after the region
            t_end = time.time() + 1.5
            while not self.rows and time.time() < t_end:
                time.sleep(0.005)
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 6 for n, v in zip(names, r[2:6]) if v == "Active"})
        busy = [c for c in sm if c > 500] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ---------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the real reference on the host cores, bounded sample
# ---------------------------------------------------------------------------------------------
REF_SNIPPET = r"""
import json, sys, time, torch
sys.path.insert(0, {root!r})
from oracle import ref_torchdistx as R
import bench
torch.set_default_dtype({{'bf16': torch.bfloat16, 'fp32': torch.float32, 'fp32->bf16': torch.float32}}[{dtype!r}])
times, n = [], 0
for i in range({reps}):
    m = R.deferred_init(lambda: bench.build_model({model!r}, layers={layers}, vocab={vocab}))
    n = sum(p.numel() for p in m.parameters())
    torch.manual_seed(i)
    t0 = time.perf_counter(); R.materialize_module(m); times.append(time.perf_counter() - t0)
    del m
print(json.dumps({{"times": times, "params": n, "threads": torch.get_num_threads()}}))
"""


def reference_sample(model: str, layers: int, reps: int):
    """Runs the reference (subprocess: it registers the same dispatch keys as torchdistx_b200)."""
    dtype = MODELS[model][2]
    code = REF_SNIPPET.format(root=ROOT, model=model, layers=layers, reps=reps, dtype=dtype,
                              vocab=SAMPLE_VOCAB.get(model))
    # torchrun exports OMP_NUM_THREADS=1 to its workers: the reference arm gets every host core it can use
    env = {k: v for k, v in os.environ.items() if k not in ("OMP_NUM_THREADS", "MKL_NUM_THREADS")}
    out = subprocess.run([sys.executable, "-c", code], check=True, capture_output=True, text=True, cwd=ROOT,
                         env=env, timeout=1500)
    return json.loads(out.stdout.strip().splitlines()[-1])


# Bounded CPU sample of the same workload (a few seconds of CPU work per repetition): one decoder
# layer of the named model at full width (all seven Llama linears: dead uniform_ + live normal_,
# exactly the chains of the full model) with the vocabulary cut to 2048 rows so that the two
# vocab-sized matrices do not dominate; GPT-2 XL: 4 of its 48 blocks, full vocabulary.
SAMPLE_VOCAB = {"llama3-8b": 2048, "llama3-8b-cast": 2048, "llama3-70b": 2048}


def sample_layers(model: str) -> int:
    return {"llama3-8b": 1, "llama3-8b-cast": 1, "llama3-70b": 1, "gpt2-xl": 4, "llama-tiny": 4}[model]


def run_reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    layers = sample_layers(a.model)
    res = reference_sample(a.model, layers, a.warmup + a.steps)
    ts = res["times"][a.warmup:]
    ms = 1e3 * sum(ts) / len(ts)
    value = res["params"] / (sum(ts) / len(ts))
    sample = (f"{a.model} cut to {layers} decoder layer(s)"
              f"{', vocab ' + str(SAMPLE_VOCAB[a.model]) if a.model in SAMPLE_VOCAB else ''} "
              f"({res['params']:,} params), {MODELS[a.model][2]}, device=cpu, reference materialize_module")
    line = {"impl": "reference", "metric": "materialize_module params/s", "value": value, "unit": "params/s",
            "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": MODELS[a.model][2], "data": "synthetic (random init of the named architecture)",
            "config": {"workload": f"{a.model} materialize_module", "sample": sample},
            "cpu_baseline": {"value": value, "unit": "params/s", "cores": res["threads"], "kind": "reference",
                             "sample": sample,
                             "note": "ATen CPU RNG kernels are serial under the generator mutex; threads only help fills"},
            "e2e": {"value": value, "unit": "params/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# baseline B (SURVEY 8d): the reference itself replaying on the GPU with stock ATen kernels
# ---------------------------------------------------------------------------------------------
GPU_REF_SNIPPET = r"""
import json, sys, time, torch
sys.path.insert(0, {root!r})
from oracle import ref_torchdistx as R
import bench
torch.cuda.set_device({index})
times, n = [], 0
for i in range({reps}):
    with torch.device('cuda:{index}'):
        m = R.deferred_init(lambda: bench.build_model({model!r}))
    n = sum(p.numel() for p in m.parameters())
    torch.manual_seed(i); torch.cuda.synchronize()
    t0 = time.perf_counter(); R.materialize_module(m); torch.cuda.synchronize(); times.append(time.perf_counter() - t0)
    del m
print(json.dumps({{"times": times, "params": n}}))
"""


def reference_on_gpu(model: str, index: int, reps: int = 3):
    """`oracle/_ref` (the reference's own engine) with the model recorded for cuda: one dispatcher
    call and one stock ATen kernel per recorded op, dead ops included (deferred_init.cc:218-220)."""
    code = GPU_REF_SNIPPET.format(root=ROOT, model=model, index=index, reps=reps)
    out = subprocess.run([sys.executable, "-c", code], check=True, capture_output=True, text=True, cwd=ROOT,
                         timeout=600)  # (a side measurement: a stuck child must not take the headline with it)
    return json.loads(out.stdout.strip().splitlines()[-1])


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
def desc_bytes(C, d):
    return d.elem_count * (4 if d.dtype in (C.TDX_F32, C.TDX_RAW32) else 8 if d.dtype == C.TDX_RAW64
                           else 1 if d.dtype == C.TDX_RAW8 else 2)


class Ctx:
    """What every measurement of one run shares."""


DUMP_BYTES = 60 << 20  # the arrays of --dump-outputs, in all (+ .npy headers and manifest.json: < 64 MB)


def dump_outputs(model, out_dir: str):
    """Writes each parameter and buffer of `model` as out_dir/<name>.npy -- float32 (exact for 16- and
    32-bit floats) or float64 (float64 and integer tensors) -- and out_dir/manifest.json.  Tensors share
    DUMP_BYTES, the smallest first; one that does not fit whole is written as the elements at the sorted
    flat indices numpy.random.default_rng(zlib.crc32(name)).choice(numel, size=k, replace=False)."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    tensors = sorted(dict(list(model.named_parameters()) + list(model.named_buffers())).items(),
                     key=lambda kv: kv[1].numel())
    left, manifest = DUMP_BYTES, {}
    for i, (name, t) in enumerate(tensors):
        wide = t.dtype == torch.float64 or not t.is_floating_point()
        out_dtype = torch.float64 if wide else torch.float32
        n = t.numel()
        k = min(n, left // (len(tensors) - i) // (8 if wide else 4))
        flat = t.detach().reshape(-1)
        entry = {"shape": list(t.shape), "dtype": str(t.dtype), "numel": n, "written": k}
        if k < n:
            idx = np.sort(np.random.default_rng(zlib.crc32(name.encode())).choice(n, size=k, replace=False))
            flat = flat[torch.from_numpy(idx).to(flat.device)]
            entry["sample"] = "numpy.random.default_rng(zlib.crc32(name)).choice(numel, size=written, replace=False), sorted"
        arr = flat.to(out_dtype).cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), arr)
        left -= arr.nbytes
        manifest[name] = entry
    with open(os.path.join(out_dir, "manifest.json"), "w") as f:
        json.dump(manifest, f, indent=1)


def measure_model(cx, model: str, steps: int, warmup: int, first_call: bool = False, roofline_only: bool = False,
                  dump_dir: str | None = None):
    """value / e2e / roofline of one model, the procedure of the module docstring.
    `roofline_only` (for ncu): one materialize, then 3 + steps launches of the dominant kernel's plan.
    `dump_dir`: where dump_outputs writes the model the timed `value` launches wrote into."""
    import torch
    import torch.distributed as dist

    from torchdistx_b200 import _cabi as C
    from torchdistx_b200 import parallel
    from torchdistx_b200.deferred_init import (deferred_init, last_descriptors, last_materialize_stats,
                                               materialize_module)

    dev, world, rank, local, lib, stream = cx.dev, cx.world, cx.rank, cx.local, cx.lib, cx.stream
    shard = (rank, world) if world > 1 else None
    if getattr(cx, "as_rank_of", 0) > 1:  # diagnostic: one process builds rank 0's share of a W-way sharded model
        shard = (0, cx.as_rank_of)
    dtype = MODELS[model][2]
    res = {"model": model, "dtype": dtype}

    # ---- record K+W+1 zero-storage models (untimed) -----------------------------------------
    t0 = time.perf_counter()
    fakes = [deferred_init(build_model, model) for _ in range(1 if roofline_only else warmup + steps + 1)]
    res["record_s_per_model"] = (time.perf_counter() - t0) / len(fakes)
    n_params = res["params"] = sum(p.numel() for p in fakes[0].parameters())
    res["tensors"] = len(list(fakes[0].parameters())) + len(list(fakes[0].buffers()))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- e2e: public API, H2D of descriptors + D2H of a result inside the timed region ---------
    probe = torch.empty(32, dtype=torch.float32 if dtype == "fp32" else torch.bfloat16).pin_memory()
    last_name = list(dict(fakes[0].named_parameters()))[-1]  # looked up outside the timed region
    host_split = {"api_return_ms": 0.0, "sync_ms": 0.0, "n": 0, "on": False}

    def step(m):
        t0 = time.perf_counter()
        if world > 1:
            # the path's one collective (16 B broadcast) on the first call; afterwards the ranks'
            # generators advance in lock step and the call returns without communicating
            parallel.sync_rng(dev)
        materialize_module(m, device=dev, shard=shard)
        t1 = time.perf_counter()
        last = m.get_parameter(last_name)
        probe.copy_(last.detach().flatten()[:32], non_blocking=True)  # D2H read of the step's result
        torch.cuda.current_stream().synchronize()
        t2 = time.perf_counter()
        if host_split["on"]:
            host_split["api_return_ms"] += (t1 - t0) * 1e3
            host_split["sync_ms"] += (t2 - t0) * 1e3
            host_split["n"] += 1

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(0 if roofline_only else warmup):
        if i == 0 and first_call:
            # the very first materialize_module of the process: CUDA module load, cold caching
            # allocator (cudaMalloc), pinned staging buffers -- what a user who calls it once pays
            barrier()
            t0 = time.perf_counter()
            step(fakes[i])
            res["e2e_cold_ms"] = max_over_ranks((time.perf_counter() - t0) * 1e3)
            res["cold_alloc_ms"] = last_materialize_stats().get("alloc_us", 0) / 1e3
        else:
            step(fakes[i])
        fakes[i] = None
    st = last_materialize_stats()
    res["h2d"] = int(st.get("upload_bytes", 0))  # plan images (descriptors, prefix sums, work lists) per step
    barrier()
    # Each step is timed on its own (events on the launching stream, bracketed by a synchronize);
    # tearing down the previous step's model -- Python GC of ~500 modules, hundreds of allocator
    # frees -- happens between the timed regions: it is not part of the API under test.
    total = 0.0
    host_split["on"] = True
    clk_e2e = ClockSampler(local, 100 if rank == 0 else 500)
    # Python's cyclic GC is collected once before and switched off across the timed steps, as `timeit`
    # does: a collection triggered by the ~600 objects a step creates walks the whole heap of THIS
    # harness (a dozen recorded models), which is not the API's cost -- and tens of milliseconds of
    # it between steps let the GPU fall back to its idle clocks before every timed call.
    gc.collect()
    gc.disable()
    with clk_e2e:
        for i in range(*((0, 0) if roofline_only else (warmup, warmup + steps))):
            barrier()
            e0.record()
            step(fakes[i])
            e1.record()
            e1.synchronize()
            total += e0.elapsed_time(e1)
            fakes[i] = None  # untimed: release the model (refcounts: no collector needed) before the next step allocates
    gc.enable()
    res["e2e_ms"] = max_over_ranks(total / steps) if not roofline_only else 0.0
    res["clk_e2e"] = clk_e2e.summary()
    res["host_split"] = {"api_return": round(host_split["api_return_ms"] / max(host_split["n"], 1), 3),
                         "gpu_done": round(host_split["sync_ms"] / max(host_split["n"], 1), 3)}
    if world > 1:
        assert parallel.check_agreement(dev), "ranks disagree on the generator state after the timed steps"

    # ---- value: plan resident in HBM, kernels only ----------------------------------------------
    keep = fakes[-1]
    materialize_module(keep, device=dev, shard=shard)  # allocates the outputs we re-launch into
    descs = last_descriptors()
    st = res["stats"] = last_materialize_stats()
    res["descs"] = len(descs)
    my_bytes = res["my_bytes"] = sum(desc_bytes(C, d) for d in descs)
    ws_bytes = lib.tdx_init_workspace_bytes(len(descs))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    plan = C.TdxPlan()
    C.check(lib.tdx_plan_upload(descs, len(descs), ws.data_ptr(), ws_bytes, stream, ctypes.byref(plan)))
    clk = ClockSampler(local, 20 if rank == 0 else 500)
    res["ms"], res["launches_per_step"] = 1.0, 0
    if not roofline_only:
        for _ in range(max(warmup, 3)):
            C.check(lib.tdx_plan_launch(ctypes.byref(plan), ws.data_ptr(), stream))
        res["launches_per_step"] = lib.tdx_last_launch_count()
        barrier()
        with clk:
            e0.record()
            for _ in range(steps):
                C.check(lib.tdx_plan_launch(ctypes.byref(plan), ws.data_ptr(), stream))
            e1.record()
            barrier()
        res["ms"] = max_over_ranks(e0.elapsed_time(e1) / steps)
        if dump_dir:
            dump_outputs(keep, dump_dir if world == 1 else os.path.join(dump_dir, f"rank{rank}"))
    res["clk"] = clk.summary()

    # ---- roofline of the dominant kernel (most bytes), timed alone with the same events ----------
    fam = {}
    for d in descs:
        fam.setdefault((d.src, d.dtype if d.src != C.TDX_SRC_CONST else -1), []).append(d)
    dom_key = max(fam, key=lambda k: sum(desc_bytes(C, d) for d in fam[k]))
    dom = (C.TdxInitDesc * len(fam[dom_key]))(*fam[dom_key])
    dom_bytes = sum(desc_bytes(C, d) for d in dom)
    ws2 = torch.empty(lib.tdx_init_workspace_bytes(len(dom)), dtype=torch.uint8, device=dev)
    plan2 = C.TdxPlan()
    C.check(lib.tdx_plan_upload(dom, len(dom), ws2.data_ptr(), ws2.numel(), stream, ctypes.byref(plan2)))
    for _ in range(3):
        C.check(lib.tdx_plan_launch(ctypes.byref(plan2), ws2.data_ptr(), stream))
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        C.check(lib.tdx_plan_launch(ctypes.byref(plan2), ws2.data_ptr(), stream))
    e1.record()
    torch.cuda.synchronize()
    dom_ms = e0.elapsed_time(e1) / steps
    wide = any(d.algo & 0x0f == C.TDX_ALGO_WIDE32 for d in dom) and dom_key[1] != C.TDX_F32
    kname = {C.TDX_SRC_CONST: "tdx_fill_kernel", C.TDX_SRC_UNIFORM: "tdx_rng_kernel<GenUniform*> / tdx_lut16_kernel<TabUniform>",
             C.TDX_SRC_NORMAL: ("tdx_rng_kernel<GenNormalBM32<float>>" if dom_key[1] == C.TDX_F32 else
                                "tdx_rng_kernel<GenNormalBM32<16-bit>> (TDX_ALGO_WIDE32)" if wide else
                                "tdx_lut16_kernel<TabNormal, 16-bit> (+ tdx_rng_kernel<GenNormalICDF16> for descriptors < 2^18 elements)")}[dom_key[0]]
    peak, peak_src = peaks()
    achieved = dom_bytes / dom_ms / 1e6
    res["roofline"] = {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak, "unit": "GB/s",
                       "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                       "bytes_per_launch": dom_bytes, "ms_per_launch": dom_ms}
    del keep, ws, ws2, fakes
    gc.collect()
    torch.cuda.empty_cache()
    return res


def kernel_sweep(cx, max_bytes: int):
    """BASELINE config 5 at this run's N: one tensor of 1 MB .. 16 GB (x4 steps), each rank writing
    bytes / N of it (its dim-0 chunk: elem_begin = rank * n / N), normal_ / uniform_ /
    kaiming_uniform_ (= uniform_ with bound 1/sqrt(fan_in)) in bf16 and fp32; GB/s of the slowest
    rank x N, L2 flushed before every timed launch below 256 MB per rank."""
    import torch
    import torch.distributed as dist

    from torchdistx_b200 import _cabi as C

    dev, world, rank, lib, stream = cx.dev, cx.world, cx.rank, cx.lib, cx.stream
    peak, _ = peaks()
    ws = torch.empty(lib.tdx_init_workspace_bytes(1), dtype=torch.uint8, device=dev)
    flush = torch.empty(192 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    kinds = {"normal_bf16": (C.TDX_BF16, C.TDX_SRC_NORMAL, 0.0, 0.02), "uniform_bf16": (C.TDX_BF16, C.TDX_SRC_UNIFORM, -0.05, 0.05),
             "kaiming_uniform_bf16": (C.TDX_BF16, C.TDX_SRC_UNIFORM, -1 / 64, 1 / 64),
             "normal_f32": (C.TDX_F32, C.TDX_SRC_NORMAL, 0.0, 0.02), "uniform_f32": (C.TDX_F32, C.TDX_SRC_UNIFORM, -0.05, 0.05),
             "kaiming_uniform_f32": (C.TDX_F32, C.TDX_SRC_UNIFORM, -1 / 64, 1 / 64)}
    rows = []
    nbytes = 1 << 20
    while nbytes <= max_bytes:
        mine = nbytes // world
        buf = torch.empty(max(mine, 16), dtype=torch.uint8, device=dev)
        row = {"bytes": nbytes}
        for name, (dt, src, p0, p1) in kinds.items():
            isz = 4 if dt == C.TDX_F32 else 2
            n = mine // isz
            d = C.make_desc(buf.data_ptr(), dtype=dt, src=src, elem_begin=rank * n, elem_count=n, seed=1234, offset=8,
                            p0=p0, p1=p1)
            arr = (C.TdxInitDesc * 1)(d)
            plan = C.TdxPlan()
            C.check(lib.tdx_plan_upload(arr, 1, ws.data_ptr(), ws.numel(), stream, ctypes.byref(plan)))
            for _ in range(3):
                C.check(lib.tdx_plan_launch(ctypes.byref(plan), ws.data_ptr(), stream))
            torch.cuda.synchronize()
            ts = []
            for _ in range(5):
                if mine < (256 << 20):
                    flush.zero_()
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                C.check(lib.tdx_plan_launch(ctypes.byref(plan), ws.data_ptr(), stream))
                e.record()
                e.synchronize()
                ts.append(s.elapsed_time(e))
            ms = sorted(ts)[len(ts) // 2]
            if world > 1:
                t = torch.tensor([ms], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t.item())
            row[name] = {"gbs": round(nbytes / ms / 1e6, 1), "frac_per_gpu": round(nbytes / world / ms / 1e6 / peak, 3)}
        rows.append(row)
        del buf
        nbytes *= 4
    del flush
    torch.cuda.empty_cache()
    return rows


def fsdp2_handoff_check(cx):
    """SURVEY 8f.1, asserted where the driver has >= 2 GPUs: after `fully_shard` on the meta device
    every rank fills the local shards FSDP owns IN PLACE from an InitPlan; the gathered parameters
    must equal the unsharded materialisation bit for bit."""
    import torch
    import torch.distributed as dist
    from torch.distributed.fsdp import fully_shard

    from torchdistx_b200 import parallel
    from torchdistx_b200.deferred_init import deferred_init, materialize_module
    from torchdistx_b200.plan import InitPlan, init_sharded_module

    plan = InitPlan.from_module(deferred_init(build_model, "llama-tiny"))
    with torch.device("meta"):
        model = build_model("llama-tiny")
    for layer in model.model.layers:
        fully_shard(layer)
    fully_shard(model)
    model.to_empty(device=cx.dev)
    torch.manual_seed(77)
    parallel.sync_rng(cx.dev, force=True)
    init_sharded_module(model, plan, cx.rank, cx.world, device=cx.dev)
    got = {n: p.full_tensor() for n, p in model.named_parameters()}
    ref = deferred_init(build_model, "llama-tiny")
    torch.manual_seed(77)
    parallel.sync_rng(cx.dev, force=True)
    materialize_module(ref, device=cx.dev)
    bad = [n for n, p in ref.named_parameters() if not torch.equal(got[n], p.detach())]
    flag = torch.tensor([len(bad)], device=cx.dev)
    dist.all_reduce(flag)
    assert int(flag.item()) == 0, f"FSDP2 hand-off mismatch on {bad[:3]}"
    return "ok: llama-tiny, fully_shard on meta -> init_sharded_module in place -> full_tensor() == unsharded materialize_module, bit for bit"


def run_ours(a):
    import torch
    import torch.distributed as dist

    from torchdistx_b200 import _cabi as C
    from torchdistx_b200 import parallel

    cx = Ctx()
    world = cx.world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = cx.rank = int(os.environ.get("RANK", "0"))
    local = cx.local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback exists)"
    torch.cuda.set_device(local)
    dev = cx.dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == a.gpus, f"--gpus {a.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run)"
    cx.lib = C.load()
    cx.as_rank_of = a.as_rank_of
    cx.stream = torch.cuda.current_stream().cuda_stream
    dtype = MODELS[a.model][2]

    if a.roofline_only:  # for ncu: one materialize, then launches of the dominant kernel's plan only
        measure_model(cx, a.model, a.steps, 0, roofline_only=True)
        return

    torch.manual_seed(1234)
    parallel.sync_rng(dev)  # the one collective: 16 bytes, rank 0 -> all
    main = measure_model(cx, a.model, a.steps, a.warmup, first_call=True, dump_dir=a.dump_outputs)

    # ---- the other BASELINE configs, measured in the same run (smaller step counts) ----------------
    extra = {}
    if not a.no_extra:
        side = []
        if a.model == "llama3-8b":
            side = ["gpt2-xl", "llama3-8b-cast"] if world == 1 else ["llama3-70b"] if world == 8 else []
        for name in side:
            try:
                r = measure_model(cx, name, max(3, a.steps // 2), 3)
                extra[name] = {"params": r["params"], "dtype": r["dtype"], "value": r["params"] / (r["ms"] / 1e3),
                               "ms_per_step": r["ms"], "hbm_gbs_per_gpu": r["my_bytes"] / (r["ms"] / 1e3) / 1e9,
                               "e2e": {"value": r["params"] / (r["e2e_ms"] / 1e3), "ms_per_step": r["e2e_ms"],
                                       "api_return_ms": r["host_split"]["api_return"]},
                               "roofline": r["roofline"], "fused_tensors": r["stats"]["fused_tensors"],
                               "generic_ops": r["stats"]["generic_ops"], "descriptors_per_rank": r["descs"]}
            except Exception as e:  # a side measurement must not cost the headline
                extra[name] = {"error": f"{type(e).__name__}: {str(e)[-300:]}"}
        try:
            extra["kernel_sweep"] = {"what": kernel_sweep.__doc__.split("\n\n")[0].replace("\n    ", " "),
                                     "rows": kernel_sweep(cx, 16 << 30)}
        except Exception as e:
            extra["kernel_sweep"] = {"error": f"{type(e).__name__}: {str(e)[-300:]}"}
        if world > 1:
            try:
                extra["fsdp2_handoff_check"] = fsdp2_handoff_check(cx)
            except Exception as e:
                extra["fsdp2_handoff_check"] = f"FAILED: {type(e).__name__}: {str(e)[-300:]}"

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- baselines on rank 0 at N = 1: the reference on the host cores (bounded sample), and the
    # reference replaying on the GPU with stock ATen kernels (baseline B, whole model) --------------
    cpu = None
    if world == 1 and not a.no_cpu_baseline:
        try:
            layers = sample_layers(a.model)
            res = reference_sample(a.model, layers, 1)
            cpu = {"value": res["params"] / res["times"][0], "unit": "params/s", "cores": res["threads"],
                   "kind": "reference",
                   "sample": f"{a.model} cut to {layers} decoder layer(s)"
                             f"{', vocab ' + str(SAMPLE_VOCAB[a.model]) if a.model in SAMPLE_VOCAB else ''} "
                             f"({res['params']:,} params), {dtype}, device=cpu, 1 repetition, {res['times'][0]:.1f} s"}
        except Exception as e:  # the oracle is test infrastructure: report, do not hide
            cpu = {"value": None, "unit": "params/s", "cores": os.cpu_count(), "kind": "reference",
                   "sample": f"unavailable: {type(e).__name__}: {str(e)[-200:]}"}
        if not a.no_extra:
            try:
                torch.cuda.empty_cache()
                g = reference_on_gpu(a.model, local)
                best = min(g["times"][1:])
                extra["gpu_baseline"] = {"what": "the reference's own engine (oracle/_ref) with the model recorded for cuda: "
                                                 "materialize_module replays every recorded op through stock ATen kernels "
                                                 "(baseline B of SURVEY 8d); wall clock incl. synchronize, best of 2 after a warm-up call",
                                         "model": a.model, "value": g["params"] / best, "unit": "params/s",
                                         "ms_per_step": best * 1e3, "first_call_ms": g["times"][0] * 1e3}
            except Exception as e:
                extra["gpu_baseline"] = {"error": f"{type(e).__name__}: {str(e)[-300:]}"}

    c1, c2, st = main["clk"], main["clk_e2e"], main["stats"]
    ms, e2e_ms, n_params, my_bytes = main["ms"], main["e2e_ms"], main["params"], main["my_bytes"]
    total_bytes = my_bytes * world if world > 1 else my_bytes
    rf = main["roofline"]
    if world == 1 and a.model == "llama3-8b":
        try:  # DRAM bytes of one launch of the dominant kernel, from the committed ncu capture (N = 1 only)
            rf["traffic"] = json.load(open(os.path.join(ROOT, "profiles", "ncu_bench_summary.json"))).get(a.model, {}).get("dram_bytes_per_launch")
        except Exception:
            pass
    rf["secondary_ceiling"] = ("dispatch port: Philox4x32-10 alone is ~74 of the ~120 cycles a 16-byte vector takes "
                               "(benchmarks/philox_rate.cu); see DESIGN.md section 4")
    line = {
        "metric": "materialize_module params/s", "value": n_params / (ms / 1e3), "unit": "params/s",
        "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": dtype, "data": "synthetic (random init of the named architecture, HF config; no checkpoint)",
        "config": {"workload": f"{a.model} deferred_init -> materialize_module on cuda, dim-0 sharded over {world} GPU(s)",
                   "params": n_params, "tensors": main["tensors"], "descriptors_per_rank": main["descs"],
                   "fused_tensors": st["fused_tensors"], "generic_ops": st["generic_ops"],
                   "elided_rng_ops": st["elided_rng_ops"], "record_s_per_model": main["record_s_per_model"],
                   "host_us": {k: round(st[k]) for k in ("traverse_us", "plan_us", "eval_us", "alloc_us", "launch_us", "wrap_us", "assign_us", "first_submit_us", "last_submit_us", "deferred_us", "helper_start_us", "helper_done_us", "submissions", "template_hits")},
                   "e2e_host_split_ms": main["host_split"],
                   "l2": "outputs per step (GBs) exceed the 126 MB L2; no flush needed",
                   "collective": "one 16-byte broadcast of (seed, offset) before the first step; later steps derive their offsets locally (parallel.sync_rng), agreement asserted after the timed region",
                   "timed_region_value": "tdx_plan_launch only (plan resident in HBM)",
                   "timed_region_e2e": "per step: sync_rng + materialize_module (traversal, plan, alloc, H2D descriptors, kernels) + 64 B D2H + sync; model teardown between steps untimed; Python GC collected once before and disabled across the timed steps (as timeit does)"},
        "hbm_gbs": total_bytes / (ms / 1e3) / 1e9, "hbm_gbs_per_gpu": my_bytes / (ms / 1e3) / 1e9,
        "e2e": {"value": n_params / (e2e_ms / 1e3), "unit": "params/s", "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": main["h2d"], "d2h_bytes_per_step": 64,
                "cold_first_call_ms": main.get("e2e_cold_ms"), "cold_first_call_alloc_ms": main.get("cold_alloc_ms"),
                "cold_note": "first materialize_module of the process: CUDA module load + cold caching allocator (one cudaMalloc per submission slab) + pinned staging; every later number is warm"},
        "gpu_launches": main["launches_per_step"] * a.steps,
        "roofline": rf,
        "cpu_baseline": cpu,
        "clocks": {"sm_mhz": c1["sm_mhz"], "sm_max_mhz": c1["sm_max_mhz"], "reasons": c1["reasons"],
                   "e2e_sm_mhz": c2["sm_mhz"], "e2e_reasons": c2["reasons"]},
        "extra": extra,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--model", default="llama3-8b", choices=sorted(MODELS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true",
                    help="skip the side measurements (the other BASELINE configs, the kernel sweep, baseline B)")
    ap.add_argument("--as-rank-of", type=int, default=0,
                    help="diagnostic (N = 1 only): build rank 0's dim-0 shard of a model sharded W ways -- the kernels "
                         "and host path of one rank of an N = W job without W GPUs; the line's params/s are then 1/W of a job's")
    ap.add_argument("--roofline-only", action="store_true",
                    help="for ncu: one materialize (1 launch per family), then 3+steps launches of the "
                         "dominant kernel's plan only; prints nothing")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the materialised model's parameters and buffers to DIR "
                         "as <name>.npy (float32/float64, 64 MB at most; a fixed seeded sample of large tensors)")
    a = ap.parse_args()
    a.warmup = max(a.warmup, 3) if a.impl == "ours" else a.warmup
    if a.impl == "reference":
        run_reference_arm(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
