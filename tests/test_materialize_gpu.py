"""GPU parity, engine level: deferred_init -> materialize_module on cuda through the public API,
against the REAL reference (oracle/_ref, CPU) and against the engine's own invariants.  What the
reference materialised is stored in tests/golden/reference_gpu_cases.pt.gz
(tests/golden/make_reference_outputs.py; format: oracle/golden.py): whole where the program is
deterministic (the same at two seeds), as moments and quantiles where it draws random numbers.

Tiers (SURVEY.md section 8c):
  T0  tensors whose recorded program is deterministic: bit-exact with the reference;
  T1  RNG tensors: same distribution as the reference's CPU sample under the same seed --
      |mean - mean_ref| <= 5 sigma sqrt(2/N), |std/std_ref - 1| <= 5/sqrt(N) (+2^-8 for bf16 vs the
      reference's bf16 path, which draws its normals from 8-bit uniforms:
      $TORCH/include/ATen/native/cpu/DistributionTemplates.h:207-256 with
      $TORCH/include/ATen/core/TransformationHelper.h:84-99 digits = 8), hard range checks,
      two-sample KS at alpha = 1e-4 on tensors >= 4096 elements (against the reference's sample
      rebuilt from 512 quantiles), no NaN/Inf;
  T2  exact self-consistency: same seed -> same bits, other seed -> other bits, shards
      concatenate to the unsharded tensor, dead-pass elision == explicit offset skip, the torch
      generator is advanced.
"""
import math

import numpy as np
import pytest
import torch
from torch import nn

from oracle import cases
from oracle import golden
from oracle import tdx_oracle as O
from torchdistx_b200.deferred_init import (deferred_init, is_deferred, last_materialize_stats,
                                           materialize_module, materialize_tensor)
from torchdistx_b200.fake import is_fake

pytestmark = pytest.mark.gpu
CASES = [("init_zoo", "fp32"), ("init_zoo", "bf16"), ("tiny_llama", "fp32"), ("tiny_llama", "bf16"),
         ("tiny_gpt2", "fp32"), ("mlp_stack", "fp32"), ("torch_transformer", "fp32"), ("clones", "fp32"), ("cast_variant", "fp32")]


@pytest.fixture(scope="module")
def reference():
    """The real reference, CPU device, seed 5: a tensor (deterministic program: equal at seeds 5 and 6)
    or its `golden.summary` (RNG program), per case."""
    ref = golden.load("reference_gpu_cases")
    return {(c, t): ref[f"{c}_{t}"] for c, t in CASES}


def build_on_cuda(case, dtype, seed=5, **kw):
    torch.set_default_dtype(cases.DTYPES[dtype])
    try:
        m = deferred_init(lambda: cases.build(case, dtype, "cuda"))
    finally:
        torch.set_default_dtype(torch.float32)
    assert is_deferred(m)
    torch.manual_seed(seed)
    materialize_module(m, **kw)
    return m


def named_tensors(m):
    return dict(list(m.named_parameters()) + list(m.named_buffers()))


@pytest.mark.parametrize("case,dtype", CASES)
def test_t0_t1_against_reference(case, dtype, reference):
    from scipy import stats

    ref = reference[(case, dtype)]
    m = build_on_cuda(case, dtype)
    st = last_materialize_stats()
    mine = named_tensors(m)
    assert set(mine) <= set(ref)
    n_rng = 0
    for k, t in mine.items():
        r = ref[k]
        r_dtype, r_shape = (r["dtype"], r["shape"]) if isinstance(r, dict) else (str(r.dtype), tuple(r.shape))
        assert t.is_cuda and not is_fake(t) and str(t.dtype) == r_dtype and tuple(t.shape) == r_shape, k
        assert isinstance(t, nn.Parameter) == (k in dict(m.named_parameters())), k
        x = t.detach().cpu()
        if not isinstance(r, dict):  # T0: deterministic program
            assert torch.equal(x, r), k
            continue
        n_rng += 1  # T1
        xf = x.double().flatten()
        n = xf.numel()
        assert torch.isfinite(xf).all(), k
        sd = r["std"]
        slack = 2 ** -8 if dtype == "bf16" else 0.0
        assert abs(xf.mean().item() - r["mean"]) <= 5 * sd * math.sqrt(2 / n) + slack * sd, k
        assert abs(xf.std().item() / sd - 1) <= 5 / math.sqrt(n) + 4 * slack, k
        lo, hi = r["min"], r["max"]
        span = hi - lo
        assert xf.min().item() >= lo - 0.5 * span and xf.max().item() <= hi + 0.5 * span, k
        if n >= 4096 and dtype == "fp32":
            assert stats.ks_2samp(xf.numpy(), golden.expand(r["quantiles"], n)).pvalue > 1e-4, k
    assert n_rng > 0
    # everything large went through the fused path
    fused_bytes = st["bytes_written"]
    total = sum(t.numel() * t.element_size() for t in mine.values())
    assert fused_bytes >= 0.95 * total, (st, total)


def test_t1_bf16_against_fp32_reference_distribution(reference):
    """The reference's own bf16 CPU normal is coarse (8-bit uniforms); the engine's bf16 output is
    checked against the reference's fp32 sample of the same program instead."""
    from scipy import stats

    ref = reference[("tiny_llama", "fp32")]
    m = build_on_cuda("tiny_llama", "bf16")
    for k, t in named_tensors(m).items():
        r = ref[k]
        if not isinstance(r, dict) or r["numel"] < 4096:  # (deterministic programs have std 0)
            continue
        x = t.detach().double().flatten().cpu()
        rb = torch.from_numpy(golden.expand(r["quantiles"], r["numel"])).to(torch.bfloat16).double()  # same rounding grid
        assert stats.ks_2samp(x.numpy(), rb.numpy()).pvalue > 1e-4, k
        assert abs(x.std().item() / r["std"] - 1) <= 5 / math.sqrt(r["numel"]) + 2 ** -9, k


def test_t2_determinism_seed_and_generator_advance():
    a = named_tensors(build_on_cuda("tiny_llama", "bf16", seed=11))
    off_after = torch.cuda.default_generators[0].get_offset()
    b = named_tensors(build_on_cuda("tiny_llama", "bf16", seed=11))
    c = named_tensors(build_on_cuda("tiny_llama", "bf16", seed=12))
    assert off_after > 0 and off_after % 4 == 0
    for k in a:
        assert torch.equal(a[k], b[k]), k
    w = "model.layers.0.mlp.up_proj.weight"
    assert (a[w] != c[w]).float().mean() > 0.9
    # later torch RNG does not replay our stream
    torch.manual_seed(11)
    m = build_on_cuda("mlp_stack", "fp32", seed=11)
    x = torch.randn(4096, device="cuda")
    assert not torch.equal(x, named_tensors(m)["0.weight"].flatten()[:4096])


@pytest.mark.parametrize("world", [2, 4, 8])
def test_t2_dim0_shards_concatenate_bit_exact(world):
    full = named_tensors(build_on_cuda("tiny_llama", "bf16", seed=3))
    params = dict(build_on_cuda("tiny_llama", "bf16", seed=3).named_parameters()).keys()
    shards = [named_tensors(build_on_cuda("tiny_llama", "bf16", seed=3, shard=(r, world))) for r in range(world)]
    for k, t in full.items():
        if k in params and t.dim() > 0:
            assert shards[0][k].shape[0] == -(-t.shape[0] // world)
            assert torch.equal(torch.cat([s[k] for s in shards], 0), t), k
        else:  # buffers are replicated
            for s in shards:
                assert torch.equal(s[k], t), k
    assert sum(s["lm_head.weight"].numel() for s in shards) == full["lm_head.weight"].numel()


def test_t2_ragged_shards_match_torch_chunk():
    class Odd(nn.Module):
        def __init__(self):
            super().__init__()
            self.w = nn.Parameter(torch.empty(10, 7, device="cuda").normal_())
            self.v = nn.Parameter(torch.empty(3, device="cuda").uniform_())
            self.s = nn.Parameter(torch.zeros((), device="cuda"))

    def build(**kw):
        m = deferred_init(Odd)
        torch.manual_seed(1)
        materialize_module(m, **kw)
        return m

    full = build()
    for world in (3, 4, 8):
        for r in range(world):
            s = build(shard=(r, world))
            for name in ("w", "v"):
                chunks = torch.chunk(getattr(full, name).detach(), world, 0)
                exp = chunks[r] if r < len(chunks) else getattr(full, name).detach()[:0]
                assert torch.equal(getattr(s, name).detach(), exp), (name, world, r)
            assert torch.equal(s.s, full.s)


def test_t2_dead_pass_elision_equals_explicit_offset_skip():
    n = 64 * 48

    def double_init():
        lin = nn.Linear(48, 64, bias=False, device="cuda")  # records uniform_ (dead) ...
        nn.init.normal_(lin.weight, 0.0, 0.02)  # ... then normal_ (live)
        return lin

    def single_init():
        return nn.Parameter(torch.empty(64, 48, device="cuda").normal_(0.0, 0.02))

    m = deferred_init(double_init)
    torch.manual_seed(21)
    materialize_module(m)
    st = last_materialize_stats()
    assert st["elided_rng_ops"] == 1 and st["fused_tensors"] == 1 and st["kernel_launches"] == 1
    p = deferred_init(single_init)
    torch.manual_seed(21)
    g = torch.cuda.default_generators[0]
    g.set_offset(g.get_offset() + O.offset_increment(n))  # what the dead uniform_ consumed
    assert torch.equal(materialize_tensor(p), m.weight)


def test_device_override_builds_cpu_recordings_on_cuda(reference):
    torch.set_default_dtype(torch.float32)
    m = deferred_init(lambda: cases.build("init_zoo", "fp32", "cpu"))
    assert m.kaiming.weight.device.type == "cpu"
    was_fake = {k for k, t in named_tensors(m).items() if is_fake(t)}
    # torch.tensor(0) (BatchNorm.num_batches_tracked) is never intercepted: a real tensor stays as it is
    assert "bn.num_batches_tracked" not in was_fake
    torch.manual_seed(5)
    materialize_module(m, device="cuda")
    ref = reference[("init_zoo", "fp32")]
    for k, t in named_tensors(m).items():
        assert t.is_cuda == (k in was_fake), k
        if not isinstance(ref[k], dict):
            assert torch.equal(t.detach().cpu(), ref[k]), k
    # and the same recording built on cuda directly gives the same bits
    m2 = build_on_cuda("init_zoo", "fp32", seed=5)
    for k, t in named_tensors(m).items():
        assert torch.equal(t.cpu(), named_tensors(m2)[k].cpu()), k


def test_identity_class_and_requires_grad_on_cuda():
    m = deferred_init(lambda: nn.Linear(8, 8, device="cuda"))
    w = materialize_tensor(m.weight)
    assert materialize_tensor(m.weight) is w and isinstance(w, nn.Parameter) and w.requires_grad
    materialize_module(m)
    assert m.weight is w and not is_deferred(m)


def test_generic_replay_on_cuda_for_unfusable_programs():
    def build():
        a = torch.randn(16, 16, device="cuda")
        return nn.Parameter(a @ a.t())  # not an init pattern: replayed by ATen on the GPU

    p = deferred_init(build)
    out = materialize_tensor(p)
    st = last_materialize_stats()
    # (the randn operand folds: dependencies of a generic replay are built by the kernels too)
    assert out.is_cuda and st["generic_ops"] >= 2 and st["fused_tensors"] == 1
    assert torch.allclose(out, out.t())


def test_generic_replay_reads_a_fused_tensor_that_is_still_in_the_batch():
    """Unfusable buffers no longer force a submission of the pending fused descriptors -- unless the
    replayed program reads one of them; then the batch must reach the stream first."""
    class M(nn.Module):
        def __init__(self):
            super().__init__()
            self.w = nn.Parameter(torch.full((1 << 12,), 0.5, device="cuda"))           # fused, pending
            self.u = nn.Parameter(torch.empty(1 << 12, device="cuda").uniform_(1, 2))   # fused, pending
            self.register_buffer("cs", torch.cumsum(self.w.detach() * 2, 0))            # generic, reads w
            self.register_buffer("iv", 1.0 / torch.arange(1, 9, device="cuda"))         # generic, independent
            self.register_buffer("us", torch.sort(self.u.detach())[0])                  # generic, reads u

    m = deferred_init(M)
    materialize_module(m)
    st = last_materialize_stats()
    assert st["fused_tensors"] >= 2 and st["generic_ops"] >= 3  # (w, u; `w * 2` folds to a constant fill as well)
    assert torch.equal(m.cs, torch.arange(1, (1 << 12) + 1, device="cuda", dtype=torch.float32))
    assert torch.equal(m.iv, 1.0 / torch.arange(1, 9, device="cuda"))
    assert torch.equal(m.us, torch.sort(m.u.detach())[0]) and float(m.us[0]) >= 1.0 and float(m.us[-1]) < 2.0


def test_cfg1_linear128_on_cpu_still_bit_exact_with_cuda_present():
    torch.manual_seed(0)
    m = deferred_init(nn.Linear, 128, 128)
    torch.manual_seed(0)
    materialize_module(m)
    torch.manual_seed(0)
    e = nn.Linear(128, 128)
    assert torch.equal(m.weight, e.weight) and torch.equal(m.bias, e.bias)


def test_clones_of_rng_tensors_are_bit_identical_to_their_source():
    m = build_on_cuda("clones", "fp32", seed=9)
    st = last_materialize_stats()
    assert st["fused_tensors"] == 4 and st["generic_ops"] == 0
    assert torch.equal(m.a, m.b) and torch.equal(m.a, m.c)
    assert torch.equal(m.d, m.a * 2.0)
    assert m.a.data_ptr() != m.b.data_ptr()


def test_cast_of_an_rng_tensor_equals_the_cast_of_its_materialised_source():
    """`.to(bf16)` / `.half()` after an fp32 init is fused with the fp32 stream (TDX_ALGO_WIDE32):
    the 16-bit tensor IS the rounded fp32 tensor, bit for bit, when both are kept."""
    m = build_on_cuda("cast_variant", "fp32", seed=4)
    st = last_materialize_stats()
    assert st["generic_ops"] == 0 and st["fused_tensors"] == len(list(m.parameters()))
    assert m.b.dtype == torch.bfloat16 and torch.equal(m.b, m.a.to(torch.bfloat16))
    assert m.v.dtype == torch.float16 and torch.equal(m.v, m.u.to(torch.float16))
    assert m.body[0].weight.dtype == torch.bfloat16 and m.head.weight.dtype == torch.float16
    w = m.head.weight.float()
    assert w.min() >= -0.05 and w.max() <= 0.05 and 0.012 < w.std() < 0.025
    # steps before the cast run in fp32, the cast rounds once, later steps round to bf16 one by one
    assert m.w.dtype == torch.bfloat16
    assert torch.equal(m.w, m.a.detach().to(torch.bfloat16).mul_(3.0).add_(1.0))


def test_fused_constant_folding_equals_generic_replay_on_random_programs():
    """Deterministic programs drawn at random (factories, fills, scalar arithmetic, clamps, casts,
    clones, aliases): the fused path (constants folded through ATen on a 1-element tensor, one fill
    kernel) must equal op-by-op ATen replay on the GPU bit for bit."""
    import random

    from torchdistx_b200 import _C

    rng = random.Random(1234)
    dtypes = [torch.float32, torch.bfloat16, torch.float16, torch.float64, torch.int64, torch.int32, torch.bool]

    def program(seed):
        r = random.Random(seed)
        dt = r.choice(dtypes)
        shape = r.choice([(7,), (33, 5), (4, 3, 2), (1,), (257,)])
        steps = []
        kind = r.choice(["zeros", "ones", "full", "empty_fill"])
        for _ in range(r.randrange(0, 5)):
            if dt in (torch.bool,):
                steps.append(r.choice(["clone", "view", "detach"]))
            elif dt in (torch.int64, torch.int32):
                steps.append(r.choice([("mul_", r.randrange(-3, 4)), ("add_", r.randrange(-5, 6)), "clone", "view",
                                       ("clamp_", -4, 9), ("to", torch.float32), ("to", torch.int64)]))
            else:
                steps.append(r.choice([("mul_", r.uniform(-2, 2)), ("add_", r.uniform(-1, 1)), ("mul", 1.5), ("add", -0.25),
                                       "clone", "view", "detach", ("clamp_", -0.5, 0.75), ("fill_", r.uniform(-3, 3)),
                                       "zero_", ("to", r.choice([torch.float32, torch.bfloat16, torch.float16]))]))

        def build():
            if kind == "zeros":
                t = torch.zeros(shape, dtype=dt, device="cuda")
            elif kind == "ones":
                t = torch.ones(shape, dtype=dt, device="cuda")
            elif kind == "full":
                t = torch.full(shape, True if dt == torch.bool else 3, dtype=dt, device="cuda")
            else:
                t = torch.empty(shape, dtype=dt, device="cuda").fill_(True if dt == torch.bool else 2)
            for s in steps:
                if s == "clone":
                    t = t.clone()
                elif s == "view":
                    t = t.view(-1).view(shape)
                elif s == "detach":
                    t = t.detach()
                elif s == "zero_":
                    t.zero_()
                elif s[0] == "to":
                    t = t.to(s[1])
                elif s[0] in ("mul_", "add_", "fill_"):
                    getattr(t, s[0])(s[1])
                elif s[0] in ("mul", "add"):
                    t = getattr(t, s[0])(s[1])
                elif s[0] == "clamp_":
                    t.clamp_(s[1], s[2])
            return t

        return build

    fused_count = 0
    for i in range(60):
        build = program(rng.randrange(1 << 30))
        a = _C.materialize_tensor(deferred_init(build), None, None, True)
        fused_count += last_materialize_stats()["fused_tensors"]
        b = _C.materialize_tensor(deferred_init(build), None, None, False)
        assert last_materialize_stats()["fused_tensors"] == 0
        assert a.dtype == b.dtype and a.shape == b.shape, i
        assert torch.equal(a.reshape(-1).view(torch.uint8), b.reshape(-1).view(torch.uint8)), (i, a.dtype)
    assert fused_count >= 50  # nearly all of these programs fold
