"""GPU tests of the round-2 engine work: analysis cached on the recording, slab-backed outputs with
storages of their own, partial writes through views (padding_idx), sharding vs cached values,
cross-recording dependencies, InitPlan with clones."""
import copy
import os
import subprocess
import sys

import pytest
import torch
from torch import nn

from oracle import cases
from oracle import golden
from torchdistx_b200.deferred_init import (deferred_init, is_deferred, last_materialize_stats, materialize_module,
                                           materialize_tensor)
from torchdistx_b200.plan import InitPlan

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def named(m):
    return dict(list(m.named_parameters()) + list(m.named_buffers()))


def bits(t):
    return t.detach().contiguous().reshape(-1).view(torch.uint8)


# ---- analysis at the end of the recording ------------------------------------------------------
def test_templates_serve_every_fused_tensor_and_change_nothing():
    def build():
        return deferred_init(lambda: cases.build("tiny_llama", "bf16", "cuda"))

    torch.manual_seed(3)
    m = build()
    materialize_module(m)
    st = last_materialize_stats()
    assert st["fused_tensors"] > 0 and st["template_hits"] >= st["fused_tensors"], st
    import os
    if os.environ.get("TDX_HOST_THREADS", "1") != "0":
        # the walking thread built the outputs ahead of the planner, which adopted every one of them
        assert st["prebuilt_outputs"] == st["fused_tensors"], st
    assert st["generic_ops"] == 0  # rotary inv_freq is an index program (TDX_SRC_IOTA + 4 epilogue steps) now
    # the same module through the uncached route (materialize_tensor on a recording whose templates
    # do not cover constant folding: `init_zoo.const`) and through generic replay: same bits
    torch.manual_seed(3)
    m2 = build()
    for k, t in named(m2).items():
        owner, _, key = k.rpartition(".")
        mod = m2.get_submodule(owner) if owner else m2
        (mod._parameters if key in mod._parameters else mod._buffers)[key] = materialize_tensor(t)
    a, b = named(m), named(m2)
    # (materialize order differs: module order vs named order are the same traversal here)
    for k in a:
        assert torch.equal(bits(a[k]), bits(b[k])), k


# ---- slab-backed outputs -------------------------------------------------------------------------
def test_outputs_share_a_slab_but_own_their_storages():
    from torchdistx_b200 import _C

    m = deferred_init(lambda: cases.build("mlp_stack", "fp32", "cuda"))
    torch.manual_seed(0)
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    materialize_module(m)
    ts = list(named(m).values())
    nbytes = sum(t.numel() * t.element_size() for t in ts)
    assert before + nbytes <= torch.cuda.memory_allocated() <= before + nbytes + 256 * len(ts) + (1 << 20)
    storages = {t.untyped_storage()._cdata for t in ts}
    assert len(storages) == len(ts)  # no two tensors share a StorageImpl
    for t in ts:
        assert t.untyped_storage().nbytes() == t.numel() * t.element_size()
        assert t.data_ptr() % 256 == 0 and t.is_contiguous()
    # the tensors do not overlap
    spans = sorted((t.data_ptr(), t.data_ptr() + t.numel() * t.element_size()) for t in ts)
    assert all(spans[i][1] <= spans[i + 1][0] for i in range(len(spans) - 1))
    # memory goes back when the last tensor of the slab dies (and the recording, which also names
    # the tensors, has been let go of on the helper thread)
    del m, ts, t  # (`t`: the loop variable above still names the last tensor)
    _C._drain()
    torch.cuda.synchronize()
    assert torch.cuda.memory_allocated() <= before + (1 << 16)

    # usable like any tensor: autograd, save/load, storage resize
    m = deferred_init(lambda: cases.build("mlp_stack", "fp32", "cuda"))
    materialize_module(m)
    y = m(torch.randn(3, 64, device="cuda"))
    y.sum().backward()
    assert all(p.grad is not None for p in m.parameters())
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    import io
    buf = io.BytesIO()
    torch.save(m.state_dict(), buf)
    assert buf.getbuffer().nbytes < 2 * sum(v.numel() * v.element_size() for v in sd.values()) + (1 << 16)
    buf.seek(0)
    back = torch.load(buf)
    assert all(torch.equal(back[k], sd[k]) for k in sd)
    w = next(m.parameters())
    keep = w.detach().clone()
    w.untyped_storage().resize_(w.untyped_storage().nbytes() * 2)  # re-allocates through the caching allocator
    assert torch.equal(w.detach(), keep)


def test_per_tensor_allocation_switch(tmp_path):
    code = ("import torch, sys; sys.path.insert(0, %r)\n"
            "from oracle import cases\n"
            "from torchdistx_b200.deferred_init import deferred_init, materialize_module\n"
            "m = deferred_init(lambda: cases.build('mlp_stack', 'fp32', 'cuda'))\n"
            "torch.manual_seed(0); materialize_module(m)\n"
            "from torchdistx_b200 import _C; _C._drain()\n"
            "w = m[0].weight; before = torch.cuda.memory_allocated()\n"
            "m[0]._parameters['weight'] = None; del w\n"
            "assert torch.cuda.memory_allocated() < before, 'freeing one tensor must release its memory'\n"
            "print('ok')\n" % ROOT)
    env = dict(os.environ, TDX_SLAB="0")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=ROOT, timeout=300)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


# ---- partial writes through views ----------------------------------------------------------------
@pytest.fixture(scope="module")
def padded_reference():
    """The real reference, fp32, seed 5 (tests/golden/make_reference_outputs.py): per weight its padded
    row and the `golden.summary` of the other rows."""
    return golden.load("reference_gpu_cases")["padded_embeddings_fp32"]


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_padding_idx_embeddings_fuse_and_match_the_reference(dtype, padded_reference):
    import math

    m = deferred_init(lambda: cases.build("padded_embeddings", dtype, "cuda"))
    torch.manual_seed(5)
    materialize_module(m)
    st = last_materialize_stats()
    assert st["generic_ops"] == 0 and st["fused_tensors"] == 4, st
    assert st["descriptors"] == 3 + 2 + 2 + 3, st
    ref = padded_reference
    # the padded rows: bit-exact zeros (T0); everything else: the reference's distribution (T1)
    for name, row in (("torch_style", 3), ("hf_style", 0), ("last_row", 256)):
        w = getattr(m, name).weight.detach()
        r_row, rr = ref[f"{name}.weight"]["padded_row"], ref[f"{name}.weight"]["rest"]
        assert torch.equal(w[row].cpu(), torch.zeros_like(r_row, dtype=w.dtype)) and torch.equal(r_row, torch.zeros_like(r_row))
        rest = torch.cat([w[:row], w[row + 1:]]).double().flatten()
        n = rest.numel()
        assert n == rr["numel"]
        assert (rest != 0).float().mean().item() > 0.99
        slack = 2.0 ** -8 if dtype == "bf16" else 0.0
        assert abs(rest.mean().item() - rr["mean"]) <= 5 * rr["std"] / math.sqrt(n), name
        assert abs(rest.std().item() / rr["std"] - 1) <= 5 / math.sqrt(2 * n) + slack, name
    h = m.halves.detach().float().cpu()
    assert torch.equal(h[32:], torch.full((32, 32), 0.5))
    assert abs(h[:16].std().item() / 0.2 - 1) < 0.15 and abs(h[16:32].std().item() / 0.1 - 1) < 0.15


def test_padding_idx_shards_concatenate_to_the_unsharded_tensor():
    def build(shard):
        m = deferred_init(lambda: cases.build("padded_embeddings", "bf16", "cuda"))
        torch.manual_seed(9)
        materialize_module(m, shard=shard)
        return named(m)

    full = build(None)
    for world in (2, 3, 8):
        parts = [build((r, world)) for r in range(world)]
        for k, t in full.items():
            chunks = [p[k] for p in parts if p[k].numel()]
            assert torch.equal(bits(torch.cat(chunks)), bits(t)), (k, world)


# ---- sharding and values cached on the recording (ADVICE r1) ------------------------------------------
class BufferFromParam(nn.Module):
    def __init__(self):
        super().__init__()
        self.w = nn.Parameter(torch.empty(16, 8).normal_(0.0, 0.5))
        self.register_buffer("b", torch.sin(self.w.detach()) + 1.0)  # a generic reader of the parameter


def test_buffer_computed_from_a_sharded_parameter_sees_the_whole_parameter():
    def build():
        return deferred_init(lambda: _on_cuda(BufferFromParam))

    torch.manual_seed(21)
    full = build()
    materialize_module(full)
    for rank in range(2):
        torch.manual_seed(21)
        m = build()
        materialize_module(m, shard=(rank, 2))  # parameter first (a chunk), then the buffer that reads all of it
        assert torch.equal(m.w.detach(), torch.chunk(full.w.detach(), 2, 0)[rank])
        assert torch.equal(m.b, full.b)
    # the other order: the buffer's dependency materialises the parameter whole, the sharded call chunks it
    torch.manual_seed(21)
    m = build()
    materialize_module(m, buffers_only=True)
    assert torch.equal(m.b, full.b) and is_deferred(m.w)
    materialize_module(m, shard=(1, 2))
    assert torch.equal(m.w.detach(), torch.chunk(full.w.detach(), 2, 0)[1])


def _on_cuda(cls):
    with torch.device("cuda:0"):
        return cls()


# ---- a generic op reading a fused tensor of an EARLIER recording (ADVICE r1) ---------------------------
def test_cross_recording_dependency_sees_initialised_memory():
    torch.manual_seed(4)
    m1 = deferred_init(lambda: _on_cuda(lambda: nn.Linear(64, 64)))
    scale = torch.arange(64, dtype=torch.float32, device="cuda:0")  # a real, non-scalar operand: generic op

    class Derived(nn.Module):
        def __init__(self):
            super().__init__()
            self.v = nn.Parameter((m1.weight.detach() * scale).clone())

    m2 = deferred_init(Derived)
    materialize_module(m2)  # materialises m1.weight (fused, pending in the batch) and multiplies it
    w1 = materialize_tensor(m1.weight)
    assert torch.equal(m2.v.detach(), w1.detach() * scale)
    assert w1.detach().abs().max().item() > 0


# ---- InitPlan and clones (ADVICE r1) -------------------------------------------------------------------
def test_plan_reproduces_modules_with_deepcopied_layers(tmp_path):
    def build():
        def fn():
            with torch.device("cuda"):
                layer = nn.Linear(32, 32)
                return nn.ModuleList([layer, copy.deepcopy(layer), nn.TransformerEncoder(
                    nn.TransformerEncoderLayer(32, 4, 64), num_layers=2, enable_nested_tensor=False)])
        return deferred_init(fn)

    plan = InitPlan.from_module(build())
    plan.save(str(tmp_path / "p.json"))
    torch.manual_seed(8)
    got = InitPlan.load(str(tmp_path / "p.json")).materialize(device="cuda")
    off_plan = torch.cuda.default_generators[0].get_offset()
    m = build()
    torch.manual_seed(8)
    materialize_module(m)
    assert off_plan == torch.cuda.default_generators[0].get_offset()
    for k, t in named(m).items():
        assert torch.equal(bits(got[k]), bits(t)), k
    assert torch.equal(m[0].weight, m[1].weight)  # deepcopy semantics: the copy equals its source


def test_plan_with_segments_round_trips(tmp_path):
    m = deferred_init(lambda: cases.build("padded_embeddings", "bf16", "cuda"))
    plan = InitPlan.from_module(m)
    plan.save(str(tmp_path / "p.json"))
    for shard in (None, (1, 3)):
        torch.manual_seed(2)
        got = InitPlan.load(str(tmp_path / "p.json")).materialize(device="cuda", shard=shard)
        m2 = deferred_init(lambda: cases.build("padded_embeddings", "bf16", "cuda"))
        torch.manual_seed(2)
        materialize_module(m2, shard=shard)
        for k, t in named(m2).items():
            assert torch.equal(bits(got[k]), bits(t)), (k, shard)


def test_plan_build_leaves_the_generators_alone():
    m = deferred_init(lambda: cases.build("tiny_llama", "bf16", "cuda"))  # inv_freq is embedded by value
    torch.manual_seed(77)
    s_cpu, s_cuda = torch.get_rng_state(), torch.cuda.get_rng_state()
    InitPlan.from_module(m)
    assert torch.equal(torch.get_rng_state(), s_cpu) and torch.equal(torch.cuda.get_rng_state(), s_cuda)


# ---- FSDP1 flat-parameter layout (SURVEY 8e) ---------------------------------------------------------
@pytest.mark.parametrize("world,align", [(1, 0), (2, 0), (3, 8), (8, 8)])
def test_flat_shard_equals_chunks_of_the_flattened_module(world, align):
    from torchdistx_b200.deferred_init import materialize_flat_shard

    def build():
        return deferred_init(lambda: cases.build("padded_embeddings", "bf16", "cuda:0"))

    torch.manual_seed(31)
    full = build()
    full_params = [materialize_tensor(p) for p in full.parameters()]  # (the order FSDP flattens in: parameters())
    flat_parts, offsets, total = [], [], 0
    for p in full_params:
        if align > 1 and total % align:
            pad = align - total % align
            flat_parts.append(torch.zeros(pad, dtype=p.dtype, device=p.device))
            total += pad
        offsets.append(total)
        flat_parts.append(p.detach().flatten())
        total += p.numel()
    flat = torch.cat(flat_parts)
    chunk = -(-total // world)
    padded = torch.cat([flat, torch.zeros(chunk * world - total, dtype=flat.dtype, device=flat.device)])
    off_end = torch.cuda.default_generators[0].get_offset()
    for rank in range(world):
        torch.manual_seed(31)
        m = build()
        shard, offs = materialize_flat_shard(list(m.parameters()), rank, world, align_numel=align)
        assert offs == offsets + [total]
        assert shard.shape == (chunk,) and torch.equal(bits(shard), bits(padded[rank * chunk:(rank + 1) * chunk])), rank
        assert torch.cuda.default_generators[0].get_offset() == off_end  # every rank consumed the same offsets
        assert all(is_deferred(p) for p in m.parameters())
    # into a caller-owned buffer (FSDP's flat_param._local_shard)
    torch.manual_seed(31)
    m = build()
    buf = torch.full((chunk + 5,), 7.0, dtype=torch.bfloat16, device="cuda:0")
    shard, _ = materialize_flat_shard(list(m.parameters()), world - 1, world, align_numel=align, out=buf)
    assert shard.data_ptr() == buf.data_ptr()
    assert torch.equal(bits(buf[:chunk]), bits(padded[(world - 1) * chunk:])) and bool((buf[chunk:] == 7.0).all())


def test_flat_shard_with_an_unfusable_parameter_falls_back_to_replay_and_copy():
    from torchdistx_b200.deferred_init import materialize_flat_shard

    class M(nn.Module):
        def __init__(self):
            super().__init__()
            self.a = nn.Parameter(torch.empty(33, 7).normal_())
            self.b = nn.Parameter(torch.sin(torch.arange(40, dtype=torch.float32)))  # generic program
            self.c = nn.Parameter(torch.full((5,), 2.0))

    def build():
        return deferred_init(lambda: _on_cuda(M))

    torch.manual_seed(1)
    full = build()
    flat = torch.cat([materialize_tensor(p).detach().flatten() for p in full.parameters()])
    chunk = -(-flat.numel() // 2)
    padded = torch.cat([flat, flat.new_zeros(2 * chunk - flat.numel())])
    for rank in range(2):
        torch.manual_seed(1)
        shard, _ = materialize_flat_shard(list(build().parameters()), rank, 2)
        assert torch.equal(shard, padded[rank * chunk:(rank + 1) * chunk])


# ---- index programs (SURVEY 8f.2): arange and what models build on it --------------------------------
def test_rotary_inv_freq_is_one_descriptor_and_equals_the_aten_replay():
    from torchdistx_b200 import _C

    def build():
        return deferred_init(lambda: cases.build("tiny_llama", "bf16", "cuda:0"))

    m = build()
    materialize_module(m)
    st = last_materialize_stats()
    assert st["generic_ops"] == 0 and st["fused_tensors"] == st["tensors"], st
    g = build()
    _C.materialize_module(g, False, None, None, None, False)  # fused=False: every op replayed by ATen on the GPU
    assert last_materialize_stats()["fused_tensors"] == 0
    for name in ("model.rotary_emb.inv_freq", "model.rotary_emb.original_inv_freq"):
        a, b = named(m)[name], named(g)[name]
        assert a.dtype == b.dtype == torch.float32 and a.shape == b.shape
        # same arithmetic as ATen's CUDA kernels (x * (1/dim), powf, 1/x): bit for bit
        assert torch.equal(a, b), (name, (a - b).abs().max().item())


def test_rotary_buffers_of_a_model_converted_to_bf16_fuse_and_equal_the_aten_replay():
    """BASELINE cfg 3's `.to(torch.bfloat16)` variant: Module.to converts the rotary buffers as well.
    One 16-bit iota descriptor each; bit for bit what ATen's CUDA kernels give op by op."""
    from torchdistx_b200 import _C

    def build():
        return deferred_init(lambda: cases.build("tiny_llama", "fp32", "cuda:0").to(torch.bfloat16))

    m = build()
    materialize_module(m)
    st = last_materialize_stats()
    assert st["generic_ops"] == 0 and st["fused_tensors"] == st["tensors"], st
    g = build()
    _C.materialize_module(g, False, None, None, None, False)  # fused=False: every op replayed by ATen on the GPU
    for name in ("model.rotary_emb.inv_freq", "model.rotary_emb.original_inv_freq"):
        a, b = named(m)[name], named(g)[name]
        assert a.dtype == b.dtype == torch.bfloat16 and a.shape == b.shape
        assert torch.equal(a, b), (name, (a.float() - b.float()).abs().max().item())


def test_iota_descriptors_through_the_c_abi():
    import numpy as np

    from oracle import tdx_oracle as O
    from torchdistx_b200 import _cabi as C

    lib = C.load()
    n = 5000
    ws = torch.empty(lib.tdx_init_workspace_bytes(4), dtype=torch.uint8, device="cuda")
    ids = torch.empty(n, dtype=torch.int64, device="cuda")
    half = torch.empty(n - 7, dtype=torch.int64, device="cuda")
    freq = torch.empty(n, dtype=torch.float32, device="cuda")
    epi = [(C.TDX_EPI_MUL, 1.0 / 128), (C.TDX_EPI_RPOW, 500000.0), (C.TDX_EPI_RECIP, 0.0), (C.TDX_EPI_MUL, 1.0)]
    descs = [C.make_desc(ids.data_ptr(), dtype=C.TDX_I64, src=C.TDX_SRC_IOTA, elem_count=n, p0=3, p1=-2),
             C.make_desc(half.data_ptr(), dtype=C.TDX_I64, src=C.TDX_SRC_IOTA, elem_begin=7, elem_count=n - 7, p0=3, p1=-2),
             C.make_desc(freq.data_ptr(), dtype=C.TDX_F32, src=C.TDX_SRC_IOTA, elem_count=n, p0=0, p1=2, epi=epi)]
    C.launch(descs, ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert torch.equal(ids.cpu(), 3 - 2 * torch.arange(n)) and torch.equal(half, ids[7:])
    assert np.array_equal(O.generate(descs[0]).view(np.int64), ids.cpu().numpy())
    # against ATen's CUDA kernels: the same program, op by op
    x = torch.arange(0, 2 * n, 2, dtype=torch.int64, device="cuda").to(torch.float32) / 128
    ref = (1.0 / (500000.0 ** x)) * 1.0
    assert torch.equal(freq, ref), (freq - ref).abs().max().item()
    # against the CPU restatement: libm's powf and CUDA's agree to a couple of ulp, not bit for bit
    exp = torch.from_numpy(O.generate(descs[2]).view(np.float32).copy())
    torch.testing.assert_close(freq.cpu(), exp, rtol=4 * 2.0 ** -23, atol=1e-45)
    # 16-bit outputs: the fp32 program rounded once at the store == `freq.to(dtype)`, in the iota kernel
    # and in the table kernel's work list alike
    for dt, tdt in ((C.TDX_BF16, torch.bfloat16), (C.TDX_F16, torch.float16)):
        out = torch.empty(n - 3, dtype=tdt, device="cuda")
        d16 = C.make_desc(out.data_ptr(), dtype=dt, src=C.TDX_SRC_IOTA, elem_begin=3, elem_count=n - 3, p0=0, p1=2, epi=epi)
        C.launch([d16], ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert torch.equal(out, freq[3:].to(tdt))
    big = torch.empty(1 << 26, dtype=torch.bfloat16, device="cuda")
    out = torch.empty(n, dtype=torch.bfloat16, device="cuda")
    ws2 = torch.empty(lib.tdx_init_workspace_bytes(2), dtype=torch.uint8, device="cuda")
    launches = C.launch([C.make_desc(big.data_ptr(), dtype=C.TDX_BF16, src=C.TDX_SRC_NORMAL, elem_count=big.numel(), seed=1, p1=0.02),
                         C.make_desc(out.data_ptr(), dtype=C.TDX_BF16, src=C.TDX_SRC_IOTA, elem_count=n, p0=0, p1=2, epi=epi)],
                        ws2.data_ptr(), ws2.numel(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert launches == 1 and torch.equal(out, freq.to(torch.bfloat16))


def test_position_ids_and_arange_buffers_fold():
    class M(nn.Module):
        def __init__(self):
            super().__init__()
            self.register_buffer("position_ids", torch.arange(512).expand((1, -1)))
            self.register_buffer("steps", torch.arange(2, 40, 3))
            self.register_buffer("half_steps", torch.arange(10, dtype=torch.float32) / 4)

    m = deferred_init(lambda: _on_cuda(M))
    materialize_module(m)
    st = last_materialize_stats()
    assert st["generic_ops"] == 0 and st["fused_tensors"] == 3, st
    assert torch.equal(m.position_ids.cpu(), torch.arange(512).expand((1, -1)))
    assert torch.equal(m.steps.cpu(), torch.arange(2, 40, 3)) and m.steps.dtype == torch.int64
    assert torch.equal(m.half_steps.cpu(), torch.arange(10, dtype=torch.float32) / 4)
