"""T0' parity (SURVEY.md section 8c): for CPU-device tensors the engine replays through ATen and
must equal the REAL reference bit for bit, RNG included -- same mt19937 stream, same materialize
order, dead ops included.  What the reference materialised (oracle/_ref, run on these cases by
tests/golden/make_reference_outputs.py) is stored as the digest of every tensor's bytes."""
import pytest
import torch

from oracle import cases
from oracle import golden
from torchdistx_b200.deferred_init import deferred_init, materialize_module

CASES = [
    ("linear128", "fp32"), ("init_zoo", "fp32"), ("init_zoo", "bf16"), ("mlp_stack", "fp32"),
    ("tiny_llama", "fp32"), ("tiny_llama", "bf16"), ("tiny_gpt2", "fp32"),
    ("torch_transformer", "fp32"), ("clones", "fp32"), ("cast_variant", "fp32"),
] + [(f"family_{name}", "fp32") for name in cases.FAMILIES] + [("family_llama", "bf16"), ("family_gpt2", "bf16")]
# (families: real HF / torch.nn constructors at toy sizes -- Llama, Mistral, Qwen2, Mixtral, Gemma-2, Phi-3,
#  GPT-2, OPT, BERT, T5, ViT, LSTM, Conv+BatchNorm, MultiheadAttention, nn.Transformer)
SEED = 5


@pytest.fixture(scope="module")
def reference_outputs():
    return golden.load("reference_cpu_parity")


@pytest.mark.parametrize("case,dtype", CASES)
def test_cpu_materialize_equals_reference_bit_exact(case, dtype, reference_outputs):
    ref = reference_outputs[f"{case}_{dtype}"]
    torch.set_default_dtype(cases.DTYPES[dtype])
    try:
        m = deferred_init(lambda: cases.build(case, dtype))
        torch.manual_seed(SEED)
        materialize_module(m)
    finally:
        torch.set_default_dtype(torch.float32)
    mine = dict(list(m.named_parameters()) + list(m.named_buffers()))
    # tied parameters stay ONE object here (named_parameters de-duplicates them); the oracle
    # driver re-wraps per slot, so it may list more names
    assert set(mine) <= set(ref) and len(mine) >= len(ref) - 2
    for k, t in mine.items():
        r = ref[k]
        assert str(t.dtype) == r["dtype"] and tuple(t.shape) == r["shape"], k
        assert golden.digest(t) == r["digest"], k
