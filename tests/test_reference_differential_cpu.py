"""Differential run against the REAL reference on random linked scripts, CPU device: both engines
replay recorded ATen ops there, so every bit is comparable, random draws included (SURVEY.md 8c
T0'); the eager run of the same script is the third opinion.  What the reference materialised
(oracle/_ref, run on the same scripts by tests/golden/make_reference_outputs.py) is stored as
`oracle.golden.value_digest`s: equal digests are what `same` below calls the same.

What is asserted
  * there is no script on which the reference reproduces the eager construction and this engine
    does not: whenever reference == eager, engine == reference, bit for bit;
  * this engine reproduces the eager construction on at least 95 % of the scripts (the rest draw
    random numbers in an order that construction and materialisation legitimately do not share:
    a tensor's whole history is replayed when its turn comes, reference deferred_init.cc:541-622);
  * the one systematic difference, pinned by a minimal program: the reference LOSES in-place writes
    made through a view of a tensor before its last alias op -- `t = ones(4, 4); t[1].zero_();
    Parameter(t)` materialises as all ones there (the same write AFTER the Parameter exists, which
    is what nn.Embedding(padding_idx=...) does, is kept).  Eager PyTorch is the arbiter: the engine
    keeps the write.  On these scripts the reference matches eager far less often than the engine
    for that reason (printed, and asserted only as "not more often")."""
import pytest
import torch
from torch import nn

from oracle import fuzz_programs as P
from oracle import golden
from torchdistx_b200.deferred_init import deferred_init, materialize_module

N = 300


def same(x, y):
    return (x.dtype == y.dtype and x.shape == y.shape and torch.equal(torch.isnan(x), torch.isnan(y))
            and torch.equal(torch.nan_to_num(x.float()), torch.nan_to_num(y.float())))


@pytest.fixture(scope="module")
def reference_runs():
    return golden.load("reference_differential")


def test_engine_is_never_wrong_where_the_reference_is_right(reference_runs):
    engine_eq_eager = ref_eq_eager = both = 0
    assert len(reference_runs["scripts"]) == N
    for seed in range(N):
        ref = reference_runs["scripts"][seed]
        assert not isinstance(ref, str), (seed, ref)  # (the reference accepted every script)
        progs, links = P.differential_script(seed)
        m = deferred_init(P.LinkedHolder, progs, links)
        torch.manual_seed(seed)
        materialize_module(m)
        torch.manual_seed(seed)
        eager = P.LinkedHolder(progs, links)
        mine = {k: v.detach() for k, v in m.named_parameters()}
        want = {k: v.detach() for k, v in eager.named_parameters()}
        assert set(mine) == set(ref) == set(want)
        e_ok = all(same(mine[k], want[k]) for k in want)
        r_ok = all(ref[k] == golden.value_digest(want[k]) for k in want)
        if r_ok:
            assert all(golden.value_digest(mine[k]) == ref[k] for k in ref), seed
        engine_eq_eager += e_ok
        ref_eq_eager += r_ok
        both += e_ok and r_ok
    print(f"\n{N} scripts: engine == eager on {engine_eq_eager}, reference == eager on {ref_eq_eager}, both on {both}")
    assert engine_eq_eager >= 0.95 * N and ref_eq_eager <= engine_eq_eager and both == ref_eq_eager


def test_write_through_a_view_before_the_last_alias_is_kept(reference_runs):
    def before():
        t = torch.ones(4, 4)
        t[1].zero_()
        return nn.ParameterList([nn.Parameter(t)])

    def after():
        t = nn.Parameter(torch.ones(4, 4))
        with torch.no_grad():
            t[1].zero_()
        return nn.ParameterList([t])

    for fn in (before, after):
        m = deferred_init(fn)
        materialize_module(m)
        assert torch.equal(m[0].detach(), fn()[0].detach()), fn.__name__
    # the reference, same two programs: row 1 of what it materialised (make_reference_outputs.VIEW_WRITE)
    out = reference_runs["view_write"]
    assert "after [0.0, 0.0, 0.0, 0.0]" in out, out
    # (if a later reference build keeps the write, this line is what changes -- and the docstring above)
    assert "before [1.0, 1.0, 1.0, 1.0]" in out, out
