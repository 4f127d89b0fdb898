"""What the real reference computed, stored under tests/golden/ (TEST INFRASTRUCTURE).

The reference can only be compiled where its sources are (oracle/build_ref.py); the tests that
compare with it read these files instead, so they run from a checkout alone.
tests/golden/make_reference_outputs.py runs the compiled reference and rewrites them.

Three forms, chosen by what a test compares:
  * `digest`        the bytes of a tensor (with its dtype and shape): bit-exact comparisons;
  * `value_digest`  the values as `float32` with NaN positions and -0.0 == 0.0, for comparisons
                    that are exact up to those (tests/test_reference_differential_cpu.py);
  * `summary`       float64 moments, min / max and `quantiles`: the sorted sample at M evenly
                    spaced probabilities.  `expand` rebuilds a sample of any size from them whose
                    empirical CDF is within 1/M of the original's, so a two-sample Kolmogorov-Smirnov
                    test against it keeps its sample sizes and nearly all of its power.
"""
from __future__ import annotations

import gzip
import hashlib
import io
import os

import numpy as np
import torch

DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def path(name: str) -> str:
    return os.path.join(DIR, name + ".pt.gz")


def save(name: str, obj) -> str:
    buf = io.BytesIO()
    torch.save(obj, buf)
    with open(path(name), "wb") as f:
        f.write(gzip.compress(buf.getvalue(), compresslevel=9, mtime=0))
    return path(name)


def load(name: str):
    with open(path(name), "rb") as f:
        return torch.load(io.BytesIO(gzip.decompress(f.read())))


def _hash(*parts: bytes) -> str:
    h = hashlib.sha256()
    for p in parts:
        h.update(p)
    return h.hexdigest()[:32]


def digest(t: torch.Tensor) -> str:
    t = t.detach().cpu().contiguous()
    return _hash(str(t.dtype).encode(), str(tuple(t.shape)).encode(), t.reshape(-1).view(torch.uint8).numpy().tobytes())


def value_digest(t: torch.Tensor) -> str:
    t = t.detach().cpu()
    v = torch.nan_to_num(t.float()) + 0.0  # (-0.0 + 0.0 is +0.0)
    return _hash(str(t.dtype).encode(), str(tuple(t.shape)).encode(), torch.isnan(t).numpy().tobytes(),
                 v.contiguous().numpy().tobytes())


def quantiles(sample: torch.Tensor, m: int) -> torch.Tensor:
    """The sorted sample at probabilities (i + 1/2) / m, i < m (the whole sorted sample if it is no larger)."""
    s = sample.detach().cpu().reshape(-1).sort().values
    n = s.numel()
    if n <= m:
        return s.clone()
    return s[((torch.arange(m, dtype=torch.float64) + 0.5) * n / m).long()].clone()


def summary(t: torch.Tensor, m: int = 0) -> dict:
    """Moments and range of `t`, and its `quantiles(t, m)` if m > 0."""
    d = t.detach().cpu().reshape(-1).double()
    out = {"numel": t.numel(), "dtype": str(t.dtype), "shape": tuple(t.shape), "mean": d.mean().item(),
           "std": d.std().item(), "min": d.min().item(), "max": d.max().item()}
    if m > 0:
        out["quantiles"] = quantiles(t, m)
    return out


def expand(q: torch.Tensor, n: int) -> np.ndarray:
    """A sample of `n` values (float64, sorted) with the distribution `quantiles(...)` recorded."""
    q = q.double().numpy()
    m = q.size
    if m == n:
        return q
    return np.interp((np.arange(n) + 0.5) / n, (np.arange(m) + 0.5) / m, q)
