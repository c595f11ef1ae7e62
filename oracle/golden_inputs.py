"""Seeded inputs shared by oracle/make_golden.py (which runs the unmodified reference)
and tests/ (which run the oracle and the CUDA path on the same inputs).

Test infrastructure.  Everything is derived from numpy PCG64 streams so that the
fixtures under tests/golden/ only need to hold OUTPUTS plus an input checksum.
"""
from __future__ import annotations

import zlib

import numpy as np
import torch


def fill_state_dict(module: torch.nn.Module, seed: int) -> None:
    """Deterministically overwrite every parameter/buffer of `module` (by state_dict order)."""
    rng = np.random.default_rng(seed)
    sd = module.state_dict()
    new = {}
    for name, t in sd.items():
        shape = tuple(t.shape)
        leaf = name.rsplit(".", 1)[-1]
        if leaf == "num_batches_tracked":
            new[name] = torch.zeros_like(t)
            continue
        if leaf == "centers":
            new[name] = t.clone()
            continue
        if leaf == "running_mean":
            a = rng.normal(0.0, 0.1, size=shape)
        elif leaf == "running_var":
            a = rng.uniform(0.5, 1.5, size=shape)
        elif leaf == "weight" and len(shape) == 1:          # norm affine scale
            a = rng.uniform(0.5, 1.5, size=shape)
        elif leaf == "bias" and _is_norm(module, name):
            a = rng.uniform(-0.2, 0.2, size=shape)
        elif leaf == "weight":                              # Linear [out, in]
            bound = 1.0 / np.sqrt(shape[1])
            a = rng.uniform(-bound, bound, size=shape)
        else:                                               # Linear bias
            a = rng.uniform(-0.1, 0.1, size=shape)
        new[name] = torch.from_numpy(np.asarray(a)).to(t.dtype)
    module.load_state_dict(new)


def _is_norm(module, name):
    parent = name.rsplit(".", 1)[0]
    m = module
    for part in parent.split("."):
        m = getattr(m, part) if not part.isdigit() else m[int(part)]
    return isinstance(m, (torch.nn.BatchNorm1d, torch.nn.LayerNorm))


def features(seed: int, n: int, d: int, scale: float = 1.0) -> torch.Tensor:
    rng = np.random.default_rng(seed)
    return torch.from_numpy((rng.normal(size=(n, d)) * scale).astype(np.float32))


def checksum(*arrays) -> int:
    c = 0
    for a in arrays:
        if isinstance(a, torch.Tensor):
            a = a.detach().cpu().numpy()
        c = zlib.crc32(np.ascontiguousarray(a).tobytes(), c)
    return c


def sample(a, n: int = 4096) -> np.ndarray:
    """A fixed subset of at most `n` elements of `a`: the flattened array at an odd stride, which visits every column
    of the power-of-two-wide feature and weight matrices.  Large fixture arrays are stored as this sample (bounds the
    file size); tests compare the same subset of what they compute."""
    if isinstance(a, torch.Tensor):
        a = a.detach().cpu().numpy()
    a = np.asarray(a).reshape(-1)
    return a[::max(1, -(-a.size // n)) | 1]


# JVASP-98225 (32 atoms: 16 K + 16 Bi) cartesian coordinates are read by make_golden.py
# from the reference test (alignn/tests/test_force_reduction.py:22-55) at generation time
# and stored inside tests/golden/jvasp_98225.npz; tests read them from there.


def cell_volumes(batch_num_nodes) -> torch.Tensor:
    """g.ndata["V"] (graphs.py:560): the cell volume repeated on every atom of a crystal; crystal b gets 90 + 17 b A^3."""
    bnn = [int(n) for n in batch_num_nodes]
    return torch.cat([torch.full((n,), 90.0 + 17.0 * b) for b, n in enumerate(bnn)])
