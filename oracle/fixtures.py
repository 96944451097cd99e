"""Storage form of the golden fixtures under ``tests/golden/`` (make_golden.py writes them with ``save``, the tests
read them with ``load``), which keeps every file below 1 MB:

* a parameter the reference initialised with ``ref_oracle.reference_init_`` is not stored: ``rand_<key>`` holds
  [seed, offset, *shape], the seed of the generator it was drawn from and the number of float64 draws before it in
  that generator's stream; ``load`` draws it again and checks it against ``head_<key>``, its first stored values;
* an array named in ``save(sampled=...)`` with more than ``SAMPLE_ABOVE`` entries keeps every ``every_<key>``-th entry
  of its flattened values; ``pick`` takes the same entries of a tensor compared with it.
"""
from __future__ import annotations

import numpy as np
import torch

from . import ref_oracle as O

SAMPLE_ABOVE = 16384


def save(path: str, arrays: dict, drawn: dict | None = None, sampled=(), every: int = 5) -> None:
    """``drawn``: {key: (seed, offset)} of the arrays ``reference_init_`` produced."""
    drawn = drawn or {}
    out = {}
    for k, a in arrays.items():
        a = np.asarray(a)
        if k in drawn:
            out["rand_" + k] = np.array([*drawn[k], *a.shape], dtype=np.int64)
            out["head_" + k] = a.reshape(-1)[:8]
        elif k in sampled and a.size > SAMPLE_ABOVE:
            out[k] = a.reshape(-1)[::every]
            out["every_" + k] = np.int64(every)
        else:
            out[k] = a
    np.savez_compressed(path, **out)


def load(path: str) -> dict:
    z = np.load(path)
    out = {k: z[k] for k in z.files if not k.startswith(("rand_", "head_"))}
    by_seed = {}
    for k in z.files:
        if k.startswith("rand_"):
            seed, off, *shape = (int(v) for v in z[k])
            by_seed.setdefault(seed, []).append((off, k[len("rand_"):], shape))
    for seed, entries in by_seed.items():
        g = torch.Generator().manual_seed(seed)
        pos = 0
        for off, key, shape in sorted(entries):
            torch.rand(off - pos, generator=g, dtype=torch.float64)        # the draws in front of this parameter
            p = torch.empty(shape)
            O.reference_init_([p], g)
            pos = off + p.numel()
            out[key] = p.numpy()
            if not np.array_equal(out[key].reshape(-1)[:8], z["head_" + key]):
                raise RuntimeError(f"{path}: {key} drawn again differs from the values the fixture was made with")
    return out


def pick(z: dict, key: str, t):
    """The entries of ``t`` that the fixture keeps for ``key``: all of them, or every n-th of the flattened tensor."""
    if "every_" + key not in z:
        return t
    return t.reshape(-1)[::int(z["every_" + key])]
