"""oracle/fixture.py -- TEST INFRASTRUCTURE ONLY.

Compact fixtures of reference outputs too large to commit whole: a seeded sample of the cells, the largest
magnitude, the Frobenius norm and a seeded random projection of every cell.  Written by oracle/gen_golden_live.py,
read by the tests.
"""
from __future__ import annotations

import numpy as np


def _projection(shape, seed=7):
    rng = np.random.default_rng(seed)
    return np.exp(2j * np.pi * rng.random(shape))


def summarise(prefix: str, a, n: int = 512, seed: int = 11) -> dict:
    a = np.asarray(a)
    idx = np.sort(np.random.default_rng(seed).choice(a.size, size=min(n, a.size), replace=False))
    return {prefix + "_shape": np.array(a.shape, dtype=np.int64), prefix + "_idx": idx.astype(np.int32),
            prefix + "_val": a.ravel()[idx], prefix + "_amax": np.max(np.abs(a)), prefix + "_fro": np.linalg.norm(a),
            prefix + "_proj": np.sum(a * _projection(a.shape))}


def errors(got, d, prefix: str):
    """(max-abs error over the sampled cells / the reference's max-abs, relative difference of the Frobenius norms,
    projection error / (||ref||_F sqrt(cells)) -- a lower bound of the relative Frobenius error ||got - ref|| / ||ref||)"""
    got = np.asarray(got)
    assert tuple(got.shape) == tuple(int(v) for v in d[prefix + "_shape"]), (got.shape, d[prefix + "_shape"])
    amax, fro = float(d[prefix + "_amax"]), float(d[prefix + "_fro"])
    e_max = float(np.max(np.abs(got.ravel()[d[prefix + "_idx"]] - d[prefix + "_val"]))) / amax
    e_fro = abs(float(np.linalg.norm(got)) - fro) / fro
    e_proj = abs(complex(np.sum(got * _projection(got.shape))) - complex(d[prefix + "_proj"])) / (fro * np.sqrt(got.size))
    return e_max, e_fro, e_proj
