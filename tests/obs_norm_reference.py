"""NumPy reference of the running observation normalization (include/minppo_b200.h, minppo_obs_norm).

* ``normalize_obs``: the transform, in float32 with the kernels' operation order, so that it reproduces the GPU's
  normalized observations bit for bit: s = 1 / sqrt(var + float32(eps)), y = (x - mean) * s, clamp to [-clip, clip]
  when clip > 0.
* ``fold_obs_stats``: Chan's parallel merge of a batch into the running (count, mean, var), in float64:
  n' = n + n_b, mean' = mean + d n_b / n', var' = (var n + M2_b + d^2 n n_b / n') / n' with d = mean_b - mean.
"""
from __future__ import annotations

import numpy as np


def normalize_obs(obs, mean, var, eps: float = 1e-8, clip: float = 10.0) -> np.ndarray:
    """obs f32 [..., D] -> normalized f32 [..., D]."""
    f = np.float32
    x = np.asarray(obs, f)
    s = f(1.0) / np.sqrt(np.asarray(var, f) + f(eps))
    y = (x - np.asarray(mean, f)) * s
    if clip > 0:
        y = np.clip(y, -f(clip), f(clip))
    return y.astype(f)


def fold_obs_stats(mean, var, count, obs):
    """Fold the rows of obs [..., D] into (mean [D], var [D], count); everything float64.  Returns (mean', var', count')."""
    x = np.asarray(obs, np.float64).reshape(-1, np.shape(mean)[-1])
    n, nb = np.float64(count), np.float64(x.shape[0])
    y = x - x[0]                     # batch moments about the first row: no cancellation of a large common offset
    ym = y.mean(axis=0)
    mb = x[0] + ym
    m2b = ((y - ym) ** 2).sum(axis=0)
    mu, v = np.asarray(mean, np.float64), np.asarray(var, np.float64)
    n1 = n + nb
    d = mb - mu
    return mu + d * nb / n1, (v * n + m2b + d * d * n * nb / n1) / n1, n1
