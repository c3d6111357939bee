"""Parameter tree <-> flat fp32 arena, and the checkpoint pickle layout.

The reference pickles the flax variable dict ``{'params': {'MLP_0': {'Dense_i': {'kernel',
'bias'}}, 'MLP_1': {...}, 'log_std': ...}}`` (/root/reference/minppo/train.py:86-89, 112, 314;
SURVEY.md section 5).  The C ABI sees the same tree flattened in JAX's sorted-key order into
one contiguous arena (include/minppo_b200.h, minppo_param_layout).  Leaves are NumPy arrays
here (the reference's are jax.Array; unpickling those needs JAX).

A checkpoint of a policy trained with observation normalization carries the statistics as an optional sibling of
"params": ``{"params": ..., "obs_normalizer": {"mean", "var", "count", "eps", "clip"}}``
(minppo_b200.obs_norm.ObsNormalizer.to_tree); everything that reads "params" ignores it.
"""
from __future__ import annotations

import os
import pickle
from typing import Dict, List, Optional, Tuple

import numpy as np


def leaf_paths(num_layers: int) -> List[Tuple[str, ...]]:
    """Sorted flatten order: MLP_0 < MLP_1 < log_std; Dense_i ascending; bias < kernel."""
    out: List[Tuple[str, ...]] = []
    for mlp in ("MLP_0", "MLP_1"):
        for i in range(num_layers + 1):
            out.append((mlp, f"Dense_{i}", "bias"))
            out.append((mlp, f"Dense_{i}", "kernel"))
    out.append(("log_std",))
    return out


def leaf_shapes(obs_dim: int, act_dim: int, hidden: int, num_layers: int) -> List[Tuple[int, ...]]:
    shapes: List[Tuple[int, ...]] = []
    for out_dim in (act_dim, 1):
        fan_in = obs_dim
        for i in range(num_layers + 1):
            o = hidden if i < num_layers else out_dim
            shapes.append((o,))
            shapes.append((fan_in, o))
            fan_in = o
    shapes.append((act_dim,))
    return shapes


def param_count(obs_dim: int, act_dim: int, hidden: int, num_layers: int) -> int:
    return int(sum(int(np.prod(s)) for s in leaf_shapes(obs_dim, act_dim, hidden, num_layers)))


def _get(tree: Dict, path: Tuple[str, ...]):
    node = tree["params"]
    for k in path:
        node = node[k]
    return node


def flatten_params(tree: Dict, num_layers: int) -> np.ndarray:
    return np.concatenate([np.asarray(_get(tree, p), np.float32).ravel() for p in leaf_paths(num_layers)])


def unflatten_params(flat: np.ndarray, obs_dim: int, act_dim: int, hidden: int, num_layers: int) -> Dict:
    flat = np.asarray(flat, np.float32)
    tree: Dict = {"params": {}}
    off = 0
    for path, shape in zip(leaf_paths(num_layers), leaf_shapes(obs_dim, act_dim, hidden, num_layers)):
        n = int(np.prod(shape))
        node = tree["params"]
        for k in path[:-1]:
            node = node.setdefault(k, {})
        node[path[-1]] = flat[off:off + n].reshape(shape).copy()
        off += n
    if off != flat.size:
        raise ValueError(f"arena has {flat.size} elements, layout needs {off}")
    return tree


OBS_NORMALIZER_KEY = "obs_normalizer"
OBS_NORMALIZER_FIELDS = ("mean", "var", "count", "eps", "clip")


def save_model(params: Dict, filename: str, obs_normalizer: Optional[Dict] = None) -> None:
    """Same pickle as train.py:86-89.  The reference calls os.makedirs(os.path.dirname(f)),
    which raises for a bare filename such as the default 'trained_model.pkl' (SURVEY.md
    section 5); the empty dirname is guarded here.  ``obs_normalizer``: the observation statistics
    (ObsNormalizer.to_tree()), stored beside "params"."""
    if obs_normalizer is not None:
        missing = [k for k in OBS_NORMALIZER_FIELDS if k not in obs_normalizer]
        if missing:
            raise ValueError(f"obs_normalizer lacks {missing}")
        params = {**params, OBS_NORMALIZER_KEY: {k: obs_normalizer[k] for k in OBS_NORMALIZER_FIELDS}}
    d = os.path.dirname(filename)
    if d:
        os.makedirs(d, exist_ok=True)
    with open(filename, "wb") as f:
        pickle.dump(params, f)


def load_model(filename: str) -> Dict:
    """/root/reference/minppo/infer.py:17-19."""
    with open(filename, "rb") as f:
        return pickle.load(f)
