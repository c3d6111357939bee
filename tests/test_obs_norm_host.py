"""Observation normalization, host side (no GPU): the NumPy reference (tests/obs_norm_reference.py), the ctypes mirror of
struct minppo_obs_norm, ObsNormalizer's checks and tree form, and the checkpoint layout with and without the
"obs_normalizer" entry."""
import ctypes as C
import os

import numpy as np
import pytest

from minppo_b200 import _lib, params
from oracle import ppo_numpy as P
from tests.obs_norm_reference import fold_obs_stats, normalize_obs
from tests.test_abi import _header_fields


def _batches(offset: float, scale: float, sizes, D=7, seed=0):
    g = np.random.default_rng(seed)
    return [(offset + scale * g.standard_normal((n, D))).astype(np.float32) for n in sizes]


@pytest.mark.parametrize("offset,scale", [(0.0, 1.0), (3.0, 0.5), (1e4, 1e-2)])
def test_fold_of_batches_equals_moments_of_their_concatenation(offset, scale):
    """Chan's merge from the initial state (mean 0, var 1, count 0) over batches of different sizes: the float64 mean and
    population variance of all rows, including data far from 0 relative to its spread."""
    bs = _batches(offset, scale, (5, 1000, 37, 4096))
    D = bs[0].shape[1]
    mean, var, count = np.zeros(D), np.ones(D), 0.0
    for b in bs:
        mean, var, count = fold_obs_stats(mean, var, count, b)
    allx = np.concatenate(bs).astype(np.float64)
    y = allx - allx[0]                         # exact in float64: the moments of y carry no cancellation of the offset
    assert count == allx.shape[0]
    np.testing.assert_allclose(mean, allx[0] + y.mean(0), rtol=1e-12, atol=0)
    # atol: near 1e4 the float64 running mean itself is rounded to 1.8e-12 (its ulp), which reaches the variance through
    # the d^2 term of the merge (measured 1.7e-16 here); a sum of squares of the raw values would be off by ~1e-8
    np.testing.assert_allclose(var, y.var(0), rtol=1e-12, atol=1e-15)


def test_normalize_obs_formula_and_clip():
    g = np.random.default_rng(1)
    x = (g.standard_normal((64, 5)) * 30).astype(np.float32)
    mean = g.standard_normal(5).astype(np.float32)
    var = np.array([1e-4, 1e-2, 1.0, 1e2, 1e4], np.float32)
    y = normalize_obs(x, mean, var, 1e-8, 10.0)
    assert y.dtype == np.float32 and np.abs(y).max() == np.float32(10.0)
    raw = normalize_obs(x, mean, var, 1e-8, 0.0)                 # clip <= 0: no clamp
    assert np.abs(raw).max() > 10.0
    np.testing.assert_array_equal(y, np.clip(raw, -10, 10))
    # float32 throughout, in the kernels' order: (x - mean) * (1 / sqrt(var + eps))
    s = np.float32(1) / np.sqrt(var + np.float32(1e-8))
    np.testing.assert_array_equal(raw, (x - mean) * s)
    # the initial state (mean 0, var 1) leaves in-range observations unchanged
    np.testing.assert_array_equal(normalize_obs(x / 10, np.zeros(5), np.ones(5), 1e-8, 10.0), x / 10)


def test_ctypes_mirror_matches_header():
    names = _header_fields("typedef struct minppo_obs_norm {", "} minppo_obs_norm;")
    assert names == [f[0] for f in _lib.MinppoObsNorm._fields_] == ["mean", "var", "count", "eps", "clip"]
    assert C.sizeof(_lib.MinppoObsNorm) == 3 * 8 + 2 * 8


def test_obs_normalizer_checks_and_tree_round_trip():
    torch = pytest.importorskip("torch")
    from minppo_b200.obs_norm import ObsNormalizer

    cpu = torch.device("cpu")
    n = ObsNormalizer.create(6, cpu, eps=1e-6, clip=5.0)
    assert n.mean.dtype == torch.float32 and n.var.dtype == torch.float32 and n.count.dtype == torch.float64
    assert torch.equal(n.mean, torch.zeros(6)) and torch.equal(n.var, torch.ones(6)) and float(n.count) == 0.0
    n.check(6, cpu)
    with pytest.raises(ValueError):
        n.check(7, cpu)
    bad = ObsNormalizer(n.mean, n.var, n.count.float(), n.eps, n.clip)
    with pytest.raises(TypeError):
        bad.check(6, cpu)
    n.mean.copy_(torch.arange(6, dtype=torch.float32))
    n.count.fill_(123.0)
    tree = n.to_tree()
    assert set(tree) == set(params.OBS_NORMALIZER_FIELDS)
    m = ObsNormalizer.from_tree(tree, cpu)
    assert torch.equal(m.mean, n.mean) and torch.equal(m.var, n.var) and torch.equal(m.count, n.count)
    assert (m.eps, m.clip) == (1e-6, 5.0)


def test_checkpoint_round_trip_with_and_without_obs_normalizer(tmp_path):
    D, A, H, L = 11, 3, 64, 2
    tree = P.init_params(D, A, H, L, seed=0, dtype=np.float32)
    flat = params.flatten_params(tree, L)
    plain = os.path.join(tmp_path, "plain.pkl")
    params.save_model(tree, plain)
    got = params.load_model(plain)
    assert set(got) == {"params"}
    np.testing.assert_array_equal(params.flatten_params(got, L), flat)

    stats = {"mean": np.linspace(-1, 1, D).astype(np.float32), "var": np.full(D, 2.5, np.float32),
             "count": np.float64(4096.0), "eps": 1e-8, "clip": 10.0}
    normed = os.path.join(tmp_path, "normed.pkl")
    params.save_model(tree, normed, obs_normalizer=stats)
    got = params.load_model(normed)
    assert set(got) == {"params", params.OBS_NORMALIZER_KEY}
    np.testing.assert_array_equal(params.flatten_params(got, L), flat)     # flattening reads only "params"
    for k in params.OBS_NORMALIZER_FIELDS:
        np.testing.assert_array_equal(got[params.OBS_NORMALIZER_KEY][k], stats[k])
    assert set(tree) == {"params"}                                          # the caller's tree is not modified
    with pytest.raises(ValueError):
        params.save_model(tree, normed, obs_normalizer={"mean": stats["mean"]})
