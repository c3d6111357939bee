"""CPU checks of the per-minibatch PPO statistics: the reference in tests/update_stats_reference.py (self-consistency,
bit-identity with the oracle's update, a scalar float64 restatement) and the C-ABI declaration / export of
minppo_update_with_stats."""
import math
import os
import re

import numpy as np
import pytest

from oracle import ppo_numpy as P
from oracle import synth, threefry
from tests.update_stats_reference import update_with_stats

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

PROBLEMS = {
    "small": (dict(num_envs=16, num_steps=8, num_minibatches=4, update_epochs=2, anneal_lr=False), 37, 3),
    "tight_clip": (dict(num_envs=16, num_steps=8, num_minibatches=2, update_epochs=2, anneal_lr=False, clip_eps=0.05,
                        hidden_size=64, num_layers=1), 20, 5),
}


def _problem(name, perturb: bool):
    kw, D, A = PROBLEMS[name]
    hp = P.Hyper(**kw)
    pr = synth.make_problem(hp, D, A, seed=2, done_p=0.05)
    if perturb:
        g = np.random.default_rng(4)
        tr = pr["traj"]
        tr["log_prob"] = (tr["log_prob"] + 0.3 * g.standard_normal(tr["log_prob"].shape)).astype(np.float32)
        tr["value"] = (tr["value"] + 0.3 * g.standard_normal(tr["value"].shape)).astype(np.float32)
    return hp, pr


def _run(hp, pr, dtype=np.float64, gemm="exact", **kw):
    p0 = P.tree_like(pr["params"], lambda x: x.astype(dtype))
    return update_with_stats(p0, P.init_opt_state(p0), pr["traj"], pr["last_val"], pr["rng"], hp, dtype=dtype,
                             gemm=gemm, **kw)


@pytest.mark.parametrize("name", list(PROBLEMS))
@pytest.mark.parametrize("perturb", [False, True])
@pytest.mark.parametrize("dtype,gemm", [(np.float64, "exact"), (np.float32, "bf16")])
def test_stats_are_consistent(name, perturb, dtype, gemm):
    hp, pr = _problem(name, perturb)
    params, opt, rng, losses, aux = _run(hp, pr, dtype, gemm)
    st = aux["stats"]
    assert st.shape == (hp.update_epochs, hp.num_minibatches, 4) and np.all(np.isfinite(st))
    # (r - 1) - log r >= 0 for every r > 0; in float32 rounding can leave a row a few ulps below 0
    assert np.all(st[..., 0] >= (0.0 if dtype == np.float64 else -1e-7))
    assert np.all((st[..., 1:3] >= 0) & (st[..., 1:3] <= 1))
    # every fraction is a count over the minibatch's rows
    counts = st[..., 1:3] * hp.minibatch_size
    assert np.allclose(counts, np.round(counts), atol=1e-4)
    assert np.array_equal(st[..., 3], aux["grad_norms"])
    if perturb:                                    # 0.3 N(0, 1) of log_prob / value noise: some rows clip on both losses
        assert st[0, 0, 1] > 0 and st[0, 0, 2] > 0 and st[0, 0, 0] > 1e-3


def test_update_with_stats_is_the_oracle_update_bit_for_bit():
    hp, pr = _problem("small", True)
    p0 = P.tree_like(pr["params"], lambda x: x.astype(np.float32))
    want = P.update(p0, P.init_opt_state(p0), pr["traj"], pr["last_val"], pr["rng"], hp, dtype=np.float32, gemm="bf16")
    got = _run(hp, pr, np.float32, "bf16")
    flat = lambda t: P.flatten_params(t, hp.num_layers, np.float64)
    assert np.array_equal(flat(got[0]), flat(want[0]))
    assert np.array_equal(flat(got[1]["mu"]), flat(want[1]["mu"])) and np.array_equal(flat(got[1]["nu"]), flat(want[1]["nu"]))
    assert got[1]["count"] == want[1]["count"]
    assert np.array_equal(got[2], want[2]) and np.array_equal(got[3], want[3])
    for k in want[4]:
        assert np.array_equal(got[4][k], want[4][k]), k


def test_on_policy_log_prob_gives_zero_kl_and_no_clipping_at_the_first_step():
    """log_prob recomputed from the starting parameters on the same float64 forward: r == 1 at step (0, 0)."""
    hp, pr = _problem("small", False)
    tr = pr["traj"]
    T, N, D = tr["obs"].shape
    mean, log_std, _, _ = P.actor_critic_forward(pr["params"], tr["obs"].reshape(T * N, D).astype(np.float64), hp)
    logp, _, _ = P.gaussian_log_prob(mean, log_std, tr["action"].reshape(T * N, -1).astype(np.float64))
    tr["log_prob"] = logp.reshape(T, N)
    _, _, _, _, aux = _run(hp, pr)
    st = aux["stats"]
    assert abs(st[0, 0, 0]) < 1e-14 and st[0, 0, 1] == 0
    assert np.all(st[1:, :, 0] > 0)                # later steps run on updated parameters


@pytest.mark.parametrize("name", list(PROBLEMS))
def test_first_step_matches_a_scalar_float64_restatement(name):
    """Step (0, 0) recomputed row by row with math.exp / math.expm1 from the oracle's forward pass."""
    hp, pr = _problem(name, True)
    _, _, _, _, aux = _run(hp, pr)
    tr = pr["traj"]
    flat = P.flatten_traj({k: tr[k].astype(np.float64) for k in ("obs", "action", "value", "log_prob")})
    _, sub = threefry.split(np.asarray(pr["rng"], np.uint32), 2, hp.prng_mode)
    idx = threefry.permutation(sub, hp.batch_size, hp.prng_mode)[:hp.minibatch_size]
    params = P.tree_like(pr["params"], lambda x: x.astype(np.float64))
    mean, log_std, v, _ = P.actor_critic_forward(params, flat["obs"][idx], hp)
    kl = clip = vclip = 0.0
    for i, row in enumerate(idx):
        lp = 0.0
        for j in range(mean.shape[1]):
            z = (flat["action"][row, j] - mean[i, j]) / math.exp(log_std[j])
            lp += -0.5 * z * z - 0.5 * math.log(2 * math.pi) - log_std[j]
        lr = lp - flat["log_prob"][row]
        kl += math.expm1(lr) - lr
        clip += abs(math.exp(lr) - 1.0) > hp.clip_eps
        vclip += abs(v[i] - flat["value"][row]) > hp.clip_eps
    n = hp.minibatch_size
    got = aux["stats"][0, 0]
    assert abs(got[0] - kl / n) <= 1e-12 * max(1.0, kl / n)
    assert got[1] == clip / n and got[2] == vclip / n


def test_expm1_form_keeps_small_kl_accurate_in_float32():
    """Why the kernels use expm1f: at |log r| ~ 1e-3 the float32 difference (r - 1) - log r loses ~10 % to cancellation."""
    lr = np.float32(1e-3) * np.linspace(-1, 1, 101, dtype=np.float32)
    lr = lr[lr != 0]
    exact = np.expm1(lr.astype(np.float64)) - lr.astype(np.float64)
    naive = (np.exp(lr) - np.float32(1)) - lr
    stable = np.expm1(lr) - lr
    assert np.max(np.abs(stable - exact) / exact) < 1e-3
    assert np.max(np.abs(naive - exact) / exact) > 5e-2


def test_header_declares_and_library_exports_update_with_stats():
    text = open(os.path.join(ROOT, "include", "minppo_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    assert re.search(r"int\s+minppo_update_with_stats\s*\([^;]*float\*\s*losses_out,\s*float\*\s*stats_out,\s*int32_t\s+use_graph",
                     text)
    from minppo_b200 import _lib

    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__

        __graft_entry__.build()
    lib = _lib.load()
    assert "minppo_update_with_stats" in _lib.SYMBOLS and hasattr(lib, "minppo_update_with_stats")
    from minppo_b200.learner import STATS_COLUMNS

    assert STATS_COLUMNS == ("approx_kl", "clip_fraction", "value_clip_fraction", "grad_norm")
