"""The per-leaf gradient comparator of tests/test_gpu_gradient_leaves.py, checked without a device.

* It rejects gradients that are wrong in the ways a kernel goes wrong (a scaled leaf, a dropped row, a coefficient applied
  twice or not at all, a split-K partial counted twice), including errors the whole-gradient bound of
  test_single_minibatch_gradient lets through.
* Its bounds can be met: on every case of the GPU matrix, the oracle with the kernels' bf16 rounding points is within
  the float64 per-leaf bound of the exact oracle, so a GPU failure points at the GPU.
* The float64 clip + Adam restatement the GPU optimizer is checked against is the oracle's optax chain.
"""
import numpy as np
import pytest

from minppo_b200.params import param_count
from oracle import ppo_numpy as P
from oracle import synth
from tests.gradient_cases import CASES, learner_path
from tests.helpers import (LEAF_BOUND_BF16, LEAF_BOUND_FP64, clip_adam_flat, compare_leaves, flat_grads, fp64_leaf_bounds,
                           leaf_errors, leaves_over, perturb_policy, rel_err, single_step_oracle_grads)


def _problem(name):
    case = CASES[name]
    hp = P.Hyper(**case["hp"])
    pr = synth.make_problem(hp, case["D"], case["A"], seed=9, done_p=0.02)
    perturb_policy(pr)
    return case, hp, pr


def _hidden(pth, L):
    return pth[0] in ("MLP_0", "MLP_1") and pth[1] != f"Dense_{L}"


def _mutate(tree, pred, fn):
    out = P.tree_like(tree, lambda x: np.array(x, copy=True))
    for pth in P.leaf_order(len(tree["params"]["MLP_0"]) - 1):
        if pred(pth):
            P.set_leaf(out, pth, fn(P.get_leaf(out, pth)))
    return out


MUTATION_SHAPES = ["d1_a1_mb200", "l1_a9_mb127"]    # ent_coef != 0 and vf_coef != 1: every mutation changes something


@pytest.mark.parametrize("name", MUTATION_SHAPES)
def test_comparator_rejects_wrong_gradients(name):
    case, hp, pr = _problem(name)
    D, A, H, L = case["D"], case["A"], hp.hidden_size, hp.num_layers
    assert hp.ent_coef != 0 and hp.vf_coef != 1
    _, gbf = single_step_oracle_grads(hp, pr, np.float32, "bf16")
    _, g64 = single_step_oracle_grads(hp, pr, np.float64, "exact")
    mb = hp.minibatch_size
    S = learner_path(case["hp"], D, A, 148, case["cfg"])["S"]
    bias0 = ("MLP_0", "Dense_0", "bias")
    kernel_last_hidden = ("MLP_1", f"Dense_{L - 1}", "kernel")
    # the hidden bias leaf without one minibatch row (a ragged tile edge dropped): the same sums over the other rows.  The
    # last row that contributes at all (a row whose probability ratio is clipped has no actor gradient).
    for r in range(mb - 1, -1, -1):
        _, g_drop = single_step_oracle_grads(hp, pr, np.float32, "bf16", rows=np.delete(np.arange(mb), r))
        if not np.array_equal(P.get_leaf(g_drop, bias0), P.get_leaf(gbf, bias0)):
            break
    mutations = {
        "hidden_x1.05": _mutate(gbf, lambda p: _hidden(p, L), lambda x: 1.05 * x),
        "bias_row_dropped": _mutate(gbf, lambda p: p == bias0, lambda x: P.get_leaf(g_drop, bias0)),
        "critic_vf_twice": _mutate(gbf, lambda p: p[0] == "MLP_1", lambda x: hp.vf_coef * x),
        "log_std_no_entropy": _mutate(gbf, lambda p: p == ("log_std",), lambda x: x + hp.ent_coef),
        "split_partial_twice": _mutate(gbf, lambda p: p == kernel_last_hidden, lambda x: x + x / S),
    }
    gbf_flat = flat_grads(gbf, L)
    for what, bad in mutations.items():
        bad_flat = flat_grads(bad, L)
        e_bf, e_64 = compare_leaves(bad_flat, gbf, g64, D, A, H, L)
        assert leaves_over(e_bf, LEAF_BOUND_BF16), (what, e_bf)
        # the whole-gradient bound of test_single_minibatch_gradient, relative to the largest entry
        old_ok = rel_err(bad_flat, gbf_flat) < 5e-3
        if what in ("hidden_x1.05", "bias_row_dropped"):
            assert old_ok, what
    # and the unmutated emulated gradient passes both per-leaf bounds
    e_bf, e_64 = compare_leaves(gbf_flat, gbf, g64, D, A, H, L)
    assert not leaves_over(e_bf, LEAF_BOUND_BF16) and not leaves_over(e_64, LEAF_BOUND_FP64, fp64_leaf_bounds(hp))


def _distinct_problems():
    """One CASES entry per distinct oracle problem (learner options do not change the oracle)."""
    seen, out = set(), []
    for name, case in CASES.items():
        key = (tuple(sorted(case["hp"].items())), case["D"], case["A"])
        if key not in seen:
            seen.add(key)
            out.append(name)
    return out


@pytest.mark.parametrize("name", _distinct_problems())
def test_emulated_oracle_meets_the_fp64_leaf_bound(name):
    case, hp, pr = _problem(name)
    _, gbf = single_step_oracle_grads(hp, pr, np.float32, "bf16")
    _, g64 = single_step_oracle_grads(hp, pr, np.float64, "exact")
    errs = leaf_errors(flat_grads(gbf, hp.num_layers), g64, case["D"], case["A"], hp.hidden_size, hp.num_layers)
    assert not leaves_over(errs, LEAF_BOUND_FP64, fp64_leaf_bounds(hp)), errs


@pytest.mark.parametrize("name", list(CASES))
def test_cases_reach_their_paths_on_a_b200(name):
    """At the B200's 148 SMs the library plans for every case the path it names (the GPU test asserts the same with the
    device's own SM count and the library's launch count)."""
    case = CASES[name]
    path = learner_path(case["hp"], case["D"], case["A"], 148, case["cfg"], case.get("force_cap"))
    for k, v in case["expect"].items():
        assert path[k] == v, (k, path)
    assert path["P"] == param_count(case["D"], case["A"], case["hp"]["hidden_size"], case["hp"]["num_layers"])


@pytest.mark.parametrize("count", [0, 37])
@pytest.mark.parametrize("max_norm", [1e6, 1e-3])
def test_flat_clip_adam_is_the_oracle_chain(count, max_norm):
    D, A, H, L = 37, 3, 64, 2
    hp = P.Hyper(num_envs=8, num_steps=4, num_minibatches=1, update_epochs=1, anneal_lr=count > 0,
                 total_timesteps=128, max_grad_norm=max_norm)
    g = np.random.default_rng(count)
    n = param_count(D, A, H, L)
    p, gr = g.standard_normal(n), 1e-2 * g.standard_normal(n)
    mu, nu = (1e-3 * g.standard_normal(n), g.uniform(0, 1e-6, n)) if count else (np.zeros(n), np.zeros(n))
    un = lambda x: P.unflatten_params(x, D, A, H, L)
    tp, to, tn = P.clip_adam_step(un(p), un(gr), {"count": count, "mu": un(mu), "nu": un(nu)}, hp)
    fp, fmu, fnu, fn = clip_adam_flat(p, gr, mu, nu, count, hp)
    assert (fn < max_norm) == (max_norm > 1)
    np.testing.assert_allclose(fp, P.flatten_params(tp, L, np.float64), rtol=1e-13, atol=0)
    np.testing.assert_allclose(fmu, P.flatten_params(to["mu"], L, np.float64), rtol=1e-13, atol=0)
    np.testing.assert_allclose(fnu, P.flatten_params(to["nu"], L, np.float64), rtol=1e-13, atol=0)
    assert abs(fn - tn) <= 1e-13 * tn and to["count"] == count + 1
