"""Every gradient leaf and the optimizer step of the learner, against float64 references, on every learner path.

The whole-gradient comparison of test_gpu_update.py is relative to the largest entry, which sits in an output head; the
hidden-layer leaves are ~1e-4 of it, and Adam's normalised step hides a leaf's gradient scale from the parameter checks.
So here each leaf is held to its own scale (tests/helpers.py: compare_leaves), and the optimizer is checked on its own,
in float64, from the gradient the GPU reduced.

(a) one minibatch step per case of tests/gradient_cases.py (E = M = 1: read("grad") is that step's gradient), each case
    asserting the path it reaches;
(b) multi-step updates at learning rate 0: the parameters stay put, so every step is comparable to the oracle tightly;
(c) clip + Adam restated in float64 on the GPU's own gradient, on every optimizer path.
The measured errors are written to $MINPPO_TEST_METRICS_DIR/leaf_metrics.json when that variable is set.
"""
import json
import os

import numpy as np
import pytest

from oracle import ppo_numpy as P
from oracle import synth
from tests.gradient_cases import CASES, learner_path
from tests.helpers import (LEAF_BOUND_BF16, LEAF_BOUND_FP64, clip_adam_flat, compare_leaves, flat_grads, fp64_leaf_bounds,
                           leaf_slices, leaves_over, perturb_policy, rel_err, run_gpu_update, single_step_oracle_grads)

pytestmark = pytest.mark.gpu

METRICS = {}


@pytest.fixture(scope="module", autouse=True)
def _dump_metrics():
    yield
    out = os.environ.get("MINPPO_TEST_METRICS_DIR")
    if not out:
        return
    try:
        os.makedirs(out, exist_ok=True)
        with open(os.path.join(out, "leaf_metrics.json"), "w") as f:
            json.dump(METRICS, f, indent=1, sort_keys=True)
    except OSError:
        pass


@pytest.fixture(scope="module")
def sm_count(cuda_device):
    import torch

    return torch.cuda.get_device_properties(cuda_device).multi_processor_count


def _run(hp, pr, device, monkeypatch, case, opt=None):
    if case.get("force_cap"):
        monkeypatch.setenv("MINPPO_FORCE_CAP", str(case["force_cap"]))      # read once, by the Learner's constructor
    try:
        return run_gpu_update(hp, pr, device, opt=opt, **case["cfg"])
    finally:
        monkeypatch.delenv("MINPPO_FORCE_CAP", raising=False)


def _check_path(case, hp_kw, sm_count, got):
    path = learner_path(hp_kw, case["D"], case["A"], sm_count, case["cfg"], case.get("force_cap"))
    for k, v in case["expect"].items():
        assert path[k] == v, (k, path)
    assert got["launches"] == path["launches"], path
    return path


# ---- (a) one step per case, per leaf ------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(CASES))
def test_single_step_gradient_per_leaf(name, cuda_device, sm_count, monkeypatch):
    case = CASES[name]
    hp = P.Hyper(**case["hp"])
    D, A, H, L = case["D"], case["A"], hp.hidden_size, hp.num_layers
    pr = synth.make_problem(hp, D, A, seed=9, done_p=0.02)
    perturb_policy(pr)
    got = _run(hp, pr, cuda_device, monkeypatch, case)
    path = _check_path(case, case["hp"], sm_count, got)

    ls64, g64 = single_step_oracle_grads(hp, pr, np.float64, "exact")
    lsbf, gbf = single_step_oracle_grads(hp, pr, np.float32, "bf16")
    e_bf, e_64 = compare_leaves(got["grad"], gbf, g64, D, A, H, L)
    m = {"path": {k: path[k] for k in ("fused", "maxu", "fast", "dw_nsplit", "S", "two_launch", "launches")},
         "max_leaf_vs_bf16": max(e_bf.values()), "max_leaf_vs_fp64": max(e_64.values()),
         "leaf_vs_bf16": e_bf, "leaf_vs_fp64": e_64,
         "loss_vs_bf16": rel_err(got["losses"][0, 0], np.array(lsbf))}
    METRICS["a/" + name] = m
    assert np.all(np.isfinite(got["grad"]))
    assert not leaves_over(e_bf, LEAF_BOUND_BF16), m
    assert not leaves_over(e_64, LEAF_BOUND_FP64, fp64_leaf_bounds(hp)), m
    assert m["loss_vs_bf16"] < 2e-3, m


# ---- (b) multi-step updates at learning rate 0 ----------------------------------------------------------------------
FROZEN = {
    # config 1 of BASELINE.json: 128 steps on 5-row minibatches, fused
    "c1": dict(hp=dict(num_envs=16, num_steps=10, num_minibatches=32, update_epochs=4), D=225, A=10, cfg={}),
    "layerwise_h512": dict(hp=dict(num_envs=25, num_steps=12, num_minibatches=3, update_epochs=2, hidden_size=512),
                           D=225, A=10, cfg={}),
    "padded": dict(hp=dict(num_envs=50, num_steps=16, num_minibatches=4, update_epochs=2), D=225, A=10, cfg={},
                   force_cap=520),
    "splits3": dict(hp=dict(num_envs=64, num_steps=16, num_minibatches=2, update_epochs=2), D=225, A=10,
                    cfg=dict(dw_splits=3)),
}


@pytest.mark.parametrize("name", list(FROZEN))
def test_frozen_parameter_update_every_step(name, cuda_device, sm_count, monkeypatch):
    """opt.lr = 0 (no annealing): Adam still reduces, clips and updates mu / nu at every step and rewrites the bf16
    weight images, but the parameters do not move, so every step of the update is evaluated at the initial parameters
    and can be held to the oracle as tightly as a single step."""
    case = dict(FROZEN[name])
    hp_kw = dict(case["hp"], anneal_lr=False, opt_lr=0.0)
    hp = P.Hyper(**hp_kw)
    D, A, H, L = case["D"], case["A"], hp.hidden_size, hp.num_layers
    case["cfg"] = dict(case["cfg"], fast_tanh=False)
    pr = synth.make_problem(hp, D, A, seed=5, done_p=0.02)
    perturb_policy(pr)
    got = _run(hp, pr, cuda_device, monkeypatch, case)
    path = learner_path(hp_kw, D, A, sm_count, case["cfg"], case.get("force_cap"))
    assert got["launches"] == path["launches"], path
    if name == "splits3":
        assert path["S"] == 3
    if name == "layerwise_h512":
        assert not path["fused"]

    p64, o64, rng64, l64, aux64 = P.update(P.tree_like(pr["params"], lambda x: x.astype(np.float64)),
                                           P.init_opt_state(P.tree_like(pr["params"], lambda x: x.astype(np.float64))),
                                           pr["traj"], pr["last_val"], pr["rng"], hp, dtype=np.float64, gemm="exact")
    p0 = P.tree_like(pr["params"], lambda x: x.astype(np.float32))
    pbf, obf, _, lbf, auxbf = P.update(p0, P.init_opt_state(p0), pr["traj"], pr["last_val"], pr["rng"], hp,
                                       dtype=np.float32, gemm="bf16", perms=aux64["perms"])
    EM = hp.update_epochs * hp.num_minibatches
    flat0 = P.flatten_params(pr["params"], L)
    assert np.array_equal(got["params"].view(np.uint32), flat0.view(np.uint32))
    assert got["step"] == EM == o64["count"]
    assert np.array_equal(got["perms"], aux64["perms"])
    assert np.array_equal(got["rng"], rng64)

    # the last step's gradient: the last minibatch of the last epoch, at the initial parameters
    mbs = hp.minibatch_size
    rows = aux64["perms"][-1][(hp.num_minibatches - 1) * mbs:]

    def last_grads(dtype, gemm):
        adv, tgt = P.gae(pr["traj"]["reward"], pr["traj"]["value"], pr["traj"]["done"], pr["last_val"], hp.gamma,
                         hp.gae_lambda, dtype)
        flat = P.flatten_traj({"obs": pr["traj"]["obs"].astype(dtype), "action": pr["traj"]["action"].astype(dtype),
                               "value": pr["traj"]["value"].astype(dtype),
                               "log_prob": pr["traj"]["log_prob"].astype(dtype), "adv": adv, "tgt": tgt})
        return P.loss_and_grads(P.tree_like(pr["params"], lambda x: x.astype(dtype)),
                                {k: v[rows] for k, v in flat.items()}, hp, gemm)[1]

    e_bf, e_64 = compare_leaves(got["grad"], last_grads(np.float32, "bf16"), last_grads(np.float64, "exact"), D, A, H, L)
    mu_err = {n: rel_err(got["mu"][s], flat_grads(obf["mu"], L)[s]) for n, s in leaf_slices(D, A, H, L)}
    nu_err = {n: rel_err(got["nu"][s], flat_grads(obf["nu"], L)[s]) for n, s in leaf_slices(D, A, H, L)}
    m = {"loss_vs_bf16": rel_err(got["losses"], lbf), "loss_vs_fp64": rel_err(got["losses"], l64),
         "gnorm_vs_bf16": rel_err(got["grad_norms"], auxbf["grad_norms"]),
         "max_leaf_vs_bf16": max(e_bf.values()), "max_leaf_vs_fp64": max(e_64.values()),
         "leaf_vs_bf16": e_bf, "leaf_vs_fp64": e_64, "max_mu_leaf": max(mu_err.values()),
         "max_nu_leaf": max(nu_err.values()), "mu_leaf": mu_err, "nu_leaf": nu_err, "launches": got["launches"]}
    METRICS["b/" + name] = m
    assert m["loss_vs_bf16"] < 1e-5, m
    assert m["gnorm_vs_bf16"] < 1e-3, m
    assert not leaves_over(e_bf, LEAF_BOUND_BF16), m
    assert not leaves_over(e_64, LEAF_BOUND_FP64, fp64_leaf_bounds(hp)), m
    assert not leaves_over(mu_err, 5e-3), m
    assert not leaves_over(nu_err, 1e-2), m


# ---- (c) clip + Adam in float64 on the GPU's own gradient -----------------------------------------------------------
# one shape per optimizer path; 32-row batches unless the path needs more rows
OPT_PATHS = {
    "dwopt1": dict(hp=dict(num_envs=8, num_steps=4, hidden_size=256), D=225, A=10, cfg={},
                   expect=dict(two_launch=False, maxu=1, fast=True)),
    "dwopt2": dict(hp=dict(num_envs=8, num_steps=4, hidden_size=256), D=415, A=20, cfg={},
                   expect=dict(two_launch=False, maxu=2, fast=True)),
    "dwopt4_fast": dict(hp=dict(num_envs=8, num_steps=4, hidden_size=256), D=1000, A=10, cfg={},
                        expect=dict(two_launch=False, maxu=4, fast=True)),
    "dwopt4_nonfast": dict(hp=dict(num_envs=8, num_steps=4, hidden_size=512), D=1000, A=64, cfg={},
                           expect=dict(two_launch=False, maxu=4, fast=False)),
    # 4 splits need 4 k-blocks: 256 rows
    "two_launch": dict(hp=dict(num_envs=32, num_steps=8, hidden_size=256), D=1000, A=10, cfg=dict(dw_splits=4),
                       expect=dict(two_launch=True)),
}


@pytest.mark.parametrize("mode", ["noclip", "clip", "resumed"])
@pytest.mark.parametrize("name", list(OPT_PATHS))
def test_optimizer_step_matches_fp64_on_the_gpu_gradient(name, mode, cuda_device, sm_count, monkeypatch):
    """E = M = 1: the gradient the optimizer consumed is read back (P + 2 loss sums), and clip_by_global_norm + Adam are
    recomputed in float64 from the same float32 inputs.  What remains is the kernels' float32 rounding."""
    case = dict(OPT_PATHS[name])
    B = case["hp"]["num_envs"] * case["hp"]["num_steps"]
    hp_kw = dict(case["hp"], num_minibatches=1, update_epochs=1, anneal_lr=False,
                 max_grad_norm=1e-3 if mode == "clip" else 1e6)
    count = 0
    if mode == "resumed":
        # the schedule divides the step count by mb * E (train.py:100): 37 steps of a 32-row minibatch are one past
        # the first schedule boundary; larger minibatches start one boundary later
        count = 37 if B <= 37 else B + 37
        hp_kw.update(anneal_lr=True, total_timesteps=4 * B)
    hp = P.Hyper(**hp_kw)
    D, A, H, L = case["D"], case["A"], hp.hidden_size, hp.num_layers
    if mode == "resumed":
        frac = 1.0 - (count // (hp.minibatch_size * hp.update_epochs)) / hp.num_updates
        assert 0.0 < frac < 1.0
    pr = synth.make_problem(hp, D, A, seed=3, done_p=0.02)
    perturb_policy(pr)
    Pn = P.flatten_params(pr["params"], L).size
    g = np.random.default_rng(17)
    if mode == "resumed":
        mu0 = (1e-3 * g.standard_normal(Pn)).astype(np.float32)
        nu0 = g.uniform(0.0, 1e-6, Pn).astype(np.float32)
    else:
        mu0 = np.zeros(Pn, np.float32)
        nu0 = np.zeros(Pn, np.float32)
    got = _run(hp, pr, cuda_device, monkeypatch, case, opt={"count": count, "mu": mu0, "nu": nu0})
    _check_path(case, hp_kw, sm_count, got)

    p_in = P.flatten_params(pr["params"], L)
    gflat = got["grad"]
    gnorm_gpu = float(got["grad_norms"][0, 0])
    p_ref, mu_ref, nu_ref, gnorm_ref = clip_adam_flat(p_in, gflat[:Pn], mu0, nu0, count, hp)
    # the restatement is optax's chain as the oracle states it
    unflat = lambda x: P.unflatten_params(np.asarray(x, np.float64), D, A, H, L)
    tp, to, tn = P.clip_adam_step(unflat(p_in), unflat(gflat[:Pn]), {"count": count, "mu": unflat(mu0), "nu": unflat(nu0)},
                                  hp)
    assert np.allclose(P.flatten_params(tp, L, np.float64), p_ref, rtol=1e-12, atol=0)
    assert np.allclose(P.flatten_params(to["mu"], L, np.float64), mu_ref, rtol=1e-12, atol=0)
    assert abs(tn - gnorm_ref) <= 1e-12 * gnorm_ref
    # which branch of clip_by_global_norm ran
    assert (gnorm_gpu >= hp.max_grad_norm) == (mode == "clip")

    lr = abs(float(P.learning_rate(count, hp, np.float64)))
    ulp = np.spacing(np.abs(p_ref).astype(np.float32)).astype(np.float64)
    dp = np.abs(got["params"].astype(np.float64) - p_ref)
    # + 2e-5 of the step itself: the kernels take the Adam constants as float32, and 0.999f is 0.999 + 1.3e-8, so the
    # bias correction 1 - b2^(count + 1) carries (count + 1) x that rounding: 1.3e-5 relative at count = 37, 6.3e-6 in the
    # step.  Where nu is small (resumed state) the step reaches ~40 lr: measured 2.7e-4 lr off the float64 step there.
    step = np.abs(p_ref - p_in.astype(np.float64))
    p_excess = dp / (2 * ulp + 1e-4 * lr + 2e-5 * step)
    mu_tol = np.empty(Pn)
    nu_tol = np.empty(Pn)
    for _, s in leaf_slices(D, A, H, L):
        mu_tol[s] = 1e-5 * np.abs(mu_ref[s]) + 1e-6 * np.abs(mu_ref[s]).max()
        nu_tol[s] = 1e-5 * np.abs(nu_ref[s]) + 1e-6 * np.abs(nu_ref[s]).max()
    mu_excess = np.abs(got["mu"] - mu_ref) / mu_tol
    nu_excess = np.abs(got["nu"] - nu_ref) / nu_tol

    # losses: from the two loss sums the kernels reduced next to the gradient, and the pre-update log_std
    mb = hp.minibatch_size
    value_loss = 0.5 * float(gflat[Pn]) / mb
    actor_loss = -float(gflat[Pn + 1]) / mb
    log_std = np.asarray(pr["params"]["params"]["log_std"], np.float64)
    entropy = A * (0.5 + 0.5 * np.log(2 * np.pi)) + np.log(np.abs(np.exp(log_std))).sum()
    total = actor_loss + hp.vf_coef * value_loss - hp.ent_coef * entropy
    loss_scale = max(abs(total), abs(actor_loss), hp.vf_coef * abs(value_loss), hp.ent_coef * abs(entropy))
    lgpu = got["losses"][0, 0].astype(np.float64)
    m = {"gnorm_rel": abs(gnorm_gpu - gnorm_ref) / gnorm_ref, "gnorm": gnorm_gpu, "lr": lr,
         "param_max_ulp": float((dp / ulp).max()), "param_max_in_lr": float(dp.max() / lr),
         "param_max_over_bound": float(p_excess.max()),
         "mu_max_rel": float((np.abs(got["mu"] - mu_ref) / np.maximum(np.abs(mu_ref), 1e-30)).max()),
         "mu_max_over_bound": float(mu_excess.max()), "nu_max_over_bound": float(nu_excess.max()),
         "total_loss_rel": abs(lgpu[0] - total) / loss_scale,
         "loss_cols_rel": [abs(lgpu[1] - value_loss) / abs(value_loss), abs(lgpu[2] - actor_loss) / abs(actor_loss),
                           abs(lgpu[3] - entropy) / abs(entropy)]}
    METRICS[f"c/{name}/{mode}"] = m
    assert got["step"] == count + 1
    assert m["gnorm_rel"] <= 1e-5, m
    assert m["param_max_over_bound"] <= 1.0, m
    assert m["mu_max_over_bound"] <= 1.0, m
    assert m["nu_max_over_bound"] <= 1.0, m
    # total = actor + vf * value - ent * entropy, relative to the largest of its terms (a sum is exact to its terms' ulp)
    assert m["total_loss_rel"] <= 1e-6, m
    assert max(m["loss_cols_rel"]) <= 1e-6, m
