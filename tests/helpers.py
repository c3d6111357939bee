"""Shared glue for the parity tests: oracle Hyper <-> product Config, running one update through
the C ABI (via minppo_b200.learner) and collecting everything as NumPy."""
from __future__ import annotations

import numpy as np

from oracle import ppo_numpy as P
from oracle import threefry


def hyper_to_config(hp: P.Hyper, fast_tanh: bool = True, use_graph: bool = True, dw_splits: int = 0, fused: bool = True):
    from minppo_b200.config import Config

    c = Config()
    c.model.hidden_size, c.model.num_layers, c.model.use_tanh = hp.hidden_size, hp.num_layers, hp.use_tanh
    c.opt.lr, c.opt.max_grad_norm = hp.opt_lr, hp.max_grad_norm
    c.rl.num_env_steps, c.rl.gamma, c.rl.gae_lambda = hp.num_steps, hp.gamma, hp.gae_lambda
    c.rl.clip_eps, c.rl.ent_coef, c.rl.vf_coef = hp.clip_eps, hp.ent_coef, hp.vf_coef
    c.training.lr, c.training.num_envs, c.training.total_timesteps = hp.training_lr, hp.num_envs, hp.total_timesteps
    c.training.num_minibatches, c.training.num_steps = hp.num_minibatches, hp.num_steps
    c.training.update_epochs, c.training.anneal_lr = hp.update_epochs, hp.anneal_lr
    c.learner.prng_mode = "legacy" if hp.prng_mode == threefry.LEGACY else "partitionable"
    c.learner.fast_tanh, c.learner.use_graph, c.learner.dw_splits = fast_tanh, use_graph, dw_splits
    c.learner.fused = fused
    return c


def run_gpu_update(hp: P.Hyper, problem, device, opt=None, **cfg_kw):
    """One update on the GPU.  Returns dict of NumPy arrays: params (flat), mu, nu, step, rng,
    losses [E,M,4], advantages, targets, perms, grad (last minibatch, flat P+4), grad_norms.
    ``opt``: optimizer state to start from, {"count", "mu", "nu"} with trees or flat arrays."""
    import torch

    from minppo_b200.learner import Learner, Memory, TrainState

    cfg = hyper_to_config(hp, **cfg_kw)
    D, A = problem["obs_dim"], problem["act_dim"]
    learner = Learner(cfg, D, A, device)
    flat = P.flatten_params(problem["params"], hp.num_layers)
    ts = TrainState.create(flat, device)
    if opt is not None:
        as_flat = lambda x: np.asarray(x, np.float32) if isinstance(x, np.ndarray) else P.flatten_params(x, hp.num_layers)
        ts.mu.copy_(torch.as_tensor(as_flat(opt["mu"])))
        ts.nu.copy_(torch.as_tensor(as_flat(opt["nu"])))
        ts.step.fill_(int(opt["count"]))
    tr = problem["traj"]
    t = lambda x: torch.as_tensor(np.ascontiguousarray(x)).to(device)
    mem = Memory(done=t(tr["done"]), action=t(tr["action"]), value=t(tr["value"]), reward=t(tr["reward"]),
                 log_prob=t(tr["log_prob"]), obs=t(tr["obs"]))
    rng = torch.as_tensor(problem["rng"].view(np.int32)).to(device)
    ts, rng_out, losses = learner.update(ts, mem, t(problem["last_val"]), rng)
    learner.check()
    out = {
        "params": ts.params.cpu().numpy(), "mu": ts.mu.cpu().numpy(), "nu": ts.nu.cpu().numpy(),
        "step": int(ts.step.item()), "rng": rng_out.cpu().numpy().view(np.uint32), "losses": losses.cpu().numpy(),
        "advantages": learner.read("advantages").cpu().numpy(), "targets": learner.read("targets").cpu().numpy(),
        "perms": learner.read("perms").cpu().numpy(), "grad": learner.read("grad").cpu().numpy(),
        "grad_norms": learner.read("grad_norms").cpu().numpy().reshape(hp.update_epochs, hp.num_minibatches),
        "launches": learner.launches_per_update(),
    }
    learner.close()
    return out


def flat_grads(grads, num_layers: int) -> np.ndarray:
    return P.flatten_params(grads, num_layers, np.float64)


def rel_err(a, b) -> float:
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


# ---- per-leaf gradient comparator ---------------------------------------------------------------
# The output heads carry ~99.9% of the gradient norm and the largest entries, so an error relative to the WHOLE
# gradient cannot see the hidden layers (their leaves are ~1e-4 of the largest entry).  Each leaf is held to its own scale.
LEAF_BOUND_BF16 = 5e-3       # against the oracle with the kernels' bf16 rounding points (float32, gemm="bf16")
LEAF_BOUND_FP64 = 5e-2       # against the exact float64 oracle


def fp64_leaf_bounds(hp: P.Hyper) -> dict:
    """Per-leaf bounds against the float64 oracle where bf16 rounding ALONE costs more than LEAF_BOUND_FP64: the oracle
    with the kernels' rounding points (float32, gemm="bf16") is that far from the exact one on the CPU
    (tests/test_gradient_check_host.py holds it to these bounds).  Hidden-layer gradients are sums over rows with
    cancelling signs, so a few discrete flips move them by a large fraction of their (small) result:
    * relu layers (the critic always; the actor with model.use_tanh = false): a pre-activation within bf16 rounding of 0
      flips relu'.  Measured up to 0.20 at 65 to 2,048 rows (critic Dense_1/kernel, D = 415 / A = 20), 0.44 on the
      5-row minibatches of config 1 (critic Dense_1/bias);
    * a narrow clip (rl.clip_eps = 0.05): rows whose probability ratio is within rounding of 1 +- eps change clip branch
      and drop their whole actor gradient (or regain it), every actor leaf included.  Measured up to 0.16 (actor
      Dense_0/kernel).
    A dropped or doubled contribution, a sign error or a zero leaf still fails these; the per-leaf bound against the
    emulating oracle (LEAF_BOUND_BF16) is the tight check of the same leaves."""
    out = {}
    for pth in P.leaf_order(hp.num_layers):
        name = "/".join(pth)
        hidden = pth[0] != "log_std" and pth[1] != f"Dense_{hp.num_layers}"
        relu = pth[0] == "MLP_1" or (pth[0] == "MLP_0" and not hp.use_tanh)
        if (hidden and relu) or (hp.clip_eps < 0.1 and pth[0] != "MLP_1"):
            out[name] = 0.5
    return out


def leaf_slices(D: int, A: int, H: int, L: int):
    """[("MLP_0/Dense_0/bias", slice), ...] over the flat arena, in P.leaf_order."""
    out, off = [], 0
    for pth, shp in zip(P.leaf_order(L), P.leaf_shapes(D, A, H, L)):
        n = int(np.prod(shp))
        out.append(("/".join(pth), slice(off, off + n)))
        off += n
    return out


def leaf_errors(g, ref_tree, D: int, A: int, H: int, L: int) -> dict:
    """max|g - ref| / max|ref| over each leaf.  g: flat gradient (at least P entries); ref_tree: an oracle gradient tree."""
    g = np.asarray(g, np.float64)
    ref = flat_grads(ref_tree, L)
    return {name: rel_err(g[s], ref[s]) for name, s in leaf_slices(D, A, H, L)}


def compare_leaves(g, tree_bf16, tree_fp64, D: int, A: int, H: int, L: int):
    """(err_bf16, err_fp64): per-leaf errors of a flat gradient against the bf16-emulating and the exact oracle."""
    return leaf_errors(g, tree_bf16, D, A, H, L), leaf_errors(g, tree_fp64, D, A, H, L)


def leaves_over(errs: dict, bound: float, overrides: dict | None = None) -> dict:
    """The leaves whose error exceeds ``bound`` (or the leaf's entry in ``overrides``)."""
    overrides = overrides or {}
    return {k: v for k, v in errs.items() if not v <= overrides.get(k, bound)}


def single_step_oracle_grads(hp: P.Hyper, pr, dtype, gemm, rows=None):
    """Losses and gradient tree of the first minibatch step of an update with E = M = 1: the whole batch in the order of
    the first epoch's permutation.  ``rows``: positions in that order to keep (the rest are dropped, with the mean and
    the advantage statistics of the full minibatch kept), for building a gradient with rows missing."""
    p0 = P.tree_like(pr["params"], lambda x: x.astype(dtype))
    adv, tgt = P.gae(pr["traj"]["reward"], pr["traj"]["value"], pr["traj"]["done"], pr["last_val"], hp.gamma,
                     hp.gae_lambda, dtype)
    flat = P.flatten_traj({"obs": pr["traj"]["obs"].astype(dtype), "action": pr["traj"]["action"].astype(dtype),
                           "value": pr["traj"]["value"].astype(dtype), "log_prob": pr["traj"]["log_prob"].astype(dtype),
                           "adv": adv, "tgt": tgt})
    _, sub = threefry.split(pr["rng"], 2, hp.prng_mode)
    perm = threefry.permutation(sub, hp.batch_size, hp.prng_mode)
    mb = {k: v[perm] for k, v in flat.items()}
    if rows is None:
        return P.loss_and_grads(p0, mb, hp, gemm)
    a = mb["adv"]
    return P.loss_and_grads(p0, {k: v[rows] for k, v in mb.items()}, hp, gemm, n_total=a.shape[0],
                            adv_mean_std=(a.mean(), a.std()))


def perturb_policy(pr, seed: int = 1) -> None:
    """Move log_prob and value of the trajectory off the policy's own (0.3 N(0, 1)), so that ratio != 1 and the
    clipped branches of both losses are taken."""
    g = np.random.default_rng(seed)
    tr = pr["traj"]
    tr["log_prob"] = (tr["log_prob"] + 0.3 * g.standard_normal(tr["log_prob"].shape)).astype(np.float32)
    tr["value"] = (tr["value"] + 0.3 * g.standard_normal(tr["value"].shape)).astype(np.float32)


def clip_adam_flat(p, g, mu, nu, count: int, hp: P.Hyper):
    """optax.chain(clip_by_global_norm(max_grad_norm), adam(lr, b1, b2, eps, eps_root)) and apply_updates on flat
    float64 arrays, with the learning-rate schedule of train.py:98-101 at ``count`` (the step count before this step).
    Returns (params', mu', nu', grad_norm)."""
    f = np.float64
    p, g, mu, nu = (np.asarray(x, f) for x in (p, g, mu, nu))
    g_norm = np.sqrt(np.sum(g * g))
    if not g_norm < hp.max_grad_norm:
        g = (g / g_norm) * f(hp.max_grad_norm)
    lr = P.learning_rate(count, hp, f)
    c1 = 1.0 - f(hp.b1) ** f(count + 1)
    c2 = 1.0 - f(hp.b2) ** f(count + 1)
    mu = (1.0 - f(hp.b1)) * g + f(hp.b1) * mu
    nu = (1.0 - f(hp.b2)) * (g * g) + f(hp.b2) * nu
    u = (mu / c1) / (np.sqrt(nu / c2 + f(hp.eps_root)) + f(hp.eps))
    return p + (-lr) * u, mu, nu, g_norm
