"""Reference for the per-minibatch statistics of ``Learner.update(..., stats=...)`` (include/minppo_b200.h,
minppo_update_with_stats): the oracle's update loop (oracle/ppo_numpy.py ``update``) restated step for step with the
same primitives, plus, per minibatch step, the four statistics evaluated in that step's forward pass (parameters
before the step's Adam update):

    approx_kl            mean(expm1(log r) - log r)       r = exp(logp_new - logp_old)
    clip_fraction        mean(|r - 1| > clip_eps)
    value_clip_fraction  mean(|v - v_old| > clip_eps)
    grad_norm            the pre-clip global gradient norm of clip_adam_step

``update_with_stats`` returns exactly what ``P.update`` returns (the same calls in the same order: bit-identical), with
``aux["stats"]`` [E, M, 4] and ``aux["ambiguous"]`` [E, M, 2] added: the rows whose |r - 1| (column 0) or |v - v_old|
(column 1) lies within ``delta`` of clip_eps, whose clip indicator another implementation's rounding may flip."""
from __future__ import annotations

import numpy as np

from oracle import ppo_numpy as P
from oracle import threefry

STATS_COLUMNS = ("approx_kl", "clip_fraction", "value_clip_fraction", "grad_norm")


def minibatch_stats(params, mb, hp: P.Hyper, gemm="exact", delta: float = 0.0):
    """(approx_kl, clip_fraction, value_clip_fraction, ambiguous ratio rows, ambiguous value rows) of one minibatch,
    from the same forward pass and log-prob arithmetic as ``P.loss_and_grads``."""
    dt = mb["obs"].dtype.type
    eps = dt(hp.clip_eps)
    mean, log_std, v, _ = P.actor_critic_forward(params, mb["obs"], hp, gemm)
    logp, _, _ = P.gaussian_log_prob(mean, log_std, mb["action"])
    logr = logp - mb["log_prob"]
    ratio = np.exp(logr)
    dr = np.abs(ratio - dt(1.0))
    dv = np.abs(v - mb["value"])
    kl = (np.expm1(logr) - logr).mean()
    return (kl, (dr > eps).mean(), (dv > eps).mean(),
            int((np.abs(dr - eps) <= delta).sum()), int((np.abs(dv - eps) <= delta).sum()))


def update_with_stats(params, opt, traj, last_val, rng, hp: P.Hyper, dtype=np.float64, gemm="exact", perms=None,
                      delta: float = 0.0):
    cast = lambda x: np.asarray(x, dtype)
    params = P.tree_like(params, cast)
    opt = {"count": int(opt["count"]), "mu": P.tree_like(opt["mu"], cast), "nu": P.tree_like(opt["nu"], cast)}
    adv, tgt = P.gae(traj["reward"], traj["value"], traj["done"], last_val, hp.gamma, hp.gae_lambda, dtype)
    flat = P.flatten_traj({"obs": cast(traj["obs"]), "action": cast(traj["action"]),
                           "value": cast(traj["value"]), "log_prob": cast(traj["log_prob"]),
                           "adv": adv, "tgt": tgt})
    B, M, mbs = hp.batch_size, hp.num_minibatches, hp.minibatch_size
    if mbs * M != B:
        raise ValueError("`batch_size` must be equal to `num_steps * num_envs`")
    rng = np.asarray(rng, np.uint32)
    losses = np.zeros((hp.update_epochs, M, 4), dtype)
    gnorms = np.zeros((hp.update_epochs, M), dtype)
    stats = np.zeros((hp.update_epochs, M, 4), dtype)
    ambiguous = np.zeros((hp.update_epochs, M, 2), np.int64)
    used_perms = []
    for e in range(hp.update_epochs):
        rng, sub = threefry.split(rng, 2, hp.prng_mode)
        perm = threefry.permutation(sub, B, hp.prng_mode) if perms is None else perms[e]
        used_perms.append(perm)
        for k in range(M):
            idx = perm[k * mbs:(k + 1) * mbs]
            mb = {name: arr[idx] for name, arr in flat.items()}
            kl, cf, vcf, amb_r, amb_v = minibatch_stats(params, mb, hp, gemm, delta)
            ls, grads = P.loss_and_grads(params, mb, hp, gemm)
            params, opt, gn = P.clip_adam_step(params, grads, opt, hp)
            losses[e, k] = ls
            gnorms[e, k] = gn
            stats[e, k] = (kl, cf, vcf, gn)
            ambiguous[e, k] = (amb_r, amb_v)
    aux = {"advantages": adv, "targets": tgt, "perms": np.stack(used_perms), "grad_norms": gnorms, "stats": stats,
           "ambiguous": ambiguous}
    return params, opt, rng, losses, aux
