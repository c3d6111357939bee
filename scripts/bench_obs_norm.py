"""Cost of running observation normalization (``Learner.update(..., obs_norm=...)``, ``policy_step(..., obs_norm=...)``).

    python scripts/bench_obs_norm.py [--rounds 5] [--steps 20] [--warmup 3] [--policy-iters 200]

configs[1] of bench.py (2048 envs x 128 steps, 256x256 MLPs, 4 epochs x 32 minibatches) at D = 225 / A = 10 and
D = 415 / A = 20, one learner context per shape:
* ms per update without and with normalization, alternating in one process: `rounds` rounds, each timing `steps`
  updates of each mode (graph replays between CUDA events; the statistics keep folding, as in training);
* the two branches of the update's fork, from one eager profiled update per mode (minppo_ctx_profile: the branch runs
  serialised there, so each class time is that of its launches alone): the GAE -> permutation -> row-list chain
  (classes gae, perm_sort, rows_and_adv_stats) against the operand images (obs_image, which with normalization also
  holds the finalize and merge launches, and weight_images);
* the rollout policy step (sampled) at 2048 envs without and with normalization, µs per call (CUDA events around
  `policy-iters` calls, alternating, `rounds` rounds).
Prints one JSON line per shape with medians, per-round values, the card name and power limit read in the same run, and
a parity flag (the normalized update equals the update on observations normalized on the host).  Writes nothing."""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import BenchShape, make_config, synth_shard  # noqa: E402
from scripts.bench_update_stats import card  # noqa: E402
from tests.obs_norm_reference import normalize_obs  # noqa: E402


def med(v):
    return {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v)),
            "per_round": [round(x, 4) for x in v]}


def one_shape(D, A, args, dev):
    import torch

    from minppo_b200 import _lib
    from minppo_b200.learner import Learner, Memory, TrainState
    from minppo_b200.obs_norm import ObsNormalizer
    from minppo_b200.params import flatten_params

    hp = BenchShape(num_envs=2048, num_steps=128, num_minibatches=32, update_epochs=4)
    learner = Learner(make_config(hp, True), D, A, dev)
    params, traj, last_val = synth_shard(hp, 0, 1, dims=(D, A))
    flat = flatten_params(params, hp.num_layers)
    t = lambda x: torch.as_tensor(np.ascontiguousarray(x)).to(dev)
    obs = (1.0 + 2.0 * traj["obs"]).astype(np.float32)       # statistics away from the initial state
    mem = Memory(done=t(traj["done"]), action=t(traj["action"]), value=t(traj["value"]), reward=t(traj["reward"]),
                 log_prob=t(traj["log_prob"]), obs=t(obs))
    lv = t(last_val)
    rng = torch.tensor([0, 1337], dtype=torch.int32, device=dev)
    rng_out = torch.empty_like(rng)
    losses = torch.empty((hp.update_epochs, hp.num_minibatches, 4), dtype=torch.float32, device=dev)
    norm = ObsNormalizer.create(D, dev)
    norm.fold(mem.obs)                                      # warm-up fold: non-trivial statistics

    # parity: normalized update == update on host-normalized observations, from the same state
    out = []
    s0 = [x.clone() for x in (norm.mean, norm.var, norm.count)]
    m, v = norm.mean.cpu().numpy(), norm.var.cpu().numpy()
    mem_pre = mem._replace(obs=t(normalize_obs(obs, m, v, norm.eps, norm.clip)))
    for memb, nrm in ((mem, norm), (mem_pre, None)):
        ts = TrainState.create(flat, dev)
        learner.update(ts, memb, lv, rng, losses, rng_out, obs_norm=nrm)
        out.append((losses.clone(), ts.params.clone()))
    learner.check()
    same = bool(torch.equal(out[0][0], out[1][0]) and torch.equal(out[0][1], out[1][1]))
    del mem_pre
    for x, y in zip((norm.mean, norm.var, norm.count), s0):
        x.copy_(y)

    ts = TrainState.create(flat, dev)
    modes = {"plain": None, "obs_norm": norm}
    launches = {}
    for k, nrm in modes.items():
        for _ in range(max(args.warmup, 3)):
            learner.update(ts, mem, lv, rng, losses, rng_out, obs_norm=nrm)
        launches[k] = learner.launches_per_update()
    torch.cuda.synchronize(dev)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = {k: [] for k in modes}
    for _ in range(args.rounds):
        for k, nrm in modes.items():
            ev0.record()
            for _ in range(args.steps):
                learner.update(ts, mem, lv, rng, losses, rng_out, obs_norm=nrm)
            ev1.record()
            torch.cuda.synchronize(dev)
            times[k].append(ev0.elapsed_time(ev1) / args.steps)

    # branch lengths of the fork, from one eager profiled update per mode
    n = len(_lib.PROFILE_CLASSES)
    branches = {}
    learner.use_graph = False
    for k, nrm in modes.items():
        learner.lib.minppo_ctx_profile(learner._h, 1)
        learner.update(ts, mem, lv, rng, losses, rng_out, obs_norm=nrm)
        msv, cnt = (C.c_float * n)(), (C.c_int32 * n)()
        _lib.check(learner.lib.minppo_ctx_profile_read(learner._h, msv, cnt, n))
        learner.lib.minppo_ctx_profile(learner._h, 0)
        cls = dict(zip(_lib.PROFILE_CLASSES, (float(x) for x in msv)))
        branches[k] = {"chain_ms (gae + perm_sort + rows_and_adv_stats)":
                       cls["gae"] + cls["perm_sort"] + cls["rows_and_adv_stats"],
                       "images_ms (obs_image + weight_images)": cls["obs_image"] + cls["weight_images"],
                       "obs_image_ms": cls["obs_image"]}
    learner.use_graph = True

    # rollout policy step at 2048 envs (sampled)
    o = mem.obs[0].contiguous()
    ptimes = {k: [] for k in modes}
    for k, nrm in modes.items():
        for _ in range(10):
            learner.policy_step(ts.params, o, rng, weights_current=True, obs_norm=nrm)
    torch.cuda.synchronize(dev)
    for _ in range(args.rounds):
        for k, nrm in modes.items():
            ev0.record()
            for _ in range(args.policy_iters):
                learner.policy_step(ts.params, o, rng, weights_current=True, obs_norm=nrm)
            ev1.record()
            torch.cuda.synchronize(dev)
            ptimes[k].append(ev0.elapsed_time(ev1) * 1e3 / args.policy_iters)
    learner.check()
    learner.close()
    return {
        "workload": f"configs[1]: 2048 envs x 128 steps, 256x256 MLPs, 4 epochs x 32 minibatches, D={D}/A={A}",
        "timing": f"CUDA events around {args.steps} graph replays per mode and round, {args.rounds} rounds, alternating",
        "update_ms": {k: med(v) for k, v in times.items()},
        "update_median_diff_ms": float(np.median(times["obs_norm"]) - np.median(times["plain"])),
        "launches_per_update": launches,
        "fork_branches_eager_profile": branches,
        "policy_step_us_2048_envs": {k: med(v) for k, v in ptimes.items()},
        "normalized_update_equals_prenormalized": same,
    }


def main():
    import torch

    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--policy-iters", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_obs_norm.py needs a CUDA device")
    dev = torch.device("cuda:0")
    for D, A in ((225, 10), (415, 20)):
        print(json.dumps({**one_shape(D, A, args, dev), "card": card()}), flush=True)


if __name__ == "__main__":
    main()
