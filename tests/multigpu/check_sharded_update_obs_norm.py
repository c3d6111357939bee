"""Observation normalization in the env-sharded learner update (run under torchrun on a box with >= 2 B200s;
tests/test_gpu_obs_norm.py drives it):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29617 \
        tests/multigpu/check_sharded_update_obs_norm.py

Every rank runs two normalized updates on its shard of ONE global batch (the second replays the captured graph), over
the peer-memory exchange and over ncclAllReduce (MINPPO_NCCL_ALLREDUCE=1); rank 0 also runs them on one GPU over the
whole batch.  Checks: the statistics are bit-identical on every rank and within the tolerances of
tests/test_gpu_obs_norm.py of the float64 fold of the global batch; the parameters are bit-identical on every rank and
equal the single-GPU ones with the tolerances of tests/multigpu/check_sharded_update.py."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from minppo_b200.learner import Learner, Memory, TrainState, nccl_unique_id  # noqa: E402
from oracle import ppo_numpy as P  # noqa: E402
from oracle import synth  # noqa: E402
from tests.helpers import hyper_to_config, rel_err  # noqa: E402
from tests.obs_norm_reference import fold_obs_stats  # noqa: E402
from tests.test_gpu_obs_norm import check_fold, make_stats  # noqa: E402

MODES = {"peer": {}, "nccl": {"MINPPO_NCCL_ALLREDUCE": "1"}}


def run(hp, pr, dev, world, rank, nccl_id, n0, Nl):
    learner = Learner(hyper_to_config(hp), pr["obs_dim"], pr["act_dim"], dev, world, rank, nccl_id)
    ts = TrainState.create(P.flatten_params(pr["params"], hp.num_layers), dev)
    t = lambda x: torch.as_tensor(np.ascontiguousarray(x)).to(dev)
    tr = {k: v[:, n0:n0 + Nl] for k, v in pr["traj"].items()}
    mem = Memory(done=t(tr["done"]), action=t(tr["action"]), value=t(tr["value"]), reward=t(tr["reward"]),
                 log_prob=t(tr["log_prob"]), obs=t(tr["obs"]))
    rng = torch.as_tensor(pr["rng"].view(np.int32)).to(dev)
    S = make_stats(pr["obs_dim"], dev)
    for _ in range(2):
        ts, rng_out, losses = learner.update(ts, mem, t(pr["last_val"][n0:n0 + Nl]), rng, obs_norm=S)
    learner.check()
    stats = torch.cat([S.mean.double(), S.var.double(), S.count])
    out = {"params": ts.params.clone(), "losses": losses.cpu().numpy(), "stats": stats}
    learner.close()
    return out


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    dist.init_process_group("nccl", device_id=dev)
    hp = P.Hyper(num_envs=64 * world, num_steps=32, num_minibatches=4, update_epochs=2, anneal_lr=False)
    pr = synth.make_problem(hp, seed=3)
    g = np.random.default_rng(5)
    pr["traj"]["obs"] = (1.5 + 2.0 * g.standard_normal(pr["traj"]["obs"].shape)).astype(np.float32)
    D = pr["obs_dim"]
    Nl = hp.num_envs // world
    ref = None
    if rank == 0:
        ref = run(hp, pr, dev, 1, 0, None, 0, hp.num_envs)
        S0 = make_stats(D, dev)
        m, v, c = S0.mean.cpu().numpy(), S0.var.cpu().numpy(), float(S0.count.item())
        for _ in range(2):
            m, v, c = fold_obs_stats(m, v, c, pr["traj"]["obs"])
            m, v = m.astype(np.float32), v.astype(np.float32)       # stored as f32 between updates
        want = (m.astype(np.float64), v.astype(np.float64), c)
    ok = True
    for mode, env in MODES.items():
        saved = {k: os.environ.get(k) for k in env}
        os.environ.update(env)
        ids = [nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        got = run(hp, pr, dev, world, rank, ids[0], rank * Nl, Nl)
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k)
            else:
                os.environ[k] = v
        alls = [torch.empty_like(got["stats"]) for _ in range(world)]
        dist.all_gather(alls, got["stats"])
        allp = [torch.empty_like(got["params"]) for _ in range(world)]
        dist.all_gather(allp, got["params"])
        if rank == 0:
            st = got["stats"].cpu().numpy()
            try:
                errs = check_fold((st[:D], st[D:2 * D], float(st[-1])), want, label=mode)
                fold_ok = True
            except AssertionError as e:
                errs, fold_ok = repr(e)[:400], False
            nsteps = 2 * hp.update_epochs * hp.num_minibatches
            dpar = float((got["params"] - ref["params"]).abs().max())
            checks = {
                "statistics identical on all ranks": all(torch.equal(alls[0], x) for x in alls),
                "statistics vs float64 fold of the global batch": fold_ok,
                "params identical on all ranks": all(torch.equal(allp[0], x) for x in allp),
                "losses vs single GPU": rel_err(got["losses"], ref["losses"]) < 2e-3,
                "params vs single GPU": dpar < hp.opt_lr * (2.0 + 0.15 * nsteps),
            }
            print(f"[{mode}] world={world} fold errors (mean, var) {errs} max |dparam| {dpar:.2e} {checks}", flush=True)
            ok = ok and all(checks.values())
    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.broadcast(flag, src=0)
    dist.destroy_process_group()
    if rank == 0:
        print("MULTIGPU OBS NORM", "OK" if ok else "FAILED", flush=True)
    sys.exit(0 if int(flag.item()) else 1)


if __name__ == "__main__":
    main()
