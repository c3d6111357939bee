"""Per-minibatch statistics of the env-sharded learner update (run under torchrun on a box with >= 2 B200s;
tests/test_gpu_update_stats.py drives it):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29613 \
        tests/multigpu/check_sharded_update_stats.py

Every rank runs the update on its shard of ONE global batch with a ``stats`` buffer, three times: over the peer-memory
exchange one-shot, over the peer-memory exchange two-phase (MINPPO_PX_TWO_PHASE), and over ncclAllReduce
(MINPPO_NCCL_ALLREDUCE=1).  Checks: the statistics are bit-identical on every rank, and rank 0's match the reference
of the global batch (tests/update_stats_reference.py, bf16 rounding points) with the tolerances of
tests/test_gpu_update_stats.py."""
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
from tests.helpers import hyper_to_config, perturb_policy  # noqa: E402
from tests.test_gpu_update_stats import DELTA, check_stats  # noqa: E402
from tests.update_stats_reference import update_with_stats  # noqa: E402

MODES = {"peer_one_shot": {"MINPPO_PX_TWO_PHASE": "0"}, "peer_two_phase": {"MINPPO_PX_TWO_PHASE": "1"},
         "nccl": {"MINPPO_NCCL_ALLREDUCE": "1"}}


def run(hp, pr, dev, world, rank, nccl_id, n0, Nl):
    learner = Learner(hyper_to_config(hp), pr["obs_dim"], pr["act_dim"], dev, world, rank, nccl_id)
    ts = TrainState.create(P.flatten_params(pr["params"], hp.num_layers), dev)
    t = lambda x: torch.as_tensor(np.ascontiguousarray(x)).to(dev)
    tr = {k: v[:, n0:n0 + Nl] for k, v in pr["traj"].items()}
    mem = Memory(done=t(tr["done"]), action=t(tr["action"]), value=t(tr["value"]), reward=t(tr["reward"]),
                 log_prob=t(tr["log_prob"]), obs=t(tr["obs"]))
    rng = torch.as_tensor(pr["rng"].view(np.int32)).to(dev)
    stats = torch.full((hp.update_epochs, hp.num_minibatches, 4), float("nan"), device=dev)
    learner.update(ts, mem, t(pr["last_val"][n0:n0 + Nl]), rng, stats=stats)
    learner.check()
    peer = learner.peer_exchange
    learner.close()
    return stats, peer


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    dist.init_process_group("nccl", device_id=dev)
    hp = P.Hyper(num_envs=64 * world, num_steps=32, num_minibatches=4, update_epochs=2, anneal_lr=False)
    pr = synth.make_problem(hp, seed=3, done_p=0.02)
    perturb_policy(pr)
    Nl = hp.num_envs // world
    ref = None
    if rank == 0:
        p0 = P.tree_like(pr["params"], lambda x: x.astype(np.float32))
        ref = update_with_stats(p0, P.init_opt_state(p0), pr["traj"], pr["last_val"], pr["rng"], hp, dtype=np.float32,
                                gemm="bf16", delta=DELTA)[4]
    ok = True
    for mode, env in MODES.items():
        saved = {k: os.environ.get(k) for k in env}
        os.environ.update(env)
        ids = [nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        stats, peer = run(hp, pr, dev, world, rank, ids[0], rank * Nl, Nl)
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k)
            else:
                os.environ[k] = v
        gathered = [torch.empty_like(stats) for _ in range(world)]
        dist.all_gather(gathered, stats)
        if rank == 0:
            same = all(torch.equal(gathered[0], x) for x in gathered)
            try:
                m = check_stats(stats.cpu().numpy(), ref["stats"], ref["ambiguous"], hp.minibatch_size, mode)
                good = True
            except AssertionError as e:
                m, good = repr(e)[:800], False
            mode_ok = same and good and peer == (mode != "nccl")
            print(f"[{mode}] world={world} peer_exchange={peer} stats identical on all ranks={same} {m}", flush=True)
            ok = ok and mode_ok
    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.broadcast(flag, src=0)
    dist.destroy_process_group()
    if rank == 0:
        print("MULTIGPU STATS", "OK" if ok else "FAILED", flush=True)
    sys.exit(0 if int(flag.item()) else 1)


if __name__ == "__main__":
    main()
