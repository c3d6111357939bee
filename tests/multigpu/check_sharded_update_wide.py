"""Multi-GPU parity check at model.hidden_size = 512 (the layer-wise path with two column groups per hidden layer), run
under torchrun on a box with >= 2 B200s:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29613 \
        tests/multigpu/check_sharded_update_wide.py

Same checks as check_sharded_update.py: permutations, rng and the shards' policy step bit-exact against the single-GPU
run; parameters bit-identical on every rank; losses / parameters equal to the single-GPU update up to fp32 summation order
(2e-3 of the largest loss, lr * (2 + 0.15 n) on the parameters); and against the oracle with the bf16 rounding points
emulated.  Collected by tests/test_gpu_wide_hidden.py where >= 2 GPUs are visible."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from minppo_b200.learner import nccl_unique_id  # noqa: E402
from oracle import ppo_numpy as P  # noqa: E402
from oracle import synth  # noqa: E402
from tests.helpers import rel_err  # noqa: E402
from tests.multigpu.check_sharded_update import run  # noqa: E402


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    dist.init_process_group("nccl", device_id=dev)
    hp = P.Hyper(anneal_lr=False, num_envs=64 * world, num_steps=32, num_minibatches=4, update_epochs=2, hidden_size=512)
    pr = synth.make_problem(hp, seed=3)
    Nl = hp.num_envs // world
    ids = [nccl_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    got = run(hp, pr, dev, world, rank, ids[0], rank * Nl, Nl)
    mine = torch.from_numpy(got["params"]).to(dev)
    allp = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(allp, mine)
    same = all(torch.equal(allp[0], x) for x in allp)
    allpol = [torch.empty_like(got["pol"]) for _ in range(world)]
    dist.all_gather(allpol, got["pol"])
    ok = True
    if rank == 0:
        ref = run(hp, pr, dev, 1, 0, None, 0, hp.num_envs)
        lr = hp.opt_lr
        nsteps = 2 * hp.update_epochs * hp.num_minibatches
        p_o = P.tree_like(pr["params"], lambda x: x.astype(np.float32))
        o_o = P.init_opt_state(p_o)
        for _ in range(2):
            p_o, o_o, rng_o, l_o, aux_o = P.update(p_o, o_o, pr["traj"], pr["last_val"], pr["rng"], hp, dtype=np.float32,
                                                   gemm="bf16")
        flat_o = P.flatten_params(p_o, hp.num_layers, np.float64)
        checks = {
            "params identical on all ranks": same,
            "perms bit-exact": bool(np.array_equal(got["perms"], ref["perms"])),
            "policy step of the shards == single GPU, bit-exact":
                bool(torch.equal(torch.cat(allpol, dim=0), ref["pol"]) and np.array_equal(got["pol_rng"], ref["pol_rng"])),
            "rng bit-exact": bool(np.array_equal(got["rng"], ref["rng"])),
            "step": got["step"] == ref["step"] == nsteps,
            "losses": rel_err(got["losses"], ref["losses"]) < 2e-3,
            "params": float(np.abs(got["params"] - ref["params"]).max()) < lr * (2.0 + 0.15 * nsteps),
            "losses vs oracle (bf16 rounding emulated)": rel_err(got["losses"], l_o) < 2e-3,
            "perms vs oracle bit-exact": bool(np.array_equal(got["perms"], aux_o["perms"])),
            "params vs oracle rms <= 1 lr": float(np.sqrt(np.mean((got["params"] - flat_o) ** 2))) < lr,
        }
        print(f"[hidden 512] world={world} loss rel err {rel_err(got['losses'], ref['losses']):.2e} "
              f"max |dparam| {np.abs(got['params'] - ref['params']).max():.2e}  {checks}", flush=True)
        ok = all(checks.values())
    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.broadcast(flag, src=0)
    dist.destroy_process_group()
    if rank == 0:
        print("MULTIGPU PARITY", "OK" if ok else "FAILED", flush=True)
    sys.exit(0 if int(flag.item()) else 1)


if __name__ == "__main__":
    main()
