"""Cost of the per-minibatch statistics output (``Learner.update(..., stats=...)``) at configs[1].

    python scripts/bench_update_stats.py [--rounds 8] [--steps 20] [--warmup 3]

configs[1] of bench.py (2048 envs x 128 steps, 256x256 MLPs, 4 epochs x 32 minibatches, D = 225 / A = 10 stand-in) on
one learner context: `rounds` rounds, each timing `steps` updates with stats=None and then `steps` updates writing a
stats buffer (graph replays between CUDA events; the two pointer sets are two cached graphs).  The statistics sums are
computed either way; the buffer only adds the per-step write.  Prints one JSON line: ms per update of each mode (median,
min, max over the rounds), the median difference, the card name and power limit read in the same run, and a parity
flag (the two modes give bitwise the same losses from the same state).  Writes nothing."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import OBS_DIM, ACT_DIM, BenchShape, make_config, synth_shard  # noqa: E402


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        name, power, clk = (x.strip() for x in r.stdout.strip().split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except (OSError, ValueError, subprocess.SubprocessError) as e:
        return {"error": str(e)[:200]}


def main():
    import torch

    from minppo_b200.learner import Learner, Memory, TrainState
    from minppo_b200.params import flatten_params

    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=8)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_update_stats.py needs a CUDA device")
    dev = torch.device("cuda:0")
    hp = BenchShape(num_envs=2048, num_steps=128, num_minibatches=32, update_epochs=4)
    D, A = OBS_DIM, ACT_DIM
    learner = Learner(make_config(hp, True), D, A, dev)
    params, traj, last_val = synth_shard(hp, 0, 1, dims=(D, A))
    flat = flatten_params(params, hp.num_layers)
    t = lambda x: torch.as_tensor(np.ascontiguousarray(x)).to(dev)
    mem = Memory(done=t(traj["done"]), action=t(traj["action"]), value=t(traj["value"]), reward=t(traj["reward"]),
                 log_prob=t(traj["log_prob"]), obs=t(traj["obs"]))
    lv = t(last_val)
    rng = torch.tensor([0, 1337], dtype=torch.int32, device=dev)
    rng_out = torch.empty_like(rng)
    losses = torch.empty((hp.update_epochs, hp.num_minibatches, 4), dtype=torch.float32, device=dev)
    stats = torch.empty((hp.update_epochs, hp.num_minibatches, 4), dtype=torch.float32, device=dev)

    # parity: the same starting state with and without the buffer gives bitwise the same losses
    out = []
    for s in (None, stats):
        ts = TrainState.create(flat, dev)
        learner.update(ts, mem, lv, rng, losses, rng_out, stats=s)
        out.append(losses.clone())
    learner.check()
    same = bool(torch.equal(out[0], out[1]))

    ts = TrainState.create(flat, dev)
    modes = {"stats_none": None, "stats_buffer": stats}
    for s in modes.values():
        for _ in range(max(args.warmup, 3)):
            learner.update(ts, mem, lv, rng, losses, rng_out, stats=s)
    torch.cuda.synchronize(dev)
    times = {k: [] for k in modes}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.rounds):
        for k, s in modes.items():
            ev0.record()
            for _ in range(args.steps):
                learner.update(ts, mem, lv, rng, losses, rng_out, stats=s)
            ev1.record()
            torch.cuda.synchronize(dev)
            times[k].append(ev0.elapsed_time(ev1) / args.steps)
    learner.check()
    learner.close()
    summary = {k: {"median_ms": float(np.median(v)), "min_ms": float(np.min(v)), "max_ms": float(np.max(v)),
                   "per_round_ms": [round(x, 4) for x in v]} for k, v in times.items()}
    print(json.dumps({
        "workload": f"configs[1]: 2048 envs x 128 steps, 256x256 MLPs, 4 epochs x 32 minibatches, D={D}/A={A} stand-in",
        "timing": f"CUDA events around {args.steps} graph replays per round, {args.rounds} rounds, modes alternating",
        **summary,
        "median_diff_ms": summary["stats_buffer"]["median_ms"] - summary["stats_none"]["median_ms"],
        "losses_identical_with_and_without_stats": same, "card": card(),
    }), flush=True)


if __name__ == "__main__":
    main()
