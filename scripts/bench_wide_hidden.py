"""Learner throughput at model.hidden_size > 256 (layer-wise tcgen05 path, two column groups per hidden layer).

    python scripts/bench_wide_hidden.py [--hidden 384 512] [--steps 20] [--warmup 3]

configs[1] of bench.py (2048 envs x 128 steps, 4 epochs x 32 minibatches, D = 225 / A = 10 stand-in) at each hidden
width; one JSON line per width on stdout with:
  * ms per update and M transitions/s: graph replays between CUDA events, after `warmup` updates;
  * the FLOP-based fraction of the sustained bf16 peak DESIGN.md section 5 uses (1,384.7 TFLOP/s) -- a whole-update rate
    over a kernel peak, not a kernel's share of peak.  Work per transition and epoch is 6 F - 4 D H multiply-adds x 2,
    F = forward multiply-adds of both nets (no dX GEMM for the first layer);
  * the eager PyTorch-on-GPU proxy of bench.py at the same shape;
  * a parity flag: one fresh-state update against bench.py's CPU restatement (tolerance 1e-2 of the largest loss);
  * the card name and power limit, read in the same run.
Writes nothing; the lines kept are committed under profiles/."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import OBS_DIM, ACT_DIM, BenchShape, cpu_update_time, gpu_proxy_time, make_config, synth_shard  # noqa: E402

SUSTAINED_BF16_TFLOPS = 1384.7          # DESIGN.md section 5: measured sustained dense bf16 rate on the B200


def update_flops(hp: BenchShape, D: int, A: int) -> float:
    H, L = hp.hidden_size, hp.num_layers
    fwd_macs = 2 * D * H + 2 * (L - 1) * H * H + H * (A + 1)
    return 2.0 * (3 * fwd_macs - 2 * D * H) * hp.batch_size * hp.update_epochs


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        name, power, clk = (x.strip() for x in r.stdout.strip().split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except (OSError, ValueError, subprocess.SubprocessError) as e:
        return {"error": str(e)[:200]}


def run(H: int, steps: int, warmup: int, dev):
    import torch

    from minppo_b200.learner import Learner, Memory, TrainState
    from minppo_b200.params import flatten_params

    hp = BenchShape(num_envs=2048, num_steps=128, num_minibatches=32, update_epochs=4, hidden_size=H)
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

    # parity: one update from the initial state against the CPU restatement
    ts = TrainState.create(flat, dev)
    learner.update(ts, mem, lv, rng, losses, rng_out)
    learner.check()
    gl = losses.cpu().numpy().astype(np.float64)
    _, _, cpu_losses = cpu_update_time(hp, 1, (D, A))
    err = float(np.abs(gl - cpu_losses).max() / np.abs(cpu_losses).max())

    # device-resident timing: graph replays (the state keeps training; inputs stay resident)
    for _ in range(max(warmup, 3)):
        learner.update(ts, mem, lv, rng, losses, rng_out)
    torch.cuda.synchronize(dev)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        learner.update(ts, mem, lv, rng, losses, rng_out)
    ev1.record()
    torch.cuda.synchronize(dev)
    learner.check()
    ms = ev0.elapsed_time(ev1) / steps
    launches = learner.launches_per_update()
    learner.close()

    proxy = gpu_proxy_time(hp, dev, steps=3, try_compile=False, dims=(D, A))
    pl = proxy.pop("_losses")
    proxy["losses_vs_cpu_restatement"] = float(np.abs(pl - cpu_losses).max() / np.abs(cpu_losses).max())
    proxy["speedup_of_this_repo_over_eager_proxy"] = proxy["eager_ms_per_update"] / ms
    flops = update_flops(hp, D, A)
    return {
        "workload": f"configs[1]: 2048 envs x 128 steps, {H}x{H} MLPs (2 hidden layers), 4 epochs x 32 minibatches, "
                    f"D={D}/A={A} stand-in",
        "hidden_size": H, "path": "layer-wise tcgen05 GEMMs, 2 column groups per hidden layer",
        "ms_per_update": ms, "M_transitions_per_s": hp.batch_size / (ms * 1e-3) / 1e6,
        "updates_timed": steps, "warmup_updates": max(warmup, 3), "timing": "CUDA events around graph replays",
        "launches_per_update": launches,
        "tflop_per_update": flops / 1e12, "achieved_tflops": flops / (ms * 1e-3) / 1e12,
        "frac_of_sustained_bf16_peak": flops / (ms * 1e-3) / 1e12 / SUSTAINED_BF16_TFLOPS,
        "peak_note": f"whole-update FLOP rate over the sustained bf16 peak of DESIGN.md section 5 ({SUSTAINED_BF16_TFLOPS} TFLOP/s)",
        "parity_at_bench_shape": bool(np.isfinite(err) and err < 1e-2), "max_rel_err_losses_vs_cpu": err, "tolerance": 1e-2,
        "gpu_proxy": proxy, "card": card(),
    }


def main():
    import torch

    ap = argparse.ArgumentParser()
    ap.add_argument("--hidden", type=int, nargs="+", default=[384, 512])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_wide_hidden.py needs a CUDA device")
    dev = torch.device("cuda:0")
    for H in args.hidden:
        print(json.dumps(run(H, max(args.steps, 20), args.warmup, dev)), flush=True)


if __name__ == "__main__":
    main()
