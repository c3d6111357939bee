#!/usr/bin/env python
"""bench.py -- learner transitions/sec (GAE + all PPO epochs) on synthetic stompy_pro-shaped
trajectories (BASELINE.json metric; SURVEY.md section 8d).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is ONE learner update of the hot path (/root/reference/minppo/train.py:185-281): GAE
over the [T x N] trajectory, E epochs x M minibatches of shuffle/gather + ActorCritic
forward/backward + PPO loss + global-norm clip + Adam.

  N == 1 : BASELINE.json configs[1]: 2048 envs x 128 steps, 256x256 MLPs, 4 epochs x 32 minibatches.
  N  > 1 : the same shard on EVERY GPU (2048 envs x 128 steps per GPU, global batch 2048*N envs, env-sharded,
           global permutation, per-minibatch gradient all-reduce) -> "scaling": "weak"; at N = 8 this is
           configs[3]'s 16384 envs.  `--workload c4` runs configs[3] literally (16384 x 64 global, strong).

`value`  = unique transitions per second = T*N / t_update, inputs resident in HBM, CUDA-graph replay.
`e2e`    = same metric through Learner.update_host: pinned HOST buffers, H2D of the trajectory +
           train state and D2H of the new train state + losses inside the timed region.
D = 225 / A = 10 are a DECLARED STAND-IN for stompy_pro (its MJCF is fetched at run time by the
reference; SURVEY.md F9).  `--impl reference`: JAX is not installable in this image, so the
reference arm times the oracle's PyTorch-CPU restatement of the same update ("kind": "port").

Separation: the product arm (`run_ours`) imports only `minppo_b200` (+ numpy / torch for input generation and device
memory); `oracle/` is imported by exactly two legs -- `cpu_update_time` (the `cpu_baseline` object at N = 1) and
`run_reference` (`--impl reference`).
"""
from __future__ import annotations

import argparse
import dataclasses
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np

OBS_DIM, ACT_DIM = 225, 10          # declared stand-in (SURVEY.md F9)
METRIC = "learner transitions/sec (GAE+PPO epochs)"
UNIT = "transitions/s"


def workload(n_gpus: int, which: str = "auto"):
    """auto: configs[1] on every GPU (2048 envs x 128 steps PER GPU, env-sharded: the global batch and the
    global minibatch grow with N -> weak scaling; at N = 8 this is configs[3]'s 16384 envs).
    c4: configs[3] literally (16384 envs x 64 steps GLOBAL, strong scaling)."""
    if which == "c4":
        return dict(name=f"configs[3]: 16384 envs x 64 steps env-sharded over {n_gpus} GPU(s), 256x256 MLPs, "
                         "4 epochs x 32 minibatches", num_envs=16384, num_steps=64, num_minibatches=32,
                    update_epochs=4, scaling="strong")
    if n_gpus == 1:
        return dict(name="configs[1]: 2048 envs x 128 steps, 256x256 MLPs, 4 epochs x 32 minibatches",
                    num_envs=2048, num_steps=128, num_minibatches=32, update_epochs=4, scaling="weak")
    return dict(name=f"configs[1] per GPU, env-sharded: {2048 * n_gpus} envs x 128 steps over {n_gpus} GPUs "
                     "(2048 envs per GPU), 256x256 MLPs, 4 epochs x 32 minibatches, per-minibatch gradient all-reduce",
                num_envs=2048 * n_gpus, num_steps=128, num_minibatches=32, update_epochs=4, scaling="weak")


@dataclasses.dataclass
class BenchShape:
    """The learner shape of one workload (the reference's defaults, config.py:50-84, where not given)."""
    num_envs: int
    num_steps: int
    num_minibatches: int
    update_epochs: int
    hidden_size: int = 256
    num_layers: int = 2
    use_tanh: bool = True
    gamma: float = 0.99
    gae_lambda: float = 0.95

    @property
    def batch_size(self) -> int:
        return self.num_envs * self.num_steps

    @property
    def minibatch_size(self) -> int:
        return self.batch_size // self.num_minibatches


def bench_config(w, world: int, dims, hp, fast_tanh: bool):
    """The `config` object of the JSON line -- identical on every arm (`--impl ours | reference`), so that the driver's
    same-config check compares like with like."""
    return {"workload": w["name"], "obs_dim": dims[0], "act_dim": dims[1],
            "shape_note": f"D={dims[0]}/A={dims[1]} are a declared stand-in for stompy_pro (SURVEY.md F9)",
            "parallelism": f"env-sharded dp{world}" if world > 1 else "single GPU",
            "l2_policy": f"inputs larger than L2 (obs {hp.batch_size // world * dims[0] * 4 / 1e6:.0f} MB per update and GPU vs 126 MB L2)",
            "fast_tanh": bool(fast_tanh)}


def make_shape(w) -> BenchShape:
    return BenchShape(num_envs=w["num_envs"], num_steps=w["num_steps"], num_minibatches=w["num_minibatches"],
                      update_epochs=w["update_epochs"])


def make_config(hp: BenchShape, fast_tanh: bool):
    """The product's Config for this shape: anneal_lr=True with the default 1e9 total timesteps (config.py:79, 83)."""
    from minppo_b200.config import Config

    c = Config()
    c.model.hidden_size, c.model.num_layers, c.model.use_tanh = hp.hidden_size, hp.num_layers, hp.use_tanh
    c.rl.num_env_steps, c.rl.gamma, c.rl.gae_lambda = hp.num_steps, hp.gamma, hp.gae_lambda
    c.training.num_envs, c.training.num_steps = hp.num_envs, hp.num_steps
    c.training.num_minibatches, c.training.update_epochs, c.training.anneal_lr = hp.num_minibatches, hp.update_epochs, True
    c.learner.fast_tanh, c.learner.use_graph = fast_tanh, True
    return c


def make_hyper(hp: BenchShape):
    """CPU arm only: the oracle's hyper-parameter record for the same shape."""
    from oracle import ppo_numpy as P

    return P.Hyper(num_envs=hp.num_envs, num_steps=hp.num_steps, num_minibatches=hp.num_minibatches,
                   update_epochs=hp.update_epochs, anneal_lr=True)


def tree_map(tree, fn):
    return {k: tree_map(v, fn) if isinstance(v, dict) else fn(v) for k, v in tree.items()}


def init_param_tree(hidden: int, num_layers: int, seed: int = 0, dims=None):
    """Synthetic parameters in the checkpoint tree layout (train.py:86-89) with the init GAINS of train.py:63/68
    (sqrt(2) hidden, 0.01 last layer) as plain scaled normals -- random-init weights of the architecture."""
    g = np.random.default_rng(seed)
    obs_dim, act_dim = dims or (OBS_DIM, ACT_DIM)
    p = {"params": {}}
    for mlp, out_dim in (("MLP_0", act_dim), ("MLP_1", 1)):
        d = {}
        fan_in = obs_dim
        for i in range(num_layers):
            d[f"Dense_{i}"] = {"kernel": (g.standard_normal((fan_in, hidden)) * np.sqrt(2.0 / fan_in)).astype(np.float32),
                               "bias": (0.01 * g.standard_normal(hidden)).astype(np.float32)}
            fan_in = hidden
        d[f"Dense_{num_layers}"] = {"kernel": (g.standard_normal((fan_in, out_dim)) * (0.01 / np.sqrt(fan_in))).astype(np.float32),
                                    "bias": (0.01 * g.standard_normal(out_dim)).astype(np.float32)}
        p["params"][mlp] = d
    p["params"]["log_std"] = (0.05 * g.standard_normal(act_dim)).astype(np.float32)
    return p


def synth_shard(hp, rank: int, world: int, seed: int = 0, dims=None):
    """Synthetic shard [T, N/world, ...] in float32 NumPy.  Params from the init gains; value / log_prob
    from a forward pass under those params; reward ~ N(0,1); done ~ B(0.01).  The same arguments give the same
    bits in every run: the forward pass runs on one CPU thread (BLAS sums in an order that depends on how it splits
    the work over threads, and it may choose that split anew in each run) and in float64, rounded once to float32.
    Input generation only: nothing here touches oracle/ or the product."""
    import torch

    T, Nl = hp.num_steps, hp.num_envs // world
    obs_dim, act_dim = dims or (OBS_DIM, ACT_DIM)
    params = init_param_tree(hp.hidden_size, hp.num_layers, seed, dims=(obs_dim, act_dim))
    g = torch.Generator().manual_seed(1234 + rank)
    obs = torch.randn(T * Nl, obs_dim, generator=g)
    pt = tree_map(params, lambda x: torch.from_numpy(x).double())["params"]

    def mlp(m, x, tanh):
        for i in range(hp.num_layers):
            x = torch.addmm(m[f"Dense_{i}"]["bias"], x, m[f"Dense_{i}"]["kernel"])
            x = x.tanh_() if tanh else x.relu_()
        return torch.addmm(m[f"Dense_{hp.num_layers}"]["bias"], x, m[f"Dense_{hp.num_layers}"]["kernel"])

    threads = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        with torch.no_grad():
            obs64 = obs.double()
            mean = mlp(pt["MLP_0"], obs64, hp.use_tanh)
            value = mlp(pt["MLP_1"], obs64, False)[:, 0]
            del obs64
            scale = torch.exp(pt["log_std"])
            action = mean + scale * torch.randn(mean.shape, generator=g).double()
            z = (action - mean) / scale
            log_prob = (-0.5 * z * z - 0.5 * np.log(2 * np.pi)).sum(-1) - torch.log(scale).sum()
            last_val = mlp(pt["MLP_1"], torch.randn(Nl, obs_dim, generator=g).double(), False)[:, 0]
    finally:
        torch.set_num_threads(threads)
    traj = {
        "obs": obs.reshape(T, Nl, obs_dim).numpy(), "action": action.float().reshape(T, Nl, act_dim).numpy(),
        "value": value.float().reshape(T, Nl).numpy(), "log_prob": log_prob.float().reshape(T, Nl).numpy(),
        "reward": torch.randn(T, Nl, generator=g).numpy(),
        "done": (torch.rand(T, Nl, generator=g) < 0.01).numpy(),
    }
    return params, traj, last_val.float().numpy()


DUMP_LIMIT_BYTES = 63 << 20          # array data: with the .npy headers, a dump stays under 64 MB


def dump_outputs(out_dir: str, arrays) -> None:
    """Write each array as <out_dir>/<name>.npy: floating point as float32, integers as float64 (exact for 32-bit words).
    If together they exceed DUMP_LIMIT_BYTES, each array larger than an equal share of the limit is replaced by the same
    seeded sample of its flattened elements in every run, so that two builds can still be compared element for element."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.asarray(v, np.float64 if np.issubdtype(np.asarray(v).dtype, np.integer) else np.float32)
              for k, v in arrays.items()}
    share = DUMP_LIMIT_BYTES // len(arrays)
    over = sum(a.nbytes for a in arrays.values()) > DUMP_LIMIT_BYTES
    for name, a in arrays.items():
        if over and a.nbytes > share:
            idx = np.sort(np.random.default_rng(0).choice(a.size, share // a.itemsize, replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        if self.thread is not None:
            self.thread.join(timeout=2)
        if not self.rows:
            # the timed region was shorter than one sampling period: one query right after it (clocks have not ramped
            # down yet) is better than no evidence at all
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.idx)],
                                     capture_output=True, text=True, timeout=10).stdout
                self.rows = [l.strip() for l in out.splitlines() if l.strip()]
            except Exception:
                pass
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        # under load = samples in the upper half of what was seen (the sampler also sees idle gaps)
        load = sorted(sm)[len(sm) // 2:] if sm else []
        return {"sm_mhz": float(np.median(load)) if load else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------
# CPU arm: the oracle's PyTorch-CPU restatement, ONE WHOLE update per step (nothing extrapolated)
# ------------------------------------------------------------------------------------------
def cpu_update_time(hp, repeats: int = 1, dims=None):
    """Seconds for one FULL learner update (GAE + E permutations + E shuffled copies + E*M minibatch steps) of
    oracle/ppo_torch.py on the host cores, every step measured.  Returns (seconds, cores, losses[E, M, 4]) -- the
    losses are what bench.py's parity check compares the GPU arm's fresh-state update against."""
    import torch

    from oracle import ppo_numpy as P
    from oracle import ppo_torch as PT

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    D, A = dims or (OBS_DIM, ACT_DIM)
    params, traj, last_val = synth_shard(hp, 0, 1, dims=(D, A))
    hp = make_hyper(hp)                                   # the oracle's record of the same shape
    pt = PT.to_torch(params, torch.float32)
    tr = {k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in traj.items()}
    lv = torch.from_numpy(last_val)
    rng = np.array([0, 1337], np.uint32)
    best, losses = None, None
    for _ in range(repeats):
        opt = {"count": 0, "mu": P.tree_like(pt, torch.zeros_like), "nu": P.tree_like(pt, torch.zeros_like)}
        t0 = time.perf_counter()
        _, _, _, ls, _ = PT.update(pt, opt, tr, lv, rng, hp)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
        losses = ls.numpy()
    return best, cores, losses


CPU_SAMPLE = ("one WHOLE learner update per step (GAE + 4 permutations + 4 shuffled epoch copies + all 128 minibatch "
              "steps), nothing extrapolated; CPU restatement (PyTorch fp32 eager, all host threads), not JAX")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = workload(args.gpus, args.workload)
    hp = make_shape(w)
    B = hp.batch_size
    dims = (args.obs_dim, args.act_dim)
    for _ in range(min(args.warmup, 1)):
        cpu_update_time(hp, 1, dims)
    times = []
    cores = os.cpu_count() or 1
    for _ in range(args.steps):
        t, cores, _ = cpu_update_time(hp, 1, dims)
        times.append(t)
    t_upd = float(np.median(times))
    val = B / t_upd
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": t_upd * 1e3, "higher_is_better": True,
        "scaling": w["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(w, args.gpus, dims, hp, bool(args.fast_tanh)),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": CPU_SAMPLE},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------
# GPU proxy arm: the SAME restatement in eager PyTorch on the B200 (SURVEY.md 8d: the stand-in comparator for the
# north_star's "20x the reference JAX-on-GPU learner", which cannot be measured in an image without JAX)
# ------------------------------------------------------------------------------------------
def gpu_proxy_time(hp, dev, steps: int = 3, try_compile: bool = True, dims=None):
    """oracle/ppo_torch.update on `dev`: every one of the E*M minibatch steps measured (CUDA events around whole
    updates, median).  The permutations are precomputed on the host OUTSIDE the timed region (in favour of the
    proxy); GAE, the shuffled epoch copies, forward/backward (autograd), clip and Adam all run as eager torch ops.
    `try_compile`: additionally time the same update with the per-minibatch loss+grad function under torch.compile
    (inductor); reported only if it compiles and runs offline."""
    import torch

    from oracle import ppo_numpy as P
    from oracle import ppo_torch as PT
    from oracle import threefry

    D, A = dims or (OBS_DIM, ACT_DIM)
    params, traj, last_val = synth_shard(hp, 0, 1, dims=(D, A))
    hpo = make_hyper(hp)
    pt = P.tree_like(PT.to_torch(params, torch.float32), lambda x: x.to(dev))
    tr = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in traj.items()}
    lv = torch.from_numpy(last_val).to(dev)
    rng = np.array([0, 1337], np.uint32)
    perms, key = [], rng
    for _ in range(hpo.update_epochs):
        key, sub = threefry.split(key, 2, hpo.prng_mode)
        perms.append(torch.from_numpy(threefry.permutation(sub, hpo.batch_size, hpo.prng_mode).astype(np.int64)).to(dev))

    def timed(compiled: bool):
        PT.set_compiled(compiled)
        ts = []
        for it in range(steps + 1):
            opt = {"count": 0, "mu": P.tree_like(pt, torch.zeros_like), "nu": P.tree_like(pt, torch.zeros_like)}
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _, _, _, ls, _ = PT.update(pt, opt, tr, lv, rng, hpo, perms=perms)
            e1.record()
            torch.cuda.synchronize(dev)
            if it > 0:                                     # first pass = warm-up (allocator, autotune, compile)
                ts.append(e0.elapsed_time(e1))
        return float(np.median(ts)), ls.cpu().numpy()

    out = {"kind": "proxy: oracle/ppo_torch.py restatement in eager PyTorch on this B200 (fp32 cuBLAS GEMMs, TF32 off), "
                   "NOT the reference JAX learner (JAX is not installable in this image)",
           "steps_measured": hpo.update_epochs * hpo.num_minibatches, "updates_timed": steps,
           "note": "permutations precomputed outside the timed region (in favour of the proxy)"}
    ms, ls = timed(False)
    out["eager_ms_per_update"] = ms
    out["eager_transitions_per_s"] = hpo.batch_size / (ms * 1e-3)
    out["_losses"] = ls
    if try_compile:
        try:
            cms, _ = timed(True)
            out["compiled_ms_per_update"] = cms
            out["compiled_transitions_per_s"] = hpo.batch_size / (cms * 1e-3)
        except Exception as e:          # inductor needs a working triton + compiler toolchain offline
            out["compiled_error"] = (type(e).__name__ + ": " + str(e))[:300]
        finally:
            PT.set_compiled(False)
    return out


def run_torch_gpu(args):
    """`--impl torch_gpu`: the GPU proxy alone (rank 0, one GPU), as its own JSON line."""
    import torch

    if int(os.environ.get("RANK", "0")) != 0:
        return
    dev = torch.device(f"cuda:{int(os.environ.get('LOCAL_RANK', '0'))}")
    w = workload(1, args.workload)
    hp = make_shape(w)
    proxy = gpu_proxy_time(hp, dev, steps=max(args.steps, 1), try_compile=bool(args.proxy_compile), dims=(args.obs_dim, args.act_dim))
    proxy.pop("_losses", None)
    ms = proxy["eager_ms_per_update"]
    print(json.dumps({"impl": "torch_gpu", "metric": METRIC, "value": hp.batch_size / (ms * 1e-3), "unit": UNIT, "n_gpus": 1,
                      "steps": args.steps, "warmup": 1, "ms_per_step": ms, "higher_is_better": True, "scaling": w["scaling"],
                      "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                      "config": {"workload": w["name"], "obs_dim": args.obs_dim, "act_dim": args.act_dim}, "gpu_proxy": proxy}), flush=True)


# ------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    from minppo_b200 import _lib
    from minppo_b200.learner import HostBatch, Learner, Memory, TrainState, calculate_gae, nccl_unique_id
    from minppo_b200.params import flatten_params

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N > 1")
    torch.cuda.set_device(local_rank)
    dev = torch.device(f"cuda:{local_rank}")
    if os.environ.get("MINPPO_BENCH_ENABLE_P2P") and torch.cuda.device_count() > 1:
        # development probe: a cross-device copy makes torch enable peer access on this context (does a context with
        # peer mappings pay more per kernel boundary?)
        other = (local_rank + 1) % torch.cuda.device_count()
        torch.zeros(1024, device=dev).to(f"cuda:{other}")
        torch.zeros(1024, device=f"cuda:{other}").to(dev)
        torch.cuda.synchronize()
    nccl_id = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        ids = [nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        nccl_id = ids[0]

    w = workload(world, args.workload)
    hp = make_shape(w)
    B = hp.batch_size
    cfg = make_config(hp, bool(args.fast_tanh))
    D_OBS, D_ACT = args.obs_dim, args.act_dim
    learner = Learner(cfg, D_OBS, D_ACT, dev, world, rank, nccl_id)
    params, traj, last_val = synth_shard(hp, rank, world, dims=(D_OBS, D_ACT))
    flat = flatten_params(params, hp.num_layers)
    t = lambda x: torch.as_tensor(np.ascontiguousarray(x)).to(dev)
    mem = Memory(done=t(traj["done"]), action=t(traj["action"]), value=t(traj["value"]), reward=t(traj["reward"]),
                 log_prob=t(traj["log_prob"]), obs=t(traj["obs"]))
    lv = t(last_val)
    ts = TrainState.create(flat, dev)
    rng = torch.tensor([0, 1337], dtype=torch.int32, device=dev)
    rng_out = torch.empty_like(rng)
    losses = torch.empty((hp.update_epochs, hp.num_minibatches, 4), dtype=torch.float32, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def one_update():
        learner.update(ts, mem, lv, rng, losses, rng_out)

    sampler = ClockSampler(local_rank) if rank == 0 else None
    # ---- device-resident number ---------------------------------------------------------------
    for _ in range(max(args.warmup, 3)):
        one_update()
    barrier()
    learner.check()
    if sampler:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(args.steps):
        one_update()
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if sampler else None
    learner.check()
    if args.dump_outputs and rank == 0:
        # what Learner.update hands its caller after the last timed step (rank 0's copy when sharded)
        dump_outputs(args.dump_outputs, {"params": ts.params.cpu().numpy(), "mu": ts.mu.cpu().numpy(),
                                         "nu": ts.nu.cpu().numpy(), "step": ts.step.cpu().numpy(),
                                         "rng_out": rng_out.cpu().numpy().view(np.uint32), "losses": losses.cpu().numpy()})
    tt = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms_per_step = float(tt.item()) / args.steps
    value = B / (ms_per_step * 1e-3)
    final_losses = losses.cpu().numpy()
    if args.quick:
        if os.environ.get("MINPPO_TRACE"):
            # development: phase stamps of the dwopt kernel of the last minibatch step (one eager update on every rank)
            learner.use_graph = False
            one_update()
            nsm = torch.cuda.get_device_properties(dev).multi_processor_count
            o2 = torch.empty((nsm, 16), dtype=torch.int64, device=dev)
            _lib.check(learner.lib.minppo_ctx_read(learner._h, 8, o2.data_ptr(), o2.numel() * 8,
                                                   torch.cuda.current_stream(dev).cuda_stream))
            torch.cuda.synchronize(dev)
            t2 = o2.cpu().numpy()
            if rank == 0:
                seq = [0, 1, 2, 13, 14, 15, 3, 4, 5] if world > 1 else [0, 1, 2, 3, 4, 5]
                lab = {1: "phase 1 done", 2: "barrier 1 passed", 13: "local reduce + pushes issued", 14: "barrier A passed",
                       15: "peer flags seen", 3: "reduce done, block sums written", 4: "barrier 2 passed", 5: "end"}
                prev = 0
                for k in seq[1:]:
                    dt = (t2[:128, k] - t2[:128, 0]).mean()
                    print(f"dwopt trace: {lab[k]:34s} {dt:9.0f} (+{dt - prev:.0f})")
                    prev = dt
        if rank == 0:
            print(json.dumps({"quick": True, "ms_per_step": ms_per_step, "value": value, "n_gpus": world,
                              "skip": os.environ.get("MINPPO_SKIP", "0"), "clocks": clocks}), flush=True)
        learner.close()
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- end-to-end through host buffers --------------------------------------------------------
    hb = HostBatch(learner)
    for k in ("obs", "action", "value", "reward", "log_prob", "last_val"):
        hb.h[k].copy_(torch.from_numpy(np.ascontiguousarray(traj[k] if k != "last_val" else last_val)))
    hb.h["done"].copy_(torch.from_numpy(traj["done"].view(np.uint8)))
    hb.h["rng"].copy_(torch.tensor([0, 1337], dtype=torch.int32))
    hb.h["params"].copy_(torch.from_numpy(flat))
    for _ in range(2):
        learner.update_host(hb)
    barrier()
    e2e_steps = max(3, min(args.steps, 10))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        learner.update_host(hb)          # blocks until the results are on the host
    barrier()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    et_block = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(et_block, op=dist.ReduceOp.MAX)
    e2e_blocking = {"value": B / float(et_block.item()), "unit": UNIT, "ms_per_step": float(et_block.item()) * 1e3,
                    "h2d_bytes_per_step": hb.h2d_bytes(), "d2h_bytes_per_step": hb.d2h_bytes(),
                    "api": "Learner.update_host: blocking round trip, trajectory + FULL train state H2D, train state + losses D2H"}

    # ---- end-to-end, streaming: HostPipeline (train state resident, trajectory H2D + params / losses D2H EVERY update,
    #      the copy of update i + 1 under the kernels of update i) -----------------------------------------------------------
    from minppo_b200.learner import HostPipeline

    ts_pipe = TrainState.create(flat, dev)
    pipe = HostPipeline(learner, ts_pipe, torch.tensor([0, 1337], dtype=torch.int32, device=dev))
    host_traj = {k: hb.h[k] for k in ("obs", "action", "value", "reward", "log_prob", "done", "last_val")}
    for _ in range(3):                                   # warm-up: both buffer sets, both cached graphs
        pipe.submit(host_traj)
        pipe.result()
    barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        pipe.submit(host_traj)                           # H2D of THIS update's trajectory + the update + D2H of its results
        if i >= 1:
            pipe.result()                                # update i - 1 is on the host (losses, params)
    pipe.result()
    barrier()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    et = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(et, op=dist.ReduceOp.MAX)
    e2e_val = B / float(et.item())
    e2e_h2d, e2e_d2h = pipe.h2d_bytes(), pipe.d2h_bytes()

    # ---- per-kernel-class timing (eager, CUDA events on the launching stream) ----------------------
    prof = None
    gae_roof = None
    if rank == 0:
        import ctypes as C

        learner.use_graph = False
        learner.lib.minppo_ctx_profile(learner._h, 1)
        one_update()
        n = len(_lib.PROFILE_CLASSES)
        msv = (C.c_float * n)()
        cnt = (C.c_int32 * n)()
        _lib.check(learner.lib.minppo_ctx_profile_read(learner._h, msv, cnt, n))
        learner.lib.minppo_ctx_profile(learner._h, 0)
        learner.use_graph = True
        prof = {name: {"ms_per_update": float(msv[i]), "scopes": int(cnt[i])} for i, name in enumerate(_lib.PROFILE_CLASSES)}
    if world > 1:
        # the other ranks must take part in the collectives of rank 0's profiled update
        if rank != 0:
            learner.use_graph = False
            one_update()
            learner.use_graph = True
        barrier()

    if rank == 0:
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peaks = json.load(f)
        except OSError:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        tf_peak = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1590.0)))
        peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
        # dominant kernel = the tensor-core class with the most time; ALGORITHMIC FLOPs per launch
        # (SURVEY.md 8d: F MACs forward, F - 2DH for dX, F for dW per transition; D unpadded)
        H, L, D, A = hp.hidden_size, hp.num_layers, D_OBS, D_ACT
        rows = hp.minibatch_size / world
        F_hidden = 2 * D * H + 2 * (L - 1) * H * H            # MACs per row, hidden-layer contractions, both nets
        F_heads = H * A + H
        fused_path = prof["head_loss"]["scopes"] == 0           # fused step kernel: fwd + heads + loss + dX in one launch
        if fused_path:
            flops = {"fwd_gemm": 2 * rows * ((F_hidden + F_heads) + (F_hidden - 2 * D * H + F_heads) + F_heads),
                     "dw_gemm": 2 * rows * F_hidden}
            ap = 16 if A <= 16 else 32
            n_par = 2 * (D * H + H + (L - 1) * (H * H + H)) + (H * A + A) + (H + 1) + A
            nsm = torch.cuda.get_device_properties(dev).multi_processor_count
            maxu = 1 if n_par <= 4 * nsm * 512 else (2 if n_par <= 8 * nsm * 512 else 4)
            names = {"fwd_gemm": f"fused_step_kernel<{ap}> (forward + heads + PPO loss + backward-to-dZ + bias-gradient column "
                                 "sums, both nets)",
                     "dw_gemm": f"dwopt_kernel<{maxu}> (split-K weight gradients of all layers and both nets + gradient "
                                "reduction + global-norm clip + Adam, one launch)"}
        else:
            flops = {"fwd_gemm": 2 * rows * F_hidden / L, "bwd_gemm": 2 * rows * 2 * H * H, "dw_gemm": 2 * rows * F_hidden}
            names = {k: f"umma_gemm_kernel ({k})" for k in flops}
        dom = max(flops, key=lambda k: prof[k]["ms_per_update"])
        launches = max(prof[dom]["scopes"], 1)
        dur_s = prof[dom]["ms_per_update"] * 1e-3 / launches
        achieved = flops[dom] / dur_s / 1e12 if dur_s > 0 else 0.0
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                traffic = json.load(f).get(dom)          # dram bytes per launch from the committed ncu --set full capture
        except (OSError, ValueError):
            pass
        step_flops = 2 * rows * (3 * (F_hidden + F_heads) - 2 * D * H)
        roofline = {"bound": "tensor", "kernel": names[dom], "achieved": achieved, "peak": tf_peak,
                    "unit": "TFLOP/s", "frac": achieved / tf_peak, "traffic": traffic,
                    "flops_per_launch": flops[dom], "avg_launch_us": dur_s * 1e6, "peak_source": peak_src + ", sustained bf16",
                    "whole_step": {"flops_per_minibatch_step": step_flops,
                                   "achieved_tflops": step_flops * hp.update_epochs * hp.num_minibatches / (ms_per_step * 1e-3) / 1e12,
                                   "note": "all kernels of one update (graph replay) against the same peak"}}
        # GAE against the HBM roofline at a bandwidth-relevant size (config 3 scale: 128 x 1M)
        Tg, Ng = 128, 1 << 20
        gg = torch.Generator(device=dev).manual_seed(0)
        r_ = torch.randn(Tg, Ng, device=dev, generator=gg)
        v_ = torch.randn(Tg, Ng, device=dev, generator=gg)
        d_ = torch.rand(Tg, Ng, device=dev, generator=gg) < 0.01
        lv_ = torch.randn(Ng, device=dev, generator=gg)
        gm = Memory(d_, None, v_, r_, None, None)
        for _ in range(3):
            calculate_gae(gm, lv_, hp.gamma, hp.gae_lambda)
        torch.cuda.synchronize(dev)
        reps, batches = 10, []
        for _ in range(3):                                       # median of three batches of 10 calls
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            for _ in range(reps):
                calculate_gae(gm, lv_, hp.gamma, hp.gae_lambda)   # 2.3 GB per call >> 126 MB L2
            g1.record()
            torch.cuda.synchronize(dev)
            batches.append(g0.elapsed_time(g1) / reps)
        gms = float(np.median(batches))
        gbytes = Tg * Ng * 17 + 4 * Ng
        # the launch plan of gae.cu (gae_plan): VEC = 4 when N % 4 == 0; one pass over T (gae_single_kernel<4, UNROLL>, UNROLL = 8
        # below 1024 float4 columns per SM, else 4) unless fewer than 384 columns per SM force the T-chunked kernel
        cols_per_sm = (Ng // 4) / torch.cuda.get_device_properties(dev).multi_processor_count
        gae_kernel = ("gae_chunked_kernel<4, 4>" if cols_per_sm < 384 else
                      ("gae_single_kernel<4, 8>" if cols_per_sm < 1024 else "gae_single_kernel<4, 4>"))
        gae_roof = {"bound": "hbm", "kernel": gae_kernel, "shape": [Tg, Ng], "achieved": gbytes / (gms * 1e-3) / 1e9,
                    "peak": hbm_peak, "unit": "GB/s", "frac": gbytes / (gms * 1e-3) / 1e9 / hbm_peak,
                    "frac_of_8TBs_spec": gbytes / (gms * 1e-3) / 1e9 / 8000.0, "bytes_per_transition": 17, "ms": gms,
                    "peak_source": peak_src}
        del r_, v_, d_, lv_, gm

        # ---- the rollout's policy step (minppo_policy_step, train.py:157-160) on this config's env count ---------
        pol = None
        try:
            pobs = torch.randn(hp.num_envs // world, D_OBS, device=dev)
            for _ in range(5):
                learner.policy_step(ts.params, pobs, rng, weights_current=True)
            torch.cuda.synchronize(dev)
            p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            p0.record()
            for _ in range(50):
                learner.policy_step(ts.params, pobs, rng, weights_current=True)
            p1.record()
            torch.cuda.synchronize(dev)
            pol = {"us_per_env_step": p0.elapsed_time(p1) / 50 * 1e3, "envs": hp.num_envs // world,
                   "note": "eager call through the Python host (one fused launch: observation conversion + both hidden "
                           "layers + heads + sampler), weights current"}
            # the same call captured once into a CUDA graph and replayed (what a captured T-step rollout pays per env step)
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            pg = torch.cuda.CUDAGraph()
            with torch.cuda.stream(side):
                with torch.cuda.graph(pg, stream=side):
                    learner.policy_step(ts.params, pobs, rng, weights_current=True)
            torch.cuda.current_stream(dev).wait_stream(side)
            for _ in range(5):
                pg.replay()
            torch.cuda.synchronize(dev)
            p0.record()
            for _ in range(200):
                pg.replay()
            p1.record()
            torch.cuda.synchronize(dev)
            pol["graph_replay_us_per_env_step"] = p0.elapsed_time(p1) / 200 * 1e3
            # T = 32 consecutive policy steps (rng chained through two ping-pong keys) captured as ONE graph: what the
            # network evaluation of a captured rollout costs per env step once the per-launch host cost is amortised
            Tr = 32
            keys = [rng.clone(), torch.empty_like(rng)]
            pact = torch.empty((hp.num_envs // world, D_ACT), dtype=torch.float32, device=dev)
            plp = torch.empty((hp.num_envs // world,), dtype=torch.float32, device=dev)
            pval = torch.empty_like(plp)
            rg = torch.cuda.CUDAGraph()
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                with torch.cuda.graph(rg, stream=side):
                    for t_ in range(Tr):
                        _lib.check(learner.lib.minppo_policy_step(
                            learner._h, ts.params.data_ptr(), pobs.data_ptr(), keys[t_ % 2].data_ptr(), keys[(t_ + 1) % 2].data_ptr(),
                            pact.data_ptr(), plp.data_ptr(), pval.data_ptr(), None, _lib.POLICY_WEIGHTS_CURRENT,
                            torch.cuda.current_stream(dev).cuda_stream))
            torch.cuda.current_stream(dev).wait_stream(side)
            for _ in range(3):
                rg.replay()
            torch.cuda.synchronize(dev)
            p0.record()
            for _ in range(20):
                rg.replay()
            p1.record()
            torch.cuda.synchronize(dev)
            pol["rollout_graph_us_per_env_step"] = p0.elapsed_time(p1) / (20 * Tr) * 1e3
            pol["rollout_graph_steps"] = Tr
        except Exception as e:  # a measurement extra must never lose the bench line
            pol = {"error": str(e)[:200]}

        # ---- CPU baseline beside it, the parity check at THIS shape, and the GPU proxy (N == 1 only) -------------
        cpu = None
        parity = None
        proxy = None
        if world == 1 and not args.no_cpu_baseline:
            t_cpu, cores, cpu_losses = cpu_update_time(hp, 1, (D_OBS, D_ACT))
            cpu = {"value": B / t_cpu, "unit": UNIT, "cores": cores, "kind": "port", "sample": CPU_SAMPLE,
                   "ms_per_update": t_cpu * 1e3}
            # parity at the benchmarked shape, outside the timed region: ONE update from the SAME initial state through
            # the product path, all E*M losses against the CPU restatement's (fp32 GEMMs there, bf16 tensor-core GEMMs
            # here: tolerance 1e-2 of the largest loss; tests/test_gpu_update.py holds the same shape to 2e-3 against the
            # oracle with the bf16 rounding points emulated)
            ts0 = TrainState.create(flat, dev)
            fresh = torch.empty_like(losses)
            learner.update(ts0, mem, lv, rng, fresh, rng_out)
            torch.cuda.synchronize(dev)
            gl = fresh.cpu().numpy().astype(np.float64)
            err = float(np.abs(gl - cpu_losses).max() / np.abs(cpu_losses).max())
            parity = {"parity_at_bench_shape": bool(np.isfinite(err) and err < 1e-2), "max_rel_err_losses": err,
                      "tolerance": 1e-2, "losses_compared": int(gl.size),
                      "first_loss_gpu": [float(x) for x in gl[0, 0]], "first_loss_cpu": [float(x) for x in cpu_losses[0, 0]],
                      "last_loss_gpu": [float(x) for x in gl[-1, -1]], "last_loss_cpu": [float(x) for x in cpu_losses[-1, -1]]}
            if not parity["parity_at_bench_shape"]:
                print(json.dumps({"error": "parity check at the benchmarked shape FAILED", **parity}), file=sys.stderr, flush=True)
        if world == 1 and not args.no_gpu_proxy:
            try:
                proxy = gpu_proxy_time(hp, dev, steps=3, try_compile=bool(args.proxy_compile), dims=(D_OBS, D_ACT))
                pl = proxy.pop("_losses")
                if cpu is not None:
                    proxy["losses_vs_cpu_restatement"] = float(np.abs(pl - cpu_losses).max() / np.abs(cpu_losses).max())
                proxy["speedup_of_this_repo_over_eager_proxy"] = proxy["eager_ms_per_update"] / ms_per_step
                if "compiled_ms_per_update" in proxy:
                    proxy["speedup_of_this_repo_over_compiled_proxy"] = proxy["compiled_ms_per_update"] / ms_per_step
                proxy["north_star_target"] = ">= 20x the reference JAX-on-GPU learner (not measurable here; this proxy stands in)"
            except Exception as e:  # a comparator must never lose the bench line
                proxy = {"error": (type(e).__name__ + ": " + str(e))[:300]}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": w["scaling"],
            "vs_baseline": None, "dtype": "bf16 tensor-core GEMMs (fp32 accumulate), fp32 elsewhere", "data": "synthetic",
            "config": bench_config(w, world, (D_OBS, D_ACT), hp, bool(args.fast_tanh)),
            "sample_passes_per_s": value * hp.update_epochs,
            "clocks": clocks,
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": e2e_h2d, "d2h_bytes_per_step": e2e_d2h,
                    "ms_per_step": float(et.item()) * 1e3,
                    "api": "HostPipeline.submit / result: pinned-host trajectory H2D and params + losses + rng D2H EVERY update, "
                           "train state resident on the device, two updates in flight (the copy of update i + 1 runs under "
                           "the kernels of update i)"},
            "e2e_blocking": e2e_blocking,
            "gpu_launches": learner.launches_per_update() * args.steps,
            "launches_per_update": learner.launches_per_update(),
            "roofline": roofline, "gae_roofline": gae_roof, "kernel_classes": prof, "policy_step": pol,
            "final_loss": [float(x) for x in final_losses[-1, -1]],
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if parity is not None:
            line.update(parity)
        if proxy is not None:
            line["gpu_proxy"] = proxy
        print(json.dumps(line), flush=True)
    learner.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "torch_gpu"])
    ap.add_argument("--fast-tanh", type=int, default=1, help="library default (config.learner.fast_tanh)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-proxy", action="store_true")
    ap.add_argument("--proxy-compile", type=int, default=1, help="also time the GPU proxy under torch.compile if it works offline")
    ap.add_argument("--obs-dim", type=int, default=OBS_DIM, help="observation width (default: the declared stand-in)")
    ap.add_argument("--act-dim", type=int, default=ACT_DIM, help="action width (default: the declared stand-in)")
    ap.add_argument("--workload", default="auto", choices=["auto", "c4"],
                    help="auto: configs[1] per GPU (weak scaling); c4: configs[3] global batch (strong scaling)")
    ap.add_argument("--quick", action="store_true", help="device-resident timing only (development)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (params, mu, nu, step, rng_out, "
                         "losses) as DIR/<name>.npy, under 64 MB in all (a seeded sample of larger outputs); "
                         "--impl ours only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "reference":
        run_reference(args)
    elif args.impl == "torch_gpu":
        run_torch_gpu(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
