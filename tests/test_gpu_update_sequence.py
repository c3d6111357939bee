"""Consecutive updates on one context equal fresh-context updates bit for bit.

dwopt_kernel's split-K completion counters live in the context and must be back at zero after every launch: a count
left over from the previous minibatch step or update would let phase 2 read partials before they are written.  One
context runs two updates through its CUDA graph (capture, then replay) and a third enqueued directly; each must equal
the same update run on a fresh context from the same starting state.  The two-launch shape (D = 1000 with 4 dW splits:
160 GEMM CTAs, more than one per SM) runs dwopt without GEMM CTAs after the stand-alone GEMM: its spare CTAs count the
small-leaf counter up, and that counter too must be back at zero."""
import numpy as np
import pytest

from oracle import ppo_numpy as P
from oracle import synth
from tests.gradient_cases import learner_path
from tests.helpers import hyper_to_config

pytestmark = pytest.mark.gpu


def _memory(problem, device):
    import torch

    from minppo_b200.learner import Memory

    t = lambda x: torch.as_tensor(np.ascontiguousarray(x)).to(device)
    tr = problem["traj"]
    return Memory(done=t(tr["done"]), action=t(tr["action"]), value=t(tr["value"]), reward=t(tr["reward"]),
                  log_prob=t(tr["log_prob"]), obs=t(tr["obs"])), t(problem["last_val"])


def _snapshot(ts, rng):
    return [x.clone() for x in (ts.params, ts.mu, ts.nu, ts.step, rng)]


@pytest.mark.parametrize("fused,D,extra", [(True, 225, {}), (False, 225, {}), (True, 1000, dict(dw_splits=4))],
                         ids=["True", "False", "two_launch"])
def test_graph_replays_then_direct_update_equal_fresh_contexts(fused, D, extra, cuda_device):
    import torch

    from minppo_b200.learner import Learner, TrainState

    hp_kw = dict(num_envs=64, num_steps=32, num_minibatches=4, update_epochs=2, anneal_lr=True)
    hp = P.Hyper(**hp_kw)
    path = learner_path(hp_kw, D, 10, torch.cuda.get_device_properties(cuda_device).multi_processor_count,
                        dict(extra, fused=fused))
    assert path["two_launch"] == bool(extra), path
    pr = synth.make_problem(hp, D, 10, seed=11, done_p=0.02)
    cfg = hyper_to_config(hp, use_graph=True, fused=fused, **extra)
    mem, lv = _memory(pr, cuda_device)

    lrn = Learner(cfg, D, 10, cuda_device)
    ts = TrainState.create(P.flatten_params(pr["params"], hp.num_layers), cuda_device)
    rng = torch.as_tensor(pr["rng"].view(np.int32)).to(cuda_device)
    runs = []
    for k in range(3):
        lrn.use_graph = k < 2                  # capture + launch, replay, then enqueued directly
        start = _snapshot(ts, rng)
        ts, rng_out, losses = lrn.update(ts, mem, lv, rng)
        lrn.check()
        assert lrn.launches_per_update() == path["launches"], path
        rng = rng_out.clone()
        runs.append((start, [x.clone() for x in (ts.params, ts.mu, ts.nu, ts.step, rng_out, losses)]))
    lrn.close()

    for k, (start, got) in enumerate(runs):
        fresh = Learner(cfg, D, 10, cuda_device)
        p0, m0, n0, s0, r0 = start
        ts = TrainState(params=p0.clone(), mu=m0.clone(), nu=n0.clone(), step=s0.clone())
        ts, rng_out, losses = fresh.update(ts, mem, lv, r0.clone())
        fresh.check()
        want = (ts.params, ts.mu, ts.nu, ts.step, rng_out, losses)
        for name, g, w in zip(("params", "mu", "nu", "step", "rng", "losses"), got, want):
            assert torch.equal(g, w), (k, name)
        fresh.close()
