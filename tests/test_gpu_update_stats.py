"""Per-minibatch PPO statistics of ``Learner.update(..., stats=...)`` (include/minppo_b200.h, minppo_update_with_stats):
approx_kl, clip_fraction, value_clip_fraction and grad_norm of every minibatch step.

* Passing ``stats`` changes nothing else: parameters, moments, step, rng, losses, the reduced gradient and the launch
  count are bitwise those of an update without it, with and without the CUDA graph.
* Parity at every step against tests/update_stats_reference.py run with the kernels' bf16 rounding points (float32,
  gemm="bf16"), on the fused path, the layer-wise path (num_layers 1 and 3), act_dim 48, hidden_size 512, the
  two-launch path and a narrow clip_eps.  Tolerances:
  - approx_kl: |gpu - ref| <= KL_REL * max|ref| + KL_ABS.  KL is a mean of (r - 1) - log r, so an error in log r of
    the size the losses carry (they are held to 2e-3 of their largest value in tests/test_gpu_update.py) moves it by
    about |log r| times that error.  Measured on a B200 (1000 W): at most 1.7e-4 of max|ref| over these cases (a
    narrow clip_eps, whose parameters drift furthest from the reference's); bound 2e-3, like the losses.
  - clip fractions are counts: a row whose |r - 1| or |v - v_old| lies within rounding of clip_eps may land on
    either side.  The reference also counts the rows within DELTA of the boundary; GPU and reference counts may
    differ by at most that number.  DELTA = 1e-3 covers the drift of r and v between the two implementations after
    several Adam steps (the per-step parameters differ by a few bf16 ulps); measured count differences were 0 on every
    step of these cases.
  - grad_norm is bitwise the norm buffer the context already keeps (``read("grad_norms")``).
* Rollout consistency: log_prob from ``Learner.policy_step`` at the starting parameters gives clip_fraction == 0 and
  approx_kl at rounding level at step (0, 0).
* A raised device error flag (row-list overflow) makes every statistic NaN.
* Graph handling: ping-pong ``stats`` buffers replay the cached graphs; a caller's capture with use_graph = False
  reproduces the directly enqueued statistics bit for bit.
* Multi-GPU: tests/multigpu/check_sharded_update_stats.py under torchrun (skipped below 2 GPUs).
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import ppo_numpy as P
from oracle import synth
from tests.helpers import hyper_to_config, perturb_policy, rel_err
from tests.update_stats_reference import update_with_stats

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

KL_REL, KL_ABS = 2e-3, 1e-7
DELTA = 1e-3
METRICS = {}


@pytest.fixture(scope="module", autouse=True)
def _dump_metrics():
    """MINPPO_TEST_METRICS_DIR: where to write the measured errors (update_stats_metrics.json)."""
    yield
    out = os.environ.get("MINPPO_TEST_METRICS_DIR")
    if out:
        os.makedirs(out, exist_ok=True)
        with open(os.path.join(out, "update_stats_metrics.json"), "w") as f:
            json.dump(METRICS, f, indent=1, sort_keys=True)


def _inputs(pr, hp, device):
    import torch

    from minppo_b200.learner import Memory, TrainState

    t = lambda x: torch.as_tensor(np.ascontiguousarray(x)).to(device)
    tr = pr["traj"]
    mem = Memory(done=t(tr["done"]), action=t(tr["action"]), value=t(tr["value"]), reward=t(tr["reward"]),
                 log_prob=t(tr["log_prob"]), obs=t(tr["obs"]))
    ts = TrainState.create(P.flatten_params(pr["params"], hp.num_layers), device)
    rng = torch.as_tensor(pr["rng"].view(np.int32)).to(device)
    return ts, mem, t(pr["last_val"]), rng


def _stats_buf(hp, device, fill=float("nan")):
    import torch

    return torch.full((hp.update_epochs, hp.num_minibatches, 4), fill, dtype=torch.float32, device=device)


def check_stats(got, ref, ambiguous, mb: int, label: str = ""):
    """Assert GPU statistics ``got`` [E, M, 4] against the reference ``ref`` with its ambiguous-row counts; returns the
    measured errors.  (Also used by tests/multigpu/check_sharded_update_stats.py.)"""
    got = np.asarray(got, np.float64)
    ref = np.asarray(ref, np.float64)
    assert np.all(np.isfinite(got)), label
    kl_err = np.abs(got[..., 0] - ref[..., 0]).max()
    kl_scale = np.abs(ref[..., 0]).max()
    dcount = np.abs(np.rint(got[..., 1:3] * mb) - np.rint(ref[..., 1:3] * mb))
    m = {"kl_err_rel_to_max": float(kl_err / max(kl_scale, 1e-30)), "kl_max": float(kl_scale),
         "clip_count_diff_max": int(dcount[..., 0].max()), "vclip_count_diff_max": int(dcount[..., 1].max()),
         "ambiguous_max": [int(x) for x in ambiguous.max(axis=(0, 1))],
         "clip_fraction_mean": float(ref[..., 1].mean()), "vclip_fraction_mean": float(ref[..., 2].mean()),
         "gnorm_rel_err": rel_err(got[..., 3], ref[..., 3])}
    assert kl_err <= KL_REL * kl_scale + KL_ABS, (label, m)
    assert np.all(dcount <= ambiguous), (label, m, np.argwhere(dcount > ambiguous)[:8].tolist())
    assert m["gnorm_rel_err"] < 2e-2, (label, m)
    return m


def _run_with_stats(hp, pr, device, **cfg_kw):
    import torch

    from minppo_b200.learner import Learner

    lrn = Learner(hyper_to_config(hp, **cfg_kw), pr["obs_dim"], pr["act_dim"], device)
    ts, mem, lv, rng = _inputs(pr, hp, device)
    stats = _stats_buf(hp, device)
    lrn.update(ts, mem, lv, rng, stats=stats)
    lrn.check()
    out = {"stats": stats.cpu().numpy(), "grad_norms": lrn.read("grad_norms").cpu().numpy(),
           "losses": lrn._losses.cpu().numpy()}
    lrn.close()
    torch.cuda.synchronize(device)
    return out


# name: (hyper-parameters, D, A, learner config)
PARITY_CASES = {
    # fused step kernel (num_layers = 2, act_dim <= 32, hidden_size <= 256)
    "fused_wide_tanh": (dict(num_envs=64, num_steps=32, num_minibatches=4, update_epochs=2, anneal_lr=False), 415, 20, {}),
    "fused_a17_relu": (dict(num_envs=32, num_steps=16, num_minibatches=2, update_epochs=2, anneal_lr=False,
                            hidden_size=128, use_tanh=False), 600, 17, {}),
    "fused_a24_h64": (dict(num_envs=32, num_steps=8, num_minibatches=2, update_epochs=2, anneal_lr=False,
                           hidden_size=64, ent_coef=0.01), 100, 24, {}),
    # layer-wise kernels (head_loss.cu)
    "layerwise_l1": (dict(num_envs=24, num_steps=16, num_minibatches=3, update_epochs=2, anneal_lr=False,
                          hidden_size=128, num_layers=1, ent_coef=0.01), 37, 3, dict(fused=False)),
    "layerwise_l3_relu": (dict(num_envs=32, num_steps=16, num_minibatches=2, update_epochs=2, anneal_lr=False,
                               hidden_size=192, num_layers=3, use_tanh=False), 256, 16, dict(fused=False)),
    "layerwise_l2": (dict(num_envs=64, num_steps=32, num_minibatches=4, update_epochs=2, anneal_lr=False), 225, 10,
                     dict(fused=False)),
    # act_dim 48: head_loss_kernel<64>
    "a48": (dict(num_envs=32, num_steps=16, num_minibatches=2, update_epochs=2, anneal_lr=False), 64, 48, {}),
    # hidden_size 512: two column groups per hidden layer
    "h512": (dict(num_envs=32, num_steps=16, num_minibatches=2, update_epochs=2, anneal_lr=False, hidden_size=512),
             64, 10, {}),
    # stand-alone dW GEMM launch, then dwopt without GEMM CTAs
    "two_launch": (dict(num_envs=32, num_steps=16, num_minibatches=2, update_epochs=1, anneal_lr=False), 1000, 10,
                   dict(dw_splits=4)),
    # a narrow clip: many rows near both boundaries
    "fused_clip005": (dict(num_envs=64, num_steps=32, num_minibatches=4, update_epochs=2, anneal_lr=False,
                           clip_eps=0.05), 225, 10, {}),
}


@pytest.mark.parametrize("name", list(PARITY_CASES))
def test_stats_match_the_reference_at_every_step(name, cuda_device):
    kw, D, A, cfg = PARITY_CASES[name]
    hp = P.Hyper(**kw)
    pr = synth.make_problem(hp, D, A, seed=7, done_p=0.02)
    perturb_policy(pr)
    got = _run_with_stats(hp, pr, cuda_device, **cfg)
    p0 = P.tree_like(pr["params"], lambda x: x.astype(np.float32))
    _, _, _, lref, aux = update_with_stats(p0, P.init_opt_state(p0), pr["traj"], pr["last_val"], pr["rng"], hp,
                                           dtype=np.float32, gemm="bf16", delta=DELTA)
    # grad_norm column: bitwise the context's own norm buffer
    assert np.array_equal(got["stats"][..., 3].ravel(), got["grad_norms"])
    m = check_stats(got["stats"], aux["stats"], aux["ambiguous"], hp.minibatch_size, name)
    m["loss_vs_reference"] = rel_err(got["losses"], lref)
    METRICS[name] = m
    # the perturbed trajectory clips on both losses: the counts are not trivially zero
    assert aux["stats"][..., 1].max() > 0 and aux["stats"][..., 2].max() > 0


CHANGE_CASES = {
    "fused": (dict(num_envs=64, num_steps=32, num_minibatches=4, update_epochs=2, anneal_lr=True), 225, 10, {}),
    "layerwise": (dict(num_envs=64, num_steps=32, num_minibatches=4, update_epochs=2, anneal_lr=True), 225, 10,
                  dict(fused=False)),
    "two_launch": PARITY_CASES["two_launch"],
}


@pytest.mark.parametrize("use_graph", [True, False])
@pytest.mark.parametrize("name", list(CHANGE_CASES))
def test_stats_change_nothing_else(name, use_graph, cuda_device):
    import torch

    from minppo_b200.learner import Learner

    kw, D, A, cfg = CHANGE_CASES[name]
    hp = P.Hyper(**kw)
    pr = synth.make_problem(hp, D, A, seed=3, done_p=0.02)
    perturb_policy(pr)
    lrn = Learner(hyper_to_config(hp, use_graph=use_graph, **cfg), D, A, cuda_device)
    ts, mem, lv, rng = _inputs(pr, hp, cuda_device)
    start = [x.clone() for x in (ts.params, ts.mu, ts.nu, ts.step)]
    losses = torch.empty((hp.update_epochs, hp.num_minibatches, 4), device=cuda_device)
    rng_out = torch.empty_like(rng)
    P_ = lrn.P

    def run(stats):
        for dst, src in zip((ts.params, ts.mu, ts.nu, ts.step), start):
            dst.copy_(src)
        losses.zero_()
        lrn.update(ts, mem, lv, rng, losses, rng_out, stats=stats)
        lrn.check()
        res = [x.clone() for x in (ts.params, ts.mu, ts.nu, ts.step, rng_out, losses)]
        res += [lrn.read("grad")[:P_ + 2], lrn.read("grad_norms")]
        return res, lrn.launches_per_update()

    a, la = run(None)
    stats = _stats_buf(hp, cuda_device)
    b, lb = run(stats)
    c, lc = run(None)
    assert la == lb == lc
    names = ("params", "mu", "nu", "step", "rng", "losses", "grad[:P+2]", "grad_norms")
    for n, x, y, z in zip(names, a, b, c):
        assert torch.equal(x, y) and torch.equal(x, z), n
    assert torch.isfinite(stats).all()
    assert torch.equal(stats[..., 3].reshape(-1), a[-1])
    lrn.close()


@pytest.mark.parametrize("fused", [True, False])
def test_rollout_log_prob_gives_zero_kl_and_no_clipping_at_the_first_step(fused, cuda_device):
    """The trajectory's actions, log-probs and values come from Learner.policy_step at the starting parameters (the
    rollout of train.py:157-160): the first minibatch step evaluates the same policy, so r == 1 up to rounding."""
    import torch

    from minppo_b200.learner import Learner, Memory

    hp = P.Hyper(num_envs=64, num_steps=32, num_minibatches=4, update_epochs=2, anneal_lr=False)
    pr = synth.make_problem(hp, 225, 10, seed=5, done_p=0.02)
    lrn = Learner(hyper_to_config(hp, fused=fused), 225, 10, cuda_device)
    ts, mem, lv, rng = _inputs(pr, hp, cuda_device)
    acts, logps, vals = [], [], []
    key = rng
    for t in range(hp.num_steps):
        a, lp, v, key, _ = lrn.policy_step(ts.params, mem.obs[t].contiguous(), key)
        acts.append(a), logps.append(lp), vals.append(v)
    mem = Memory(done=mem.done, action=torch.stack(acts), value=torch.stack(vals), reward=mem.reward,
                 log_prob=torch.stack(logps), obs=mem.obs)
    stats = _stats_buf(hp, cuda_device)
    lrn.update(ts, mem, lv, rng, stats=stats)
    lrn.check()
    st = stats.cpu().numpy()
    METRICS[f"rollout_fused={fused}"] = {"kl_00": float(st[0, 0, 0]), "clip_00": float(st[0, 0, 1]),
                                         "kl_last": float(st[-1, -1, 0])}
    assert st[0, 0, 1] == 0.0
    assert abs(st[0, 0, 0]) < 1e-6
    assert st[-1, -1, 0] > 10 * abs(st[0, 0, 0])       # later steps see updated parameters
    lrn.close()


def test_row_list_overflow_makes_every_statistic_nan(cuda_device, monkeypatch):
    import torch

    from minppo_b200 import _lib
    from minppo_b200.learner import Learner

    monkeypatch.setenv("MINPPO_FORCE_CAP", "256")                # minibatches have 512 rows
    hp = P.Hyper(num_envs=64, num_steps=32, num_minibatches=4, update_epochs=2, anneal_lr=True)
    pr = synth.make_problem(hp, 225, 10, seed=3)
    lrn = Learner(hyper_to_config(hp), 225, 10, cuda_device)
    monkeypatch.delenv("MINPPO_FORCE_CAP")
    ts, mem, lv, rng = _inputs(pr, hp, cuda_device)
    stats = _stats_buf(hp, cuda_device, fill=0.0)
    _, _, losses = lrn.update(ts, mem, lv, rng, stats=stats)
    torch.cuda.synchronize(cuda_device)
    assert torch.isnan(losses).all()
    assert torch.isnan(stats).all()
    with pytest.raises(_lib.MinppoError):
        lrn.check()
    lrn.close()


def test_ping_pong_stats_buffers_replay_and_match_eager(cuda_device):
    """Four consecutive updates writing their statistics alternately into two buffers: with use_graph the two pointer
    sets are two cached graphs, replayed; every update's statistics equal those of the directly enqueued run."""
    import torch

    from minppo_b200.learner import Learner

    hp = P.Hyper(num_envs=64, num_steps=32, num_minibatches=4, update_epochs=2, anneal_lr=True)
    pr = synth.make_problem(hp, 225, 10, seed=8, done_p=0.02)
    perturb_policy(pr)
    results = {}
    for use_graph in (True, False):
        lrn = Learner(hyper_to_config(hp, use_graph=use_graph), 225, 10, cuda_device)
        ts, mem, lv, rng = _inputs(pr, hp, cuda_device)
        bufs = [_stats_buf(hp, cuda_device), _stats_buf(hp, cuda_device)]
        rng_out = torch.empty_like(rng)
        seq = []
        for i in range(4):
            lrn.update(ts, mem, lv, rng, stats=bufs[i % 2], rng_out=rng_out)
            rng = rng_out.clone()
            seq.append(bufs[i % 2].clone())
        lrn.check()
        results[use_graph] = (seq, ts.params.clone())
        lrn.close()
    for i, (g, e) in enumerate(zip(results[True][0], results[False][0])):
        assert torch.isfinite(g).all() and torch.equal(g, e), i
    assert not torch.equal(results[True][0][0], results[True][0][2])     # the training moved on between the updates
    assert torch.equal(results[True][1], results[False][1])


def test_callers_capture_reproduces_eager_stats(cuda_device):
    import torch

    from minppo_b200.learner import Learner

    hp = P.Hyper(num_envs=64, num_steps=32, num_minibatches=4, update_epochs=2, anneal_lr=True)
    pr = synth.make_problem(hp, 225, 10, seed=5, done_p=0.02)
    perturb_policy(pr)
    cfg = hyper_to_config(hp, use_graph=False)

    lrn = Learner(cfg, 225, 10, cuda_device)
    ts, mem, lv, rng = _inputs(pr, hp, cuda_device)
    want = _stats_buf(hp, cuda_device)
    lrn.update(ts, mem, lv, rng, stats=want)
    lrn.check()
    lrn.close()

    lrn = Learner(cfg, 225, 10, cuda_device)
    ts, mem, lv, rng = _inputs(pr, hp, cuda_device)
    p0, m0, n0, s0 = ts.params.clone(), ts.mu.clone(), ts.nu.clone(), ts.step.clone()
    stats = _stats_buf(hp, cuda_device, fill=0.0)
    losses = torch.zeros((hp.update_epochs, hp.num_minibatches, 4), device=cuda_device)
    rng_out = torch.zeros_like(rng)
    side = torch.cuda.Stream(device=cuda_device)
    side.wait_stream(torch.cuda.current_stream(cuda_device))
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            lrn.update(ts, mem, lv, rng, losses, rng_out, stats=stats)
    torch.cuda.current_stream(cuda_device).wait_stream(side)
    torch.cuda.synchronize(cuda_device)
    assert not torch.isnan(stats).any() and (stats == 0).all(), "capture must not execute anything"
    for rep in range(2):
        ts.params.copy_(p0); ts.mu.copy_(m0); ts.nu.copy_(n0); ts.step.copy_(s0)
        stats.zero_()
        graph.replay()
        torch.cuda.synchronize(cuda_device)
        lrn.check()
        assert torch.equal(stats, want), rep
    lrn.close()


def test_sharded_update_stats_all_visible_gpus():
    import torch

    n = torch.cuda.device_count() if torch.cuda.is_available() else 0
    if n < 2:
        pytest.skip("needs >= 2 GPUs on one box")
    n = 8 if n >= 8 else (4 if n >= 4 else 2)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
                        "--master-addr", "127.0.0.1", "--master-port", "29613",
                        os.path.join(ROOT, "tests", "multigpu", "check_sharded_update_stats.py")],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0 and "MULTIGPU STATS OK" in r.stdout, (r.stdout[-3000:], r.stderr[-3000:])
