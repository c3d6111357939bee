"""Running observation normalization on the GPU (include/minppo_b200.h, minppo_obs_norm; minppo_b200.obs_norm).

1. ``Learner.update(..., obs_norm=S)`` is bitwise the update without normalization on observations normalized on the
   host (tests/obs_norm_reference.py normalize_obs, float32): params, mu, nu, step, rng, losses and statistics, on the
   fused and the layer-wise paths, hidden_size 384, act_dim 48, num_layers 3 and obs_dim 37, with and without the CUDA
   graph.  S has random means, variances over 1e-4 ... 1e4 and a clip that clamps entries.
2. The statistics it leaves equal the float64 fold of the batch (fold_obs_stats): count exactly, mean within
   1e-6 (|mu| + sigma), var within 1e-5 relative (1e-4 on data at 1e4 +- 1e-2, where a sum of squares would fail);
   three updates equal the fold of their concatenation; two runs and ``ObsNormalizer.fold`` give the same bits.  The
   stand-alone fold is checked the same way at D = 37, 415 and 1000 (every register layout of the moments kernel),
   with 2^20 + 3 rows at D = 37.
3. ``policy_step`` (sampled and mode) and ``bootstrap_value`` with S are bitwise the calls on host-normalized
   observations without it, on both paths, and leave S unchanged.
4. The graph cache keys on clip: the same buffers with another clip replay a graph of their own.
5. InferencePolicy normalizes when the checkpoint carries "obs_normalizer".
6. Multi-GPU: tests/multigpu/check_sharded_update_obs_norm.py under torchrun (skipped below 2 GPUs).
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import ppo_numpy as P
from oracle import synth
from tests.helpers import hyper_to_config, perturb_policy
from tests.obs_norm_reference import fold_obs_stats, normalize_obs
from tests.test_gpu_update_stats import _inputs, _stats_buf

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

MEAN_TOL, VAR_TOL, VAR_TOL_OFFSET = 1e-6, 1e-5, 1e-4


def make_stats(D: int, device, seed: int = 11, clip: float = 5.0, count: float = 1000.0):
    """A non-trivial ObsNormalizer: means N(0, 0.5), variances log-uniform over 1e-4 ... 1e4 (the small ones push
    N(0, 1) observations far past the clip)."""
    import torch

    from minppo_b200.obs_norm import ObsNormalizer

    g = np.random.default_rng(seed)
    mean = (0.5 * g.standard_normal(D)).astype(np.float32)
    var = (10.0 ** g.uniform(-4, 4, D)).astype(np.float32)
    t = lambda x: torch.as_tensor(x).to(device)
    return ObsNormalizer(t(mean), t(var), t(np.array([count])), 1e-8, clip)


def host(n):
    return n.mean.cpu().numpy(), n.var.cpu().numpy(), float(n.count.item())


def check_fold(got, want, offset: bool = False, label: str = ""):
    """got: (mean, var, count) from the GPU; want: the float64 fold."""
    gm, gv, gc = got
    wm, wv, wc = want
    assert gc == wc, (label, gc, wc)
    sig = np.sqrt(wv)
    merr = np.abs(gm.astype(np.float64) - wm) / (np.abs(wm) + sig)
    verr = np.abs(gv.astype(np.float64) - wv) / wv
    assert merr.max() <= MEAN_TOL, (label, float(merr.max()))
    assert verr.max() <= (VAR_TOL_OFFSET if offset else VAR_TOL), (label, float(verr.max()))
    return float(merr.max()), float(verr.max())


# name: (hyper-parameters, D, A, learner config)
SHAPES = {
    "fused_default": (dict(), 225, 10, {}),
    "layerwise": (dict(), 225, 10, dict(fused=False)),
    "h384": (dict(hidden_size=384), 225, 10, {}),
    "a48": (dict(), 225, 48, {}),
    "l3": (dict(num_layers=3, hidden_size=128), 225, 10, {}),
    "d37": (dict(), 37, 10, {}),
}
BASE = dict(num_envs=64, num_steps=32, num_minibatches=4, update_epochs=2, anneal_lr=True)


def _with_obs(mem, obs):
    from minppo_b200.learner import Memory

    return Memory(done=mem.done, action=mem.action, value=mem.value, reward=mem.reward, log_prob=mem.log_prob, obs=obs)


@pytest.mark.parametrize("use_graph", [True, False])
@pytest.mark.parametrize("name", list(SHAPES))
def test_update_equals_update_on_prenormalized_obs(name, use_graph, cuda_device):
    import torch

    from minppo_b200.learner import Learner

    kw, D, A, cfg = SHAPES[name]
    hp = P.Hyper(**{**BASE, **kw})
    pr = synth.make_problem(hp, D, A, seed=4, done_p=0.02)
    perturb_policy(pr)
    lrn = Learner(hyper_to_config(hp, use_graph=use_graph, **cfg), D, A, cuda_device)
    ts, mem, lv, rng = _inputs(pr, hp, cuda_device)
    S = make_stats(D, cuda_device)
    s0 = [x.clone() for x in (S.mean, S.var, S.count)]
    m, v, _ = host(S)
    pre = normalize_obs(pr["traj"]["obs"], m, v, S.eps, S.clip)
    assert np.abs(pre).max() == np.float32(S.clip)                # the clip is reached
    mem_pre = _with_obs(mem, torch.as_tensor(pre).to(cuda_device))
    start = [x.clone() for x in (ts.params, ts.mu, ts.nu, ts.step)]
    losses = torch.empty((hp.update_epochs, hp.num_minibatches, 4), device=cuda_device)
    rng_out = torch.empty_like(rng)
    stats = _stats_buf(hp, cuda_device)

    def run(memb, norm):
        for dst, src in zip((ts.params, ts.mu, ts.nu, ts.step), start):
            dst.copy_(src)
        lrn.update(ts, memb, lv, rng, losses, rng_out, stats=stats, obs_norm=norm)
        lrn.check()
        return [x.clone() for x in (ts.params, ts.mu, ts.nu, ts.step, rng_out, losses, stats)], lrn.launches_per_update()

    a, la = run(mem, S)
    assert float(S.count.item()) == 1000.0 + hp.batch_size           # the fold ran
    for dst, src in zip((S.mean, S.var, S.count), s0):
        dst.copy_(src)
    b, lb = run(mem_pre, None)
    assert all(torch.equal(x, y) for x, y in zip((S.mean, S.var, S.count), s0))
    for n, x, y in zip(("params", "mu", "nu", "step", "rng", "losses", "stats"), a, b):
        assert torch.equal(x, y), (name, use_graph, n)
    assert la == lb + 2                                               # finalize + merge
    assert torch.isfinite(a[5]).all()
    lrn.close()


def _fold_problem(hp, D, A, seed, offset=0.0, scale=1.0):
    pr = synth.make_problem(hp, D, A, seed=seed, done_p=0.02)
    g = np.random.default_rng(seed + 7)
    pr["traj"]["obs"] = (offset + scale * g.standard_normal(pr["traj"]["obs"].shape)).astype(np.float32)
    return pr


@pytest.mark.parametrize("data", ["unit", "offset"])
def test_update_statistics_match_the_float64_fold(data, cuda_device):
    """unit: N(0, 1) observations folded into a non-trivial state (count 1000).  offset: 1e4 + 1e-2 N(0, 1) from count 0,
    so that the statistics are the batch's own moments, which a sum of squares could not resolve."""
    import torch

    from minppo_b200.learner import Learner
    from minppo_b200.obs_norm import ObsNormalizer

    hp = P.Hyper(**BASE)
    D, A = 225, 10
    offset, scale, count = (0.0, 1.0, 1000.0) if data == "unit" else (1e4, 1e-2, 0.0)
    pr = _fold_problem(hp, D, A, seed=2, offset=offset, scale=scale)
    lrn = Learner(hyper_to_config(hp), D, A, cuda_device)
    ts, mem, lv, rng = _inputs(pr, hp, cuda_device)
    S = make_stats(D, cuda_device, count=count)
    m, v, c = host(S)
    F = ObsNormalizer(S.mean.clone(), S.var.clone(), S.count.clone(), S.eps, S.clip)
    lrn.update(ts, mem, lv, rng, obs_norm=S)
    lrn.check()
    check_fold(host(S), fold_obs_stats(m, v, c, pr["traj"]["obs"]), offset=data == "offset", label=data)
    # the stand-alone fold of the same observations from the same state: bitwise the update's result
    F.fold(mem.obs)
    torch.cuda.synchronize(cuda_device)
    for x, y in zip((F.mean, F.var, F.count), (S.mean, S.var, S.count)):
        assert torch.equal(x, y), data
    lrn.close()


def test_update_statistics_are_bit_reproducible(cuda_device):
    import torch

    from minppo_b200.learner import Learner

    hp = P.Hyper(**BASE)
    pr = _fold_problem(hp, 225, 10, seed=3, offset=2.0, scale=3.0)
    out = []
    for use_graph in (True, True, False):
        lrn = Learner(hyper_to_config(hp, use_graph=use_graph), 225, 10, cuda_device)
        ts, mem, lv, rng = _inputs(pr, hp, cuda_device)
        S = make_stats(225, cuda_device)
        lrn.update(ts, mem, lv, rng, obs_norm=S)
        lrn.check()
        out.append([x.clone() for x in (S.mean, S.var, S.count, ts.params)])
        lrn.close()
    for o in out[1:]:
        assert all(torch.equal(x, y) for x, y in zip(out[0], o))


def test_three_updates_equal_the_fold_of_their_concatenation(cuda_device):
    from minppo_b200.learner import Learner
    from minppo_b200.obs_norm import ObsNormalizer

    hp = P.Hyper(**BASE)
    D, A = 225, 10
    lrn = Learner(hyper_to_config(hp), D, A, cuda_device)
    S = ObsNormalizer.create(D, cuda_device)
    obs = []
    for k in range(3):
        pr = _fold_problem(hp, D, A, seed=20 + k, offset=1.5 * k - 1.0, scale=0.5 + k)
        ts, mem, lv, rng = _inputs(pr, hp, cuda_device)
        lrn.update(ts, mem, lv, rng, obs_norm=S)
        obs.append(pr["traj"]["obs"].reshape(-1, D))
    lrn.check()
    want = fold_obs_stats(np.zeros(D), np.ones(D), 0.0, np.concatenate(obs))
    check_fold(host(S), want, label="three updates")
    lrn.close()


@pytest.mark.parametrize("D,rows", [(37, (1 << 20) + 3), (415, 70001), (1000, 20011)])
def test_stand_alone_fold_matches_the_float64_fold(D, rows, cuda_device):
    import torch

    from minppo_b200.obs_norm import ObsNormalizer

    g = np.random.default_rng(D)
    x = (g.uniform(-3, 3, D) + g.uniform(0.1, 4, D) * g.standard_normal((rows, D))).astype(np.float32)
    S = make_stats(D, cuda_device, count=333.0)
    m, v, c = host(S)
    S.fold(torch.as_tensor(x).to(cuda_device))
    check_fold(host(S), fold_obs_stats(m, v, c, x), label=f"D={D}")


def test_fold_refuses_obs_dim_past_the_moments_kernel(cuda_device):
    import torch

    from minppo_b200 import _lib
    from minppo_b200.obs_norm import ObsNormalizer

    S = ObsNormalizer.create(1100, cuda_device)
    with pytest.raises(_lib.MinppoError, match="obs_dim=1100 unsupported"):
        S.fold(torch.zeros((16, 1100), device=cuda_device))


@pytest.mark.parametrize("fused", [True, False])
def test_policy_step_equals_policy_step_on_prenormalized_obs(fused, cuda_device):
    import torch

    from minppo_b200.learner import Learner

    hp = P.Hyper(num_envs=300, num_steps=2, num_minibatches=2, update_epochs=1)
    D, A = 225, 10
    pr = synth.make_problem(hp, D, A, seed=9)
    lrn = Learner(hyper_to_config(hp, fused=fused), D, A, cuda_device)
    ts, mem, lv, rng = _inputs(pr, hp, cuda_device)
    obs = mem.obs[0].contiguous()
    S = make_stats(D, cuda_device)
    s0 = [x.clone() for x in (S.mean, S.var, S.count)]
    m, v, _ = host(S)
    pre = torch.as_tensor(normalize_obs(obs.cpu().numpy(), m, v, S.eps, S.clip)).to(cuda_device)
    for key in (rng, None):
        a = lrn.policy_step(ts.params, obs, key, want_mean=True, obs_norm=S)
        b = lrn.policy_step(ts.params, pre, key, want_mean=True)
        for x, y in zip(a, b):
            assert (x is None and y is None) or torch.equal(x, y), (fused, key is None)
    assert torch.equal(lrn.bootstrap_value(ts.params, obs, obs_norm=S), lrn.bootstrap_value(ts.params, pre))
    assert not torch.equal(lrn.bootstrap_value(ts.params, obs, obs_norm=S), lrn.bootstrap_value(ts.params, obs))
    torch.cuda.synchronize(cuda_device)
    assert all(torch.equal(x, y) for x, y in zip((S.mean, S.var, S.count), s0))
    lrn.close()


def test_graph_cache_keys_on_clip(cuda_device):
    """The same buffers with another clip must not replay the graph captured for the first clip."""
    import torch

    from minppo_b200.learner import Learner

    hp = P.Hyper(**BASE)
    D, A = 225, 10
    pr = synth.make_problem(hp, D, A, seed=6, done_p=0.02)
    lrn = Learner(hyper_to_config(hp, use_graph=True), D, A, cuda_device)
    ts, mem, lv, rng = _inputs(pr, hp, cuda_device)
    S = make_stats(D, cuda_device)
    s0 = [x.clone() for x in (S.mean, S.var, S.count)]
    start = [x.clone() for x in (ts.params, ts.mu, ts.nu, ts.step)]

    def run(clip, prenormalized):
        for dst, src in zip((ts.params, ts.mu, ts.nu, ts.step, S.mean, S.var, S.count), start + s0):
            dst.copy_(src)
        S.clip = clip
        if prenormalized:
            m, v, _ = host(S)
            memb = _with_obs(mem, torch.as_tensor(normalize_obs(pr["traj"]["obs"], m, v, S.eps, clip)).to(cuda_device))
            lrn.update(ts, memb, lv, rng)
        else:
            lrn.update(ts, mem, lv, rng, obs_norm=S)
        lrn.check()
        return ts.params.clone()

    p5, p2 = run(5.0, False), run(2.0, False)
    assert torch.equal(p5, run(5.0, True)) and torch.equal(p2, run(2.0, True))
    assert not torch.equal(p5, p2)
    lrn.close()


def test_inference_policy_normalizes_with_the_checkpoint_statistics(tmp_path, cuda_device):
    import torch

    from minppo_b200.infer import InferencePolicy
    from minppo_b200.params import save_model

    hp = P.Hyper(num_envs=256, num_steps=2, num_minibatches=2, update_epochs=1)
    D, A = 225, 10
    tree = P.tree_like(P.init_params(D, A, hp.hidden_size, hp.num_layers, seed=5), lambda x: x.astype(np.float32))
    S = make_stats(D, cuda_device)
    ckpt = os.path.join(tmp_path, "policy.pkl")
    save_model(tree, ckpt, obs_normalizer=S.to_tree())
    cfg = hyper_to_config(hp)
    with_norm = InferencePolicy.from_checkpoint(ckpt, cfg, hp.num_envs, cuda_device)
    plain = InferencePolicy(tree, cfg, hp.num_envs, cuda_device)
    assert with_norm.obs_norm is not None and plain.obs_norm is None
    obs = np.random.default_rng(0).standard_normal((hp.num_envs, D)).astype(np.float32)
    m, v, _ = host(S)
    a, va = with_norm.act(torch.as_tensor(obs).to(cuda_device))
    b, vb = plain.act(torch.as_tensor(normalize_obs(obs, m, v, S.eps, S.clip)).to(cuda_device))
    assert torch.equal(a, b) and torch.equal(va, vb)
    c, _ = plain.act(torch.as_tensor(obs).to(cuda_device))
    assert not torch.equal(a, c)
    with_norm.close(), plain.close()


def test_sharded_update_obs_norm_all_visible_gpus():
    import torch

    n = torch.cuda.device_count() if torch.cuda.is_available() else 0
    if n < 2:
        pytest.skip("needs >= 2 GPUs on one box")
    n = 8 if n >= 8 else (4 if n >= 4 else 2)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
                        "--master-addr", "127.0.0.1", "--master-port", "29617",
                        os.path.join(ROOT, "tests", "multigpu", "check_sharded_update_obs_norm.py")],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0 and "MULTIGPU OBS NORM OK" in r.stdout, (r.stdout[-3000:], r.stderr[-3000:])
