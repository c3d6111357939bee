"""act_dim 33 .. 64: wider than the fused step kernel's 32-wide heads, so training, the rollout policy step, the bootstrap
value and InferencePolicy run on the layer-wise kernels (head_loss_kernel<64>, policy_head_kernel<64>) whatever
learner.fused says.

* Update parity against the oracle, the same method and tolerances as test_update_parity (tests/test_gpu_update.py).
* The single-minibatch gradient per leaf, on the leaves the head kernel produces.
* That learner.fused = True does not enter the fused kernels at A > 32 (same launch count as learner.fused = False).
* Policy step (modes included), the rollout log-prob against the first epoch's recomputation, InferencePolicy, capture
  into a caller's CUDA graph and the refusal above 64.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import ppo_numpy as P
from oracle import synth, threefry
from tests.helpers import flat_grads, hyper_to_config, rel_err, run_gpu_update

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CASES = {
    # one past the fused kernel's limit, plausible humanoid observation width
    "a33_d415": dict(hp=dict(num_envs=64, num_steps=32, num_minibatches=4, update_epochs=2, anneal_lr=False), D=415, A=33),
    # entropy bonus, annealed learning rate
    "a48_d415_ent_anneal": dict(hp=dict(num_envs=64, num_steps=32, num_minibatches=4, update_epochs=2, anneal_lr=True,
                                        ent_coef=0.01), D=415, A=48),
    # the head kernel's shared-memory worst case: W3a staged in two 256-row chunks
    "a64_h512": dict(hp=dict(num_envs=64, num_steps=32, num_minibatches=4, update_epochs=2, anneal_lr=False,
                             hidden_size=512), D=225, A=64),
    # the first width where a fully resident W3a would overflow; a short second chunk (448 = 256 + 192)
    "a40_h448": dict(hp=dict(num_envs=64, num_steps=32, num_minibatches=4, update_epochs=2, anneal_lr=False,
                             hidden_size=448), D=225, A=40),
    # one hidden layer, relu actor, D below one k-block, ragged row counts
    "a64_l1_relu_ragged": dict(hp=dict(num_envs=24, num_steps=16, num_minibatches=3, update_epochs=2, anneal_lr=False,
                                       hidden_size=128, num_layers=1, use_tanh=False), D=37, A=64),
    # three hidden layers, partitionable PRNG
    "a40_l3_partitionable": dict(hp=dict(num_envs=32, num_steps=16, num_minibatches=2, update_epochs=2, anneal_lr=False,
                                         hidden_size=192, num_layers=3, prng_mode=threefry.PARTITIONABLE), D=256, A=40),
}


def _oracle(hp, pr, dtype, gemm, perms=None):
    p0 = P.tree_like(pr["params"], lambda x: x.astype(dtype))
    return P.update(p0, P.init_opt_state(p0), pr["traj"], pr["last_val"], pr["rng"], hp, dtype=dtype, gemm=gemm,
                    perms=perms)


def _leaf_rms_in_lr(got_flat, ref_tree, hp, D, A, lr):
    out, off = {}, 0
    ref = P.flatten_params(ref_tree, hp.num_layers, np.float64)
    for pth, shp in zip(P.leaf_order(hp.num_layers), P.leaf_shapes(D, A, hp.hidden_size, hp.num_layers)):
        n = int(np.prod(shp))
        d = got_flat[off:off + n].astype(np.float64) - ref[off:off + n]
        out["/".join(pth)] = float(np.sqrt(np.mean(d * d)) / lr)
        off += n
    return out


@pytest.mark.parametrize("name", list(CASES))
def test_wide_action_update_parity(name, cuda_device):
    case = CASES[name]
    hp = P.Hyper(**case["hp"])
    D, A = case["D"], case["A"]
    pr = synth.make_problem(hp, D, A, seed=7, done_p=0.02)
    got = run_gpu_update(hp, pr, cuda_device)
    p64, o64, rng64, l64, aux64 = _oracle(hp, pr, np.float64, "exact")
    pbf, obf, _, lbf, auxbf = _oracle(hp, pr, np.float32, "bf16", perms=aux64["perms"])

    assert np.array_equal(got["perms"], aux64["perms"])
    assert np.array_equal(got["rng"], rng64)
    assert got["step"] == hp.update_epochs * hp.num_minibatches == o64["count"]
    assert np.abs(got["advantages"] - aux64["advantages"]).max() <= 1e-5 * np.abs(aux64["advantages"]).max()
    assert np.abs(got["targets"] - aux64["targets"]).max() <= 1e-5 * np.abs(aux64["targets"]).max()

    lr = hp.opt_lr if not hp.anneal_lr else hp.training_lr
    flat64 = P.flatten_params(p64, hp.num_layers, np.float64)
    m = {
        "loss_vs_bf16_oracle": rel_err(got["losses"], lbf),
        "loss_vs_fp64_oracle": rel_err(got["losses"], l64),
        "gnorm_vs_bf16_oracle": rel_err(got["grad_norms"], auxbf["grad_norms"]),
        "param_absdiff_vs_fp64_oracle_in_lr": float(np.abs(got["params"] - flat64).max() / lr),
        "param_rms_vs_fp64_oracle_in_lr": float(np.sqrt(np.mean((got["params"] - flat64) ** 2)) / lr),
        "param_leaf_rms_vs_bf16_oracle_in_lr": _leaf_rms_in_lr(got["params"], pbf, hp, D, A, lr),
    }
    print(name, m)
    assert np.all(np.isfinite(got["losses"])) and np.all(np.isfinite(got["params"]))
    assert m["loss_vs_bf16_oracle"] < 2e-3, m
    assert m["loss_vs_fp64_oracle"] < 3e-2, m
    assert m["gnorm_vs_bf16_oracle"] < 2e-2, m
    nsteps = hp.update_epochs * hp.num_minibatches
    assert m["param_absdiff_vs_fp64_oracle_in_lr"] < 2.0 + 0.15 * nsteps, m
    assert m["param_rms_vs_fp64_oracle_in_lr"] < 1.0, m
    assert max(m["param_leaf_rms_vs_bf16_oracle_in_lr"].values()) < 1.0, m


@pytest.mark.parametrize("name", ["a48_d415_ent_anneal", "a64_h512"])
def test_wide_action_single_minibatch_gradient(name, cuda_device):
    """E = 1, M = 1 (as test_single_minibatch_gradient in tests/test_gpu_update.py): the gradient the optimizer saw, leaf
    by leaf against the oracle with the bf16 rounding points emulated.  The leaves the actor half of the head kernel
    produces (the actor's head kernel and bias, log_std, the actor's last hidden bias) are each held to 5e-3 of their own
    largest entry.  The critic half does the same arithmetic as at A <= 32; its leaves are held, with every other leaf,
    to 5e-3 of the largest gradient entry (at H = 512 the critic's small hidden-layer gradients reach ~1e-2 of their
    own largest entry through bf16 rounding flips of dZ, whatever act_dim is)."""
    case = CASES[name]
    kw = dict(case["hp"])
    kw.update(num_minibatches=1, update_epochs=1)
    hp = P.Hyper(**kw)
    D, A, L = case["D"], case["A"], hp.num_layers
    pr = synth.make_problem(hp, D, A, seed=9, done_p=0.02)
    g = np.random.default_rng(1)                              # ratio != 1: both clip branches
    pr["traj"]["log_prob"] = (pr["traj"]["log_prob"] + 0.3 * g.standard_normal(pr["traj"]["log_prob"].shape)).astype(np.float32)
    pr["traj"]["value"] = (pr["traj"]["value"] + 0.3 * g.standard_normal(pr["traj"]["value"].shape)).astype(np.float32)
    got = run_gpu_update(hp, pr, cuda_device)

    p0 = P.tree_like(pr["params"], lambda x: x.astype(np.float32))
    adv, tgt = P.gae(pr["traj"]["reward"], pr["traj"]["value"], pr["traj"]["done"], pr["last_val"], hp.gamma,
                     hp.gae_lambda, np.float32)
    flat = P.flatten_traj({"obs": pr["traj"]["obs"], "action": pr["traj"]["action"], "value": pr["traj"]["value"],
                           "log_prob": pr["traj"]["log_prob"], "adv": adv, "tgt": tgt})
    _, sub = threefry.split(pr["rng"], 2, hp.prng_mode)
    perm = threefry.permutation(sub, hp.batch_size, hp.prng_mode)
    lsbf, gr = P.loss_and_grads(p0, {k: v[perm] for k, v in flat.items()}, hp, "bf16")
    gbf = flat_grads(gr, L)
    ggpu = got["grad"][:gbf.size].astype(np.float64)
    leaf_err, off = {}, 0
    for pth, shp in zip(P.leaf_order(L), P.leaf_shapes(D, A, hp.hidden_size, L)):
        n = int(np.prod(shp))
        leaf_err["/".join(pth)] = rel_err(ggpu[off:off + n], gbf[off:off + n])
        off += n
    print(name, leaf_err)
    assert rel_err(ggpu, gbf) < 5e-3
    assert rel_err(got["losses"][0, 0], np.array(lsbf)) < 2e-3
    for leaf in (f"MLP_0/Dense_{L}/kernel", f"MLP_0/Dense_{L}/bias", "log_std", f"MLP_0/Dense_{L - 1}/bias"):
        assert leaf_err[leaf] < 5e-3, (leaf, leaf_err)


def test_fused_flag_does_not_enter_the_fused_kernels_above_32(cuda_device):
    hp = P.Hyper(num_envs=64, num_steps=32, num_minibatches=4, update_epochs=1, anneal_lr=False)
    pr = synth.make_problem(hp, 225, 33, seed=3)
    a = run_gpu_update(hp, pr, cuda_device, fused=True)
    b = run_gpu_update(hp, pr, cuda_device, fused=False)
    assert a["launches"] == b["launches"]
    for k in ("params", "losses"):
        assert np.array_equal(a[k], b[k]), k
    # against A = 32 on the fused path (fewer launches: one fused step kernel per minibatch step)
    c = run_gpu_update(hp, synth.make_problem(hp, 225, 32, seed=3), cuda_device, fused=True)
    assert c["launches"] < a["launches"]


# ---- rollout policy step / inference ----------------------------------------------------------------------------------
def _policy_setup(device, A, hidden=256, seed=11, **hpkw):
    import torch

    from minppo_b200.learner import Learner

    hp = P.Hyper(**{**dict(num_envs=300, num_steps=4, num_minibatches=2, update_epochs=1, anneal_lr=False,
                           hidden_size=hidden), **hpkw})
    D = 225
    pr = synth.make_problem(hp, D, A, seed=seed)
    pr["params"]["params"]["log_std"] = np.linspace(-0.7, 0.3, A).astype(np.float32)
    learner = Learner(hyper_to_config(hp), D, A, device)
    obs = np.random.default_rng(77).standard_normal((hp.num_envs, D)).astype(np.float32)
    flat = torch.as_tensor(P.flatten_params(pr["params"], hp.num_layers)).to(device)
    return hp, pr, learner, flat, torch.as_tensor(obs).to(device)


@pytest.mark.parametrize("A,H", [(48, 256), (64, 512)])
def test_wide_action_policy_step_vs_oracle(A, H, cuda_device):
    import torch

    hp, pr, learner, flat, dobs = _policy_setup(cuda_device, A, H)
    rng = torch.as_tensor(pr["rng"].view(np.int32)).to(cuda_device)
    action, log_prob, value, rng2, mean = learner.policy_step(flat, dobs, rng, want_mean=True)
    learner.check()
    action, log_prob, value, mean = (x.cpu().numpy() for x in (action, log_prob, value, mean))
    p32 = P.tree_like(pr["params"], lambda x: x.astype(np.float32))
    a_o, lp_o, v_o, rng_o, m_o = P.policy_step(p32, dobs.cpu().numpy(), pr["rng"], hp, hp.prng_mode, gemm="bf16")
    assert action.shape == (hp.num_envs, A)
    assert np.array_equal(rng2.cpu().numpy().view(np.uint32), rng_o)
    for got, ref, name in ((mean, m_o, "mean"), (value, v_o, "value")):
        scale = np.abs(ref).max()
        d = np.abs(got - ref)
        assert d.max() <= 5e-3 * scale and d.mean() <= 2e-4 * scale, (name, d.max(), d.mean(), scale)
    ls = pr["params"]["params"]["log_std"].astype(np.float64)
    _, akey = threefry.split(pr["rng"], 2, hp.prng_mode)
    eps_o = threefry.normal_f32(akey, action.size, hp.prng_mode, erfinv="xla").reshape(action.shape)
    eps = (action.astype(np.float64) - mean.astype(np.float64)) / np.exp(ls)
    assert np.all(np.abs(eps - eps_o) <= 2e-6 * np.maximum(1.0, np.abs(eps_o))), np.abs(eps - eps_o).max()
    z = (action.astype(np.float64) - mean) / np.exp(ls)
    lp64 = (-0.5 * z * z - 0.5 * np.log(2 * np.pi)).sum(-1) - ls.sum()
    assert np.abs(log_prob - lp64).max() <= 1e-4
    assert np.abs(log_prob - lp_o).max() <= 1e-4
    learner.close()


def test_wide_action_policy_step_modes(cuda_device):
    """No sampling (action = mode), critic-only bootstrap value, and the weights-current fast path, at A = 64."""
    import torch

    hp, pr, learner, flat, dobs = _policy_setup(cuda_device, 64)
    rng = torch.as_tensor(pr["rng"].view(np.int32)).to(cuda_device)
    a1, lp1, v1, r1, m1 = learner.policy_step(flat, dobs, rng, want_mean=True)
    a2, lp2, v2, r2, m2 = learner.policy_step(flat, dobs, rng, weights_current=True, want_mean=True)
    for x, y in ((a1, a2), (lp1, lp2), (v1, v2), (r1, r2), (m1, m2)):
        assert torch.equal(x, y)
    a0, lp0, v0, r0, m0 = learner.policy_step(flat, dobs, None, want_mean=True)
    assert r0 is None and torch.equal(a0, m0) and torch.equal(m0, m1) and torch.equal(v0, v1)
    ls = pr["params"]["params"]["log_std"].astype(np.float64)
    assert np.allclose(lp0.cpu().numpy(), -0.5 * 64 * np.log(2 * np.pi) - ls.sum(), atol=1e-4)
    assert torch.equal(learner.bootstrap_value(flat, dobs), v1)
    learner.check()
    learner.close()


def test_wide_action_rollout_log_prob_matches_first_epoch(cuda_device):
    """As test_rollout_log_prob_matches_first_epoch (tests/test_gpu_policy.py) at A = 64: the learner's first minibatch
    sees ratio == 1 and v == v_old, so actor_loss ~ 0 and value_loss = 0.5 * mean((v_old - tgt)^2)."""
    import torch

    from minppo_b200.learner import Learner, Memory, TrainState

    hp = P.Hyper(num_envs=256, num_steps=8, num_minibatches=1, update_epochs=1, anneal_lr=False)
    D, A = 225, 64
    pr = synth.make_problem(hp, D, A, seed=4)
    learner = Learner(hyper_to_config(hp), D, A, cuda_device)
    ts = TrainState.create(P.flatten_params(pr["params"], hp.num_layers), cuda_device)
    obs = torch.as_tensor(pr["traj"]["obs"]).to(cuda_device)
    rng = torch.as_tensor(pr["rng"].view(np.int32)).to(cuda_device)
    acts, lps, vals = [], [], []
    for t in range(hp.num_steps):
        a, lp, v, rng, _ = learner.policy_step(ts.params, obs[t].contiguous(), rng, weights_current=t > 0)
        acts.append(a); lps.append(lp); vals.append(v)
    mem = Memory(done=torch.as_tensor(pr["traj"]["done"]).to(cuda_device), action=torch.stack(acts),
                 value=torch.stack(vals), reward=torch.as_tensor(pr["traj"]["reward"]).to(cuda_device),
                 log_prob=torch.stack(lps), obs=obs)
    last_val = learner.bootstrap_value(ts.params, obs[-1].contiguous(), weights_current=True)
    ts, _, losses = learner.update(ts, mem, last_val, rng)
    learner.check()
    total, value_loss, actor_loss, _ = losses.cpu().numpy()[0, 0]
    tgt = learner.read("targets").cpu().numpy()
    v_old = torch.stack(vals).cpu().numpy()
    assert abs(actor_loss) < 1e-5
    assert abs(value_loss - 0.5 * np.mean((v_old - tgt) ** 2)) <= 1e-5 * max(1.0, value_loss)
    learner.close()


def test_inference_policy_act_64(cuda_device, tmp_path):
    import torch

    from minppo_b200.infer import InferencePolicy
    from minppo_b200.params import save_model

    hp, pr, learner, flat, dobs = _policy_setup(cuda_device, 64, 512)
    ref_a, _, ref_v, _, _ = learner.policy_step(flat, dobs, None)
    path = str(tmp_path / "trained_model.pkl")
    save_model(P.tree_like(pr["params"], lambda x: x.astype(np.float32)), path)
    pol = InferencePolicy.from_checkpoint(path, hyper_to_config(hp), hp.num_envs, cuda_device)
    assert (pol.obs_dim, pol.act_dim) == (225, 64)
    for _ in range(2):                                         # second call: weights-current fast path
        a, v = pol.act(dobs)
        assert torch.equal(a, ref_a) and torch.equal(v, ref_v)
    rng = torch.as_tensor(pr["rng"].view(np.int32)).to(cuda_device)
    sa, slp, sv, rng2 = pol.act(dobs, rng)
    ra, rlp, rv, rrng, _ = learner.policy_step(flat, dobs, rng)
    assert torch.equal(sa, ra) and torch.equal(slp, rlp) and torch.equal(rng2, rrng)
    pol.close()
    learner.close()


# ---- capture into a caller's CUDA graph (use_graph = 0: the XLA-FFI mode) ---------------------------------------------
def test_a64_update_and_policy_step_replay_from_a_callers_capture(cuda_device):
    import torch

    from minppo_b200.learner import Learner, Memory, TrainState

    hp = P.Hyper(num_envs=64, num_steps=32, num_minibatches=4, update_epochs=2, anneal_lr=True)
    D, A = 225, 64
    pr = synth.make_problem(hp, D, A, seed=5, done_p=0.02)
    cfg = hyper_to_config(hp, use_graph=False)
    obs = torch.as_tensor(np.random.default_rng(0).standard_normal((hp.num_envs, D)).astype(np.float32)).to(cuda_device)
    t = lambda x: torch.as_tensor(np.ascontiguousarray(x)).to(cuda_device)
    tr = pr["traj"]
    mem = Memory(done=t(tr["done"]), action=t(tr["action"]), value=t(tr["value"]), reward=t(tr["reward"]),
                 log_prob=t(tr["log_prob"]), obs=t(tr["obs"]))
    lv = t(pr["last_val"])
    rng = torch.as_tensor(pr["rng"].view(np.int32)).to(cuda_device)

    def fresh():
        return TrainState.create(P.flatten_params(pr["params"], hp.num_layers), cuda_device)

    lrn = Learner(cfg, D, A, cuda_device)
    ts = fresh()
    losses = torch.empty((hp.update_epochs, hp.num_minibatches, 4), device=cuda_device)
    rng_out = torch.empty_like(rng)
    lrn.update(ts, mem, lv, rng, losses, rng_out)
    act, logp, val, rng2, _ = lrn.policy_step(ts.params, obs, rng_out)
    lrn.check()
    want = [x.clone() for x in (ts.params, ts.mu, ts.nu, ts.step, losses, rng_out, act, logp, val, rng2)]
    lrn.close()

    lrn = Learner(cfg, D, A, cuda_device)
    ts = fresh()
    p0, m0, n0, s0 = ts.params.clone(), ts.mu.clone(), ts.nu.clone(), ts.step.clone()
    losses = torch.zeros((hp.update_epochs, hp.num_minibatches, 4), device=cuda_device)
    rng_out = torch.zeros_like(rng)
    side = torch.cuda.Stream(device=cuda_device)
    side.wait_stream(torch.cuda.current_stream(cuda_device))
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            lrn.update(ts, mem, lv, rng, losses, rng_out)
            act, logp, val, rng2, _ = lrn.policy_step(ts.params, obs, rng_out)
    torch.cuda.current_stream(cuda_device).wait_stream(side)
    torch.cuda.synchronize(cuda_device)
    assert torch.equal(ts.params, p0) and int(ts.step.item()) == 0
    for rep in range(2):
        ts.params.copy_(p0); ts.mu.copy_(m0); ts.nu.copy_(n0); ts.step.copy_(s0)
        graph.replay()
        torch.cuda.synchronize(cuda_device)
        lrn.check()
        got = (ts.params, ts.mu, ts.nu, ts.step, losses, rng_out, act, logp, val, rng2)
        for i, (g, w) in enumerate(zip(got, want)):
            assert torch.equal(g, w), (rep, i)
    lrn.close()


@pytest.mark.parametrize("A", [65, 128])
def test_wide_action_refusal(A, cuda_device):
    from minppo_b200 import _lib
    from minppo_b200.learner import Learner

    with pytest.raises(_lib.MinppoError) as e:
        Learner(hyper_to_config(P.Hyper(num_envs=16, num_steps=4, num_minibatches=4)), 8, A, cuda_device)
    assert e.value.code == _lib.ERR_UNSUPPORTED and "<= 64" in str(e.value)


def test_sharded_wide_action_update_parity_all_visible_gpus():
    import torch

    n = torch.cuda.device_count() if torch.cuda.is_available() else 0
    if n < 2:
        pytest.skip("needs >= 2 GPUs on one box")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29614",
                        os.path.join(ROOT, "tests", "multigpu", "check_sharded_update_wide_action.py")],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0 and "MULTIGPU PARITY OK" in r.stdout, (r.stdout[-2000:], r.stderr[-2000:])
