"""model.hidden_size above one 256-column GEMM tile (320 .. 512): every hidden layer runs on the layer-wise tcgen05 GEMMs
as two column groups of one launch (fused step kernel: H <= 256 only).

* Update parity against the oracle, the same method and tolerances as test_update_parity (tests/test_gpu_update.py).
* Zero-padding embedding, independent of the oracle: a 256-wide net widened to 512 by hidden units whose incoming and
  outgoing weights and biases are all zero.  Those units compute exact zeros (tanh(0) = relu(0) = 0) and get exactly
  zero gradient, so Adam leaves them at 0; every product they add to a real unit's fp32 accumulator is +0.  The first
  minibatch's losses (forward only) are therefore bit-identical to the 256-wide layer-wise run; later steps differ only
  through the summation order of the global gradient norm (more, all-zero, elements spread over the optimizer threads).
* Policy step, InferencePolicy, capture into a caller's CUDA graph and the refusals at 512 wide.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import ppo_numpy as P
from oracle import synth
from tests.helpers import hyper_to_config, rel_err, run_gpu_update

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CASES = {
    "h512": dict(hp=dict(num_envs=64, num_steps=32, num_minibatches=4, update_epochs=2, anneal_lr=False,
                         hidden_size=512), D=225, A=10),
    "h512_l1_relu_ragged": dict(hp=dict(num_envs=24, num_steps=16, num_minibatches=3, update_epochs=2, anneal_lr=False,
                                        hidden_size=512, num_layers=1, use_tanh=False), D=37, A=3),
    # 192 + 128 column groups, 32-wide head template, D > 256
    "h320_d415_a32": dict(hp=dict(num_envs=64, num_steps=32, num_minibatches=4, update_epochs=2, anneal_lr=False,
                                  hidden_size=320), D=415, A=32),
    # 256 + 192 column groups, entropy bonus, annealed learning rate
    "h448_ent_anneal": dict(hp=dict(num_envs=64, num_steps=32, num_minibatches=4, update_epochs=2, anneal_lr=True,
                                    hidden_size=448, ent_coef=0.01), D=225, A=10),
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
def test_wide_update_parity(name, cuda_device):
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


# ---- zero-padding embedding of a 256-wide net into a 512-wide one ---------------------------------------------------
def _pad_tree(tree, num_layers, H):
    """Copy of a parameter tree with every hidden layer zero-padded to H units."""
    out = P.tree_like(tree, lambda x: x)
    for mlp in ("MLP_0", "MLP_1"):
        for i in range(num_layers + 1):
            d = tree["params"][mlp][f"Dense_{i}"]
            k, b = np.asarray(d["kernel"]), np.asarray(d["bias"])
            rows = k.shape[0] if i == 0 else H
            cols = H if i < num_layers else k.shape[1]
            kp = np.zeros((rows, cols), k.dtype)
            kp[:k.shape[0], :k.shape[1]] = k
            bp = np.zeros((cols,), b.dtype)
            bp[:b.shape[0]] = b
            out["params"][mlp][f"Dense_{i}"] = {"kernel": kp, "bias": bp}
    return out


def _pad_mask(D, A, H0, H, L):
    """Flat mask of the 512-wide arena: True at the padding entries."""
    n = sum(int(np.prod(s)) for s in P.leaf_shapes(D, A, H0, L))
    ones = P.unflatten_params(np.ones(n, np.float32), D, A, H0, L)
    return P.flatten_params(_pad_tree(ones, L, H), L) == 0


@pytest.mark.parametrize("use_tanh", [True, False])
def test_zero_padded_512_equals_256_layerwise(use_tanh, cuda_device):
    kw = dict(num_envs=64, num_steps=32, num_minibatches=4, update_epochs=1, anneal_lr=False, use_tanh=use_tanh)
    hp256, hp512 = P.Hyper(hidden_size=256, **kw), P.Hyper(hidden_size=512, **kw)
    D, A, L = 225, 10, 2
    pr = synth.make_problem(hp256, D, A, seed=5, done_p=0.02)
    pr512 = dict(pr)
    pr512["params"] = _pad_tree(pr["params"], L, 512)
    a = run_gpu_update(hp256, pr, cuda_device, fused=False, dw_splits=4)
    b = run_gpu_update(hp512, pr512, cuda_device, dw_splits=4)
    pad = _pad_mask(D, A, 256, 512, L)
    assert pad.sum() == P.flatten_params(pr512["params"], L).size - a["params"].size
    assert np.all(b["params"][pad] == 0.0) and np.all(b["mu"][pad] == 0.0) and np.all(b["nu"][pad] == 0.0)
    assert np.array_equal(b["losses"][0, 0], a["losses"][0, 0])
    assert rel_err(b["losses"], a["losses"]) < 2e-4
    lr = hp256.opt_lr
    nsteps = hp256.update_epochs * hp256.num_minibatches
    assert np.abs(b["params"][~pad] - a["params"]).max() < lr * (2.0 + 0.15 * nsteps)
    assert np.array_equal(b["perms"], a["perms"]) and np.array_equal(b["rng"], a["rng"])


# ---- rollout policy step / inference ----------------------------------------------------------------------------------
def _policy_setup(device, hidden=512, fused=True, seed=11):
    import torch

    from minppo_b200.learner import Learner

    hp = P.Hyper(num_envs=300, num_steps=4, num_minibatches=2, update_epochs=1, anneal_lr=False, hidden_size=hidden)
    D, A = 225, 10
    pr = synth.make_problem(hp, D, A, seed=seed)
    pr["params"]["params"]["log_std"] = np.linspace(-0.7, 0.3, A).astype(np.float32)
    learner = Learner(hyper_to_config(hp, fused=fused), D, A, device)
    obs = np.random.default_rng(77).standard_normal((hp.num_envs, D)).astype(np.float32)
    return hp, pr, learner, torch.as_tensor(obs).to(device)


def test_policy_step_h512_vs_oracle(cuda_device):
    import torch

    from oracle import threefry

    hp, pr, learner, dobs = _policy_setup(cuda_device)
    flat = torch.as_tensor(P.flatten_params(pr["params"], hp.num_layers)).to(cuda_device)
    rng = torch.as_tensor(pr["rng"].view(np.int32)).to(cuda_device)
    action, log_prob, value, rng2, mean = learner.policy_step(flat, dobs, rng, want_mean=True)
    vb = learner.bootstrap_value(flat, dobs)
    learner.check()
    assert torch.equal(vb, value)
    action, log_prob, value, mean = (x.cpu().numpy() for x in (action, log_prob, value, mean))
    p32 = P.tree_like(pr["params"], lambda x: x.astype(np.float32))
    a_o, lp_o, v_o, rng_o, m_o = P.policy_step(p32, dobs.cpu().numpy(), pr["rng"], hp, hp.prng_mode, gemm="bf16")
    assert np.array_equal(rng2.cpu().numpy().view(np.uint32), rng_o)
    for got, ref, name in ((mean, m_o, "mean"), (value, v_o, "value")):
        scale = np.abs(ref).max()
        d = np.abs(got - ref)
        assert d.max() <= 5e-3 * scale and d.mean() <= 2e-4 * scale, (name, d.max(), d.mean(), scale)
    ls = pr["params"]["params"]["log_std"].astype(np.float64)
    _, akey = threefry.split(pr["rng"], 2, hp.prng_mode)
    eps_o = threefry.normal_f32(akey, action.size, hp.prng_mode, erfinv="xla").reshape(action.shape)
    eps = (action.astype(np.float64) - mean.astype(np.float64)) / np.exp(ls)
    assert np.all(np.abs(eps - eps_o) <= 2e-6 * np.maximum(1.0, np.abs(eps_o)))
    assert np.abs(log_prob - lp_o).max() <= 1e-4
    learner.close()


def test_policy_step_zero_padded_512_equals_256_layerwise(cuda_device):
    import torch

    hp, pr, small, dobs = _policy_setup(cuda_device, hidden=256, fused=False)
    _, _, wide, _ = _policy_setup(cuda_device, hidden=512)
    L = hp.num_layers
    f256 = torch.as_tensor(P.flatten_params(pr["params"], L)).to(cuda_device)
    f512 = torch.as_tensor(P.flatten_params(_pad_tree(pr["params"], L, 512), L)).to(cuda_device)
    rng = torch.as_tensor(pr["rng"].view(np.int32)).to(cuda_device)
    a = small.policy_step(f256, dobs, rng, want_mean=True)
    b = wide.policy_step(f512, dobs, rng, want_mean=True)
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    assert torch.equal(small.bootstrap_value(f256, dobs), wide.bootstrap_value(f512, dobs))
    small.close()
    wide.close()


def test_inference_policy_h512(cuda_device, tmp_path):
    import torch

    from minppo_b200.infer import InferencePolicy
    from minppo_b200.params import save_model

    hp, pr, learner, dobs = _policy_setup(cuda_device)
    flat = torch.as_tensor(P.flatten_params(pr["params"], hp.num_layers)).to(cuda_device)
    ref_a, _, ref_v, _, _ = learner.policy_step(flat, dobs, None)
    path = str(tmp_path / "trained_model.pkl")
    save_model(P.tree_like(pr["params"], lambda x: x.astype(np.float32)), path)
    pol = InferencePolicy.from_checkpoint(path, hyper_to_config(hp), hp.num_envs, cuda_device)
    for _ in range(2):                                         # second call: weights-current fast path
        a, v = pol.act(dobs)
        assert torch.equal(a, ref_a) and torch.equal(v, ref_v)
    pol.close()
    learner.close()


# ---- capture into a caller's CUDA graph (use_graph = 0: the XLA-FFI mode) ---------------------------------------------
def test_h512_update_and_policy_step_replay_from_a_callers_capture(cuda_device):
    import torch

    from minppo_b200.learner import Learner, Memory, TrainState

    hp = P.Hyper(num_envs=64, num_steps=32, num_minibatches=4, update_epochs=2, anneal_lr=True, hidden_size=512)
    pr = synth.make_problem(hp, 225, 10, seed=5, done_p=0.02)
    cfg = hyper_to_config(hp, use_graph=False)
    obs = torch.as_tensor(np.random.default_rng(0).standard_normal((hp.num_envs, 225)).astype(np.float32)).to(cuda_device)
    t = lambda x: torch.as_tensor(np.ascontiguousarray(x)).to(cuda_device)
    tr = pr["traj"]
    mem = Memory(done=t(tr["done"]), action=t(tr["action"]), value=t(tr["value"]), reward=t(tr["reward"]),
                 log_prob=t(tr["log_prob"]), obs=t(tr["obs"]))
    lv = t(pr["last_val"])
    rng = torch.as_tensor(pr["rng"].view(np.int32)).to(cuda_device)

    def fresh():
        return TrainState.create(P.flatten_params(pr["params"], hp.num_layers), cuda_device)

    lrn = Learner(cfg, 225, 10, cuda_device)
    ts = fresh()
    losses = torch.empty((hp.update_epochs, hp.num_minibatches, 4), device=cuda_device)
    rng_out = torch.empty_like(rng)
    lrn.update(ts, mem, lv, rng, losses, rng_out)
    act, logp, val, rng2, _ = lrn.policy_step(ts.params, obs, rng_out)
    lrn.check()
    want = [x.clone() for x in (ts.params, ts.mu, ts.nu, ts.step, losses, rng_out, act, logp, val, rng2)]
    lrn.close()

    lrn = Learner(cfg, 225, 10, cuda_device)
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


@pytest.mark.parametrize("H,L,limit", [(576, 2, "<= 512"), (384, 3, "num_layers <= 2")])
def test_wide_hidden_refusals(H, L, limit, cuda_device):
    from minppo_b200 import _lib
    from minppo_b200.learner import Learner

    with pytest.raises(_lib.MinppoError) as e:
        Learner(hyper_to_config(P.Hyper(num_envs=16, num_steps=4, num_minibatches=4, hidden_size=H, num_layers=L)), 8, 2,
                cuda_device)
    assert e.value.code == _lib.ERR_UNSUPPORTED and limit in str(e.value)


def test_sharded_wide_update_parity_all_visible_gpus():
    import torch

    n = torch.cuda.device_count() if torch.cuda.is_available() else 0
    if n < 2:
        pytest.skip("needs >= 2 GPUs on one box")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29613",
                        os.path.join(ROOT, "tests", "multigpu", "check_sharded_update_wide.py")],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0 and "MULTIGPU PARITY OK" in r.stdout, (r.stdout[-2000:], r.stderr[-2000:])
