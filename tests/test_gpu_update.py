"""One full learner update through the C ABI against the oracle (train.py:181-281).

GEMM precision of the CUDA path (declared): BF16 operands on tcgen05 tensor cores, FP32
accumulation; hidden activations and dZ stored as BF16; heads, loss, reductions, clip and Adam
in FP32.  Two comparisons per case:

* vs the oracle with the SAME rounding points emulated (gemm="bf16", float32): isolates
  algorithmic agreement from precision.  Tolerances: losses 2e-3 * max|loss|, gradient
  5e-3 * max|g| -- what remains is fp32 summation order and one-bf16-ulp rounding flips.
* vs the float64 oracle: shows the precision cost.  Tolerances: losses 3e-2 * max|loss|;
  parameters after n Adam steps: max |dp| <= lr * (2 + 0.15 n) and rms(dp) <= lr.  Adam's
  normalised step is ~lr per step and sign-sensitive where a gradient is near zero, so drift is
  measured in units of lr and allowed to grow with the step count (config 1 takes 128 steps on
  5-row minibatches; measured 16.4 lr max, 0.68 lr rms).
Bit-exact items: permutations, rng key, Adam step count.
"""
import json
import os

import numpy as np
import pytest

from oracle import ppo_numpy as P
from oracle import synth, threefry
from tests.helpers import (LEAF_BOUND_BF16, LEAF_BOUND_FP64, flat_grads, fp64_leaf_bounds, leaf_slices, leaves_over,
                           rel_err, run_gpu_update)

pytestmark = pytest.mark.gpu

METRICS = {}


@pytest.fixture(scope="module", autouse=True)
def _dump_metrics():
    yield
    out = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    try:
        os.makedirs(out, exist_ok=True)
        with open(os.path.join(out, "parity_metrics.json"), "w") as f:
            json.dump(METRICS, f, indent=1, sort_keys=True)
    except OSError:
        pass


CASES = {
    # config 1 of BASELINE.json: N=16, T=10 -> B=160, M=32 -> mb=5, E=4 (plumbing / parity shape)
    "c1": dict(hp=dict(num_envs=16, num_steps=10, num_minibatches=32, update_epochs=4, anneal_lr=False), D=225, A=10),
    # medium: several 128-row tiles per minibatch, annealed LR with the default 1e9 timesteps
    "medium": dict(hp=dict(num_envs=64, num_steps=32, num_minibatches=4, update_epochs=2, anneal_lr=True), D=225, A=10),
    # ragged shapes: D not a multiple of 64 below one k-block, small A, narrower net, 1 hidden layer
    "ragged": dict(hp=dict(num_envs=24, num_steps=16, num_minibatches=3, update_epochs=2, anneal_lr=False,
                           hidden_size=128, num_layers=1, ent_coef=0.01), D=37, A=3),
    # 3 hidden layers, relu actor (model.use_tanh=false), aligned D, partitionable PRNG
    "deep": dict(hp=dict(num_envs=32, num_steps=16, num_minibatches=2, update_epochs=2, anneal_lr=False,
                         hidden_size=192, num_layers=3, use_tanh=False, prng_mode=threefry.PARTITIONABLE), D=256, A=16),
    # ---- shape-genericity of the FUSED step kernel (num_layers = 2; SURVEY F9: D, A come from the MJCF at run time) ----
    # a plausible real humanoid (env.py:245-261 with ~20 actuators): D > 256 streams X k-blocks through the 4 slots,
    # A > 16 takes the 32-wide head template, P > 303k takes two register-resident units per optimizer thread
    "wide": dict(hp=dict(num_envs=64, num_steps=32, num_minibatches=4, update_epochs=2, anneal_lr=False), D=415, A=20),
    # A at the limit, 3 k-blocks of H, D one element past a k-block boundary
    "a32_h192": dict(hp=dict(num_envs=48, num_steps=16, num_minibatches=2, update_epochs=2, anneal_lr=False,
                             hidden_size=192), D=321, A=32),
    # odd A just past the 16-wide template, narrow net, 10 k-blocks of D (slots refilled 6 times)
    "a17_h128_d600": dict(hp=dict(num_envs=32, num_steps=16, num_minibatches=2, update_epochs=2, anneal_lr=False,
                                  hidden_size=128, use_tanh=False), D=600, A=17),
    # one k-block of H, A = 24
    "a24_h64": dict(hp=dict(num_envs=32, num_steps=8, num_minibatches=2, update_epochs=2, anneal_lr=False,
                            hidden_size=64, ent_coef=0.01), D=100, A=24),
    # 16 k-blocks of D, P = 646k: four register-resident units per optimizer thread
    "d1000": dict(hp=dict(num_envs=32, num_steps=16, num_minibatches=2, update_epochs=1, anneal_lr=False), D=1000, A=10),
    # the same with 4 dW splits: 4 x 40 GEMM CTAs do not fit one CTA per SM (148), so every step takes the two-launch
    # sequence (stand-alone dW GEMM, then dwopt without GEMM CTAs) instead of the merged dwopt launch
    "d1000_two_launch": dict(hp=dict(num_envs=32, num_steps=16, num_minibatches=2, update_epochs=1, anneal_lr=False),
                             D=1000, A=10, cfg=dict(dw_splits=4)),
}
FUSED_SHAPE_CASES = ["wide", "a32_h192", "a17_h128_d600", "a24_h64", "d1000"]


def _oracle(hp, pr, dtype, gemm, perms=None):
    p0 = P.tree_like(pr["params"], lambda x: x.astype(dtype))
    return P.update(p0, P.init_opt_state(p0), pr["traj"], pr["last_val"], pr["rng"], hp, dtype=dtype, gemm=gemm,
                    perms=perms)


@pytest.mark.parametrize("name", list(CASES))
def test_update_parity(name, cuda_device):
    case = CASES[name]
    hp = P.Hyper(**case["hp"])
    pr = synth.make_problem(hp, case["D"], case["A"], seed=7, done_p=0.02)
    got = run_gpu_update(hp, pr, cuda_device, **case.get("cfg", {}))

    p64, o64, rng64, l64, aux64 = _oracle(hp, pr, np.float64, "exact")
    pbf, obf, _, lbf, auxbf = _oracle(hp, pr, np.float32, "bf16", perms=aux64["perms"])

    # bit-exact: permutations, key chain, step count
    assert np.array_equal(got["perms"], aux64["perms"])
    assert np.array_equal(got["rng"], rng64)
    assert got["step"] == hp.update_epochs * hp.num_minibatches == o64["count"]
    # GAE: 1e-5 relative (north_star)
    assert np.abs(got["advantages"] - aux64["advantages"]).max() <= 1e-5 * np.abs(aux64["advantages"]).max()
    assert np.abs(got["targets"] - aux64["targets"]).max() <= 1e-5 * np.abs(aux64["targets"]).max()

    lr = hp.opt_lr if not hp.anneal_lr else hp.training_lr
    flat64 = P.flatten_params(p64, hp.num_layers, np.float64)
    flatbf = P.flatten_params(pbf, hp.num_layers, np.float64)
    m = {
        "loss_vs_bf16_oracle": rel_err(got["losses"], lbf),
        "loss_vs_fp64_oracle": rel_err(got["losses"], l64),
        "gnorm_vs_bf16_oracle": rel_err(got["grad_norms"], auxbf["grad_norms"]),
        "gnorm_vs_fp64_oracle": rel_err(got["grad_norms"], aux64["grad_norms"]),
        "param_absdiff_vs_bf16_oracle_in_lr": float(np.abs(got["params"] - flatbf).max() / lr),
        "param_absdiff_vs_fp64_oracle_in_lr": float(np.abs(got["params"] - flat64).max() / lr),
        "param_rms_vs_fp64_oracle_in_lr": float(np.sqrt(np.mean((got["params"] - flat64) ** 2)) / lr),
        "first_loss_gpu": [float(x) for x in got["losses"][0, 0]],
        "first_loss_fp64": [float(x) for x in l64[0, 0]],
        "launches": got["launches"],
        "param_leaf_rms_vs_bf16_oracle_in_lr": _per_leaf_rms_in_lr(got["params"], pbf, hp, case["D"], case["A"], lr),
    }
    METRICS[name] = m
    assert np.all(np.isfinite(got["losses"])) and np.all(np.isfinite(got["params"]))
    assert m["loss_vs_bf16_oracle"] < 2e-3, m
    assert m["loss_vs_fp64_oracle"] < 3e-2, m
    assert m["gnorm_vs_bf16_oracle"] < 2e-2, m
    nsteps = hp.update_epochs * hp.num_minibatches
    assert m["param_absdiff_vs_fp64_oracle_in_lr"] < 2.0 + 0.15 * nsteps, m
    assert m["param_rms_vs_fp64_oracle_in_lr"] < 1.0, m
    # per leaf (a wrong small leaf would vanish in the global figures): rms <= 1 lr against the emulated oracle
    assert max(m["param_leaf_rms_vs_bf16_oracle_in_lr"].values()) < 1.0, m


# ---- the benchmarked shapes (BASELINE.json configs[1] and configs[3]) -----------------------------------
BENCH_CASES = {
    # configs[1]: what bench.py times at N = 1 (mb = 8192: 64 row tiles per net, split-K over 128 k-blocks)
    "configs1": dict(hp=dict(num_envs=2048, num_steps=128, num_minibatches=32, update_epochs=4, anneal_lr=True), D=225, A=10),
    # configs[3] on ONE GPU (mb = 32768: 256 row tiles per net = several waves of the fused step kernel)
    "configs3": dict(hp=dict(num_envs=16384, num_steps=64, num_minibatches=32, update_epochs=4, anneal_lr=True), D=225, A=10),
}


def _per_leaf_rms_in_lr(got_flat, ref_tree, hp, D, A, lr):
    out, off = {}, 0
    ref = P.flatten_params(ref_tree, hp.num_layers, np.float64)
    for pth, shp in zip(P.leaf_order(hp.num_layers), P.leaf_shapes(D, A, hp.hidden_size, hp.num_layers)):
        n = int(np.prod(shp))
        d = got_flat[off:off + n].astype(np.float64) - ref[off:off + n]
        out["/".join(pth)] = float(np.sqrt(np.mean(d * d)) / lr)
        off += n
    assert off == ref.size
    return out


@pytest.mark.parametrize("name", list(BENCH_CASES))
def test_update_parity_at_bench_shape(name, cuda_device):
    """ONE full update (E x M = 128 sequential minibatch steps) at the shapes bench.py reports, against the
    oracle run with the same bf16 rounding points (float32, gemm="bf16").  Tolerances: permutations / rng / step
    count bit-exact; advantages and targets 1e-5 relative; every one of the 128 losses 2e-3 of the largest loss;
    every gradient norm 2e-2; parameters PER LEAF rms <= 1 lr (Adam moves a parameter ~lr per step, 128 steps)."""
    case = BENCH_CASES[name]
    hp = P.Hyper(**case["hp"])
    D, A = case["D"], case["A"]
    pr = synth.make_problem(hp, D, A, seed=11, done_p=0.01)
    got = run_gpu_update(hp, pr, cuda_device)
    pbf, obf, rngbf, lbf, auxbf = _oracle(hp, pr, np.float32, "bf16")

    assert np.array_equal(got["perms"], auxbf["perms"])
    assert np.array_equal(got["rng"], rngbf)
    assert got["step"] == hp.update_epochs * hp.num_minibatches == obf["count"]
    assert np.abs(got["advantages"] - auxbf["advantages"]).max() <= 1e-5 * np.abs(auxbf["advantages"]).max()
    assert np.abs(got["targets"] - auxbf["targets"]).max() <= 1e-5 * np.abs(auxbf["targets"]).max()
    lr = hp.training_lr
    leaf_rms = _per_leaf_rms_in_lr(got["params"], pbf, hp, D, A, lr)
    m = {
        "loss_vs_bf16_oracle": rel_err(got["losses"], lbf),
        "loss_vs_bf16_oracle_per_column": [rel_err(got["losses"][..., j], lbf[..., j]) for j in (0, 1, 3)],
        "gnorm_vs_bf16_oracle": float(np.abs(got["grad_norms"] - auxbf["grad_norms"]).max() / np.abs(auxbf["grad_norms"]).max()),
        "param_leaf_rms_in_lr": leaf_rms,
        "param_absdiff_vs_bf16_oracle_in_lr": float(np.abs(got["params"] - P.flatten_params(pbf, hp.num_layers, np.float64)).max() / lr),
        "last_loss_gpu": [float(x) for x in got["losses"][-1, -1]],
        "last_loss_oracle": [float(x) for x in lbf[-1, -1]],
        "launches": got["launches"],
    }
    METRICS["bench_shape_" + name] = m
    assert np.all(np.isfinite(got["losses"])) and np.all(np.isfinite(got["params"]))
    assert m["loss_vs_bf16_oracle"] < 2e-3, m
    assert m["gnorm_vs_bf16_oracle"] < 2e-2, m
    assert max(leaf_rms.values()) < 1.0, m


def test_update_parity_negative_lr_schedule(cuda_device):
    """SURVEY F8 on the GPU: with training.total_timesteps = num_steps * num_envs (one update) the reference's
    schedule (train.py:98-101) divides the step count by minibatch_size * update_epochs = 20, so over the 128
    steps of config 1 frac = 1, 0, -1, ..., -5: the learning rate hits zero at step 20 and is NEGATIVE after."""
    hp = P.Hyper(num_envs=16, num_steps=10, num_minibatches=32, update_epochs=4, anneal_lr=True, total_timesteps=160)
    assert hp.num_updates == 1 and hp.minibatch_size * hp.update_epochs == 20
    lrs = [float(P.learning_rate(k, hp, np.float32)) for k in range(128)]
    assert lrs[0] == np.float32(hp.training_lr) and lrs[20] == 0.0 and lrs[40] < 0 and lrs[127] == np.float32(hp.training_lr) * -5
    pr = synth.make_problem(hp, 225, 10, seed=7, done_p=0.02)
    got = run_gpu_update(hp, pr, cuda_device)
    p64, o64, rng64, l64, aux64 = _oracle(hp, pr, np.float64, "exact")
    pbf, obf, _, lbf, auxbf = _oracle(hp, pr, np.float32, "bf16", perms=aux64["perms"])
    assert np.array_equal(got["perms"], aux64["perms"])
    assert got["step"] == 128
    lr = hp.training_lr
    m = {"loss_vs_bf16_oracle": rel_err(got["losses"], lbf), "loss_vs_fp64_oracle": rel_err(got["losses"], l64),
         "param_leaf_rms_in_lr": _per_leaf_rms_in_lr(got["params"], pbf, hp, 225, 10, lr)}
    METRICS["c1_negative_lr"] = m
    # 5e-3 here (2e-3 elsewhere): with negative learning rates the update ASCENDS the loss for 88 of the 128 steps at up
    # to 5x the step size, which amplifies the bf16-ulp rounding differences between the two implementations
    # (measured 1.4e-3 .. 2.0e-3 across kernel revisions)
    assert m["loss_vs_bf16_oracle"] < 5e-3, m
    assert m["loss_vs_fp64_oracle"] < 3e-2, m
    # the schedule itself, observable: a run with the SAME inputs but a constant learning rate must differ
    hp_const = P.Hyper(num_envs=16, num_steps=10, num_minibatches=32, update_epochs=4, anneal_lr=False)
    got_const = run_gpu_update(hp_const, pr, cuda_device)
    assert np.abs(got_const["params"] - got["params"]).max() > 10 * lr
    # sum_k |lr_k| = (20 + 0 + 20 + 40 + 60 + 80 + 8 * 5) lr = 260 lr of possible travel (128 lr at constant lr)
    assert max(m["param_leaf_rms_in_lr"].values()) < 5.0, m


@pytest.mark.parametrize("name", ["medium", "ragged", "deep"] + FUSED_SHAPE_CASES)
def test_single_minibatch_gradient(name, cuda_device):
    """E = 1, M = 1: the one minibatch is the whole batch, so the gradient the optimizer saw can
    be read back and compared leaf by leaf with the hand-derived / autograd-checked oracle."""
    case = CASES[name]
    kw = dict(case["hp"])
    kw.update(num_minibatches=1, update_epochs=1)
    hp = P.Hyper(**kw)
    pr = synth.make_problem(hp, case["D"], case["A"], seed=9, done_p=0.02)
    # perturb the policy so that ratio != 1 and both clip branches are exercised
    g = np.random.default_rng(1)
    pr["traj"]["log_prob"] = (pr["traj"]["log_prob"] + 0.3 * g.standard_normal(pr["traj"]["log_prob"].shape)).astype(np.float32)
    pr["traj"]["value"] = (pr["traj"]["value"] + 0.3 * g.standard_normal(pr["traj"]["value"].shape)).astype(np.float32)
    got = run_gpu_update(hp, pr, cuda_device)

    def oracle_grads(dtype, gemm):
        p0 = P.tree_like(pr["params"], lambda x: x.astype(dtype))
        adv, tgt = P.gae(pr["traj"]["reward"], pr["traj"]["value"], pr["traj"]["done"], pr["last_val"], hp.gamma,
                         hp.gae_lambda, dtype)
        flat = P.flatten_traj({"obs": pr["traj"]["obs"].astype(dtype), "action": pr["traj"]["action"].astype(dtype),
                               "value": pr["traj"]["value"].astype(dtype), "log_prob": pr["traj"]["log_prob"].astype(dtype),
                               "adv": adv, "tgt": tgt})
        _, sub = threefry.split(pr["rng"], 2, hp.prng_mode)
        perm = threefry.permutation(sub, hp.batch_size, hp.prng_mode)
        mb = {k: v[perm] for k, v in flat.items()}
        ls, gr = P.loss_and_grads(p0, mb, hp, gemm)
        return ls, flat_grads(gr, hp.num_layers)

    ls64, g64 = oracle_grads(np.float64, "exact")
    lsbf, gbf = oracle_grads(np.float32, "bf16")
    ggpu = got["grad"][:g64.size].astype(np.float64)
    m = {
        "grad_vs_bf16_oracle": rel_err(ggpu, gbf), "grad_vs_fp64_oracle": rel_err(ggpu, g64),
        "loss_vs_bf16_oracle": rel_err(got["losses"][0, 0], np.array(lsbf)),
        "loss_vs_fp64_oracle": rel_err(got["losses"][0, 0], np.array(ls64)),
        "gnorm_gpu": float(got["grad_norms"][0, 0]), "gnorm_fp64": float(np.linalg.norm(g64)),
    }
    # per-leaf relative errors (relative to the leaf's own max): the hidden-layer leaves are ~1e-4 of the largest
    # gradient entry, so the whole-gradient figures above cannot see them
    def leaf_err(ref):
        return {k: rel_err(ggpu[s], ref[s]) for k, s in leaf_slices(case["D"], case["A"], hp.hidden_size, hp.num_layers)}

    leaf_bf, leaf_64 = leaf_err(gbf), leaf_err(g64)
    m.update({"leaf/" + k: v for k, v in leaf_bf.items()})
    m.update({"leaf_fp64/" + k: v for k, v in leaf_64.items()})
    METRICS["grad_" + name] = m
    assert m["grad_vs_bf16_oracle"] < 5e-3, m
    assert m["grad_vs_fp64_oracle"] < 5e-2, m
    assert not leaves_over(leaf_bf, LEAF_BOUND_BF16), m
    assert not leaves_over(leaf_64, LEAF_BOUND_FP64, fp64_leaf_bounds(hp)), m
    assert m["loss_vs_bf16_oracle"] < 2e-3, m
    assert abs(m["gnorm_gpu"] - m["gnorm_fp64"]) < 3e-2 * m["gnorm_fp64"], m


def test_update_deterministic_and_graph_equals_eager(cuda_device):
    """No atomics anywhere: two runs are bitwise identical, and the CUDA-graph replay equals the
    directly enqueued kernels."""
    hp = P.Hyper(**CASES["medium"]["hp"])
    pr = synth.make_problem(hp, 225, 10, seed=3)
    a = run_gpu_update(hp, pr, cuda_device, use_graph=True)
    b = run_gpu_update(hp, pr, cuda_device, use_graph=True)
    c = run_gpu_update(hp, pr, cuda_device, use_graph=False)
    for k in ("params", "mu", "nu", "losses", "grad"):
        assert np.array_equal(a[k], b[k]), k
        assert np.array_equal(a[k], c[k]), k


@pytest.mark.parametrize("fused", [True, False])
def test_precise_tanh_mode_matches_emulated_oracle_tightly(fused, cuda_device):
    """learner.fast_tanh=false evaluates tanh through ex2/rcp (abs. err ~1e-7): with the same bf16
    rounding points emulated in the oracle, losses agree to fp32 summation-order noise (1e-5)."""
    case = CASES["medium"]
    hp = P.Hyper(**case["hp"])
    pr = synth.make_problem(hp, case["D"], case["A"], seed=7, done_p=0.02)
    got = run_gpu_update(hp, pr, cuda_device, fast_tanh=False, fused=fused)
    _, _, _, lbf, auxbf = _oracle(hp, pr, np.float32, "bf16")
    METRICS[f"precise_tanh_fused={fused}"] = {"loss_vs_bf16_oracle": rel_err(got["losses"], lbf)}
    assert rel_err(got["losses"], lbf) < 1e-5
    assert rel_err(got["grad_norms"], auxbf["grad_norms"]) < 1e-3


@pytest.mark.parametrize("name", ["c1", "medium"])
def test_fused_step_kernel_equals_layerwise_kernels(name, cuda_device):
    """The fused forward+loss+backward kernel (L == 2) and the layer-wise GEMM kernels share every
    rounding point; they differ only in fp32 summation order of the head partials."""
    case = CASES[name]
    hp = P.Hyper(**case["hp"])
    pr = synth.make_problem(hp, case["D"], case["A"], seed=7, done_p=0.02)
    a = run_gpu_update(hp, pr, cuda_device, fused=True)
    b = run_gpu_update(hp, pr, cuda_device, fused=False)
    assert a["launches"] < b["launches"]
    assert rel_err(a["losses"], b["losses"]) < 2e-4
    # the gradient read back is the LAST step's; on config 1 (5-row minibatches, 128 steps) the two
    # runs have drifted apart by then, so the tight check is for the few-step case only
    # (both paths are separately held to the oracle at 5e-3; between them the fused path's tensor-core
    # heads (bf16 hi/lo split) vs the fp32 SIMT heads drift apart by ~2e-3 of the largest gradient entry)
    assert rel_err(a["grad"][:-4], b["grad"][:-4]) < (4e-3 if name == "medium" else 1e-1)
    lr = hp.opt_lr if not hp.anneal_lr else hp.training_lr
    nsteps = hp.update_epochs * hp.num_minibatches
    assert np.abs(a["params"] - b["params"]).max() < lr * (2.0 + 0.15 * nsteps)


def test_update_resumes_from_optimizer_state(cuda_device):
    """Second update starting from non-zero mu/nu/count (what RunnerState carries across
    _update_step calls, train.py:276-281) matches the oracle continuing from the same state."""
    hp = P.Hyper(**CASES["medium"]["hp"])
    pr = synth.make_problem(hp, 225, 10, seed=4)
    p0 = P.tree_like(pr["params"], lambda x: x.astype(np.float32))
    p1, o1, rng1, _, aux1 = P.update(p0, P.init_opt_state(p0), pr["traj"], pr["last_val"], pr["rng"], hp,
                                     dtype=np.float32, gemm="bf16")
    pr2 = dict(pr)
    pr2["params"], pr2["rng"] = p1, rng1
    got = run_gpu_update(hp, pr2, cuda_device, opt=o1)
    p2, o2, rng2, l2, aux2 = P.update(p1, o1, pr["traj"], pr["last_val"], rng1, hp, dtype=np.float32, gemm="bf16")
    assert got["step"] == o2["count"]
    assert np.array_equal(got["rng"], rng2)
    assert np.array_equal(got["perms"], aux2["perms"])
    assert rel_err(got["losses"], l2) < 2e-3
    lr = hp.training_lr
    assert np.abs(got["params"] - P.flatten_params(p2, hp.num_layers, np.float64)).max() < 3.2 * lr


def test_update_rejects_bad_arguments(cuda_device):
    import torch

    from minppo_b200 import _lib
    from minppo_b200.learner import Learner
    from tests.helpers import hyper_to_config

    with pytest.raises(ValueError, match="batch_size"):          # train.py:253-255
        Learner(hyper_to_config(P.Hyper(num_envs=10, num_steps=3, num_minibatches=4)), 8, 2, cuda_device)
    with pytest.raises(_lib.MinppoError) as e:
        Learner(hyper_to_config(P.Hyper(num_envs=16, num_steps=4, num_minibatches=4, hidden_size=100)), 8, 2, cuda_device)
    assert e.value.code == _lib.ERR_UNSUPPORTED
    lrn = Learner(hyper_to_config(P.Hyper(num_envs=16, num_steps=4, num_minibatches=4)), 8, 2, cuda_device)
    from minppo_b200.learner import Memory, TrainState

    ts = TrainState.create(np.zeros(lrn.P, np.float32), cuda_device)
    z = lambda *s: torch.zeros(*s, device=cuda_device)
    bad = Memory(done=torch.zeros(4, 16, dtype=torch.bool, device=cuda_device), action=z(4, 16, 2), value=z(4, 16),
                 reward=z(4, 16), log_prob=z(4, 16), obs=z(4, 16, 9))     # wrong obs dim
    with pytest.raises(ValueError, match="obs"):
        lrn.update(ts, bad, z(16), torch.zeros(2, dtype=torch.int32, device=cuda_device))
    lrn.close()


def test_dw_grid_past_one_wave_takes_the_two_launch_path(cuda_device):
    """d1000_two_launch really runs the fallback: one more launch per minibatch step than the automatic split-K factor,
    whose dW grid fits one CTA per SM (S = 2: 80 CTAs) and merges the GEMM and the optimizer into one launch."""
    case = CASES["d1000_two_launch"]
    hp = P.Hyper(**case["hp"])
    pr = synth.make_problem(hp, case["D"], case["A"], seed=7, done_p=0.02)
    auto = run_gpu_update(hp, pr, cuda_device)
    two = run_gpu_update(hp, pr, cuda_device, **case["cfg"])
    assert two["launches"] == auto["launches"] + hp.update_epochs * hp.num_minibatches


def test_row_list_overflow_raises_the_device_flag_and_poisons_the_losses(cuda_device, monkeypatch):
    """Env-sharded ranks size their per-minibatch row lists for 1.5 x the mean + 256 rows.  A list that does not fit must
    not bias the gradient silently: compact_rows raises the device-side error flag, every reported loss of that update
    becomes NaN (visible without a host round trip), and Learner.check() names the cause.  MINPPO_FORCE_CAP undersizes the
    list on one GPU."""
    import torch

    from minppo_b200 import _lib
    from minppo_b200.learner import Learner, Memory, TrainState
    from tests.helpers import hyper_to_config

    monkeypatch.setenv("MINPPO_FORCE_CAP", "256")                # minibatches have 512 rows
    hp = P.Hyper(**CASES["medium"]["hp"])
    pr = synth.make_problem(hp, 225, 10, seed=3)
    lrn = Learner(hyper_to_config(hp), 225, 10, cuda_device)
    monkeypatch.delenv("MINPPO_FORCE_CAP")
    t = lambda x: torch.as_tensor(np.ascontiguousarray(x)).to(cuda_device)
    tr = pr["traj"]
    mem = Memory(done=t(tr["done"]), action=t(tr["action"]), value=t(tr["value"]), reward=t(tr["reward"]),
                 log_prob=t(tr["log_prob"]), obs=t(tr["obs"]))
    ts = TrainState.create(P.flatten_params(pr["params"], hp.num_layers), cuda_device)
    rng = torch.as_tensor(pr["rng"].view(np.int32)).to(cuda_device)
    ts, _, losses = lrn.update(ts, mem, t(pr["last_val"]), rng)
    torch.cuda.synchronize(cuda_device)
    assert torch.isnan(losses).all()
    with pytest.raises(_lib.MinppoError) as e:
        lrn.check()
    assert e.value.code in (_lib.ERR_WORKSPACE,)
    lrn.close()
