"""Host-side pieces of bench.py that run without a GPU: the workload table, the product Config it builds, and the
synthetic parameter generator (which must stay the oracle's recipe so that the CPU arm and the GPU arm time the same
problem).  bench.py's product arm must not import oracle/ (the oracle is the checker, never the thing measured)."""
import ast
import os
import sys

import numpy as np
import pytest

import bench
from minppo_b200.config import to_c_config
from minppo_b200.params import flatten_params, param_count
from oracle import ppo_numpy as P

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_workloads_match_baseline_configs():
    w1 = bench.workload(1)
    assert (w1["num_envs"], w1["num_steps"], w1["num_minibatches"], w1["update_epochs"]) == (2048, 128, 32, 4)
    w8 = bench.workload(8)
    assert w8["num_envs"] == 16384 and w8["scaling"] == "weak"            # configs[1] per GPU == configs[3]'s env count
    c4 = bench.workload(4, "c4")
    assert (c4["num_envs"], c4["num_steps"], c4["scaling"]) == (16384, 64, "strong")
    hp = bench.make_shape(w1)
    assert hp.batch_size == 262144 and hp.minibatch_size == 8192


def test_config_built_by_bench_is_the_reference_default_shape():
    hp = bench.make_shape(bench.workload(1))
    cfg = bench.make_config(hp, True)
    c = to_c_config(cfg, bench.OBS_DIM, bench.ACT_DIM)
    assert (c.num_envs, c.num_steps, c.num_minibatches, c.update_epochs) == (2048, 128, 32, 4)
    assert (c.hidden_size, c.num_layers, c.use_tanh, c.anneal_lr) == (256, 2, 1, 1)
    assert c.total_timesteps == 1_000_000_000 and abs(c.clip_eps - 0.2) < 1e-12 and abs(c.adam_eps - 1e-5) < 1e-18
    # same numbers as the oracle's record of the shape
    ho = bench.make_hyper(hp)
    assert (ho.gamma, ho.gae_lambda, ho.clip_eps, ho.vf_coef, ho.ent_coef) == (c.gamma, c.gae_lambda, c.clip_eps, c.vf_coef, c.ent_coef)
    assert ho.minibatch_size == hp.minibatch_size and ho.anneal_lr


def test_synthetic_parameters_are_the_oracles_recipe():
    a = flatten_params(bench.init_param_tree(256, 2, 0), 2)
    b = P.flatten_params(P.init_params(bench.OBS_DIM, bench.ACT_DIM, 256, 2, 0, np.float32), 2)
    assert a.size == param_count(bench.OBS_DIM, bench.ACT_DIM, 256, 2) == 250133          # SURVEY.md 8a row 4
    assert np.array_equal(a, b)


def test_synthetic_inputs_do_not_depend_on_the_thread_count():
    """The benchmark's inputs are the same bits in every run, so that outputs of two builds can be compared exactly."""
    import torch

    hp = bench.BenchShape(num_envs=64, num_steps=16, num_minibatches=4, update_epochs=1)
    threads = torch.get_num_threads()
    shards = []
    try:
        for t in (1, 3):
            torch.set_num_threads(t)
            shards.append(bench.synth_shard(hp, 0, 1))
            assert torch.get_num_threads() == t
    finally:
        torch.set_num_threads(threads)
    (_, a, lva), (_, b, lvb) = shards
    assert np.array_equal(lva, lvb) and lva.dtype == np.float32
    for k in a:
        assert np.array_equal(a[k], b[k]), k


def test_dump_outputs_types_and_size_limit(tmp_path, monkeypatch):
    """float32 / float64 files named after the outputs; over the limit, a large array becomes the same seeded sample of
    its elements in every run, and the files stay within the limit."""
    params = np.arange(1000, dtype=np.float32) / 7
    arrays = {"params": params, "step": np.array([128], np.int32), "rng_out": np.array([0xFFFFFFFF, 7], np.uint32)}
    bench.dump_outputs(str(tmp_path / "a"), arrays)
    got = {k: np.load(tmp_path / "a" / f"{k}.npy") for k in arrays}
    assert got["params"].dtype == np.float32 and np.array_equal(got["params"], params)
    assert got["step"].dtype == np.float64 and got["step"].tolist() == [128.0]
    assert got["rng_out"].dtype == np.float64 and got["rng_out"].tolist() == [4294967295.0, 7.0]

    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 1200)
    bench.dump_outputs(str(tmp_path / "b"), arrays)
    bench.dump_outputs(str(tmp_path / "c"), arrays)
    b, c = (np.load(tmp_path / d / "params.npy") for d in "bc")
    assert np.array_equal(b, c) and b.size == 1200 // 3 // 4 and np.isin(b, params).all()
    assert sum(os.path.getsize(tmp_path / "b" / f"{k}.npy") - 128 for k in arrays) <= 1200       # 128-byte .npy header
    assert np.load(tmp_path / "b" / "step.npy").tolist() == [128.0]


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_bench_rejects_bad_arguments(argv, monkeypatch):
    monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
    with pytest.raises(SystemExit) as e:
        bench.main()
    assert e.value.code == 2


def test_product_arm_does_not_import_the_oracle():
    """Static check: `oracle` / `tests` imports appear only inside make_hyper, cpu_update_time (the CPU baseline and the
    checker of the parity flag), run_reference and gpu_proxy_time (the eager-PyTorch-on-GPU comparator)."""
    src = open(os.path.join(ROOT, "bench.py")).read()
    tree = ast.parse(src)
    allowed = {"make_hyper", "cpu_update_time", "run_reference", "gpu_proxy_time"}
    for fn in [n for n in tree.body if isinstance(n, ast.FunctionDef)]:
        mods = set()
        for n in ast.walk(fn):
            if isinstance(n, ast.ImportFrom) and n.module:
                mods.add(n.module.split(".")[0])
            elif isinstance(n, ast.Import):
                mods.update(a.name.split(".")[0] for a in n.names)
        if fn.name not in allowed:
            assert not ({"oracle", "tests"} & mods), (fn.name, mods)
    top = {n.module.split(".")[0] for n in tree.body if isinstance(n, ast.ImportFrom) and n.module} | \
          {a.name.split(".")[0] for n in tree.body if isinstance(n, ast.Import) for a in n.names}
    assert not ({"oracle", "tests"} & top)


def test_product_package_does_not_import_the_oracle():
    pkg = os.path.join(ROOT, "minppo_b200")
    for name in os.listdir(pkg):
        if name.endswith(".py"):
            tree = ast.parse(open(os.path.join(pkg, name)).read())
            for n in ast.walk(tree):
                if isinstance(n, ast.ImportFrom) and n.module:
                    assert n.module.split(".")[0] not in ("oracle", "tests"), name
                elif isinstance(n, ast.Import):
                    assert all(a.name.split(".")[0] not in ("oracle", "tests") for a in n.names), name
