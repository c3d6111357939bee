"""model.hidden_size above one 256-column GEMM tile (up to 512), host side: the C layout of the parameter arena, the
refusals that need no device, and that the parity tolerances of tests/test_gpu_wide_hidden.py are reachable at K = 512
by the bf16-emulating oracle itself before any GPU runs."""
import ctypes as C
import os

import numpy as np
import pytest

from minppo_b200 import _lib, config
from minppo_b200.params import leaf_paths, leaf_shapes, param_count
from oracle import ppo_numpy as P
from oracle import synth
from tests.helpers import rel_err


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__

        __graft_entry__.build()
    return _lib.load()


@pytest.mark.parametrize("D,A,H,L", [(225, 10, 512, 2), (415, 32, 320, 2), (37, 3, 512, 1)])
def test_param_layout_at_wide_hidden(lib, D, A, H, L):
    cc = config.to_c_config(config.load_config([f"model.hidden_size={H}", f"model.num_layers={L}"]), D, A)
    n = C.c_int32()
    offs, rows, cols = (C.c_int64 * 32)(), (C.c_int64 * 32)(), (C.c_int64 * 32)()
    total = lib.minppo_param_layout(C.byref(cc), C.byref(n), offs, rows, cols)
    shapes = leaf_shapes(D, A, H, L)
    assert total == param_count(D, A, H, L) and n.value == len(shapes) == len(leaf_paths(L))
    off = 0
    for i, shp in enumerate(shapes):
        assert offs[i] == off
        assert (rows[i], cols[i]) == ((1, shp[0]) if len(shp) == 1 else shp)
        off += int(np.prod(shp))
    if (D, A, H, L) == (225, 10, 512, 2):
        assert total == 762389


@pytest.mark.parametrize("H,L,limit", [(576, 2, b"<= 512"), (100, 2, b"multiple of 64"), (384, 3, b"num_layers <= 2")])
def test_context_refuses_unsupported_widths_before_touching_a_device(lib, H, L, limit):
    cc = config.to_c_config(config.load_config([f"model.hidden_size={H}", f"model.num_layers={L}",
                                                "training.num_envs=16", "training.num_steps=4",
                                                "rl.num_env_steps=4", "training.num_minibatches=4"]), 8, 2)
    h = C.c_void_p()
    assert lib.minppo_ctx_create(C.byref(cc), None, C.byref(h)) == _lib.ERR_UNSUPPORTED
    assert limit in lib.minppo_last_error()
    assert not h.value


def test_bf16_oracle_meets_the_fp64_tolerances_at_hidden_512():
    hp = P.Hyper(num_envs=16, num_steps=8, num_minibatches=2, update_epochs=2, anneal_lr=False, hidden_size=512)
    pr = synth.make_problem(hp, 225, 10, seed=7, done_p=0.02)
    p64 = P.tree_like(pr["params"], lambda x: x.astype(np.float64))
    pbf = P.tree_like(pr["params"], lambda x: x.astype(np.float32))
    q64, o64, rng64, l64, aux64 = P.update(p64, P.init_opt_state(p64), pr["traj"], pr["last_val"], pr["rng"], hp,
                                           dtype=np.float64, gemm="exact")
    qbf, obf, rngbf, lbf, auxbf = P.update(pbf, P.init_opt_state(pbf), pr["traj"], pr["last_val"], pr["rng"], hp,
                                           dtype=np.float32, gemm="bf16", perms=aux64["perms"])
    assert np.array_equal(rngbf, rng64)
    assert rel_err(lbf, l64) < 3e-2
    assert rel_err(auxbf["grad_norms"], aux64["grad_norms"]) < 2e-2
    lr = hp.opt_lr
    nsteps = hp.update_epochs * hp.num_minibatches
    d = P.flatten_params(qbf, hp.num_layers, np.float64) - P.flatten_params(q64, hp.num_layers, np.float64)
    assert np.abs(d).max() < lr * (2.0 + 0.15 * nsteps)
    assert np.sqrt(np.mean(d * d)) < lr
