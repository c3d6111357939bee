"""The C-ABI library loads on a CPU-only box and exports every symbol include/minppo_b200.h
declares; host-only entry points behave (no compute calls: there is no GPU here)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from minppo_b200 import _lib, config
from minppo_b200.params import leaf_paths, leaf_shapes, param_count
from oracle import ppo_numpy as P
from tests.helpers import hyper_to_config

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__

        __graft_entry__.build()
    return _lib.load()


def _header_symbols():
    text = open(os.path.join(ROOT, "include", "minppo_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(minppo_[a-z0-9_]+)\s*\(", text)))


def test_header_and_binding_agree(lib):
    hdr = _header_symbols()
    assert sorted(_lib.SYMBOLS) == hdr
    for s in hdr:
        assert hasattr(lib, s), f"libminppo_b200.so does not export {s}"


def test_version_and_error_string(lib):
    assert lib.minppo_version() >= 100
    assert isinstance(lib.minppo_last_error(), bytes)


def _header_fields(begin, end):
    text = open(os.path.join(ROOT, "include", "minppo_b200.h")).read()
    start = text.index(begin)
    body = re.sub(r"/\*.*?\*/", "", text[start:text.index(end, start)], flags=re.S)
    decls = [d.strip() for d in body.split("{", 1)[1].split(";") if d.strip()]
    return [n.strip() for d in decls for n in d.split(None, 1)[1].split(",")]


def test_struct_layout_matches_header():
    """Field order of the ctypes mirrors == field order of struct minppo_config and struct minppo_plan in the header."""
    names = _header_fields("typedef struct minppo_config {", "} minppo_config;")
    assert names == [f[0] for f in _lib.MinppoConfig._fields_]
    assert C.sizeof(_lib.MinppoConfig) == 4 * 4 + 8 + 12 * 4 + 12 * 8            # 4 i32, i64, 12 i32, 12 f64
    assert _header_fields("struct minppo_plan {", "};") == [f[0] for f in _lib.MinppoPlan._fields_]
    assert C.sizeof(_lib.MinppoPlan) == 8 + 14 * 4                                # i64, 14 i32


@pytest.mark.parametrize("H,L,A,limit", [(576, 2, 2, "<= 512"), (384, 3, 2, "num_layers <= 2"), (256, 2, 65, "<= 64")])
def test_plan_refuses_what_the_context_refuses(lib, H, L, A, limit):
    """minppo_plan runs the config check of minppo_ctx_create: the shapes test_wide_hidden_refusals and
    test_wide_action_refusal hand to a context are refused here with the same code and message, without a device."""
    hp = P.Hyper(num_envs=16, num_steps=4, num_minibatches=4, hidden_size=H, num_layers=L)
    cc = config.to_c_config(hyper_to_config(hp), 8, A)
    plan = _lib.MinppoPlan()
    assert lib.minppo_plan(C.byref(cc), 148, C.byref(plan)) == _lib.ERR_UNSUPPORTED
    assert limit in lib.minppo_last_error().decode()


@pytest.mark.parametrize("D,A,H,L", [(225, 10, 256, 2), (37, 3, 128, 1), (256, 16, 192, 3)])
def test_param_layout_matches_pickle_tree(lib, D, A, H, L):
    cfg = config.load_config([f"model.hidden_size={H}", f"model.num_layers={L}"])
    cc = config.to_c_config(cfg, D, A)
    n = C.c_int32()
    offs, rows, cols = (C.c_int64 * 32)(), (C.c_int64 * 32)(), (C.c_int64 * 32)()
    P = lib.minppo_param_layout(C.byref(cc), C.byref(n), offs, rows, cols)
    shapes = leaf_shapes(D, A, H, L)
    assert P == param_count(D, A, H, L) and n.value == len(shapes) == len(leaf_paths(L))
    off = 0
    for i, shp in enumerate(shapes):
        assert offs[i] == off
        assert (rows[i], cols[i]) == ((1, shp[0]) if len(shp) == 1 else shp)
        off += int(np.prod(shp))
    if (D, A, H, L) == (225, 10, 256, 2):
        assert P == 250133            # SURVEY.md section 8a row 4


def test_host_side_argument_validation(lib):
    """Null pointers are rejected on the host before any launch, with a message."""
    rc = lib.minppo_gae(None, None, None, None, None, None, 4, 4, 0.99, 0.95, None)
    assert rc == _lib.ERR_ARG and b"null" in lib.minppo_last_error()
    rc = lib.minppo_permutation(None, None, 0, 1, 16, None, None, 0, None)
    assert rc == _lib.ERR_ARG
    assert lib.minppo_permutation_workspace_size(4, 262144) >= 3 * 4 * 262144 * 4
    with pytest.raises(_lib.MinppoError):
        _lib.check(rc)
    assert lib.minppo_plan(None, 148, None) == _lib.ERR_ARG
    cc = config.to_c_config(config.load_config(), 225, 10)
    assert lib.minppo_plan(C.byref(cc), 0, C.byref(_lib.MinppoPlan())) == _lib.ERR_ARG
