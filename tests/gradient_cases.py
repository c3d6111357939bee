"""Shapes of the per-leaf gradient tests and the learner path each of them must reach.

``CASES`` is shared by tests/test_gpu_gradient_leaves.py (the GPU against the oracle) and
tests/test_gradient_check_host.py (the oracle against itself, no device).  Every case runs one
minibatch step (E = M = 1), so the minibatch is the whole batch: mb = num_envs * num_steps.

``learner_path`` asks the library (minppo_plan, the host-only path decision of minppo_ctx_create)
which kernels a shape reaches at an SM count, so that each case can assert the path it is meant to
reach: a heuristic change that moves a case to another path then fails the case instead of silently
testing something else.  ``launches`` counts the launches of one update on that path; the GPU tests
compare it with the count the library issued (``Learner.launches_per_update``).
"""
from __future__ import annotations

import ctypes as C
import math
import os
from unittest import mock

from minppo_b200 import _lib
from minppo_b200.config import to_c_config
from oracle import ppo_numpy as P
from oracle import threefry
from tests.helpers import hyper_to_config


def _case(N, T, D, A, H=256, L=2, cfg=None, expect=None, force_cap=None, **hp):
    kw = dict(num_envs=N, num_steps=T, num_minibatches=1, update_epochs=1, anneal_lr=False, hidden_size=H, num_layers=L)
    kw.update(hp)
    return dict(hp=kw, D=D, A=A, cfg=dict(cfg or {}), expect=dict(expect or {}), force_cap=force_cap)


# name -> shape, learner options and the path the case must reach (keys of learner_path's result)
CASES = {
    "h256_d225_mb2048": _case(64, 32, 225, 10, expect=dict(fused=True, dw_nsplit=2, maxu=1, fast=True, two_launch=False)),
    "a32_h192": _case(32, 16, 321, 32, H=192, expect=dict(fused=True, dw_nsplit=1, ap=32, two_launch=False)),
    # smallest observation and action widths; 200 rows: the last 128-row tile holds 72
    "d1_a1_mb200": _case(25, 8, 1, 1, H=64, ent_coef=0.01, expect=dict(fused=True, ap=16, two_launch=False)),
    # one row past a 64-row tile (and short of a 128-row one); relu actor
    "a17_mb65": _case(13, 5, 600, 17, H=128, use_tanh=False, expect=dict(fused=True, ap=32, two_launch=False)),
    # one row past a 128-row tile, layer-wise kernels
    "layerwise_a8_mb129": _case(43, 3, 225, 8, cfg=dict(fused=False), expect=dict(fused=False, head_amax=8)),
    # one hidden layer (always layer-wise), relu actor, one row short of a 128-row tile
    "l1_a9_mb127": _case(127, 1, 37, 9, H=128, L=1, use_tanh=False, ent_coef=0.01,
                         expect=dict(fused=False, head_amax=16)),
    "l3_a24_mb333": _case(37, 9, 100, 24, H=192, L=3, prng_mode=threefry.PARTITIONABLE,
                          expect=dict(fused=False, head_amax=32)),
    # H = 320 > GEMM_MAXN: column groups of 192 + 128; A = 40 > 32: layer-wise, 64-wide head template
    "h320_a40": _case(16, 16, 415, 40, H=320, expect=dict(fused=False, hsplit=2, dw_nsplit=2, head_amax=64)),
    # 1.55 M hidden-kernel parameters: more than four register-resident units per thread of the dwopt grid
    "h512_d1000_a64": _case(32, 8, 1000, 64, H=512, expect=dict(fused=False, maxu=4, fast=False, head_amax=64)),
    "maxu2_d415_a20": _case(32, 16, 415, 20, expect=dict(fused=True, maxu=2, fast=True, two_launch=False)),
    "maxu4_d1000": _case(32, 16, 1000, 10, expect=dict(fused=True, maxu=4, fast=True, two_launch=False)),
    # the two-launch sequence (stand-alone dW GEMM, then dwopt without GEMM CTAs): 4 (fused) / 8 (layer-wise) splits of a
    # D = 1000 network do not fit one CTA per SM
    "two_launch_fused": _case(32, 16, 1000, 10, cfg=dict(dw_splits=4), expect=dict(fused=True, S=4, two_launch=True)),
    "two_launch_layerwise": _case(32, 16, 1000, 10, cfg=dict(dw_splits=8, fused=False),
                                  expect=dict(fused=False, S=8, two_launch=True)),
    # padded row lists (what env-sharded ranks use) on one GPU: a 520-row capacity for 200-row minibatches, so the
    # kernels take the row count from the device (k-block skip, live tiles) and nothing overflows
    "padded_fused": _case(25, 8, 225, 10, force_cap=520, expect=dict(fused=True, padded=True, cap=640)),
    "padded_layerwise": _case(25, 8, 225, 10, force_cap=520, cfg=dict(fused=False),
                              expect=dict(fused=False, padded=True, cap=640)),
    # non-default PPO coefficients: the value-clip and ratio-clip branches at a narrow clip, the entropy bonus as the
    # log_std gradient's bias, precise tanh
    "coef_fused": _case(32, 16, 225, 10, clip_eps=0.05, vf_coef=1.0, ent_coef=0.02, cfg=dict(fast_tanh=False),
                        expect=dict(fused=True)),
    "coef_layerwise": _case(32, 16, 225, 10, clip_eps=0.05, vf_coef=1.0, ent_coef=0.02,
                            cfg=dict(fast_tanh=False, fused=False), expect=dict(fused=False)),
}
# split-K of the dW GEMMs at 512 rows (8 k-blocks of 64): even (1, 2, 4, 8) and uneven (3: 3 + 3 + 2 k-blocks) factors.
# (The constructor lowers a factor that would leave a split empty, 5 -> 4 at 8 k-blocks.)
for _s in (1, 2, 3, 4, 8):
    CASES[f"splits{_s}_fused"] = _case(32, 16, 225, 10, cfg=dict(dw_splits=_s), expect=dict(fused=True, S=_s, two_launch=False))
    CASES[f"splits{_s}_layerwise"] = _case(32, 16, 225, 10, cfg=dict(dw_splits=_s, fused=False),
                                           expect=dict(fused=False, S=_s, two_launch=False))


def perm_launch_count(B: int) -> int:          # prng_sort.cu
    return math.ceil(3.0 * math.log(max(B, 1)) / math.log(4294967295.0)) * 4 * 3


def learner_path(hp: dict, D: int, A: int, sm_count: int, cfg: dict | None = None, force_cap: int | None = None) -> dict:
    """The single-GPU path the library plans for a shape (minppo_plan), and the launch count of one update.
    ``cfg``: keyword arguments of tests.helpers.hyper_to_config; ``force_cap``: MINPPO_FORCE_CAP for the call."""
    h = P.Hyper(**hp)
    c = to_c_config(hyper_to_config(h, **(cfg or {})), D, A)
    plan = _lib.MinppoPlan()
    with mock.patch.dict(os.environ, {} if force_cap is None else {"MINPPO_FORCE_CAP": str(force_cap)}):
        _lib.check(_lib.load().minppo_plan(C.byref(c), sm_count, C.byref(plan)))
    fused, two_launch = bool(plan.fused), bool(plan.two_launch)
    per_step = (1 if fused else 2 * h.num_layers) + (2 if two_launch else 1)
    launches = 2 + 1 + perm_launch_count(h.batch_size) + 1 + 3 + h.update_epochs * h.num_minibatches * per_step
    return dict(fused=fused, P=plan.num_params, maxu=plan.maxu, fast=bool(plan.dwopt_fast), dw_nsplit=plan.dw_nsplit,
                hsplit=plan.hsplit, ap=plan.ap, head_amax=plan.head_amax, S=plan.S, gemm_ctas=plan.dw_gemm_ctas,
                two_launch=two_launch, padded=bool(plan.padded), cap=plan.row_cap, launches=launches)
