"""Shapes of the per-leaf gradient tests and the learner's path selection restated in Python.

``CASES`` is shared by tests/test_gpu_gradient_leaves.py (the GPU against the oracle) and
tests/test_gradient_check_host.py (the oracle against itself, no device).  Every case runs one
minibatch step (E = M = 1), so the minibatch is the whole batch: mb = num_envs * num_steps.

``learner_path`` repeats the host-side choices of minppo_ctx_create / enqueue_step
(minppo_b200/csrc/learner.cu, dwopt.cuh, head_loss.cu) from the shapes and the SM count, so that
each case can assert the path it is meant to reach: a heuristic change that moves a case to another
path then fails the case instead of silently testing something else.  ``launches`` is observable
(``Learner.launches_per_update``) and ties the restatement to the library.
"""
from __future__ import annotations

import math

from oracle import ppo_numpy as P
from oracle import threefry

DWOPT_THREADS = 512          # dwopt.cuh
GEMM_MAXN = 256              # umma_gemm.cuh: widest tcgen05 tile; wider hidden layers run as two column groups
GEMM_MAX_GROUPS = 8
FS_MAX_AP = 32               # fused_step.cuh: widest padded head of the fused step kernel


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


def param_count(D: int, A: int, H: int, L: int) -> int:
    n = 0
    for out in (A, 1):
        fan_in = D
        for i in range(L + 1):
            o = H if i < L else out
            n += o + fan_in * o
            fan_in = o
    return n + A


def perm_launch_count(B: int) -> int:          # prng_sort.cu
    return math.ceil(3.0 * math.log(max(B, 1)) / math.log(4294967295.0)) * 4 * 3


def learner_path(hp: dict, D: int, A: int, sm_count: int, cfg: dict | None = None, force_cap: int | None = None) -> dict:
    """The single-GPU path minppo_ctx_create picks for a shape (learner.cu), and the launch count of one update."""
    cfg = cfg or {}
    h = P.Hyper(**hp)
    H, L, E, M, B = h.hidden_size, h.num_layers, h.update_epochs, h.num_minibatches, h.batch_size
    mb = B // M
    padded = force_cap is not None
    cap = force_cap if padded else mb
    M_pad = (cap + 127) // 128 * 128
    Dp = (D + 63) // 64 * 64
    fused = cfg.get("fused", True) and L == 2 and H <= GEMM_MAXN and A <= FS_MAX_AP
    n_params = param_count(D, A, H, L)
    cap1 = 4 * sm_count * DWOPT_THREADS
    maxu = 1 if n_params <= cap1 else (2 if n_params <= 2 * cap1 else 4)
    dw_nsplit = 2 if H > GEMM_MAXN else (2 if fused and H % 128 == 0 and 2 * 2 * L <= GEMM_MAX_GROUPS else 1)
    per_split = sum(2 * dw_nsplit * (((Dp if l == 0 else H) + 127) // 128) for l in range(L))
    budget = sm_count - 16 if sm_count > 48 else sm_count
    S = cfg.get("dw_splits", 0) or budget // max(per_split, 1)
    kb_total = M_pad // 64
    if padded:
        kb_total = max(min(M_pad, int(mb + 3.0 * math.sqrt(mb)) + 1 + 63) // 64, 1)
    S = max(min(S, kb_total, 32), 1)
    while S > 1 and -(-kb_total // S) * (S - 1) >= kb_total:
        S -= 1
    gemm_ctas = per_split * S
    two_launch = gemm_ctas > sm_count
    # register-resident (fast) dwopt path: the 4-element units of the "late" leaves (hidden kernels; layer-wise also the
    # hidden biases, whose column sums the dW GEMM computes) fit MAXU per thread of the one-CTA-per-SM grid
    late = 0
    fan_in = D
    for _ in range(L):
        late += fan_in * H + (0 if fused else H)
        fan_in = H
    late *= 2
    fast = late // 4 <= sm_count * DWOPT_THREADS * maxu
    per_step = (1 if fused else 2 * L) + (2 if two_launch else 1)
    launches = 2 + 1 + perm_launch_count(B) + 1 + 3 + E * M * per_step
    return dict(fused=fused, P=n_params, maxu=maxu, fast=fast, dw_nsplit=dw_nsplit, hsplit=2 if H > GEMM_MAXN else 1,
                ap=16 if A <= 16 else 32, head_amax=8 if A <= 8 else (16 if A <= 16 else (32 if A <= 32 else 64)),
                S=S, gemm_ctas=gemm_ctas, two_launch=two_launch, padded=padded, cap=M_pad, launches=launches)
