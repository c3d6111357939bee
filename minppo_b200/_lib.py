"""ctypes binding of libminppo_b200.so (the C ABI in include/minppo_b200.h).

The shared library is built in-tree by ``minppo_b200/csrc/build.sh`` (nvcc, sm_100a).  There
is no fallback: if the library is missing, importing a symbol raises with the build command.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libminppo_b200.so")

OK = 0
ERR_ARG, ERR_CUDA, ERR_WORKSPACE, ERR_UNSUPPORTED, ERR_NCCL, ERR_BARRIER, ERR_NONFINITE = -1, -2, -3, -4, -5, -6, -7
PRNG_LEGACY, PRNG_PARTITIONABLE = 0, 1
MAX_LEAVES = 32

# every symbol include/minppo_b200.h declares (tests check the library exports all of them)
SYMBOLS = (
    "minppo_last_error", "minppo_version", "minppo_gae", "minppo_gae_chunked",
    "minppo_permutation_workspace_size", "minppo_permutation", "minppo_param_layout",
    "minppo_nccl_unique_id", "minppo_ctx_create", "minppo_ctx_destroy", "minppo_update",
    "minppo_ctx_check", "minppo_update_launch_count", "minppo_ctx_read", "minppo_debug_gemm",
    "minppo_ctx_profile", "minppo_ctx_profile_read", "minppo_ctx_ipc_handle", "minppo_ctx_set_peers",
    "minppo_policy_step", "minppo_update_with_stats", "minppo_plan",
    "minppo_update_normalized", "minppo_policy_step_normalized", "minppo_obs_norm_fold",
)
POLICY_WEIGHTS_CURRENT = 1
PROFILE_CLASSES = ("gae", "perm_sort", "rows_and_adv_stats", "obs_image", "weight_images", "fwd_gemm", "head_loss",
                   "bwd_gemm", "dw_gemm", "optimizer", "allreduce")


class MinppoConfig(C.Structure):
    """``struct minppo_config`` -- field order and types must match the header."""
    _fields_ = [
        ("num_envs", C.c_int32), ("num_steps", C.c_int32), ("num_minibatches", C.c_int32),
        ("update_epochs", C.c_int32), ("total_timesteps", C.c_int64), ("anneal_lr", C.c_int32),
        ("hidden_size", C.c_int32), ("num_layers", C.c_int32), ("use_tanh", C.c_int32),
        ("obs_dim", C.c_int32), ("act_dim", C.c_int32), ("prng_mode", C.c_int32),
        ("world_size", C.c_int32), ("rank", C.c_int32), ("fast_tanh", C.c_int32), ("dw_splits", C.c_int32),
        ("disable_fused", C.c_int32),
        ("training_lr", C.c_double), ("opt_lr", C.c_double), ("max_grad_norm", C.c_double),
        ("gamma", C.c_double), ("gae_lambda", C.c_double), ("clip_eps", C.c_double),
        ("ent_coef", C.c_double), ("vf_coef", C.c_double),
        ("adam_b1", C.c_double), ("adam_b2", C.c_double), ("adam_eps", C.c_double), ("adam_eps_root", C.c_double),
    ]


class MinppoPlan(C.Structure):
    """``struct minppo_plan`` -- field order and types must match the header."""
    _fields_ = [("num_params", C.c_int64)] + [(n, C.c_int32) for n in (
        "fused", "ap", "head_amax", "hsplit", "dw_nsplit", "S", "dw_gemm_ctas", "two_launch",
        "maxu", "dwopt_fast", "padded", "row_cap", "peer_exchange")]


class MinppoObsNorm(C.Structure):
    """``struct minppo_obs_norm`` -- field order and types must match the header."""
    _fields_ = [("mean", C.c_void_p), ("var", C.c_void_p), ("count", C.c_void_p), ("eps", C.c_double), ("clip", C.c_double)]


class MinppoError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"minppo_b200 error {code}: {msg}")
        self.code = code


_lib: Optional[C.CDLL] = None


def load() -> C.CDLL:
    """Load the shared library (once) and declare every prototype."""
    global _lib
    if _lib is not None:
        return _lib
    global LIB_PATH
    LIB_PATH = os.environ.get("MINPPO_B200_LIB", LIB_PATH)      # development: A/B a differently compiled build
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: the CUDA library is not built. Run `bash minppo_b200/csrc/build.sh` "
            "(or `python -c 'import __graft_entry__ as g; g.build()'`). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, f64, sz = C.c_void_p, C.c_int32, C.c_int64, C.c_double, C.c_size_t
    lib.minppo_last_error.restype = C.c_char_p
    lib.minppo_last_error.argtypes = []
    lib.minppo_version.restype = C.c_int
    lib.minppo_gae.restype = C.c_int
    lib.minppo_gae.argtypes = [vp, vp, vp, vp, vp, vp, i32, i64, f64, f64, vp]
    lib.minppo_gae_chunked.restype = C.c_int
    lib.minppo_gae_chunked.argtypes = [vp, vp, vp, vp, vp, vp, i32, i64, f64, f64, i32, vp]
    lib.minppo_permutation_workspace_size.restype = sz
    lib.minppo_permutation_workspace_size.argtypes = [i32, i64]
    lib.minppo_permutation.restype = C.c_int
    lib.minppo_permutation.argtypes = [vp, vp, i32, i32, i64, vp, vp, sz, vp]
    lib.minppo_param_layout.restype = i64
    lib.minppo_param_layout.argtypes = [C.POINTER(MinppoConfig), C.POINTER(i32), C.POINTER(i64), C.POINTER(i64),
                                        C.POINTER(i64)]
    lib.minppo_nccl_unique_id.restype = C.c_int
    lib.minppo_nccl_unique_id.argtypes = [vp]
    lib.minppo_plan.restype = C.c_int
    lib.minppo_plan.argtypes = [C.POINTER(MinppoConfig), i32, C.POINTER(MinppoPlan)]
    lib.minppo_ctx_create.restype = C.c_int
    lib.minppo_ctx_create.argtypes = [C.POINTER(MinppoConfig), vp, C.POINTER(vp)]
    lib.minppo_ctx_destroy.restype = C.c_int
    lib.minppo_ctx_destroy.argtypes = [vp]
    lib.minppo_update.restype = C.c_int
    lib.minppo_update.argtypes = [vp] + [vp] * 14 + [i32, vp]
    lib.minppo_update_with_stats.restype = C.c_int
    lib.minppo_update_with_stats.argtypes = [vp] + [vp] * 15 + [i32, vp]
    norm = C.POINTER(MinppoObsNorm)
    lib.minppo_update_normalized.restype = C.c_int
    lib.minppo_update_normalized.argtypes = [vp] + [vp] * 15 + [norm, i32, vp]
    lib.minppo_obs_norm_fold.restype = C.c_int
    lib.minppo_obs_norm_fold.argtypes = [vp, i64, i32, norm, vp]
    lib.minppo_ctx_check.restype = C.c_int
    lib.minppo_ctx_check.argtypes = [vp, vp]
    lib.minppo_update_launch_count.restype = i64
    lib.minppo_update_launch_count.argtypes = [vp]
    lib.minppo_ctx_read.restype = C.c_int
    lib.minppo_ctx_read.argtypes = [vp, i32, vp, sz, vp]
    lib.minppo_ctx_profile.restype = C.c_int
    lib.minppo_ctx_profile.argtypes = [vp, i32]
    lib.minppo_ctx_profile_read.restype = C.c_int
    lib.minppo_ctx_profile_read.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(i32), i32]
    lib.minppo_ctx_ipc_handle.restype = C.c_int
    lib.minppo_ctx_ipc_handle.argtypes = [vp, vp]
    lib.minppo_ctx_set_peers.restype = C.c_int
    lib.minppo_ctx_set_peers.argtypes = [vp, vp]
    lib.minppo_policy_step.restype = C.c_int
    lib.minppo_policy_step.argtypes = [vp] * 9 + [i32, vp]
    lib.minppo_policy_step_normalized.restype = C.c_int
    lib.minppo_policy_step_normalized.argtypes = [vp] * 9 + [norm, i32, vp]
    lib.minppo_debug_gemm.restype = C.c_int
    lib.minppo_debug_gemm.argtypes = [i32, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]
    _lib = lib
    return lib


def check(code: int) -> None:
    if code != 0:
        raise MinppoError(code, load().minppo_last_error().decode("utf-8", "replace"))
