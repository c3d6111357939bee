"""Host-side mirror of the config keys the learner reads.

Same key names, nesting and defaults as the reference's OmegaConf structured config
(/root/reference/minppo/config.py:50-84): ``model.*``, ``opt.*``, ``rl.*``, ``training.*``.
Environment / visualisation / reward / inference sub-trees are out of scope (they configure
the MJX rollout, which stays the reference's).  OmegaConf is not installed in this image, so
this is plain dataclasses plus the same dot-list override syntax (``training.num_envs=16``);
like the reference's structured config, unknown keys raise (SURVEY.md F5).
"""
from __future__ import annotations

import dataclasses
from dataclasses import dataclass, field
from typing import Any, Sequence

from . import _lib


@dataclass
class ModelConfig:                       # config.py:50-54
    hidden_size: int = 256
    num_layers: int = 2
    use_tanh: bool = True


@dataclass
class OptimizerConfig:                   # config.py:57-60
    lr: float = 3e-4
    max_grad_norm: float = 0.5


@dataclass
class ReinforcementLearningConfig:       # config.py:63-71
    num_env_steps: int = 10
    gamma: float = 0.99
    gae_lambda: float = 0.95
    clip_eps: float = 0.2
    ent_coef: float = 0.0
    vf_coef: float = 0.5


@dataclass
class TrainingConfig:                    # config.py:74-84
    lr: float = 3e-4
    seed: int = 1337
    num_envs: int = 2048
    total_timesteps: int = 1_000_000_000
    num_minibatches: int = 32
    num_steps: int = 10
    update_epochs: int = 4
    anneal_lr: bool = True
    model_save_path: str = "trained_model.pkl"


@dataclass
class LearnerExtras:
    """Keys that do not exist in the reference: how the B200 learner is run."""
    prng_mode: str = "legacy"            # "legacy" | "partitionable" (jax_threefry_partitionable, SURVEY F11)
    fast_tanh: bool = True               # tanh.approx.f32 (MUFU, rel. err ~2^-11, below the bf16 ulp of the stored
                                         # activation); False = 1 - 2/(1+exp(2x)) through ex2/rcp (abs. err ~1e-7)
    use_graph: bool = True               # replay one CUDA graph per update
    dw_splits: int = 0                   # 0 = auto
    fused: bool = True                   # fused forward+loss+backward kernel when num_layers == 2 and hidden_size <= 256
                                         # (wider layers always run layer-wise); False = layer-wise kernels


@dataclass
class Config:
    model: ModelConfig = field(default_factory=ModelConfig)
    opt: OptimizerConfig = field(default_factory=OptimizerConfig)
    rl: ReinforcementLearningConfig = field(default_factory=ReinforcementLearningConfig)
    training: TrainingConfig = field(default_factory=TrainingConfig)
    learner: LearnerExtras = field(default_factory=LearnerExtras)


def _coerce(old: Any, text: str) -> Any:
    if isinstance(old, bool):
        if text.lower() in ("true", "1", "yes"):
            return True
        if text.lower() in ("false", "0", "no"):
            return False
        raise ValueError(f"not a bool: {text!r}")
    if isinstance(old, int):
        return int(float(text)) if ("e" in text.lower() or "." in text) else int(text.replace("_", ""))
    if isinstance(old, float):
        return float(text)
    return text


def apply_overrides(cfg: Config, overrides: Sequence[str]) -> Config:
    """``key.sub=value`` dot-list overrides (what OmegaConf.from_dotlist does at config.py:122-123)."""
    for item in overrides:
        if "=" not in item:
            raise ValueError(f"override {item!r} is not of the form key=value")
        key, text = item.split("=", 1)
        node: Any = cfg
        parts = key.split(".")
        for p in parts[:-1]:
            if not dataclasses.is_dataclass(node) or not hasattr(node, p):
                raise KeyError(f"Key {key!r} is not in the structured config (unknown node {p!r})")
            node = getattr(node, p)
        leaf = parts[-1]
        if not dataclasses.is_dataclass(node) or not hasattr(node, leaf):
            raise KeyError(f"Key {key!r} is not in the structured config")
        setattr(node, leaf, _coerce(getattr(node, leaf), text))
    return cfg


def load_config(overrides: Sequence[str] = ()) -> Config:
    return apply_overrides(Config(), overrides)


def to_c_config(cfg: Config, obs_dim: int, act_dim: int, world_size: int = 1, rank: int = 0) -> "_lib.MinppoConfig":
    """Fill ``struct minppo_config``.  The reference uses rl.num_env_steps for the rollout
    length and training.num_steps for the minibatch arithmetic (train.py:179 vs 93-94); they
    must agree or the reference fails at trace time (SURVEY.md F6) -- same check here."""
    if cfg.rl.num_env_steps != cfg.training.num_steps:
        raise ValueError(
            f"rl.num_env_steps ({cfg.rl.num_env_steps}) != training.num_steps ({cfg.training.num_steps}): "
            "the reference reshapes [num_env_steps, N] to num_steps * num_envs (train.py:260) and fails; set both")
    mode = {"legacy": _lib.PRNG_LEGACY, "partitionable": _lib.PRNG_PARTITIONABLE}[cfg.learner.prng_mode]
    c = _lib.MinppoConfig()
    c.num_envs, c.num_steps = cfg.training.num_envs, cfg.training.num_steps
    c.num_minibatches, c.update_epochs = cfg.training.num_minibatches, cfg.training.update_epochs
    c.total_timesteps = int(cfg.training.total_timesteps)
    c.anneal_lr = int(cfg.training.anneal_lr)
    c.hidden_size, c.num_layers, c.use_tanh = cfg.model.hidden_size, cfg.model.num_layers, int(cfg.model.use_tanh)
    c.obs_dim, c.act_dim, c.prng_mode = obs_dim, act_dim, mode
    c.world_size, c.rank = world_size, rank
    c.fast_tanh, c.dw_splits = int(cfg.learner.fast_tanh), cfg.learner.dw_splits
    c.disable_fused = int(not cfg.learner.fused)
    c.training_lr, c.opt_lr, c.max_grad_norm = cfg.training.lr, cfg.opt.lr, cfg.opt.max_grad_norm
    c.gamma, c.gae_lambda, c.clip_eps = cfg.rl.gamma, cfg.rl.gae_lambda, cfg.rl.clip_eps
    c.ent_coef, c.vf_coef = cfg.rl.ent_coef, cfg.rl.vf_coef
    c.adam_b1, c.adam_b2, c.adam_eps, c.adam_eps_root = 0.9, 0.999, 1e-5, 0.0      # optax.adam(eps=1e-5), train.py:118
    return c
