"""Policy inference from a checkpoint: the loader the reference has (/root/reference/minppo/infer.py:17-19) plus the
forward pass its `main` never got (infer.py:27 raises NotImplementedError).

The checkpoint is the reference's pickle of the flax variable dict (train.py:86-89); it is flattened into the fp32 arena
(minppo_b200.params) and evaluated by minppo_policy_step -- the same tensor-core forward pass the rollout uses
(train.py:157-160).  `act(obs)` returns the mode of pi (deterministic evaluation); with an rng it samples like the rollout.
A checkpoint with an "obs_normalizer" entry (minppo_b200.params) is evaluated on observations normalized with the stored
statistics, as during training; without it the observations are used as they are.
"""
from __future__ import annotations

import copy
from typing import Optional

import numpy as np
import torch

from .config import Config
from .learner import Learner
from .obs_norm import ObsNormalizer
from .params import OBS_NORMALIZER_KEY, flatten_params, leaf_shapes, load_model


class InferencePolicy:
    def __init__(self, params_tree: dict, config: Config, num_envs: int, device: Optional[torch.device] = None):
        kernel0 = np.asarray(params_tree["params"]["MLP_0"]["Dense_0"]["kernel"])
        log_std = np.asarray(params_tree["params"]["log_std"])
        self.obs_dim, self.act_dim = int(kernel0.shape[0]), int(log_std.shape[0])
        L, H = config.model.num_layers, config.model.hidden_size
        want = leaf_shapes(self.obs_dim, self.act_dim, H, L)
        flat = flatten_params(params_tree, L)
        if flat.size != sum(int(np.prod(s)) for s in want):
            raise ValueError("checkpoint does not match model.hidden_size / model.num_layers of the config")
        # the context is shaped by (num_envs, num_steps, num_minibatches): inference only needs a consistent triple
        cfg = copy.deepcopy(config)
        cfg.training.num_envs = num_envs
        cfg.rl.num_env_steps = cfg.training.num_steps = 1
        cfg.training.num_minibatches = 1
        self._learner = Learner(cfg, self.obs_dim, self.act_dim, device)
        self.device = self._learner.device
        self.params = torch.as_tensor(flat).to(self.device)
        self.obs_norm = None
        if OBS_NORMALIZER_KEY in params_tree:
            self.obs_norm = ObsNormalizer.from_tree(params_tree[OBS_NORMALIZER_KEY], self.device)
            if self.obs_norm.obs_dim != self.obs_dim:
                raise ValueError(f"obs_normalizer has {self.obs_norm.obs_dim} features, the policy {self.obs_dim}")
        self._first = True

    @classmethod
    def from_checkpoint(cls, filename: str, config: Config, num_envs: int, device: Optional[torch.device] = None):
        return cls(load_model(filename), config, num_envs, device)

    def act(self, obs: torch.Tensor, rng: Optional[torch.Tensor] = None):
        """obs f32 [num_envs, obs_dim] on the policy's device.  rng None: (mode of pi, value); else
        (sampled action, log_prob, value, rng') exactly like one rollout step."""
        cur = not self._first
        self._first = False
        action, log_prob, value, rng_out, _ = self._learner.policy_step(self.params, obs, rng, weights_current=cur,
                                                                        obs_norm=self.obs_norm)
        if rng is None:
            return action, value
        return action, log_prob, value, rng_out

    def close(self) -> None:
        self._learner.close()
