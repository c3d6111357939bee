"""Running per-feature observation normalization (include/minppo_b200.h, ``minppo_obs_norm``).

``ObsNormalizer`` holds the running statistics as caller-owned device tensors, like ``TrainState``: ``mean`` f32 [D],
``var`` f32 [D] (population variance) and ``count`` f64 [1], plus the host scalars ``eps`` and ``clip``.  Passing it to
``Learner.policy_step`` / ``bootstrap_value`` evaluates the networks on

    y = clamp((x - mean) * (1 / sqrt(var + eps)), -clip, clip)        (fp32; clip <= 0: no clamp)

and leaves the statistics alone; passing it to ``Learner.update`` normalizes the trajectory with the same (entry)
statistics, which the rollout used, and then folds the update's global batch into them in place.  ``fold(obs)`` folds a
batch without an update (warming up from a random-policy rollout).  Nothing synchronises.
"""
from __future__ import annotations

import ctypes as C
import dataclasses

import numpy as np
import torch

from . import _lib


@dataclasses.dataclass
class ObsNormalizer:
    mean: torch.Tensor       # f32 [D]
    var: torch.Tensor        # f32 [D]
    count: torch.Tensor      # f64 [1]
    eps: float = 1e-8
    clip: float = 10.0       # <= 0: no clip

    @staticmethod
    def create(obs_dim: int, device, eps: float = 1e-8, clip: float = 10.0) -> "ObsNormalizer":
        """The initial state: mean = 0, var = 1, count = 0."""
        device = torch.device(device)
        return ObsNormalizer(torch.zeros(obs_dim, dtype=torch.float32, device=device),
                             torch.ones(obs_dim, dtype=torch.float32, device=device),
                             torch.zeros(1, dtype=torch.float64, device=device), float(eps), float(clip))

    @property
    def obs_dim(self) -> int:
        return int(self.mean.shape[0])

    def check(self, obs_dim: int, device: torch.device) -> None:
        """dtype, shape, device and contiguity of the three tensors (as ``Learner`` checks its inputs)."""
        for name, t, dtype, shape in (("mean", self.mean, torch.float32, (obs_dim,)),
                                      ("var", self.var, torch.float32, (obs_dim,)),
                                      ("count", self.count, torch.float64, (1,))):
            if t.dtype != dtype:
                raise TypeError(f"obs_norm.{name}: expected {dtype}, got {t.dtype}")
            if tuple(t.shape) != shape:
                raise ValueError(f"obs_norm.{name}: expected shape {shape}, got {tuple(t.shape)}")
            if t.device != device:
                raise ValueError(f"obs_norm.{name}: expected device {device}, got {t.device}")
            if not t.is_contiguous():
                raise ValueError(f"obs_norm.{name}: must be contiguous")

    def c_struct(self) -> _lib.MinppoObsNorm:
        return _lib.MinppoObsNorm(self.mean.data_ptr(), self.var.data_ptr(), self.count.data_ptr(), float(self.eps),
                                  float(self.clip))

    def fold(self, obs: torch.Tensor) -> None:
        """Fold observations f32 [..., D] (any leading shape, contiguous, on the statistics' device) into the
        statistics, exactly as an update over the same rows on one process does."""
        dev = self.mean.device
        D = self.obs_dim
        self.check(D, dev)
        if obs.dtype != torch.float32 or obs.device != dev or not obs.is_contiguous() or obs.dim() < 1 \
                or obs.shape[-1] != D:
            raise ValueError(f"obs must be a contiguous f32 [..., {D}] tensor on {dev}")
        rows = obs.numel() // D
        s = self.c_struct()
        with torch.cuda.device(dev):
            _lib.check(_lib.load().minppo_obs_norm_fold(obs.data_ptr(), rows, D, C.byref(s),
                                                        torch.cuda.current_stream(dev).cuda_stream))

    def to_tree(self) -> dict:
        """Host copy for a checkpoint (``params.save_model(..., obs_normalizer=...)``); synchronises."""
        return {"mean": self.mean.cpu().numpy(), "var": self.var.cpu().numpy(),
                "count": np.float64(self.count.item()), "eps": float(self.eps), "clip": float(self.clip)}

    @staticmethod
    def from_tree(tree: dict, device) -> "ObsNormalizer":
        device = torch.device(device)
        mean = np.ascontiguousarray(tree["mean"], np.float32).reshape(-1)
        var = np.ascontiguousarray(tree["var"], np.float32).reshape(-1)
        if mean.shape != var.shape:
            raise ValueError(f"obs_normalizer: mean {mean.shape} and var {var.shape} differ in shape")
        count = np.asarray(tree["count"], np.float64).reshape(1)
        return ObsNormalizer(torch.as_tensor(mean).to(device), torch.as_tensor(var).to(device),
                             torch.as_tensor(count).to(device), float(tree["eps"]), float(tree["clip"]))
