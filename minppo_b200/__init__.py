"""minppo_b200 -- B200-native (sm_100a) PPO learner for the hot path of kscalelabs/minppo
(/root/reference/minppo/train.py:181-281): GAE, PRNG-derived minibatch shuffle/gather,
ActorCritic forward/backward + PPO loss, global-norm clip + Adam.

Public surface:
  minppo_b200.config   -- mirror of the rl.* / training.* / opt.* / model.* config keys
  minppo_b200.params   -- checkpoint pickle layout <-> flat fp32 arena
  minppo_b200.learner  -- Learner.update (the seam of _update_step), Learner.policy_step, calculate_gae, permutations
  minppo_b200.obs_norm -- ObsNormalizer: running observation statistics for the update, the policy step and checkpoints
  minppo_b200.infer    -- InferencePolicy: checkpoint pickle -> deterministic / sampled actions (infer.py:17-27)
  minppo_b200._lib     -- ctypes binding of the C ABI (include/minppo_b200.h)
"""
__version__ = "0.1.0"

from . import config, params  # noqa: F401  (pure Python; importing them never needs the .so)


def __getattr__(name):
    # learner pulls in torch; import lazily so that `import minppo_b200` stays light
    if name in ("learner", "Learner", "Memory", "TrainState", "HostBatch", "HostPipeline", "calculate_gae", "permutations"):
        import importlib

        mod = importlib.import_module(".learner", __name__)
        return mod if name == "learner" else getattr(mod, name)
    if name in ("obs_norm", "ObsNormalizer"):
        import importlib

        mod = importlib.import_module(".obs_norm", __name__)
        return mod if name == "obs_norm" else mod.ObsNormalizer
    raise AttributeError(name)
