"""Host-side mirror of the reference's learner seam, over the C ABI.

The reference has no operator / plugin interface for this path: the seam is the span of
``_update_step`` between the rollout scan and the rebuilt ``RunnerState``
(/root/reference/minppo/train.py:181-281).  Its logical signature (SURVEY.md section 8b) is

    learner_update(params, opt_state{count, mu, nu}, traj{obs, action, value, reward,
                   log_prob, done}, last_val, rng) -> (params', opt_state', rng', losses[E, M, 4])

``Learner.update`` is that function: same names (``Memory``, ``TrainState``-like state,
``rng``), same time-major ``[T, N, ...]`` layout as ``jax.lax.scan`` stacks it, same error
for a batch that does not divide into minibatches (train.py:253-255).  torch is used only for
device memory, streams and ``torch.distributed`` plumbing; all arithmetic happens in
libminppo_b200.so (sm_100a kernels).  There is no CPU path.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
import os
from typing import Any, NamedTuple, Optional

import numpy as np
import torch

from . import _lib
from .config import Config, to_c_config
from .params import leaf_paths, leaf_shapes, param_count


class Memory(NamedTuple):
    """Same fields, order and layout as train.py:26-33 (time-major [T, N, ...])."""
    done: torch.Tensor       # bool / uint8 [T, N]
    action: torch.Tensor     # f32 [T, N, A]
    value: torch.Tensor      # f32 [T, N]
    reward: torch.Tensor     # f32 [T, N]
    log_prob: torch.Tensor   # f32 [T, N]
    obs: torch.Tensor        # f32 [T, N, D]
    info: Any = None         # EnvMetrics; unused by the loss, passed through (train.py:283)


@dataclasses.dataclass
class TrainState:
    """What flax's TrainState carries on this path (train.py:126-130): params, the Adam
    moments and the step count, as flat fp32 arenas on the device."""
    params: torch.Tensor     # f32 [P]
    mu: torch.Tensor         # f32 [P]
    nu: torch.Tensor         # f32 [P]
    step: torch.Tensor       # i32 [1]  == ScaleByAdamState.count

    @staticmethod
    def create(flat_params: np.ndarray, device: torch.device) -> "TrainState":
        p = torch.as_tensor(np.ascontiguousarray(flat_params, np.float32)).to(device)
        return TrainState(p, torch.zeros_like(p), torch.zeros_like(p), torch.zeros(1, dtype=torch.int32, device=device))


# columns of the per-minibatch statistics ``Learner.update(..., stats=...)`` writes (include/minppo_b200.h)
STATS_COLUMNS = ("approx_kl", "clip_fraction", "value_clip_fraction", "grad_norm")


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _as_u8(done: torch.Tensor) -> torch.Tensor:
    if done.dtype == torch.bool:
        return done.view(torch.uint8)          # zero-copy: bool is one byte
    if done.dtype != torch.uint8:
        raise TypeError(f"done must be bool or uint8, got {done.dtype}")
    return done


def _check(t: torch.Tensor, name: str, dtype: torch.dtype, shape, device: torch.device) -> torch.Tensor:
    if t.dtype != dtype:
        raise TypeError(f"{name}: expected {dtype}, got {t.dtype}")
    if tuple(t.shape) != tuple(shape):
        raise ValueError(f"{name}: expected shape {tuple(shape)}, got {tuple(t.shape)}")
    if t.device != device:
        raise ValueError(f"{name}: expected device {device}, got {t.device}")
    if not t.is_contiguous():
        raise ValueError(f"{name}: must be contiguous (time-major [T, N, ...])")
    return t


# ------------------------------------------------------------------------------------------
# stateless entry points
# ------------------------------------------------------------------------------------------
def calculate_gae(mem_batch: Memory, last_val: torch.Tensor, gamma: float, gae_lambda: float,
                  chunks: int = 0):
    """``_calculate_gae(mem_batch, last_val) -> (advantages, targets)`` (train.py:185-207)."""
    lib = _lib.load()
    dev = mem_batch.reward.device
    if dev.type != "cuda":
        raise ValueError("calculate_gae needs CUDA tensors; there is no CPU path")
    T, N = mem_batch.reward.shape
    reward = _check(mem_batch.reward, "reward", torch.float32, (T, N), dev)
    value = _check(mem_batch.value, "value", torch.float32, (T, N), dev)
    done = _check(_as_u8(mem_batch.done), "done", torch.uint8, (T, N), dev)
    last_val = _check(last_val, "last_val", torch.float32, (N,), dev)
    adv = torch.empty_like(reward)
    tgt = torch.empty_like(reward)
    with torch.cuda.device(dev):
        _lib.check(lib.minppo_gae_chunked(_ptr(reward), _ptr(value), _ptr(done), _ptr(last_val), _ptr(adv), _ptr(tgt),
                                          T, N, gamma, gae_lambda, chunks, _stream_ptr(dev)))
    return adv, tgt


def permutations(rng: torch.Tensor, batch_size: int, epochs: int, prng_mode: int = _lib.PRNG_LEGACY):
    """The ``epochs`` successive ``rng, _rng = split(rng); permutation(_rng, batch_size)`` of one
    update (train.py:252, 258).  rng: uint32-as-int32/uint32 [2] CUDA tensor.
    Returns (rng_out [2], perms int32 [epochs, batch_size])."""
    lib = _lib.load()
    dev = rng.device
    if dev.type != "cuda":
        raise ValueError("permutations needs CUDA tensors; there is no CPU path")
    if rng.numel() != 2 or rng.element_size() != 4:
        raise ValueError("rng must hold two 32-bit words")
    perms = torch.empty((epochs, batch_size), dtype=torch.int32, device=dev)
    rng_out = torch.empty_like(rng)
    ws_bytes = lib.minppo_permutation_workspace_size(epochs, batch_size)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.minppo_permutation(_ptr(rng), _ptr(rng_out), prng_mode, epochs, batch_size, _ptr(perms),
                                          _ptr(ws), ws_bytes, _stream_ptr(dev)))
    return rng_out, perms


def nccl_unique_id() -> bytes:
    buf = C.create_string_buffer(128)
    _lib.check(_lib.load().minppo_nccl_unique_id(buf))
    return buf.raw


# ------------------------------------------------------------------------------------------
# the learner
# ------------------------------------------------------------------------------------------
class Learner:
    """One context per (device, shape).  ``world_size > 1``: env-sharded data parallelism --
    this rank's trajectory holds envs [rank*N/G, (rank+1)*N/G) of the GLOBAL batch, every rank
    computes the global permutation, gradients are all-reduced per minibatch (SURVEY.md 8e)."""

    def __init__(self, config: Config, obs_dim: int, act_dim: int, device: Optional[torch.device] = None,
                 world_size: int = 1, rank: int = 0, nccl_id: Optional[bytes] = None):
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise RuntimeError("minppo_b200.Learner needs a CUDA (sm_100a) device; there is no CPU fallback")
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.config = config
        self.obs_dim, self.act_dim = obs_dim, act_dim
        self.world_size, self.rank = world_size, rank
        self.cconf = to_c_config(config, obs_dim, act_dim, world_size, rank)
        t = config.training
        self.T, self.N = t.num_steps, t.num_envs
        self.Nl = self.N // world_size
        self.E, self.M = t.update_epochs, t.num_minibatches
        self.P = param_count(obs_dim, act_dim, config.model.hidden_size, config.model.num_layers)
        batch = self.T * self.N
        if (batch // self.M) * self.M != batch:
            raise ValueError("`batch_size` must be equal to `num_steps * num_envs`")      # train.py:254-255
        handle = C.c_void_p()
        idbuf = C.create_string_buffer(nccl_id, 128) if nccl_id is not None else None
        with torch.cuda.device(self.device):
            _lib.check(self.lib.minppo_ctx_create(C.byref(self.cconf), idbuf, C.byref(handle)))
        self._h = handle
        self.use_graph = bool(config.learner.use_graph)
        # Persistent device slots for the rng key and the losses: the library caches one CUDA graph per POINTER SET, so the
        # natural loop `ts, rng, losses = learner.update(ts, mem, last_val, rng)` must present the same pointers every call.
        self._key_in = torch.zeros(2, dtype=torch.int32, device=self.device)
        self._key_out = torch.zeros(2, dtype=torch.int32, device=self.device)
        self._losses = torch.zeros((self.E, self.M, 4), dtype=torch.float32, device=self.device)
        self.peer_exchange = False
        if world_size > 1 and os.environ.get("MINPPO_NCCL_ALLREDUCE", "0") != "1":
            self._connect_peers()

    def _connect_peers(self) -> None:
        """Exchange the CUDA-IPC handles of the gradient exchange buffers through torch.distributed (plumbing
        only) and switch the per-minibatch all-reduce to the fused peer-memory path (include/minppo_b200.h).
        Without an initialised process group the context stays on ncclAllReduce."""
        import torch.distributed as dist

        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() != self.world_size:
            return
        buf = C.create_string_buffer(64)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.minppo_ctx_ipc_handle(self._h, buf))
            handles = [None] * self.world_size
            dist.all_gather_object(handles, buf.raw)
            table = C.create_string_buffer(b"".join(handles), 64 * self.world_size)
            _lib.check(self.lib.minppo_ctx_set_peers(self._h, table))
        dist.barrier()                       # every rank has mapped every buffer before the first update
        self.peer_exchange = True

    def close(self) -> None:
        if getattr(self, "_h", None):
            self.lib.minppo_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- layout ---------------------------------------------------------------------------
    def param_layout(self):
        n = C.c_int32()
        offs = (C.c_int64 * _lib.MAX_LEAVES)()
        rows = (C.c_int64 * _lib.MAX_LEAVES)()
        cols = (C.c_int64 * _lib.MAX_LEAVES)()
        P = self.lib.minppo_param_layout(C.byref(self.cconf), C.byref(n), offs, rows, cols)
        paths = leaf_paths(self.config.model.num_layers)
        return P, [(paths[i], offs[i], rows[i], cols[i]) for i in range(n.value)]

    # -- the update -----------------------------------------------------------------------
    def update(self, train_state: TrainState, mem_batch: Memory, last_val: torch.Tensor, rng: torch.Tensor,
               losses: Optional[torch.Tensor] = None, rng_out: Optional[torch.Tensor] = None,
               stats: Optional[torch.Tensor] = None):
        """train.py:185-281.  In place on ``train_state``; returns (train_state, rng', losses[E, M, 4])
        with losses columns (total, value_loss, actor_loss, entropy).  Nothing synchronises.

        ``stats``: optional caller-owned f32 [E, M, 4] device tensor, filled in place with per-minibatch diagnostics,
        columns ``STATS_COLUMNS``: approx_kl = mean(expm1(log r) - log r), clip_fraction = mean(|r - 1| > clip_eps),
        value_clip_fraction = mean(|v - v_old| > clip_eps) over the rows of the global minibatch, evaluated with the
        parameters before that minibatch's Adam step, and the pre-clip global gradient norm.  Passing it changes
        nothing else the update computes.

        ``rng`` is copied (8 bytes, stream-ordered) into a learner-owned slot; without ``losses`` / ``rng_out`` the
        results land in learner-owned buffers that the NEXT ``update`` overwrites (pass your own to keep them).  With
        the trajectory / train-state tensors reused across calls the pointer set is stable and every update is one CUDA
        graph replay; the library keeps the 4 most recently used pointer sets."""
        dev = self.device
        T, Nl, D, A = self.T, self.Nl, self.obs_dim, self.act_dim
        obs = _check(mem_batch.obs, "obs", torch.float32, (T, Nl, D), dev)
        action = _check(mem_batch.action, "action", torch.float32, (T, Nl, A), dev)
        value = _check(mem_batch.value, "value", torch.float32, (T, Nl), dev)
        reward = _check(mem_batch.reward, "reward", torch.float32, (T, Nl), dev)
        log_prob = _check(mem_batch.log_prob, "log_prob", torch.float32, (T, Nl), dev)
        done = _check(_as_u8(mem_batch.done), "done", torch.uint8, (T, Nl), dev)
        last_val = _check(last_val, "last_val", torch.float32, (Nl,), dev)
        _check(train_state.params, "params", torch.float32, (self.P,), dev)
        _check(train_state.mu, "mu", torch.float32, (self.P,), dev)
        _check(train_state.nu, "nu", torch.float32, (self.P,), dev)
        _check(train_state.step, "step", torch.int32, (1,), dev)
        if rng.numel() != 2 or rng.element_size() != 4 or rng.device != dev:
            raise ValueError("rng must hold two 32-bit words on the learner's device")
        if losses is None:
            losses = self._losses
        else:
            _check(losses, "losses", torch.float32, (self.E, self.M, 4), dev)
        if stats is not None:
            _check(stats, "stats", torch.float32, (self.E, self.M, len(STATS_COLUMNS)), dev)
        if rng_out is None:
            rng_out = self._key_out.view(rng.dtype)
        with torch.cuda.device(dev):
            if rng.data_ptr() != self._key_in.data_ptr():
                self._key_in.copy_(rng.reshape(2).view(torch.int32), non_blocking=True)
            _lib.check(self.lib.minppo_update_with_stats(
                self._h, _ptr(train_state.params), _ptr(train_state.mu), _ptr(train_state.nu), _ptr(train_state.step),
                _ptr(obs), _ptr(action), _ptr(value), _ptr(reward), _ptr(log_prob), _ptr(done), _ptr(last_val),
                _ptr(self._key_in), _ptr(rng_out), _ptr(losses), _ptr(stats), int(self.use_graph), _stream_ptr(dev)))
        return train_state, rng_out, losses

    # -- policy / value inference for the rollout -------------------------------------------
    def policy_step(self, params: torch.Tensor, last_obs: torch.Tensor, rng: Optional[torch.Tensor],
                    weights_current: bool = False, want_mean: bool = False):
        """train.py:157-160: ``pi, value = network.apply(params, last_obs); rng, action_rng = split(rng);
        action = pi.sample(seed=action_rng); log_prob = pi.log_prob(action)`` on this rank's ``Nl`` envs.
        Returns (action [Nl, A], log_prob [Nl], value [Nl], rng', mean or None).  ``rng=None``: no sampling
        (action = the mode of pi, rng' = None).  Nothing synchronises."""
        dev = self.device
        obs = _check(last_obs, "last_obs", torch.float32, (self.Nl, self.obs_dim), dev)
        _check(params, "params", torch.float32, (self.P,), dev)
        if rng is not None and (rng.numel() != 2 or rng.element_size() != 4 or rng.device != dev):
            raise ValueError("rng must hold two 32-bit words on the learner's device")
        action = torch.empty((self.Nl, self.act_dim), dtype=torch.float32, device=dev)
        log_prob = torch.empty((self.Nl,), dtype=torch.float32, device=dev)
        value = torch.empty((self.Nl,), dtype=torch.float32, device=dev)
        mean = torch.empty_like(action) if want_mean else None
        rng_out = torch.empty_like(rng) if rng is not None else None
        with torch.cuda.device(dev):
            _lib.check(self.lib.minppo_policy_step(
                self._h, _ptr(params), _ptr(obs), _ptr(rng), _ptr(rng_out), _ptr(action), _ptr(log_prob), _ptr(value),
                _ptr(mean), _lib.POLICY_WEIGHTS_CURRENT if weights_current else 0, _stream_ptr(dev)))
        return action, log_prob, value, rng_out, mean

    def bootstrap_value(self, params: torch.Tensor, last_obs: torch.Tensor, weights_current: bool = False) -> torch.Tensor:
        """train.py:182-183: ``_, last_val = network.apply(params, last_obs)`` (critic only)."""
        dev = self.device
        obs = _check(last_obs, "last_obs", torch.float32, (self.Nl, self.obs_dim), dev)
        _check(params, "params", torch.float32, (self.P,), dev)
        value = torch.empty((self.Nl,), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            _lib.check(self.lib.minppo_policy_step(
                self._h, _ptr(params), _ptr(obs), None, None, None, None, _ptr(value), None,
                _lib.POLICY_WEIGHTS_CURRENT if weights_current else 0, _stream_ptr(dev)))
        return value

    def check(self) -> None:
        """Synchronise and raise if the device-side error flag is set, a row list overflowed
        or a gradient norm is not finite (the reference has no such guard; SURVEY.md section 5)."""
        with torch.cuda.device(self.device):
            _lib.check(self.lib.minppo_ctx_check(self._h, _stream_ptr(self.device)))

    def launches_per_update(self) -> int:
        return int(self.lib.minppo_update_launch_count(self._h))

    # -- introspection (tests) --------------------------------------------------------------
    _WHAT = {"advantages": 0, "targets": 1, "perms": 2, "grad": 3, "grad_norms": 4, "counts": 5, "adv_stats": 6}

    def read(self, what: str) -> torch.Tensor:
        EM, B, Bl = self.E * self.M, self.T * self.N, self.T * self.Nl
        spec = {
            "advantages": ((self.T, self.Nl), torch.float32), "targets": ((self.T, self.Nl), torch.float32),
            "perms": ((self.E, B), torch.int32), "grad": ((self.P + 4,), torch.float32),
            "grad_norms": ((EM,), torch.float32), "counts": ((EM,), torch.int32),
            "adv_stats": ((2, EM), torch.float32),
        }[what]
        out = torch.empty(spec[0], dtype=spec[1], device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.minppo_ctx_read(self._h, self._WHAT[what], _ptr(out), out.numel() * out.element_size(),
                                                _stream_ptr(self.device)))
        return out

    # -- host-buffer entry point (what bench.py's e2e number times) -------------------------
    def update_host(self, host: "HostBatch") -> np.ndarray:
        """Full round trip with HOST buffers: pinned H2D copies of the trajectory, params and
        optimizer state, the update, and D2H of params / moments / step / rng / losses.  Blocks
        until the results are on the host.  Returns losses[E, M, 4] (a view of pinned memory)."""
        host.to_device(self.device)
        ts = TrainState(host.d["params"], host.d["mu"], host.d["nu"], host.d["step"])
        mem = Memory(host.d["done"], host.d["action"], host.d["value"], host.d["reward"], host.d["log_prob"],
                     host.d["obs"])
        self.update(ts, mem, host.d["last_val"], host.d["rng"], host.d["losses"], host.d["rng_out"])
        host.to_host()
        torch.cuda.current_stream(self.device).synchronize()
        return host.h["losses"].numpy()


class HostBatch:
    """Pinned host buffers + their device twins for ``Learner.update_host``."""
    IN = ("obs", "action", "value", "reward", "log_prob", "done", "last_val", "rng", "params", "mu", "nu", "step")
    OUT = ("params", "mu", "nu", "step", "rng_out", "losses")

    def __init__(self, learner: Learner):
        T, Nl, D, A, P = learner.T, learner.Nl, learner.obs_dim, learner.act_dim, learner.P
        f32, i32, u8 = torch.float32, torch.int32, torch.uint8
        spec = {
            "obs": ((T, Nl, D), f32), "action": ((T, Nl, A), f32), "value": ((T, Nl), f32), "reward": ((T, Nl), f32),
            "log_prob": ((T, Nl), f32), "done": ((T, Nl), u8), "last_val": ((Nl,), f32), "rng": ((2,), i32),
            "params": ((P,), f32), "mu": ((P,), f32), "nu": ((P,), f32), "step": ((1,), i32),
            "rng_out": ((2,), i32), "losses": ((learner.E, learner.M, 4), f32),
        }
        self.h = {k: torch.zeros(s, dtype=dt).pin_memory() for k, (s, dt) in spec.items()}
        self.d = {k: torch.empty(s, dtype=dt, device=learner.device) for k, (s, dt) in spec.items()}

    def h2d_bytes(self) -> int:
        return sum(self.h[k].numel() * self.h[k].element_size() for k in self.IN)

    def d2h_bytes(self) -> int:
        return sum(self.h[k].numel() * self.h[k].element_size() for k in self.OUT)

    def to_device(self, device) -> None:
        for k in self.IN:
            self.d[k].copy_(self.h[k], non_blocking=True)

    def to_host(self) -> None:
        for k in self.OUT:
            self.h[k].copy_(self.d[k], non_blocking=True)


class HostPipeline:
    """Streaming host entry point: trajectories arrive in pinned HOST memory (remote / CPU rollout workers), the train
    state lives on the device, and every update returns the new parameters and the losses to the host.

    ``submit(traj)`` enqueues, without blocking: the H2D copy of that update's trajectory (+ last_val) on a copy stream
    into one of two device buffer sets, the update on the compute stream (ordered after the copy by an event), and the
    D2H copies of params / rng / losses into pinned host memory.  ``result()`` blocks until the OLDEST outstanding update
    is on the host and returns (losses[E, M, 4], params[P]) views of pinned memory.  With two updates in flight the H2D
    copy of update i + 1 runs under the kernels of update i -- every update still pays for its own copies, they just no
    longer serialise with the compute (the reference keeps the trajectory on the device and has no such copy at all).
    Updates are strictly sequential on the device (update i + 1 starts from update i's parameters and rng)."""

    DEPTH = 2

    def __init__(self, learner: Learner, train_state: TrainState, rng: torch.Tensor):
        self.lrn = learner
        self.ts = train_state
        dev = learner.device
        T, Nl, D, A, P = learner.T, learner.Nl, learner.obs_dim, learner.act_dim, learner.P
        f32, u8 = torch.float32, torch.uint8
        self.spec = {"obs": ((T, Nl, D), f32), "action": ((T, Nl, A), f32), "value": ((T, Nl), f32), "reward": ((T, Nl), f32),
                     "log_prob": ((T, Nl), f32), "done": ((T, Nl), u8), "last_val": ((Nl,), f32)}
        self.dev_in = [{k: torch.empty(s, dtype=dt, device=dev) for k, (s, dt) in self.spec.items()} for _ in range(self.DEPTH)]
        self.dev_losses = [torch.empty((learner.E, learner.M, 4), dtype=f32, device=dev) for _ in range(self.DEPTH)]
        self.host_out = [{"losses": torch.empty((learner.E, learner.M, 4), dtype=f32).pin_memory(),
                          "params": torch.empty((P,), dtype=f32).pin_memory(),
                          "rng": torch.empty((2,), dtype=torch.int32).pin_memory()} for _ in range(self.DEPTH)]
        # the rng key chain lives on the device: ping-pong pair (update i reads slot i % 2, writes slot (i + 1) % 2)
        self.rng = [rng.reshape(2).view(torch.int32).clone(), torch.empty(2, dtype=torch.int32, device=dev)]
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.ev_copied = [torch.cuda.Event() for _ in range(self.DEPTH)]
        self.ev_done = [torch.cuda.Event() for _ in range(self.DEPTH)]       # update + D2H of slot k finished
        self.ev_free = [None] * self.DEPTH                                    # device inputs of slot k no longer read
        self.n_submitted = 0
        self.n_returned = 0

    def h2d_bytes(self) -> int:
        return sum(int(np.prod(s)) * torch.empty((), dtype=dt).element_size() for s, dt in self.spec.values())

    def d2h_bytes(self) -> int:
        return sum(t.numel() * t.element_size() for t in self.host_out[0].values())

    def submit(self, traj: dict) -> None:
        """``traj``: pinned host tensors obs, action, value, reward, log_prob, done (uint8 / bool), last_val."""
        if self.n_submitted - self.n_returned >= self.DEPTH:
            raise RuntimeError("HostPipeline: call result() before submitting a third update")
        k = self.n_submitted % self.DEPTH
        dev = self.lrn.device
        compute = torch.cuda.current_stream(dev)
        with torch.cuda.stream(self.copy_stream):
            if self.ev_free[k] is not None:
                self.copy_stream.wait_event(self.ev_free[k])          # the update that last read this buffer set is finished
            for name in self.spec:
                src = traj[name]
                if name == "done" and src.dtype == torch.bool:
                    src = src.view(torch.uint8)
                self.dev_in[k][name].copy_(src, non_blocking=True)
            self.ev_copied[k].record(self.copy_stream)
        compute.wait_event(self.ev_copied[k])
        d = self.dev_in[k]
        mem = Memory(d["done"], d["action"], d["value"], d["reward"], d["log_prob"], d["obs"])
        i = self.n_submitted
        self.lrn.update(self.ts, mem, d["last_val"], self.rng[i % 2], self.dev_losses[k], self.rng[(i + 1) % 2])
        ev = torch.cuda.Event()
        ev.record(compute)
        self.ev_free[k] = ev
        h = self.host_out[k]
        h["losses"].copy_(self.dev_losses[k], non_blocking=True)
        h["params"].copy_(self.ts.params, non_blocking=True)
        h["rng"].copy_(self.rng[(i + 1) % 2], non_blocking=True)
        self.ev_done[k].record(compute)
        self.n_submitted += 1

    def result(self):
        if self.n_returned >= self.n_submitted:
            raise RuntimeError("HostPipeline: nothing outstanding")
        k = self.n_returned % self.DEPTH
        self.ev_done[k].synchronize()
        self.n_returned += 1
        return self.host_out[k]["losses"].numpy(), self.host_out[k]["params"].numpy()
