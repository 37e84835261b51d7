"""Rollout producer and the wrapper base class of the drop-in boundary.

`RunnerWrapper` keeps the reference's proxying contract (derl/runners/env_runner.py:72-90):
only {env, policy, horizon, nsteps, step_count, nenvs, is_exhausted} are forwarded, `run`
is an abstract generator, `__len__` forwards, `unwrapped` is the innermost runner.
`EnvRunner` (env_runner.py:6-69) is host Python around CPU simulators — out of the
accelerated scope — and is provided so `make_ppo_runner` stays a drop-in.
"""
from abc import ABC, abstractmethod

import numpy as np
import torch

from .frame_stacks import DeviceFrameStackPacker, FrameStackRollout

_FORWARDED = frozenset(("env", "policy", "horizon", "nsteps", "step_count", "nenvs",
                        "is_exhausted"))


class _ResidentRollout:
  """Preallocated [horizon, ...] tensors on `device`, filled one step at a time
  (SURVEY.md §8f rank 3): the rollout is born in HBM instead of being stacked from T host
  lists (`np.asarray`, derl/runners/onpolicy.py:20-27) and uploaded afterwards.

  On a CUDA device every column has a PINNED host mirror of the same shape: a step's value is
  written into its mirror row (a host memcpy) and that row is handed to an asynchronous H2D copy —
  a copy from pageable memory would block the host for every step.  A mirror row is rewritten
  one rollout later at the earliest; `begin()` waits for the previous rollout's copies first."""

  def __init__(self, horizon, device):
    self.horizon, self.device = horizon, torch.device(device)
    self.buffers, self.mirrors = {}, {}
    self.pinned = self.device.type == "cuda"
    self.drained = None

  def begin(self):
    """Fresh device tensors for a new rollout (the previous ones now belong to the consumer)."""
    if self.drained is not None:
      self.drained.synchronize()
      self.drained = None
    self.buffers = {}

  def put(self, key, step, value):
    arr = np.asarray(value)
    if arr.dtype == object or arr.dtype.kind in "USV":
      return False
    host = torch.from_numpy(np.ascontiguousarray(arr))
    buf = self.buffers.get(key)
    if buf is None or buf.shape[1:] != host.shape or buf.dtype != host.dtype:
      buf = self.buffers[key] = torch.empty((self.horizon,) + tuple(host.shape), dtype=host.dtype,
                                            device=self.device)
    if not self.pinned:
      buf[step].copy_(host)
      return True
    mirror = self.mirrors.get(key)
    if mirror is None or mirror.shape != buf.shape or mirror.dtype != buf.dtype:
      mirror = self.mirrors[key] = torch.empty(buf.shape, dtype=buf.dtype, pin_memory=True)
    mirror[step].copy_(host)
    buf[step].copy_(mirror[step], non_blocking=True)
    return True

  def end(self):
    if self.pinned:
      self.drained = torch.cuda.Event()
      self.drained.record(torch.cuda.current_stream(self.device))


class EnvRunner:
  """Steps `env` with `policy` for `horizon` steps per yielded rollout.

  `resident_device` (extension, default None = reference behaviour): write every numeric
  per-step value straight into preallocated device tensors; `next_observations` is then not
  collected (nothing on the PPO path reads it) and `infos` stays a host list.  In that mode the
  rollout also carries `state["latest_values"]`: the critic's value of the final observation,
  taken from the forward pass this runner makes on it right after the last step (the same batch
  a GAE bootstrap would evaluate, derl/runners/trajectory_transforms.py:47-50) and kept on the
  device, so `derl_b200.GAE` does not run a second forward or a host round trip for it.

  `pack_frames` (extension, default False): `observations` is yielded as a
  `runners.frame_stacks.FrameStacks` — every frame plane stored once plus a per-sample stack
  index, packed one step at a time — instead of stacked arrays: about a quarter of the bytes for
  4-frame Atari stacks.  Without `resident_device` the host packs (FrameStackPacker) and the
  planes stay in pinned host memory (TransformInteractions uploads them).  With it each step's
  stacks are copied to the device and packed there (DeviceFrameStackPacker, kernel K11): planes
  and index are born in HBM, and the host does no more per step than the stacked resident route.
  `state["latest_observations"]` stays stacked in both modes.
  """

  def __init__(self, env, policy, horizon, nsteps=None, time_limit=None, resident_device=None,
               pack_frames=False):
    self.resident_device = resident_device
    self.pack_frames = pack_frames
    self.env, self.policy, self.horizon = env, policy, horizon
    self.nsteps = int(nsteps)
    if time_limit is not None and getattr(env.unwrapped, "nenvs", None) is not None:
      raise TypeError("batched envs are not supported for time_limit "
                      f"not equal to None, got env={env}, time_limit={time_limit}")
    self.time_limit = time_limit
    self.step_count = 0
    self.episode_length = 0
    self._resident = None
    self._frame_packer = None

  @property
  def nenvs(self):
    return getattr(self.env.unwrapped, "nenvs", None)

  def is_exhausted(self):
    return self.nsteps is not None and self.step_count >= self.nsteps

  def __len__(self):
    return self.nsteps if self.nsteps is not None else self.step_count

  def run(self, obs=None):
    if obs is None:
      obs = self.env.reset()
      self.episode_length = 0
    while not self.is_exhausted():
      rollout = {}
      resident = None
      if self.resident_device is not None:
        if self._resident is None:
          self._resident = _ResidentRollout(self.horizon, self.resident_device)
        resident = self._resident
        resident.begin()
      frames = None
      if self.pack_frames:
        if self.resident_device is not None and self._frame_packer is None:
          self._frame_packer = DeviceFrameStackPacker(self.resident_device, self.horizon)
        frames = FrameStackRollout(self.horizon, self.resident_device, self._frame_packer)

      def put(key, val, step):
        if resident is not None and key == "next_observations":
          return
        if frames is not None and key == "observations":
          rollout.setdefault(key, None)   # keeps the reference's key order
          frames.put(step, val)
          return
        if resident is not None and resident.put(key, step, val):
          rollout[key] = resident.buffers[key]
        else:
          rollout.setdefault(key, []).append(val)

      for step in range(self.horizon):
        act = self.policy.act(obs)
        put("observations", obs, step)
        if "actions" not in act:
          raise ValueError("result of policy.act must contain 'actions' "
                           f"but has keys {list(act.keys())}")
        for key, val in act.items():
          put(key, val, step)
        next_obs, reward, done, info = self.env.step(act["actions"])
        self.episode_length += 1
        put("rewards", reward, step)
        put("resets", done, step)
        put("infos", info, step)
        put("next_observations", next_obs, step)
        # batched envs auto-reset; a single env is reset here (env_runner.py:58-65)
        if self.nenvs is None and (done or self.episode_length == self.time_limit):
          obs = self.env.reset()
          self.episode_length = 0
        else:
          obs = next_obs
      if frames is not None:
        rollout["observations"] = frames.finish()
      rollout["state"] = dict(latest_observations=obs)
      if resident is not None:
        resident.end()
        values = self.policy.act(obs).get("values")
        if values is not None:
          rollout["state"]["latest_values"] = torch.as_tensor(np.asarray(values)).to(
              resident.device)
      self.step_count += self.horizon * (self.nenvs or 1)
      yield rollout


class RunnerWrapper(ABC):
  """Base of TransformInteractions / IterateWithMinibatches."""

  def __init__(self, runner):
    self.runner = runner
    self.unwrapped = getattr(runner, "unwrapped", runner)

  def __getattr__(self, attr):
    if attr not in _FORWARDED:
      raise AttributeError(f"'{self.__class__.__name__}' has no attribute '{attr}'")
    return getattr(self.runner, attr)

  def __len__(self):
    return len(self.runner)

  @abstractmethod
  def run(self, obs=None):
    """Generator of interaction dicts."""
