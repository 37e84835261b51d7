"""Seeded synthetic rollout source with the attribute surface of the reference's EnvRunner
(derl/runners/env_runner.py:6-69; SURVEY.md §8b "Rollout source"), for benches and tests:
no simulator is involved, the arrays have exactly the dtypes/shapes EnvRunner + np.asarray
produce (§8a a1, §8d):

  atari   observations uint8 (T,N,84,84,4), actions int64 (T,N), log_prob f32 (T,N),
          values f32 (T,N,1), rewards {-1,0,1} (T,N), resets bool (T,N),
          state.latest_observations uint8 (N,84,84,4)
  mujoco  unbatched (nenvs=None): observations f64 (T,17), actions f32 (T,6), log_prob f32
          (T,), values f32 (T,1), rewards f64 (T,), resets bool (T,),
          state.latest_observations f64 (17,)

`device="cuda"` builds the rollout directly in HBM (torch generators); `device="cpu"`
returns NumPy arrays like the reference's runner does.  No `next_observations` / `infos`.
"""
import math
import types

import numpy as np
import torch


def _space(**kw):
  return types.SimpleNamespace(**kw)


class SyntheticEnv:
  """Just enough of an env for the wrappers: spaces and `unwrapped.nenvs`."""

  def __init__(self, kind, nenvs, nactions, obs_dim, act_dim):
    self.nenvs = nenvs
    if kind == "atari":
      self.observation_space = _space(shape=(84, 84, 4), dtype=np.uint8)
      self.action_space = _space(n=nactions, shape=())
    else:
      self.observation_space = _space(shape=(obs_dim,), dtype=np.float64)
      self.action_space = _space(shape=(act_dim,), dtype=np.float32)

  @property
  def unwrapped(self):
    return self


def make_rollout(kind, horizon, nenvs, device="cuda", seed=0, nactions=4, obs_dim=17,
                 act_dim=6, rewards_dtype=None, reset_prob=None):
  """One rollout dict (see module docstring).  `nenvs=None` -> unbatched."""
  dev = torch.device(device)
  gen = torch.Generator(device=dev)
  gen.manual_seed(seed)
  lead = (horizon,) if nenvs is None else (horizon, nenvs)
  tail = () if nenvs is None else (nenvs,)
  randn = lambda shape, dtype=torch.float32: torch.randn(shape, generator=gen, device=dev,
                                                         dtype=dtype)
  rand = lambda shape: torch.rand(shape, generator=gen, device=dev)
  if kind == "atari":
    obs = torch.randint(0, 256, lead + (84, 84, 4), generator=gen, device=dev,
                        dtype=torch.uint8)
    latest = torch.randint(0, 256, tail + (84, 84, 4), generator=gen, device=dev,
                           dtype=torch.uint8)
    actions = torch.randint(0, nactions, lead, generator=gen, device=dev, dtype=torch.int64)
    log_prob = -math.log(nactions) + 0.01 * randn(lead)
    rdt = rewards_dtype or (torch.float32 if dev.type == "cuda" else torch.float64)
    rewards = (torch.sign(randn(lead)) * (rand(lead) < 0.1)).to(rdt)
    resets = rand(lead) < (0.01 if reset_prob is None else reset_prob)
  elif kind == "mujoco":
    obs = randn(lead + (obs_dim,), torch.float64)
    latest = randn(tail + (obs_dim,), torch.float64)
    actions = randn(lead + (act_dim,))
    log_prob = (-0.5 * actions ** 2 - 0.5 * math.log(2 * math.pi)).sum(-1) + 0.01 * randn(lead)
    rewards = randn(lead, rewards_dtype or torch.float64)
    resets = rand(lead) < (0.001 if reset_prob is None else reset_prob)
  else:
    raise ValueError(f"unknown rollout kind {kind!r}")
  values = randn(lead + (1,))
  rollout = dict(observations=obs, actions=actions, log_prob=log_prob, values=values,
                 rewards=rewards, resets=resets, state=dict(latest_observations=latest))
  if dev.type == "cpu":
    for key, val in rollout.items():
      if key != "state":
        rollout[key] = val.numpy()
    rollout["state"]["latest_observations"] = latest.numpy()
  return rollout


def make_frame_stack_rollout(horizon, nenvs, device="cuda", seed=0, nactions=4, k=4, height=84,
                             width=84, reset_prob=0.01, stacked=True):
  """A seeded atari-shaped rollout whose frame stacks are consistent, in both storage forms.

  Every (env, step) sees one random new frame; a stack holds the env's last k frames, and the
  first observation after a reset is the baselines-style [f, f, ..., f] (the reset frame
  repeated).  The rollout starts mid-episode with k-1 frames of history per env, so the planes
  are (horizon + k - 1) * nenvs.  Returns (stacked_rollout, frames_rollout): the same dict twice,
  sharing every column but `observations`, which is a stacked uint8 (T, N, H, W, k) array in the
  first and a `FrameStacks` in the second.  `stacked=False` skips the stacked form (None).
  `state.latest_observations` is stacked in both.
  """
  from .frame_stacks import FrameStacks
  dev = torch.device(device)
  gen = torch.Generator(device=dev)
  gen.manual_seed(seed)
  lead = (horizon, nenvs)
  randn = lambda shape: torch.randn(shape, generator=gen, device=dev)
  rand = lambda shape: torch.rand(shape, generator=gen, device=dev)
  frames = torch.randint(0, 256, ((horizon + k - 1) * nenvs, height, width), generator=gen,
                         device=dev, dtype=torch.uint8)
  latest_frame = torch.randint(0, 256, (nenvs, height, width), generator=gen, device=dev,
                               dtype=torch.uint8)
  actions = torch.randint(0, nactions, lead, generator=gen, device=dev, dtype=torch.int64)
  log_prob = -math.log(nactions) + 0.01 * randn(lead)
  rdt = torch.float32 if dev.type == "cuda" else torch.float64
  rewards = (torch.sign(randn(lead)) * (rand(lead) < 0.1)).to(rdt)
  resets = rand(lead) < reset_prob
  values = randn(lead + (1,))

  # time of the frame in channel c at step t: max(t - (k-1-c), first step of the episode); the
  # plane of (env n, time tau) is (tau + k - 1) * nenvs + n
  done = resets.cpu().numpy()
  episode_start = np.full(nenvs, -(k - 1), dtype=np.int64)
  lags = np.arange(k - 1, -1, -1, dtype=np.int64)
  envs = np.arange(nenvs, dtype=np.int64)
  index = np.empty(lead + (k,), dtype=np.int32)
  for t in range(horizon + 1):
    if t > 0:
      episode_start = np.where(done[t - 1], t, episode_start)
    tau = np.maximum(t - lags[None, :], episode_start[:, None])
    if t < horizon:
      index[t] = (tau + k - 1) * nenvs + envs[:, None]
    else:
      latest_tau = tau
  # latest stack: planes of steps < horizon from `frames`, the step-`horizon` one is new
  latest_ids = torch.from_numpy((np.minimum(latest_tau, horizon - 1) + k - 1) * nenvs
                                + envs[:, None]).to(dev)
  latest = frames[latest_ids].permute(0, 2, 3, 1).contiguous()
  fresh = torch.from_numpy(latest_tau == horizon).to(dev)
  latest = torch.where(fresh[:, None, None, :], latest_frame[..., None], latest)

  index_t = torch.from_numpy(index).to(dev)
  obs = None
  if stacked:
    obs = torch.empty(lead + (height, width, k), dtype=torch.uint8, device=dev)
    for t in range(horizon):
      obs[t] = frames[index_t[t].long()].permute(0, 2, 3, 1)
  columns = dict(actions=actions, log_prob=log_prob, values=values, rewards=rewards,
                 resets=resets)
  if dev.type == "cpu":
    columns = {key: val.numpy() for key, val in columns.items()}
    latest = latest.numpy()
    obs = obs.numpy() if obs is not None else None
  packed = FrameStacks(frames, index_t, validate=False)
  as_stacked = None if obs is None else dict(observations=obs, **columns,
                                             state=dict(latest_observations=latest))
  as_frames = dict(observations=packed, **columns, state=dict(latest_observations=latest))
  return as_stacked, as_frames


class SyntheticRolloutRunner:
  """Yields the same (or freshly seeded) synthetic rollout until `nsteps` env steps."""

  def __init__(self, policy, kind="atari", nenvs=8, horizon=128, nsteps=None, device="cuda",
               seed=0, fresh_each_rollout=False, **rollout_kwargs):
    self.policy, self.kind, self.horizon = policy, kind, horizon
    self.nsteps = None if nsteps is None else int(nsteps)
    self.device, self.seed, self.fresh = device, seed, fresh_each_rollout
    self.rollout_kwargs = rollout_kwargs
    self.env = SyntheticEnv(kind, nenvs, rollout_kwargs.get("nactions", 4),
                            rollout_kwargs.get("obs_dim", 17), rollout_kwargs.get("act_dim", 6))
    self.step_count = 0
    self._cached = None

  @property
  def nenvs(self):
    return self.env.nenvs

  def is_exhausted(self):
    return self.nsteps is not None and self.step_count >= self.nsteps

  def __len__(self):
    return self.nsteps if self.nsteps is not None else self.step_count

  def rollout(self):
    if self._cached is None or self.fresh:
      seed = self.seed + (self.step_count if self.fresh else 0)
      self._cached = make_rollout(self.kind, self.horizon, self.nenvs, self.device, seed,
                                  **self.rollout_kwargs)
    out = dict(self._cached)
    out["state"] = dict(self._cached["state"])
    return out

  def run(self, obs=None):
    while not self.is_exhausted():
      data = self.rollout()
      self.step_count += self.horizon * (self.nenvs or 1)
      yield data
