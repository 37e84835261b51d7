"""Rollouts stored as unique frame planes + stack index (derl_b200/runners/frame_stacks.py):
the host packer, the FrameStacks column in the runner wrappers, EnvRunner(pack_frames=True),
make_frame_stack_rollout, and on the GPU the K10 gather and a full PPO update from it."""
import numpy as np
import pytest
import torch

import derl_b200 as d
from derl_b200.runners.frame_stacks import FrameStackPacker, FrameStacks, unpack
from derl_b200.runners.onpolicy import IterateWithMinibatches, gather_minibatch

DEV = torch.device("cuda", 0) if torch.cuda.is_available() else None


# ------------------------------------------------------------------------------ helpers
class StackingEnv:
  """Batched env with baselines-style frame stacks: each step shifts in one new random frame;
  the first observation after a reset (and after `reset()`) is the new frame repeated k times.
  `stack=False`: every observation is fresh noise (stacks share nothing)."""

  def __init__(self, nenvs, k, hw=(12, 8), reset_prob=0.2, stack=True, seed=0):
    self.nenvs, self.k, self.hw = nenvs, k, hw
    self.reset_prob, self.stack_frames = reset_prob, stack
    self.rng = np.random.default_rng(seed)
    self.stack = None

  @property
  def unwrapped(self):
    return self

  def _frames(self):
    return self.rng.integers(0, 256, (self.nenvs,) + self.hw, dtype=np.uint8)

  def _noise(self):
    return self.rng.integers(0, 256, (self.nenvs,) + self.hw + (self.k,), dtype=np.uint8)

  def reset(self):
    self.stack = np.repeat(self._frames()[..., None], self.k, axis=-1) if self.stack_frames \
        else self._noise()
    return self.stack.copy()

  def step(self, actions):
    done = self.rng.random(self.nenvs) < self.reset_prob
    if self.stack_frames:
      self.stack = np.concatenate([self.stack[..., 1:], self._frames()[..., None]], axis=-1)
      fresh = self._frames()
      self.stack[done] = np.repeat(fresh[done][..., None], self.k, axis=-1)
    else:
      self.stack = self._noise()
    rewards = self.rng.standard_normal(self.nenvs).astype(np.float32)
    return self.stack.copy(), rewards, done, [{} for _ in range(self.nenvs)]


class ZeroPolicy:
  def __init__(self, nenvs):
    self.nenvs = nenvs

  def act(self, obs):
    return {"actions": np.zeros(self.nenvs, np.int64),
            "values": np.full(self.nenvs, 0.5, np.float32)}


def stacked_sequence(nenvs, steps, k, hw=(12, 8), reset_prob=0.0, seed=0):
  """[steps, N, H, W, k] of a baselines-style env that starts mid-episode (k-1 history frames)."""
  rng = np.random.default_rng(seed)
  stack = rng.integers(0, 256, (nenvs,) + hw + (k,), dtype=np.uint8)
  out = []
  for _ in range(steps):
    out.append(stack.copy())
    frame = rng.integers(0, 256, (nenvs,) + hw, dtype=np.uint8)
    stack = np.concatenate([stack[..., 1:], frame[..., None]], axis=-1)
    done = rng.random(nenvs) < reset_prob
    stack[done] = np.repeat(frame[done][..., None], k, axis=-1)
  return np.stack(out)


def pack_all(seq):
  packer = FrameStackPacker()
  index = np.stack([packer.pack(obs) for obs in seq])
  return packer, index


def run_env_runner(pack_frames, nenvs=5, horizon=7, rollouts=3, resident_device=None, **env_kw):
  env = StackingEnv(nenvs, **env_kw)
  runner = d.EnvRunner(env, ZeroPolicy(nenvs), horizon, nsteps=horizon * nenvs * rollouts,
                       resident_device=resident_device, pack_frames=pack_frames)
  return list(runner.run())


# ------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("k", [1, 2, 3, 4])
@pytest.mark.parametrize("reset_prob", [0.0, 0.3])
def test_packer_round_trips_baselines_stacks(k, reset_prob):
  seq = stacked_sequence(6, 9, k, reset_prob=reset_prob, seed=k)
  packer, index = pack_all(seq)
  assert index.dtype == np.int32 and index.shape == (9, 6, k)
  assert np.array_equal(unpack(packer.frames.numpy(), index), seq)
  if reset_prob == 0.0:
    assert packer.count == 9 * 6 + 6 * (k - 1)
  else:   # a reset stack [f, ..., f] adds one plane, so resets never add to the count
    assert packer.count <= 9 * 6 + 6 * (k - 1)


@pytest.mark.parametrize("k", [1, 2, 3, 4])
def test_packer_round_trips_stacks_that_share_nothing(k):
  rng = np.random.default_rng(k)
  seq = rng.integers(0, 256, (5, 4, 16, 4, k), dtype=np.uint8)
  packer, index = pack_all(seq)
  assert np.array_equal(unpack(packer.frames.numpy(), index), seq)
  assert packer.count == seq.size // (16 * 4)   # no reuse
  # capacity reserved for the standard case is outgrown without loss
  small = FrameStackPacker(capacity=3)
  index = np.stack([small.pack(obs) for obs in seq])
  assert np.array_equal(unpack(small.frames.numpy(), index), seq)


def test_packer_reuses_only_equal_bytes():
  """Equal channels inside a stack reuse one plane; a channel equal to channel c+1 of the
  previous step reuses that plane; one differing byte makes a new plane."""
  k = 4
  f = [np.full((1, 4, 4), v, np.uint8) for v in range(6)]
  packer = FrameStackPacker()
  ids0 = packer.pack(np.stack([f[1], f[1], f[1], f[1]], -1))      # reset stack: one plane
  assert packer.count == 1 and (ids0 == ids0[0, 3]).all()
  ids1 = packer.pack(np.stack([f[1], f[1], f[1], f[2]], -1))
  assert packer.count == 2 and list(ids1[0]) == [ids0[0, 3]] * 3 + [1]
  nearly = f[2].copy()
  nearly[0, 3, 3] ^= 1
  ids2 = packer.pack(np.stack([f[1], f[1], nearly, f[3]], -1))
  assert packer.count == 4 and ids2[0, 2] not in (ids1[0, 3],)
  seq = np.stack([np.stack([f[1]] * 4, -1), np.stack([f[1]] * 3 + [f[2]], -1),
                  np.stack([f[1], f[1], nearly, f[3]], -1)])
  assert np.array_equal(unpack(packer.frames.numpy(), np.stack([ids0, ids1, ids2])), seq)
  with pytest.raises(TypeError):
    packer.pack(np.zeros((1, 4, 4, k), np.float32))
  with pytest.raises(ValueError):
    packer.pack(np.zeros((2, 4, 4, k), np.uint8))


def test_frame_stacks_array_interface_and_merge_time_batch():
  seq = stacked_sequence(3, 4, 4, hw=(8, 6))
  packer, index = pack_all(seq)
  col = FrameStacks(packer.frames, index)
  assert col.shape == seq.shape and col.ndim == seq.ndim and col.dtype == torch.uint8
  assert len(col) == 4 and not col.is_cuda
  traj = {"observations": col, "resets": np.zeros((4, 3), bool),
          "rewards": np.zeros((4, 3), np.float32)}
  d.MergeTimeBatch()(traj)
  merged = traj["observations"]
  assert isinstance(merged, FrameStacks) and merged.shape == (12, 8, 6, 4)
  assert np.array_equal(unpack(merged.frames.numpy(), merged.index.numpy()),
                        seq.reshape(12, 8, 6, 4))
  assert merged.reshape(4, 3, 8, 6, 4).shape == seq.shape
  with pytest.raises(ValueError):
    merged.reshape(12, 6, 8, 4)


def test_frame_stacks_reject_out_of_range_plane_ids():
  frames = np.zeros((5, 4, 4), np.uint8)
  FrameStacks(frames, np.array([[0, 1, 2, 4]]))
  with pytest.raises(IndexError, match="5"):
    FrameStacks(frames, np.array([[0, 1, 2, 5]]))
  with pytest.raises(IndexError, match="-1"):
    FrameStacks(frames, np.array([[-1, 1, 2, 3]], np.int32))
  with pytest.raises(TypeError):
    FrameStacks(frames, np.array([[0.0, 1.0]]))
  with pytest.raises(TypeError):
    FrameStacks(frames.astype(np.int16), np.array([[0, 1]]))


@pytest.mark.parametrize("stack", [True, False])
def test_env_runner_pack_frames_yields_the_stacked_observations(stack):
  """Several rollouts of one runner (each packed from its own first step) equal the stacked run;
  latest_observations stays stacked."""
  k = 4
  want = run_env_runner(False, k=k, stack=stack)
  got = run_env_runner(True, k=k, stack=stack)
  assert len(got) == len(want) == 3
  for i, (g, w) in enumerate(zip(got, want)):
    assert list(g) == list(w)   # same keys, same order
    obs = g["observations"]
    assert isinstance(obs, FrameStacks) and obs.shape == (7, 5, 12, 8, k)
    assert np.array_equal(unpack(obs.frames.numpy(), obs.index.numpy()), np.asarray(w["observations"]))
    assert np.array_equal(g["state"]["latest_observations"], w["state"]["latest_observations"])
    for key in ("actions", "rewards", "resets"):
      assert np.array_equal(np.asarray(g[key]), np.asarray(w[key]))
    if stack:
      assert obs.num_frames <= 7 * 5 + 5 * (k - 1)
    else:
      assert obs.num_frames == 7 * 5 * k
  # no resets: the first rollout starts at reset() stacks, later ones mid-episode
  counts = [r["observations"].num_frames for r in run_env_runner(True, k=k, reset_prob=0.0)]
  assert counts == [7 * 5, 7 * 5 + 5 * (k - 1), 7 * 5 + 5 * (k - 1)]


def test_make_frame_stack_rollout_forms_agree():
  stacked, packed = d.make_frame_stack_rollout(9, 5, device="cpu", seed=4, reset_prob=0.3,
                                               height=8, width=6)
  obs = packed["observations"]
  assert obs.shape == stacked["observations"].shape == (9, 5, 8, 6, 4)
  assert obs.num_frames == (9 + 3) * 5
  assert np.array_equal(unpack(obs.frames.numpy(), obs.index.numpy()), stacked["observations"])
  for key in ("actions", "log_prob", "values", "rewards", "resets"):
    assert packed[key] is stacked[key]
  assert stacked["resets"].any()
  latest = packed["state"]["latest_observations"]
  assert latest.shape == (5, 8, 6, 4)
  # baselines stacks: channel c of step t is channel c+1 of step t-1 unless step t follows a reset
  seq = np.concatenate([stacked["observations"], latest[None]])
  for t in range(1, 10):
    cont = ~stacked["resets"][t - 1]
    assert np.array_equal(seq[t, cont, ..., :-1], seq[t - 1, cont, ..., 1:])
    reset = stacked["resets"][t - 1]
    assert (seq[t, reset] == seq[t, reset][..., :1]).all()
  _, only = d.make_frame_stack_rollout(9, 5, device="cpu", seed=4, reset_prob=0.3, height=8,
                                       width=6, stacked=False)
  assert torch.equal(only["observations"].index, obs.index)


# ------------------------------------------------------------------------------ GPU
K = torch.ops.derl_b200 if DEV is not None else None


def random_frame_stacks(nsamples, nframes, hw, k, seed):
  gen = torch.Generator(device=DEV).manual_seed(seed)
  frames = torch.randint(0, 256, (nframes,) + hw, generator=gen, device=DEV, dtype=torch.uint8)
  index = torch.randint(0, nframes, (nsamples, k), generator=gen, device=DEV, dtype=torch.int32)
  stacked = frames[index.long()].permute(0, 2, 3, 1).contiguous()
  return frames, index, stacked


@pytest.mark.gpu
@pytest.mark.parametrize("hw,k", [((84, 84), 4), ((12, 8), 4), ((84, 84), 1), ((84, 84), 3),
                                  ((10, 7), 4), ((9, 9), 2), ((5, 6), 5)])
def test_k10_is_bit_identical_to_the_stacked_gather(hw, k):
  frames, index, stacked = random_frame_stacks(3000, 900, hw, k, seed=k)
  gen = torch.Generator(device=DEV).manual_seed(7)
  perm = torch.randperm(3000, generator=gen, device=DEV)
  for start, count in ((0, 3000), (17, 1), (5, 1031), (2999, 1), (100, 0)):
    got = K.gather_frame_stacks(frames, index, perm, start, count)
    want = stacked[perm[start:start + count]]
    assert got.shape == (count,) + hw + (k,)
    assert torch.equal(got, want), (start, count)
    if count:
      assert torch.equal(got, K.gather_rows(stacked, perm, start, count))
  repeated = torch.tensor([4, 4, 4, 0, 2999, 4, 0], device=DEV)
  assert torch.equal(K.gather_frame_stacks(frames, index, repeated, 0, 7), stacked[repeated])
  with pytest.raises(ValueError, match="window"):
    K.gather_frame_stacks(frames, index, perm, 2990, 11)


@pytest.mark.gpu
def test_k10_default_shape_at_minibatch_scale_and_repeated_launches():
  frames, index, stacked = random_frame_stacks(40000, 12000, (84, 84), 4, seed=11)
  perm = torch.randperm(40000, device=DEV)
  first = K.gather_frame_stacks(frames, index, perm, 123, 39000)
  assert torch.equal(first, stacked[perm[123:123 + 39000]])
  for _ in range(3):
    assert torch.equal(K.gather_frame_stacks(frames, index, perm, 123, 39000), first)
  # an index view that is not 16-byte aligned takes the plain kernel: same bytes
  wide = torch.zeros(40000 * 4 + 1, dtype=torch.int32, device=DEV)
  wide[1:] = index.reshape(-1)
  unaligned = wide[1:].view(40000, 4)
  assert torch.equal(K.gather_frame_stacks(frames, unaligned, perm, 0, 5000), stacked[perm[:5000]])


@pytest.mark.gpu
def test_pinned_host_frame_stacks_upload_and_gather():
  stacked, packed = d.make_frame_stack_rollout(6, 40, device="cpu", seed=2, height=84, width=84)
  host = packed["observations"]
  pinned = FrameStacks(host.frames.pin_memory(), host.index.pin_memory())
  traj = dict(packed, observations=pinned)
  runner = d.TransformInteractions(type("R", (), {"run": lambda self, obs=None: iter([traj])})(),
                                   [d.MergeTimeBatch()])
  out = next(runner.run())
  col = out["observations"]
  assert isinstance(col, FrameStacks) and col.is_cuda and col.shape == (240, 84, 84, 4)
  want = torch.from_numpy(stacked["observations"]).reshape(240, 84, 84, 4).to(DEV)
  perm = torch.randperm(240, device=DEV)
  batch = gather_minibatch(out, perm, 10, 100)
  assert torch.equal(batch["observations"], want[perm[10:110]])
  assert torch.equal(batch["actions"], out["actions"][perm[10:110]])
  assert torch.equal(col.materialize(), want)
  assert torch.equal(host.materialize().cpu(), torch.from_numpy(stacked["observations"]))


@pytest.mark.gpu
def test_take_and_shuffle_work_on_frame_stacks():
  stacked, packed = d.make_frame_stack_rollout(5, 8, device=DEV, seed=5, height=12, width=8)
  a, b = dict(stacked), dict(packed)
  d.Take([6, 1, -1], axis=1)(a)
  d.Take([6, 1, -1], axis=1)(b)
  assert torch.equal(a["observations"], b["observations"])
  a, b = dict(stacked), dict(packed)
  d.MergeTimeBatch()(a)
  d.MergeTimeBatch()(b)
  np.random.seed(3)
  IterateWithMinibatches.shuffle_interactions(a)
  np.random.seed(3)
  IterateWithMinibatches.shuffle_interactions(b)
  for key in a:
    if key != "state":
      assert torch.equal(a[key], b[key]), key


@pytest.mark.gpu
@pytest.mark.parametrize("stack", [True, False])
def test_env_runner_pack_frames_resident_on_the_device(stack):
  """Device pool filled step by step from the pinned mirror; with stacks that share nothing it
  outgrows the capacity reserved for the standard case."""
  want = run_env_runner(False, k=4, stack=stack, resident_device=DEV, hw=(16, 8))
  got = run_env_runner(True, k=4, stack=stack, resident_device=DEV, hw=(16, 8))
  for g, w in zip(got, want):
    obs = g["observations"]
    assert isinstance(obs, FrameStacks) and obs.is_cuda
    assert torch.equal(obs.materialize(), w["observations"])
    assert np.array_equal(g["state"]["latest_observations"], w["state"]["latest_observations"])
    assert torch.equal(g["state"]["latest_values"], w["state"]["latest_values"])
    if not stack:
      assert obs.num_frames == 7 * 5 * 4   # beyond the 7 * 5 + 5 * 3 planes reserved


class FixedSource:
  """EnvRunner-like source yielding one rollout dict (fresh dict each time)."""

  def __init__(self, policy, rollout, nenvs, horizon):
    self.policy, self.rollout, self.horizon = policy, rollout, horizon
    self.env = d.runners.SyntheticEnv("atari", nenvs, 4, 17, 6)
    self.nsteps, self.step_count = None, 0

  def is_exhausted(self):
    return False

  def run(self, obs=None):
    while True:
      self.step_count += self.horizon * self.env.nenvs
      out = dict(self.rollout)
      out["state"] = dict(self.rollout["state"])
      yield out


@pytest.mark.gpu
@pytest.mark.parametrize("fused_gather", [False, True])
def test_ppo_update_from_frame_stacks_is_bit_identical(fused_gather):
  """Default TF32 + K6t/K7t network, micro-batched Trainer: losses and parameters after two
  updates from a FrameStacks rollout equal those from the same rollout stored stacked."""
  nsteps, nenvs, nact = 16, 24, 4
  stacked, packed = d.make_frame_stack_rollout(nsteps, nenvs, device=DEV, seed=8, nactions=nact,
                                               reset_prob=0.05)
  assert torch.backends.cudnn.allow_tf32
  results = []
  for rollout in (stacked, packed):
    torch.manual_seed(0)
    policy = d.ActorCriticPolicy(d.NatureCNNModel([nact, 1]))
    source = FixedSource(policy, rollout, nenvs, nsteps)
    runner = d.ppo_runner_wrap(source, num_epochs=2, num_minibatches=2, fused_gather=fused_gather)
    optimizer = torch.optim.Adam(policy.model.parameters(), lr=2.5e-4, eps=1e-5)
    alg = d.PPO(runner, d.Trainer(optimizer, max_grad_norm=0.5, micro_batch=64), cliprange=0.1)
    np.random.seed(21)
    it = runner.run()
    losses = [alg.step(next(it)) for _ in range(2 * 4)]
    results.append((torch.stack([l.detach() for l in losses]),
                    [p.detach().clone() for p in policy.model.parameters()]))
  (loss_s, params_s), (loss_f, params_f) = results
  assert torch.equal(loss_s, loss_f)
  for a, b in zip(params_s, params_f):
    assert torch.equal(a, b)
