"""Frame-stack packing on the GPU (K11, torch.ops.derl_b200.pack_frame_stacks,
DeviceFrameStackPacker): the same plane ids and plane bytes as the host FrameStackPacker, no host
synchronisation per step, pool growth and the overflow guard, and EnvRunner(pack_frames=True,
resident_device=...) packing on the device."""
import ctypes

import numpy as np
import pytest
import torch

import derl_b200 as d
from derl_b200 import _lib
from derl_b200.runners.frame_stacks import DeviceFrameStackPacker, FrameStackPacker, unpack
from test_frame_stacks import StackingEnv, pack_all, stacked_sequence

DEV = torch.device("cuda", 0) if torch.cuda.is_available() else None


# ------------------------------------------------------------------------------ CPU
def test_pack_abi_rejects_bad_arguments_without_a_device():
  lib = _lib.load()
  buf = ctypes.create_string_buffer(4096)
  p, null = ctypes.cast(buf, ctypes.c_void_p), ctypes.c_void_p(None)
  state = ctypes.c_void_p(ctypes.addressof(buf) + 1024)

  def call(stacks=p, prev=null, prev_ids=null, n=2, h=4, w=4, k=4, pool=p, cap=64, st=state,
           ids=p, ws=p, ws_bytes=1024):
    rc = lib.derl_b200_pack_frame_stacks(stacks, prev, prev_ids, n, h, w, k, pool, cap, st, ids,
                                         ws, ws_bytes, null)
    return rc, lib.derl_b200_last_error().decode()

  for kw in (dict(stacks=null), dict(pool=null), dict(st=null), dict(ids=null), dict(ws=null)):
    assert call(**kw) == (1, "pack_frame_stacks: null pointer"), kw
  rc, msg = call(prev=p)
  assert rc == 1 and "prev_ids" in msg
  for k in (0, 33, -1):
    rc, msg = call(k=k)
    assert rc == 1 and f"k = {k} outside 1..32" in msg
  for kw in (dict(n=-1), dict(h=-3), dict(w=0), dict(cap=-5), dict(n=0)):
    rc, msg = call(**kw)
    assert rc == 1 and "bad sizes" in msg, kw
  rc, msg = call(cap=2 ** 31)
  assert rc == 1 and "int32" in msg
  assert lib.derl_b200_pack_frame_stacks_workspace_bytes(2, 0) == 0
  assert lib.derl_b200_pack_frame_stacks_workspace_bytes(2, 33) == 0
  need = lib.derl_b200_pack_frame_stacks_workspace_bytes(2, 4)
  assert need >= 16 + 2 * 8 + 2 * 3 * 4 and need % 16 == 0
  rc, msg = call(ws_bytes=need - 1)
  assert rc == 1 and "workspace" in msg


# ------------------------------------------------------------------------------ GPU
def device_pack_all(seq, horizon=None, as_tensor=False):
  """(packer, frames, index) of the device packer over seq [T, N, H, W, k]; ids are written
  into the rows of one device index, as FrameStackRollout does."""
  packer = DeviceFrameStackPacker(DEV, horizon or len(seq))
  index = torch.empty(seq.shape[:2] + seq.shape[-1:], dtype=torch.int32, device=DEV)
  for t, obs in enumerate(seq):
    packer.pack(torch.from_numpy(obs).to(DEV) if as_tensor else obs, out=index[t])
  frames = packer.finish()
  return packer, frames.cpu().numpy(), index.cpu().numpy()


def assert_same_as_host(seq, **kw):
  want, want_index = pack_all(seq)
  _, frames, index = device_pack_all(seq, **kw)
  assert frames.shape[0] == want.count
  assert np.array_equal(index, want_index)
  assert np.array_equal(frames, want.frames.numpy())
  assert np.array_equal(unpack(frames, index), seq)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("hw", [(84, 84), (16, 8), (10, 7)])
@pytest.mark.parametrize("stacks", ["stacked", "resets", "share_nothing"])
def test_device_packer_is_bit_identical_to_the_host_packer(k, hw, stacks):
  for nenvs in (1, 5, 257):
    steps = 6 + nenvs % 4
    seed = 100 * k + nenvs
    if stacks == "share_nothing":
      rng = np.random.default_rng(seed)
      seq = rng.integers(0, 256, (steps, nenvs) + hw + (k,), dtype=np.uint8)
    else:
      seq = stacked_sequence(nenvs, steps, k, hw=hw, reset_prob=0.3 if stacks == "resets" else 0.0,
                             seed=seed)
    assert_same_as_host(seq)


@pytest.fixture(scope="module")
def full_size_sequence():
  return stacked_sequence(4096, 4, 4, hw=(84, 84), reset_prob=0.05, seed=9)


@pytest.mark.gpu
def test_device_packer_at_full_size(full_size_sequence):
  """N = 4096, 84x84x4: the vectorised path."""
  assert_same_as_host(full_size_sequence)


@pytest.mark.gpu
def test_device_packer_is_deterministic(full_size_sequence):
  _, frames_a, index_a = device_pack_all(full_size_sequence)
  _, frames_b, index_b = device_pack_all(full_size_sequence)
  assert np.array_equal(index_a, index_b)
  assert np.array_equal(frames_a, frames_b)


@pytest.mark.gpu
def test_device_packer_reuses_only_equal_bytes():
  """The cases of test_packer_reuses_only_equal_bytes: one differing byte makes a new plane."""
  k = 4
  f = [np.full((1, 4, 4), v, np.uint8) for v in range(6)]
  nearly = f[2].copy()
  nearly[0, 3, 3] ^= 1
  seq = np.stack([np.stack([f[1]] * 4, -1), np.stack([f[1]] * 3 + [f[2]], -1),
                  np.stack([f[1], f[1], nearly, f[3]], -1)])
  packer = DeviceFrameStackPacker(DEV, 3)
  ids = [packer.pack(obs).cpu().numpy() for obs in seq]
  frames = packer.finish().cpu().numpy()
  assert frames.shape[0] == 4
  assert (ids[0] == ids[0][0, 3]).all()
  assert list(ids[1][0]) == [ids[0][0, 3]] * 3 + [1]
  assert ids[2][0, 2] != ids[1][0, 3]
  assert np.array_equal(unpack(frames, np.stack(ids)), seq)
  assert_same_as_host(seq)
  with pytest.raises(TypeError):
    packer.pack(np.zeros((1, 4, 4, k), np.float32))
  with pytest.raises(ValueError):
    packer.pack(np.zeros((2, 4, 4, k), np.uint8))


@pytest.mark.gpu
@pytest.mark.parametrize("horizon", [1, 2])
def test_device_pool_grows_from_a_small_capacity(horizon):
  """Stacks that share nothing add N*k planes per step, far beyond the pool reserved for
  `horizon` steps of the standard case; the output is still the host packer's."""
  rng = np.random.default_rng(horizon)
  seq = rng.integers(0, 256, (9, 5, 16, 8, 4), dtype=np.uint8)
  assert_same_as_host(seq, horizon=horizon)
  assert_same_as_host(seq[:, :, :, :7, :3], horizon=horizon)


@pytest.mark.gpu
@pytest.mark.parametrize("capacity", [3, 12])
def test_pool_overflow_sets_the_flag_and_writes_nothing_past_the_pool(capacity):
  K = torch.ops.derl_b200
  rng = np.random.default_rng(capacity)
  step = torch.from_numpy(rng.integers(0, 256, (5, 16, 8, 4), dtype=np.uint8)).to(DEV)
  big = torch.full((capacity + 40, 16, 8), 0xAB, dtype=torch.uint8, device=DEV)
  pool = big[:capacity]
  state = torch.zeros(2, dtype=torch.int64, device=DEV)
  ids = torch.full((5, 4), -7, dtype=torch.int32, device=DEV)
  K.pack_frame_stacks(step, None, None, pool, state, ids)   # needs 20 planes
  assert state.tolist() == [0, 1]
  assert (big[capacity:] == 0xAB).all()
  assert (ids == -7).all()
  # the flag is sticky: a later step that would fit does nothing either
  roomy = torch.zeros((64, 16, 8), dtype=torch.uint8, device=DEV)
  K.pack_frame_stacks(step, None, None, roomy, state, ids)
  assert state.tolist() == [0, 1] and (ids == -7).all() and not roomy.any()


@pytest.mark.gpu
def test_device_packer_raises_on_overflow(monkeypatch):
  rng = np.random.default_rng(1)
  seq = rng.integers(0, 256, (2, 5, 16, 8, 4), dtype=np.uint8)
  packer = DeviceFrameStackPacker(DEV, 2)
  packer.pack(seq[0])
  packer._pool = packer._pool[:24]
  monkeypatch.setattr(packer, "_reserve", lambda need, nk: None)
  packer.pack(seq[1])   # needs 20 more planes than the 20 it has
  with pytest.raises(RuntimeError, match="overflow"):
    packer.finish()


@pytest.mark.gpu
def test_device_packer_does_not_synchronise():
  seq = stacked_sequence(33, 8, 4, hw=(84, 84), reset_prob=0.2, seed=5)
  steps = [torch.from_numpy(obs).to(DEV) for obs in seq]
  packer = DeviceFrameStackPacker(DEV, len(seq))
  index = torch.empty((8, 33, 4), dtype=torch.int32, device=DEV)
  torch.cuda.synchronize()
  torch.cuda.set_sync_debug_mode("error")
  try:
    for t, obs in enumerate(steps):
      packer.pack(obs, out=index[t])
  finally:
    torch.cuda.set_sync_debug_mode(0)
  frames = packer.finish()
  _, want_frames, want_index = device_pack_all(seq)
  assert np.array_equal(index.cpu().numpy(), want_index)
  assert np.array_equal(frames.cpu().numpy(), want_frames)
  # a new rollout on the same packer starts from an empty pool, with no previous step
  packer.reset()
  again = torch.stack([packer.pack(obs) for obs in steps])
  assert torch.equal(again, index) and torch.equal(packer.finish(), frames)


class SyncPolicy:
  """Returns host arrays, like a policy that runs on the GPU and copies its outputs back."""

  def __init__(self, nenvs):
    self.nenvs = nenvs

  def act(self, obs):
    values = torch.full((self.nenvs,), 0.5, device=DEV).cpu().numpy()
    return {"actions": np.zeros(self.nenvs, np.int64), "values": values}


def collect(nenvs, horizon, rollouts, **kw):
  env = StackingEnv(nenvs, 4, hw=(16, 8), stack=kw.pop("stack"))
  runner = d.EnvRunner(env, SyncPolicy(nenvs), horizon, nsteps=horizon * nenvs * rollouts,
                       pack_frames=True, **kw)
  return list(runner.run())


@pytest.mark.gpu
@pytest.mark.parametrize("stack", [True, False])
def test_env_runner_packs_resident_rollouts_on_the_device(stack, monkeypatch):
  host = collect(5, 7, 3, stack=stack)

  def no_host_packing(self, obs):
    raise AssertionError("the resident route must not pack on the host")

  monkeypatch.setattr(FrameStackPacker, "pack", no_host_packing)
  got = collect(5, 7, 3, stack=stack, resident_device=DEV)
  assert len(got) == len(host) == 3
  for g, w in zip(got, host):
    obs, want = g["observations"], w["observations"]
    assert obs.is_cuda and obs.index.is_cuda and not want.is_cuda
    assert torch.equal(obs.index.cpu(), want.index)
    assert torch.equal(obs.frames.cpu(), want.frames)
    assert np.array_equal(g["state"]["latest_observations"], w["state"]["latest_observations"])
