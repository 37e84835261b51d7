"""Runner wrappers of the PPO data path: the rollout-transform hook and the epoch /
minibatch iterator, with the rollout resident in HBM.

Reference: derl/runners/onpolicy.py — TransformInteractions :11-30, IterateWithMinibatches
:33-62, ppo_runner_wrap :65-75, make_ppo_runner :78-82.

What changes underneath the unchanged API: the reference copies the whole rollout once per
epoch (`val[indices]` for every key, :47-49) and again per minibatch (:59-62), on the host.
Here the rollout is uploaded once, never physically shuffled, and each minibatch is ONE
permutation-indexed gather (torch.ops.derl_b200.gather_rows / gather_columns) driven by the
composed permutation P_e = P_{e-1}[perm_e] — which selects exactly the rows the reference's
in-place shuffles select.  The global NumPy RNG is consumed identically (one
`np.random.permutation(S)` per epoch), so seeded runs see the same minibatches.
"""
import numpy as np
import torch

from .. import _lib, ops  # noqa: F401
from .env_runner import EnvRunner, RunnerWrapper
from .frame_stacks import FrameStacks
from .host_column import HostColumn, eligible as _lazy_eligible
from .row_selection import RowSelection
from .summary import PeriodicSummaries
from .trajectory_transforms import (GAE, MergeTimeBatch, NormalizeAdvantages, policy_device,
                                    to_device)

_K = torch.ops.derl_b200
WIDE_ROW_BYTES = 2048  # rows at least this wide go through the TMA bulk-copy gather


class TransformInteractions(RunnerWrapper):
  """Applies a list of callables to every interactions dict the wrapped runner yields.

  `asarray=True` (reference: `np.asarray` of every value, :20-27) here means "make it a
  dense array ON THE DEVICE": lists of per-step arrays are stacked and uploaded once;
  tensors already on the device pass through untouched; non-numeric values (e.g. `infos`)
  stay NumPy object arrays on the host.
  """

  def __init__(self, runner, transforms=None, asarray=True, lazy_upload=True):
    super().__init__(runner)
    self.transforms = transforms or []
    self.asarray = asarray
    # wide columns handed over in PINNED host memory are uploaded by the first epoch's gathers
    # (overlapped with the update) instead of one blocking copy; see runners/host_column.py
    self.lazy_upload = lazy_upload

  def _densify(self, key, val, device):
    if isinstance(val, (torch.Tensor, HostColumn, RowSelection)):
      return val
    if isinstance(val, FrameStacks):
      return val.to_device(device)
    try:
      arr = np.asarray(val)
    except ValueError:
      raise ValueError(f"cannot convert value under key '{key}' to np.ndarray")
    if arr.dtype == object or arr.dtype.kind in "USV":
      return arr
    if self.lazy_upload and key == "observations":
      host = _lazy_eligible(arr)
      if host is not None:
        return HostColumn(host, device)
    return to_device(arr, device)

  def run(self, obs=None):
    for interactions in self.runner.run(obs=obs):
      if self.asarray:
        device = policy_device(getattr(self, "policy", None))
        for key in [k for k in interactions if k != "state"]:
          interactions[key] = self._densify(key, interactions[key], device)
      for transform in self.transforms:
        transform(interactions)
      yield interactions


def _row_bytes(t):
  return (t[0].numel() * t.element_size()) if t.shape[0] > 0 else 0


def gather_minibatch(interactions, perm, start, count, host_perm=None, perm_ready=None,
                     fused_gather=False):
  """dict of rows perm[start:start+count] of every array in `interactions`.

  Wide columns (frame stacks) use the TMA row gather, all narrow columns share one launch
  which also reduces the float64 moments of `advantages` (attached as `_derl_moments`).
  fused_gather: a resident `observations` column is handed on as a `RowSelection` (source +
  row indices) for the network's stem kernels to read in place instead of being copied.
  A `FrameStacks` column is always rebuilt into stacked rows by K10 (fused_gather or not).
  """
  out, narrow = {}, []
  for key, val in interactions.items():
    if key == "state":
      out[key] = val
    elif isinstance(val, FrameStacks):
      out[key] = val.gather(perm, start, count)
    elif isinstance(val, HostColumn):
      if fused_gather and key == "observations" and val.complete:
        out[key] = RowSelection(val.resident, perm, start, count)
      else:
        out[key] = val.gather(perm, start, count, perm_ready)
    elif isinstance(val, torch.Tensor):
      if not val.is_cuda:
        raise TypeError(f"interactions['{key}'] is a CPU tensor; the rollout must be resident "
                        "on the GPU (derl_b200 has no host gather path)")
      if _row_bytes(val) >= WIDE_ROW_BYTES:
        if fused_gather and key == "observations" and val.is_contiguous():
          out[key] = RowSelection(val, perm, start, count)
        else:
          out[key] = _K.gather_rows(val, perm, start, count)
      else:
        narrow.append(key)
    else:  # host object arrays (infos): plain NumPy fancy index with the same rows
      rows = host_perm[start:start + count] if host_perm is not None \
          else perm[start:start + count].cpu().numpy()
      out[key] = np.asarray(val)[rows]
  for lo in range(0, len(narrow), _lib.MAX_COLUMNS):
    keys = narrow[lo:lo + _lib.MAX_COLUMNS]
    cols = [interactions[k] for k in keys]
    adv_col = -1
    if "advantages" in keys:
      adv = interactions["advantages"]
      if adv.dtype == torch.float32 and _row_bytes(adv) == 4:
        adv_col = keys.index("advantages")
    *gathered, moments = _K.gather_columns(cols, perm, start, count, adv_col)
    for key, val in zip(keys, gathered):
      out[key] = val
    if adv_col >= 0:
      out["advantages"]._derl_moments = moments
  return {k: out[k] for k in interactions}  # keep the reference's key order


class IterateWithMinibatches(RunnerWrapper):
  """Iterates over interactions with minibatches for a given number of epochs."""

  def __init__(self, runner, num_epochs=3, num_minibatches=4, shuffle_before_epoch=True,
               fused_gather=False):
    super().__init__(runner)
    self.num_epochs = num_epochs
    self.num_minibatches = num_minibatches
    self.shuffle_before_epoch = shuffle_before_epoch
    self.fused_gather = fused_gather   # extension: see runners/row_selection.py

  @staticmethod
  def _sample_size(interactions):
    return interactions["observations"].shape[0]

  @staticmethod
  def _upload(order, device):
    # staged through pinned memory: a pageable copy would block the host until the stream has
    # drained, once per epoch (the pinned block is recycled by the host allocator after the copy)
    host = torch.from_numpy(np.ascontiguousarray(order, dtype=np.int64))
    if torch.device(device).type != "cuda":
      return host.to(device)
    pinned = torch.empty(host.shape, dtype=torch.int64, pin_memory=True)
    pinned.copy_(host)
    return pinned.to(device, non_blocking=True)

  @staticmethod
  def shuffle_interactions(interactions):
    """Physically shuffles every key but "state" with one np.random.permutation (:43-49).
    Kept for API parity; `run` never needs the physical shuffle."""
    size = IterateWithMinibatches._sample_size(interactions)
    order = np.random.permutation(size)
    device = next((v.device for v in interactions.values()
                   if isinstance(v, torch.Tensor) and v.is_cuda), None)
    if device is None:
      raise TypeError("shuffle_interactions needs the rollout resident on the GPU")
    for key, val in interactions.items():
      if isinstance(val, HostColumn):
        interactions[key] = val.materialize()
    perm = IterateWithMinibatches._upload(order, device)
    interactions.update(gather_minibatch(interactions, perm, 0, size, host_perm=order))

  def minibatches(self, interactions):
    """The epochs x minibatches of ONE rollout (the body of the reference's run loop, :52-62)."""
    size = self._sample_size(interactions)
    device = next((v.device for v in interactions.values()
                   if isinstance(v, torch.Tensor) and v.is_cuda), None)
    if device is None:
      raise TypeError("IterateWithMinibatches needs the rollout resident on the GPU "
                      "(wrap the runner in TransformInteractions first)")
    order, perm, perm_ready = None, None, None
    for _ in range(self.num_epochs):
      if self.shuffle_before_epoch:
        draw = np.random.permutation(size)                  # same RNG stream as :46
        order = draw if order is None else order[draw]      # compose: shuffles were in place
        perm = self._upload(order, device)
        perm_ready = torch.cuda.current_stream(device).record_event()
      elif perm is None:
        order = np.arange(size)
        perm = self._upload(order, device)
        perm_ready = torch.cuda.current_stream(device).record_event()
      mbsize = size // self.num_minibatches
      for start in range(0, size, mbsize):
        count = min(start + mbsize, size) - start
        yield gather_minibatch(interactions, perm, start, count, host_perm=order,
                               perm_ready=perm_ready, fused_gather=self.fused_gather)

  def run(self, obs=None):
    for interactions in self.runner.run(obs=obs):
      yield from self.minibatches(interactions)


def ppo_runner_wrap(runner, gamma=0.99, lambda_=0.95, num_epochs=3, num_minibatches=4,
                    fused_gather=False):
  """Wraps a rollout source for PPO: [GAE, MergeTimeBatch?] -> minibatches -> normalise
  (reference :65-75; MergeTimeBatch only for non-recurrent policies on batched envs)."""
  env, policy = runner.env, runner.policy
  transforms = [GAE(policy, gamma=gamma, lambda_=lambda_, normalize=False)]
  if not policy.is_recurrent() and getattr(env.unwrapped, "nenvs", None):
    transforms.append(MergeTimeBatch())
  runner = TransformInteractions(runner, transforms)
  runner = IterateWithMinibatches(runner, num_epochs, num_minibatches, fused_gather=fused_gather)
  return TransformInteractions(runner, [NormalizeAdvantages()])


def make_ppo_runner(env, policy, horizon, nsteps, nlogs=1e5, **wrap_kwargs):
  """EnvRunner -> PeriodicSummaries -> ppo_runner_wrap (reference :78-82)."""
  runner = EnvRunner(env, policy, horizon, nsteps)
  runner = PeriodicSummaries.make_with_nlogs(runner, nlogs)
  return ppo_runner_wrap(runner, **wrap_kwargs)
