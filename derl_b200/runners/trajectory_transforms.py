"""Rollout transforms with the reference's protocol (`transform(trajectory_dict)`, in-place),
computing on the B200 through torch.ops.derl_b200.*.

Reference: derl/runners/trajectory_transforms.py — GAE :5-72, MergeTimeBatch :75-81,
NormalizeAdvantages :84-92, Take :95-103.  Values of the trajectory dict may be CUDA
tensors (the resident-rollout pipeline of this package) or NumPy arrays (a caller coming
from the reference's host pipeline): NumPy in -> NumPy out, tensor in -> tensor out; either
way the arithmetic runs in the CUDA kernels, never on the host.
"""
import numpy as np
import torch

from .. import ops  # noqa: F401  (registers torch.ops.derl_b200)

_K = torch.ops.derl_b200


def policy_device(policy=None):
  """Device the rollout should live on: the policy model's, else the current CUDA device."""
  model = getattr(policy, "model", None)
  if model is not None:
    try:
      dev = next(model.parameters()).device
      if dev.type == "cuda":
        return dev
    except StopIteration:
      pass
  return torch.device("cuda", torch.cuda.current_device())


def to_device(value, device):
  """NumPy array / tensor -> contiguous tensor on `device` (one upload, pinned if large)."""
  if isinstance(value, torch.Tensor):
    return value.to(device).contiguous()
  arr = np.ascontiguousarray(value)
  host = torch.from_numpy(arr)
  return host.to(device, non_blocking=False)


def _is_array(value):
  from .frame_stacks import FrameStacks
  from .host_column import HostColumn
  return isinstance(value, (np.ndarray, torch.Tensor, HostColumn, FrameStacks))


class GAE:
  """Generalized Advantage Estimator (Schulman et al. 2016) on the sm_100a scan kernel.

  Same constructor, keys, errors and return value as the reference (:10-16, :18-72).  The
  reverse scan is bit-identical to the reference's NumPy loop (float64 register
  arithmetic, float32 stores); `normalize` uses float64 moments reduced on the device.
  `variant` picks the kernel (0 auto, 1 direct, 2 TMA) — an extension, default auto.
  """

  def __init__(self, policy, gamma=0.99, lambda_=0.95, normalize=None, epsilon=1e-8,
               variant=0):
    self.policy = policy
    self.gamma = gamma
    self.lambda_ = lambda_
    self.normalize = normalize
    self.epsilon = epsilon
    self.variant = variant

  def bootstrap_value(self, trajectory):
    """policy.act(latest_observations)["values"], as the reference asks for it (:47-50)."""
    state = trajectory["state"]
    if state.get("latest_values") is not None:   # EnvRunner(resident_device=): already evaluated
      return state["latest_values"]
    value_tensor = getattr(self.policy, "value_tensor", None)
    if value_tensor is not None and state.get("policy_state", None) is None:
      return value_tensor(state["latest_observations"])   # stays on the device: no sync
    return self.policy.act(state["latest_observations"], state=state.get("policy_state", None),
                           update_state=False)["values"]

  def __call__(self, trajectory):
    if "advantages" in trajectory:
      raise ValueError("trajectory cannot contain 'advantages'")
    if "value_targets" in trajectory:
      raise ValueError("trajectory cannot contain 'value_targets'")
    rewards, resets, values = (trajectory[k] for k in ("rewards", "resets", "values"))
    if (not 0 <= values.ndim - rewards.ndim <= 1
        or values.ndim == rewards.ndim + 1 and values.shape[-1] != 1):
      raise ValueError(
          f"trajectory['values'] of shape {tuple(values.shape)} "
          "must have the same number of dimensions as "
          f"trajectory['rewards'] which has shape {tuple(rewards.shape)} "
          "or have last dimension of size 1")
    as_numpy = isinstance(values, np.ndarray)
    device = values.device if isinstance(values, torch.Tensor) and values.is_cuda \
        else policy_device(self.policy)

    values_d = to_device(values, device)
    if values_d.dtype != torch.float32:
      raise TypeError(f"trajectory['values'] must be float32, got {values_d.dtype}")
    squeezed_shape = tuple(values.shape[:-1]) if values.ndim == rewards.ndim + 1 \
        else tuple(values.shape)
    rewards_d = to_device(rewards, device)
    if rewards_d.dtype not in (torch.float32, torch.float64):
      rewards_d = rewards_d.to(torch.float64)  # ints/halves promote like NumPy would
    resets_d = to_device(resets, device)
    if resets_d.dtype not in (torch.bool, torch.uint8):
      raise TypeError(f"trajectory['resets'] must be bool or uint8, got {resets_d.dtype}")
    last_value = to_device(self.bootstrap_value(trajectory), device).to(torch.float32)

    nsteps = squeezed_shape[0]
    nenvs = int(np.prod(squeezed_shape[1:], dtype=np.int64)) if len(squeezed_shape) > 1 else 1
    if tuple(rewards_d.shape) != squeezed_shape or tuple(resets_d.shape) != squeezed_shape:
      raise ValueError(f"rewards {tuple(rewards_d.shape)} and resets {tuple(resets_d.shape)} "
                       f"must match values {squeezed_shape}")
    if last_value.numel() != nenvs:
      raise ValueError(f"bootstrap values have {last_value.numel()} elements, "
                       f"expected {nenvs}")
    nelem = nsteps * nenvs
    do_normalize = bool(self.normalize or (self.normalize is None and nelem > 1))
    adv, targets, stats = _K.gae(rewards_d.reshape(nsteps, nenvs), values_d.reshape(nsteps, nenvs),
                                 resets_d.reshape(nsteps, nenvs), last_value.reshape(nenvs),
                                 float(self.gamma), float(self.lambda_), do_normalize,
                                 int(self.variant))
    if do_normalize:
      adv = _K.normalize(adv, stats, float(self.epsilon))
    adv = adv.reshape(squeezed_shape)
    targets = targets.reshape(tuple(values.shape))
    if as_numpy:
      adv, targets = adv.cpu().numpy(), targets.cpu().numpy()
    trajectory["advantages"] = adv
    trajectory["value_targets"] = targets
    return adv, targets


class MergeTimeBatch:
  """(T, N, ...) -> (T*N, ...) for every array value; a view, no copy (:77-81)."""

  def __call__(self, trajectory):
    assert trajectory["resets"].ndim == 2, trajectory["resets"].shape
    for key, val in trajectory.items():
      if _is_array(val):
        trajectory[key] = val.reshape((-1,) + tuple(val.shape[2:]))


class NormalizeAdvantages:
  """advantages <- (adv - mean) / (std_pop + epsilon) over the minibatch (:84-92).

  When the minibatch came out of IterateWithMinibatches its float64 moments were already
  reduced inside the gather kernel and ride along on the tensor (`_derl_moments`), so this
  is a single elementwise launch.  `group`: optional torch.distributed process group —
  moments are all-reduced so every env-axis shard normalises with the GLOBAL minibatch
  statistics (SURVEY.md §8e).
  """

  def __init__(self, epsilon=1e-8, group=None):
    self.epsilon = epsilon
    self.group = group

  def __call__(self, trajectory):
    adv = trajectory["advantages"]
    as_numpy = isinstance(adv, np.ndarray)
    adv_d = to_device(adv, policy_device()) if as_numpy else adv
    if adv_d.dtype != torch.float32:
      raise TypeError(f"advantages must be float32, got {adv_d.dtype}")
    moments = getattr(adv, "_derl_moments", None)
    if moments is None:
      moments = _K.moments(adv_d.contiguous())
    if self.group is not None:
      import torch.distributed as dist
      moments = moments.clone()
      dist.all_reduce(moments, group=self.group)
    out = _K.normalize(adv_d.contiguous(), moments, float(self.epsilon))
    trajectory["advantages"] = out.cpu().numpy() if as_numpy else out


class Take:
  """Keeps data only from the given indices along `axis` for every key but "state" (:95-103).

  `np.take` semantics for device tensors too: negative indices count from the end, an index
  outside [-n, n) raises IndexError (the gather kernels never bounds-check: the indices are the
  caller's and live on the host, so they are validated THERE, once, without a device sync), and
  an index array of any rank replaces the axis by its own shape.
  """

  def __init__(self, indices, axis=1):
    self.indices = indices
    self.axis = axis

  def _checked(self, size):
    """Host int64 indices wrapped into [0, size); IndexError like NumPy's when out of bounds."""
    index = np.asarray(self.indices)
    if index.size == 0:   # np.take accepts an empty (float64) list
      index = index.astype(np.int64)
    if index.dtype == np.bool_ or not np.issubdtype(index.dtype, np.integer):
      raise TypeError(f"Take indices must be integers, got {index.dtype}")
    index = index.astype(np.int64)
    if index.size:
      lo, hi = int(index.min()), int(index.max())
      if lo < -size or hi >= size:
        bad = lo if lo < -size else hi
        raise IndexError(f"index {bad} is out of bounds for axis {self.axis} with size {size}")
    return np.where(index < 0, index + size, index)

  def __call__(self, trajectory):
    for key, val in trajectory.items():
      if key == "state":
        continue
      if hasattr(val, "materialize"):   # HostColumn, FrameStacks: stacked on the device, then index
        val = val.materialize()
      if isinstance(val, torch.Tensor):
        axis = self.axis if self.axis >= 0 else self.axis + val.ndim
        if not 0 <= axis < val.ndim:
          raise IndexError(f"axis {self.axis} is out of bounds for array of dimension {val.ndim}")
        index = self._checked(val.shape[axis])
        if index.ndim == 0:
          trajectory[key] = val.select(axis, int(index))
          continue
        flat = torch.from_numpy(np.ascontiguousarray(index.reshape(-1))).to(val.device)
        if axis == 0 and val.is_cuda and flat.numel() > 0:
          taken = _K.gather_rows(val.contiguous(), flat, 0, flat.numel())
        else:
          taken = torch.index_select(val, axis, flat)
        trajectory[key] = taken.reshape(tuple(val.shape[:axis]) + index.shape
                                        + tuple(val.shape[axis + 1:]))
      else:
        trajectory[key] = np.take(val, self.indices, axis=self.axis)
