"""Rows of a resident rollout column selected by a permutation slice — not materialised.

The reference's minibatch slice copies every selected observation row out of the rollout
(`derl/runners/onpolicy.py:57-62`) before the network reads it back (`derl/models.py:79-88,
117-123`).  With `IterateWithMinibatches(fused_gather=True)` the minibatch's `observations`
is a `RowSelection` instead: the NatureCNN stem kernels (K6t forward, K7t backward) take the
row indices and pull each 28 224-byte row straight out of the resident rollout (SURVEY §8f
rank 2), so the minibatch copy — one write and one extra read of every frame — never happens.
Anything else that touches the object gets the materialised tensor (`materialize()`, any
index other than a contiguous row slice, `.to()`, `.clone()`, `.cpu()`) — produced by the K2
gather kernel, so on a host tensor it fails loudly like every other derl_b200 op.
"""
import torch

from .. import ops  # noqa: F401

_K = torch.ops.derl_b200


class RowSelection:
  """`source[perm[start:start+count]]`, lazily."""

  def __init__(self, source, perm, start, count):
    if not (isinstance(source, torch.Tensor) and source.is_contiguous()):
      raise TypeError("RowSelection needs a contiguous tensor as its source")
    if perm.dtype != torch.int64 or perm.dim() != 1 or perm.device != source.device:
      raise TypeError("RowSelection needs a 1-D int64 permutation on the source's device")
    start, count = int(start), int(count)
    if start < 0 or count < 0 or start + count > perm.numel():
      raise ValueError(f"rows [{start}, {start + count}) outside a permutation of {perm.numel()}")
    self.source, self.perm, self.start, self.count = source, perm, start, count
    self._dense = None

  # ---- the bit of the tensor interface the runner wrappers, Trainer and the models read
  shape = property(lambda self: torch.Size((self.count,) + tuple(self.source.shape[1:])))
  ndim = property(lambda self: self.source.ndim)
  dtype = property(lambda self: self.source.dtype)
  device = property(lambda self: self.source.device)
  is_cuda = property(lambda self: self.source.is_cuda)

  def dim(self):
    return self.source.ndim

  def size(self, axis=None):
    return self.shape if axis is None else self.shape[axis]

  def is_contiguous(self):
    return True

  def __len__(self):
    return self.count

  @property
  def rows(self):
    """int64 [count] row indices into `source` (a view of the permutation)."""
    return self.perm[self.start:self.start + self.count]

  def materialize(self):
    if self._dense is None:
      self._dense = _K.gather_rows(self.source, self.perm, self.start, self.count)
    return self._dense

  def __getitem__(self, key):
    if isinstance(key, tuple) and len(key) == 0:
      return self
    if isinstance(key, slice) and key.step in (None, 1):
      lo, hi, _ = key.indices(self.count)
      return RowSelection(self.source, self.perm, self.start + lo, max(hi - lo, 0))
    return self.materialize()[key]

  def to(self, *args, **kwargs):
    return self.materialize().to(*args, **kwargs)

  def clone(self):
    return self.materialize().clone()

  def cpu(self):
    return self.materialize().cpu()

  def __repr__(self):
    return (f"RowSelection(source={tuple(self.source.shape)} {self.source.dtype}, "
            f"rows=perm[{self.start}:{self.start + self.count}])")


def dense(value):
  """`value` as an ordinary tensor (materialises a RowSelection)."""
  return value.materialize() if isinstance(value, RowSelection) else value
