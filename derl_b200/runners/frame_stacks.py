"""Atari rollouts stored as unique frames plus a per-sample stack index.

Consecutive frame stacks share k-1 of their k frames, so a stacked [T, N, 84, 84, 4] uint8
`observations` column (14.8 GB at 4096 envs x 128 steps) stores every frame four times.  The
format defined here stores each frame plane once:

  frames  uint8 [F, H, W]        the unique planes (7056 B each at 84x84, a multiple of 16 B)
  index   int32 [S, k]           (or [T, N, k] before MergeTimeBatch): for sample s, channel c,
                                 the id of the plane that channel is, so that
                                 stacked[s, y, x, c] == frames[index[s, c], y, x]   byte for byte.

It is exact by construction and makes no assumption about how an env wrapper stacks or resets:
stacks that share nothing simply compress to nothing.  The minibatch gather (K10,
torch.ops.derl_b200.gather_frame_stacks) rebuilds the stacked [count, H, W, k] rows bit for bit,
so everything downstream of the gather is unchanged.

  FrameStacks        the column: enough of the array interface for the runner wrappers
  FrameStackPacker   host packer, one env step [N, H, W, k] at a time (NumPy)
  DeviceFrameStackPacker  the same packing on the GPU (K11), planes in a device pool
  FrameStackRollout  one rollout's observations collected by EnvRunner(pack_frames=True)
  unpack             NumPy restatement of the format (frames, index) -> stacked array
"""
import numpy as np
import torch

from .. import ops  # noqa: F401  (registers torch.ops.derl_b200)
from .host_column import _side_stream

_K = torch.ops.derl_b200


def unpack(frames, index):
  """stacked[..., y, x, c] = frames[index[..., c], y, x] with NumPy (the format's definition)."""
  frames, index = np.asarray(frames), np.asarray(index)
  return np.moveaxis(frames[index], -3, -1)


def _as_tensor(value):
  return value if isinstance(value, torch.Tensor) else torch.from_numpy(np.asarray(value))


class FrameStacks:
  """A stacked uint8 [..., H, W, k] column held as unique planes + stack index.

  `shape` reports the stacked shape.  Arrays supplied by a caller are validated once, here
  (plane ids in [0, F), else IndexError); the gather kernel then trusts them.  A FrameStacks in
  host memory is uploaded by `to_device` (the runner wrappers do it) and gathered on the device.
  """

  def __init__(self, frames, index, validate=True):
    frames, index = _as_tensor(frames), _as_tensor(index)
    if frames.dtype != torch.uint8 or frames.dim() != 3:
      raise TypeError(f"frames must be uint8 [F, H, W], got {frames.dtype} {tuple(frames.shape)}")
    if index.dim() < 2 or index.dtype.is_floating_point or index.dtype == torch.bool:
      raise TypeError(f"index must be an integer [..., k] array, got {index.dtype} "
                      f"{tuple(index.shape)}")
    if frames.device != index.device:
      raise ValueError(f"frames ({frames.device}) and index ({index.device}) must share a device")
    if validate and index.numel() > 0:
      lo, hi = int(index.min()), int(index.max())
      if lo < 0 or hi >= frames.shape[0]:
        bad = lo if lo < 0 else hi
        raise IndexError(f"plane id {bad} is out of range for {frames.shape[0]} frames")
    self.frames = frames.contiguous()
    self.index = index.to(torch.int32).contiguous()
    self._ready = None   # event of a pending upload: the first gather waits on it

  # ---- just enough of the array interface for the runner wrappers
  shape = property(lambda self: torch.Size(tuple(self.index.shape[:-1])
                                           + tuple(self.frames.shape[1:])
                                           + (self.index.shape[-1],)))
  ndim = property(lambda self: self.index.dim() + 2)
  dtype = property(lambda self: self.frames.dtype)
  device = property(lambda self: self.frames.device)
  is_cuda = property(lambda self: self.frames.is_cuda)

  def __len__(self):
    return self.shape[0]

  @property
  def num_frames(self):
    return self.frames.shape[0]

  def reshape(self, *shape):
    """Reshape of the sample axes (the trailing H, W, k stay): MergeTimeBatch's [T, N] -> [S]."""
    shape = tuple(shape[0]) if len(shape) == 1 and isinstance(shape[0], (tuple, list)) else shape
    tail = tuple(self.shape[-3:])
    if tuple(shape[-3:]) != tail:
      raise ValueError(f"FrameStacks can only reshape its sample axes: {tuple(shape)} does not end "
                       f"with {tail}")
    out = FrameStacks(self.frames, self.index.reshape(tuple(shape[:-3]) + (tail[-1],)),
                      validate=False)
    out._ready = self._ready
    return out

  def to_device(self, device):
    """The same column on `device`: frames and index are copied with one asynchronous copy each
    on the shared per-device upload stream; the first gather waits for them."""
    device = torch.device(device)
    if self.is_cuda and self.device == device:
      return self
    frames = torch.empty(self.frames.shape, dtype=self.frames.dtype, device=device)
    index = torch.empty(self.index.shape, dtype=self.index.dtype, device=device)
    main = torch.cuda.current_stream(device)
    side = _side_stream(device)
    side.wait_stream(main)        # the allocations above belong to the main stream
    with torch.cuda.stream(side):
      frames.copy_(self.frames, non_blocking=True)
      index.copy_(self.index, non_blocking=True)
    frames.record_stream(side)
    index.record_stream(side)
    out = FrameStacks(frames, index, validate=False)
    out._ready = side.record_event()
    return out

  def _wait(self):
    if self._ready is not None:
      torch.cuda.current_stream(self.device).wait_event(self._ready)
      self._ready = None

  def gather(self, perm, start, count):
    """Stacked rows perm[start:start+count] as a [count, H, W, k] device tensor (K10)."""
    if not self.is_cuda:
      raise TypeError("FrameStacks.gather needs the column on the GPU (to_device first)")
    self._wait()
    return _K.gather_frame_stacks(self.frames, self.index.reshape(-1, self.index.shape[-1]), perm,
                                  int(start), int(count))

  def materialize(self):
    """The stacked tensor on the device (uploading first if the column is in host memory)."""
    src = self if self.is_cuda else self.to_device(torch.device("cuda",
                                                                torch.cuda.current_device()))
    samples = src.index[..., 0].numel()
    perm = torch.arange(samples, dtype=torch.int64, device=src.device)
    return src.gather(perm, 0, samples).reshape(self.shape)

  def __repr__(self):
    return (f"FrameStacks(shape={tuple(self.shape)}, frames={self.num_frames}, "
            f"device={self.device})")


def _pinned(shape, dtype, pinned=True):
  return torch.empty(shape, dtype=dtype, pin_memory=pinned)


def _next_channel_differs(a, b, k, scratch):
  """[N, k-1] bool: channel c of stack a[n] differs from channel c+1 of stack b[n] somewhere.
  a, b: [N, P*k] byte views of NHWC stacks.  One contiguous compare of every byte with the next
  byte, then an OR over the P pixels per channel by repeated halving (each pass contiguous)."""
  np.not_equal(a[:, :-1], b[:, 1:], out=scratch[:, :-1])
  scratch[:, -1] = False
  x = scratch.view(np.uint8).reshape(a.shape[0], -1, k)
  p = x.shape[1]
  while p > 1:
    h = p // 2
    np.bitwise_or(x[:, :h], x[:, p - h:p], out=x[:, :h])
    p -= h
  return x[:, 0, :k - 1].astype(bool)


class FrameStackPacker:
  """Packs a stream of stacked steps obs_t ([N, H, W, k] uint8) into unique planes.

  Channel k-1 is always a new plane.  For c = k-2 ... 0, in order, channel c reuses the id of
  channel c+1 of the same stack if their bytes are equal (covers a reset stack [f, f, f, f]),
  else the id of channel c+1 of the same env's previous step if those bytes are equal, else it
  becomes a new plane.  Reuse happens only on byte equality, so unpacking is exact whatever the
  env does; on the usual stacking wrappers a rollout stores T*N + N*(k-1) planes.

  The planes live in one growing uint8 [capacity, H, W] array (`pinned=True`: page-locked torch
  memory, so that they can be copied to a GPU asynchronously).
  """

  def __init__(self, capacity=0, pinned=False):
    self.capacity, self.pinned = int(capacity), pinned
    self.count = 0
    self._store = None        # torch uint8 [capacity, H, W]
    self._prev, self._prev_ids = None, None
    self._diff = None         # bool scratch of one step's size

  @property
  def frames(self):
    """torch uint8 [count, H, W]: the planes packed so far (a view of the store)."""
    return self._store[:self.count]

  def _reserve(self, need, plane_shape):
    if self._store is not None and need <= self._store.shape[0]:
      return
    cap = max(need, self.capacity, int(self._store.shape[0] * 1.5) if self._store is not None else 0)
    store = _pinned((cap,) + plane_shape, torch.uint8, self.pinned)
    if self._store is not None and self.count:
      store[:self.count].copy_(self._store[:self.count])
    self._store, self.capacity = store, cap

  def pack(self, obs):
    """Appends one step; returns its int32 [N, k] plane ids."""
    obs = np.ascontiguousarray(obs)
    if obs.dtype != np.uint8 or obs.ndim != 4:
      raise TypeError(f"expected uint8 [N, H, W, k] observations, got {obs.dtype} {obs.shape}")
    nenvs, k = obs.shape[0], obs.shape[-1]
    if self._prev is not None and self._prev.shape != obs.shape:
      raise ValueError(f"step shape {obs.shape} differs from the previous step's {self._prev.shape}")
    # same[:, c]: channel c == channel c+1 of the stack; prev[:, c]: == channel c+1 one step back
    flat = obs.reshape(nenvs, -1)
    if self._diff is None or self._diff.shape != flat.shape:
      self._diff = np.empty(flat.shape, dtype=bool)
    same = ~_next_channel_differs(flat, flat, k, self._diff)
    if self._prev is not None:
      prev = ~_next_channel_differs(flat, self._prev.reshape(nenvs, -1), k, self._diff)
    else:
      prev = np.zeros_like(same)
    new = ~same & ~prev
    self._reserve(self.count + nenvs + int(new.sum()), obs.shape[1:3])
    planes = self._store.numpy()
    ids = np.empty((nenvs, k), dtype=np.int32)
    ids[:, k - 1] = np.arange(self.count, self.count + nenvs, dtype=np.int32)
    planes[self.count:self.count + nenvs] = obs[..., k - 1]
    self.count += nenvs
    for c in range(k - 2, -1, -1):
      col = ids[:, c + 1].copy()
      if self._prev_ids is not None:
        col[~same[:, c]] = self._prev_ids[~same[:, c], c + 1]
      fresh = np.flatnonzero(new[:, c])
      col[fresh] = np.arange(self.count, self.count + fresh.size, dtype=np.int32)
      planes[self.count:self.count + fresh.size] = obs[fresh, :, :, c]
      self.count += fresh.size
      ids[:, c] = col
    self._prev, self._prev_ids = obs.copy(), ids
    return ids


class DeviceFrameStackPacker:
  """FrameStackPacker on the GPU (K11, torch.ops.derl_b200.pack_frame_stacks): the same ids and
  plane bytes for the same steps, with the planes in a device pool and no host synchronisation
  per step.

  `pack(obs, out=None)` takes a NumPy [N, H, W, k] uint8 step or a CUDA uint8 tensor of that
  shape and writes the int32 [N, k] ids into `out` (a device row, e.g. one row of a rollout's
  index) or returns them as a new device tensor.  A NumPy step goes through one of two pinned
  staging slots (rewritten only once the slot's previous copy has completed) and an asynchronous
  copy into one of two device stack buffers, which hold the current and the previous step; a CUDA
  step is copied device to device, since the caller may reuse its tensor.  Everything runs on the
  current stream, and the buffers are allocated once and reused across rollouts.

  The plane count stays on the device.  After each step it is copied into a pinned per-step ring
  and an event is recorded; before a step the pool is grown (stream-ordered device copy) if the
  latest count known to have arrived, plus N*k planes for every step since, could exceed it.
  `reset()` starts a rollout with a fresh pool of `horizon*N + N*(k-1)` planes (the standard
  stacking case) plus N*k headroom; `finish()` reads the count once, raises RuntimeError if a step
  overflowed the pool, and returns the planes [count, H, W].
  """

  def __init__(self, device, horizon):
    self.device = torch.device(device)
    self.horizon = max(int(horizon), 1)
    self._shape = None
    self._stacks = None       # device uint8 [2, N, H, W, k]: current and previous step
    self._staging = None      # pinned uint8 [2, N, H, W, k]
    self._staged = [None, None]   # event of each staging slot's last copy
    self._state = torch.zeros(2, dtype=torch.int64, device=self.device)
    self._counts = torch.zeros(self.horizon, dtype=torch.int64, pin_memory=True)
    self._count_events = [torch.cuda.Event() for _ in range(self.horizon)]
    self.reset()

  def reset(self):
    """Start a rollout: no previous step, count 0, a new pool (the old one now belongs to the
    FrameStacks that `finish` returned)."""
    self._pool, self._prev_ids = None, None
    self._steps = 0
    self._known = (-1, 0)     # (step, plane count after it) last read from the pinned ring
    self._pending = []        # steps whose count copy has not been read yet, oldest first
    self._state.zero_()

  def _buffers(self, shape):
    if self._shape == shape:
      return
    if self._steps:
      raise ValueError(f"step shape {shape} differs from the previous step's {self._shape}")
    self._shape = shape
    self._stacks = torch.empty((2,) + shape, dtype=torch.uint8, device=self.device)
    self._staging, self._staged = None, [None, None]

  def _bound(self, nk):
    """Upper bound of the plane count after the step about to be packed."""
    while self._pending and self._count_events[self._pending[0] % self.horizon].query():
      step = self._pending.pop(0)
      self._known = (step, int(self._counts[step % self.horizon]))
    step, count = self._known
    return count + (self._steps - step) * nk

  def _reserve(self, need, nk):
    cap = 0 if self._pool is None else self._pool.shape[0]
    if need <= cap:
      return
    if self._pool is None:
      nenvs, k = self._shape[0], self._shape[-1]
      need = max(need, self.horizon * nenvs + nenvs * (k - 1) + nk)
    grown = torch.empty((max(need, cap * 3 // 2),) + self._shape[1:3], dtype=torch.uint8,
                        device=self.device)
    if cap:
      used = min(cap, self._bound(nk) - nk)   # the count before this step is at most this
      grown[:used].copy_(self._pool[:used])
    self._pool = grown

  def pack(self, obs, out=None):
    """Appends one step; returns its int32 [N, k] plane ids (a device tensor, `out` if given)."""
    if isinstance(obs, torch.Tensor) and obs.is_cuda:
      src = obs
    else:
      src = np.ascontiguousarray(obs)
    if src.dtype not in (np.uint8, torch.uint8) or src.ndim != 4:
      raise TypeError(f"expected uint8 [N, H, W, k] observations, got {src.dtype} "
                      f"{tuple(src.shape)}")
    shape = tuple(src.shape)
    self._buffers(shape)
    nenvs, k = shape[0], shape[-1]
    slot = self._steps % 2
    cur = self._stacks[slot]
    if isinstance(src, torch.Tensor):
      cur.copy_(src)
    else:
      if self._staging is None:
        self._staging = torch.empty((2,) + shape, dtype=torch.uint8, pin_memory=True)
      if self._staged[slot] is not None:
        self._staged[slot].synchronize()
      np.copyto(self._staging[slot].numpy(), src)
      cur.copy_(self._staging[slot], non_blocking=True)
      self._staged[slot] = torch.cuda.current_stream(self.device).record_event()
    nk = nenvs * k
    self._reserve(self._bound(nk), nk)
    if out is not None and self._prev_ids is not None and \
        out.data_ptr() == self._prev_ids.data_ptr():
      raise ValueError("out must not be the previous step's ids: the kernel reads them")
    ids = out if out is not None else torch.empty((nenvs, k), dtype=torch.int32,
                                                  device=self.device)
    prev = self._stacks[1 - slot] if self._prev_ids is not None else None
    _K.pack_frame_stacks(cur, prev, self._prev_ids, self._pool, self._state, ids)
    ring = self._steps % self.horizon
    if len(self._pending) == self.horizon:     # the ring slot is still in flight
      self._count_events[ring].synchronize()
      self._bound(nk)
    self._counts[ring].copy_(self._state[0], non_blocking=True)
    self._count_events[ring].record(torch.cuda.current_stream(self.device))
    self._pending.append(self._steps)
    self._prev_ids = ids
    self._steps += 1
    return ids

  def finish(self):
    """The planes packed since `reset`: uint8 [count, H, W] on the device (one host read)."""
    count, overflow = self._state.tolist()
    if overflow:
      raise RuntimeError("frame-plane pool overflowed: a step needed more planes than the pool "
                         "holds, so this rollout's frames are incomplete")
    if self._pool is None:
      raise RuntimeError("nothing was packed since reset()")
    return self._pool[:count]


class FrameStackRollout:
  """`observations` of one EnvRunner rollout, packed as it is collected.

  device None: FrameStackPacker packs on the host; planes and index accumulate in host memory
  (pinned when CUDA is available) and `finish` returns a host FrameStacks (TransformInteractions
  uploads it).  device given: a DeviceFrameStackPacker (`packer`, reused across rollouts when the
  caller passes one) packs on the GPU, writing every step's ids straight into the device index;
  `finish` returns a device FrameStacks.
  """

  def __init__(self, horizon, device=None, packer=None):
    self.horizon = horizon
    self.device = None if device is None else torch.device(device)
    self.packer, self.index = packer, None
    self._dev_index = None

  def put(self, step, obs):
    if not isinstance(obs, torch.Tensor):
      obs = np.asarray(obs)
    if self.device is not None:
      if self._dev_index is None:
        nenvs, k = obs.shape[0], obs.shape[-1]
        if self.packer is None:
          self.packer = DeviceFrameStackPacker(self.device, self.horizon)
        self.packer.reset()
        self._dev_index = torch.empty((self.horizon, nenvs, k), dtype=torch.int32,
                                      device=self.device)
      self.packer.pack(obs, out=self._dev_index[step])
      return
    if self.packer is None:
      nenvs, k = obs.shape[0], obs.shape[-1]
      pinned = torch.cuda.is_available()   # page-locked only where a GPU will read it
      self.packer = FrameStackPacker(self.horizon * nenvs + nenvs * (k - 1), pinned=pinned)
      self.index = _pinned((self.horizon, nenvs, k), torch.int32, pinned)
    self.index[step].numpy()[...] = self.packer.pack(obs)

  def finish(self):
    if self.device is None:
      return FrameStacks(self.packer.frames, self.index, validate=False)
    return FrameStacks(self.packer.finish(), self._dev_index, validate=False)
