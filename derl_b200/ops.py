"""torch.library custom ops (`torch.ops.derl_b200.*`) over the C ABI in include/derl_b200.h.

PyTorch is plumbing here: it owns device memory (caching allocator) and the current stream;
every op body is a pointer hand-off to libderl_b200.so.  The ops are registered for CUDA
only — called with CPU tensors the dispatcher raises, by design (no CPU fallback).
"""
import ctypes
import os
from typing import List, Optional, Tuple

import torch
from torch import Tensor

from . import _lib

_lib.load()  # fail at import time, loudly, if the CUDA library is absent

_VP = ctypes.c_void_p


def _stream(t):
  return _VP(torch.cuda.current_stream(t.device).cuda_stream)


def _p(t):
  return _VP(t.data_ptr()) if t is not None and t.numel() > 0 else _VP(None)


def _need(cond, msg):
  if not cond:
    raise ValueError(msg)


# DERL_B200_CHECK_INDICES=1: validate gather indices and categorical action indices on the host
# (one device sync per call).  Off by default: the runner wrappers only ever pass permutations
# they built themselves, `Take` validates its (host) indices before any launch, and actions come
# out of the policy's own sampler.
CHECK_INDICES = os.environ.get("DERL_B200_CHECK_INDICES", "0") not in ("", "0")


def _check_indices(perm, start, count, nrows):
  if CHECK_INDICES and count > 0:
    window = perm[start:start + count]
    lo, hi = int(window.min()), int(window.max())
    if lo < 0 or hi >= nrows:
      raise IndexError(f"gather index out of range: [{lo}, {hi}] not within [0, {nrows})")


def _dense(t, name, dtypes=None):
  _need(t.is_contiguous(), f"{name} must be contiguous")
  if dtypes is not None:
    _need(t.dtype in dtypes, f"{name} must have dtype in {dtypes}, got {t.dtype}")
  return t


# When set to a list, every library call appends (kernel name, start event, end event)
# recorded on the launching stream: bench.py reads per-kernel device times from it.
PROFILE = None


class _device_of:
  """Make the tensor's device current for the duration of a library call."""

  def __init__(self, t, name=None):
    self.idx = t.device.index
    self.prev = None
    self.name = name
    self.start = None

  def __enter__(self):
    cur = torch.cuda.current_device()
    if self.idx is not None and cur != self.idx:
      self.prev = cur
      torch.cuda.set_device(self.idx)
    if PROFILE is not None and self.name is not None:
      self.start = torch.cuda.Event(enable_timing=True)
      self.start.record()

  def __exit__(self, *exc):
    if self.start is not None:
      end = torch.cuda.Event(enable_timing=True)
      end.record()
      PROFILE.append((self.name, self.start, end))
    if self.prev is not None:
      torch.cuda.set_device(self.prev)


# --------------------------------------------------------------------------- K1: GAE
@torch.library.custom_op("derl_b200::gae", mutates_args=(), device_types="cuda")
def gae(rewards: Tensor, values: Tensor, resets: Tensor, last_value: Tensor, gamma: float,
        lambda_: float, want_stats: bool = False,
        variant: int = 0) -> Tuple[Tensor, Tensor, Tensor]:
  """(advantages [T,N] f32, value_targets [T,N] f32, stats f64[3] or empty)."""
  _need(values.dim() == 2, f"values must be [T, N], got {tuple(values.shape)}")
  nsteps, nenvs = values.shape
  _dense(rewards, "rewards", (torch.float32, torch.float64))
  _dense(values, "values", (torch.float32,))
  _dense(resets, "resets", (torch.bool, torch.uint8))
  _dense(last_value, "last_value", (torch.float32,))
  _need(rewards.shape == values.shape and resets.shape == values.shape,
        f"rewards {tuple(rewards.shape)}, resets {tuple(resets.shape)} and values "
        f"{tuple(values.shape)} must have the same [T, N] shape")
  _need(last_value.numel() == nenvs, f"last_value must have {nenvs} elements")
  _need(nsteps >= 1 and nenvs >= 1, "empty rollout")
  lib = _lib.load()
  adv = torch.empty_like(values)
  targets = torch.empty_like(values)
  if want_stats:
    stats = torch.empty(_lib.GAE_STATS, dtype=torch.float64, device=values.device)
    ws_bytes = lib.derl_b200_gae_workspace_bytes(nsteps, nenvs)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=values.device)
  else:
    stats = torch.empty(0, dtype=torch.float64, device=values.device)
    ws_bytes, ws = 0, None
  with _device_of(values, "gae"):
    _lib.check(lib.derl_b200_gae(_p(rewards), int(rewards.dtype == torch.float64), _p(values),
                                 _p(resets), _p(last_value), nsteps, nenvs, float(gamma),
                                 float(lambda_), _p(adv), _p(targets), _p(stats), _p(ws),
                                 ws_bytes, int(variant), _stream(values)), "gae")
  return adv, targets, stats


@gae.register_fake
def _(rewards, values, resets, last_value, gamma, lambda_, want_stats=False, variant=0):
  stats = values.new_empty(_lib.GAE_STATS if want_stats else 0, dtype=torch.float64)
  return torch.empty_like(values), torch.empty_like(values), stats


@torch.library.custom_op("derl_b200::moments", mutates_args=(), device_types="cuda")
def moments(x: Tensor) -> Tensor:
  """float64 {sum, sum of squares, count} of a float32 tensor."""
  _dense(x, "x", (torch.float32,))
  _need(x.numel() >= 1, "moments of an empty tensor")
  lib = _lib.load()
  stats = torch.empty(3, dtype=torch.float64, device=x.device)
  ws_bytes = lib.derl_b200_moments_workspace_bytes(x.numel())
  ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
  with _device_of(x, "moments"):
    _lib.check(lib.derl_b200_moments(_p(x), x.numel(), _p(stats), _p(ws), ws_bytes, _stream(x)),
               "moments")
  return stats


@moments.register_fake
def _(x):
  return x.new_empty(3, dtype=torch.float64)


@torch.library.custom_op("derl_b200::normalize", mutates_args=(), device_types="cuda")
def normalize(x: Tensor, stats: Tensor, epsilon: float) -> Tensor:
  """(x - mean) / (std_pop + epsilon) from device-resident {sum, sumsq, count}."""
  _dense(x, "x", (torch.float32,))
  _dense(stats, "stats", (torch.float64,))
  _need(stats.numel() >= 3 and x.numel() >= 1, "normalize: bad stats or empty input")
  out = torch.empty_like(x)
  with _device_of(x, "normalize"):
    _lib.check(_lib.load().derl_b200_normalize(_p(x), _p(out), x.numel(), _p(stats),
                                               float(epsilon), _stream(x)), "normalize")
  return out


@normalize.register_fake
def _(x, stats, epsilon):
  return torch.empty_like(x)


# --------------------------------------------------------------------------- K2: gather
@torch.library.custom_op("derl_b200::gather_rows", mutates_args=(), device_types="cuda")
def gather_rows(src: Tensor, perm: Tensor, start: int, count: int) -> Tensor:
  """out[j] = src[perm[start + j]] along dim 0 (bit-exact copy of whole rows)."""
  _dense(src, "src")
  _dense(perm, "perm", (torch.int64,))
  _need(src.dim() >= 1 and src.shape[0] >= 1, "src must have at least one row")
  _need(0 <= start and 0 <= count and start + count <= perm.numel(),
        f"window [{start}, {start + count}) outside perm of {perm.numel()}")
  _check_indices(perm, start, count, src.shape[0])
  out = src.new_empty((count,) + tuple(src.shape[1:]))
  row_bytes = src[0].numel() * src.element_size()
  if count == 0 or row_bytes == 0:
    return out
  with _device_of(src, "gather_rows"):
    _lib.check(_lib.load().derl_b200_gather_rows(_p(src), src.shape[0], row_bytes, _p(perm),
                                                 start, count, _p(out), _stream(src)),
               "gather_rows")
  return out


@gather_rows.register_fake
def _(src, perm, start, count):
  return src.new_empty((count,) + tuple(src.shape[1:]))


@torch.library.custom_op("derl_b200::gather_rows_upload", mutates_args=("resident",),
                         device_types="cuda")
def gather_rows_upload(host_ptr: int, perm: Tensor, start: int, count: int, resident: Tensor,
                       max_ctas: int = 8) -> Tensor:
  """First-epoch upload gather: rows perm[start:start+count] of a column living in PINNED HOST
  memory at `host_ptr` (same shape/dtype as `resident`) are copied once over PCIe and written
  both to the returned minibatch tensor and to `resident[perm[...]]`."""
  _dense(resident, "resident")
  _dense(perm, "perm", (torch.int64,))
  _need(host_ptr != 0 and host_ptr % 16 == 0, "host pointer must be non-null and 16-byte aligned")
  _need(resident.dim() >= 1 and resident.shape[0] >= 1, "resident must have at least one row")
  _need(0 <= start and 0 <= count and start + count <= perm.numel(),
        f"window [{start}, {start + count}) outside perm of {perm.numel()}")
  out = resident.new_empty((count,) + tuple(resident.shape[1:]))
  row_bytes = resident[0].numel() * resident.element_size()
  if count == 0:
    return out
  with _device_of(resident, "gather_rows_upload"):
    _lib.check(_lib.load().derl_b200_gather_rows_upload(
        _VP(host_ptr), resident.shape[0], row_bytes, _p(perm), start, count, _p(out),
        _p(resident), int(max_ctas), _stream(resident)), "gather_rows_upload")
  return out


@gather_rows_upload.register_fake
def _(host_ptr, perm, start, count, resident, max_ctas=8):
  return resident.new_empty((count,) + tuple(resident.shape[1:]))


# --------------------------------------------------------------------------- K10: frame stacks
@torch.library.custom_op("derl_b200::gather_frame_stacks", mutates_args=(), device_types="cuda")
def gather_frame_stacks(frames: Tensor, index: Tensor, perm: Tensor, start: int,
                        count: int) -> Tensor:
  """out[j, y, x, c] = frames[index[perm[start + j], c], y, x]: the stacked [count, H, W, k]
  uint8 minibatch, rebuilt from unique planes (runners/frame_stacks.py).  Plane ids are not
  checked here; FrameStacks validates caller-supplied ones when it is built."""
  _dense(frames, "frames", (torch.uint8,))
  _dense(index, "index", (torch.int32,))
  _dense(perm, "perm", (torch.int64,))
  _need(frames.dim() == 3 and frames.shape[0] >= 1, f"frames must be [F, H, W], got "
        f"{tuple(frames.shape)}")
  _need(index.dim() == 2 and index.shape[0] >= 1 and index.shape[1] >= 1,
        f"index must be [S, k], got {tuple(index.shape)}")
  _need(frames.device == index.device == perm.device, "frames, index and perm must share a device")
  _need(0 <= start and 0 <= count and start + count <= perm.numel(),
        f"window [{start}, {start + count}) outside perm of {perm.numel()}")
  _check_indices(perm, start, count, index.shape[0])
  n_frames, height, width = frames.shape
  n_samples, k = index.shape
  out = frames.new_empty((count, height, width, k))
  if count == 0:
    return out
  with _device_of(frames, "gather_frame_stacks"):
    _lib.check(_lib.load().derl_b200_gather_frame_stacks(
        _p(frames), n_frames, height, width, _p(index), n_samples, k, _p(perm), start, count,
        _p(out), _stream(frames)), "gather_frame_stacks")
  return out


@gather_frame_stacks.register_fake
def _(frames, index, perm, start, count):
  return frames.new_empty((count,) + tuple(frames.shape[1:]) + (index.shape[1],))


# --------------------------------------------------------------------------- K11: frame packing
@torch.library.custom_op("derl_b200::pack_frame_stacks", mutates_args=("pool", "state", "ids"),
                         device_types="cuda")
def pack_frame_stacks(stacks: Tensor, prev_stacks: Optional[Tensor], prev_ids: Optional[Tensor],
                      pool: Tensor, state: Tensor, ids: Tensor) -> None:
  """Packs one step of stacks [N, H, W, k] uint8 into the planes pool [capacity, H, W] exactly as
  FrameStackPacker.pack does: writes the step's int32 [N, k] plane ids into `ids`, appends the new
  planes to `pool` and advances state = int64 {plane count, overflow flag}, all on the device.
  prev_stacks / prev_ids are the previous step's stacks and ids (None on a rollout's first step).
  A step that would not fit in `pool` sets the (sticky) overflow flag instead of writing."""
  _dense(stacks, "stacks", (torch.uint8,))
  _dense(pool, "pool", (torch.uint8,))
  _dense(state, "state", (torch.int64,))
  _dense(ids, "ids", (torch.int32,))
  _need(stacks.dim() == 4, f"stacks must be [N, H, W, k], got {tuple(stacks.shape)}")
  nenvs, height, width, k = stacks.shape
  _need(pool.dim() == 3 and tuple(pool.shape[1:]) == (height, width),
        f"pool must be [capacity, {height}, {width}], got {tuple(pool.shape)}")
  _need(state.numel() == 2, "state must hold {count, overflow}")
  _need(tuple(ids.shape) == (nenvs, k), f"ids must be [{nenvs}, {k}], got {tuple(ids.shape)}")
  _need((prev_stacks is None) == (prev_ids is None), "prev_stacks and prev_ids go together")
  if prev_stacks is not None:
    _dense(prev_stacks, "prev_stacks", (torch.uint8,))
    _dense(prev_ids, "prev_ids", (torch.int32,))
    _need(prev_stacks.shape == stacks.shape and tuple(prev_ids.shape) == (nenvs, k),
          "the previous step must have the same shape as this one")
  tensors = [stacks, pool, state, ids] + ([prev_stacks, prev_ids] if prev_stacks is not None else [])
  _need(all(t.device == stacks.device for t in tensors), "all tensors must share a device")
  lib = _lib.load()
  ws_bytes = lib.derl_b200_pack_frame_stacks_workspace_bytes(nenvs, k)
  ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=stacks.device)
  with _device_of(stacks, "pack_frame_stacks"):
    _lib.check(lib.derl_b200_pack_frame_stacks(
        _p(stacks), _p(prev_stacks), _p(prev_ids), nenvs, height, width, k, _p(pool),
        pool.shape[0], _p(state), _p(ids), _p(ws), ws_bytes, _stream(stacks)), "pack_frame_stacks")


@pack_frame_stacks.register_fake
def _(stacks, prev_stacks, prev_ids, pool, state, ids):
  return None


@torch.library.custom_op("derl_b200::gather_columns", mutates_args=(), device_types="cuda")
def gather_columns(columns: List[Tensor], perm: Tensor, start: int, count: int,
                   moments_col: int = -1) -> List[Tensor]:
  """Gathers every narrow column in one launch; the returned list has one extra trailing
  entry: float64 {sum, sumsq, count} of columns[moments_col] over the gathered rows (empty
  when moments_col < 0)."""
  ncol = len(columns)
  _need(1 <= ncol <= _lib.MAX_COLUMNS, f"between 1 and {_lib.MAX_COLUMNS} columns, got {ncol}")
  _dense(perm, "perm", (torch.int64,))
  _need(0 <= start and 0 <= count and start + count <= perm.numel(),
        f"window [{start}, {start + count}) outside perm of {perm.numel()}")
  dev = columns[0].device
  _check_indices(perm, start, count, min(c.shape[0] for c in columns))
  outs, row_bytes = [], []
  for i, col in enumerate(columns):
    _dense(col, f"columns[{i}]")
    _need(col.dim() >= 1 and col.shape[0] >= 1, f"columns[{i}] has no rows")
    outs.append(col.new_empty((count,) + tuple(col.shape[1:])))
    row_bytes.append(col[0].numel() * col.element_size())
    _need(row_bytes[-1] >= 1, f"columns[{i}] has empty rows")
  lib = _lib.load()
  if moments_col >= 0:
    _need(columns[moments_col].dtype == torch.float32 and row_bytes[moments_col] == 4,
          "moments column must be float32 with one element per row")
    stats = torch.empty(3, dtype=torch.float64, device=dev)
    ws_bytes = lib.derl_b200_moments_workspace_bytes(count)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
  else:
    stats, ws_bytes, ws = torch.empty(0, dtype=torch.float64, device=dev), 0, None
  if count > 0:
    srcs = (_VP * ncol)(*[c.data_ptr() for c in columns])
    dsts = (_VP * ncol)(*[o.data_ptr() for o in outs])
    rbs = (ctypes.c_int64 * ncol)(*row_bytes)
    with _device_of(columns[0], "gather_columns"):
      _lib.check(lib.derl_b200_gather_columns(ncol, srcs, rbs, dsts, _p(perm), start, count,
                                              int(moments_col), _p(stats), _p(ws), ws_bytes,
                                              _stream(columns[0])), "gather_columns")
  return outs + [stats]


@gather_columns.register_fake
def _(columns, perm, start, count, moments_col=-1):
  outs = [c.new_empty((count,) + tuple(c.shape[1:])) for c in columns]
  return outs + [columns[0].new_empty(3 if moments_col >= 0 else 0, dtype=torch.float64)]


# --------------------------------------------------------------------------- K4: frames
_S2D_DTYPES = {torch.float32: 0, torch.bfloat16: 1, torch.float16: 2}


@torch.library.custom_op("derl_b200::frames_to_s2d", mutates_args=(), device_types="cuda")
def frames_to_s2d(frames: Tensor, block: int, dtype: torch.dtype, divisor: float) -> Tensor:
  """uint8 NHWC frames [B,H,W,C] -> [B, H/block, W/block, block*block*C] of `dtype`, values
  divided by `divisor` in float32 (space-to-depth + cast + scale in one pass)."""
  _dense(frames, "frames", (torch.uint8,))
  _need(frames.dim() == 4, f"frames must be [B, H, W, C], got {tuple(frames.shape)}")
  _need(dtype in _S2D_DTYPES, f"dtype must be one of {list(_S2D_DTYPES)}")
  batch, height, width, chans = frames.shape
  _need(block * chans == 16 and height % block == 0 and width % block == 0,
        f"frames_to_s2d needs block*C == 16 and H, W multiples of block (got {tuple(frames.shape)}, "
        f"block={block})")
  out = torch.empty((batch, height // block, width // block, block * block * chans), dtype=dtype,
                    device=frames.device)
  with _device_of(frames, "frames_to_s2d"):
    _lib.check(_lib.load().derl_b200_frames_to_s2d(_p(frames), batch, height, width, chans, block,
                                                   _p(out), _S2D_DTYPES[dtype], float(divisor),
                                                   _stream(frames)), "frames_to_s2d")
  return out


@frames_to_s2d.register_fake
def _(frames, block, dtype, divisor):
  batch, height, width, chans = frames.shape
  return frames.new_empty((batch, height // block, width // block, block * block * chans),
                          dtype=dtype)


@torch.library.custom_op("derl_b200::space_to_depth", mutates_args=(), device_types="cuda")
def space_to_depth(x: Tensor, block: int, inverse: bool = False) -> Tensor:
  """NHWC-contiguous [B,H,W,C] -> [B,H/block,W/block,block*block*C] (inverse: the other way)."""
  _dense(x, "x")
  _need(x.dim() == 4, f"expected [B, H, W, C], got {tuple(x.shape)}")
  batch, height, width, chans = x.shape
  if inverse:
    _need(chans % (block * block) == 0, "channels must be divisible by block^2")
    chans //= block * block
    height, width = height * block, width * block
  _need(height % block == 0 and width % block == 0 and (chans * x.element_size()) % 16 == 0,
        f"space_to_depth: unsupported shape {tuple(x.shape)} for block {block}")
  shape = (batch, height, width, chans) if inverse else \
      (batch, height // block, width // block, block * block * chans)
  out = x.new_empty(shape)
  with _device_of(x, "space_to_depth"):
    _lib.check(_lib.load().derl_b200_space_to_depth(_p(x), batch, height, width,
                                                    chans * x.element_size(), block,
                                                    int(inverse), _p(out), _stream(x)),
               "space_to_depth")
  return out


@space_to_depth.register_fake
def _(x, block, inverse=False):
  batch, height, width, chans = x.shape
  if inverse:
    return x.new_empty((batch, height * block, width * block, chans // (block * block)))
  return x.new_empty((batch, height // block, width // block, block * block * chans))


def _s2d_setup(ctx, inputs, output):
  ctx.block, ctx.inverse = inputs[1], inputs[2]


def _s2d_backward(ctx, grad):
  return torch.ops.derl_b200.space_to_depth(grad.contiguous(), ctx.block, not ctx.inverse), \
      None, None


space_to_depth.register_autograd(_s2d_backward, setup_context=_s2d_setup)


# --------------------------------------------------------------------------- K6t: stem conv
@torch.library.custom_op("derl_b200::stem_conv_relu", mutates_args=(), device_types="cuda")
def stem_conv_relu(frames: Tensor, weight: Tensor, bias: Tensor, dtype: torch.dtype,
                   out_block: int = 1, rows: Optional[Tensor] = None) -> Tensor:
  """relu(conv2d(frames/255, weight, bias, stride 4)) for uint8 NHWC frames [B,84,84,4] and the
  Atari stem weight [32,4,8,8] (K6t); returns the channels-last activation [B,20,20,32], or its
  space-to-depth(2) arrangement [B,10,10,128] when out_block == 2.  A bfloat16 output is the
  float32 one rounded to nearest even.  `rows` (int64 [B']): the
  batch is frames[rows] — the minibatch gather fused into the layer, nothing materialised."""
  _dense(frames, "frames", (torch.uint8,))
  batch = _check_rows(frames, rows)
  _need(tuple(frames.shape[1:]) == (84, 84, 4), f"frames must be [B,84,84,4], got {tuple(frames.shape)}")
  _dense(weight, "weight", (torch.float32,))
  _dense(bias, "bias", (torch.float32,))
  _need(tuple(weight.shape) == (32, 4, 8, 8) and tuple(bias.shape) == (32,),
        "stem_conv_relu is specialised to weight [32,4,8,8], bias [32]")
  _need(dtype in (torch.float32, torch.bfloat16), "dtype must be float32 or bfloat16")
  _need(out_block in (1, 2), "out_block must be 1 or 2")
  shape = (batch, 20, 20, 32) if out_block == 1 else (batch, 10, 10, 128)
  out = torch.empty(shape, dtype=dtype, device=frames.device)
  with _device_of(frames, "stem_conv_relu"):
    _lib.check(_lib.load().derl_b200_stem_conv_relu(
        _p(frames), _p(rows) if rows is not None else None, batch, _p(weight), _p(bias), _p(out),
        _S2D_DTYPES[dtype], out_block, _stream(frames)), "stem_conv_relu")
  return out


def _check_rows(frames, rows):
  """Batch size of a (frames, rows) pair; rows must be a dense int64 vector on frames' device."""
  if rows is None:
    return frames.shape[0]
  _dense(rows, "rows", (torch.int64,))
  _need(rows.dim() == 1 and rows.device == frames.device, "rows must be a 1-D tensor on the "
        "frames' device")
  if CHECK_INDICES and rows.numel():
    lo, hi = int(rows.min()), int(rows.max())
    _need(0 <= lo and hi < frames.shape[0], f"rows out of range [0, {frames.shape[0]})")
  return rows.numel()


@stem_conv_relu.register_fake
def _(frames, weight, bias, dtype, out_block=1, rows=None):
  batch = frames.shape[0] if rows is None else rows.shape[0]
  shape = (batch, 20, 20, 32) if out_block == 1 else (batch, 10, 10, 128)
  return frames.new_empty(shape, dtype=dtype)


@torch.library.custom_op("derl_b200::stem_conv_relu_mask", mutates_args=(), device_types="cuda")
def stem_conv_relu_mask(frames: Tensor, weight: Tensor, bias: Tensor, out_block: int = 1,
                        rows: Optional[Tensor] = None) -> Tuple[Tensor, Tensor]:
  """K6t (tcgen05 + tensor memory): float32 `stem_conv_relu` that also returns the ReLU mask,
  int32 [B, 14, 32]: bit l of word (t, c) = (channel c at padded pixel 21 oy + ox = 32 t + l is
  > 0) — what `stem_backward_masked` reads instead of the 32x larger float32 activation."""
  _dense(frames, "frames", (torch.uint8,))
  batch = _check_rows(frames, rows)
  _need(tuple(frames.shape[1:]) == (84, 84, 4), f"frames must be [B,84,84,4], got {tuple(frames.shape)}")
  _dense(weight, "weight", (torch.float32,))
  _dense(bias, "bias", (torch.float32,))
  _need(tuple(weight.shape) == (32, 4, 8, 8) and tuple(bias.shape) == (32,),
        "stem_conv_relu_mask is specialised to weight [32,4,8,8], bias [32]")
  _need(out_block in (1, 2), "out_block must be 1 or 2")
  shape = (batch, 20, 20, 32) if out_block == 1 else (batch, 10, 10, 128)
  out = torch.empty(shape, dtype=torch.float32, device=frames.device)
  mask = torch.empty((batch, 14, 32), dtype=torch.int32, device=frames.device)
  with _device_of(frames, "stem_conv_relu"):
    _lib.check(_lib.load().derl_b200_stem_conv_relu_mask(
        _p(frames), _p(rows) if rows is not None else None, batch, _p(weight), _p(bias), _p(out),
        _p(mask), out_block, _stream(frames)), "stem_conv_relu_mask")
  return out, mask


@stem_conv_relu_mask.register_fake
def _(frames, weight, bias, out_block=1, rows=None):
  batch = frames.shape[0] if rows is None else rows.shape[0]
  shape = (batch, 20, 20, 32) if out_block == 1 else (batch, 10, 10, 128)
  return (frames.new_empty(shape, dtype=torch.float32),
          frames.new_empty((batch, 14, 32), dtype=torch.int32))


@torch.library.custom_op("derl_b200::stem_backward_masked", mutates_args=(), device_types="cuda")
def stem_backward_masked(frames: Tensor, grad_out: Tensor, mask: Tensor, blocked: bool,
                         rows: Optional[Tensor] = None) -> Tuple[Tensor, Tensor]:
  """K7t (tcgen05 + tensor memory): (grad_weight [32,4,8,8], grad_bias [32]) of the stem from the
  uint8 frames, the gradient w.r.t. its output (channels-last [B,32,20,20], or [B,128,10,10]
  when `blocked`) and the ReLU mask `stem_conv_relu_mask` returned."""
  _dense(frames, "frames", (torch.uint8,))
  _need(tuple(frames.shape[1:]) == (84, 84, 4), f"frames must be [B,84,84,4], got {tuple(frames.shape)}")
  batch = _check_rows(frames, rows)
  _need(batch >= 1, "stem_backward_masked needs at least one frame")
  want = (batch, 128, 10, 10) if blocked else (batch, 32, 20, 20)
  _need(grad_out.dtype == torch.float32 and tuple(grad_out.shape) == want
        and grad_out.is_contiguous(memory_format=torch.channels_last),
        f"grad_out must be a channels_last float32 tensor of shape {want}")
  _dense(mask, "mask", (torch.int32,))
  _need(tuple(mask.shape) == (batch, 14, 32), f"mask must be int32 [{batch}, 14, 32]")
  grad_w = torch.empty((32, 4, 8, 8), dtype=torch.float32, device=frames.device)
  grad_b = torch.empty(32, dtype=torch.float32, device=frames.device)
  lib = _lib.load()
  ws_bytes = lib.derl_b200_stem_backward_workspace_bytes()
  ws = torch.empty(ws_bytes, dtype=torch.uint8, device=frames.device)
  with _device_of(frames, "stem_backward"):
    _lib.check(lib.derl_b200_stem_backward_masked(
        _p(frames), _p(rows) if rows is not None else None, batch, _p(grad_out), _p(mask),
        int(blocked), _p(grad_w), _p(grad_b), _p(ws), ws_bytes, _stream(frames)),
        "stem_backward_masked")
  return grad_w, grad_b


@stem_backward_masked.register_fake
def _(frames, grad_out, mask, blocked, rows=None):
  return frames.new_empty((32, 4, 8, 8), dtype=torch.float32), \
      frames.new_empty(32, dtype=torch.float32)


# --------------------------------------------------------------------------- K5: ReLU bwd
@torch.library.custom_op("derl_b200::relu_bwd_bias", mutates_args=(), device_types="cuda")
def relu_bwd_bias(grad_out: Tensor, out: Tensor, unblock: int = 1) -> Tuple[Tensor, Tensor]:
  """(grad_out masked by out > 0, per-channel sum of it as float32) for channels-last
  [B, C, H, W] tensors — threshold_backward and the bias gradient in one pass.  unblock > 1:
  the inputs are a space-to-depth(unblock) arrangement; the masked gradient comes back in the
  plain [B, C / unblock^2, H * unblock, W * unblock] layout, the sums keep C entries."""
  _need(grad_out.dim() == 4 and grad_out.shape == out.shape, "expected two [B, C, H, W] tensors")
  _need(grad_out.dtype == out.dtype and out.dtype in _S2D_DTYPES, "unsupported dtype")
  _need(out.is_contiguous(memory_format=torch.channels_last)
        and grad_out.is_contiguous(memory_format=torch.channels_last),
        "relu_bwd_bias needs channels_last tensors")
  batch, chans, height, width = out.shape
  if unblock > 1:
    _need(chans % (4 * unblock * unblock) == 0, "channels must be a multiple of 4 * unblock^2")
    grad_pre = torch.empty((batch, chans // unblock ** 2, height * unblock, width * unblock),
                           dtype=out.dtype, device=out.device,
                           memory_format=torch.channels_last)
  else:
    grad_pre = torch.empty_like(out)
  bias_grad = torch.empty(chans, dtype=torch.float32, device=out.device)
  lib = _lib.load()
  ws_bytes = lib.derl_b200_relu_bwd_bias_workspace_bytes(chans)
  ws = torch.empty(ws_bytes, dtype=torch.uint8, device=out.device)
  with _device_of(out, "relu_bwd_bias"):
    _lib.check(lib.derl_b200_relu_bwd_bias(_p(grad_out), _p(out), _p(grad_pre), _p(bias_grad),
                                           batch * height * width, chans,
                                           _S2D_DTYPES[out.dtype], unblock, height, width,
                                           _p(ws), ws_bytes, _stream(out)), "relu_bwd_bias")
  return grad_pre, bias_grad


@relu_bwd_bias.register_fake
def _(grad_out, out, unblock=1):
  batch, chans, height, width = out.shape
  shape = (batch, chans // unblock ** 2, height * unblock, width * unblock)
  return (out.new_empty(shape).contiguous(memory_format=torch.channels_last),
          out.new_empty(chans, dtype=torch.float32))


# --------------------------------------------------------------------------- K9: linear heads
@torch.library.custom_op("derl_b200::linear_heads", mutates_args=(), device_types="cuda")
def linear_heads(hidden: Tensor, hidden_bias: Optional[Tensor], weight: Tensor,
                 bias: Tensor) -> Tensor:
  """out [B, U] = (hidden [B, 512] + hidden_bias [512]) @ weight [U, 512].T + bias [U]: the
  stacked nn.Linear heads of the actor-critic network (derl/models.py:201-202) in one pass."""
  _dense(hidden, "hidden", (torch.float32,))
  _dense(weight, "weight", (torch.float32,))
  _dense(bias, "bias", (torch.float32,))
  _need(hidden.dim() == 2 and weight.dim() == 2 and hidden.shape[1] == weight.shape[1],
        "hidden [B, F] and weight [U, F] expected")
  _need(bias.shape == (weight.shape[0],), "bias must be [U]")
  if hidden_bias is not None:
    _dense(hidden_bias, "hidden_bias", (torch.float32,))
    _need(hidden_bias.shape == (hidden.shape[1],), "hidden_bias must be [F]")
  batch, features = hidden.shape
  units = weight.shape[0]
  out = torch.empty((batch, units), dtype=torch.float32, device=hidden.device)
  with _device_of(hidden, "linear_heads"):
    _lib.check(_lib.load().derl_b200_linear_heads_forward(
        _p(hidden), _p(hidden_bias), _p(weight), _p(bias), _p(out), batch, features, units,
        _stream(hidden)), "linear_heads")
  return out


@linear_heads.register_fake
def _(hidden, hidden_bias, weight, bias):
  return hidden.new_empty((hidden.shape[0], weight.shape[0]))


@torch.library.custom_op("derl_b200::linear_heads_backward", mutates_args=(), device_types="cuda")
def linear_heads_backward(hidden: Tensor, hidden_bias: Optional[Tensor], weight: Tensor,
                          grad_out: Tensor) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
  """(grad_hidden [B, 512], grad_weight [U, 512], grad_bias [U], grad_hidden_bias [512] or an
  empty tensor when hidden_bias is None) of `linear_heads`."""
  _dense(hidden, "hidden", (torch.float32,))
  _dense(weight, "weight", (torch.float32,))
  _dense(grad_out, "grad_out", (torch.float32,))
  batch, features = hidden.shape
  units = weight.shape[0]
  _need(grad_out.shape == (batch, units), "grad_out must be [B, U]")
  _need(batch >= 1, "linear_heads_backward needs at least one row")
  if hidden_bias is not None:
    _dense(hidden_bias, "hidden_bias", (torch.float32,))
  grad_hidden = torch.empty_like(hidden)
  grad_weight = torch.empty_like(weight)
  grad_bias = torch.empty(units, dtype=torch.float32, device=hidden.device)
  grad_hb = torch.empty(features if hidden_bias is not None else 0, dtype=torch.float32,
                        device=hidden.device)
  lib = _lib.load()
  ws_bytes = lib.derl_b200_linear_heads_workspace_bytes(units)
  ws = torch.empty(ws_bytes, dtype=torch.uint8, device=hidden.device)
  with _device_of(hidden, "linear_heads_backward"):
    _lib.check(lib.derl_b200_linear_heads_backward(
        _p(hidden), _p(hidden_bias), _p(weight), _p(grad_out), _p(grad_hidden), _p(grad_weight),
        _p(grad_bias), _p(grad_hb), batch, features, units, _p(ws), ws_bytes, _stream(hidden)),
        "linear_heads_backward")
  return grad_hidden, grad_weight, grad_bias, grad_hb


@linear_heads_backward.register_fake
def _(hidden, hidden_bias, weight, grad_out):
  return (torch.empty_like(hidden), torch.empty_like(weight), weight.new_empty(weight.shape[0]),
          weight.new_empty(hidden.shape[1] if hidden_bias is not None else 0))


def _linear_heads_setup(ctx, inputs, output):
  hidden, hidden_bias, weight, _ = inputs
  ctx.save_for_backward(hidden, weight, *([] if hidden_bias is None else [hidden_bias]))
  ctx.has_hidden_bias = hidden_bias is not None


def _linear_heads_bw(ctx, grad_out):
  hidden, weight, *rest = ctx.saved_tensors
  hidden_bias = rest[0] if ctx.has_hidden_bias else None
  grad_hidden, grad_weight, grad_bias, grad_hb = torch.ops.derl_b200.linear_heads_backward(
      hidden, hidden_bias, weight, grad_out.contiguous())
  return grad_hidden, (grad_hb if ctx.has_hidden_bias else None), grad_weight, grad_bias


linear_heads.register_autograd(_linear_heads_bw, setup_context=_linear_heads_setup)


# --------------------------------------------------------------------------- K3: PPO / A2C loss
def _loss_buffers(ref, nb):
  lib = _lib.load()
  loss = torch.empty((), dtype=torch.float32, device=ref.device)
  stats = torch.empty(_lib.LOSS_STATS, dtype=torch.float32, device=ref.device)
  ws_bytes = lib.derl_b200_ppo_loss_workspace_bytes(nb)
  ws = torch.empty(ws_bytes, dtype=torch.uint8, device=ref.device)
  return lib, loss, stats, ws, ws_bytes


def _check_value_side(who, nb, values, value_targets, old_values, a2c):
  if values is None:
    return
  _need(value_targets is not None and (a2c or old_values is not None),
        f"{who}: value head needs value_targets" + ("" if a2c else " and old values"))
  for name, t in (("values", values), ("value_targets", value_targets),
                  ("old values", old_values)):
    if t is None:
      continue
    _dense(t, name, (torch.float32,))
    _need(t.numel() == nb, f"{who}: {name} must have one element per sample")


def _check_policy_side(who, nb, old_log_prob, advantages, a2c):
  _need(advantages is not None and (a2c or old_log_prob is not None),
        f"{who}: policy head needs advantages" + ("" if a2c else " and log_prob"))
  for name, t in (("log_prob", old_log_prob), ("advantages", advantages)):
    if t is None:
      continue
    _dense(t, name, (torch.float32,))
    _need(t.numel() == nb, f"{who}: {name} length differs from the batch size")


def _grad_like(t, ref):
  return torch.empty_like(t) if t is not None else ref.new_empty(0)


def _run_categorical(a2c, logits, values, actions, old_log_prob, advantages, value_targets,
                     old_values, cliprange, value_loss_coef, entropy_coef):
  """Shared body of ppo_loss_categorical / a2c_loss_categorical: one launch of K3."""
  who = "a2c_loss_categorical" if a2c else "ppo_loss_categorical"
  ref = logits if logits is not None else values
  _need(ref is not None, f"{who}: both the policy head and the value head are absent")
  nb, nact = ref.shape[0], 1
  if logits is not None:
    _dense(logits, "logits", (torch.float32,))
    _need(logits.dim() == 2, f"logits must be [B, A], got {tuple(logits.shape)}")
    nact = logits.shape[1]
    _check_policy_side(who, nb, old_log_prob, advantages, a2c)
    _need(actions is not None, f"{who}: actions missing")
    _dense(actions, "actions", (torch.int64,))
    _need(actions.numel() == nb, f"{who}: one action index per sample")
    if CHECK_INDICES and nb:   # the kernel maps an out-of-range action to 0 (memory safety only)
      lo, hi = int(actions.min()), int(actions.max())
      if lo < 0 or hi >= nact:
        raise IndexError(f"{who}: action index out of range: [{lo}, {hi}] not within [0, {nact})")
  _check_value_side(who, nb, values, value_targets, old_values, a2c)
  lib, loss, stats, ws, ws_bytes = _loss_buffers(ref, nb)
  dlogits, dvalues = _grad_like(logits, ref), _grad_like(values, ref)
  with _device_of(ref, who):
    if a2c:
      code = lib.derl_b200_a2c_loss_categorical(
          _p(logits), nb, nact, _p(actions), _p(advantages), _p(values), _p(value_targets),
          float(value_loss_coef), float(entropy_coef), _p(loss), _p(dlogits), _p(dvalues),
          _p(stats), _p(ws), ws_bytes, _stream(ref))
    else:
      code = lib.derl_b200_ppo_loss_categorical(
          _p(logits), nb, nact, _p(actions), _p(old_log_prob), _p(advantages), _p(values),
          _p(value_targets), _p(old_values), int(cliprange is not None),
          float(cliprange or 0.), float(value_loss_coef), float(entropy_coef), _p(loss),
          _p(dlogits), _p(dvalues), _p(stats), _p(ws), ws_bytes, _stream(ref))
    _lib.check(code, who)
  return loss, dlogits, dvalues, stats


def _run_gaussian(a2c, loc, scale, values, actions, old_log_prob, advantages, value_targets,
                  old_values, cliprange, value_loss_coef, entropy_coef):
  """Shared body of ppo_loss_gaussian / a2c_loss_gaussian."""
  who = "a2c_loss_gaussian" if a2c else "ppo_loss_gaussian"
  ref = loc if loc is not None else values
  _need(ref is not None, f"{who}: both the policy head and the value head are absent")
  nb, ndim = ref.shape[0], 1
  if loc is not None:
    _need(scale is not None and actions is not None, f"{who}: scale/actions missing")
    for name, t in (("loc", loc), ("scale", scale), ("actions", actions)):
      _dense(t, name, (torch.float32,))
    _need(loc.dim() == 2 and scale.shape == loc.shape and actions.shape == loc.shape,
          f"loc {tuple(loc.shape)}, scale {tuple(scale.shape)} and actions "
          f"{tuple(actions.shape)} must all be [B, D]")
    ndim = loc.shape[1]
    _check_policy_side(who, nb, old_log_prob, advantages, a2c)
  _check_value_side(who, nb, values, value_targets, old_values, a2c)
  lib, loss, stats, ws, ws_bytes = _loss_buffers(ref, nb)
  dloc = _grad_like(loc, ref)
  dscale = _grad_like(scale if loc is not None else None, ref)
  dvalues = _grad_like(values, ref)
  with _device_of(ref, who):
    if a2c:
      code = lib.derl_b200_a2c_loss_gaussian(
          _p(loc), _p(scale), nb, ndim, _p(actions), _p(advantages), _p(values),
          _p(value_targets), float(value_loss_coef), float(entropy_coef), _p(loss), _p(dloc),
          _p(dscale), _p(dvalues), _p(stats), _p(ws), ws_bytes, _stream(ref))
    else:
      code = lib.derl_b200_ppo_loss_gaussian(
          _p(loc), _p(scale), nb, ndim, _p(actions), _p(old_log_prob), _p(advantages), _p(values),
          _p(value_targets), _p(old_values), int(cliprange is not None), float(cliprange or 0.),
          float(value_loss_coef), float(entropy_coef), _p(loss), _p(dloc), _p(dscale),
          _p(dvalues), _p(stats), _p(ws), ws_bytes, _stream(ref))
    _lib.check(code, who)
  return loss, dloc, dscale, dvalues, stats


def _scaled_backward(ngrads, nrest, has_of):
  """autograd of a loss op: the kernel already produced d loss / d head; scale by grad(loss).
  ngrads saved gradient tensors, nrest non-differentiable trailing inputs; has_of(inputs) says
  which heads exist (absent heads get None)."""
  def setup(ctx, inputs, output):
    ctx.set_materialize_grads(False)
    ctx.save_for_backward(*output[1:1 + ngrads])
    ctx.has = has_of(inputs)

  def backward(ctx, g_loss, *unused):
    rest = (None,) * nrest
    if g_loss is None:
      return (None,) * ngrads + rest
    return tuple((g_loss * d) if present else None
                 for d, present in zip(ctx.saved_tensors, ctx.has)) + rest
  return backward, setup


@torch.library.custom_op("derl_b200::ppo_loss_categorical", mutates_args=(), device_types="cuda")
def ppo_loss_categorical(logits: Optional[Tensor], values: Optional[Tensor],
                         actions: Optional[Tensor], old_log_prob: Optional[Tensor],
                         advantages: Optional[Tensor], value_targets: Optional[Tensor],
                         old_values: Optional[Tensor], cliprange: Optional[float],
                         value_loss_coef: float,
                         entropy_coef: float) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
  """(loss [], dloss/dlogits, dloss/dvalues, stats f32[16]); absent heads give empty grads."""
  return _run_categorical(False, logits, values, actions, old_log_prob, advantages,
                          value_targets, old_values, cliprange, value_loss_coef, entropy_coef)


@ppo_loss_categorical.register_fake
def _(logits, values, actions, old_log_prob, advantages, value_targets, old_values, cliprange,
      value_loss_coef, entropy_coef):
  ref = logits if logits is not None else values
  return ref.new_empty(()), _grad_like(logits, ref), _grad_like(values, ref), \
      ref.new_empty(_lib.LOSS_STATS)


_bw, _su = _scaled_backward(2, 8, lambda i: (i[0] is not None, i[1] is not None))
ppo_loss_categorical.register_autograd(_bw, setup_context=_su)


@torch.library.custom_op("derl_b200::ppo_loss_gaussian", mutates_args=(), device_types="cuda")
def ppo_loss_gaussian(loc: Optional[Tensor], scale: Optional[Tensor], values: Optional[Tensor],
                      actions: Optional[Tensor], old_log_prob: Optional[Tensor],
                      advantages: Optional[Tensor], value_targets: Optional[Tensor],
                      old_values: Optional[Tensor], cliprange: Optional[float],
                      value_loss_coef: float,
                      entropy_coef: float) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
  """(loss [], dloss/dloc, dloss/dscale, dloss/dvalues, stats f32[16])."""
  return _run_gaussian(False, loc, scale, values, actions, old_log_prob, advantages,
                       value_targets, old_values, cliprange, value_loss_coef, entropy_coef)


@ppo_loss_gaussian.register_fake
def _(loc, scale, values, actions, old_log_prob, advantages, value_targets, old_values,
      cliprange, value_loss_coef, entropy_coef):
  ref = loc if loc is not None else values
  return (ref.new_empty(()), _grad_like(loc, ref), _grad_like(scale, ref),
          _grad_like(values, ref), ref.new_empty(_lib.LOSS_STATS))


_bw, _su = _scaled_backward(3, 8, lambda i: (i[0] is not None, i[0] is not None, i[2] is not None))
ppo_loss_gaussian.register_autograd(_bw, setup_context=_su)


@torch.library.custom_op("derl_b200::a2c_loss_categorical", mutates_args=(), device_types="cuda")
def a2c_loss_categorical(logits: Optional[Tensor], values: Optional[Tensor],
                         actions: Optional[Tensor], advantages: Optional[Tensor],
                         value_targets: Optional[Tensor], value_loss_coef: float,
                         entropy_coef: float) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
  """Advantage actor-critic loss (categorical head): (loss [], dlogits, dvalues, stats f32[16])."""
  return _run_categorical(True, logits, values, actions, None, advantages, value_targets, None,
                          None, value_loss_coef, entropy_coef)


@a2c_loss_categorical.register_fake
def _(logits, values, actions, advantages, value_targets, value_loss_coef, entropy_coef):
  ref = logits if logits is not None else values
  return ref.new_empty(()), _grad_like(logits, ref), _grad_like(values, ref), \
      ref.new_empty(_lib.LOSS_STATS)


_bw, _su = _scaled_backward(2, 5, lambda i: (i[0] is not None, i[1] is not None))
a2c_loss_categorical.register_autograd(_bw, setup_context=_su)


@torch.library.custom_op("derl_b200::a2c_loss_gaussian", mutates_args=(), device_types="cuda")
def a2c_loss_gaussian(loc: Optional[Tensor], scale: Optional[Tensor], values: Optional[Tensor],
                      actions: Optional[Tensor], advantages: Optional[Tensor],
                      value_targets: Optional[Tensor], value_loss_coef: float,
                      entropy_coef: float) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
  """Advantage actor-critic loss (diagonal-Gaussian head)."""
  return _run_gaussian(True, loc, scale, values, actions, None, advantages, value_targets, None,
                       None, value_loss_coef, entropy_coef)


@a2c_loss_gaussian.register_fake
def _(loc, scale, values, actions, advantages, value_targets, value_loss_coef, entropy_coef):
  ref = loc if loc is not None else values
  return (ref.new_empty(()), _grad_like(loc, ref), _grad_like(scale, ref),
          _grad_like(values, ref), ref.new_empty(_lib.LOSS_STATS))


_bw, _su = _scaled_backward(3, 5, lambda i: (i[0] is not None, i[0] is not None, i[2] is not None))
a2c_loss_gaussian.register_autograd(_bw, setup_context=_su)


# --------------------------------------------------------------------------- K8: MLP PPO update
@torch.library.custom_op("derl_b200::ppo_mlp_update",
                         mutates_args=("params", "exp_avg", "exp_avg_sq"), device_types="cuda")
def ppo_mlp_update(params: List[Tensor], exp_avg: List[Tensor], exp_avg_sq: List[Tensor],
                   observations: Tensor, actions: Tensor, old_log_prob: Tensor,
                   advantages: Tensor, value_targets: Tensor, old_values: Tensor, perm: Tensor,
                   num_epochs: int, minibatch: int, normalize: bool, adv_epsilon: float,
                   cliprange: Optional[float], value_loss_coef: float, entropy_coef: float,
                   max_grad_norm: Optional[float], lr: float, beta1: float, beta2: float,
                   adam_eps: float, adam_step: int) -> Tuple[Tensor, Tensor]:
  """One whole PPO update (all epochs x minibatches) of the two-MLP actor-critic in one launch;
  updates `params`, `exp_avg`, `exp_avg_sq` in place.  Returns (losses [nsteps], stats
  [nsteps, 16]).  Tensor order: policy W1 b1 W2 b2 W3 b3, value W1 b1 W2 b2 W3 b3, logstd."""
  _need(len(params) == 13 and len(exp_avg) == 13 and len(exp_avg_sq) == 13,
        "ppo_mlp_update: 13 parameter / exp_avg / exp_avg_sq tensors expected")
  _dense(observations, "observations", (torch.float32, torch.float64))
  _need(observations.dim() == 2, "observations must be [S, obs_dim]")
  size, obs_dim = observations.shape
  act_dim = params[12].numel()
  shapes = [(64, obs_dim), (64,), (64, 64), (64,), (act_dim, 64), (act_dim,),
            (64, obs_dim), (64,), (64, 64), (64,), (1, 64), (1,), (act_dim,)]
  for group, name in ((params, "params"), (exp_avg, "exp_avg"), (exp_avg_sq, "exp_avg_sq")):
    for i, (t, shape) in enumerate(zip(group, shapes)):
      _dense(t, f"{name}[{i}]", (torch.float32,))
      _need(tuple(t.shape) == shape, f"{name}[{i}] must have shape {shape}, got {tuple(t.shape)}")
  _dense(actions, "actions", (torch.float32,))
  _need(tuple(actions.shape) == (size, act_dim), "actions must be [S, act_dim]")
  for name, t in (("log_prob", old_log_prob), ("advantages", advantages),
                  ("value_targets", value_targets), ("values", old_values)):
    _dense(t, name, (torch.float32,))
    _need(t.numel() == size, f"{name} must have one element per sample")
  _dense(perm, "perm", (torch.int64,))
  _need(perm.numel() == num_epochs * size, "perm must hold num_epochs * S row indices")
  _need(1 <= minibatch <= size and num_epochs >= 1, "bad minibatch size / epoch count")
  nsteps = num_epochs * ((size + minibatch - 1) // minibatch)
  losses = torch.empty(nsteps, dtype=torch.float32, device=observations.device)
  stats = torch.empty((nsteps, _lib.LOSS_STATS), dtype=torch.float32, device=observations.device)
  table = lambda ts: (_VP * 13)(*[t.data_ptr() for t in ts])
  lib = _lib.load()
  ws_bytes = lib.derl_b200_ppo_mlp_update_workspace_bytes(obs_dim, act_dim)
  ws = torch.empty(ws_bytes, dtype=torch.uint8, device=observations.device)
  with _device_of(observations, "ppo_mlp_update"):
    _lib.check(_lib.load().derl_b200_ppo_mlp_update(
        table(params), table(exp_avg), table(exp_avg_sq), obs_dim, act_dim, _p(observations),
        int(observations.dtype == torch.float64), _p(actions), _p(old_log_prob), _p(advantages),
        _p(value_targets), _p(old_values), size, _p(perm), num_epochs, minibatch, int(normalize),
        float(adv_epsilon), int(cliprange is not None), float(cliprange or 0.),
        float(value_loss_coef), float(entropy_coef),
        float(max_grad_norm) if max_grad_norm is not None else -1.0, float(lr), float(beta1),
        float(beta2), float(adam_eps), int(adam_step), _p(losses), _p(stats), _p(ws), ws_bytes,
        _stream(observations)), "ppo_mlp_update")
  return losses, stats


@ppo_mlp_update.register_fake
def _(params, exp_avg, exp_avg_sq, observations, actions, old_log_prob, advantages, value_targets,
      old_values, perm, num_epochs, minibatch, normalize, adv_epsilon, cliprange, value_loss_coef,
      entropy_coef, max_grad_norm, lr, beta1, beta2, adam_eps, adam_step):
  nsteps = num_epochs * ((observations.shape[0] + minibatch - 1) // minibatch)
  return (observations.new_empty(nsteps, dtype=torch.float32),
          observations.new_empty((nsteps, _lib.LOSS_STATS), dtype=torch.float32))
