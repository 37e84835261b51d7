"""Policy networks of the PPO path, state_dict-compatible with the reference.

Reference: derl/models.py — collocate_inputs :72-91, NatureCNNBase :94-124,
broadcast_inputs :141-163, NatureCNNModel :166-214, MLP :224-237, MuJoCoModel :240-271,
make_model :281-298.  Only the options PPO uses are carried (no noisy / dueling /
distributional heads: those belong to DQN / SAC, outside the hot path).

The hidden conv / linear layers stay library calls (cuDNN / cuBLAS tensor-core kernels); the
stem — the one layer that touches the uint8 frames — runs on derl_b200's own INT8 tensor-core
kernels (K6t forward; K7t backward of a float32 forward) whenever a reduced-precision
tensor-core path is allowed (TF32 or autocast).  B200-specific choices around them: an NHWC uint8
frame stack viewed as NCHW *is* a channels_last tensor, so the trunk runs channels_last end to end
and the reference's NCHW `.contiguous()` transpose copy (models.py:123) never happens; strided
convs with kernel = 2 x stride run as 2x2/1 convs on space-to-depth tensors.
"""
import numpy as np
import torch
from torch import nn


def _device():
  return "cuda" if torch.cuda.is_available() else "cpu"


def orthogonal_init(layer):
  """Orthogonal weights, zero biases (reference :127-138)."""
  if hasattr(layer, "weight"):
    nn.init.orthogonal_(layer.weight)
  if hasattr(layer, "bias"):
    nn.init.zeros_(layer.bias)


def _collocate(module, inputs, cast_dtype):
  """NumPy -> tensor, then onto the module's device (and dtype when asked)."""
  param = next(module.parameters())
  out = []
  for x in inputs:
    if isinstance(x, np.ndarray):
      x = torch.from_numpy(x)
    want_dtype = param.dtype if cast_dtype and x.dtype != param.dtype else None
    if x.device != param.device or want_dtype is not None:
      x = x.to(device=param.device, dtype=want_dtype)
    out.append(x)
  return out


def _broadcast(ndims, forward, module, inputs):
  """Pad leading axes up to `ndims`, call, strip them again (reference :141-163)."""
  rank = inputs[0].ndim
  for i, x in enumerate(inputs):
    if x.ndim != rank:
      raise ValueError("for broadcasting all inputs must have the same "
                       "number of dimensions, got "
                       f"inputs[0].shape={inputs[0].shape}, "
                       f"inputs[{i}].shape={inputs[i].shape}")
  extra = ndims - rank
  outputs = forward(module, *[x[(None,) * extra] for x in inputs])

  def strip(out):
    if isinstance(out, (tuple, list)):
      return type(out)(strip(o) for o in out)
    return out.reshape(out.shape[extra:])
  return strip(outputs)


class _ConvBiasReLU(torch.autograd.Function):
  """conv2d + bias + ReLU as ONE cuDNN call forward (`cudnn_convolution_relu`: the bias add
  and the activation run in the convolution's epilogue instead of two more passes over the
  activation tensor), and threshold + `convolution_backward` backward.  The ReLU mask is
  recovered from the output, so the pre-activation tensor is never materialised or saved."""

  @staticmethod
  def forward(ctx, inputs, weight, bias, stride, padding):
    out = torch.cudnn_convolution_relu(inputs, weight, bias, stride, padding, (1, 1), 1)
    ctx.save_for_backward(inputs, weight, out)
    ctx.conf = (stride, padding)
    return out

  @staticmethod
  def backward(ctx, grad_out):
    inputs, weight, out = ctx.saved_tensors
    stride, padding = ctx.conf
    chans = out.shape[1]
    # ReLU mask + bias gradient in one derl_b200 kernel (K5) where its shape rules allow
    if (chans % 4 == 0 and 256 % (chans // 4) == 0
        and out.is_contiguous(memory_format=torch.channels_last)):
      from . import ops  # noqa: F401
      grad_out = grad_out.contiguous(memory_format=torch.channels_last)
      grad_pre, grad_b = torch.ops.derl_b200.relu_bwd_bias(grad_out, out)
      grad_in, grad_w, _ = torch.ops.aten.convolution_backward(
          grad_pre, inputs, weight, None, stride, padding, (1, 1), False, (0, 0), 1,
          [ctx.needs_input_grad[0], True, False])
      return grad_in, grad_w, grad_b.to(weight.dtype), None, None
    grad_pre = torch.ops.aten.threshold_backward(grad_out, out, 0)
    grad_in, grad_w, grad_b = torch.ops.aten.convolution_backward(
        grad_pre, inputs, weight, [weight.shape[0]], stride, padding, (1, 1), False, (0, 0), 1,
        [ctx.needs_input_grad[0], True, True])
    return grad_in, grad_w, grad_b, None, None


class _StemConvReLU(torch.autograd.Function):
  """The 8x8/4 stem + bias + ReLU straight from uint8 frames (derl_b200 K6t) forward,
  optionally emitting the space-to-depth(2) arrangement the next layer consumes.  A float32
  forward that needs a gradient also emits the ReLU mask as bits (K6t), and the backward is K7t
  (ReLU mask + bias gradient + weight gradient in one INT8 tensor-core pass over the same uint8
  frames).  Otherwise (bf16 autocast) the backward is K5 (ReLU mask + bias gradient) and the
  weight gradient of the equivalent space-to-depth conv (K4 re-creates the float frames, cuDNN
  wgrad), mapped back to [32, 4, 8, 8].  With `rows` the kernels read frames[rows] in place: the
  minibatch gather fused into the layer (runners/row_selection.py)."""

  @staticmethod
  def forward(ctx, frames, weight, bias, dtype, out_block, rows=None):
    """rows: int64 indices — the batch is frames[rows], read in place (fused minibatch gather)."""
    mask = None
    wants_backward = any(ctx.needs_input_grad[1:3])   # no mask for rollouts / no_grad forwards
    if dtype == torch.float32 and wants_backward:
      out, mask = torch.ops.derl_b200.stem_conv_relu_mask(frames, weight.contiguous(), bias,
                                                          out_block, rows)
    else:
      out = torch.ops.derl_b200.stem_conv_relu(frames, weight.contiguous(), bias, dtype,
                                               out_block, rows)
    out = out.permute(0, 3, 1, 2)   # channels-last storage seen as NCHW
    # with the mask the backward never reads the activation (its consumer, the next layer, keeps
    # it alive anyway); without it the activation itself is the mask
    ctx.save_for_backward(frames, out if mask is None else mask, rows)
    ctx.has_mask = mask is not None
    ctx.weight_dtype, ctx.out_block = weight.dtype, out_block
    return out

  @staticmethod
  def backward(ctx, grad_out):
    frames, out, rows = ctx.saved_tensors
    grad_out = grad_out.contiguous(memory_format=torch.channels_last)
    if ctx.has_mask:
      grad_w, grad_b = torch.ops.derl_b200.stem_backward_masked(frames, grad_out, out,
                                                                ctx.out_block == 2, rows)
      return None, grad_w.to(ctx.weight_dtype), grad_b, None, None, None
    if rows is not None:   # the library route below wants the batch's frames as one tensor
      frames = torch.ops.derl_b200.gather_rows(frames, rows, 0, rows.numel())
    # out_block 2: [B,128,10,10] with (i, j, c) channels; K5 stores the masked gradient
    # straight in the plain [B,32,20,20] layout the weight-gradient conv needs
    grad_pre, grad_b = torch.ops.derl_b200.relu_bwd_bias(grad_out, out, ctx.out_block)
    if ctx.out_block == 2:
      grad_b = grad_b.view(4, 32).sum(0)
    s2d = torch.ops.derl_b200.frames_to_s2d(frames, 4, out.dtype, 255.0).permute(0, 3, 1, 2)
    shape_only = s2d.new_empty((32, 64, 2, 2)).contiguous(memory_format=torch.channels_last)
    _, grad_w2, _ = torch.ops.aten.convolution_backward(
        grad_pre, s2d, shape_only, None, (1, 1), (0, 0), (1, 1), False, (0, 0), 1,
        [False, True, False])
    # [O, (i, j, c), a, b] -> [O, c, 4a + i, 4b + j]
    grad_w = grad_w2.reshape(32, 4, 4, 4, 2, 2).permute(0, 3, 4, 1, 5, 2).reshape(32, 4, 8, 8)
    return None, grad_w.to(ctx.weight_dtype), grad_b, None, None, None


def _conv_out(size, conv):
  return (size + 2 * conv.padding[0] - conv.dilation[0] * (conv.kernel_size[0] - 1) - 1) \
      // conv.stride[0] + 1


class NatureCNNBase(nn.Sequential):
  """conv8x8/4 -> conv4x4/2 -> conv3x3/1 (ReLU each) -> flatten -> linear 512 (no ReLU)."""

  def __init__(self, input_shape=(84, 84, 4), permute=True):
    super().__init__()
    self.permute = permute
    channels, height, width = input_shape
    if permute:
      height, width, channels = input_shape
    convs = [nn.Conv2d(channels, 32, 8, 4), nn.Conv2d(32, 64, 4, 2), nn.Conv2d(64, 64, 3, 1)]
    for i, conv in enumerate(convs):
      height, width = _conv_out(height, conv), _conv_out(width, conv)
      self.add_module(f"conv-{i}", conv)
      self.add_module(f"relu-{i}", nn.ReLU())
    self.add_module("flatten", nn.Flatten())
    self.add_module("linear", nn.Linear(height * width * convs[-1].out_channels, 512))

  custom_stem = True             # K6t: stem conv straight from uint8 frames (needs TF32 allowed
                                 # or autocast: it is a reduced-precision tensor-core path)
  space_to_depth = True          # class-wide switches (tests compare the formulations)
  space_to_depth_hidden = True   # ... also for strided convs after the stem (the 4x4/2 layer):
                                 # avoids cuDNN's strided dgrad + layout folds (-5 % per update)
  fused_conv_relu = True
  defer_linear_bias = False   # set by NatureCNNModel around its call: see `deferred_bias`
  deferred_bias = None

  @staticmethod
  def _s2d_weight(conv):
    """[O, C, 2s, 2s] -> [O, s*s*C, 2, 2]: weights of the equivalent 2x2 / stride-1 conv over
    the space-to-depth(s) tensor (channel order (i, j, c), like the activations)."""
    s, out_ch, in_ch = conv.stride[0], conv.out_channels, conv.in_channels
    weight = conv.weight.view(out_ch, in_ch, 2, s, 2, s).permute(0, 3, 5, 1, 2, 4)
    return weight.reshape(out_ch, s * s * in_ch, 2, 2).contiguous(
        memory_format=torch.channels_last)

  @staticmethod
  def _s2d_ok(conv, height, width):
    s = conv.stride[0]
    return (s > 1 and conv.stride == (s, s) and conv.kernel_size == (2 * s, 2 * s)
            and conv.padding == (0, 0) and conv.dilation == (1, 1) and conv.groups == 1
            and height % s == 0 and width % s == 0)

  def _conv_relu(self, hidden, conv, pre_s2d=False):
    """conv + bias + ReLU.  A strided conv with kernel = 2 x stride is evaluated as a 2x2 /
    stride-1 conv over the space-to-depth activation (same parameters, same sums): cuDNN's
    strided dgrad + its layout folds for the 4x4/2 layer were 14 % of the update in situ, the
    stride-1 form runs on plain implicit-GEMM kernels and the re-arrangement is one
    derl_b200.space_to_depth pass (or free when the stem kernel already emitted that layout:
    `pre_s2d`).  On the GPU conv, bias and ReLU are one cuDNN call."""
    weight, bias, stride = conv.weight, conv.bias, conv.stride
    if pre_s2d:
      weight, stride = self._s2d_weight(conv), (1, 1)
    elif (self.space_to_depth and self.space_to_depth_hidden and hidden.is_cuda
          and self._s2d_ok(conv, *hidden.shape[2:])):
      s, (batch, chans, height, width) = stride[0], hidden.shape
      nhwc = hidden.permute(0, 2, 3, 1)   # a view: channels-last storage is NHWC-contiguous
      if nhwc.is_contiguous() and (chans * hidden.element_size()) % 16 == 0:
        from . import ops  # noqa: F401
        hidden = torch.ops.derl_b200.space_to_depth(nhwc, s, False).permute(0, 3, 1, 2)
      else:
        blocks = nhwc.reshape(batch, height // s, s, width // s, s, chans)
        hidden = blocks.permute(0, 1, 3, 2, 4, 5).reshape(batch, height // s, width // s,
                                                          s * s * chans).permute(0, 3, 1, 2)
      weight, stride = self._s2d_weight(conv), (1, 1)
    if (self.fused_conv_relu and hidden.is_cuda and bias is not None and conv.groups == 1
        and conv.dilation == (1, 1) and isinstance(conv.padding, tuple)):
      if hidden.dtype != weight.dtype:         # autocast: run the whole layer in that dtype
        weight, bias = weight.to(hidden.dtype), bias.to(hidden.dtype)
      return _ConvBiasReLU.apply(hidden, weight, bias, stride, conv.padding)
    return torch.relu(nn.functional.conv2d(hidden, weight, bias, stride, conv.padding))

  def _forward_frames(self, frames):
    """uint8 NHWC frames on the GPU.  The 8x8/4 stem over 4 channels is a 2x2/1 conv over the
    space-to-depth(4) tensor with 64 channels: cuDNN has only a scalar NHWC engine for C = 4
    (13 ms per 16384 frames, 49 % of the update before this change) but tensor-core implicit
    GEMM for C = 64.  Re-indexing, uint8 -> float cast and the /255 are ONE pass of the
    frames_to_s2d kernel (IEEE division: the reference's `.float() / 255` values exactly)."""
    conv = self[0]
    s = conv.stride[0]
    from . import ops  # noqa: F401  (registers torch.ops.derl_b200)
    from .runners.row_selection import RowSelection
    selection = frames if isinstance(frames, RowSelection) else None
    autocast = torch.is_autocast_enabled("cuda")
    dtype = torch.get_autocast_dtype("cuda") if autocast else conv.weight.dtype
    pre_s2d = False
    if (self.custom_stem and (autocast or torch.backends.cudnn.allow_tf32)
        and tuple(frames.shape[1:]) == (84, 84, 4) and tuple(conv.weight.shape) == (32, 4, 8, 8)
        and conv.weight.dtype == torch.float32 and dtype in (torch.float32, torch.bfloat16)):
      nxt = list(self.children())[2]
      pre_s2d = (self.space_to_depth and self.space_to_depth_hidden and isinstance(nxt, nn.Conv2d)
                 and nxt.stride == (2, 2) and self._s2d_ok(nxt, 20, 20))
      if selection is not None:   # fused gather: the stem kernels read the rollout rows in place
        hidden = _StemConvReLU.apply(selection.source, conv.weight, conv.bias, dtype,
                                     2 if pre_s2d else 1, selection.rows)
      else:
        hidden = _StemConvReLU.apply(frames, conv.weight, conv.bias, dtype, 2 if pre_s2d else 1)
    else:
      if selection is not None:
        frames = selection.materialize()
      s2d = torch.ops.derl_b200.frames_to_s2d(frames, s, dtype, 255.0).permute(0, 3, 1, 2)
      weight, bias = self._s2d_weight(conv), conv.bias
      if self.fused_conv_relu:
        if s2d.dtype != weight.dtype:
          weight, bias = weight.to(s2d.dtype), bias.to(s2d.dtype)
        hidden = _ConvBiasReLU.apply(s2d, weight, bias, (1, 1), (0, 0))
      else:
        hidden = torch.relu(nn.functional.conv2d(s2d, weight, bias))
    layers = list(self.children())[2:]          # after conv-0, relu-0
    while len(layers) >= 2 and isinstance(layers[0], nn.Conv2d) and isinstance(layers[1], nn.ReLU):
      hidden = self._conv_relu(hidden, layers[0], pre_s2d)
      pre_s2d = False
      layers = layers[2:]
    if (len(layers) == 2 and isinstance(layers[0], nn.Flatten) and isinstance(layers[1], nn.Linear)
        and hidden.is_contiguous(memory_format=torch.channels_last)):
      # nn.Flatten orders features (c, h, w); the activations lie (h, w, c) in memory.  Re-index
      # the linear layer's 1.6 M weights instead of transposing B x 3136 activations (and their
      # gradients) on every pass: the flatten becomes a view.
      batch, chans, height, width = hidden.shape
      linear = layers[1]
      weight = linear.weight.view(-1, chans, height, width).permute(0, 2, 3, 1).reshape(
          linear.out_features, -1)
      flat = hidden.permute(0, 2, 3, 1).reshape(batch, -1)
      if self.defer_linear_bias and linear.bias is not None and flat.dtype == linear.bias.dtype:
        # the caller (NatureCNNModel with fused heads, K9) adds the bias inside its own kernel and
        # gets its gradient from the heads' column sums instead of a [B, 512] reduction
        self.__dict__["deferred_bias"] = linear.bias   # not a second registration of the Parameter
        return nn.functional.linear(flat, weight.to(flat.dtype), None)
      return nn.functional.linear(flat, weight.to(flat.dtype), linear.bias.to(flat.dtype)
                                  if linear.bias is not None else None)
    for layer in layers:                        # flatten, linear
      hidden = layer(hidden)
    return hidden

  def _s2d_applies(self, inputs):
    conv = self[0]
    return (self.space_to_depth and self.permute and inputs.is_cuda and inputs.dtype == torch.uint8
            and inputs.ndim == 4 and inputs.is_contiguous() and conv.bias is not None
            and self._s2d_ok(conv, inputs.shape[1], inputs.shape[2])
            and conv.stride[0] * inputs.shape[3] == 16)

  def forward(self, inputs):
    inputs, = _collocate(self, [inputs], cast_dtype=False)
    if self._s2d_applies(inputs):
      return self._forward_frames(inputs)
    if hasattr(inputs, "materialize"):   # a RowSelection on a path without the fused stem
      inputs = inputs.materialize()
    if self.permute:
      inputs = inputs.permute(0, 3, 1, 2)   # NHWC storage seen as NCHW == channels_last
    if inputs.dtype == torch.uint8:
      inputs = inputs.float() / 255         # elementwise: keeps the channels_last strides
    return super().forward(inputs)


class NatureCNNModel(nn.Module):
  """Nature-DQN trunk with linear heads; `output_units=[A, 1]` for actor-critic PPO."""

  def __init__(self, output_units, input_shape=(84, 84, 4), init_fn=orthogonal_init):
    super().__init__()
    self.single_output = not isinstance(output_units, (list, tuple))
    self.output_units = [output_units] if self.single_output else list(output_units)
    self.base = NatureCNNBase(input_shape)
    self.output_layers = nn.ModuleList([nn.Linear(512, n) for n in self.output_units])
    self.init_fn = init_fn
    if init_fn:
      self.apply(init_fn)
    self.autocast_dtype = None  # e.g. torch.bfloat16: run trunk + heads under autocast
    self.to(_device())
    if next(self.parameters()).is_cuda:
      self.to(memory_format=torch.channels_last)

  fused_heads = True  # all output layers as ONE derl_b200 kernel over the 512 features (K9)

  def _heads_fusable(self):
    layers = list(self.output_layers)
    return (self.fused_heads and self.autocast_dtype is None
            and not torch.is_autocast_enabled("cuda")
            and all(type(l) is nn.Linear and l.bias is not None and l.in_features == 512
                    and l.weight.is_cuda and l.weight.dtype == torch.float32 for l in layers)
            and 1 <= sum(l.out_features for l in layers) <= 32)

  def _fused_heads(self, observations):
    """Trunk with its last bias deferred, then every head in one kernel (K9)."""
    base = self.base
    base.__dict__.update(defer_linear_bias=True, deferred_bias=None)
    try:
      hidden = base(observations)
      hidden_bias = base.__dict__["deferred_bias"]
    finally:
      base.__dict__.update(defer_linear_bias=False, deferred_bias=None)
    layers = list(self.output_layers)
    if not (hidden.is_cuda and hidden.dtype == torch.float32 and hidden.dim() == 2
            and hidden.is_contiguous()):
      if hidden_bias is not None:
        hidden = hidden + hidden_bias
      return [layer(hidden) for layer in layers]
    from . import ops  # noqa: F401
    weight = torch.cat([l.weight for l in layers], 0) if len(layers) > 1 else layers[0].weight
    bias = torch.cat([l.bias for l in layers], 0) if len(layers) > 1 else layers[0].bias
    out = torch.ops.derl_b200.linear_heads(hidden, hidden_bias, weight.contiguous(),
                                           bias.contiguous())
    if len(layers) == 1:
      return [out]
    return [o.contiguous() for o in torch.split(out, [l.out_features for l in layers], 1)]

  def _forward(self, observations):
    if self.autocast_dtype is not None:
      with torch.autocast("cuda", dtype=self.autocast_dtype):
        hidden = self.base(observations)
        outputs = [layer(hidden).float() for layer in self.output_layers]
    elif self._heads_fusable():
      outputs = self._fused_heads(observations)
    else:
      hidden = self.base(observations)
      outputs = [layer(hidden) for layer in self.output_layers]
    return outputs[0] if self.single_output else outputs

  def forward(self, *inputs):
    return _broadcast(4, NatureCNNModel._forward, self, inputs)


class MLP(nn.Sequential):
  """Linear/activation stack without an activation after the last layer."""

  def __init__(self, in_features, out_features, hidden_features=(64, 64), activation=nn.Tanh):
    sizes = (in_features, *hidden_features, out_features)
    layers = []
    for nin, nout in zip(sizes[:-1], sizes[1:]):
      layers += [nn.Linear(nin, nout), activation()]
    super().__init__(*layers[:-1])


class MuJoCoModel(nn.Module):
  """One MLP per output; state-independent logstd; returns (loc, std[B,D], *others)."""

  def __init__(self, observation_dim, output_units, mlp=MLP, init_fn=orthogonal_init):
    super().__init__()
    if not isinstance(output_units, (tuple, list)):
      output_units = [output_units]
    self.module_list = nn.ModuleList(mlp(observation_dim, n) for n in output_units)
    self.init_fn = init_fn
    if init_fn is not None:
      self.apply(init_fn)
    self.logstd = nn.Parameter(torch.zeros(output_units[0]))
    self.to(_device())

  def _forward(self, observations):
    observations, = _collocate(self, [observations], cast_dtype=True)
    first, *others = (module(observations) for module in self.module_list)
    std = torch.exp(self.logstd)[None].expand(observations.shape[0], -1).contiguous()
    return (first, std, *others)

  def forward(self, *inputs):
    return _broadcast(2, MuJoCoModel._forward, self, inputs)


def make_model(observation_space, action_space, other_outputs=None, **kwargs):
  """Default model for the spaces (reference :281-298): Discrete -> NatureCNNModel,
  Box -> MuJoCoModel.  Spaces are duck-typed (`.n` / `.shape`), gym is not imported."""
  if isinstance(other_outputs, int) or other_outputs is None:
    other_outputs = [other_outputs] if other_outputs is not None else []
  if hasattr(action_space, "spaces"):
    action_space = action_space.spaces[0]
  if hasattr(action_space, "n"):
    return NatureCNNModel(input_shape=observation_space.shape,
                          output_units=[action_space.n, *other_outputs], **kwargs)
  if getattr(action_space, "shape", None) is not None:
    if len(observation_space.shape) != 1 or len(action_space.shape) != 1:
      raise ValueError(f"expected vector shape, got shape={observation_space.shape}")
    return MuJoCoModel(observation_dim=observation_space.shape[0],
                       output_units=[action_space.shape[0], *other_outputs], **kwargs)
  raise ValueError(f"unsupported action space {action_space}")
