"""NumPy model of the arithmetic of the derl_b200 stem kernels (test infrastructure).

K6t (csrc/stem_tc.cu) and K7t (csrc/stem_bwd_tc.cu) evaluate the reference's
first layer (derl/models.py:102-103,117-123: `.float()/255` -> nn.Conv2d(4, 32, 8, 4) -> nn.ReLU)
and its backward on the INT8 tensor cores: one operand (the uint8 frame) is exact, the other
(weights forward, the masked gradient backward) is expressed as two signed 8-bit digit planes,
value ~= s * (q1 + q2 / 254).  This module restates that number format step by step so that
its error bounds can be pinned on the CPU against the float64 formulation of the reference; the
forward restates K6t's arithmetic exactly, so the GPU tests compare the kernel with it bit for bit.
"""
import numpy as np

MAGIC = np.float32(12582912.0)   # 1.5 * 2^23: x + MAGIC - MAGIC == rint(x) for |x| < 2^22
F = np.float32


def patches(frames):
  """uint8 [B,84,84,4] -> int64 view [B,20,20,8,8,4]: x[b, 4oy+kh, 4ox+kw, c]."""
  b, h, w, c = frames.shape
  sb, sh, sw, sc = frames.strides
  view = np.lib.stride_tricks.as_strided(frames, (b, 20, 20, 8, 8, c),
                                         (sb, 4 * sh, 4 * sw, sh, sw, sc), writeable=False)
  return view.astype(np.int64)


def weight_digits(weight):
  """csrc/stem_tc.cu (digit planes of the weights): per output channel s = max|w| / 127,
  q1 = rint(w / s), q2 = clamp(rint((w - q1 s) * 254 / s), +-127), all in float32."""
  w = weight.astype(F)
  m = np.abs(w).reshape(w.shape[0], -1).max(1)
  s = np.where(m > 0, m / F(127), F(1)).astype(F)
  inv = (F(1) / s).astype(F)
  sb, ib = s[:, None, None, None], inv[:, None, None, None]
  q1 = np.rint(w * ib).astype(F)
  q2 = np.clip(np.rint(((w - q1 * sb) * F(254)) * ib), -127, 127).astype(F)
  return s, q1.astype(np.int64), q2.astype(np.int64)


def stem_forward(frames, weight, bias, chunk=64):
  """K6t: relu(conv(frames / 255, weight, bias, stride 4)) -> float32 [B,20,20,32], bit for bit:
  both = acc1 * 254 + acc2 (exact), y = relu(float(both) * float32(s / 64770) + bias), each step
  rounded to float32 as in the kernel's epilogue.  The digit sums run as a float32 matmul, which
  is exact: every partial sum is an integer of magnitude <= 256 * 255 * 127 < 2^24."""
  s, q1, q2 = weight_digits(weight)
  w = np.concatenate([q1, q2]).transpose(2, 3, 1, 0).reshape(256, 64).astype(F)   # [(kh,kw,c), n']
  es = (s / F(64770)).astype(F)
  b = bias.astype(F)
  out = np.empty((frames.shape[0], 20, 20, 32), F)
  for i in range(0, frames.shape[0], chunk):
    acc = (patches(frames[i:i + chunk]).reshape(-1, 256).astype(F) @ w).astype(np.int64)
    both = acc[:, :32] * 254 + acc[:, 32:]
    y = (both.astype(F) * es).astype(F) + b
    out[i:i + chunk] = np.maximum(y, F(0)).reshape(-1, 20, 20, 32)
  return out, (s, q1, q2)


def gradient_digits(masked):
  """csrc/stem_bwd_tc.cu `quantise2`: per (frame, channel) s = max|g| / 127; x = g / s;
  q1 = rint(x) and q2 = rint((x - q1) * 254) by the magic-number trick (the second one through
  one fused multiply-add), |q2| <= 127 because |x - q1| <= 1/2."""
  g = masked.astype(F)                                   # [B,20,20,32]
  m = np.abs(g).max(axis=(1, 2), keepdims=True)
  s = np.where(m > 0, m / F(127), F(1)).astype(F)
  inv = (F(1) / s).astype(F)
  x = (g * inv).astype(F)
  q1 = ((x + MAGIC).astype(F) - MAGIC).astype(F)
  d = (x - q1).astype(F)
  q2 = (d.astype(np.float64) * 254.0 + float(MAGIC)).astype(F) - MAGIC   # fma: one rounding
  return s, q1.astype(np.int64), q2.astype(np.int64)


def stem_backward(frames, grad_out, out):
  """K7t: (grad_weight [32,4,8,8], grad_bias [32]) of the layer given the gradient w.r.t. its
  output and the saved output (both [B,20,20,32]; the ReLU mask is out > 0); per-frame int
  accumulation is exact, frames are combined in float64 here (the kernel: float32 per CTA, then
  float64 across CTAs)."""
  masked = np.where(out > 0, grad_out, 0).astype(F)
  s, q1, q2 = gradient_digits(masked)
  x = patches(frames)
  acc1 = np.einsum("bijn,bijklc->bnckl", q1, x)         # exact integers
  acc2 = np.einsum("bijn,bijklc->bnckl", q2, x)
  per_frame = acc1.astype(np.float64) + acc2.astype(np.float64) / 254.0
  grad_w = (per_frame * s.reshape(-1, 32, 1, 1, 1).astype(np.float64)).sum(0) / 255.0
  grad_b = masked.astype(np.float64).sum((0, 1, 2))
  return grad_w, grad_b, (s, q1, q2)
