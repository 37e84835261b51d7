"""NumPy model of the arithmetic of the derl_b200 stem kernels (test infrastructure).

K6 / K6t (csrc/stem.cu, csrc/stem_tc.cu) and K7t (csrc/stem_bwd_tc.cu) evaluate the reference's
first layer (derl/models.py:102-103,117-123: `.float()/255` -> nn.Conv2d(4, 32, 8, 4) -> nn.ReLU)
and its backward on the INT8 tensor cores: one operand (the uint8 frame) is exact, the other
(weights forward, the masked gradient backward) is expressed as two signed 8-bit digit planes,
value ~= s * (q1 + q2 / 254).  This module restates that number format step by step so that
its error bounds can be pinned on the CPU against the float64 formulation of the reference.
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
  """csrc/stem.cu (digit planes of the weights): per output channel s = max|w| / 127,
  q1 = rint(w / s), q2 = clamp(rint((w - q1 s) * 254 / s), +-127), all in float32."""
  w = weight.astype(F)
  m = np.abs(w).reshape(w.shape[0], -1).max(1)
  s = np.where(m > 0, m / F(127), F(1)).astype(F)
  inv = (F(1) / s).astype(F)
  sb, ib = s[:, None, None, None], inv[:, None, None, None]
  q1 = np.rint(w * ib).astype(F)
  q2 = np.clip(np.rint(((w - q1 * sb) * F(254)) * ib), -127, 127).astype(F)
  return s, q1.astype(np.int64), q2.astype(np.int64)


def stem_forward(frames, weight, bias):
  """K6: relu(conv(frames / 255, weight, bias, stride 4)) -> float32 [B,20,20,32]."""
  s, q1, q2 = weight_digits(weight)
  x = patches(frames)
  acc1 = np.einsum("bijklc,nckl->bijn", x, q1)          # exact integers (|.| < 2^24)
  acc2 = np.einsum("bijklc,nckl->bijn", x, q2)
  scale = (s * F(1.0 / 255.0)).astype(F)
  y = (acc1.astype(F) + acc2.astype(F) * F(1.0 / 254.0)).astype(F) * scale
  y = y.astype(F) + bias.astype(F)
  return np.maximum(y, F(0)).astype(F), (s, q1, q2)


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
