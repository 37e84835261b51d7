"""Pins, on the CPU, the number format the INT8 stem kernels (K6t forward, K7t backward) use
against the float64 formulation of the reference's first layer (derl/models.py:102-103,
117-123).  The GPU parity tests check the kernels against float32 convolutions; these tests
check the format itself: digit ranges, the <= s/508 residual, and the end-to-end error of the
activations and of the weight gradient — the claims made in DESIGN.md §3 K6t / K7t."""
import numpy as np

from stem_model import gradient_digits, patches, stem_backward, stem_forward, weight_digits


def _inputs(batch, seed):
  rng = np.random.RandomState(seed)
  frames = rng.randint(0, 256, (batch, 84, 84, 4)).astype(np.uint8)
  weight = (rng.standard_normal((32, 4, 8, 8)) * 0.08).astype(np.float32)
  bias = (rng.standard_normal(32) * 0.1).astype(np.float32)
  return rng, frames, weight, bias


def _exact_forward(frames, weight, bias):
  pre = np.einsum("bijklc,nckl->bijn", patches(frames).astype(np.float64) / 255.0,
                  weight.astype(np.float64)) + bias.astype(np.float64)
  return np.maximum(pre, 0.0)


def test_weight_digit_planes_residual_and_range():
  _, _, weight, _ = _inputs(1, 0)
  weight[5] = 0.0                                        # an all-zero channel keeps s = 1
  s, q1, q2 = weight_digits(weight)
  assert np.abs(q1).max() <= 127 and np.abs(q2).max() <= 127 and s[5] == 1.0
  recon = s[:, None, None, None].astype(np.float64) * (q1 + q2 / 254.0)
  resid = np.abs(recon - weight.astype(np.float64)).reshape(32, -1).max(1)
  assert np.all(resid <= s.astype(np.float64) / 508.0 * 1.01 + 1e-12)


def test_forward_model_error_against_float64_convolution():
  _, frames, weight, bias = _inputs(3, 1)
  got, _ = stem_forward(frames, weight, bias)
  want = _exact_forward(frames, weight, bias)
  assert got.dtype == np.float32 and got.shape == (3, 20, 20, 32)
  err = np.abs(got - want).max() / np.abs(want).max()
  assert err < 1e-4, err                                 # DESIGN: <= 1e-4 of the activation scale
  assert ((got > 0) != (want > 0)).mean() < 1e-3         # ReLU mask flips only within ~1e-5 of 0


def test_gradient_digit_planes_per_frame_and_channel():
  rng = np.random.RandomState(2)
  g = (rng.standard_normal((4, 20, 20, 32)) * rng.rand(4, 1, 1, 32) * 1e-3).astype(np.float32)
  g[1, :, :, 7] = 0.0                                    # dead channel in one frame
  g[2, 3, 4, :] *= 50                                    # outliers set the per-channel scale
  s, q1, q2 = gradient_digits(g)
  assert s.shape == (4, 1, 1, 32) and s[1, 0, 0, 7] == 1.0
  assert np.abs(q1).max() <= 127 and np.abs(q2).max() <= 127
  recon = s.astype(np.float64) * (q1 + q2 / 254.0)
  # s / 508 plus the float32 rounding of g / s (|x| <= 127: 127 * 2^-24 in digit units)
  assert np.all(np.abs(recon - g) <= s.astype(np.float64) / 508.0 * 1.01 + 1e-18)


def test_backward_model_error_against_float64_gradient():
  rng, frames, weight, bias = _inputs(6, 3)
  out, _ = stem_forward(frames, weight, bias)
  grad = (rng.standard_normal(out.shape) * rng.rand(6, 1, 1, 1) * 1e-3).astype(np.float32)
  got_w, got_b, _ = stem_backward(frames, grad, out)
  masked = np.where(out > 0, grad, 0).astype(np.float64)
  want_w = np.einsum("bijn,bijklc->nckl", masked, patches(frames).astype(np.float64) / 255.0)
  want_b = masked.sum((0, 1, 2))
  err_w = np.abs(got_w - want_w).max() / np.abs(want_w).max()
  err_b = np.abs(got_b - want_b).max() / np.abs(want_b).max()
  assert got_w.shape == (32, 4, 8, 8)
  assert err_w < 5e-5 and err_b < 1e-12, (err_w, err_b)  # DESIGN: 2.3e-5 measured on the GPU
