"""Hardware check of the tcgen05 stem backward (K7t) and of the ReLU mask K6t emits, against
float32 autograd (tolerances of tests/test_gpu_parity.py)."""
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import derl_b200  # noqa: E402,F401

K = torch.ops.derl_b200


def s2d2(x):   # [B,20,20,32] -> [B,10,10,128]
  return K.space_to_depth(x.contiguous(), 2, False)


def expected_mask(out):
  """[B, 14, 32] words: bit l of (t, c) = out[b, oy, ox, c] > 0 at padded pixel 21 oy + ox = 32 t + l."""
  batch = out.shape[0]
  m = torch.arange(448, device=out.device)
  oy, ox = m // 21, m % 21
  valid = (m < 420) & (ox < 20)
  pos = torch.zeros(batch, 448, 32, dtype=torch.int64, device=out.device)
  pos[:, valid] = (out[:, oy[valid], ox[valid], :] > 0).to(torch.int64)
  weights = (1 << torch.arange(32, device=out.device, dtype=torch.int64)).view(1, 1, 32, 1)
  return (pos.view(batch, 14, 32, 32) * weights).sum(2)


def profile_only():
  """A short run for ncu: K6t (with mask) and K7t on 8192 frames."""
  gen = torch.Generator(device="cuda").manual_seed(1)
  weight = torch.randn(32, 4, 8, 8, device="cuda", generator=gen) * 0.1
  bias = torch.randn(32, device="cuda", generator=gen) * 0.1
  frames = torch.randint(0, 256, (8192, 84, 84, 4), dtype=torch.uint8, device="cuda", generator=gen)
  g_in = torch.randn(8192, 128, 10, 10, device="cuda", generator=gen).contiguous(
      memory_format=torch.channels_last)
  for _ in range(3):
    out, mask = K.stem_conv_relu_mask(frames, weight, bias, 2, None)
    K.stem_conv_relu(frames, weight, bias, torch.float32, 2, None)
    K.stem_backward_masked(frames, g_in, mask, True, None)
  torch.cuda.synchronize()
  return 0


def main():
  if "--profile" in sys.argv:
    return profile_only()
  gen = torch.Generator(device="cuda").manual_seed(1)
  weight = (torch.randn(32, 4, 8, 8, device="cuda", generator=gen) * 0.1).requires_grad_()
  bias = (torch.randn(32, device="cuda", generator=gen) * 0.1).requires_grad_()
  torch.backends.cudnn.allow_tf32 = False
  ok = True
  for batch in (1, 2, 5, 148, 149, 600):
    frames = torch.randint(0, 256, (batch, 84, 84, 4), dtype=torch.uint8, device="cuda",
                           generator=gen)
    out, mask = K.stem_conv_relu_mask(frames, weight.detach(), bias.detach(), 1, None)
    torch.cuda.synchronize()
    mask_ok = torch.equal(mask.to(torch.int64) & 0xffffffff, expected_mask(out))
    grad = torch.randn(batch, 20, 20, 32, device="cuda", generator=gen)
    grad[batch // 2] *= 1e-3    # a frame with small gradients: block floating point is per frame
    # float32 reference with the SAME ReLU mask (the kernels' own: a sign flip of a near-zero
    # pre-activation between the int8 path and cuDNN is not what is being measured here)
    src = frames.permute(0, 3, 1, 2).float() / 255
    pre = torch.nn.functional.conv2d(src, weight, bias, stride=4)
    keep = (out > 0).permute(0, 3, 1, 2).float()
    gw, gb = torch.autograd.grad(pre, (weight, bias), grad.permute(0, 3, 1, 2) * keep)
    for blocked in (False, True):
      g_in = (s2d2(grad) if blocked else grad).permute(0, 3, 1, 2)
      t0 = time.time()
      nw, nb = K.stem_backward_masked(frames, g_in, mask, blocked, None)
      torch.cuda.synchronize()
      ew = (nw - gw).abs().max().item() / gw.abs().max().item()
      eb = (nb - gb).abs().max().item() / gb.abs().max().item()
      good = ew < 2e-4 and eb < 1e-5
      ok = ok and good and mask_ok
      print(f"batch {batch} blocked {int(blocked)}: mask {mask_ok}  dW err {ew:.2e}  db err {eb:.2e}  "
            f"{'ok' if good else 'BAD'} ({time.time() - t0:.2f}s)", flush=True)
    rows = torch.randint(0, batch, (batch + 3,), device="cuda", generator=gen)
    out_r, mask_r = K.stem_conv_relu_mask(frames, weight.detach(), bias.detach(), 2, rows)
    grad_r = torch.randn(batch + 3, 128, 10, 10, device="cuda", generator=gen).contiguous(
        memory_format=torch.channels_last)
    a = K.stem_backward_masked(frames, grad_r, mask_r, True, rows)
    b = K.stem_backward_masked(frames[rows].contiguous(), grad_r, mask_r, True, None)
    same = torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    again = K.stem_backward_masked(frames, grad_r, mask_r, True, rows)
    det = torch.equal(a[0], again[0])
    ok = ok and same and det
    print(f"batch {batch}: rows == materialised gather {same}, deterministic {det}", flush=True)
  # timing
  nb_ = 32768
  frames = torch.randint(0, 256, (nb_, 84, 84, 4), dtype=torch.uint8, device="cuda", generator=gen)
  out, mask = K.stem_conv_relu_mask(frames, weight.detach(), bias.detach(), 2, None)
  g_in = torch.randn(nb_, 128, 10, 10, device="cuda", generator=gen).contiguous(
      memory_format=torch.channels_last)
  K.stem_backward_masked(frames, g_in, mask, True, None)
  s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  s.record()
  for _ in range(5):
    K.stem_backward_masked(frames, g_in, mask, True, None)
  e.record()
  torch.cuda.synchronize()
  ms = s.elapsed_time(e) / 5
  print(f"K7t: {ms:.3f} ms per {nb_} frames, {nb_ * (28224 + 51200 + 1600) / ms / 1e6:.0f} GB/s of "
        f"its own algorithmic bytes", flush=True)
  s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  s.record()
  for _ in range(5):
    K.stem_conv_relu_mask(frames, weight.detach(), bias.detach(), 2, None)
  e.record()
  torch.cuda.synchronize()
  ms = s.elapsed_time(e) / 5
  print(f"K6t with mask: {ms:.3f} ms per {nb_} frames, {nb_ * (28224 + 51200 + 1600) / ms / 1e6:.0f} GB/s",
        flush=True)
  print("OK" if ok else "MISMATCH", flush=True)
  return 0 if ok else 1


if __name__ == "__main__":
  sys.exit(main())
