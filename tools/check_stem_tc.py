"""Hardware check of the tcgen05 stem kernel (K6t) against the NumPy restatement of its number
format (tests/stem_model.py, bit-exact expected), the bf16 output against the float32 one rounded
to nearest even (bit-exact), and an fp32 convolution (<= 1e-4 of the activation scale); then the
kernel's time with float32 and with bf16 output.  Progressive batch sizes, flushed output, so that
a hang or a wrong descriptor shows where it happened."""
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import derl_b200  # noqa: E402,F401
import stem_model  # noqa: E402

K = torch.ops.derl_b200


def run(frames, weight, bias, dtype, out_block, rows):
  out = K.stem_conv_relu(frames, weight, bias, dtype, out_block, rows)
  torch.cuda.synchronize()
  return out


def main():
  torch.manual_seed(0)
  gen = torch.Generator(device="cuda").manual_seed(1)
  weight = torch.randn(32, 4, 8, 8, device="cuda", generator=gen) * 0.1
  bias = torch.randn(32, device="cuda", generator=gen) * 0.1
  torch.backends.cudnn.allow_tf32 = False
  ok = True
  for batch in (1, 2, 3, 7, 148, 149, 300, 1000):
    frames = torch.randint(0, 256, (batch, 84, 84, 4), dtype=torch.uint8, device="cuda",
                           generator=gen)
    model, _ = stem_model.stem_forward(frames.cpu().numpy(), weight.cpu().numpy(),
                                       bias.cpu().numpy())
    model = torch.from_numpy(model).cuda()
    for out_block in (1, 2):
      for use_rows in (False, True):
        rows = torch.randint(0, batch, (batch + 5,), device="cuda", generator=gen) \
            if use_rows else None
        t0 = time.time()
        want = model if rows is None else model[rows]
        if out_block == 2:
          want = K.space_to_depth(want, 2, False)
        got = run(frames, weight, bias, torch.float32, out_block, rows)
        half = run(frames, weight, bias, torch.bfloat16, out_block, rows)
        same = torch.equal(got, want)
        same_half = torch.equal(half, got.to(torch.bfloat16))
        diff = (got - want).abs().max().item()
        msg = f"batch {batch} out_block {out_block} rows {use_rows}: model bit-identical {same} " \
              f"max|diff| {diff:.3e}, bf16 = rn(f32) {same_half} ({time.time() - t0:.2f}s)"
        if not same:
          bad = (got != want).nonzero()
          msg += f"  first mismatches {bad[:4].tolist()} of {bad.shape[0]}"
        ok = ok and same and same_half
        print(msg, flush=True)
    src = frames.permute(0, 3, 1, 2).float() / 255
    want = torch.relu(torch.nn.functional.conv2d(src, weight, bias, stride=4)).permute(0, 2, 3, 1)
    got = run(frames, weight, bias, torch.float32, 1, None)
    err = (got - want).abs().max().item() / want.abs().max().item()
    print(f"batch {batch}: vs fp32 conv, max err / scale = {err:.3e}", flush=True)
    ok = ok and err < 1e-4
  # timing, 32768 frames, both output types
  frames = torch.randint(0, 256, (32768, 84, 84, 4), dtype=torch.uint8, device="cuda", generator=gen)
  for dtype, size in ((torch.float32, 4), (torch.bfloat16, 2)):
    for block in (1, 2):
      run(frames, weight, bias, dtype, block, None)
      s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      s.record()
      for _ in range(5):
        K.stem_conv_relu(frames, weight, bias, dtype, block, None)
      e.record()
      torch.cuda.synchronize()
      ms = s.elapsed_time(e) / 5
      gbs = 32768 * (28224 + 400 * 32 * size) / ms / 1e6
      print(f"{str(dtype)[6:]:8s} out_block {block}: {ms:.3f} ms per 32768 frames, {gbs:.0f} GB/s",
            flush=True)
  print("OK" if ok else "MISMATCH", flush=True)
  return 0 if ok else 1


if __name__ == "__main__":
  sys.exit(main())
