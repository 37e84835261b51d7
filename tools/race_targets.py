"""One small launch of every kernel with an mbarrier / TMA pipeline (K1 TMA scan, K2 row gather,
K6t stem forward, K7t stem backward), for `compute-sanitizer --tool racecheck` (shared-
memory hazards) or `--tool memcheck` / `--tool synccheck`:

    compute-sanitizer --tool racecheck python tools/race_targets.py [repeats]
"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import derl_b200  # noqa: E402,F401

K = torch.ops.derl_b200


def main():
  repeats = int(sys.argv[1]) if len(sys.argv) > 1 else 1
  gen = torch.Generator(device="cuda").manual_seed(0)
  for _ in range(repeats):
    # K1: TMA variant, several time tiles, ragged last strip
    nsteps, nenvs = 70, 304
    rewards = torch.randn(nsteps, nenvs, device="cuda", generator=gen)
    values = torch.randn(nsteps, nenvs, device="cuda", generator=gen)
    resets = torch.rand(nsteps, nenvs, device="cuda", generator=gen) < 0.05
    last = torch.randn(nenvs, device="cuda", generator=gen)
    K.gae(rewards, values, resets, last, 0.99, 0.95, True, 2)
    # K2: TMA row gather (28 224-byte rows), more units than CTAs
    frames = torch.randint(0, 256, (400, 84, 84, 4), dtype=torch.uint8, device="cuda", generator=gen)
    perm = torch.randperm(400, device="cuda", generator=gen)
    K.gather_rows(frames, perm, 3, 390)
    # K6t (bf16, float32 with mask, float32) / K7t
    weight = torch.randn(32, 4, 8, 8, device="cuda", generator=gen) * 0.1
    bias = torch.randn(32, device="cuda", generator=gen) * 0.1
    K.stem_conv_relu(frames, weight, bias, torch.bfloat16, 2, None)
    out, mask = K.stem_conv_relu_mask(frames, weight, bias, 2, perm)
    K.stem_conv_relu(frames, weight, bias, torch.float32, 1, None)
    grad = torch.randn(400, 128, 10, 10, device="cuda", generator=gen).contiguous(
        memory_format=torch.channels_last)
    K.stem_backward_masked(frames, grad, mask, True, perm)
  torch.cuda.synchronize()
  print("race targets done")


if __name__ == "__main__":
  main()
