"""Launches each hand-written kernel a few times at its headline size, for ncu captures:

  python tools/profile_kernels.py                       # plain run (must exit 0 first)
  ncu --set full --clock-control none --import-source on \
      -k regex:'gather_rows_tma|gae_tma|gae_direct|ppo_loss|ppo_mlp|gather_columns|frames_to_s2d|relu_bwd|stem_' -c 80 \
      -o gpurun_out/kernels python tools/profile_kernels.py

Sizes: gather = one 131072-row minibatch out of a 4096x128 frame-stack rollout (14.8 GB,
config 3); GAE = T2048 x N65536 (config 5 maximum, 2.28 GB of traffic); loss = B 131072.
Prints CUDA-event times so the plain run doubles as a quick microbenchmark.
"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import derl_b200  # noqa: E402,F401

K = torch.ops.derl_b200
DEV = "cuda"
REPS = int(os.environ.get("REPS", "3"))


def timed(name, fn, nbytes):
  times = []
  for _ in range(REPS):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    fn()
    e.record()
    torch.cuda.synchronize()
    times.append(s.elapsed_time(e))
  ms = min(times)
  print(f"{name:28s} {ms:9.4f} ms  {nbytes / ms / 1e6:9.1f} GB/s", flush=True)


def main():
  gen = torch.Generator(device=DEV).manual_seed(0)
  # ---- GAE sweep maximum
  nsteps, nenvs = 2048, 65536
  rewards = torch.randn(nsteps, nenvs, device=DEV, generator=gen)
  values = torch.randn(nsteps, nenvs, device=DEV, generator=gen)
  resets = torch.rand(nsteps, nenvs, device=DEV, generator=gen) < 0.01
  last = torch.randn(nenvs, device=DEV, generator=gen)
  nbytes = 17.0 * nsteps * nenvs
  timed("gae_tma   T2048 N65536", lambda: K.gae(rewards, values, resets, last, .99, .95, False, 2),
        nbytes)
  timed("gae_direct T2048 N65536", lambda: K.gae(rewards, values, resets, last, .99, .95, False, 1),
        nbytes)
  nsm = 128 * 4096
  timed("gae_tma   T128 N4096", lambda: K.gae(rewards[:128, :4096].contiguous(),
                                               values[:128, :4096].contiguous(),
                                               resets[:128, :4096].contiguous(), last[:4096],
                                               .99, .95, False, 2), 17.0 * nsm)
  del rewards, values, resets
  # ---- loss, config-3 minibatch
  nb, nact = 131072, 4
  logits = torch.randn(nb, nact, device=DEV, generator=gen)
  vals = torch.randn(nb, 1, device=DEV, generator=gen)
  acts = torch.randint(0, nact, (nb,), device=DEV, generator=gen)
  vec = lambda: torch.randn(nb, device=DEV, generator=gen)
  old_lp, adv, vt, vold = vec() * .1 - 1.4, vec(), vec().reshape(nb, 1), vec().reshape(nb, 1)
  timed("ppo_loss_categorical B131072",
        lambda: K.ppo_loss_categorical(logits, vals, acts, old_lp, adv, vt, vold, .1, .25, .01),
        (8 * nact + 32.0) * nb)
  loc, scale = torch.randn(nb, 6, device=DEV, generator=gen), torch.rand(nb, 6, device=DEV) + .5
  cact = torch.randn(nb, 6, device=DEV, generator=gen)
  timed("ppo_loss_gaussian B131072",
        lambda: K.ppo_loss_gaussian(loc, scale, vals, cact, old_lp, adv, vt, vold, .2, .25, 0.),
        (20 * 6 + 24.0) * nb)
  # ---- gather, config-3 minibatch
  nsamples = int(os.environ.get("SAMPLES", 4096 * 128))
  obs = torch.randint(0, 256, (nsamples, 84, 84, 4), device=DEV, dtype=torch.uint8, generator=gen)
  perm = torch.from_numpy(np.random.RandomState(0).permutation(nsamples)).to(DEV)
  mb = nsamples // 4
  state = {"i": 0}

  def gather():
    state["i"] = (state["i"] + 1) % 4
    return K.gather_rows(obs, perm, state["i"] * mb, mb)
  timed("gather_rows_tma 131072x28224", gather, (8 + 2 * 28224.0) * mb)
  wstem = torch.randn(32, 4, 8, 8, device=DEV, generator=gen) * .1
  bstem = torch.zeros(32, device=DEV)
  for blk in (1, 2):
    timed(f"stem_conv_relu 32768 f32 blk{blk}",
          lambda: K.stem_conv_relu(obs[:32768], wstem, bstem, torch.float32, blk),
          32768 * (28224 + 400 * 32 * 4.0))
  timed("stem_conv_relu_mask 32768 blk2 (K6t)",
        lambda: K.stem_conv_relu_mask(obs[:32768], wstem, bstem, 2),
        32768 * (28224 + 400 * 32 * 4.0 + 1792))
  timed("stem_conv_relu 32768 bf16 blk2 (K6t)",
        lambda: K.stem_conv_relu(obs[:32768], wstem, bstem, torch.bfloat16, 2),
        32768 * (28224 + 400 * 32 * 2.0))
  act, relu_mask = K.stem_conv_relu_mask(obs[:32768], wstem, bstem, 2)
  act = act.permute(0, 3, 1, 2)
  gact = torch.randn_like(act) * 1e-3
  timed("stem_backward_masked 32768 (K7t)",
        lambda: K.stem_backward_masked(obs[:32768], gact, relu_mask, True),
        32768 * (28224 + 51200.0 + 1792))
  del act, gact, relu_mask
  frames = obs[:16384]
  for dt, nb in ((torch.float32, 5.0), (torch.bfloat16, 3.0)):
    timed(f"frames_to_s2d 16384 {str(dt)[6:]}", lambda: K.frames_to_s2d(frames, 4, dt, 255.0),
          nb * frames.numel())
  act = torch.relu(torch.randn(32768, 32, 20, 20, device=DEV, generator=gen)).contiguous(
      memory_format=torch.channels_last)
  gact = torch.randn_like(act)
  timed("relu_bwd_bias 32768x32x20x20", lambda: K.relu_bwd_bias(gact, act), 12.0 * act.numel())
  del act, gact
  for hw in (9, 7):   # the conv2 / conv3 activations of a 32768-frame micro-batch
    act = torch.relu(torch.randn(32768, 64, hw, hw, device=DEV, generator=gen)).contiguous(
        memory_format=torch.channels_last)
    gact = torch.randn_like(act)
    timed(f"relu_bwd_bias 32768x64x{hw}x{hw}", lambda: K.relu_bwd_bias(gact, act), 12.0 * act.numel())
    del act, gact
  cols = [adv.repeat(4), vt.reshape(-1).repeat(4), vold.reshape(-1).repeat(4), old_lp.repeat(4),
          acts.repeat(4)]
  timed("gather_columns 5 cols", lambda: K.gather_columns(cols, perm, mb, mb, 0),
        (8 + 2 * 24.0) * mb)
  # ---- K8: one whole MuJoCo-shaped update (2048 samples, 10 epochs x 32 minibatches of 64)
  size, odim, adim = 2048, 17, 6
  shapes = [(64, odim), (64,), (64, 64), (64,), (adim, 64), (adim,),
            (64, odim), (64,), (64, 64), (64,), (1, 64), (1,), (adim,)]
  params = [torch.randn(sh, device=DEV, generator=gen) * .1 for sh in shapes]
  m1 = [torch.zeros_like(p) for p in params]
  m2 = [torch.zeros_like(p) for p in params]
  mobs = torch.randn(size, odim, device=DEV, generator=gen, dtype=torch.float64)
  mact = torch.randn(size, adim, device=DEV, generator=gen)
  mcol = lambda: torch.randn(size, device=DEV, generator=gen)
  mlp, madv, mvt, mval = mcol() * .1 - 8, mcol(), mcol(), mcol()
  mperm = torch.cat([torch.randperm(size, device=DEV, generator=gen) for _ in range(10)])
  timed("ppo_mlp_update 2048 x 10 x 32 (K8)",
        lambda: K.ppo_mlp_update(params, m1, m2, mobs, mact, mlp, madv, mvt, mval, mperm, 10, 64,
                                 True, 1e-8, .2, .25, 0., .5, 3e-4, .9, .999, 1e-5, 0),
        320 * 64 * (17 * 8 + 6 * 4 + 16.0))


if __name__ == "__main__":
  main()
