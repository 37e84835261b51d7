#!/usr/bin/env python
"""Atari rollouts stored as unique frames (FrameStacks, K10) against the stacked column (K2).

    python tools/bench_frame_stacks.py                 # every arm, one JSON line on stdout
    python tools/bench_frame_stacks.py --packer-only   # the host packer arm alone (no GPU)

Arms, each timed with CUDA events in one process, the two forms alternating step by step:
  kernel    K10 vs K2 per 131 072-row minibatch of a 4096 x 128 rollout (ms, GB/s of algorithmic
            bytes, fraction of the HBM peak of bench.peaks()); inputs are 3.8 / 14.8 GB >> L2
  update    full PPO update (4 epochs x 4 minibatches, TF32 network, 65 536-row micro-batches),
            rollout resident in HBM, stacked vs FrameStacks, same seeds
  e2e       the same update with the rollout starting in pinned host memory: stacked HostColumn
            vs FrameStacks (frames + index uploaded by one copy each)
  capacity  32 768 envs x 128 steps as FrameStacks on one GPU: update time, peak allocation
  packer    FrameStackPacker.pack per step at N = 4096 (host CPU time)
  device_packer  DeviceFrameStackPacker (K11) at N = 4096, 84x84x4: host time per `pack` call
            (NumPy step: pinned staging copy + launches), K11 device time per step from CUDA events
            (launches queued behind a sleep kernel, so no host gap is timed; L2 overwritten with
            256 MB before every step, so the previous step's stacks are not L2-resident), its
            algorithmic bytes and share of HBM peak, and the H2D bytes per step
  collect   seconds per 128-step rollout of EnvRunner(resident_device=...) at N = 4096 on a cheap
            stacking env that shifts in frames from a pre-generated bank: stacked vs
            pack_frames=True (device packing), alternating; the host-packing route
            (pack_frames=True without resident_device) once; and the env + policy alone
    python tools/bench_frame_stacks.py --pack-only     # packer, device_packer and collect arms
The GPU name, power limit and SM clock are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time
import types

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

import bench  # noqa: E402  (build_alg, timed_updates, peaks, ClockSampler, ...)

ROW = 84 * 84 * 4


def gpu_info(index):
  out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.sm,"
                        "clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True).stdout.strip()
  name, power, sm, sm_max = [x.strip() for x in out.split(",")]
  return {"name": name, "power_limit_w": float(power), "sm_mhz_idle": float(sm),
          "sm_max_mhz": float(sm_max)}


def packer_arm(nenvs, steps, seed=0):
  from derl_b200.runners.frame_stacks import FrameStackPacker
  rng = np.random.default_rng(seed)
  stack = rng.integers(0, 256, (nenvs, 84, 84, 4), dtype=np.uint8)
  packer = FrameStackPacker(steps * nenvs + nenvs * 3)
  times = []
  for _ in range(steps):
    t0 = time.perf_counter()
    packer.pack(stack)
    times.append(time.perf_counter() - t0)
    frame = rng.integers(0, 256, (nenvs, 84, 84), dtype=np.uint8)
    stack = np.concatenate([stack[..., 1:], frame[..., None]], axis=-1)
  steady = times[1:]   # the first step allocates the plane store
  return {"nenvs": nenvs, "steps": steps, "ms_per_step": float(np.mean(steady)) * 1e3,
          "ms_per_step_max": float(np.max(steady)) * 1e3, "first_step_ms": times[0] * 1e3,
          "planes": packer.count, "threads": torch.get_num_threads(),
          "what": "host CPU time of FrameStackPacker.pack on [N, 84, 84, 4] uint8 steps"}


class BankEnv:
  """Batched env with baselines-style 84x84x4 stacks that shifts in one frame per step from a
  pre-generated bank, so that collection timings are not dominated by an emulator."""

  def __init__(self, nenvs, bank=8, seed=0):
    rng = np.random.default_rng(seed)
    self.bank = rng.integers(0, 256, (bank, nenvs, 84, 84), dtype=np.uint8)
    self.nenvs, self.t = nenvs, 0
    self.unwrapped = self
    self.stack = None

  def reset(self):
    self.stack = np.stack([self.bank[i] for i in range(4)], -1)
    self.t = 4
    return self.stack

  def step(self, actions):
    self.stack = np.concatenate([self.stack[..., 1:],
                                 self.bank[self.t % len(self.bank)][..., None]], -1)
    self.t += 1
    return self.stack, np.zeros(self.nenvs, np.float32), np.zeros(self.nenvs, bool), {}


class SyncPolicy:
  """Host outputs read back from the device every step, as a GPU policy's are."""

  def __init__(self, nenvs, device):
    self.nenvs, self.device = nenvs, device

  def act(self, obs):
    values = torch.zeros(self.nenvs, device=self.device).cpu().numpy()
    return {"actions": np.zeros(self.nenvs, np.int64), "values": values}


def device_packer_arm(nenvs, steps, peak, peak_kind, device):
  from derl_b200.runners.frame_stacks import DeviceFrameStackPacker
  K = torch.ops.derl_b200
  env = BankEnv(nenvs, seed=3)
  # a bank of 8 frames makes the stacks periodic in 8 steps: cycling these continues the sequence
  host_steps = [env.reset()] + [env.step(None)[0] for _ in range(7)]
  plane = 84 * 84
  # host time per pack call, NumPy input (the EnvRunner route); the device is drained each step,
  # as policy.act does in EnvRunner, so the staging slot never waits
  packer = DeviceFrameStackPacker(device, steps)
  host_ms = []
  for i in range(steps):
    t0 = time.perf_counter()
    packer.pack(host_steps[i % len(host_steps)])
    host_ms.append((time.perf_counter() - t0) * 1e3)
    torch.cuda.synchronize()
  packer.finish()
  del packer
  # K11 device time per step: steps on the device, launches queued behind a sleep kernel
  dev_steps = [torch.from_numpy(s).to(device) for s in host_steps]
  pool = torch.empty((steps * nenvs * 4 + nenvs * 4, 84, 84), dtype=torch.uint8, device=device)
  state = torch.zeros(2, dtype=torch.int64, device=device)
  index = torch.empty((steps, nenvs, 4), dtype=torch.int32, device=device)
  flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)
  for _ in range(2):   # warm-up pass, then the timed pass from an empty pool
    state.zero_()
    torch.cuda.synchronize()
    torch.cuda._sleep(200_000_000)
    events, counts = [], []
    for i in range(steps):
      flush.fill_(i & 255)
      a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      a.record()
      prev = dev_steps[(i - 1) % len(dev_steps)] if i else None
      K.pack_frame_stacks(dev_steps[i % len(dev_steps)], prev, index[i - 1] if i else None, pool,
                          state, index[i])
      b.record()
      events.append((a, b))
      counts.append(state[0].clone())
    torch.cuda.synchronize()
  ms = [a.elapsed_time(b) for a, b in events]
  counts = [0] + [int(c) for c in counts]
  new_planes = [counts[i + 1] - counts[i] for i in range(steps)]
  # steady state: steps after the first (which has no previous step and stores every channel)
  stack_bytes = nenvs * plane * 4
  steady = ms[1:]
  bytes_step = [2 * stack_bytes + 16 * nenvs + new_planes[i] * plane + 16 * nenvs
                for i in range(1, steps)]
  t = float(np.median(steady))
  algo = float(np.median(bytes_step))
  return {"nenvs": nenvs, "steps": steps, "hw": [84, 84], "k": 4,
          "host_ms_per_pack": float(np.median(host_ms[1:])),
          "host_ms_per_pack_max": float(np.max(host_ms[1:])), "host_first_pack_ms": host_ms[0],
          "k11_ms_per_step": t, "k11_ms_min": float(np.min(steady)),
          "k11_first_step_ms": ms[0], "planes_per_step": new_planes[1], "planes_first_step": new_planes[0],
          "algorithmic_bytes_per_step": algo, "GBps": algo / t / 1e6, "frac": algo / t / 1e6 / peak,
          "peak_GBps": peak, "peak_source": peak_kind, "l2": "256 MB overwritten before every step",
          "h2d_bytes_per_step": stack_bytes,
          "what": "host: wall time of DeviceFrameStackPacker.pack on a NumPy step; K11: CUDA events "
                  "around the three launches of one step"}


def collect_arm(nenvs, horizon, rollouts, device):
  import derl_b200 as d

  def runner(**kw):
    env = BankEnv(nenvs, seed=4)
    return d.EnvRunner(env, SyncPolicy(nenvs, device), horizon, nsteps=10 ** 12, **kw).run()

  def timed(it):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = next(it)
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out

  arms = {"stacked": runner(resident_device=device),
          "device_packing": runner(resident_device=device, pack_frames=True)}
  sec = {name: [] for name in arms}
  planes = None
  for i in range(rollouts + 1):
    for name, it in arms.items():
      s, out = timed(it)
      if name == "device_packing":
        planes = out["observations"].num_frames
      del out
      if i:
        sec[name].append(s)
  del arms
  torch.cuda.empty_cache()
  env, policy = BankEnv(nenvs, seed=4), SyncPolicy(nenvs, device)
  obs = env.reset()
  t0 = time.perf_counter()
  for _ in range(horizon):
    policy.act(obs)
    obs = env.step(None)[0]
  env_s = time.perf_counter() - t0
  host_s, out = timed(runner(pack_frames=True))
  host_planes = out["observations"].num_frames
  del out
  result = {"envs": nenvs, "horizon": horizon, "rollouts": rollouts,
            "env_and_policy_s": env_s, "host_packing_s": host_s, "host_packing_planes": host_planes,
            "device_packing_planes": planes,
            "what": "seconds per rollout of EnvRunner.run (resident_device unless host_packing), "
                    "a bank-fed stacking env and a policy that reads its output back each step; "
                    "host_packing is one first rollout (its pinned plane store is allocated in it)"}
  for name, s in sec.items():
    result[name + "_s"] = float(np.mean(s))
    result[name + "_s_each"] = [float(x) for x in s]
  return result


def kernel_arm(stacked_obs, packed_obs, reps, mb_rows, peak, peak_kind):
  K = torch.ops.derl_b200
  src = stacked_obs.reshape(-1, 84, 84, 4)
  frames, index = packed_obs.frames, packed_obs.index.reshape(-1, 4)
  samples = src.shape[0]
  perm = torch.randperm(samples, device=src.device)
  windows = samples // mb_rows
  arms = {"K2_gather_rows": lambda s: K.gather_rows(src, perm, s, mb_rows),
          "K10_gather_frame_stacks": lambda s: K.gather_frame_stacks(frames, index, perm, s,
                                                                     mb_rows)}
  for w in range(windows):   # warm-up, and the two kernels agree on every window
    assert torch.equal(arms["K2_gather_rows"](w * mb_rows),
                       arms["K10_gather_frame_stacks"](w * mb_rows)), w
  torch.cuda.synchronize()
  ms = {name: [] for name in arms}
  for r in range(reps):
    for name, fn in arms.items():
      a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      a.record()
      out = fn((r % windows) * mb_rows)
      b.record()
      b.synchronize()
      ms[name].append(a.elapsed_time(b))
      del out
  bytes_of = {"K2_gather_rows": (8 + 2 * ROW) * mb_rows,
              "K10_gather_frame_stacks": (8 + 4 * 4 + 2 * ROW) * mb_rows}
  result = {"rows": mb_rows, "reps": reps, "peak_GBps": peak, "peak_source": peak_kind}
  for name in arms:
    t = float(np.median(ms[name]))
    gbps = bytes_of[name] / t / 1e6
    result[name] = {"median_ms": t, "min_ms": float(np.min(ms[name])),
                    "bytes_per_launch": bytes_of[name], "GBps": gbps, "frac": gbps / peak}
  result["K10_over_K2"] = result["K10_gather_frame_stacks"]["median_ms"] / \
      result["K2_gather_rows"]["median_ms"]
  return result


class FixedSource:
  """EnvRunner-like source yielding the same rollout dict again and again."""

  def __init__(self, policy, rollout, nenvs, horizon):
    self.policy, self.rollout, self.horizon, self.nenvs = policy, rollout, horizon, nenvs
    self.env = types.SimpleNamespace(nenvs=nenvs)
    self.env.unwrapped = self.env
    self.nsteps, self.step_count = None, 0

  def is_exhausted(self):
    return False

  def run(self, obs=None):
    while True:
      self.step_count += self.horizon * self.nenvs
      out = dict(self.rollout)
      out["state"] = dict(self.rollout["state"])
      yield out


def make_alg(d, args, rollout, nenvs, horizon, device):
  torch.manual_seed(0)
  policy = d.ActorCriticPolicy(d.NatureCNNModel([args.nactions, 1]))
  source = FixedSource(policy, rollout, nenvs, horizon)
  return bench.build_alg(args, d, source, 1, device)


def alternate(arms, nbatches, steps, read_losses):
  """{name: (alg, runner)} -> {name: [seconds per update]}; one warm-up each, then the arms take
  turns, each update seeded alike."""
  sec = {name: [] for name in arms}
  for i in range(steps + 1):
    for name, (alg, runner) in arms.items():
      np.random.seed(1000 + i)
      s, losses = bench.timed_updates(alg, runner, nbatches, 1, 0, 1, read_losses)
      if i:
        sec[name].append(s)
  return sec


def pinned_copy(value):
  if isinstance(value, torch.Tensor):
    out = torch.empty(value.shape, dtype=value.dtype, pin_memory=True)
    out.copy_(value)
    return out
  return value


def main():
  p = argparse.ArgumentParser()
  p.add_argument("--envs", type=int, default=4096)
  p.add_argument("--horizon", type=int, default=128)
  p.add_argument("--capacity-envs", type=int, default=32768)
  p.add_argument("--kernel-reps", type=int, default=40)
  p.add_argument("--steps", type=int, default=3, help="timed updates per arm (update, e2e)")
  p.add_argument("--packer-only", action="store_true")
  p.add_argument("--pack-only", action="store_true",
                 help="packer, device_packer and collect arms only")
  p.add_argument("--pack-steps", type=int, default=64, help="steps timed by device_packer")
  p.add_argument("--collect-rollouts", type=int, default=2)
  p.add_argument("--no-capacity", action="store_true")
  p.add_argument("--no-e2e", action="store_true")
  cli = p.parse_args()
  line = {"metric": "frame_stacks", "packer": packer_arm(4096, 9)}
  if cli.packer_only:
    print(json.dumps(line), flush=True)
    return
  assert torch.cuda.is_available(), "the GPU arms need a B200; --packer-only runs without one"
  import derl_b200 as d
  d.summary.stop_recording()
  device = torch.device("cuda", 0)
  torch.cuda.set_device(device)
  torch.backends.cudnn.benchmark = True
  torch.backends.cudnn.allow_tf32 = True
  torch.backends.cuda.matmul.allow_tf32 = True
  args = types.SimpleNamespace(epochs=4, minibatches=4, micro_batch=65536, nactions=4)
  nenvs, horizon = cli.envs, cli.horizon
  nbatches = args.epochs * args.minibatches
  samples = horizon * nenvs * args.epochs
  peak, peak_kind = bench.peaks()
  line["gpu"] = gpu_info(0)
  line["device_packer"] = device_packer_arm(cli.envs, cli.pack_steps, peak, peak_kind, device)
  torch.cuda.empty_cache()
  line["collect"] = collect_arm(cli.envs, cli.horizon, cli.collect_rollouts, device)
  torch.cuda.empty_cache()
  if cli.pack_only:
    line["gpu_after"] = gpu_info(0)
    print(json.dumps(line), flush=True)
    return

  stacked, packed = d.make_frame_stack_rollout(horizon, nenvs, device=device, seed=1000)
  line["rollout"] = {"envs": nenvs, "horizon": horizon,
                     "stacked_bytes": stacked["observations"].numel(),
                     "frames": packed["observations"].num_frames,
                     "frame_stacks_bytes": packed["observations"].frames.numel()
                     + packed["observations"].index.numel() * 4}

  with bench.ClockSampler(0) as clocks:
    line["kernel"] = kernel_arm(stacked["observations"], packed["observations"], cli.kernel_reps,
                                horizon * nenvs // args.minibatches, peak, peak_kind)
  line["kernel"]["clocks"] = clocks.summary()

  arms = {"stacked": make_alg(d, args, stacked, nenvs, horizon, device),
          "frame_stacks": make_alg(d, args, packed, nenvs, horizon, device)}
  with bench.ClockSampler(0) as clocks:
    sec = alternate(arms, nbatches, cli.steps, False)
  line["update"] = {name: {"ms_per_update": float(np.mean(s)) * 1e3,
                           "M_samples_per_s": samples / float(np.mean(s)) / 1e6,
                           "ms_each": [x * 1e3 for x in s]} for name, s in sec.items()}
  line["update"]["clocks"] = clocks.summary()
  del arms
  torch.cuda.empty_cache()

  if not cli.no_e2e:
    host_stacked = {k: (v if k == "state" else pinned_copy(v).numpy()) for k, v in stacked.items()}
    host_stacked["state"] = {"latest_observations":
                             pinned_copy(stacked["state"]["latest_observations"]).numpy()}
    obs = packed["observations"]
    host_packed = dict(host_stacked, observations=d.FrameStacks(
        pinned_copy(obs.frames.cpu()), pinned_copy(obs.index.cpu()), validate=False))
    del stacked, packed, obs
    torch.cuda.empty_cache()
    arms = {"stacked_host_column": make_alg(d, args, host_stacked, nenvs, horizon, device),
            "frame_stacks_host": make_alg(d, args, host_packed, nenvs, horizon, device)}
    sec = alternate(arms, nbatches, cli.steps, True)
    h2d = bench.concurrent_h2d_gbps(host_stacked["observations"], device, 1)
    narrow = sum(v.nbytes for k, v in host_stacked.items() if k not in ("state", "observations"))
    obs_bytes = {"stacked_host_column": host_stacked["observations"].nbytes,
                 "frame_stacks_host": host_packed["observations"].frames.numel()
                 + host_packed["observations"].index.numel() * 4}
    perm_bytes = args.epochs * horizon * nenvs * 8
    line["e2e"] = {"h2d_GBps": h2d}
    for name, s in sec.items():
      total = obs_bytes[name] + narrow + perm_bytes
      line["e2e"][name] = {"ms_per_update": float(np.mean(s)) * 1e3,
                           "M_samples_per_s": samples / float(np.mean(s)) / 1e6,
                           "h2d_bytes_per_update": total,
                           "h2d_floor_ms": total / h2d / 1e6}
    del arms, host_stacked, host_packed
  else:
    del stacked, packed
  torch.cuda.empty_cache()

  if not cli.no_capacity:
    cap_envs = cli.capacity_envs
    torch.cuda.reset_peak_memory_stats(device)
    _, big = d.make_frame_stack_rollout(horizon, cap_envs, device=device, seed=2000,
                                        stacked=False)
    alg, runner = make_alg(d, args, big, cap_envs, horizon, device)
    np.random.seed(5)
    bench.timed_updates(alg, runner, nbatches, 0, 1, 1, False)
    sec_c, losses = bench.timed_updates(alg, runner, nbatches, 1, 0, 1, False)
    line["capacity"] = {"envs": cap_envs, "horizon": horizon, "gpus": 1,
                        "frames": big["observations"].num_frames,
                        "stacked_bytes_equivalent": cap_envs * horizon * ROW,
                        "ms_per_update": sec_c * 1e3,
                        "M_samples_per_s": horizon * cap_envs * args.epochs / sec_c / 1e6,
                        "max_memory_allocated": torch.cuda.max_memory_allocated(device),
                        "last_loss": float(losses[-1])}
    del alg, runner, big
    torch.cuda.empty_cache()
  line["gpu_after"] = gpu_info(0)
  print(json.dumps(line), flush=True)


if __name__ == "__main__":
  main()
