"""Parity tests proper: the CUDA path (through torch.ops.derl_b200 -> ctypes -> C ABI) against
the oracle and the committed golden vectors.  Integer / byte / index work is bit-exact; GAE
is bit-exact; float32 loss terms within the tolerance stated at each assert (north_star:
fp32 relative 1e-5).  Run on a B200: `pytest -m gpu`."""
import ctypes

import numpy as np
import pytest
import torch

import derl_b200 as d
from derl_b200 import _lib
from oracle import derl_oracle as O

import stem_model

pytestmark = pytest.mark.gpu
K = torch.ops.derl_b200
DEV = "cuda"


def cuda(x):
  return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


def run_gae(rewards, values, resets, last_value, gamma, lambda_, variant=0, want_stats=False):
  nsteps = values.shape[0]
  adv, vt, stats = K.gae(cuda(rewards).reshape(nsteps, -1), cuda(values).reshape(nsteps, -1),
                         cuda(resets).reshape(nsteps, -1), cuda(last_value).reshape(-1),
                         gamma, lambda_, want_stats, variant)
  return adv.cpu().numpy(), vt.cpu().numpy(), stats.cpu().numpy()


def variants_for(nenvs):
  return (0, 1, 2) if nenvs % 16 == 0 and nenvs >= 32 else (0, 1)


class ConstPolicy:
  def __init__(self, last_value, model=None):
    self.last_value, self.model = last_value, model

  def act(self, inputs, state=None, update_state=True, training=False):
    return {"values": self.last_value}

  def is_recurrent(self):
    return False


# =============================================================================== K1: GAE
def test_device_is_sm100_and_library_sees_it():
  assert torch.cuda.get_device_capability()[0] == 10
  assert _lib.load().derl_b200_device_ok() == 0


def test_gae_golden_vectors_bit_exact(golden):
  g = golden("live_gae.npz")
  for i in range(g.ncases):
    c = g.case(i)
    norm = {-1: None, 0: False, 1: True}[int(c["normalize"])]
    nsteps = c["values"].shape[0]
    nenvs = c["values"].size // nsteps
    for variant in variants_for(nenvs):
      traj = dict(rewards=c["rewards"], values=c["values"], resets=c["resets"],
                  state=dict(latest_observations=None))
      gae = d.GAE(ConstPolicy(c["last_value"]), gamma=float(c["gamma"]),
                  lambda_=float(c["lambda_"]), normalize=norm, variant=variant)
      adv, vt = gae(traj)
      assert isinstance(adv, np.ndarray) and adv.dtype == np.float32  # NumPy in -> NumPy out
      assert adv.shape == c["advantages"].shape and vt.shape == c["value_targets"].shape
      np.testing.assert_array_equal(vt, c["value_targets"], err_msg=f"case {i} v{variant}")
      normalized = norm or (norm is None and adv.size > 1)
      if not normalized:
        np.testing.assert_array_equal(adv, c["advantages"], err_msg=f"case {i} v{variant}")
      else:  # float64 device moments vs NumPy's float32 pairwise mean/std: tolerance, not bits
        scale = np.abs(c["advantages"]).max()
        np.testing.assert_allclose(adv, c["advantages"], rtol=1e-5, atol=2e-6 * scale)
      assert traj["advantages"] is adv and traj["value_targets"] is vt


def test_gae_reference_fixture(golden):
  g = golden("ref_a2c_atari_gae.npz")
  gamma = float(g["gamma"])
  values = g["values"][..., 0]
  last_value = ((g["advantages"][-1].astype(np.float64) - (g["rewards"][-1] - values[-1]))
                / gamma).astype(np.float32)
  adv, vt, _ = run_gae(g["rewards"], values, g["resets"], last_value, gamma, float(g["lambda_"]))
  np.testing.assert_array_equal(adv[:-1], g["advantages"][:-1])
  np.testing.assert_allclose(adv[-1], g["advantages"][-1], rtol=1e-6)


@pytest.mark.parametrize("nsteps,nenvs,rdtype,reset_prob", [
    (128, 4096, np.float32, 0.01),   # config 3
    (128, 8, np.float64, 0.01),      # config 1
    (2048, 1, np.float64, 0.001),    # config 2 (unbatched)
    (512, 1040, np.float64, 0.05),   # N % 16 == 0, not a multiple of 32: ragged last strip
    (37, 48, np.float32, 0.3),       # T not a multiple of the time tile
    (1, 64, np.float32, 0.5),        # single step: only the two-rounding last row
    (15, 33, np.float64, 0.2),       # direct path only
    (16, 32, np.float32, 1.0),       # every step resets
    (512, 65536, np.float32, 0.01),  # sweep-sized (570 MB of traffic)
])
def test_gae_random_vs_oracle_bit_exact(nsteps, nenvs, rdtype, reset_prob):
  rng = np.random.RandomState(nsteps * 7 + nenvs)
  rewards = rng.standard_normal((nsteps, nenvs)).astype(rdtype)
  values = rng.standard_normal((nsteps, nenvs)).astype(np.float32)
  resets = rng.random((nsteps, nenvs)) < reset_prob
  last_value = rng.standard_normal(nenvs).astype(np.float32)
  want_a, want_vt = O.gae_c(rewards, values, resets, last_value, 0.99, 0.95)
  for variant in variants_for(nenvs):
    adv, vt, stats = run_gae(rewards, values, resets, last_value, 0.99, 0.95, variant, True)
    np.testing.assert_array_equal(adv, want_a, err_msg=f"variant {variant}")
    np.testing.assert_array_equal(vt, want_vt, err_msg=f"variant {variant}")
    a64 = want_a.astype(np.float64)
    np.testing.assert_allclose(stats, [a64.sum(), (a64 * a64).sum(), a64.size], rtol=1e-12)


@pytest.mark.parametrize("cfg", [0, 1, 2, 5])
def test_gae_tma_tile_configurations_are_bit_identical(cfg, monkeypatch):
  """Every TMA tile shape (strip width, warps per CTA, chains per lane, stages) computes the
  same bits as the oracle, including ragged strips and a partial top time-chunk."""
  monkeypatch.setenv("DERL_GAE_TMA_CFG", str(cfg))
  for nsteps, nenvs, rdtype in ((100, 1040, np.float64), (16, 128, np.float32),
                                (3, 48, np.float32), (257, 4096, np.float32)):
    rng = np.random.RandomState(cfg * 100 + nsteps)
    rewards = rng.standard_normal((nsteps, nenvs)).astype(rdtype)
    values = rng.standard_normal((nsteps, nenvs)).astype(np.float32)
    resets = rng.random((nsteps, nenvs)) < 0.05
    last_value = rng.standard_normal(nenvs).astype(np.float32)
    want_a, want_vt = O.gae_c(rewards, values, resets, last_value, 0.99, 0.95)
    adv, vt, stats = run_gae(rewards, values, resets, last_value, 0.99, 0.95, 2, True)
    np.testing.assert_array_equal(adv, want_a)
    np.testing.assert_array_equal(vt, want_vt)
    a64 = want_a.astype(np.float64)
    np.testing.assert_allclose(stats, [a64.sum(), (a64 * a64).sum(), a64.size], rtol=1e-12)


def test_gae_special_values_follow_ieee_like_numpy():
  """inf / nan / signed zeros propagate exactly as NumPy's float64 arithmetic does."""
  nsteps, nenvs = 6, 32
  rng = np.random.RandomState(3)
  rewards = rng.standard_normal((nsteps, nenvs))
  values = rng.standard_normal((nsteps, nenvs)).astype(np.float32)
  resets = rng.random((nsteps, nenvs)) < 0.3
  rewards[2, 0], values[3, 1], rewards[4, 2] = np.inf, np.nan, -0.0
  values[4, 2], values[5, 2], resets[4, 2] = 0.0, -1.0, True
  last_value = rng.standard_normal(nenvs).astype(np.float32)
  with np.errstate(all="ignore"):
    want_a, want_vt = O.gae(rewards, values, resets, last_value, 0.99, 0.95, normalize=False)
  assert np.isnan(want_a).any() and np.isinf(want_a).any()
  for variant in (1, 2):
    adv, vt, _ = run_gae(rewards, values, resets, last_value, 0.99, 0.95, variant)
    # NaN payload bits are not specified by IEEE (x86 yields 0x7FC00000, sm_100 0x7FFFFFFF):
    # compare NaN-ness, then every other bit including the sign of zeros
    for got, want in ((adv, want_a), (vt, want_vt)):
      np.testing.assert_array_equal(np.isnan(got), np.isnan(want))
      finite = ~np.isnan(want)
      np.testing.assert_array_equal(got[finite].view(np.uint32), want[finite].view(np.uint32))


def test_gae_tensor_in_tensor_out_and_unbatched():
  rng = np.random.RandomState(5)
  nsteps = 300
  traj_np = dict(rewards=rng.standard_normal(nsteps), resets=rng.random(nsteps) < .05,
                 values=rng.standard_normal((nsteps, 1)).astype(np.float32))
  last_value = rng.standard_normal(1).astype(np.float32)
  want_a, want_vt = O.gae(traj_np["rewards"], traj_np["values"], traj_np["resets"], last_value,
                          normalize=False)
  traj = {k: cuda(v) for k, v in traj_np.items()}
  traj["state"] = dict(latest_observations=None)
  adv, vt = d.GAE(ConstPolicy(cuda(last_value)), normalize=False)(traj)
  assert adv.is_cuda and adv.shape == (nsteps,) and vt.shape == (nsteps, 1)
  np.testing.assert_array_equal(adv.cpu().numpy(), want_a)
  np.testing.assert_array_equal(vt.cpu().numpy(), want_vt)


def test_gae_host_entry_point_of_the_c_abi():
  """derl_b200_gae_host called with plain NumPy buffers, as a ctypes binding in the
  reference's tree would (INTEGRATION.md)."""
  lib = _lib.load()
  rng = np.random.RandomState(9)
  nsteps, nenvs = 64, 96
  rewards = rng.standard_normal((nsteps, nenvs))
  values = rng.standard_normal((nsteps, nenvs)).astype(np.float32)
  resets = (rng.random((nsteps, nenvs)) < .1).astype(np.uint8)
  last_value = rng.standard_normal(nenvs).astype(np.float32)
  adv, vt = np.empty_like(values), np.empty_like(values)
  ptr = lambda a: a.ctypes.data_as(ctypes.c_void_p)
  for normalize in (0, 1):
    rc = lib.derl_b200_gae_host(ptr(rewards), 1, ptr(values), ptr(resets), ptr(last_value),
                                nsteps, nenvs, 0.99, 0.95, normalize, 1e-8, ptr(adv), ptr(vt),
                                None)
    _lib.check(rc, "gae_host")
    want_a, want_vt = O.gae(rewards, values, resets.astype(bool), last_value, 0.99, 0.95,
                            normalize=bool(normalize))
    np.testing.assert_array_equal(vt, want_vt)
    if normalize:
      np.testing.assert_allclose(adv, want_a, rtol=1e-5, atol=1e-5)
    else:
      np.testing.assert_array_equal(adv, want_a)


def test_moments_and_normalize_vs_numpy():
  rng = np.random.RandomState(11)
  for n in (1, 2, 255, 4097, 1 << 20):
    x = (rng.standard_normal(n) * 3 + 0.7).astype(np.float32)
    stats = K.moments(cuda(x))
    x64 = x.astype(np.float64)
    np.testing.assert_allclose(stats.cpu().numpy(), [x64.sum(), (x64 * x64).sum(), n], rtol=1e-12)
    if n > 1:
      out = K.normalize(cuda(x), stats, 1e-8).cpu().numpy()
      want = O.normalize_advantages(x)
      # float64 device moments vs NumPy float32 pairwise mean/std -> agree to ~1 ulp of the scale
      np.testing.assert_allclose(out, want, rtol=1e-5, atol=2e-6)
      assert abs(out.mean()) < 1e-5 and abs(out.std() - 1) < 1e-4


# =============================================================================== K2: gather
@pytest.mark.parametrize("row_shape,dtype,nrows", [
    ((84, 84, 4), np.uint8, 300),      # frame stacks: TMA bulk path, 28224-B rows
    ((2048,), np.uint8, 257),          # smallest row on the TMA path
    ((65536 + 16,), np.uint8, 40),     # rows wider than one stage: 3 chunks
    ((28672 * 2,), np.uint8, 33),      # exactly two full stages
    ((17,), np.float64, 1000),         # MuJoCo observations: 136-B rows, vector path
    ((6,), np.float32, 999),           # actions [B, 6]
    ((3,), np.uint8, 500),             # odd byte rows
    ((2047,), np.uint8, 129),          # unaligned wide rows: byte path
    ((), np.int64, 4096),              # scalar column
])
def test_gather_rows_bit_exact(row_shape, dtype, nrows):
  rng = np.random.RandomState(nrows)
  if np.issubdtype(dtype, np.integer):
    src = rng.randint(0, 255, (nrows,) + row_shape).astype(dtype)
  else:
    src = rng.standard_normal((nrows,) + row_shape).astype(dtype)
  perm = rng.permutation(nrows).astype(np.int64)
  src_d, perm_d = cuda(src), cuda(perm)
  for start, count in ((0, nrows), (0, 1), (nrows - 1, 1), (nrows // 3, nrows // 2), (5, 0)):
    out = K.gather_rows(src_d, perm_d, start, count).cpu().numpy()
    np.testing.assert_array_equal(out, src[perm[start:start + count]])
    np.testing.assert_array_equal(out, O.gather_rows_c(src, perm, start, count))
  # repeated indices are legal for an index gather (Take), not only permutations
  idx = rng.randint(0, nrows, 2 * nrows).astype(np.int64)
  out = K.gather_rows(src_d, cuda(idx), 0, idx.size).cpu().numpy()
  np.testing.assert_array_equal(out, src[idx])


def test_gather_index_validation_switch(monkeypatch):
  from derl_b200 import ops
  src, bad = cuda(np.arange(40, dtype=np.float32).reshape(10, 4)), cuda(np.array([0, 3, 10]))
  monkeypatch.setattr(ops, "CHECK_INDICES", True)
  with pytest.raises(IndexError, match="out of range"):
    K.gather_rows(src, bad, 0, 3)
  assert torch.equal(K.gather_rows(src, bad, 0, 2), src[[0, 3]])


def test_gather_columns_bit_exact_with_fused_moments():
  rng = np.random.RandomState(21)
  n = 5000
  cols = dict(actions=rng.randint(0, 18, n).astype(np.int64),
              log_prob=rng.standard_normal(n).astype(np.float32),
              advantages=(rng.standard_normal(n) * 2 + .3).astype(np.float32),
              value_targets=rng.standard_normal((n, 1)).astype(np.float32),
              values=rng.standard_normal((n, 1)).astype(np.float32),
              rewards=rng.standard_normal(n), resets=rng.random(n) < .1,
              cont_actions=rng.standard_normal((n, 6)).astype(np.float32),
              odd=rng.randint(0, 255, (n, 3)).astype(np.uint8),
              half=rng.standard_normal((n, 5)).astype(np.float16))
  keys = list(cols)
  perm = rng.permutation(n).astype(np.int64)
  dev = [cuda(cols[k]) for k in keys]
  for start, count in ((0, n), (1234, 1250), (n - 1, 1), (0, 0)):
    *outs, moments = K.gather_columns(dev, cuda(perm), start, count, keys.index("advantages"))
    rows = perm[start:start + count]
    for key, out in zip(keys, outs):
      np.testing.assert_array_equal(out.cpu().numpy(), cols[key][rows], err_msg=key)
    if count:
      a = cols["advantages"][rows].astype(np.float64)
      np.testing.assert_allclose(moments.cpu().numpy(), [a.sum(), (a * a).sum(), count],
                                 rtol=1e-12)
  *outs, moments = K.gather_columns(dev[:2], cuda(perm), 0, 100, -1)
  assert moments.numel() == 0 and len(outs) == 2


def test_gather_full_config3_minibatch_against_torch_index():
  """4096 envs x 128 steps of frame stacks (14.8 GB resident), one 131072-sample minibatch:
  bit-identical to torch's own advanced indexing, and a gather with the inverse permutation
  restores the rollout (round trip) on a 1/8 slice."""
  nsamples = 4096 * 128
  gen = torch.Generator(device=DEV).manual_seed(0)
  obs = torch.randint(0, 256, (nsamples, 84, 84, 4), generator=gen, device=DEV,
                      dtype=torch.uint8)
  np.random.seed(0)
  perm = torch.from_numpy(np.random.permutation(nsamples)).to(DEV)
  mb = nsamples // 4
  out = K.gather_rows(obs, perm, mb, mb)
  for lo in range(0, mb, 16384):
    want = obs[perm[mb + lo:mb + lo + 16384]]
    assert torch.equal(out[lo:lo + 16384], want)
  del want
  inverse = torch.empty_like(perm)
  inverse[perm[mb:2 * mb]] = torch.arange(mb, device=DEV)
  # rows perm[mb:2mb] scattered back: out[inverse[r]] == obs[r] for every r in that set
  some = perm[mb:mb + 65536]
  back = K.gather_rows(out, inverse[some].contiguous(), 0, some.numel())
  assert torch.equal(back, obs[some])


def test_minibatch_pipeline_matches_reference_golden(golden):
  """TransformInteractions[GAE, MergeTimeBatch] -> IterateWithMinibatches ->
  TransformInteractions[NormalizeAdvantages] under np.random.seed: same rows in every
  minibatch as the reference selected (ids bit-exact, ragged tails included)."""
  g = golden("live_minibatches.npz")
  for i in range(g.ncases):
    c = g.case(i)
    nsteps, nenvs = c["ids"].shape
    rollout = {k: c[k] for k in ("observations", "ids", "actions", "log_prob", "values",
                                 "rewards", "resets")}
    rollout["state"] = dict(latest_observations=np.zeros((nenvs, 4, 3, 2), np.uint8))

    class Source:
      env = type("E", (), {"nenvs": nenvs, "unwrapped": property(lambda s: s)})()
      policy = ConstPolicy(c["last_value"])
      horizon, step_count = 1, 0
      nsteps = 1

      def run(self, obs=None):
        yield dict(rollout)

    runner = d.ppo_runner_wrap(Source(), num_epochs=int(c["epochs"]),
                               num_minibatches=int(c["nmb"]))
    np.random.seed(int(c["seed"]))
    flat_obs = c["observations"].reshape((nsteps * nenvs,) + c["observations"].shape[2:])
    ids, advs, sizes = [], [], []
    for batch in runner.run():
      assert list(batch.keys())[:3] == ["observations", "ids", "actions"]
      rows = batch["ids"].cpu().numpy()
      np.testing.assert_array_equal(batch["observations"].cpu().numpy(), flat_obs[rows])
      np.testing.assert_array_equal(batch["resets"].cpu().numpy(), c["resets"].reshape(-1)[rows])
      ids.append(rows)
      advs.append(batch["advantages"].cpu().numpy())
      sizes.append(len(rows))
    np.testing.assert_array_equal(sizes, c["mb_sizes"])
    np.testing.assert_array_equal(np.concatenate(ids), c["mb_ids"])
    # normalisation: float64 moments on device vs NumPy float32 pairwise -> tolerance
    np.testing.assert_allclose(np.concatenate(advs), c["mb_advantages"], rtol=1e-5, atol=2e-6)


@pytest.mark.parametrize("nmb,shuffle", [(4, True), (3, True), (4, False)])
def test_first_epoch_upload_from_pinned_host_memory(nmb, shuffle, monkeypatch):
  """Observations handed over in pinned host memory become a HostColumn: the first epoch's
  minibatches are pulled over PCIe by the gather kernel (side stream) and mirrored into the
  device-resident copy; later epochs read HBM.  Every minibatch is bit-identical to the
  all-resident pipeline and the resident copy ends up equal to the host array."""
  from derl_b200.runners import host_column
  monkeypatch.setattr(host_column, "MIN_BYTES", 0)
  nsteps, nenvs = 10, 7   # S = 70: ragged tail for nmb = 3 and 4
  rng = np.random.RandomState(8)
  pinned = torch.empty((nsteps, nenvs, 84, 84, 4), dtype=torch.uint8, pin_memory=True)
  pinned.copy_(torch.from_numpy(rng.randint(0, 256, pinned.shape).astype(np.uint8)))
  base = dict(actions=rng.randint(0, 4, (nsteps, nenvs)).astype(np.int64),
              log_prob=rng.standard_normal((nsteps, nenvs)).astype(np.float32),
              values=rng.standard_normal((nsteps, nenvs, 1)).astype(np.float32),
              rewards=rng.standard_normal((nsteps, nenvs)), resets=rng.random((nsteps, nenvs)) < .1)
  last_value = rng.standard_normal((nenvs, 1)).astype(np.float32)

  def batches(observations):
    rollout = dict(observations=observations, **base,
                   state=dict(latest_observations=np.zeros((nenvs, 84, 84, 4), np.uint8)))

    class Source:
      env = type("E", (), {"nenvs": nenvs, "unwrapped": property(lambda s: s)})()
      policy = ConstPolicy(last_value)
      horizon, step_count = 1, 0
      nsteps = 1

      def run(self, obs=None):
        yield dict(rollout)

    inner = d.TransformInteractions(Source(), [d.GAE(Source.policy, normalize=False),
                                               d.MergeTimeBatch()])
    runner = d.IterateWithMinibatches(inner, 3, nmb, shuffle_before_epoch=shuffle)
    np.random.seed(5)
    out = []
    for batch in runner.run():
      out.append({k: v.clone() for k, v in batch.items() if isinstance(v, torch.Tensor)})
    return out

  lazy = batches(pinned.numpy())
  eager = batches(pinned.numpy().copy())   # pageable copy -> ordinary one-shot upload
  assert len(lazy) == len(eager) == 3 * len(range(0, 70, 70 // nmb))
  for a, b in zip(lazy, eager):
    assert a.keys() == b.keys()
    for k in a:
      assert torch.equal(a[k], b[k]), k
  # direct check of the column object
  col = host_column.HostColumn(pinned.reshape(70, 84, 84, 4), DEV)
  perm = cuda(np.random.RandomState(1).permutation(70))
  parts = [col.gather(perm, lo, min(lo + 24, 70) - lo) for lo in range(0, 70, 24)]
  assert col.complete
  torch.cuda.synchronize()
  assert torch.equal(col.resident.cpu(), pinned.reshape(70, 84, 84, 4))
  assert torch.equal(torch.cat(parts).cpu(), pinned.reshape(70, 84, 84, 4)[perm.cpu()])
  # a non-sequential access pattern falls back to one bulk upload
  col2 = host_column.HostColumn(pinned.reshape(70, 84, 84, 4), DEV)
  mid = col2.gather(perm, 30, 10)
  assert col2.complete and torch.equal(mid.cpu(), pinned.reshape(70, 84, 84, 4)[perm.cpu()[30:40]])


def test_iterate_without_shuffle_and_too_many_minibatches():
  rollout = dict(observations=torch.arange(10, device=DEV).reshape(10, 1).float(),
                 advantages=torch.arange(10, device=DEV).float(), state=dict(k=1))

  class Source:
    env, policy, horizon, nsteps, step_count, nenvs = None, None, 10, 10, 0, None

    def run(self, obs=None):
      yield dict(rollout)

  batches = list(d.IterateWithMinibatches(Source(), 2, 3, shuffle_before_epoch=False).run())
  assert [b["observations"].shape[0] for b in batches] == [3, 3, 3, 1] * 2
  assert torch.equal(batches[1]["advantages"], torch.tensor([3., 4., 5.], device=DEV))
  assert batches[0]["state"] == dict(k=1)
  with pytest.raises(ValueError):  # range() step 0, as in the reference
    list(d.IterateWithMinibatches(Source(), 1, 11).run())


# =============================================================================== K3: loss
class HeadPolicy:
  def __init__(self, head, values):
    self.head, self.values = head, values
    self.model = torch.nn.Linear(1, 1).to(DEV)

  def act(self, inputs, state=None, update_state=True, training=False):
    dist = d.policies.CategoricalHead(*self.head) if len(self.head) == 1 \
        else d.policies.DiagNormalHead(*self.head)
    return {"distribution": dist, "values": self.values}


def loss_case_inputs(c):
  head = [cuda(c[f"head{j}"]).requires_grad_() for j in range(2) if f"head{j}" in c]
  values = cuda(c["pred_values"]).requires_grad_()
  batch = {k: c[k] for k in ("actions", "log_prob", "advantages", "value_targets", "values")}
  clip = None if float(c["cliprange"]) < 0 else float(c["cliprange"])
  return head, values, batch, clip


def test_ppo_loss_golden_forward_backward_and_scalars(golden):
  """Reference PPOLoss + torch autograd outputs (tests/golden/live_ppo_loss.npz).
  Tolerance: rtol 1e-5 on the loss (north_star); gradients rtol 1e-5 with an absolute floor
  of 1e-5 * max|grad| for elements that are themselves rounding noise."""
  g = golden("live_ppo_loss.npz")
  for i in range(g.ncases):
    c = g.case(i)
    head, values, batch, clip = loss_case_inputs(c)
    fn = d.PPOLoss(HeadPolicy(head, values), cliprange=clip, value_loss_coef=float(c["vcoef"]),
                   entropy_coef=float(c["ecoef"]))
    loss = fn(batch)
    assert loss.shape == () and loss.is_cuda and fn.call_count == 1
    loss.backward()
    np.testing.assert_allclose(loss.item(), c["loss"], rtol=1e-5, err_msg=f"case {i}")
    dv = values.grad.cpu().numpy()
    np.testing.assert_allclose(dv, c["dvalues"], rtol=1e-5, atol=1e-5 * np.abs(c["dvalues"]).max())
    for j, h in enumerate(head):
      want = c[f"dhead{j}"]
      np.testing.assert_allclose(h.grad.cpu().numpy(), want, rtol=1e-5,
                                 atol=1e-5 * np.abs(want).max(), err_msg=f"case {i} head{j}")
    stats = fn.last_stats.cpu().numpy()
    for key in ("loss", "policy_loss", "entropy", "value_loss", "advantages", "value_targets",
                "value_preds", "r_squared"):
      np.testing.assert_allclose(stats[d.alg.ppo.STAT[key]], c[f"log_ppo_{key}"], rtol=2e-5,
                                 atol=2e-7, err_msg=f"case {i} {key}")
    # the two partial entry points (policy_loss / value_loss)
    head2, values2, _, _ = loss_case_inputs(c)
    fn2 = d.PPOLoss(HeadPolicy(head2, values2), cliprange=clip,
                    value_loss_coef=float(c["vcoef"]), entropy_coef=float(c["ecoef"]))
    np.testing.assert_allclose(fn2.policy_loss(batch).item(), c["policy_loss"], rtol=1e-5,
                               atol=1e-7)
    np.testing.assert_allclose(fn2.value_loss(batch).item(), c["value_loss"], rtol=1e-5)


def test_a2c_loss_golden_forward_backward_and_scalars(golden):
  """A2CLoss on the fused kernels (a2c mode) against the reference's A2CLoss + autograd
  (tests/golden/live_a2c_loss.npz), both heads, incl. the logged scalars."""
  g = golden("live_a2c_loss.npz")
  for i in range(g.ncases):
    c = g.case(i)
    head = [cuda(c[f"head{j}"]).requires_grad_() for j in range(2) if f"head{j}" in c]
    values = cuda(c["pred_values"]).requires_grad_()
    batch = {k: c[k] for k in ("actions", "advantages", "value_targets")}
    fn = d.A2CLoss(HeadPolicy(head, values), value_loss_coef=float(c["vcoef"]),
                   entropy_coef=float(c["ecoef"]))
    assert fn.name == "a2c"
    loss = fn(batch)
    loss.backward()
    np.testing.assert_allclose(loss.item(), c["loss"], rtol=1e-5, err_msg=f"case {i}")
    np.testing.assert_allclose(values.grad.cpu().numpy(), c["dvalues"], rtol=1e-5,
                               atol=1e-5 * np.abs(c["dvalues"]).max())
    for j, h in enumerate(head):
      want = c[f"dhead{j}"]
      np.testing.assert_allclose(h.grad.cpu().numpy(), want, rtol=1e-5,
                                 atol=1e-5 * np.abs(want).max(), err_msg=f"case {i} head{j}")
    stats = fn.last_stats.cpu().numpy()
    for key in ("loss", "policy_loss", "entropy", "value_loss", "advantages", "value_targets",
                "value_preds", "r_squared"):
      np.testing.assert_allclose(stats[d.alg.ppo.STAT[key]], c[f"log_a2c_{key}"], rtol=2e-5,
                                 atol=2e-7, err_msg=f"case {i} {key}")
    head2 = [cuda(c[f"head{j}"]) for j in range(2) if f"head{j}" in c]
    fn2 = d.A2CLoss(HeadPolicy(head2, cuda(c["pred_values"])), value_loss_coef=float(c["vcoef"]),
                    entropy_coef=float(c["ecoef"]))
    np.testing.assert_allclose(fn2.value_loss(batch).item(), c["log_a2c_value_loss"], rtol=1e-5)
    np.testing.assert_allclose(
        fn2.policy_loss(batch).item(),
        c["log_a2c_policy_loss"] - float(c["ecoef"]) * c["log_a2c_entropy"], rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("kind,width", [("categorical", 4), ("categorical", 18),
                                        ("categorical", 130), ("gaussian", 6),
                                        ("gaussian", 40)])
def test_ppo_loss_large_batch_vs_oracle(kind, width):
  """B = 131072 (config-3 minibatch) against the oracle's torch restatement on the CPU and
  its autograd gradients; also checks run-to-run determinism of the two-stage reduction."""
  nb = 131072 if width <= 18 else 20000
  rng = np.random.RandomState(width)
  batch = dict(log_prob=(rng.standard_normal(nb) * .2 - 1.5).astype(np.float32),
               advantages=rng.standard_normal(nb).astype(np.float32),
               value_targets=rng.standard_normal((nb, 1)).astype(np.float32),
               values=rng.standard_normal((nb, 1)).astype(np.float32))
  pred = (batch["values"] + rng.standard_normal((nb, 1)) * .15).astype(np.float32)
  if kind == "categorical":
    head = [rng.standard_normal((nb, width)).astype(np.float32)]
    batch["actions"] = rng.randint(0, width, nb).astype(np.int64)
  else:
    head = [rng.standard_normal((nb, width)).astype(np.float32),
            np.exp(rng.standard_normal((nb, width)) * .2).astype(np.float32)]
    batch["actions"] = (head[0] + .5 * rng.standard_normal((nb, width))).astype(np.float32)
    batch["log_prob"] = (batch["log_prob"] - width).astype(np.float32)
  cpu_head = [torch.tensor(h, requires_grad=True) for h in head]
  cpu_values = torch.tensor(pred, requires_grad=True)
  want = O.ppo_loss(cpu_head, cpu_values, batch, 0.1, 0.25, 0.01)
  want.backward()
  results = []
  for _ in range(2):
    dev_head = [cuda(h).requires_grad_() for h in head]
    dev_values = cuda(pred).requires_grad_()
    fn = d.PPOLoss(HeadPolicy(dev_head, dev_values), cliprange=0.1, value_loss_coef=0.25,
                   entropy_coef=0.01)
    loss = fn(batch)
    loss.backward()
    results.append((loss.item(), [h.grad.clone() for h in dev_head], dev_values.grad.clone()))
  loss_val, dhead, dvalues = results[0]
  np.testing.assert_allclose(loss_val, want.item(), rtol=1e-5)
  for got, ref in zip(dhead + [dvalues], [h.grad for h in cpu_head] + [cpu_values.grad]):
    ref = ref.numpy()
    np.testing.assert_allclose(got.cpu().numpy(), ref, rtol=1e-5, atol=1e-5 * np.abs(ref).max())
  assert results[1][0] == loss_val and torch.equal(results[1][2], dvalues)  # deterministic
  assert all(torch.equal(a, b) for a, b in zip(results[1][1], dhead))


def test_ppo_loss_grad_scales_with_upstream_gradient():
  rng = np.random.RandomState(1)
  nb, width = 512, 5
  logits = cuda(rng.standard_normal((nb, width)).astype(np.float32)).requires_grad_()
  values = cuda(rng.standard_normal((nb, 1)).astype(np.float32)).requires_grad_()
  args = (cuda(rng.randint(0, width, nb)), cuda(rng.standard_normal(nb).astype(np.float32)),
          cuda(rng.standard_normal(nb).astype(np.float32)),
          cuda(rng.standard_normal((nb, 1)).astype(np.float32)),
          cuda(rng.standard_normal((nb, 1)).astype(np.float32)))
  loss, dlogits, dvalues, _ = K.ppo_loss_categorical(logits, values, *args, 0.2, 0.25, 0.01)
  (3.0 * loss).backward()
  assert torch.allclose(logits.grad, 3.0 * dlogits) and torch.allclose(values.grad, 3.0 * dvalues)


def test_ppo_pybullet_fixture_through_the_product_model(golden):
  """testdata/ppo/pybullet through derl_b200.MuJoCoModel + PPOLoss on the GPU: loss0 and all
  13 parameter gradients at the reference's own tolerance (rtol = atol = 1e-5)."""
  g = golden("ref_ppo_pybullet.npz")
  torch.manual_seed(0)
  model = d.MuJoCoModel(26, [6, 1])
  assert next(model.parameters()).is_cuda
  torch.backends.cuda.matmul.allow_tf32 = False
  fn = d.PPOLoss(d.ActorCriticPolicy(model), cliprange=float(g["cliprange"]),
                 value_loss_coef=float(g["value_loss_coef"]),
                 entropy_coef=float(g["entropy_coef"]))
  batch = {k: g[k] for k in ("observations", "actions", "log_prob", "values", "advantages",
                             "value_targets")}
  loss = fn(batch)
  loss.backward()
  np.testing.assert_allclose(loss.item(), g["loss0"], rtol=1e-5, atol=1e-5)
  for j, p in enumerate(model.parameters()):
    np.testing.assert_allclose(p.grad.cpu().numpy(), g[f"grad_{j}"], rtol=1e-5, atol=1e-5,
                               err_msg=f"grad_{j}")


def run_golden_update(g, kind, micro_batch=None, fused_gather=False, graphed_warmup=None):
  """The golden rollouts through the whole drop-in pipeline (GAE -> minibatches -> normalise ->
  fused loss -> backward -> clip -> Adam) with the reference's seeds; returns (losses, model)."""
  torch.manual_seed(0)
  if kind == "mujoco":
    model = d.MuJoCoModel(g["r0_observations"].shape[-1], [g["r0_actions"].shape[-1], 1])
    nenvs = None
  else:
    model = d.NatureCNNModel([4, 1])
    nenvs = int(g["nenvs"])
  policy = d.ActorCriticPolicy(model)
  rollouts = []
  for r in range(int(g["nrollouts"])):
    data = {k: g[f"r{r}_{k}"] for k in ("observations", "actions", "log_prob", "values",
                                         "rewards", "resets")}
    data["state"] = dict(latest_observations=g[f"r{r}_latest_observations"])
    rollouts.append(data)

  class Source:
    env = type("E", (), {"nenvs": nenvs, "unwrapped": property(lambda s: s)})()
    horizon, nsteps, step_count = 1, 1, 0

    def __init__(self):
      self.policy = policy
      self.nenvs = nenvs

    def run(self, obs=None):
      for data in rollouts:
        yield dict(data)

  runner = d.ppo_runner_wrap(Source(), num_epochs=int(g["epochs"]),
                             num_minibatches=int(g["nmb"]))
  if fused_gather:
    runner.runner.fused_gather = True
  if graphed_warmup is None:
    optimizer = torch.optim.Adam(model.parameters(), lr=float(g["lr"]), eps=1e-5)
    trainer = d.Trainer(optimizer, max_grad_norm=.5, micro_batch=micro_batch)
  else:   # CUDA-graph replay of the step after `graphed_warmup` eager steps per minibatch shape
    lr = d.LinearAnneal(float(g["lr"]), 10 ** 12, device=DEV)
    optimizer = torch.optim.Adam(model.parameters(), lr=lr.get_tensor(), eps=1e-5, capturable=True)
    trainer = d.GraphedTrainer(optimizer, anneals=[lr], max_grad_norm=.5, warmup=graphed_warmup,
                               micro_batch=micro_batch)
  run_golden_update.trainer = trainer
  alg = d.PPO(runner, trainer, cliprange=float(g["cliprange"]),
              value_loss_coef=float(g["value_loss_coef"]), entropy_coef=float(g["entropy_coef"]))
  np.random.seed(int(g["seed"]))
  losses = [alg.step(batch).item() for batch in runner.run()]
  return losses, model


@pytest.mark.parametrize("name,kind", [("live_update_mujoco.npz", "mujoco"),
                                       ("live_update_atari.npz", "atari")])
def test_full_ppo_update_matches_reference_losses(golden, name, kind):
  """Two rollouts through the whole drop-in pipeline with the reference's seeds: the sequence
  of losses the reference's own classes produced.  float32 network on both sides (TF32 off);
  tolerance 1e-4 relative: GPU-vs-CPU float32 GEMM/conv rounding compounds over Adam steps."""
  torch.backends.cuda.matmul.allow_tf32 = False
  torch.backends.cudnn.allow_tf32 = False
  try:
    g = golden(name)
    losses, model = run_golden_update(g, kind)
  finally:
    torch.backends.cudnn.allow_tf32 = True
  np.testing.assert_allclose(losses, g["losses"], rtol=1e-4, atol=1e-5)
  final = torch.cat([p.detach().reshape(-1) for p in model.parameters()]).double()
  # a sum over 1.7 M parameters with cancellation: 1e-4 of the sum is ~1e-8 per parameter
  np.testing.assert_allclose(final.sum().item(), float(g["final_param_sum"]), rtol=1e-4)


@pytest.mark.parametrize("name,kind", [("live_update_mujoco.npz", "mujoco"),
                                       ("live_update_atari.npz", "atari")])
def test_graph_replayed_update_matches_reference_losses(golden, name, kind):
  """GraphedTrainer (SURVEY §8f rank 1: forward + fused loss + backward + clip + capturable Adam
  captured once per minibatch shape, then replayed) against the ORACLE, not against the eager
  path: the reference's golden loss sequence and final parameter sum, at the tolerance of the
  eager float32 test.  One eager warm-up step per shape, every later step is a graph replay."""
  torch.backends.cuda.matmul.allow_tf32 = False
  torch.backends.cudnn.allow_tf32 = False
  try:
    g = golden(name)
    losses, model = run_golden_update(g, kind, graphed_warmup=1)
  finally:
    torch.backends.cudnn.allow_tf32 = True
  assert run_golden_update.trainer.replays == len(losses) - 1
  np.testing.assert_allclose(losses, g["losses"], rtol=1e-4, atol=1e-5)
  _check_param_sum(model, g)


def _check_param_sum(model, g, tol=2e-7):
  """|sum(p) - golden| <= tol * sum|p|.  Capturable Adam evaluates its bias corrections in
  float32 on the device (the eager optimizer in Python doubles): ~1e-7 relative per parameter,
  and the golden sum cancels from sum|p| = 25 771 down to -13.4."""
  final = torch.cat([p.detach().reshape(-1) for p in model.parameters()]).double()
  dev = abs(final.sum().item() - float(g["final_param_sum"]))
  assert dev <= tol * float(g["final_param_abs_sum"]), dev


@pytest.mark.parametrize("tf32", [False, True])
def test_graph_replayed_micro_batched_update_with_fused_gather(golden, tf32):
  """The large-configuration step as CUDA graphs: GraphedTrainer(micro_batch=) replays one graph
  per row chunk (ragged: 12-row minibatches in chunks of 5) plus one update graph, and with
  `fused_gather=True` a chunk graph's observation input is the int64 row vector, not frames.
  float32: the reference's golden losses at the eager test's tolerance.  TF32 (the benchmarked
  arithmetic, where the stem kernels gather rows by index inside the graph): the TF32 bounds of
  `test_benchmarked_configuration_tracks_the_fp32_reference_losses`."""
  torch.backends.cuda.matmul.allow_tf32 = tf32
  torch.backends.cudnn.allow_tf32 = tf32
  try:
    g = golden("live_update_atari.npz")
    losses, model = run_golden_update(g, "atari", micro_batch=5, fused_gather=True,
                                      graphed_warmup=1)
  finally:
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = True
  assert run_golden_update.trainer.replays == len(losses) - 1
  rel = np.abs(np.asarray(losses) - g["losses"]) / np.abs(g["losses"])
  if tf32:
    assert rel[0] <= TF32_FIRST_LOSS_RTOL and rel.max() <= TF32_LOSS_RTOL, rel
  else:
    np.testing.assert_allclose(losses, g["losses"], rtol=1e-4, atol=1e-5)
    _check_param_sum(model, g)


# Tolerances of the benchmarked (default `bench.py`) arithmetic against the reference's float32
# losses.  Two different things are bounded:
#  * the FIRST loss is a pure forward pass on identical parameters — it measures the arithmetic
#    itself: TF32 tensor-core conv/GEMM (10-bit mantissa operands, fp32 accumulation) plus the
#    INT8 two-digit stem K6t (operand residual <= 1/508 of a channel's scale).  Measured on B200
#    (profiles/r02_tf32_parity.txt): 9.2e-5 relative (6.2e-5 for the TF32 library path); bound 5e-4.
#  * later losses follow 1..7 Adam steps.  Adam's update lr * m / (sqrt(v) + eps) is sign-like in
#    its first steps, so a 1e-3 relative gradient perturbation (TF32's operand rounding) moves
#    1.7 M parameters by O(lr) in slightly different directions and the 12-sample minibatch
#    losses drift by ~1 % — for cuDNN/cuBLAS TF32 alone (custom_stem off) just as for the
#    default path with K6t/K7t (measured side by side: worst step 1.65e-2 vs 1.75e-2).  Bound
#    3e-2, and the default path must not drift more than 2x what the TF32 library path does.
TF32_FIRST_LOSS_RTOL = 5e-4
TF32_LOSS_RTOL = 3e-2
TF32_PARAM_SUM_TOL = 2e-5   # of sum |p| (25771): the sum itself cancels to -13.4


def _tf32_update(golden, custom_stem, fused_gather):
  g = golden("live_update_atari.npz")
  torch.backends.cuda.matmul.allow_tf32 = True
  torch.backends.cudnn.allow_tf32 = True
  saved = d.NatureCNNBase.custom_stem
  d.NatureCNNBase.custom_stem = custom_stem
  try:
    losses, model = run_golden_update(g, "atari", micro_batch=5, fused_gather=fused_gather)
  finally:
    d.NatureCNNBase.custom_stem = saved
    torch.backends.cuda.matmul.allow_tf32 = False
  rel = np.abs(np.asarray(losses) - g["losses"]) / np.abs(g["losses"])
  final = torch.cat([p.detach().reshape(-1) for p in model.parameters()]).double()
  dsum = abs(final.sum().item() - float(g["final_param_sum"])) / float(g["final_param_abs_sum"])
  return rel, dsum


@pytest.mark.parametrize("fused_gather", [False, True])
def test_benchmarked_configuration_tracks_the_fp32_reference_losses(golden, fused_gather):
  """The configuration bench.py times by default — allow_tf32 on (cuDNN/cuBLAS TF32), the INT8
  stem kernels K6t/K7t on, space-to-depth hidden layers on, micro-batched gradient accumulation
  (ragged chunks: 12-row minibatches in chunks of 5), optionally the fused gather — run on the
  reference's golden rollouts and compared with the losses the reference's float32 CPU classes
  produced (tests/golden/live_update_atari.npz).  This pins the benchmarked arithmetic end to
  end against the oracle with stated tolerances (see the comment above)."""
  assert d.NatureCNNBase.custom_stem and d.NatureCNNBase.space_to_depth_hidden
  launches = _lib.launch_count()
  rel, dsum = _tf32_update(golden, True, fused_gather)
  assert _lib.launch_count() - launches >= 8 * 3 * 2, "K6t/K7t did not run"
  lib_rel, lib_dsum = _tf32_update(golden, False, False)   # cuDNN/cuBLAS TF32 only, no K6t/K7t
  print(f"\n[tf32 parity] default path (fused_gather={fused_gather}): loss rel dev per step "
        f"{np.array2string(rel, precision=2)}, param-sum dev {dsum:.2e} of sum|p|\n"
        f"[tf32 parity] TF32 library path (no K6t/K7t):    loss rel dev per step "
        f"{np.array2string(lib_rel, precision=2)}, param-sum dev {lib_dsum:.2e} of sum|p|")
  assert rel[0] <= TF32_FIRST_LOSS_RTOL, rel
  assert rel.max() <= TF32_LOSS_RTOL, rel
  assert rel.max() <= 2.0 * max(lib_rel.max(), 5e-3), (rel, lib_rel)
  assert dsum <= TF32_PARAM_SUM_TOL, dsum


def test_stem_kernels_run_in_the_default_configuration():
  """Guard for the test above: with allow_tf32 the model routes its first layer through K6t
  (forward) and K7t (backward), and with TF32 off it does not."""
  from derl_b200 import ops
  frames = torch.randint(0, 256, (6, 84, 84, 4), dtype=torch.uint8, device=DEV)
  torch.manual_seed(0)
  model = d.NatureCNNModel([4, 1])
  for tf32, expect in ((True, True), (False, False)):
    torch.backends.cudnn.allow_tf32 = tf32
    ops.PROFILE = []
    try:
      logits, values = model(frames)
      (logits.sum() + values.sum()).backward()
      names = {n for n, _, _ in ops.PROFILE}
    finally:
      ops.PROFILE = None
      torch.backends.cudnn.allow_tf32 = True
    assert ("stem_conv_relu" in names) == expect and ("stem_backward" in names) == expect, names


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
def test_frames_to_s2d_kernel_bit_exact(dtype):
  """K4: uint8 NHWC -> space-to-depth, /255 (IEEE float32 division), cast — against the same
  expression evaluated by NumPy / torch on the host, bit for bit."""
  rng = np.random.RandomState(4)
  for batch, height, width in ((3, 84, 84), (1, 4, 4), (257, 8, 12)):
    frames = rng.randint(0, 256, (batch, height, width, 4)).astype(np.uint8)
    out = K.frames_to_s2d(cuda(frames), 4, dtype, 255.0)
    blocks = frames.reshape(batch, height // 4, 4, width // 4, 4, 4).transpose(0, 1, 3, 2, 4, 5)
    want = torch.from_numpy(blocks.reshape(batch, height // 4, width // 4, 64).astype(np.float32)
                            / np.float32(255)).to(dtype)
    assert out.shape == want.shape and out.dtype == dtype
    assert torch.equal(out.cpu(), want)
  raw = K.frames_to_s2d(cuda(frames), 4, torch.float32, 1.0)
  assert torch.equal(raw.cpu(), torch.from_numpy(
      blocks.reshape(batch, height // 4, width // 4, 64).astype(np.float32)))
  with pytest.raises(ValueError, match="block\\*C == 16"):
    K.frames_to_s2d(cuda(frames), 2, torch.float32, 255.0)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
def test_relu_backward_bias_kernel_vs_aten(dtype):
  """K5: masked gradient bit-identical to ATen's threshold_backward; bias gradient equal to
  the float64 column sums to float32 accuracy; deterministic across launches."""
  gen = torch.Generator(device=DEV).manual_seed(6)
  for shape in ((37, 32, 20, 20), (5, 64, 9, 9), (3, 64, 7, 7), (1, 4, 1, 1), (300, 128, 3, 5)):
    out = torch.relu(torch.randn(shape, device=DEV, generator=gen)).to(dtype).contiguous(
        memory_format=torch.channels_last)
    grad = torch.randn(shape, device=DEV, generator=gen).to(dtype).contiguous(
        memory_format=torch.channels_last)
    grad_pre, bias = K.relu_bwd_bias(grad, out)
    want = torch.ops.aten.threshold_backward(grad, out, 0)
    assert torch.equal(grad_pre, want) and grad_pre.stride() == out.stride()
    want_bias = want.double().sum((0, 2, 3))
    assert torch.allclose(bias.double(), want_bias, rtol=1e-5, atol=1e-4)
    again = K.relu_bwd_bias(grad, out)[1]
    assert torch.equal(again, bias)
  with pytest.raises(ValueError, match="channels_last"):
    K.relu_bwd_bias(torch.zeros(2, 8, 3, 3, device=DEV), torch.zeros(2, 8, 3, 3, device=DEV))
  # unblock: inputs in space-to-depth(2) arrangement, masked gradient back in the plain layout
  plain_out = torch.relu(torch.randn(9, 20, 20, 32, device=DEV, generator=gen)).to(dtype)
  plain_grad = torch.randn(9, 20, 20, 32, device=DEV, generator=gen).to(dtype)
  s2d = lambda x: K.space_to_depth(x, 2, False).permute(0, 3, 1, 2)
  grad_pre, bias = K.relu_bwd_bias(s2d(plain_grad), s2d(plain_out), 2)
  want = torch.ops.aten.threshold_backward(plain_grad, plain_out, 0)
  assert grad_pre.shape == (9, 32, 20, 20)
  assert torch.equal(grad_pre.permute(0, 2, 3, 1), want)
  assert torch.allclose(bias.view(4, 32).sum(0).double(), want.double().sum((0, 1, 2)),
                        rtol=1e-5, atol=1e-3)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_space_to_depth_kernel_and_its_inverse(dtype):
  gen = torch.Generator(device=DEV).manual_seed(3)
  for shape, block in (((5, 20, 20, 32), 2), ((3, 8, 12, 8), 4), ((2, 6, 6, 64), 3)):
    x = torch.randn(shape, device=DEV, generator=gen).to(dtype).requires_grad_()
    batch, height, width, chans = shape
    want = x.detach().reshape(batch, height // block, block, width // block, block, chans) \
        .permute(0, 1, 3, 2, 4, 5).reshape(batch, height // block, width // block, -1)
    got = K.space_to_depth(x, block, False)
    assert torch.equal(got, want)
    assert torch.equal(K.space_to_depth(got.detach(), block, True), x.detach())
    grad = torch.randn_like(got)
    got.backward(grad)
    assert torch.equal(x.grad, K.space_to_depth(grad, block, True))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_stem_conv_kernel_vs_float32_convolution(dtype):
  """K6t: conv 8x8/4 + bias + ReLU straight from uint8 frames (INT8 MMA, weights as two signed
  8-bit digit planes) against the reference formulation in float32 (`.float()/255` -> conv2d ->
  relu, TF32 off).  The digits keep each weight to 1.6e-5 of its channel's largest: 1e-4 relative
  on activations of O(1) (bf16 output: bf16 rounding)."""
  torch.backends.cudnn.allow_tf32 = False
  gen = torch.Generator(device=DEV).manual_seed(12)
  weight = torch.randn(32, 4, 8, 8, device=DEV, generator=gen) * 0.1
  bias = torch.randn(32, device=DEV, generator=gen) * 0.1
  for batch in (1, 2, 3, 301):
    frames = torch.randint(0, 256, (batch, 84, 84, 4), device=DEV, dtype=torch.uint8, generator=gen)
    out = K.stem_conv_relu(frames, weight, bias, dtype, 1)
    want = torch.relu(torch.nn.functional.conv2d(frames.permute(0, 3, 1, 2).float() / 255, weight,
                                                 bias, stride=4)).permute(0, 2, 3, 1)
    assert out.shape == (batch, 20, 20, 32) and out.dtype == dtype
    blocked = K.stem_conv_relu(frames, weight, bias, dtype, 2)   # same values, s2d(2) layout
    assert torch.equal(blocked, K.space_to_depth(out, 2, False))
    tol = 1e-4 if dtype == torch.float32 else 1e-2
    assert torch.allclose(out.float(), want, rtol=tol, atol=tol * float(want.abs().max())), \
        (out.float() - want).abs().max()
    assert (out.float() - want).abs().max() <= tol * want.abs().max()
  torch.backends.cudnn.allow_tf32 = True


def test_stem_forward_kernels_with_fused_row_gather_are_bit_identical():
  """K6t with `rows`: frame i of the batch is source[rows[i]], pulled straight out of the
  resident rollout (SURVEY §8f rank 2).  Same bytes in, deterministic kernels: bit-identical to
  running them on the materialised gather, for both output layouts, with repeated rows (the
  backward's `rows` is checked by test_stem_tcgen05_pair_against_its_number_format)."""
  gen = torch.Generator(device=DEV).manual_seed(33)
  weight = torch.randn(32, 4, 8, 8, device=DEV, generator=gen) * 0.05
  bias = torch.randn(32, device=DEV, generator=gen) * 0.1
  source = torch.randint(0, 256, (97, 84, 84, 4), device=DEV, dtype=torch.uint8, generator=gen)
  for count in (1, 5, 300):   # 300 > 97: rows repeat; > 148 CTAs (one per SM): second frames per CTA
    rows = torch.randint(0, 97, (count,), device=DEV, generator=gen)
    dense = source[rows]
    for blk in (1, 2):
      for dtype in (torch.float32, torch.bfloat16):
        assert torch.equal(K.stem_conv_relu(source, weight, bias, dtype, blk, rows),
                           K.stem_conv_relu(dense, weight, bias, dtype, blk))
  with pytest.raises(ValueError, match="rows"):
    K.stem_conv_relu(source, weight, bias, torch.float32, 1, rows.int())


def test_fused_gather_minibatches_and_update_match_the_materialised_pipeline():
  """IterateWithMinibatches(fused_gather=True) hands `observations` on as a RowSelection; the
  NatureCNN stem reads the rollout rows in place.  Minibatch contents (materialised on demand),
  loss and every parameter gradient equal the materialised pipeline's; Trainer's micro-batch
  row slicing stays lazy; paths without the fused stem fall back to the materialised tensor."""
  from derl_b200.runners.row_selection import RowSelection
  nsteps, nenvs, nact = 12, 6, 4
  torch.manual_seed(1)
  policy = d.ActorCriticPolicy(d.NatureCNNModel([nact, 1]))
  torch.backends.cudnn.deterministic = True
  make_source = lambda: d.SyntheticRolloutRunner(policy, "atari", nenvs=nenvs, horizon=nsteps,
                                                 seed=3, nactions=nact)
  rollout = make_source().rollout()

  def run(fused):
    runner = d.ppo_runner_wrap(make_source(), num_epochs=2, num_minibatches=3, fused_gather=fused)
    np.random.seed(7)
    loss_fn = d.PPOLoss(policy, cliprange=0.1)
    out = []
    it = runner.run()
    for _ in range(6):
      batch = next(it)
      policy.model.zero_grad()
      loss = loss_fn(batch)
      loss.backward()
      out.append((batch, loss.detach().clone(), [p.grad.clone() for p in policy.model.parameters()]))
    return out

  eager, fused = run(False), run(True)
  for (be, le, ge), (bf, lf, gf) in zip(eager, fused):
    assert isinstance(bf["observations"], RowSelection) and isinstance(be["observations"], torch.Tensor)
    assert bf["observations"].shape == be["observations"].shape
    assert torch.equal(bf["observations"].materialize(), be["observations"])
    assert torch.equal(bf["observations"][3:20].materialize(), be["observations"][3:20])
    assert torch.equal(bf["observations"][5], be["observations"][5])
    for key in be:
      if key not in ("observations", "state"):
        assert torch.equal(bf[key], be[key]), key
    assert torch.equal(lf, le)
    for a, b in zip(gf, ge):
      assert torch.equal(a, b)
  # micro-batched Trainer: row chunks of a RowSelection are RowSelections; same update
  params0 = [p.detach().clone() for p in policy.model.parameters()]
  finals = []
  for fused_flag in (False, True):
    with torch.no_grad():
      for p, p0 in zip(policy.model.parameters(), params0):
        p.copy_(p0)
    runner = d.ppo_runner_wrap(make_source(), num_epochs=1, num_minibatches=2,
                               fused_gather=fused_flag)
    np.random.seed(9)
    optimizer = torch.optim.SGD(policy.model.parameters(), lr=1e-3)
    alg = d.PPO(runner, d.Trainer(optimizer, max_grad_norm=0.5, micro_batch=16), cliprange=0.1)
    it = runner.run()
    losses = [alg.step(next(it)) for _ in range(2)]
    finals.append((torch.stack(losses), [p.detach().clone() for p in policy.model.parameters()]))
  assert torch.equal(finals[0][0], finals[1][0])
  for a, b in zip(finals[0][1], finals[1][1]):
    assert torch.equal(a, b)
  # strict-fp32 network (no K6t/K7t): the selection is materialised for the library stem
  torch.backends.cudnn.allow_tf32 = False
  sel = RowSelection(rollout["observations"].reshape(-1, 84, 84, 4),
                     torch.randperm(nsteps * nenvs, device=DEV), 10, 17)
  with torch.no_grad():
    a = policy.model(sel)
    b = policy.model(sel.materialize())
  torch.backends.cudnn.allow_tf32 = True
  torch.backends.cudnn.deterministic = False
  assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
  with pytest.raises(ValueError):
    RowSelection(sel.source, sel.perm, 70, 5)


def test_stem_autograd_matches_cudnn_path():
  """NatureCNN with the K6t stem (TF32 allowed) vs the cuDNN stem: outputs and all parameter
  gradients agree to TF32-level tolerance; the stem weight gradient lands in [32,4,8,8] layout."""
  torch.manual_seed(0)
  model = d.NatureCNNModel([4, 1])
  frames = torch.randint(0, 256, (64, 84, 84, 4), dtype=torch.uint8, device=DEV)
  res = {}
  for custom, hidden in ((True, True), (True, False), (False, True)):
    d.NatureCNNBase.custom_stem, d.NatureCNNBase.space_to_depth_hidden = custom, hidden
    model.zero_grad()
    logits, values = model(frames)
    (logits.square().sum() + values.sum()).backward()
    res[custom, hidden] = (logits.detach().clone(), [p.grad.clone() for p in model.parameters()])
  d.NatureCNNBase.custom_stem = d.NatureCNNBase.space_to_depth_hidden = True
  base = res[False, True]
  for key in ((True, True), (True, False)):
    assert torch.allclose(res[key][0], base[0], rtol=2e-2, atol=2e-3), key
    for a, b in zip(res[key][1], base[1]):
      assert a.shape == b.shape
      assert (a - b).abs().max() <= 2e-2 * b.abs().max() + 1e-6, key


def test_space_to_depth_first_conv_equals_plain_formulation():
  """NatureCNNBase runs the 8x8/4 stem as a 2x2/1 conv on the space-to-depth tensor with
  re-indexed weights (derl_b200/models.py): same parameters, same function as the
  reference's NCHW float/255 pipeline (derl/models.py:117-124) — outputs and parameter
  gradients agree to float32 rounding (TF32 off)."""
  torch.backends.cudnn.allow_tf32 = False
  torch.backends.cuda.matmul.allow_tf32 = False
  torch.manual_seed(0)
  model = d.NatureCNNModel([6, 1])
  frames = torch.randint(0, 256, (37, 84, 84, 4), dtype=torch.uint8, device=DEV)
  outs = {}
  for s2d, fused in ((True, True), (True, False), (False, False), ("hidden", True)):
    d.NatureCNNBase.space_to_depth, d.NatureCNNBase.fused_conv_relu = bool(s2d), fused
    d.NatureCNNBase.space_to_depth_hidden = s2d == "hidden"
    model.zero_grad()  # (TF32 is off here, so the K6t stem is not in play: cuDNN float32 stem)
    logits, values = model(frames)
    (logits.square().sum() + values.sum()).backward()
    outs[s2d, fused] = (logits.detach().clone(), values.detach().clone(),
                        [p.grad.clone() for p in model.parameters()])
  d.NatureCNNBase.space_to_depth = d.NatureCNNBase.fused_conv_relu = True
  d.NatureCNNBase.space_to_depth_hidden = True
  torch.backends.cudnn.allow_tf32 = True
  plain = outs[False, False]
  for key in ((True, True), (True, False), ("hidden", True)):
    for a, b in zip(outs[key][:2], plain[:2]):
      assert torch.allclose(a, b, rtol=1e-5, atol=1e-6), key
    for a, b in zip(outs[key][2], plain[2]):
      assert torch.allclose(a, b, rtol=1e-4, atol=1e-5 * float(b.abs().max())), key
  outs = {True: outs[True, True]}
  # and the CPU path (reference formulation) agrees with the GPU one
  cpu = d.NatureCNNModel([6, 1]).to("cpu")
  cpu.load_state_dict(model.state_dict())
  want = cpu(frames.cpu())[0]
  assert torch.allclose(outs[True][0].cpu(), want, rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize("kind", ["mujoco", "atari"])
def test_graphed_trainer_matches_eager_trainer(kind):
  """GraphedTrainer (CUDA-graph replay of forward + fused loss + backward + clip + Adam) walks
  the same parameter trajectory as the eager Trainer on the same minibatch stream."""
  torch.backends.cudnn.allow_tf32 = False
  torch.backends.cuda.matmul.allow_tf32 = False
  # Adam turns rounding-level gradient noise into O(lr) parameter differences wherever a
  # gradient is ~0, so the two runs must use the same (deterministic) cuDNN algorithms
  torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
  results = {}
  for graphed in (False, True):
    torch.manual_seed(0)
    model = d.MuJoCoModel(17, [6, 1]) if kind == "mujoco" else d.NatureCNNModel([4, 1])
    policy = d.ActorCriticPolicy(model)
    nenvs, horizon = (None, 256) if kind == "mujoco" else (4, 32)
    source = d.SyntheticRolloutRunner(policy, kind, nenvs, horizon, nsteps=None, device=DEV, seed=2)
    runner = d.ppo_runner_wrap(source, num_epochs=2, num_minibatches=4)
    if graphed:
      lr = d.LinearAnneal(2.5e-4, 10 ** 6, device=DEV)
      opt = torch.optim.Adam(model.parameters(), lr=lr.get_tensor(), eps=1e-5, capturable=True)
      trainer = d.GraphedTrainer(opt, anneals=[lr], max_grad_norm=.5, warmup=2)
    else:
      lr = d.LinearAnneal(2.5e-4, 10 ** 6)
      opt = torch.optim.Adam(model.parameters(), lr=lr.get_tensor(), eps=1e-5)
      trainer = d.Trainer(opt, anneals=[lr], max_grad_norm=.5)
    alg = d.PPO(runner, trainer, cliprange=.2)
    np.random.seed(4)
    it = runner.run()
    losses = [alg.step(next(it)).item() for _ in range(20)]
    results[graphed] = (losses, torch.cat([p.detach().reshape(-1) for p in model.parameters()]),
                        alg.loss_fn.call_count, trainer.step_count)
    if graphed:
      assert trainer.replays == 18
  torch.backends.cudnn.allow_tf32 = True
  torch.backends.cudnn.deterministic = False
  np.testing.assert_allclose(results[True][0], results[False][0], rtol=2e-3, atol=1e-5)
  assert torch.allclose(results[True][1], results[False][1], rtol=1e-2, atol=3e-4)
  assert results[True][2:] == results[False][2:] == (20, 20)


# =============================================================================== plumbing
def test_ops_are_cuda_graph_capturable():
  """GAE + gather + loss captured once and replayed on new data in the same buffers."""
  rng = np.random.RandomState(2)
  nsteps, nenvs, nact = 32, 64, 4
  size = nsteps * nenvs
  rewards = cuda(rng.standard_normal((nsteps, nenvs)).astype(np.float32))
  values = cuda(rng.standard_normal((nsteps, nenvs)).astype(np.float32))
  resets = cuda(rng.random((nsteps, nenvs)) < .1)
  last_value = cuda(rng.standard_normal(nenvs).astype(np.float32))
  logits = cuda(rng.standard_normal((size, nact)).astype(np.float32))
  actions = cuda(rng.randint(0, nact, size))
  old_lp = cuda((rng.standard_normal(size) * .1 - 1.4).astype(np.float32))
  perm = cuda(rng.permutation(size))

  def step():
    adv, vt, _ = K.gae(rewards, values, resets, last_value, 0.99, 0.95, False, 0)
    *cols, moments = K.gather_columns([adv.reshape(-1), vt.reshape(-1), values.reshape(-1),
                                       old_lp, actions], perm, 0, size, 0)
    nadv = K.normalize(cols[0], moments, 1e-8)
    lg = K.gather_rows(logits, perm, 0, size)
    return K.ppo_loss_categorical(lg, cols[2].clone(), cols[4], cols[3], nadv, cols[1], cols[2],
                                  0.1, 0.25, 0.01)

  stream = torch.cuda.Stream()
  stream.wait_stream(torch.cuda.current_stream())
  with torch.cuda.stream(stream):
    for _ in range(2):
      eager = step()
  torch.cuda.current_stream().wait_stream(stream)
  graph = torch.cuda.CUDAGraph()
  with torch.cuda.graph(graph):
    captured = step()
  graph.replay()
  torch.cuda.synchronize()
  assert captured[0].item() == eager[0].item() and torch.equal(captured[1], eager[1])
  rewards.add_(1.0)  # new data, same buffers
  want = step()
  graph.replay()
  torch.cuda.synchronize()
  assert captured[0].item() == want[0].item() and torch.equal(captured[1], want[1])


def test_plain_c_caller_of_the_abi(tmp_path):
  """gcc-compiled tests/abi_smoke.c (no Python in the loop) gets bit-identical GAE."""
  import test_abi
  test_abi.test_plain_c_caller_links_and_runs(tmp_path)


def test_launch_counter_counts_our_kernels():
  before = _lib.launch_count()
  K.moments(torch.ones(100, device=DEV))
  assert _lib.launch_count() == before + 1


# =============================================================================== Take / EnvRunner
@pytest.mark.parametrize("axis,indices", [(0, [3, 0, 0, -1]), (0, 2), (1, [1, -2]),
                                          (0, [[0, 1], [4, -5]]), (1, 0)])
def test_take_on_device_tensors_matches_np_take(axis, indices):
  """derl/runners/trajectory_transforms.py:95-103 on CUDA tensors: axis 0 goes through the
  gather_rows kernel (28 224-byte rows take the TMA path), other axes through index_select; a
  HostColumn (pinned host column of the e2e path) is uploaded first.  Bit-exact vs np.take."""
  from derl_b200.runners.host_column import HostColumn
  rng = np.random.RandomState(2)
  obs = rng.randint(0, 256, (5, 3, 84, 84, 4)).astype(np.uint8)
  adv = rng.standard_normal((5, 3)).astype(np.float32)
  state = dict(latest_observations=obs[0])
  traj = dict(observations=cuda(obs), advantages=cuda(adv), state=state)
  d.Take(indices, axis=axis)(traj)
  for key, src in (("observations", obs), ("advantages", adv)):
    want = np.take(src, indices, axis=axis)
    assert traj[key].is_cuda and tuple(traj[key].shape) == want.shape
    assert np.array_equal(traj[key].cpu().numpy(), want), key
  assert traj["state"] is state
  pinned = torch.from_numpy(obs.reshape(15, 84, 84, 4)).pin_memory()
  column = HostColumn(pinned, torch.device(DEV))
  traj = dict(observations=column)
  if axis == 0:
    d.Take(indices, axis=0)(traj)
    assert np.array_equal(traj["observations"].cpu().numpy(),
                          np.take(obs.reshape(15, 84, 84, 4), indices, axis=0))


def test_take_out_of_range_raises_before_any_launch():
  x = torch.zeros(4, 3, 28224, dtype=torch.uint8, device=DEV)
  before = _lib.launch_count()
  for bad, axis in (([0, 4], 0), ([-5], 0), (3, 1)):
    with pytest.raises(IndexError, match="out of bounds"):
      d.Take(bad, axis=axis)(dict(observations=x))
  assert _lib.launch_count() == before


def test_env_runner_resident_on_cuda_feeds_gae_without_a_second_forward():
  """SURVEY §8f rank 3: EnvRunner(resident_device="cuda") writes each step through pinned
  staging rows into preallocated device tensors (equal to the reference-style stacked lists),
  and hands GAE the critic's value of the final observation from its own forward pass on it
  (`state["latest_values"]`, on the device): GAE's result is bit-identical to the oracle's on the
  stacked host arrays, and the policy is not called again."""
  class Env:
    nenvs = 4
    unwrapped = property(lambda self: self)

    def __init__(self):
      self.t = 0
      self.rng = np.random.RandomState(5)

    def _obs(self):
      return self.rng.randint(0, 256, (4, 84, 84, 4)).astype(np.uint8)

    def reset(self):
      self.t = 0
      return self._obs()

    def step(self, actions):
      self.t += 1
      return (self._obs(), self.rng.standard_normal(4), self.rng.rand(4) < 0.2, [{}] * 4)

  class CountingPolicy(d.ActorCriticPolicy):
    calls = 0

    def act(self, inputs, state=None, update_state=True, training=False):
      CountingPolicy.calls += 1
      return super().act(inputs, state, update_state, training)

  torch.manual_seed(0)
  torch.backends.cudnn.allow_tf32 = False
  try:
    policy = CountingPolicy(d.NatureCNNModel([4, 1]))
    runner = d.EnvRunner(Env(), policy, horizon=6, nsteps=48, resident_device=DEV)
    gen = runner.run()
    rollouts = [next(gen), next(gen)]
    assert runner.is_exhausted()
    for rollout in rollouts:
      for key in ("observations", "actions", "log_prob", "values", "rewards", "resets"):
        assert rollout[key].is_cuda and rollout[key].shape[:2] == (6, 4), key
      assert rollout["observations"].dtype == torch.uint8
      assert rollout["rewards"].dtype == torch.float64 and rollout["resets"].dtype == torch.bool
      assert rollout["state"]["latest_values"].is_cuda
    # the two rollouts own different device tensors (the first is not overwritten by the second)
    assert rollouts[0]["observations"].data_ptr() != rollouts[1]["observations"].data_ptr()
    assert not torch.equal(rollouts[0]["observations"], rollouts[1]["observations"])
    # replay the env: the resident tensors hold exactly what the per-step lists would
    env = Env()
    first = env.reset()
    assert np.array_equal(rollouts[0]["observations"][0].cpu().numpy(), first)
    calls = CountingPolicy.calls
    rollout = rollouts[1]
    host = {k: rollout[k].cpu().numpy() for k in ("rewards", "values", "resets")}
    last_value = rollout["state"]["latest_values"].cpu().numpy()
    adv, targets = d.GAE(policy, normalize=False)(rollout)
    assert CountingPolicy.calls == calls, "GAE ran a second forward for the bootstrap value"
    want_adv, want_targets = O.gae(host["rewards"], host["values"], host["resets"], last_value,
                                   normalize=False)
    assert np.array_equal(adv.cpu().numpy(), want_adv)
    assert np.array_equal(targets.cpu().numpy(), want_targets)
  finally:
    torch.backends.cudnn.allow_tf32 = True


# =============================================================================== K8: fused MLP update
class _ArraySource:
  """EnvRunner-shaped source over prepared rollouts (unbatched env: nenvs None)."""

  def __init__(self, rollouts, policy, horizon):
    self.rollouts, self.policy, self.horizon = rollouts, policy, horizon
    self.env = type("E", (), {"nenvs": None, "unwrapped": property(lambda s: s)})()
    self.nenvs, self.step_count = None, 0
    self.nsteps = horizon * len(rollouts)

  def is_exhausted(self):
    return self.step_count >= self.nsteps

  def __len__(self):
    return self.nsteps

  def run(self, obs=None):
    for data in self.rollouts:
      self.step_count += self.horizon
      yield {k: (dict(v) if k == "state" else v) for k, v in data.items()}


def _mujoco_alg(rollouts, obs_dim, act_dim, epochs, nmb, lr=3e-4, hp=None, max_grad_norm=.5):
  torch.manual_seed(0)
  model = d.MuJoCoModel(obs_dim, [act_dim, 1])
  policy = d.ActorCriticPolicy(model)
  horizon = rollouts[0]["rewards"].shape[0]
  runner = d.ppo_runner_wrap(_ArraySource(rollouts, policy, horizon), num_epochs=epochs,
                             num_minibatches=nmb)
  optimizer = torch.optim.Adam(model.parameters(), lr=lr, eps=1e-5)
  alg = d.PPO(runner, d.Trainer(optimizer, max_grad_norm=max_grad_norm),
              **(hp or dict(cliprange=.2, value_loss_coef=.25, entropy_coef=0.)))
  return alg, model, optimizer


def test_fused_mlp_update_matches_the_reference_golden_update(golden):
  """K8 (one launch per rollout: gather, normalise, forward, PPO loss, backward, clip, Adam for
  every epoch x minibatch) through `PPO.learn()` on the reference's golden MuJoCo-shaped
  rollouts: the 16 losses the reference's classes produced and its final parameters, at the
  tolerance of the per-minibatch GPU path (rtol 1e-4: float32 summation order differs from the
  CPU's, and the difference compounds over Adam steps)."""
  from derl_b200.alg.fused_mlp import FusedMLPUpdate
  g = golden("live_update_mujoco.npz")
  rollouts = []
  for r in range(int(g["nrollouts"])):
    data = {k: g[f"r{r}_{k}"] for k in ("observations", "actions", "log_prob", "values",
                                         "rewards", "resets")}
    data["state"] = dict(latest_observations=g[f"r{r}_latest_observations"])
    rollouts.append(data)
  alg, model, optimizer = _mujoco_alg(rollouts, g["r0_observations"].shape[-1],
                                      g["r0_actions"].shape[-1], int(g["epochs"]), int(g["nmb"]),
                                      lr=float(g["lr"]),
                                      hp=dict(cliprange=float(g["cliprange"]),
                                              value_loss_coef=float(g["value_loss_coef"]),
                                              entropy_coef=float(g["entropy_coef"])))
  assert FusedMLPUpdate.plan(alg) is not None, "the stock MuJoCo pipeline must take the fused path"
  np.random.seed(int(g["seed"]))
  launches = _lib.launch_count()
  losses = []
  source = alg.runner.unwrapped
  for r in range(len(rollouts)):   # learn() one rollout at a time to collect every loss
    source.nsteps = source.horizon * (r + 1)
    source.rollouts = rollouts[r:r + 1]
    alg.learn(progress=False)
    losses += alg.last_losses.cpu().tolist()
  per_update = int(g["epochs"]) * int(g["nmb"])
  assert len(losses) == per_update * len(rollouts)
  # per rollout: GAE + the one update kernel (the bootstrap forward is library code)
  assert _lib.launch_count() - launches == 2 * len(rollouts)
  np.testing.assert_allclose(losses, g["losses"], rtol=1e-4, atol=1e-5)
  state = model.state_dict()
  for key, val in state.items():
    np.testing.assert_allclose(val.cpu().numpy(), g["final_" + key], rtol=1e-4, atol=1e-6,
                               err_msg=key)
  assert alg.trainer.step_count == len(losses) and alg.loss_fn.call_count == len(losses)
  steps = {float(s["step"]) for s in optimizer.state.values()}
  assert steps == {float(len(losses))}
  assert all(p.grad is None for p in model.parameters())


@pytest.mark.parametrize("size,nmb,epochs,obs_dim,act_dim,obs_dtype,hp,clip_norm", [
    (384, 4, 2, 17, 6, np.float64, None, .5),    # 96-row minibatches: a full and a partial 64-row pass
    (100, 3, 2, 11, 3, np.float32, None, .5),    # ragged: 33, 33, 33, 1
    (2048, 32, 2, 26, 8, np.float64, None, .5),  # BASELINE configs[1] minibatch shape, pybullet-sized obs
    # no clipping anywhere (cliprange=None drops both clips, alg/ppo.py:47,83; no clip_grad_norm_)
    # and an entropy bonus
    (256, 4, 2, 17, 6, np.float64, dict(cliprange=None, value_loss_coef=.5, entropy_coef=.01), None),
])
def test_fused_mlp_update_equals_the_per_minibatch_path(size, nmb, epochs, obs_dim, act_dim,
                                                        obs_dtype, hp, clip_norm):
  """Same seeds, same rollout: `PPO.learn()` on the fused kernel vs minibatch-by-minibatch
  `alg.step` (gather kernels + library MLP + K3 + torch clip/Adam).  The two are float32
  evaluations of the same formulas in different summation orders: the first loss (identical
  parameters) agrees to 1e-5, later losses and the final parameters to what a few Adam steps
  of that noise give (1e-3 of the loss; 2e-5 absolute on parameters of O(0.1-1))."""
  rng = np.random.RandomState(size)
  rollout = dict(observations=rng.standard_normal((size, obs_dim)).astype(obs_dtype),
                 actions=rng.standard_normal((size, act_dim)).astype(np.float32),
                 log_prob=(rng.standard_normal(size) * .1 - 1.4 * act_dim).astype(np.float32),
                 values=(rng.standard_normal((size, 1)) * .1).astype(np.float32),
                 rewards=rng.standard_normal(size), resets=rng.rand(size) < .01,
                 state=dict(latest_observations=rng.standard_normal(obs_dim).astype(obs_dtype)))
  results = []
  for fused in (True, False):
    alg, model, _ = _mujoco_alg([rollout], obs_dim, act_dim, epochs, nmb, hp=hp,
                                max_grad_norm=clip_norm)
    np.random.seed(3)
    if fused:
      alg.learn(progress=False)
      losses = alg.last_losses.cpu().numpy()
    else:
      losses = np.asarray([alg.step(batch).item() for batch in alg.runner.run()])
    results.append((losses, [p.detach().cpu().numpy() for p in model.parameters()]))
  (fl, fp), (el, ep) = results
  assert fl.shape == el.shape
  np.testing.assert_allclose(fl[0], el[0], rtol=1e-5)
  np.testing.assert_allclose(fl, el, rtol=1e-3, atol=1e-5)
  for a, b in zip(fp, ep):
    np.testing.assert_allclose(a, b, rtol=0, atol=2e-5)


def test_fused_mlp_plan_rejects_what_it_does_not_model():
  """Anything but the stock pipeline falls back to the per-minibatch path."""
  from derl_b200.alg.fused_mlp import FusedMLPUpdate
  rng = np.random.RandomState(0)
  rollout = dict(observations=rng.standard_normal((64, 5)), rewards=rng.standard_normal(64))
  alg, model, opt = _mujoco_alg([rollout], 5, 2, 2, 4)
  assert FusedMLPUpdate.plan(alg) is not None
  alg.trainer.micro_batch = 16
  assert FusedMLPUpdate.plan(alg) is None
  alg.trainer.micro_batch = None
  opt.param_groups[0]["weight_decay"] = 0.1
  assert FusedMLPUpdate.plan(alg) is None
  opt.param_groups[0]["weight_decay"] = 0
  alg.runner.runner.fused_gather = True
  assert FusedMLPUpdate.plan(alg) is None
  alg.runner.runner.fused_gather = False
  wide = d.MuJoCoModel(5, [2, 1], mlp=lambda i, o: d.MLP(i, o, hidden_features=(32, 32)))
  alg.model = wide
  assert FusedMLPUpdate.plan(alg) is None
  assert _lib.load().derl_b200_ppo_mlp_update_smem_bytes(376, 17) == 0   # Humanoid: too wide
  assert _lib.load().derl_b200_ppo_mlp_update_smem_bytes(17, 6) > 0


# =============================================================================== K6t: tcgen05 stem
@pytest.mark.parametrize("batch", [1, 3, 149, 700])
@pytest.mark.parametrize("out_block", [1, 2])
def test_stem_forward_kernel_against_its_number_format(batch, out_block):
  """K6t (csrc/stem_tc.cu: tcgen05.mma kind::i8, accumulators in tensor memory, TMA-permuted
  frame tile as a no-swizzle K-major operand) computes exact int32 digit sums and a separately
  rounded fp32 epilogue, so its float32 output equals the NumPy restatement of that arithmetic
  (tests/stem_model.py) bit for bit — with and without the fused gather (`rows`, repeated indices
  included).  The bf16 output is the float32 one rounded to nearest even, and the float32 output
  stays within 1e-4 of the activation scale of the float32 convolution
  (derl/models.py:102-103,117-123)."""
  gen = torch.Generator(device=DEV).manual_seed(batch)
  weight = torch.randn(32, 4, 8, 8, device=DEV, generator=gen) * 0.1
  bias = torch.randn(32, device=DEV, generator=gen) * 0.1
  frames = torch.randint(0, 256, (batch, 84, 84, 4), dtype=torch.uint8, device=DEV, generator=gen)
  rows = torch.randint(0, batch, (batch + 3,), device=DEV, generator=gen)
  model, _ = stem_model.stem_forward(frames.cpu().numpy(), weight.cpu().numpy(),
                                     bias.cpu().numpy())
  model = torch.from_numpy(model).to(DEV)
  for sel in (None, rows):
    want = model if sel is None else model[sel]
    if out_block == 2:
      want = K.space_to_depth(want, 2, False)
    got = K.stem_conv_relu(frames, weight, bias, torch.float32, out_block, sel)
    assert torch.equal(got, want), f"rows={'yes' if sel is not None else 'no'}"
    half = K.stem_conv_relu(frames, weight, bias, torch.bfloat16, out_block, sel)
    assert torch.equal(half, got.to(torch.bfloat16)), f"bf16, rows={'yes' if sel is not None else 'no'}"
  if out_block == 1:
    torch.backends.cudnn.allow_tf32 = False
    try:
      src = frames.permute(0, 3, 1, 2).float() / 255
      want = torch.relu(torch.nn.functional.conv2d(src, weight, bias, stride=4)).permute(0, 2, 3, 1)
    finally:
      torch.backends.cudnn.allow_tf32 = True
    got = K.stem_conv_relu(frames, weight, bias, torch.float32, 1, None)
    assert (got - want).abs().max().item() <= 1e-4 * want.abs().max().item()


def test_stem_tcgen05_kernel_is_deterministic_under_repetition():
  """Stress for the mbarrier rings of K6t (TMA -> MMA -> two epilogue groups -> TMA store): 30
  launches over batch sizes that leave CTAs with 0, 1 or many frames must all give the first
  launch's bytes (a race in the pipeline shows up as a sporadic difference), for the float32 and
  the bf16 staging layouts."""
  gen = torch.Generator(device=DEV).manual_seed(9)
  weight = torch.randn(32, 4, 8, 8, device=DEV, generator=gen) * 0.1
  bias = torch.randn(32, device=DEV, generator=gen) * 0.1
  for batch in (5, 148, 151, 2000):
    frames = torch.randint(0, 256, (batch, 84, 84, 4), dtype=torch.uint8, device=DEV,
                           generator=gen)
    for dtype in (torch.float32, torch.bfloat16):
      ref = K.stem_conv_relu(frames, weight, bias, dtype, 2, None)
      for _ in range(30):
        again = K.stem_conv_relu(frames, weight, bias, dtype, 2, None)
        assert torch.equal(again, ref)


def _expected_relu_mask(plain_out):
  """[B, 14, 32] words of derl_b200_stem_conv_relu_mask from the plain [B, 20, 20, 32] activation:
  bit l of (tile t, channel c) = out > 0 at padded pixel 21 oy + ox = 32 t + l."""
  batch = plain_out.shape[0]
  m = torch.arange(448, device=plain_out.device)
  oy, ox = m // 21, m % 21
  valid = (m < 420) & (ox < 20)
  pos = torch.zeros(batch, 448, 32, dtype=torch.int64, device=plain_out.device)
  pos[:, valid] = (plain_out[:, oy[valid], ox[valid], :] > 0).to(torch.int64)
  weights = (1 << torch.arange(32, device=plain_out.device, dtype=torch.int64)).view(1, 1, 32, 1)
  return (pos.view(batch, 14, 32, 32) * weights).sum(2)


@pytest.mark.parametrize("blocked", [False, True])
def test_stem_tcgen05_pair_against_its_number_format(blocked):
  """K6t + K7t (the pair a training step uses): the forward's float32 output is the plain
  `stem_conv_relu` output bit for bit, its ReLU signs differ from the float32 convolution's only
  for the few activations within ~1e-4 of zero, and its ReLU mask is exactly (output > 0) in the
  padded pixel-tile layout.  The backward (tcgen05, frame as an MN-major operand, gradient digits
  K-major, accumulators folded per frame from tensor memory) under that mask equals the float64
  gradients of its number format — the dequantised digits s (q1 + q2 / 254) of
  tests/stem_model.py — to float32 summation-order noise (1e-6 of the largest entry: the per-frame
  integer sums are exact), and float32 autograd within the format's tolerance (2e-4 / 1e-5).
  With the fused gather it is bit-identical to the materialised rows, and it is deterministic."""
  torch.backends.cudnn.allow_tf32 = False
  try:
    gen = torch.Generator(device=DEV).manual_seed(5)
    weight = torch.randn(32, 4, 8, 8, device=DEV, generator=gen) * 0.05
    bias = torch.randn(32, device=DEV, generator=gen) * 0.1
    block = 2 if blocked else 1
    for batch in (1, 3, 4, 150, 310, 333):
      frames = torch.randint(0, 256, (batch, 84, 84, 4), device=DEV, dtype=torch.uint8,
                             generator=gen)
      out, mask = K.stem_conv_relu_mask(frames, weight, bias, block, None)
      assert torch.equal(out, K.stem_conv_relu(frames, weight, bias, torch.float32, block, None))
      plain = K.space_to_depth(out, 2, True) if blocked else out
      assert torch.equal(mask.to(torch.int64) & 0xffffffff, _expected_relu_mask(plain))
      inputs = frames.permute(0, 3, 1, 2).float() / 255
      exact = torch.relu(torch.nn.functional.conv2d(inputs, weight, bias, stride=4))
      keep = plain.permute(0, 3, 1, 2) > 0
      assert int((keep != (exact > 0)).sum()) <= max(2, exact.numel() // 20000)
      grad = torch.randn(batch, 32, 20, 20, device=DEV, generator=gen) * \
          torch.rand(batch, 1, 1, 1, device=DEV, generator=gen) * 1e-3
      g_nhwc = grad.permute(0, 2, 3, 1).contiguous()
      if blocked:
        g_nhwc = K.space_to_depth(g_nhwc, 2, False)
      g_in = g_nhwc.permute(0, 3, 1, 2)
      new_w, new_b = K.stem_backward_masked(frames, g_in, mask, blocked, None)
      masked = grad * keep
      s, q1, q2 = stem_model.gradient_digits(masked.permute(0, 2, 3, 1).cpu().numpy())
      digits = torch.from_numpy(s * (q1 + q2 / 254.0)).to(DEV).permute(0, 3, 1, 2)
      fmt_w = torch.nn.grad.conv2d_weight(frames.permute(0, 3, 1, 2).double(), weight.shape,
                                          digits, stride=4) / 255.0
      fmt_b = masked.double().sum((0, 2, 3))
      assert (new_w - fmt_w).abs().max() <= 1e-6 * fmt_w.abs().max()
      assert (new_b - fmt_b).abs().max() <= 1e-6 * fmt_b.abs().max()
      want_w = torch.nn.grad.conv2d_weight(inputs, weight.shape, masked, stride=4)
      want_b = masked.sum((0, 2, 3))
      assert (new_w - want_w).abs().max() < 2e-4 * want_w.abs().max()
      assert (new_b - want_b).abs().max() < 1e-5 * want_b.abs().max()
      # fused gather: bit-identical to the materialised rows; repeated launches bit-identical
      rows = torch.randint(0, batch, (batch + 2,), device=DEV, generator=gen)
      out_r, mask_r = K.stem_conv_relu_mask(frames, weight, bias, block, rows)
      g_r = g_in[rows].contiguous(memory_format=torch.channels_last)
      a = K.stem_backward_masked(frames, g_r, mask_r, blocked, rows)
      b = K.stem_backward_masked(frames[rows].contiguous(), g_r, mask_r, blocked, None)
      assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
      for _ in range(5):
        again = K.stem_backward_masked(frames, g_r, mask_r, blocked, rows)
        assert torch.equal(again[0], a[0]) and torch.equal(again[1], a[1])
  finally:
    torch.backends.cudnn.allow_tf32 = True


def test_model_routes_float32_stem_through_the_tcgen05_pair(monkeypatch):
  """NatureCNNModel in a float32 training step under allow_tf32 runs its stem forward through K6t
  (`stem_conv_relu_mask`: the mask is saved, not the activation) and its backward through K7t
  (`stem_backward_masked`), and the stem's weight and bias gradients are bit for bit what that op
  returns for the arguments the model passed it."""
  calls = {"stem_conv_relu_mask": [], "stem_backward_masked": []}
  for name in calls:
    def record(*args, _op=getattr(K, name), _calls=calls[name]):
      _calls.append(args)
      return _op(*args)
    monkeypatch.setattr(K, name, record)
  frames = torch.randint(0, 256, (40, 84, 84, 4), dtype=torch.uint8, device=DEV)
  torch.manual_seed(0)
  model = d.NatureCNNModel([4, 1])
  logits, values = model(frames)
  (logits.square().sum() + values.sum()).backward()
  monkeypatch.undo()
  assert [len(v) for v in calls.values()] == [1, 1], calls
  grad_w, grad_b = K.stem_backward_masked(*calls["stem_backward_masked"][0])
  stem = next(m for m in model.modules() if isinstance(m, torch.nn.Conv2d))
  assert stem.kernel_size == (8, 8)
  assert torch.equal(stem.weight.grad, grad_w) and torch.equal(stem.bias.grad, grad_b)


# ------------------------------------------------------------------------------ K9: linear heads
@pytest.mark.parametrize("batch,units,with_hidden_bias", [
    (1, 5, True), (7, 5, False), (1000, 5, True), (4099, 19, True), (300, 32, False), (64, 1, True)])
def test_linear_heads_match_float64_linear_layers(batch, units, with_hidden_bias):
  """K9 forward and backward against the same formulas in float64 (`F.linear` heads on
  hidden + bias, derl/models.py:201-202): float32 FMA arithmetic, so 1e-5 of each tensor's scale;
  twice the same launch is bit-identical (fixed summation order)."""
  K = torch.ops.derl_b200
  gen = torch.Generator(device=DEV).manual_seed(batch * 37 + units)
  hidden = torch.randn(batch, 512, device=DEV, generator=gen)
  hb = torch.randn(512, device=DEV, generator=gen) * .3 if with_hidden_bias else None
  weight = torch.randn(units, 512, device=DEV, generator=gen) * .05
  bias = torch.randn(units, device=DEV, generator=gen)
  grad_out = torch.randn(batch, units, device=DEV, generator=gen)
  leaves = [t.clone().requires_grad_() for t in (hidden, weight, bias)]
  hb_leaf = hb.clone().requires_grad_() if hb is not None else None
  out = K.linear_heads(leaves[0], hb_leaf, leaves[1], leaves[2])
  out.backward(grad_out)
  h64, w64, b64 = (t.double().requires_grad_() for t in (hidden, weight, bias))
  hb64 = hb.double().requires_grad_() if hb is not None else None
  want = torch.nn.functional.linear(h64 + hb64 if hb is not None else h64, w64, b64)
  want.backward(grad_out.double())

  def close(got, ref, what):
    scale = ref.abs().max().item() + 1e-30
    assert (got.double() - ref).abs().max().item() <= 1e-5 * scale, what
  close(out, want, "out")
  close(leaves[0].grad, h64.grad, "grad_hidden")
  close(leaves[1].grad, w64.grad, "grad_weight")
  close(leaves[2].grad, b64.grad, "grad_bias")
  if hb is not None:
    close(hb_leaf.grad, hb64.grad, "grad_hidden_bias")
  again = K.linear_heads_backward(hidden, hb, weight, grad_out)
  once = K.linear_heads_backward(hidden, hb, weight, grad_out)
  assert all(torch.equal(a, b) for a, b in zip(again, once))
  assert torch.equal(K.linear_heads(hidden, hb, weight, bias), out.detach())


def test_model_with_fused_heads_equals_the_library_heads():
  """NatureCNNModel.fused_heads on/off (float32 library arithmetic, TF32 off): same outputs and
  parameter gradients to 2e-5 of their scale — including the trunk's deferred linear bias, whose
  gradient comes from the heads' column sums."""
  frames = torch.randint(0, 256, (48, 84, 84, 4), dtype=torch.uint8, device=DEV)
  saved = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
  torch.backends.cudnn.allow_tf32 = False
  torch.backends.cuda.matmul.allow_tf32 = False
  try:
    results = []
    for fused in (True, False):
      torch.manual_seed(0)
      model = d.NatureCNNModel([6, 1])
      with torch.no_grad():   # orthogonal_init zeroes the biases: make them count
        for p in model.parameters():
          if p.dim() == 1:
            p.copy_(torch.randn_like(p) * .1)
      model.fused_heads = fused
      logits, values = model(frames)
      assert logits.shape == (48, 6) and values.shape == (48, 1)
      assert logits.is_contiguous() and values.is_contiguous()
      (logits.square().sum() + (values * torch.arange(48, device=DEV)[:, None]).sum()).backward()
      results.append(([logits.detach(), values.detach()],
                      {n: p.grad.clone() for n, p in model.named_parameters()}))
    (outs_a, grads_a), (outs_b, grads_b) = results
    for a, b in zip(outs_a, outs_b):
      assert (a - b).abs().max() <= 2e-5 * b.abs().max()
    for name in grads_b:
      a, b = grads_a[name], grads_b[name]
      assert (a - b).abs().max() <= 2e-5 * b.abs().max() + 1e-12, name
  finally:
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved
