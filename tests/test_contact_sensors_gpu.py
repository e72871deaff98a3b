"""Contact force sensors (so101_contact_sensors) on the device: closed forms of tests/kat_analytic.py, parity with the float64
restatement over the oracle's efc_force (tests/contact_sensor_reference.py) on the harvested solver-tier batch, invariance of the
rollout when sensors are on, bit-identical readout in every float64 solver tier, the zero rules and argument validation."""
import ctypes

import numpy as np
import pytest
import torch

import contact_sensor_reference as csr
import kat_analytic as ka
from so101_sim_b200.model import body_set
from test_analytic_gpu import _kat_env, _put
from test_solver_tiers_gpu import MODELS, _oracle_substep, _two_arm_states, batch

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


# ------------------------------------------------------------------------------------------------ closed forms
# float32 bars, relative to the load: set from the values measured on a B200 (printed by each test)
F32_BAR = 1e-3   # measured on a B200: resting box 7.5e-6, stack 3.2e-4 (DESIGN.md section 7c)


@pytest.mark.parametrize('precision', ['f64', 'f32'])
def test_resting_box_carries_its_weight(built, precision):
  env = _kat_env(built, 1, precision)
  box = body_set(env.model, 'object')
  env.set_contact_sensors([(box, 'others')])
  _put(env, [ka.scene_state(env.model['qpos0'], (0.25, 0.0, ka.TABLE_TOP + ka.BOX_HALF[2]))])
  zero = torch.zeros(1, 6, device=DEV)
  for _ in range(100):
    env.step(zero)
  r = env.contact_sensors()[0, 0].double().cpu().numpy()
  w = ka.BOX_MASS * ka.G
  err = max(abs(r[2] / w - 1), abs(r[3] / w - 1), np.abs(r[:2]).max() / w)
  print(f'{precision} resting box readout / m g: {r[:4] / w}, count {r[4]}; worst relative error {err:.3g}')
  assert r[4] == 4
  assert err < (1e-6 if precision == 'f64' else F32_BAR)
  env.close()


@pytest.mark.parametrize('precision', ['f64', 'f32'])
def test_stack_passes_the_load_down(built, precision):
  env = _kat_env(built, 1, precision)
  box, cap, static = body_set(env.model, 'object'), body_set(env.model, 'container'), body_set(env.model, 'static')
  env.set_contact_sensors([(cap, box), (box, static), (box, cap)])
  _put(env, [ka.stack_state(env.model['qpos0'])])
  zero = torch.zeros(1, 6, device=DEV)
  for _ in range(150):
    env.step(zero)
  r = env.contact_sensors()[0].double().cpu().numpy()
  wc, wb = ka.CAP_MASS * ka.G, (ka.BOX_MASS + ka.CAP_MASS) * ka.G
  err = max(abs(r[0, 2] / wc - 1), abs(r[0, 3] / wc - 1), abs(r[1, 2] / wb - 1), abs(r[1, 3] / wb - 1),
            np.abs(r[0, :2]).max() / wc, np.abs(r[1, :2]).max() / wb)
  print(f'{precision} stack: (capsule, box) / m_cap g {r[0, :4] / wc}, (box, static) / (m_box + m_cap) g {r[1, :4] / wb}; '
        f'worst relative error {err:.3g}')
  assert r[0, 4] == 2 and r[1, 4] == 4
  assert err < (1e-6 if precision == 'f64' else F32_BAR)
  assert np.array_equal(r[2, :3], -r[0, :3]) and np.array_equal(r[2, 3:], r[0, 3:])
  env.close()


@pytest.mark.parametrize('precision', ['f64', 'f32'])
def test_sliding_box_sits_on_the_friction_cone(built, precision):
  """A box on the table given 0.3 m/s along +x, one substep per step, 12 steps.  Momentum balance: the readout (box, others)
  is the net contact force on the box, so m (v' - v) / h = F - m g z on every step (its centre of mass is the body origin).
  On the steps where all four corners slide, the friction force opposes the velocity and |F_t| / F_n = mu (elliptic cone,
  within the 1 % soft-cone margin of test_oracle_analytic's sliding test).  The float64 oracle gives the same sequence: the box
  hops for four steps after the velocity is set, lands on all four corners, then rocks on two, where one of them sticks and the
  ratio drops below mu."""
  env = _kat_env(built, 1, precision, control_timestep=0.002)
  box = body_set(env.model, 'object')
  env.set_contact_sensors([(box, 'others')])
  _put(env, [ka.scene_state(env.model['qpos0'], (0.1, 0.0, ka.TABLE_TOP + ka.BOX_HALF[2]))])
  zero = torch.zeros(1, 6, device=DEV)
  for _ in range(500):
    env.step(zero)
  q, v = env.get_state(torch.float64)
  v[:, 6] = 0.3
  env.set_state(q, v)
  w = ka.BOX_MASS * ka.G
  ratios, worst = [], 0.0
  for _ in range(12):
    v0 = env.get_state(torch.float64)[1][0, 6:9].cpu().numpy()
    env.step(zero)
    v1 = env.get_state(torch.float64)[1][0, 6:9].cpu().numpy()
    r = env.contact_sensors()[0, 0].double().cpu().numpy()
    worst = max(worst, float(np.abs(ka.BOX_MASS * (v1 - v0) / ka.DT + np.array([0, 0, w]) - r[:3]).max() / w))
    if r[4] == 4:
      ratios.append(float(np.hypot(r[0], r[1]) / r[2]))
      assert r[0] < 0 and abs(r[1]) < 1e-3 * abs(r[0]), r
  print(f'{precision} sliding box: momentum balance worst error / m g {worst:.3g}; |F_t| / F_n on the steps with four sliding '
        f'contacts {ratios} (mu = {ka.MU})')
  assert worst < (1e-6 if precision == 'f64' else 1e-3)
  assert len(ratios) >= 2 and all(abs(x / ka.MU - 1) < 1e-2 for x in ratios)
  env.close()


# ------------------------------------------------------------------------------------------------ oracle parity
def _sensor_sets(meta):
  narm = int(meta['nu'][0]) // 6
  jaws = sorted({b for k in range(narm) for b in body_set(meta, 'gripper', k)})
  arm = sorted({b for k in range(narm) for b in body_set(meta, 'arm', k)})
  obj, cont, static = body_set(meta, 'object'), body_set(meta, 'container'), body_set(meta, 'static')
  return [(jaws, obj), (obj, cont), (obj, static), (arm, static)]


def _parity_batch(model):
  """The harvested batch of test_solver_tiers_gpu, plus the constructed state csr.jaw_object_state: the harvest's only
  jaw-on-object contacts (none in the one-arm scene, three in the two-arm scene) come in states that also touch a curved static
  obstacle, where forces are compared to a looser bar, so the grasp force is pinned by this state."""
  jaw = csr.jaw_object_state(model)
  assert not jaw['curved']
  return list(batch(model)) + [jaw]


def _sensor_batch(model, precision, recs, pairs):
  from test_solver_tiers_gpu import _env
  env = _env(model, precision, len(recs), control_timestep=0.002)
  env.set_initial_state(torch.tensor(np.stack([r['q'] for r in recs])), torch.tensor(np.stack([r['v'] for r in recs])))
  env.reset()
  env.set_contact_sensors(pairs)
  env.step(torch.tensor(np.stack([r['a'] for r in recs]), dtype=torch.float32, device=DEV))
  out = dict(s=env.contact_sensors().double().cpu().numpy(), tier=env.debug_read('tier').flatten().cpu().numpy(), counters=env.counters())
  env.close()
  return out


def _err(got, want):
  """Force error of one sensor row relative to max(1 N, the reference's largest component)."""
  return float(np.abs(got[:4] - want[:4]).max() / max(1.0, np.abs(want[:4]).max()))


# Bars of the float64 parity test, set from the errors measured on a B200 (DESIGN.md section 7c): 5.3e-8 at worst away from
# curved obstacles (the readout is float32: one rounding is up to 6e-8 of the largest component), 4.6e-3 on states touching one
F64_BAR, F64_BAR_CURVED = 2e-7, 2e-2


@pytest.mark.parametrize('model', MODELS)
def test_f64_readout_matches_the_oracle_in_every_tier(built, model):
  """One float64 substep of every harvested state and of the constructed jaw-on-object state: the readout of jaw / object,
  object / container, object / static and arm / static against the restatement over the oracle's efc_force.  Counts equal
  exactly.  Forces, relative to max(1 N, the largest reference component), agree to F64_BAR; on states touching a curved static
  obstacle EPA stops by tolerance (test_solver_tiers_gpu), which moves contact points and depths, so there the bar is
  F64_BAR_CURVED.  The jaw / object rows of states away from curved obstacles must include a nonzero force."""
  recs = _parity_batch(model)
  from oracle.oracle import OracleSim
  meta = OracleSim(model).meta
  pairs = _sensor_sets(meta)
  got = _sensor_batch(model, 'f64', recs, pairs)
  assert got['counters']['diverged'] == 0 and got['counters']['contacts_dropped'] == 0
  worst, worst_curved, worst_jaw = {t: 0.0 for t in range(3)}, 0.0, 0.0
  jaw_states, jaw_forces, bad = 0, 0, []
  for e, r in enumerate(recs):
    o, cons = _oracle_substep(model, r)
    want = csr.readout(meta, cons, o.field('efc_force'), pairs)
    jaw_states += want[0, 4] > 0
    if not np.array_equal(got['s'][e][:, 4], want[:, 4]):
      bad.append(('count', e, got['s'][e][:, 4].tolist(), want[:, 4].tolist()))
    err = max(_err(got['s'][e][k], want[k]) for k in range(len(pairs)))
    t = int(got['tier'][e])
    if want[0, 4] > 0:
      print(f'  state {e} (tier {t}, curved {r["curved"]}): jaw / object readout {got["s"][e][0].tolist()}, restatement {want[0].tolist()}')
    if r['curved']:
      worst_curved = max(worst_curved, err)
      continue
    worst[t] = max(worst[t], err)
    if want[0, 4] > 0:
      jaw_forces += want[0, 3] > 0
      worst_jaw = max(worst_jaw, _err(got['s'][e][0], want[0]))
  print(f'{model} f64 sensor readout vs oracle: {len(recs)} states, {jaw_states} with jaw / object contacts ({jaw_forces} with force '
        f'away from curved obstacles, worst jaw / object error {worst_jaw:.3g}); worst relative force error per tier {worst}, '
        f'on curved obstacles {worst_curved:.3g}')
  assert not bad, bad
  assert jaw_forces >= 1
  assert all(w < F64_BAR for w in worst.values()), worst
  assert worst_curved < F64_BAR_CURVED


@pytest.mark.parametrize('model', MODELS)
def test_f32_readout_error_per_tier(built, model):
  """The same batch in the float32 product arithmetic: force error against the float64 restatement, reported per tier
  (median, worst; measured on a B200 in DESIGN.md section 7c).  A float32 narrow phase may find a contact more or fewer at a tier
  edge, so counts are not compared, and the worst states are arms driven centimetres into the table or the props, where float32
  contact rows are stiff (as in test_solver_tiers_gpu): the median is bounded, at 10x the measured 4e-5."""
  recs = _parity_batch(model)
  from oracle.oracle import OracleSim
  meta = OracleSim(model).meta
  pairs = _sensor_sets(meta)
  got = _sensor_batch(model, 'f32', recs, pairs)
  errs = {t: [] for t in range(3)}
  for e, r in enumerate(recs):
    o, cons = _oracle_substep(model, r)
    want = csr.readout(meta, cons, o.field('efc_force'), pairs)
    errs[int(got['tier'][e])].append(max(_err(got['s'][e][k], want[k]) for k in range(len(pairs))))
  stats = {t: (len(x), float(np.median(x)), float(np.max(x))) for t, x in errs.items() if x}
  print(f'{model} f32 sensor readout vs oracle, relative force error per tier (states, median, worst): {stats}')
  assert np.isfinite(got['s']).all()
  assert all(s[1] < 4e-4 for s in stats.values()), stats


# ------------------------------------------------------------------------------------------------ invariance and determinism
def _rollout(model, precision, sensors, steps=30, n=64):
  from test_solver_tiers_gpu import _env
  env = _env(model, precision, n)
  if model == 'so100_handover_banana':
    env.sample_prop_initial_states(seed=11, settle_steps=0)
  else:
    env.set_initial_state(*_two_arm_states(model, n, seed=11)); env.reset()
  if sensors:
    env.set_contact_sensors(_sensor_sets(env.model))
  g = torch.Generator(device=DEV); g.manual_seed(5)
  spec = env.action_spec()
  lo, hi = torch.tensor(spec.minimum, device=DEV), torch.tensor(spec.maximum, device=DEV)
  acts = (lo + torch.rand(steps, n, env.nu, generator=g, device=DEV) * (hi - lo)) * 0.6
  c0 = env.counters()
  trace, readouts = [], []
  for t in range(steps):
    ts = env.step(acts[t])
    trace.append(torch.cat([ts.step_type.double()[:, None], ts.reward.double()[:, None], ts.discount.double()[:, None]]
                           + [o.double() for o in ts.observation.values() if o.shape[1]], 1).cpu())
    if sensors:
      readouts.append(env.contact_sensors().cpu())
  c1 = env.counters()
  q, v = env.get_state(torch.float64)
  res = dict(q=q.cpu(), v=v.cpu(), trace=torch.stack(trace), dropped=env.contacts_dropped_per_env().cpu(),
             launches=c1['kernel_launches'] - c0['kernel_launches'], graphs=c1['graph_launches'] - c0['graph_launches'],
             readout=torch.stack(readouts) if sensors else None)
  env.close()
  return res


@pytest.mark.parametrize('model', MODELS)
@pytest.mark.parametrize('precision', ['f32', 'f64'])
def test_sensors_do_not_change_the_rollout(built, model, precision):
  """30 random-action steps with the four sensors on and off: state, observations, reward, discount and step type are bit
  for bit the same, and so are the kernel launches and graph launches per step (the sensor pass runs inside the solve
  kernels; its only other work is a memset node in the step graph).  Envs that lost contacts to a full buffer in either run are
  left out: which contacts survive then depends on arrival order, so two runs with sensors off differ there too."""
  off, on = _rollout(model, precision, False), _rollout(model, precision, True)
  keep = (off['dropped'] == 0) & (on['dropped'] == 0)
  differ = [k for k in range(len(keep)) if not (torch.equal(off['q'][k], on['q'][k]) and torch.equal(off['trace'][:, k], on['trace'][:, k]))]
  print(f'{model} {precision}: per step {off["launches"] / 30} kernel launches and {off["graphs"] / 30} graph launches, sensors off and on; '
        f'sensor rows with contacts {int((on["readout"][..., 4] > 0).sum())} of {on["readout"][..., 4].numel()}; '
        f'{int(keep.sum())} envs kept all contacts; envs that differ {differ} (dropped off / on: '
        f'{[(int(off["dropped"][k]), int(on["dropped"][k])) for k in differ]})')
  assert int(keep.sum()) >= 32
  for k in ('q', 'v'):
    assert torch.equal(off[k][keep], on[k][keep]), k
  assert torch.equal(off['trace'][:, keep], on['trace'][:, keep])
  assert off['launches'] == on['launches'] and off['graphs'] == on['graphs'] == 30
  assert int((on['readout'][..., 4] > 0).sum()) > 0 and torch.isfinite(on['readout']).all()


@pytest.mark.parametrize('model', MODELS)
def test_f64_readout_is_bit_identical_in_every_solver_tier(built, monkeypatch, model):
  """SO101_SOLVE_TIER_MIN = 0 / 1 / 2: the readout of every step is the same bits (envs that lost contacts to a full buffer in
  any run are left out, as in test_solver_tiers_gpu.test_forced_solver_tier_is_bit_identical)."""
  runs = []
  for t in (0, 1, 2):
    monkeypatch.setenv('SO101_SOLVE_TIER_MIN', str(t))
    runs.append(_rollout(model, 'f64', True, steps=25))
  keep = (torch.stack([r['dropped'] for r in runs]) == 0).all(0)
  assert int(keep.sum()) >= 32
  for r in runs[1:]:
    assert torch.equal(r['readout'][:, keep], runs[0]['readout'][:, keep])
  assert int((runs[0]['readout'][:, keep][..., 4] > 0).sum()) > 0


# ------------------------------------------------------------------------------------------------ zero rules
def _banana(n, precision='f32', time_limit=30.0, control_timestep=0.02):
  from so101_sim_b200.task_suite import create_batched_task_env
  env = create_batched_task_env('SO100HandOverBanana', num_envs=n, time_limit=time_limit, seed=0, device=DEV, reset_rounds=0, precision=precision,
                                control_timestep=control_timestep)
  env.sample_prop_initial_states(seed=3, settle_steps=5)
  env.reset()
  env.set_contact_sensors([('object', 'others'), ('container', 'static')])
  return env


def test_first_rows_after_auto_reset_and_reset_are_zero(built):
  env = _banana(8, time_limit=0.2)   # 10 control steps per episode
  zero = torch.zeros(8, 6, device=DEV)
  seen_first = 0
  for _ in range(14):
    ts = env.step(zero)
    s = env.contact_sensors()
    first = ts.step_type == 0
    seen_first += int(first.sum())
    assert torch.all(s[first] == 0)
    assert torch.all(s[~first][:, :, 4] > 0)   # the props rest on the table: every stepped env reads its contacts
  assert seen_first == 8
  before = env.contact_sensors()
  mask = torch.tensor([1, 0] * 4, dtype=torch.uint8, device=DEV)
  env.reset(mask)
  after = env.contact_sensors()
  assert torch.all(after[mask.bool()] == 0) and torch.equal(after[~mask.bool()], before[~mask.bool()])
  env.step(zero)
  env.reset()
  assert torch.all(env.contact_sensors() == 0)
  env.close()


@pytest.mark.parametrize('control_timestep', [0.02, 0.002])
def test_diverged_env_reads_zero(built, control_timestep):
  """A non-finite prop velocity fails the acceleration check on the step's first substep.  With 10 substeps per step the env is
  then frozen for the remaining ones; with one substep per step (0.002 s) it diverges on the last substep itself.  Either way
  its row is zero while the neighbouring env reads its contacts."""
  env = _banana(2, control_timestep=control_timestep)
  zero = torch.zeros(2, 6, device=DEV)
  for _ in range(int(round(0.04 / control_timestep))):   # 40 ms: the props have landed
    env.step(zero)
  q, v = env.get_state()
  v[1, 6] = float('inf')
  env.set_state(q, v)
  ts = env.step(zero)
  s = env.contact_sensors()
  assert int(ts.step_type[1]) == 2 and torch.all(s[1] == 0)
  assert int(ts.step_type[0]) == 1 and float(s[0, 0, 4]) > 0
  env.close()


def test_readout_is_zero_after_a_checkpoint_load_and_the_next_step_resumes(built):
  env = _banana(16, precision='f64')
  zero = torch.zeros(16, 6, device=DEV)
  for _ in range(3):
    env.step(zero)
  ck = env.save_checkpoint()
  env.step(zero)
  want = env.contact_sensors()
  env.load_checkpoint(ck)
  assert torch.all(env.contact_sensors() == 0)
  env.step(zero)
  assert torch.equal(env.contact_sensors(), want)
  env.close()


# ------------------------------------------------------------------------------------------------ validation
def test_invalid_sensor_specs_are_refused(built):
  from so101_sim_b200 import _lib
  from so101_sim_b200.task_suite import create_batched_task_env
  arm = create_batched_task_env('SO100ArmOnly', num_envs=4, time_limit=30.0, seed=0, device=DEV)
  with pytest.raises(ValueError):
    arm.set_contact_sensors([('gripper', 'others')])
  masks = ((ctypes.c_uint32 * 2) * 1)()
  masks[0][0], masks[0][1] = 1 << 6, 1 << 0
  assert arm._lib.so101_contact_sensors(arm._h, 1, ctypes.cast(masks, ctypes.c_void_p)) < 0   # through the handle too
  arm.close()
  env = _banana(4)
  L, h = env._lib, env._h

  def call(pairs):
    m = ((ctypes.c_uint32 * 2) * max(1, len(pairs)))()
    for k, (a, b) in enumerate(pairs):
      m[k][0], m[k][1] = a, b
    return L.so101_contact_sensors(h, len(pairs), ctypes.cast(m, ctypes.c_void_p))

  assert call([(1 << 11, 1 << 12)] * 17) < 0           # more than 16 sensors
  assert call([(0, 1 << 12)]) < 0 and call([(1 << 11, 0)]) < 0   # empty sets
  assert call([(1 << 11 | 1 << 12, 1 << 12)]) < 0      # overlapping sets
  assert call([(1 << 11, 1 << 13)]) < 0                # body 13 >= nbody (13)
  assert call([(1 << 11, 1 << 12)] * 16) == 0          # 16 is allowed
  with pytest.raises(ValueError):
    env.set_contact_sensors([('object', 'object')])
  with pytest.raises(ValueError):
    env.set_contact_sensors([('others', 'others')])
  with pytest.raises(ValueError):
    env.set_contact_sensors([(11, 13)])
  with pytest.raises(ValueError):
    env.set_contact_sensors([('object', 'others')] * 17)
  env.set_contact_sensors([('object', 'others'), ('gripper', 'object')])
  env.step(torch.zeros(4, 6, device=DEV))
  buf = torch.zeros(4 * 2 * 5 - 1, device=DEV)
  assert L.so101_contact_sensors_read(h, ctypes.c_void_p(buf.data_ptr()), buf.numel(), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)) < 0
  buf = torch.zeros(4 * 2 * 5, device=DEV)
  assert L.so101_contact_sensors_read(h, ctypes.c_void_p(buf.data_ptr()), buf.numel(), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)) == 0
  assert torch.equal(buf.view(4, 2, 5), env.contact_sensors())
  env.set_contact_sensors([])
  assert env.contact_sensors().shape == (4, 0, 5)
  env.close()
