"""GPU parity tests of the full contact scene kernel (SO100HandOverBanana) against the float64 oracle, through the C-ABI."""
import numpy as np
import pytest
import torch

from oracle.oracle import OracleSim

pytestmark = pytest.mark.gpu


def _env(built, **kw):
  from so101_sim_b200.task_suite import create_batched_task_env
  args = dict(task_name='SO100HandOverBanana', num_envs=8, time_limit=30.0, seed=0, device='cuda:0', reset_rounds=0)
  args.update(kw)
  return create_batched_task_env(**args)


def _initial(env, seed, clearance=0.002):
  env.sample_prop_initial_states(seed=seed, clearance=clearance, settle_steps=0)
  return env.get_state(torch.float64)


def _actions(env, steps, seed=1, scale=0.3):
  g = torch.Generator(device='cuda:0'); g.manual_seed(seed)
  spec = env.action_spec()
  lo, hi = torch.tensor(spec.minimum, device='cuda:0'), torch.tensor(spec.maximum, device='cuda:0')
  return (lo + torch.rand(steps, env.num_envs, 6, generator=g, device='cuda:0') * (hi - lo)) * scale


def test_f64_scene_matches_oracle(built):
  """Drop both props 2 mm onto the table while the arm moves: float64 GPU path vs float64 oracle, same algorithm.
  Envs whose bowl lands on the static cylinder obstacle (scene_pbr.xml:144-146) go through EPA on a curved surface, whose
  tolerance-terminated normal is sensitive to FMA-level round-off; they are held to 1e-4, the others to 1e-7."""
  env = _env(built, precision='f64', num_envs=4)
  q0, v0 = _initial(env, seed=3)
  acts = _actions(env, 12)
  sims = []
  for e in range(4):
    o = OracleSim('so100_handover_banana', collide=True)
    o.set_state(q0[e].cpu().numpy(), v0[e].cpu().numpy())
    sims.append(o)
  worst = np.zeros(4)
  for t in range(12):
    ts = env.step(acts[t])
    q, v = env.get_state(torch.float64)
    for e in range(4):
      r = sims[e].control_step(acts[t, e].double().cpu().numpy())
      worst[e] = max(worst[e], np.abs(q[e].cpu().numpy() - sims[e].qpos).max())
      assert float(ts.reward[e]) == r
  print('f64 scene max |dqpos| per env over 120 substeps:', worst)
  assert np.sort(worst)[:2].max() < 1e-7, worst     # at least two envs are flat-contact only
  assert worst.max() < 1e-4, worst
  assert env.counters()['contacts_dropped'] == 0 and env.counters()['diverged'] == 0
  env.close()


def test_f64_scene_implicitfast_matches_oracle(built):
  """The contact scene with integrator='implicitfast': float64 CUDA path against the oracle's implicitfast over 60 substeps."""
  env = _env(built, precision='f64', num_envs=2, integrator='implicitfast')
  q0, v0 = _initial(env, seed=3)
  acts = _actions(env, 6)
  sims = []
  for e in range(2):
    o = OracleSim('so100_handover_banana', collide=True, integrator='implicitfast')
    o.set_state(q0[e].cpu().numpy(), v0[e].cpu().numpy())
    sims.append(o)
  for t in range(6):
    env.step(acts[t])
    for e in range(2):
      sims[e].control_step(acts[t, e].double().cpu().numpy())
  q, v = env.get_state(torch.float64)
  for e in range(2):
    assert np.abs(q[e].cpu().numpy() - sims[e].qpos).max() < 1e-7 and np.abs(v[e].cpu().numpy() - sims[e].qvel).max() < 1e-5
  env.close()


def test_contacts_match_oracle(built):
  """Contact lists (geom pair, distance, position, normal) of one substep, float64 GPU vs oracle."""
  env = _env(built, precision='f64', num_envs=3, control_timestep=0.002)
  q0, v0 = _initial(env, seed=3, clearance=-0.0002)   # start slightly penetrating so that contacts exist at once
  env.debug_contacts()
  env.step(torch.zeros(3, 6, device='cuda:0'))
  got = env.debug_contacts()
  for e in (0, 2):
    o = OracleSim('so100_handover_banana', collide=True)
    o.set_state(q0[e].cpu().numpy(), v0[e].cpu().numpy()); o.forward()
    ref = o.contacts()
    assert len(ref) > 10 and len(got[e]) == len(ref)
    for g, r in zip(got[e], ref):
      assert (g[0], g[1]) == (r['geom1'], r['geom2'])
      assert abs(g[2] - r["dist"]) < 5e-6 and np.abs(g[3] - r['pos']).max() < 1e-5 and np.abs(g[4] - r['frame'][0]).max() < 1e-5
      assert g[2] < 0 and abs(np.linalg.norm(g[4]) - 1) < 1e-5
  env.close()


def test_f32_scene_tracks_oracle(built):
  """float32 product path, ALL envs of the batch against the float64 oracle over 25 control steps (250 substeps) in which the
  props drop 2 mm onto the table while the arm moves.  Bars: reward / discount / step_type exact; the arm within north_star's
  1e-4 relative for as long as it is contact-free (the tolerance is stated for contact-free rollouts); props within 0.2 mm /
  2e-3 (quaternion) through the landing transient and back within 2e-5 / 2e-5 at rest - except a prop that lands on one of the
  scene's CURVED static obstacles (capsule / cylinder, scene_pbr.xml:141-146), where EPA's termination tolerance (1e-6 in
  float32, [upstream] ccd_tolerance) bounds the contact normal only to ~sqrt(2 tol / r) and the rest pose to ~1e-3.
  Measured errors are printed."""
  N = 4
  env = _env(built, precision='f32', num_envs=N)
  q0, v0 = _initial(env, seed=5)
  acts = _actions(env, 25, scale=0.1)
  sims = []
  for e in range(N):
    o = OracleSim('so100_handover_banana', collide=True)
    o.set_state(q0[e].cpu().numpy(), v0[e].cpu().numpy())
    sims.append(o)
  meta = sims[0].meta
  arm_bodies = set(int(b) for b in meta['jnt_body'][:6])
  gbody, gtype = meta['geom_body'], meta['geom_type']
  curved_static = {g for g in range(len(gtype)) if gtype[g] in (2, 3) and meta['body_weld'][gbody[g]] == 0}
  arm_free = [True] * N       # no arm contact so far
  first_touch = [None] * N
  on_curved = [False] * N     # a prop has touched a curved static obstacle
  worst = dict(arm=0.0, arm_v=0.0, prop_p=0.0, prop_q=0.0)
  rows = []
  for t in range(25):
    ts = env.step(acts[t])
    q, v = env.get_state(torch.float64)
    for e, o in enumerate(sims):
      r = o.control_step(acts[t, e].double().cpu().numpy())
      assert float(ts.reward[e]) == r and int(ts.step_type[e]) == 1 and float(ts.discount[e]) == 1.0
      for c in o.contacts():
        if int(gbody[c['geom1']]) in arm_bodies or int(gbody[c['geom2']]) in arm_bodies:
          arm_free[e] = False
          if first_touch[e] is None: first_touch[e] = t + 1
        if c['geom1'] in curved_static or c['geom2'] in curved_static: on_curved[e] = True
      qe, ve = q[e].cpu().numpy(), v[e].cpu().numpy()
      ea = float(np.abs(qe[:6] - o.qpos[:6]).max() / max(1.0, np.abs(o.qpos[:6]).max()))
      ev = float(np.abs(ve[:6] - o.qvel[:6]).max() / max(1.0, np.abs(o.qvel[:6]).max()))
      pp = float(max(np.abs(qe[6:9] - o.qpos[6:9]).max(), np.abs(qe[13:16] - o.qpos[13:16]).max()))
      pq = float(max(np.abs(qe[9:13] - o.qpos[9:13]).max(), np.abs(qe[16:20] - o.qpos[16:20]).max()))
      rows.append((t + 1, e, ea, ev, pp, pq, arm_free[e], on_curved[e]))
      if arm_free[e]:
        worst['arm'] = max(worst['arm'], ea); worst['arm_v'] = max(worst['arm_v'], ev)
        assert ea < 1e-4 and ev < 1e-4, (t, e, ea, ev)                     # north_star: 1e-4 relative, contact-free arm
      else:
        assert ea < 1e-4 and ev < 2e-3, (t, e, ea, ev)                     # arm in contact (table / props): velocities are impact-sensitive
      if not on_curved[e]:
        worst['prop_p'] = max(worst['prop_p'], pp); worst['prop_q'] = max(worst['prop_q'], pq)
        assert pp < 2e-4 and pq < 2e-3, (t, e, pp, pq)                     # landing transient
      else:
        assert pp < 1e-3 and pq < 5e-3, (t, e, pp, pq)
  print('f32 scene, 4 envs x 25 steps, worst errors vs the float64 oracle:', {k: float(f'{x:.2g}') for k, x in worst.items()},
        '| first control step with an arm contact:', first_touch, '| prop on a curved obstacle:', on_curved)
  print('   final (env, arm rel, prop pos, prop quat):', [(r[1], float(f'{r[2]:.2g}'), float(f'{r[4]:.2g}'), float(f'{r[5]:.2g}')) for r in rows[-N:]])
  assert sum(1 for f in first_touch if f is None or f > 10) >= 2 and sum(not c for c in on_curved) >= 2   # both bars are exercised
  for r in rows[-N:]:
    if not r[7]:
      assert r[4] < 2e-5 and r[5] < 2e-5, r                               # at rest on the table: same pose as the oracle
  assert torch.isfinite(q).all() and env.counters()['diverged'] == 0 and env.counters()['contacts_dropped'] == 0
  assert int(env.contacts_dropped_per_env().sum()) == 0   # per-env view of the same counter
  env.close()


def test_scene_forced_divergence_ends_the_episode(built):
  """PhysicsError path of the contact scene (task_suite.py:153: raise_exception_on_physics_error=False): a non-finite prop
  velocity makes qacc fail [upstream] mj_checkAcc -> reward 0, discount 0, LAST for that env only; the next step() returns
  FIRST from the env's reset state.  The neighbouring env keeps stepping."""
  env = _env(built, num_envs=2)
  env.sample_prop_initial_states(seed=2, settle_steps=5)
  env.reset()
  q0, v0 = env.get_state()
  zero = torch.zeros(2, 6, device='cuda:0')
  env.step(zero)
  q, v = env.get_state()
  v[1, 6] = float('inf')
  env.set_state(q, v)
  d0 = env.counters()['diverged']
  ts = env.step(zero)
  assert int(ts.step_type[1]) == 2 and float(ts.reward[1]) == 0.0 and float(ts.discount[1]) == 0.0
  assert int(ts.step_type[0]) == 1 and float(ts.discount[0]) == 1.0
  assert env.counters()['diverged'] == d0 + 1
  ts = env.step(zero)
  assert int(ts.step_type[1]) == 0 and float(ts.reward[1]) == 0.0 and float(ts.discount[1]) == 1.0 and int(ts.step_type[0]) == 1
  qq, vv = env.get_state()
  assert torch.allclose(qq[1], q0[1]) and torch.isfinite(qq).all() and torch.isfinite(vv).all()
  env.close()


@pytest.mark.parametrize('precision', [64, 32])
def test_device_overlap_matches_the_reference_golden(built, precision):
  """The DEVICE 6-axis SAT (scene_kernel.inl overlap_oobb_oobb, the reward geometry) on the 240 box pairs whose flags were
  produced by executing the reference's own oobb_utils.py (tests/golden/oobb_overlap.json, tools/make_golden_oobb.py): every
  flag must be reproduced, in float64 and in the float32 the product path evaluates it in."""
  import ctypes, json, os
  from so101_sim_b200 import _lib
  g = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'oobb_overlap.json')))
  rows = [c['obj_pos'] + c['obj_quat'] + c['obj_half'] + c['ws_pos'] + c['ws_quat'] + c['container_half'] for c in g['cases']]
  want = torch.tensor([c['overlap'] for c in g['cases']], dtype=torch.uint8)
  cases = torch.tensor(rows, dtype=torch.float64, device='cuda:0').contiguous()
  out = torch.zeros(len(rows), dtype=torch.uint8, device='cuda:0')
  L = _lib.load()
  rc = L.so101_debug_overlap(precision, 0, ctypes.c_void_p(cases.data_ptr()), len(rows), ctypes.c_void_p(out.data_ptr()),
                             ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
  torch.cuda.synchronize()
  assert rc == 0
  got = out.cpu()
  assert int(want.sum()) > 40 and int((1 - want).sum()) > 40
  assert torch.equal(got, want), f'{int((got != want).sum())} of {len(rows)} flags differ: cases {torch.nonzero(got != want).flatten().tolist()}'


@pytest.mark.parametrize('precision', ['f64'])
def test_single_env_many_pairs_keeps_every_contact(built, precision):
  """num_envs = 1 with the banana resting inside the bowl (> 32 candidate geom pairs: 53 bowl hulls + 4 banana hulls against
  the table and each other): no hit record may be lost to a capacity that scales with the batch size (the hit list once held
  32 x num_envs records).  The state follows the float64 oracle; nothing is dropped."""
  env = _env(built, num_envs=1, precision=precision)
  q = torch.tensor(env.model['qpos0'], dtype=torch.float64).repeat(1, 1)
  q[:, :6] = 0
  q[:, 13:16] = torch.tensor([-0.25, -0.05, 0.4226], dtype=torch.float64); q[:, 16] = 1; q[:, 17:20] = 0
  q[0, 6:9] = torch.tensor([-0.25 - 0.0255, -0.05 - 0.0675, 0.4226 + 0.06], dtype=torch.float64)
  q[0, 9] = float(np.cos(0.4)); q[0, 10:12] = 0; q[0, 12] = float(np.sin(0.4))
  env.set_initial_state(q, torch.zeros(1, 18, dtype=torch.float64))
  env.reset()
  o = OracleSim('so100_handover_banana', collide=True)
  o.set_state(q[0].numpy(), np.zeros(18))
  zero = torch.zeros(1, 6, device='cuda:0')
  nmax = 0
  for t in range(15):
    ts = env.step(zero)
    r = o.control_step(np.zeros(6))
    qq, _ = env.get_state(torch.float64)
    n = int(env.debug_read('ncon')[0, 0])
    nmax = max(nmax, n)
    assert np.abs(qq[0].cpu().numpy() - o.qpos).max() < 1e-6, t
    assert float(ts.reward[0]) == r
    if r >= 1.0:   # banana at rest in the bowl: success, the env resets on the next step
      break
  assert nmax > 16 and env.counters()['contacts_dropped'] == 0
  env.close()


def test_default_creation_starts_from_settled_placements(built):
  """create -> reset -> step with no further set-up must start from sampled and settled prop placements (the reference places
  and settles the props in every initialize_episode, so100_hand_over.py:208-229,320-323), never from the blob's qpos0 with both
  props coincident at the world origin."""
  from so101_sim_b200.task_suite import create_batched_task_env
  env = create_batched_task_env('SO100HandOverBanana', num_envs=8, time_limit=30.0, seed=3, device='cuda:0')
  ts = env.reset()
  ps = ts.observation['physics_state']
  assert float(ps[:, 6].min()) >= 0.14 and float(ps[:, 6].max()) <= 0.36       # banana x in its placement range (+- settle drift / roll-off)
  assert float(ps[:, 13].min()) >= -0.33 and float(ps[:, 13].max()) <= -0.17   # bowl x
  assert abs(float(ps[:, 8].median()) - 0.4217) < 3e-3                         # bananas resting on the table top
  assert float(ps[:, :6].abs().max()) == 0.0                                   # arm qpos 0 (home is never applied, so100_task.py:308-313)
  ts = env.step(torch.zeros(8, 6, device='cuda:0'))
  assert ts.step_type.tolist() == [1] * 8 and env.counters()['diverged'] == 0
  assert float((ts.observation['physics_state'][:, 6:9] - ps[:, 6:9]).abs().max()) < 2e-3  # props stay put
  env.close()


def test_scene_observations_and_reward_flags(built):
  env = _env(built, num_envs=4)
  env.sample_prop_initial_states(seed=1, settle_steps=5)
  ts = env.reset()
  assert ts.observation['physics_state'].shape == (4, 38) and ts.observation['joints_vel'].shape == (4, 0)
  assert ts.step_type.tolist() == [0] * 4
  ts = env.step(torch.zeros(4, 6, device='cuda:0'))
  assert ts.step_type.tolist() == [1] * 4 and ts.reward.tolist() == [0.0] * 4 and ts.discount.tolist() == [1.0] * 4
  q, v = env.get_state()
  assert torch.allclose(ts.observation['physics_state'], torch.cat([q, v], dim=1))
  env.close()


def test_scene_success_reward_terminates(built):
  """Drop the banana onto the bowl's containment box: once both props are slower than 1e-3 m/s the overlap reward fires
  (so100_hand_over.py:238-275) -> reward 1, discount 0, LAST; the next step() auto-resets to FIRST (so100_task.py:292-302)."""
  env = _env(built, num_envs=2, precision='f64')
  q = torch.tensor(env.model['qpos0'], dtype=torch.float32).repeat(2, 1)
  q[:, :6] = 0
  q[:, 13:16] = torch.tensor([-0.25, -0.05, 0.4226]); q[:, 16] = 1; q[:, 17:20] = 0
  q[0, 6:9] = torch.tensor([-0.25 - 0.0255, -0.05 - 0.0675, 0.4226 + 0.09])
  q[0, 9] = float(np.cos(0.4)); q[0, 10:12] = 0; q[0, 12] = float(np.sin(0.4))
  q[1, 6:9] = torch.tensor([0.25, 0.0, 0.4237]); q[1, 9] = 1; q[1, 10:13] = 0
  v = torch.zeros(2, 18)
  env.set_initial_state(q, v)
  env.reset()
  o = OracleSim('so100_handover_banana', collide=True)
  o.set_state(q[0].double().numpy(), np.zeros(18))
  zero = torch.zeros(2, 6, device='cuda:0')
  hit = None
  for t in range(40):
    ts = env.step(zero)
    r = o.control_step(np.zeros(6))
    assert float(ts.reward[0]) == r, t
    assert float(ts.reward[1]) == 0.0 and int(ts.step_type[1]) == 1
    if r >= 1.0:
      hit = t
      break
  assert hit is not None and hit > 2
  assert float(ts.discount[0]) == 0.0 and int(ts.step_type[0]) == 2
  ts = env.step(zero)
  assert int(ts.step_type[0]) == 0 and float(ts.reward[0]) == 0.0 and float(ts.discount[0]) == 1.0
  assert int(ts.step_type[1]) == 1
  qq, _ = env.get_state()
  assert torch.allclose(qq[0].cpu(), q[0], atol=1e-6)
  env.close()


def test_f64_contact_rich_rollout_matches_oracle(built):
  """Arm driven by random targets through resting props for 25 control steps (250 substeps: arm-prop and arm-table hits,
  props pushed around, larger solver tiers): the float64 CUDA pipeline must follow the float64 oracle, same algorithm, to
  round-off amplified by the contact dynamics."""
  env = _env(built, precision='f64', num_envs=2)
  env.sample_prop_initial_states(seed=11, clearance=0.001, settle_steps=0)
  q0, v0 = env.get_state(torch.float64)
  acts = _actions(env, 25, seed=4, scale=0.3)
  o = OracleSim('so100_handover_banana', collide=True)
  o.set_state(q0[0].cpu().numpy(), v0[0].cpu().numpy())
  worst, ncon_max = 0.0, 0
  for t in range(25):
    ts = env.step(acts[t])
    r = o.control_step(acts[t, 0].double().cpu().numpy())
    q, v = env.get_state(torch.float64)
    worst = max(worst, np.abs(q[0].cpu().numpy() - o.qpos).max())
    ncon_max = max(ncon_max, int(env.debug_read('ncon')[0, 0]))
    assert float(ts.reward[0]) == r
  print('f64 contact-rich rollout: max |dqpos| =', worst, 'max contacts', ncon_max)
  # measured 1.5e-6 after 250 substeps of hard contacts (EPA terminates by tolerance on curved pairs: FMA-level differences
  # between nvcc and gcc are amplified by the contact dynamics); the bound is the one used for curved contacts above
  assert worst < 1e-4, worst
  assert env.counters()['diverged'] == 0
  env.close()


def test_step_host_returns_the_whole_timestep(built):
  """so101_step_host (the e2e path of bench.py): pinned host action in, EVERY block of the TimeStep out to pinned host tensors;
  identical to what step() leaves in the device tensors of a twin env."""
  a, b = _env(built, num_envs=4), _env(built, num_envs=4)
  for e in (a, b):
    e.sample_prop_initial_states(seed=7, settle_steps=0)
  acts = _actions(a, 6, seed=9)
  host = b.make_host_timestep()
  assert set(host) == {'commanded_joints_pos', 'joints_pos', 'undelayed_joints_pos', 'physics_state', 'delayed_physics_state', 'reward', 'discount', 'step_type'}
  for t in range(6):
    ts = a.step(acts[t])
    nbytes = b.step_host(acts[t].cpu().pin_memory(), host)
  assert nbytes == 4 * (3 * 24 + 2 * 152 + 9)
  for k in ('commanded_joints_pos', 'joints_pos', 'undelayed_joints_pos', 'physics_state', 'delayed_physics_state'):
    assert torch.equal(ts.observation[k].cpu(), host[k]), k
  assert torch.equal(ts.reward.cpu(), host['reward']) and torch.equal(ts.discount.cpu(), host['discount']) and torch.equal(ts.step_type.cpu(), host['step_type'])
  a.close(); b.close()


def test_episode_step_counters_roundtrip_and_time_limit(built):
  """so101_get/set_episode_steps: the per-env control-step counters that decide when `physics.time() >= time_limit` fires
  (1501 control steps for 30 s).  Setting env 1 to 1499 makes its next-but-one step LAST and the one after FIRST."""
  env = _env(built, num_envs=3)
  env.sample_prop_initial_states(seed=1, settle_steps=0)
  zero = torch.zeros(3, 6, device='cuda:0')
  env.step(zero)
  assert env.get_episode_steps().tolist() == [1, 1, 1]
  env.set_episode_steps(torch.tensor([1, 1499, 7]))
  kinds = [env.step(zero).step_type.tolist() for _ in range(3)]
  assert kinds == [[1, 1, 1], [1, 2, 1], [1, 0, 1]]
  assert env.get_episode_steps().tolist() == [4, 0, 10]
  env.close()


def _trace(env, acts):
  out = []
  for a in acts:
    ts = env.step(a)
    out.append([ts.step_type.clone(), ts.reward.clone(), ts.discount.clone()] + [v.clone() for _, v in sorted(ts.observation.items())])
  q, v = env.get_state(torch.float64)
  return out, q, v


def test_checkpoint_resume_is_bit_identical(built):
  """so101_checkpoint_save / _load: a rollout resumed from a checkpoint - in the same env after it has moved on, and in a second
  env created the same way - reproduces every TimeStep (delayed observations included) and the final state bit for bit.  The
  window crosses time-limit LAST steps and auto-resets from a two-round reset pool (0.3 s episodes = 16 control steps), so the
  warm starts, the delay buffers, the episode / pool counters and the auto-reset flags all have to come back."""
  from so101_sim_b200.task_suite import create_batched_task_env
  kw = dict(task_name='SO100HandOverBanana', num_envs=16, time_limit=0.3, seed=3, device='cuda:0', placement='pool', reset_rounds=2)
  env = create_batched_task_env(**kw)
  env.reset()
  acts = _actions(env, 45, seed=9)
  for t in range(11):
    env.step(acts[t])
  ck = env.save_checkpoint()
  assert ck.dtype == torch.uint8 and ck.numel() > 16 * (20 + 18) * 8
  ref, q_ref, v_ref = _trace(env, acts[11:])
  kinds = torch.stack([r[0] for r in ref])
  assert (kinds == 2).any() and (kinds == 0).any()         # the window holds LAST and FIRST steps
  env.load_checkpoint(ck)                                    # (1) rewind the same env
  again, q1, v1 = _trace(env, acts[11:])
  other = create_batched_task_env(**kw)                      # (2) a second env that never saw the first 11 steps
  other.load_checkpoint(ck)
  third, q2, v2 = _trace(other, acts[11:])
  for got, q, v in ((again, q1, v1), (third, q2, v2)):
    assert torch.equal(q, q_ref) and torch.equal(v, v_ref)
    for a, b in zip(ref, got):
      assert all(torch.equal(x, y) for x, y in zip(a, b))
  # a handle created differently refuses the checkpoint
  small = create_batched_task_env(**dict(kw, num_envs=8))
  with pytest.raises(RuntimeError, match='different model'):
    small.load_checkpoint(ck)
  with pytest.raises(RuntimeError, match='not a checkpoint'):
    env.load_checkpoint(torch.zeros(ck.numel(), dtype=torch.uint8, device='cuda:0'))
  for e in (env, other, small):
    e.close()


def test_checkpoint_carries_the_placement_machinery(built):
  """With nursery envs the checkpoint also holds the SETTLE-mode state of the hidden envs, the Philox draw counters and the ring
  of settled placements with its counters: after a load the placement statistics read as they did at the save, and the
  nursery continues from there."""
  from so101_sim_b200.task_suite import create_batched_task_env
  env = create_batched_task_env('SO100HandOverBanana', num_envs=16, time_limit=30.0, seed=5, device='cuda:0', placement='device', nursery_envs=16)
  env.reset()
  zero = torch.zeros(16, 6, device='cuda:0')
  for _ in range(40):
    env.step(zero)
  at_save = env.placement_stats()
  ck = env.save_checkpoint()
  for _ in range(60):
    env.step(zero)
  later = env.placement_stats()
  assert later['published'] > at_save['published']
  env.load_checkpoint(ck)
  assert env.placement_stats() == at_save
  for _ in range(60):
    env.step(zero)
  assert env.placement_stats()['published'] == later['published']   # the nursery's own trajectory is deterministic
  env.close()


@pytest.mark.parametrize('precision', ['f32', 'f64'])
def test_two_launch_narrow_phase_is_bit_identical(built, monkeypatch, precision):
  """Groups of 32768+ envs run the narrow phase as two launches (scene_epa_kernel: EPA as a per-lane state machine with pairs
  taken from a cursor; scene_manifold_kernel: manifold / plane contacts) instead of the fused thread-per-pair kernel.
  Forced on at 64 envs (SO101_NARROW_SPLIT = smallest group size that uses it), the states after 25 random-action control
  steps must equal the fused kernel's bit for bit, and the launch counter must show the extra launch."""
  results = []
  for split in ('1000000000', '1'):
    monkeypatch.setenv('SO101_NARROW_SPLIT', split)
    env = _env(built, num_envs=64, precision=precision)
    _initial(env, seed=11)
    acts = _actions(env, 25, seed=5)
    c0 = env.counters()['kernel_launches']
    for t in range(25):
      env.step(acts[t])
    launches = env.counters()['kernel_launches'] - c0
    q, v = env.get_state(torch.float64)
    results.append((q.clone(), v.clone(), launches, env.debug_read('ncon').flatten().clone()))
    env.close()
  assert results[0][2] == 25 * 83 and all(r[2] == 25 * 93 for r in results[1:])
  assert int(results[0][3].max()) >= 8     # the rollout has contacts
  for r in results[1:]:
    assert torch.equal(r[0], results[0][0]) and torch.equal(r[1], results[0][1]) and torch.equal(r[3], results[0][3])


def test_kernel_times_and_launch_counts(built, monkeypatch):
  """so101_kernel_times: CUDA-event time per kernel while enabled; one control step = 3 + 8 x 10 launches per group
  (begin, kinematics + dynamics, broad phase; then per substep GJK, EPA / manifold, classify, three solver tiers, kinematics + dynamics,
  broad phase or task layer)."""
  monkeypatch.delenv('SO101_NARROW_SPLIT', raising=False)
  env = _env(built, num_envs=8)
  env.sample_prop_initial_states(seed=2, settle_steps=0)
  c0 = env.counters()
  env.kernel_times(True)
  zero = torch.zeros(8, 6, device='cuda:0')
  for _ in range(3):
    env.step(zero)
  kt = env.kernel_times(False)
  c1 = env.counters()
  assert c1['kernel_launches'] - c0['kernel_launches'] == 3 * 83
  assert kt['scene_kindyn_kernel'][1] == 33 and kt['scene_broad_kernel'][1] == 33
  assert kt['scene_begin_kernel'][1] == 3 and kt['scene_gjk_kernel'][1] == 30 and kt['scene_narrow_kernel'][1] == 30
  assert kt['scene_solve_kernel'][1] == 30 and all(ms >= 0 for ms, _ in kt.values())
  assert kt['scene_solve_kernel'][0] > 0 and kt['arm_step_kernel'][1] == 0
  env.kernel_times(True); env.step(zero)
  assert env.kernel_times(False)['scene_begin_kernel'][1] == 4   # totals accumulate
  env.close()


# ------------------------------------------------------------------------------------------------ SO100HandOverPen (so100_hand_over.py:97-117)
def _pen_in_holder_state(env_or_meta, n):
  """Row 0: the pen standing inside the utensil holder (rotated so that its long axis, body y, points up); row 1..: pen lying on
  the table away from the holder."""
  q = torch.tensor(env_or_meta['qpos0'], dtype=torch.float32).repeat(n, 1)
  q[:, :6] = 0
  q[:, 13:16] = torch.tensor([-0.25, 0.05, 0.4503]); q[:, 16] = 1; q[:, 17:20] = 0
  q[:, 6:9] = torch.tensor([0.25, 0.0, 0.4283]); q[:, 9] = 1; q[:, 10:13] = 0
  q[0, 6:9] = torch.tensor([-0.25, 0.05, 0.4503 + 0.105])
  q[0, 9] = float(np.cos(np.pi / 4)); q[0, 10] = float(np.sin(np.pi / 4)); q[0, 11:13] = 0  # +90 degrees about x: y -> z
  return q


def test_pen_scene_matches_oracle_and_rewards(built):
  """SO100HandOverPen: same kernels, second model blob (pen x(1.5,1,1.5) + utensil holder x0.6, 52 hulls) and TWO overlap boxes
  that must both be touched (so100_hand_over.py:104-116,263-273).  float64 state parity over contact-rich steps, and the
  reward / discount / step_type flags equal the oracle's at every step."""
  env = _env(built, task_name='SO100HandOverPen', num_envs=3, precision='f64')
  assert env.task.get_instruction() == 'pick up the pen and put it in the container using the SO100 arm'
  q = _pen_in_holder_state(env.model, 3)
  q[2, 6:9] = torch.tensor([0.22, 0.03, 0.45])  # dropped from the reference's spawn height
  v = torch.zeros(3, 18)
  env.set_initial_state(q, v)
  env.reset()
  sims = []
  for e in range(3):
    o = OracleSim('so100_handover_pen', collide=True)
    o.set_state(q[e].double().numpy(), np.zeros(18))
    sims.append(o)
  acts = _actions(env, 30, seed=3, scale=0.1)
  seen_success = False
  for t in range(30):
    ts = env.step(acts[t])
    qg, vg = env.get_state(torch.float64)
    for e, o in enumerate(sims):
      if o is None:
        continue
      r = o.control_step(acts[t, e].double().cpu().numpy())
      assert float(ts.reward[e]) == r, (t, e)
      assert np.abs(o.qpos - qg[e].cpu().numpy()).max() < 1e-5, (t, e, np.abs(o.qpos - qg[e].cpu().numpy()).max())
      if r >= 1.0:
        assert e == 0 and float(ts.discount[e]) == 0.0 and int(ts.step_type[e]) == 2
        seen_success = True
        sims[e] = None  # the env auto-resets on the next step
  assert seen_success, 'the pen standing in the holder must trigger the two-box overlap reward once it is at rest'
  env.close()


def test_pen_f32_rollout_and_reset_pool(built):
  env = _env(built, task_name='SO100HandOverPen', num_envs=16)
  Q, V = env.randomize_resets(rounds=2, seed=3, settle_steps=60)
  assert torch.isfinite(Q).all() and float(V[..., 6:].abs().max()) < 0.1
  # both rest on the table top (z 0.42): the pen's body origin ends ~2 mm below it (the mesh is off-centre), the holder's base
  # sits at its origin; the rejection sampling keeps the holder off the static cylinder obstacle (scene_pbr.xml:144-146)
  assert float((Q[..., 8] - 0.4180).abs().max()) < 5e-3 and float((Q[..., 15] - 0.4204).abs().max()) < 2e-3
  acts = _actions(env, 20, seed=5)
  for t in range(20):
    ts = env.step(acts[t])
  assert torch.isfinite(ts.observation['physics_state']).all() and env.counters()['diverged'] == 0
  env.close()


def test_specs_match_the_reference_printouts(built):
  """action_spec bounds and observation keys / shapes as printed by the reference (examples/so101_rl_breakdown.ipynb:65,
  120-121,355-363 -> tests/golden/kat2_reset_observation.json): min/max = actuator ctrlrange with [0] -> +-pi and the gripper
  -> [0, 0.08] (so100_task.py:232-251); state dim 38; joints_vel empty."""
  import json, os
  kat2 = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'kat2_reset_observation.json')))
  env = _env(built, num_envs=2)
  spec = env.action_spec()
  assert spec.shape == (6,) and spec.dtype == np.float32
  assert np.round(spec.minimum.astype(np.float64), 2).tolist() == kat2['action_spec']['minimum']
  assert np.round(spec.maximum.astype(np.float64), 2).tolist() == kat2['action_spec']['maximum']
  assert abs(float(spec.maximum[0]) - np.pi) < 1e-6 and abs(float(spec.maximum[1]) - 3.14158) < 1e-6
  ts = env.reset()
  keys = [k for k in kat2['observation_keys'] if not k.endswith('_cam')]
  assert list(ts.observation.keys()) == keys == list(env.observation_spec().keys())
  for k, shp in env.observation_spec().items():
    assert tuple(ts.observation[k].shape[1:]) == tuple(shp), k
  assert env.observation_spec()['physics_state'] == (38,) and env.observation_spec()['joints_vel'] == (0,)
  # reset observation (KAT-2): commanded = HOME_CTRL (zero calibration), arm qpos = 0
  np.testing.assert_allclose(ts.observation['commanded_joints_pos'][0].cpu().numpy(), kat2['commanded_joints_pos'], atol=1e-5)
  assert float(ts.observation['joints_pos'].abs().max()) == 0.0
  env.close()
