"""End-effector queries and batched IK on the B200 (so101_ee_pose / so101_ee_ik through BatchedEnvironment): TCP pose against the
float64 oracle, IK against its float64 NumPy restatement, convergence, no effect on the env's state, arm independence and a
closed loop in physics."""
import numpy as np
import pytest
import torch

from ee_reference import ArmFK, ik
from so101_sim_b200.task_suite import IK_DEFAULTS, create_batched_task_env, quat_from_rotvec, quat_mul

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
CONFIGS = [('SO100ArmOnly', 'so100_arm'), ('SO100HandOverBanana', 'so100_handover_banana'), ('SO100TwoArmHandOverBanana', 'so100_twoarm_banana')]
OFFSETS = np.array([0.01, -0.02, 0.015, 0.0, 0.03, -0.01])


def _env(task, precision, n, offsets=None):
  return create_batched_task_env(task, num_envs=n, time_limit=30.0, seed=0, device=DEV, precision=precision, placement='none',
                                 calibration_offsets=offsets)


def _random_arm_q(env, n, seed, frac=0.8):
  """[n, nq] float64 states: every arm's joints uniform in frac x its joint ranges (about the range centre), the rest at qpos0."""
  rng = np.random.default_rng(seed)
  r = env.model['jnt_range'].reshape(-1, 2)[:env.nu]
  q = np.tile(env.model['qpos0'], (n, 1))
  q[:, :env.nu] = 0.5 * (r[:, 0] + r[:, 1]) + 0.5 * frac * (r[:, 1] - r[:, 0]) * (2 * rng.random((n, env.nu)) - 1)
  return q


def _set(env, q):
  env.set_state(torch.tensor(q, dtype=torch.float64, device=DEV), torch.zeros(env.num_envs, env.nv, dtype=torch.float64, device=DEV))


@pytest.mark.parametrize('precision', ['f32', 'f64'])
@pytest.mark.parametrize('task,blob', CONFIGS)
def test_ee_pose_matches_the_oracle(built, task, blob, precision):
  n = 64
  env = _env(task, precision, n, OFFSETS)
  env.reset()
  q = _random_arm_q(env, n, seed=1)
  _set(env, q)
  pos, quat = env.ee_pose('state')
  cpos, cquat = env.ee_pose('command')
  pos, quat, cpos, cquat = (t.double().cpu().numpy() for t in (pos, quat, cpos, cquat))
  ctrl = (np.float32(np.array([0.0, -1.57079, 1.57079, 1.57079, -1.57079, 0.0])) + np.float32(OFFSETS)).astype(np.float64)
  off = env.tcp_offset.astype(np.float32).astype(np.float64)
  for arm in range(env.narm):
    fk = ArmFK(blob, arm)
    for e in range(n):
      p, R = fk.pose(q[e, 6 * arm:6 * arm + 6], off)
      assert np.abs(pos[e, arm] - p).max() <= 1e-6
      xq = fk.sim.field('xquat').reshape(-1, 4)[fk.body]
      xq = xq / np.linalg.norm(xq)
      assert min(np.abs(quat[e, arm] - xq).max(), np.abs(quat[e, arm] + xq).max()) <= 1e-6
    p, R = fk.pose(ctrl, off)   # after reset() the commanded targets are home + offsets in every env
    assert np.abs(cpos[:, arm] - p).max() <= 1e-6
  env.close()


@pytest.mark.parametrize('orient', [False, True])
@pytest.mark.parametrize('iterations', [1, 16])
@pytest.mark.parametrize('precision', ['f32', 'f64'])
@pytest.mark.parametrize('task,blob', CONFIGS)
def test_solve_ik_equals_the_float64_restatement(built, task, blob, precision, iterations, orient):
  n = 24
  env = _env(task, precision, n, OFFSETS)
  env.reset()
  qt = _random_arm_q(env, n, seed=2)
  _set(env, qt)
  tp, tq = env.ee_pose('state')
  rng = np.random.default_rng(3)
  q0 = qt[:, :env.nu].copy()
  for arm in range(env.narm):
    d = rng.normal(size=(n, 5))
    q0[:, 6 * arm:6 * arm + 5] += 0.3 * d / np.linalg.norm(d, axis=1, keepdims=True)
  use_seed = iterations == 16   # the other case starts from the env's state
  if use_seed:
    seed = torch.tensor(q0, dtype=torch.float32, device=DEV)
    q0 = q0.astype(np.float32).astype(np.float64)
  else:
    qs = qt.copy(); qs[:, :env.nu] = q0
    _set(env, qs)
  grip = torch.rand(n, env.narm, generator=torch.Generator().manual_seed(4)).to(DEV)
  prm = dict(IK_DEFAULTS, iterations=iterations)
  action, err = env.solve_ik(tp, tq if orient else None, grip, seed=seed if use_seed else None, **prm)
  a2, e2 = env.solve_ik(tp, tq if orient else None, grip, seed=seed if use_seed else None, **prm)
  assert torch.equal(action, a2) and torch.equal(err, e2)   # deterministic
  action, err = action.double().cpu().numpy(), err.double().cpu().numpy()
  tp, tq = tp.double().cpu().numpy(), tq.double().cpu().numpy()
  off = env.tcp_offset.astype(np.float32).astype(np.float64)
  f32 = lambda x: float(np.float32(x))
  ref_prm = dict(iterations=iterations, damping=f32(prm['damping']), w_rot=f32(prm['w_rot']), max_step=f32(prm['max_step']), tolerance=0.0)
  offs = np.float32(OFFSETS).astype(np.float64)
  worst = 0.0
  for arm in range(env.narm):
    fk = ArmFK(blob, arm)
    for e in range(n):
      q, pe, re, _ = ik(fk, q0[e, 6 * arm:6 * arm + 6], tp[e, arm], tq[e, arm] if orient else None, off, **ref_prm)
      worst = max(worst, np.abs(action[e, 6 * arm:6 * arm + 5] - (q[:5] - offs[:5])).max())
      assert abs(err[e, arm, 0] - pe) <= 1e-6 and abs(err[e, arm, 1] - re) <= 1e-5
    assert np.array_equal(action[:, 6 * arm + 5], grip[:, arm].double().cpu().numpy())
  assert worst <= 2e-6, worst
  env.close()


@pytest.mark.parametrize('precision', ['f32', 'f64'])
def test_solve_ik_converges_and_stays_in_range(built, precision):
  n = 4096
  env = _env('SO100ArmOnly', precision, n)
  env.reset()
  qt = _random_arm_q(env, n, seed=5)
  _set(env, qt)
  tp, tq = env.ee_pose('state')
  rng = np.random.default_rng(6)
  d = rng.normal(size=(n, 5))
  q0 = qt.copy()
  q0[:, :5] += 0.3 * d / np.linalg.norm(d, axis=1, keepdims=True)
  seed = torch.tensor(q0, dtype=torch.float32, device=DEV)
  _, err = env.solve_ik(tp, tq, seed=seed)
  ok = ((err[:, 0, 0] < 1e-4) & (err[:, 0, 1] < 1e-3)).float().mean().item()
  _, err_p = env.solve_ik(tp, seed=seed)
  ok_p = (err_p[:, 0, 0] < 1e-4).float().mean().item()
  print(f'\n{precision}: pose targets reached {ok:.4f}, position targets reached {ok_p:.4f}')
  assert ok >= 0.99 and ok_p >= 0.99
  # 2 m away: finite joint targets inside the joint ranges, the miss shows in the error
  far = tp + torch.tensor([2.0, 0.0, 0.0], device=DEV)
  for quat in (None, tq):
    action, err = env.solve_ik(far, quat, seed=seed)
    r = torch.tensor(env.model['jnt_range'].reshape(-1, 2)[:5], dtype=torch.float32, device=DEV)
    assert bool(torch.isfinite(action).all()) and bool(torch.isfinite(err).all())
    assert bool((action[:, :5] >= r[:, 0] - 1e-6).all()) and bool((action[:, :5] <= r[:, 1] + 1e-6).all())
    assert bool((err[:, 0, 0] > 1.0).all())
  env.close()


def _scene_or_arm(task, n):
  env = _env(task, 'f32', n)
  if env.task.collide:
    env.sample_prop_initial_states(seed=5, clearance=0.002, settle_steps=0)
  else:
    env.sample_arm_initial_states(seed=0)
    env.reset()
  return env


@pytest.mark.parametrize('task', ['SO100ArmOnly', 'SO100HandOverBanana'])
def test_ee_calls_leave_the_rollout_bit_identical(built, task):
  n, steps = 64, 25
  a, b = _scene_or_arm(task, n), _scene_or_arm(task, n)
  g = torch.Generator(device=DEV); g.manual_seed(7)
  acts = 0.2 * (2 * torch.rand(steps, n, 6, generator=g, device=DEV) - 1)
  c0a, c0b = a.counters(), b.counters()
  for t in range(steps):
    ta = a.step(acts[t])
    pos, quat = b.ee_pose('state')
    b.ee_pose('command')
    b.solve_ik(pos[:, :, :] + 0.01, quat, torch.zeros(n, 1, device=DEV))
    tb = b.step(acts[t])
    for k in ('physics_state', 'commanded_joints_pos', 'joints_pos', 'delayed_physics_state'):
      assert torch.equal(ta.observation[k], tb.observation[k]), (t, k)
    assert torch.equal(ta.reward, tb.reward) and torch.equal(ta.step_type, tb.step_type)
    b.solve_ik(pos, None, None)
  qa, va = a.get_state(torch.float64); qb, vb = b.get_state(torch.float64)
  assert torch.equal(qa, qb) and torch.equal(va, vb)
  ca, cb = a.counters(), b.counters()
  ga, gb = ca['graph_launches'] - c0a['graph_launches'], cb['graph_launches'] - c0b['graph_launches']
  assert ga == gb == (steps if a.task.collide else 0)
  assert ca['control_steps'] == cb['control_steps']
  a.close(); b.close()


@pytest.mark.parametrize('task', ['SO100ArmOnly', 'SO100HandOverBanana'])
def test_step_ee_equals_step_of_solve_ik(built, task):
  n = 64
  a, b = _scene_or_arm(task, n), _scene_or_arm(task, n)
  g = torch.Generator(device=DEV); g.manual_seed(8)
  ws = ((-0.3, -0.4, 0.45), (0.3, 0.0, 0.8))
  for t in range(6):
    dp = 0.02 * (2 * torch.rand(n, 1, 3, generator=g, device=DEV) - 1)
    dr = 0.05 * (2 * torch.rand(n, 1, 3, generator=g, device=DEV) - 1) if t % 2 else None
    grip = torch.rand(n, 1, generator=g, device=DEV) * 0.08
    base = 'command' if t >= 3 else 'state'
    ta = a.step_ee(dp, grip, dr, base=base, workspace=ws)
    pos, quat = b.ee_pose(base)
    target = torch.minimum(torch.maximum(pos + dp, torch.tensor(ws[0], device=DEV)), torch.tensor(ws[1], device=DEV))
    tq = None if dr is None else quat_mul(quat_from_rotvec(dr), quat.double()).float()
    action, err = b.solve_ik(target, tq, grip)
    tb = b.step(action)
    assert torch.equal(ta.observation['physics_state'], tb.observation['physics_state']), t
    assert torch.equal(a.last_ee_error, err)
  a.close(); b.close()


def test_arms_are_solved_independently(built):
  n = 32
  env = _env('SO100TwoArmHandOverBanana', 'f32', n)
  env.reset()
  _set(env, _random_arm_q(env, n, seed=9, frac=0.5))
  tp, tq = env.ee_pose('state')
  target = tp + 0.03
  a1, e1 = env.solve_ik(target, tq)
  t2 = target.clone(); t2[:, 1] += torch.tensor([0.05, -0.04, 0.02], device=DEV)
  a2, e2 = env.solve_ik(t2, tq)
  assert torch.equal(a1[:, :6], a2[:, :6]) and torch.equal(e1[:, 0], e2[:, 0])
  assert not torch.equal(a1[:, 6:], a2[:, 6:])
  env.close()


def test_step_ee_closed_loop_follows_the_oracle(built):
  """step_ee in a closed loop through five targets 10 cm apart (arm-only, float64): the device run equals the float64 oracle's
  physics driven by the NumPy IK restatement over the first target.  The TCP errors per target are printed, not bounded: the
  reference's actuators (gain 50, bias -50 q + 1 qvel, no joint damping) make the arm oscillate with growing amplitude under
  any changing command, so the error after 25 steps is set by the arm model, not by the IK (DESIGN.md section 7b)."""
  from oracle.oracle import OracleSim
  n = 2
  env = _env('SO100ArmOnly', 'f64', n)
  home = np.array([0.0, -1.57079, 1.57079, 1.57079, -1.57079, 0.0])
  env.set_initial_state(torch.tensor(home, dtype=torch.float32, device=DEV).repeat(n, 1), torch.zeros(n, 6, device=DEV))
  env.reset()
  p0 = env.ee_pose('state')[0]
  path = [(0, -0.1, 0), (0, -0.1, 0.1), (0.1, -0.1, 0.1), (0.1, 0, 0.1), (0.1, 0, 0)]
  errs, first = [], []
  for d in path:
    target = p0 + torch.tensor(d, dtype=torch.float32, device=DEV)
    for _ in range(25):
      pos = env.ee_pose('state')[0]
      env.step_ee(target - pos, torch.zeros(n, 1, device=DEV))
      if d == path[0]:
        first.append((env.ee_pose('state')[0] - target).norm(dim=-1)[0].item())
    assert bool(torch.isfinite(env.last_ee_error).all())
    errs.append((env.ee_pose('state')[0] - target).norm(dim=-1).max().item())
  assert env.counters()['diverged'] == 0
  print('\nclosed-loop TCP error per target after 25 control steps (m):', ' '.join(f'{e:.4f}' for e in errs))
  fk = ArmFK('so100_arm')
  off = env.tcp_offset.astype(np.float32).astype(np.float64)
  f32 = lambda x: float(np.float32(x))
  prm = dict(iterations=IK_DEFAULTS['iterations'], damping=f32(IK_DEFAULTS['damping']), w_rot=0.0, max_step=f32(IK_DEFAULTS['max_step']))
  sim = OracleSim('so100_arm', collide=False)
  sim.set_state(np.float32(home).astype(np.float64), np.zeros(6))
  t0 = p0[0, 0].double().cpu().numpy() + np.float32(path[0])
  for k in range(25):
    q, _, _, _ = ik(fk, sim.qpos.copy(), t0, None, off, **prm)
    q[5] = 0.0
    sim.control_step(q.astype(np.float32).astype(np.float64))
    p, _ = fk.pose(sim.qpos.copy(), off)
    assert abs(np.linalg.norm(p - t0) - first[k]) < 1e-4, (k, np.linalg.norm(p - t0), first[k])
  env.close()


def test_lerobot_ee_delta_wrapper(built):
  from so101_sim_b200.lerobot import BatchedSO101LeRobotWrapper
  n = 8
  w = BatchedSO101LeRobotWrapper('SO100ArmOnly', num_envs=n, device=DEV, seed=0, action_space='ee_delta',
                                 ee_workspace=((-0.4, -0.5, 0.3), (0.4, 0.0, 0.9)))
  first = w.reset()
  assert first['action'].shape == (n, 4)
  p0, _ = w.env.ee_pose('command')
  act = torch.tensor([0.0, -0.02, 0.01, 0.05], device=DEV)
  rec = w.step(act)
  assert rec['action'].shape == (n, 4) and torch.equal(rec['action'], act.expand(n, 4))
  assert rec['observation.state'].shape == (n, 6)
  assert w.get_action_spec()['shape'] == (4,)
  # the commanded TCP moved by the delta from where the state's TCP was (reset state: qpos0), inside the workspace
  cmd = w.env.ee_pose('command')[0]
  assert bool((cmd[:, 0, 2] <= 0.9 + 1e-4).all())
  with pytest.raises(ValueError):
    w.step(torch.zeros(n, 6, device=DEV))
  w.env.close()
