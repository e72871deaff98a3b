"""Per-env state of the arm-only model on the B200: what goes in through the C-ABI comes back out row for row, starts the
episodes it should, and survives a checkpoint.  Each env gets its own distinct state and the batch is not a multiple of 32,
so a mix-up of envs, components or strides shows."""
import struct

import pytest
import torch

from so101_sim_b200.task_suite import SO100_HOME_CTRL, create_batched_task_env

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
N = 37
PRECISIONS = ['f32', 'f64']


def _env(precision, **kw):
  args = dict(num_envs=N, time_limit=30.0, seed=0, device=DEV, precision=precision)
  args.update(kw)
  return create_batched_task_env('SO100ArmOnly', **args)


def _states(env, seed, dtype=torch.float64):
  """Distinct per-env states: joints inside half their ranges, velocities up to 0.5 rad/s."""
  g = torch.Generator(device='cpu'); g.manual_seed(seed)
  r = torch.tensor(env.model['jnt_range'].reshape(-1, 2)[:6], dtype=torch.float64)
  q = 0.5 * (r[:, 0] + torch.rand(N, 6, generator=g, dtype=torch.float64) * (r[:, 1] - r[:, 0]))
  v = 0.5 * (2 * torch.rand(N, 6, generator=g, dtype=torch.float64) - 1)
  return q.to(device=DEV, dtype=dtype), v.to(device=DEV, dtype=dtype)


def _actions(env, steps, seed):
  g = torch.Generator(device=DEV); g.manual_seed(seed)
  spec = env.action_spec()
  lo, hi = torch.tensor(spec.minimum, device=DEV), torch.tensor(spec.maximum, device=DEV)
  return (lo + torch.rand(steps, N, 6, generator=g, device=DEV) * (hi - lo)) * 0.3


def _assert_first(ts, q, v, envs=slice(None)):
  """The FIRST TimeStep of envs that start from state (q, v): every observation is that state, undelayed."""
  phys = torch.cat([q, v], 1).float()
  o = ts.observation
  assert (ts.step_type[envs] == 0).all() and (ts.reward[envs] == 0).all() and (ts.discount[envs] == 1).all()
  assert torch.equal(o['physics_state'][envs], phys[envs])
  assert torch.equal(o['delayed_physics_state'][envs], phys[envs])
  assert torch.equal(o['undelayed_joints_pos'][envs], q.float()[envs])
  assert torch.equal(o['joints_pos'][envs], q.float()[envs])
  home = torch.tensor(SO100_HOME_CTRL, dtype=torch.float32, device=DEV)
  assert torch.equal(o['commanded_joints_pos'][envs], home.expand(N, 6)[envs])


@pytest.mark.parametrize('precision', PRECISIONS)
def test_state_round_trip(built, precision):
  """set_initial_state (float32 rows) and set_state_f64 (float64 rows) store each env's row; get_state returns it exactly in
  float32 and float64, and reset() starts every env from it.  The commanded targets a step stores are read back per env by
  ee_pose('command')."""
  env = _env(precision)
  q32, v32 = _states(env, 1, torch.float32)
  env.set_initial_state(q32, v32)
  q, v = env.get_state(torch.float32)
  assert torch.equal(q, q32) and torch.equal(v, v32)
  q, v = env.get_state(torch.float64)
  assert torch.equal(q, q32.double()) and torch.equal(v, v32.double())
  _assert_first(env.reset(), q32.double(), v32.double())

  q64, v64 = _states(env, 2)
  env.set_initial_state(q64, v64)   # float64 tensors go through so101_set_state_f64
  q, v = env.get_state(torch.float64)
  assert torch.equal(q, q64) and torch.equal(v, v64)
  q, v = env.get_state(torch.float32)
  assert torch.equal(q, q64.float()) and torch.equal(v, v64.float())
  _assert_first(env.reset(), q64, v64)

  q32, v32 = _states(env, 3, torch.float32)
  env.set_state(q32, v32)           # the state only: the reset state stays (q64, v64)
  q, v = env.get_state(torch.float32)
  assert torch.equal(q, q32) and torch.equal(v, v32)
  _assert_first(env.reset(), q64, v64)

  ts = env.step(_actions(env, 1, seed=4)[0])
  ctrl = ts.observation['commanded_joints_pos'].double()   # action + zero offsets: exact in both precisions
  cpos, _ = env.ee_pose('command')
  env.set_state(ctrl, torch.zeros(N, 6, dtype=torch.float64, device=DEV))
  spos, _ = env.ee_pose('state')
  assert torch.equal(cpos, spos)
  env.close()


@pytest.mark.parametrize('precision', PRECISIONS)
def test_reset_pool_entry_follows_the_episode(built, precision):
  """With a two-round reset pool every FIRST TimeStep of env e shows pool entry (episode of e) % 2, through reset() and the
  auto-resets after the time limit."""
  env = _env(precision, time_limit=0.06)   # LAST on control step 3
  pool = [_states(env, 10 + r, torch.float32) for r in range(2)]
  env.set_reset_pool(torch.stack([p[0] for p in pool]), torch.stack([p[1] for p in pool]))
  episode = torch.zeros(N, dtype=torch.long, device=DEV)

  def check(ts):
    first = ts.step_type == 0
    for r in range(2):
      envs = first & (episode % 2 == r)
      _assert_first(ts, pool[r][0].double(), pool[r][1].double(), envs)
      q, v = env.get_state(torch.float32)
      assert torch.equal(q[envs], pool[r][0][envs]) and torch.equal(v[envs], pool[r][1][envs])
    episode.add_(first.long())
    return int(first.sum())

  assert check(env.reset()) == N
  firsts = 0
  for a in _actions(env, 14, seed=5):
    firsts += check(env.step(a))
  assert firsts >= 3 * N and int(episode.min()) >= 4
  env.close()


def _trace(env, acts):
  out = []
  for a in acts:
    ts = env.step(a)
    out.append([ts.step_type.clone(), ts.reward.clone(), ts.discount.clone()] + [x.clone() for x in ts.observation.values()])
  q, v = env.get_state(torch.float64)
  return out, q, v


@pytest.mark.parametrize('precision', PRECISIONS)
def test_checkpoint_resume_is_bit_identical(built, precision):
  """A rollout resumed from a checkpoint, in the same env after it has moved on and in a second env, reproduces every TimeStep
  and the final state bit for bit.  The checkpoint is taken 20 steps into a 25-step episode and the window runs through the
  auto-reset (two-round reset pool), so the delay rings (both hold values written before the save), the warm starts, the
  commanded targets, the episode counters and the auto-reset flags all have to come back.  A checkpoint that claims the
  previous library version is refused."""
  env = _env(precision, time_limit=0.5)
  pool = [_states(env, 20 + r, torch.float32) for r in range(2)]
  Q, V = torch.stack([p[0] for p in pool]), torch.stack([p[1] for p in pool])
  env.set_reset_pool(Q, V)
  env.reset()
  acts = _actions(env, 40, seed=6)
  for t in range(20):
    env.step(acts[t])
  ck = env.save_checkpoint()
  ref, q_ref, v_ref = _trace(env, acts[20:])
  kinds = torch.stack([r[0] for r in ref])
  assert (kinds == 2).any() and (kinds == 0).any()   # the window holds LAST and FIRST steps
  env.load_checkpoint(ck)
  again, q1, v1 = _trace(env, acts[20:])
  other = _env(precision, time_limit=0.5)
  other.set_reset_pool(torch.zeros_like(Q), torch.zeros_like(V))   # room for the checkpoint's two-round pool
  other.load_checkpoint(ck)
  third, q2, v2 = _trace(other, acts[20:])
  for got, q, v in ((again, q1, v1), (third, q2, v2)):
    assert torch.equal(q, q_ref) and torch.equal(v, v_ref)
    for a, b in zip(ref, got):
      assert all(torch.equal(x, y) for x, y in zip(a, b))
  old = ck.clone()
  old[4:8] = torch.tensor(list(struct.pack('<I', env._lib.so101_abi_version() - 1)), dtype=torch.uint8, device=DEV)   # header: magic, abi
  with pytest.raises(RuntimeError, match='not a checkpoint of this library version'):
    other.load_checkpoint(old)
  env.close()
  other.close()
