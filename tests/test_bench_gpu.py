"""bench.py's GPU arm at a small size: --dump-outputs writes the TimeStep of the last timed step, the same one run after run, and
it is the TimeStep of step warmup + steps of the benchmark's rollout (so --steps sets how many steps are timed)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = 'cuda:0'
ENVS, STEPS, WARMUP = 512, 3, 2


def _bench(out):
  r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--workload', 'banana16384', '--envs', str(ENVS), '--steps', str(STEPS),
                      '--warmup', str(WARMUP), '--no-secondary', '--no-steady', '--no-cpu-baseline', '--dump-outputs', str(out)],
                     capture_output=True, text=True, timeout=600, cwd=ROOT)
  assert r.returncode == 0, r.stderr[-2000:]
  d = json.loads(r.stdout.strip().splitlines()[-1])
  assert d['steps'] == STEPS and d['config']['envs_per_gpu'] == ENVS
  return {f[:-4]: np.load(os.path.join(out, f)) for f in sorted(os.listdir(out))}


def test_bench_dump_outputs_are_the_last_timed_step(built, tmp_path):
  import bench
  from so101_sim_b200.sharding import rank_seed
  from so101_sim_b200.task_suite import create_batched_task_env
  a, b = _bench(tmp_path / 'a'), _bench(tmp_path / 'b')
  assert sorted(a) == sorted(['step_type', 'reward', 'discount', 'commanded_joints_pos', 'joints_pos', 'physics_state',
                              'undelayed_joints_pos', 'delayed_physics_state'])
  for k in a:
    assert a[k].dtype == np.float32 and a[k].shape[0] == ENVS and np.isfinite(a[k]).all(), k
    assert np.array_equal(a[k], b[k]), f'{k} differs between two runs with the same arguments'
  # the same rollout outside bench.py: env and actions made as run_workload makes them, stepped warmup + steps times
  w = bench.WORKLOADS['banana16384']
  env = create_batched_task_env(w['task'], num_envs=ENVS, time_limit=30.0, seed=rank_seed(0, 0), device=DEV, placement='device', nursery_envs=0)
  env.reset()
  acts = bench._actions(env, WARMUP + STEPS, ENVS, torch.device(DEV), rank_seed(1, 0))
  for i in range(WARMUP + STEPS):
    ts = env.step(acts[i])
  # bitwise repetition holds for envs that keep all their contacts (see bench.dump_outputs)
  assert int(env.contacts_dropped_per_env().sum()) == 0
  got = dict(step_type=ts.step_type, reward=ts.reward, discount=ts.discount, **ts.observation)
  for k in a:
    assert np.array_equal(a[k], got[k].float().cpu().numpy()), k
  env.close()
