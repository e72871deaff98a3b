"""Timing and accuracy of the end-effector layer (BatchedEnvironment.ee_pose / solve_ik) next to one control step.

For 4096 / 16384 / 131072 envs of the hand-over banana scene (float32, the bench.py headline task) it times, with CUDA events,
ee_pose, solve_ik with the default parameters and a position + orientation target, and one step; then it records the IK's
accuracy distribution on 4096 arm-only envs (targets from FK of random configurations inside 0.8 x the joint ranges, seeded
0.3 rad away).  Writes one JSON (with the card's name and power limit) to profiles/ or --out.

  python tools/bench_ee.py [--envs 4096,16384,131072] [--out profiles/ee_bench.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from so101_sim_b200.task_suite import IK_DEFAULTS, create_batched_task_env  # noqa: E402

DEV = 'cuda:0'


def timed(fn, reps):
  fn()
  torch.cuda.synchronize()
  s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  s.record()
  for _ in range(reps):
    fn()
  e.record()
  torch.cuda.synchronize()
  return s.elapsed_time(e) / reps


def card():
  q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'], capture_output=True, text=True)
  name, power = (x.strip() for x in q.stdout.strip().split(',')) if q.returncode == 0 else (torch.cuda.get_device_name(0), 'unknown')
  return name, power


def timing(n):
  env = create_batched_task_env('SO100HandOverBanana', num_envs=n, time_limit=30.0, seed=0, device=DEV, placement='none')
  env.sample_prop_initial_states(seed=5, clearance=0.002, settle_steps=0)
  pos, quat = env.ee_pose('state')
  target = pos + 0.02
  action = torch.zeros(n, env.nu, device=DEV)
  for _ in range(3):
    env.step(action)   # captures the step graph
  out = dict(envs=n, ee_pose_ms=timed(lambda: env.ee_pose('state'), 50),
             solve_ik_ms=timed(lambda: env.solve_ik(target, quat), 20),
             solve_ik_position_only_ms=timed(lambda: env.solve_ik(target), 20),
             step_ms=timed(lambda: env.step(action), 5))
  out['solve_ik_share_of_step'] = out['solve_ik_ms'] / out['step_ms']
  env.close()
  return out


def accuracy(n=4096, seed=5):
  env = create_batched_task_env('SO100ArmOnly', num_envs=n, time_limit=30.0, seed=0, device=DEV, placement='none', precision='f64')
  env.reset()
  rng = np.random.default_rng(seed)
  r = env.model['jnt_range'].reshape(-1, 2)[:6]
  qt = 0.5 * (r[:, 0] + r[:, 1]) + 0.4 * (r[:, 1] - r[:, 0]) * (2 * rng.random((n, 6)) - 1)
  env.set_state(torch.tensor(qt, device=DEV), torch.zeros(n, 6, dtype=torch.float64, device=DEV))
  tp, tq = env.ee_pose('state')
  d = rng.normal(size=(n, 5))
  q0 = qt.copy()
  q0[:, :5] += 0.3 * d / np.linalg.norm(d, axis=1, keepdims=True)
  seed_q = torch.tensor(q0, dtype=torch.float32, device=DEV)
  pct = lambda x: {f'p{p}': float(np.percentile(x, p)) for p in (50, 90, 99, 99.9, 100)}
  out = {}
  for name, quat in (('pose', tq), ('position', None)):
    _, err = env.solve_ik(tp, quat, seed=seed_q)
    e = err[:, 0].double().cpu().numpy()
    ok = (e[:, 0] < 1e-4) & ((e[:, 1] < 1e-3) if quat is not None else True)
    out[name] = dict(reached=float(ok.mean()), position_error_m=pct(e[:, 0]), orientation_error_rad=pct(e[:, 1]))
  env.close()
  return out


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--envs', default='4096,16384,131072')
  ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'ee_bench.json'))
  a = ap.parse_args()
  if not torch.cuda.is_available():
    raise SystemExit('bench_ee.py needs a CUDA device')
  name, power = card()
  res = dict(gpu=name, power_limit=power, ik_params=IK_DEFAULTS, timing=[timing(int(n)) for n in a.envs.split(',')], accuracy=accuracy())
  os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
  with open(a.out, 'w') as f:
    json.dump(res, f, indent=1)
  print(json.dumps(res))


if __name__ == '__main__':
  main()
