"""Cost of the contact force sensors (BatchedEnvironment.set_contact_sensors) on the control step.

For 131072 and 16384 envs of the hand-over banana scene (float32, the bench.py headline task, props dropped 2 mm onto the table,
random actions at 0.6 x the control range) it times windows of control steps with four sensors (gripper / object, object /
container, object / static, arm / static) and with none, alternated, `--repeats` windows each, with CUDA events.  Every window
starts from the same checkpoint (taken after 20 random-action steps) and replays the same actions, so that sensors on and off
time the same physics; two untimed steps before each window capture the step graph.  Then it times the copy of the [N, 4, 5]
readout to a caller buffer.  Writes one JSON (with the card's name and power limit read in the same run) to profiles/ or --out.

  python tools/bench_contact_sensors.py [--envs 131072,16384] [--steps 10] [--repeats 3] [--out profiles/contact_sensors_bench.json]
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from so101_sim_b200.model import body_set  # noqa: E402
from so101_sim_b200.task_suite import create_batched_task_env  # noqa: E402

DEV = 'cuda:0'


def card():
  q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'], capture_output=True, text=True)
  name, power = (x.strip() for x in q.stdout.strip().split(',')) if q.returncode == 0 else (torch.cuda.get_device_name(0), 'unknown')
  return name, power


def window_ms(env, acts, steps):
  for t in range(2):
    env.step(acts[t])
  torch.cuda.synchronize()
  s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  s.record()
  for t in range(steps):
    env.step(acts[2 + t])
  e.record()
  torch.cuda.synchronize()
  return s.elapsed_time(e) / steps


def run(n, steps, repeats):
  env = create_batched_task_env('SO100HandOverBanana', num_envs=n, time_limit=30.0, seed=0, device=DEV, placement='none')
  env.sample_prop_initial_states(seed=5, clearance=0.002, settle_steps=0)
  m = env.model
  sensors = [('gripper', 'object'), ('object', 'container'), ('object', 'static'), (body_set(m, 'arm'), 'static')]
  g = torch.Generator(device=DEV); g.manual_seed(1)
  spec = env.action_spec()
  lo, hi = torch.tensor(spec.minimum, device=DEV), torch.tensor(spec.maximum, device=DEV)
  for a in (lo + torch.rand(20, n, env.nu, generator=g, device=DEV) * (hi - lo)) * 0.6:
    env.step(a)
  ck = env.save_checkpoint()
  acts = (lo + torch.rand(steps + 2, n, env.nu, generator=g, device=DEV) * (hi - lo)) * 0.6
  on, off = [], []
  for _ in range(repeats):
    for k, dst in ((0, off), (1, on)):
      env.load_checkpoint(ck)
      env.set_contact_sensors(sensors if k else [])
      dst.append(window_ms(env, acts, steps))
  # readout copy into a preallocated buffer (so101_contact_sensors_read), sensors on
  env.set_contact_sensors(sensors)
  env.step(torch.zeros(n, env.nu, device=DEV))
  buf = torch.empty(n, len(sensors), 5, device=DEV)
  stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
  read = lambda: env._check(env._lib.so101_contact_sensors_read(env._h, ctypes.c_void_p(buf.data_ptr()), buf.numel(), stream))
  read()
  torch.cuda.synchronize()
  s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  s.record()
  for _ in range(50):
    read()
  e.record()
  torch.cuda.synchronize()
  readout = env.contact_sensors()
  rows_with_contacts = (readout[..., 4] > 0).float().mean(0).tolist()
  env.close()
  med_on, med_off = float(np.median(on)), float(np.median(off))
  return dict(envs=n, steps_per_window=steps, step_ms_sensors_off=off, step_ms_sensors_on=on, median_ms_off=med_off, median_ms_on=med_on,
              overhead_ms=med_on - med_off, overhead_rel=med_on / med_off - 1,
              spread_off_rel=(max(off) - min(off)) / med_off, spread_on_rel=(max(on) - min(on)) / med_on,
              readout_copy_ms=s.elapsed_time(e) / 50, readout_bytes=buf.numel() * 4, share_of_envs_with_contacts_per_sensor=rows_with_contacts)


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--envs', default='131072,16384')
  ap.add_argument('--steps', type=int, default=10)
  ap.add_argument('--repeats', type=int, default=3)
  ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'contact_sensors_bench.json'))
  a = ap.parse_args()
  if not torch.cuda.is_available():
    raise SystemExit('bench_contact_sensors.py needs a CUDA device')
  name, power = card()
  res = dict(gpu=name, power_limit=power, sensors=['gripper/object', 'object/container', 'object/static', 'arm/static'],
             runs=[run(int(n), a.steps, a.repeats) for n in a.envs.split(',')])
  os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
  with open(a.out, 'w') as f:
    json.dump(res, f, indent=1)
  print(json.dumps(res))


if __name__ == '__main__':
  main()
