"""CPU-only tests: host logic, C-ABI export surface, blob format."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_time_limit_step_matches_reference_accumulation():
  from so101_sim_b200.task_suite import time_limit_to_last_step
  # SURVEY.md §6: float64 accumulation of 0.002 reaches 30 only on substep 15010 -> control step 1501; 80 s -> 4001
  assert time_limit_to_last_step(30.0, 0.02) == 1501
  assert time_limit_to_last_step(80.0, 0.02) == 4001
  assert time_limit_to_last_step(float('inf'), 0.02) == 0


def test_library_exports_every_declared_symbol(built):
  """Every function declared in include/so101_b200.h must be exported by the in-tree .so (no compute calls here)."""
  from so101_sim_b200 import _lib
  hdr = open(os.path.join(ROOT, 'include', 'so101_b200.h')).read()
  declared = set(re.findall(r'\b(so101_[a-z0-9_]+)\s*\(', hdr))
  assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
  for path in (_lib.LIB_PATH, _lib.LIB_PATH_2ARM):   # one-arm build and the two-arm build of the same sources
    L = ctypes.CDLL(path)
    for sym in declared:
      assert hasattr(L, sym), (path, sym)
    assert L.so101_abi_version() == 4


def test_create_fails_loudly_without_gpu(built):
  import torch
  if torch.cuda.is_available():
    pytest.skip('GPU present')
  from so101_sim_b200.task_suite import create_batched_task_env
  with pytest.raises(RuntimeError, match='no CPU fallback'):
    create_batched_task_env('SO100ArmOnly', num_envs=4, time_limit=1.0)


def test_unknown_task_and_kwarg_filtering():
  from so101_sim_b200 import task_suite
  with pytest.raises(ValueError, match='Unknown task_name'):
    task_suite.create_batched_task_env('Nope', num_envs=1, time_limit=1.0)
  with pytest.raises(ValueError, match='Invalid object name'):
    task_suite.SO100HandOver(object_name='mug', control_timestep=0.02)


def test_calibration_mirror(tmp_path):
  from so101_sim_b200.calibration import SO101Calibration
  c = SO101Calibration()  # no file -> zero offsets (reference behaviour when the CWD-relative file is absent)
  np.testing.assert_array_equal(c.apply_calibration_to_action(np.arange(6.0)), np.arange(6.0))
  p = tmp_path / 'arm.json'
  p.write_text('{"shoulder_pan": {"homing_offset": 28}, "gripper": {"homing_offset": -158}}')
  c = SO101Calibration(str(p))
  np.testing.assert_array_equal(c.homing_offsets, [28, 0, 0, 0, 0, -158])
  with pytest.raises(ValueError):
    c.apply_calibration_to_position(np.zeros(5))


def test_blob_roundtrip_fields():
  from so101_sim_b200.model import read_blob
  arm = read_blob('so100_arm'); full = read_blob('so100_handover_banana')
  assert (arm['nq'][0], arm['nv'][0], arm['nu'][0]) == (6, 6, 6)
  assert (full['nq'][0], full['nv'][0], full['nu'][0]) == (20, 18, 6)  # SURVEY.md fact 3
  assert full['ngeom'][0] == 83                                         # 83 colliding geoms
  np.testing.assert_allclose(full['dof_armature'][:6], 0.1); np.testing.assert_allclose(full['dof_frictionloss'][:6], 0.1)
  np.testing.assert_allclose(full['act_ctrlrange'].reshape(-1, 2), [[-3.14158, 3.14158]] * 6)


def test_batched_env_config_mirrors_the_factory():
  """BatchedEnvConfig carries exactly the factory's keyword arguments (with the same defaults), round-trips through a dict /
  JSON and rejects what the factory would reject."""
  import inspect, json
  import dataclasses
  from so101_sim_b200.task_suite import BatchedEnvConfig, create_batched_task_env
  sig = inspect.signature(create_batched_task_env).parameters
  fields = {f.name: f for f in dataclasses.fields(BatchedEnvConfig)}
  assert set(fields) - {'task_kwargs'} == set(sig) - {'kwargs'}
  for name, f in fields.items():
    if name in ('task_kwargs', 'task_name', 'num_envs', 'time_limit'):
      continue
    assert f.default == sig[name].default, name
  c = BatchedEnvConfig(task_name='SO100HandOverPen', num_envs=64, precision='f64', calibration_offsets=[0, 1, 2, 3, 4, 5], cameras=[])
  again = BatchedEnvConfig.from_dict(json.loads(json.dumps(c.to_dict())))
  assert again == c and again.calibration_offsets == (0.0, 1.0, 2.0, 3.0, 4.0, 5.0) and again.cameras == ()
  for bad in (dict(task_name='NoSuchTask'), dict(num_envs=0), dict(precision='f16'), dict(placement='host'), dict(integrator='rk4')):
    with pytest.raises(ValueError):
      BatchedEnvConfig(**bad)
  with pytest.raises(ValueError, match='unknown config keys'):
    BatchedEnvConfig.from_dict({'envs': 3})


def test_bench_reference_arm_prints_the_contract_line():
  """`bench.py --impl reference` (the CPU arm: the float64 oracle on the host cores) prints one JSON line with the contract's keys,
  the same metric / config as the GPU arm, and an e2e block without copies."""
  import json, subprocess, sys
  root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
  r = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0', '--ref-seconds', '1'],
                     capture_output=True, text=True, timeout=300, cwd=root)
  assert r.returncode == 0, r.stderr[-800:]
  d = json.loads(r.stdout.strip().splitlines()[-1])
  assert d['impl'] == 'reference' and d['unit'] == 'env-steps/s' and d['higher_is_better'] is True and d['value'] > 0
  assert d['metric'].startswith('SO101 pick-place env-steps/sec') and d['config']['workload'] == 'banana131072'
  assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1 and d['cpu_baseline']['value'] == d['value']
  assert d['e2e'] == dict(value=d['value'], unit='env-steps/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0)
  assert d['vs_baseline'] is None and d['steps'] == 1 and d['warmup'] == 0


def test_bench_dump_outputs_writes_the_timestep(tmp_path):
  """bench.py --dump-outputs: every non-empty block of the TimeStep as float32 <name>.npy, one row per env; above the byte budget
  the same fixed sample of rows in every file, their env indices beside them, and the whole dump within the budget."""
  import torch
  import bench
  from so101_sim_b200.task_suite import OBSERVATION_KEYS, BatchedTimeStep
  N = 1000
  g = torch.Generator().manual_seed(0)
  obs = {k: torch.zeros(N, 0) if k.endswith('joints_vel') else torch.rand(N, 38 if 'physics' in k else 6, generator=g) for k in OBSERVATION_KEYS}
  ts = BatchedTimeStep(torch.randint(0, 3, (N,), dtype=torch.uint8, generator=g), torch.rand(N, generator=g), torch.ones(N), obs)
  src = dict(step_type=ts.step_type.float().numpy(), reward=ts.reward.numpy(), discount=ts.discount.numpy(),
             **{k: v.numpy() for k, v in obs.items() if v.numel()})
  names = bench.dump_outputs(str(tmp_path / 'full'), ts)
  assert names == sorted(k + '.npy' for k in src)
  for k, v in src.items():
    a = np.load(tmp_path / 'full' / f'{k}.npy')
    assert a.dtype == np.float32 and np.array_equal(a, v), k
  budget = 100_000
  for d in ('a', 'b'):
    names = bench.dump_outputs(str(tmp_path / d), ts, max_bytes=budget)
    assert names == sorted([k + '.npy' for k in src] + ['env_index.npy'])
    assert sum(os.path.getsize(tmp_path / d / n) for n in names) <= budget
  idx = np.load(tmp_path / 'a' / 'env_index.npy')
  assert idx.dtype == np.float64 and 200 < len(idx) < N and np.all(np.diff(idx) > 0)
  for k, v in src.items():
    a = np.load(tmp_path / 'a' / f'{k}.npy')
    assert np.array_equal(a, v[idx.astype(np.int64)]) and np.array_equal(a, np.load(tmp_path / 'b' / f'{k}.npy')), k


def test_bench_gpu_arm_refuses_to_run_without_a_gpu():
  """No CPU fallback: without a CUDA device the GPU arm stops with a message instead of measuring something else."""
  import subprocess, sys
  import torch
  if torch.cuda.is_available():
    pytest.skip('a GPU is present')
  root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
  r = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--steps', '1', '--warmup', '0'], capture_output=True, text=True, timeout=300, cwd=root)
  assert r.returncode != 0 and 'no CPU fallback' in (r.stderr + r.stdout)
