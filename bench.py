#!/usr/bin/env python3
"""Benchmark of the so101 lockstep env-step path.  Contract: one JSON line on stdout (rank 0).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference --steps K --warmup W     # CPU arm: the float64 oracle on the host cores

A "step" is one control step (0.02 s = 10 physics substeps + observations + reward/termination) of ALL lockstep envs.
Workloads (BASELINE.md §3):
  banana131072 config 5 at its single-GPU point: SO100HandOverBanana pick-and-place with contacts, 131072 lockstep envs per GPU
               (DEFAULT: the metric is "pick-place env-steps/sec at 1/2/4/8 B200" and config 5 is its sweep - 131072 envs on 1 GPU
               is the largest single-GPU pick-place configuration in BASELINE.json; with N GPUs every rank keeps 131072 envs,
               weak scaling, no per-step collective).  The pipeline's kernels are bound by their slowest warps at small batches
               (a step of 16384 envs takes as long as one of 32768), so throughput per GPU grows with the batch: 16384 envs
               ~0.44 M, 32768 ~0.87 M, 131072 ~0.84-1.0 M env-steps/s (profiles/).
  banana16384  config 3: the same scene with 16384 envs per GPU (attached as `other_workloads`)
  arm4096      config 2: arm-only, collisions off, 4096 envs per GPU (also measured and attached as `other_workloads`)
  handover8192 config 4: two-arm hand-over, 8192 envs per GPU, on a LABELLED SYNTHETIC two-SO100 scene (the reference has none);
               also attached as `other_workloads`
value  = env-steps/s with inputs resident in HBM (CUDA events around each step, L2 flushed between steps).
e2e    = env-steps/s through BatchedEnvironment.step_host(): pinned host action in, the WHOLE TimeStep (observation dict, reward,
         discount, step_type) out to pinned host tensors, copies and the stream sync inside the timed region.
steady_state = the same workload with episodes cycling through auto-reset (short episodes, staggered phases, reset pool).
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# stdout carries exactly one JSON line: NCCL's own banner / debug lines ("NCCL version ...") go to stderr
os.environ.setdefault('NCCL_DEBUG_FILE', '/dev/stderr')

WORKLOADS = {
    # name: (task, envs per GPU, blob, collide, algorithmic bytes per env-step [SURVEY.md §8d])
    'arm4096': dict(task='SO100ArmOnly', envs=4096, model='so100_arm', collide=False, bytes_per_env_step=177,
                    desc='BASELINE config 2: SO100 arm-only, collisions off, 4096 lockstep envs per GPU'),
    'banana16384': dict(task='SO100HandOverBanana', envs=16384, model='so100_handover_banana', collide=True, bytes_per_env_step=385,
                        desc='BASELINE config 3: SO100HandOverBanana with contacts, 16384 lockstep envs per GPU'),
    'banana131072': dict(task='SO100HandOverBanana', envs=131072, model='so100_handover_banana', collide=True, bytes_per_env_step=385,
                         desc='BASELINE config 5 at its single-GPU point: SO100HandOverBanana with contacts, 131072 lockstep envs per GPU '
                              '(every rank keeps 131072 envs when N > 1)'),
    # config 4: read qpos 26 + qvel 24 + action 12 words, write qpos + qvel, joints_pos + commanded_joints_pos 24 words, 9 B of flags
    'handover8192': dict(task='SO100TwoArmHandOverBanana', envs=8192, model='so100_twoarm_banana', collide=True, bytes_per_env_step=553,
                         desc='BASELINE config 4 (hand-over, two arms, 8192 envs per GPU) on a LABELLED SYNTHETIC scene: the reference has no '
                              'two-SO100 scene, this is scene_pbr.xml with two SO100 arms + the banana / bowl props'),
}
METRIC = 'SO101 pick-place env-steps/sec at 1/2/4/8 B200 vs MuJoCo CPU on host cores'
# the float32 product path keeps the integration state, the actuator model and the Euler update in float64
# (so101_sim_b200/csrc/env_state.cuh); dynamics, collision and the constraint solver run in float32
PRECISION_NOTE = {'f32': 'f32 dynamics / collision / solver, f64 integration state + actuator model + Euler update', 'f64': 'f64'}


def measured_peak_gbs():
  p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(p):
    return float(json.load(open(p))['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
  return 6650.0, 'fallback (B200_PROFILING.md)'


# ------------------------------------------------------------------------------------------------ CPU arm (oracle)
def _cpu_worker(args):
  model, collide, seconds, seed = args
  from oracle.oracle import OracleSim
  sim = OracleSim(model, collide=collide)
  rs = np.random.RandomState(seed)
  na = sim.nu   # arm dofs = actuators (6 per arm); the props' free joints follow
  lo = np.tile([-np.pi, -3.14158, -3.14158, -3.14158, -3.14158, 0.0], na // 6); hi = np.tile([np.pi, 3.14158, 3.14158, 3.14158, 3.14158, 0.08], na // 6)
  rng = sim.meta['jnt_range'].reshape(-1, 2)[:6]
  q = sim.meta['qpos0'].copy()
  if sim.nq == 6:    # config 2: arm qpos ~ U(1/4 joint range)
    q[:6] = 0.25 * rs.uniform(rng[:, 0], rng[:, 1])
    sim.set_state(q, np.zeros(sim.nv))
  else:              # configs 3 / 4: props at the reference drop height (so100_hand_over.py:37-55), settled 1 s (untimed), arms at qpos 0
    u = rs.uniform(size=5)
    while np.hypot(-0.3 + 0.1 * u[3] + 0.1778, -0.1 + 0.2 * u[4] - 0.1656) < 0.151:   # bowl vs static cylinder (see task_suite._bowl_obstacles)
      u[3:5] = rs.uniform(size=2)
    yaw = (2 * u[2] - 1) * 0.1 * np.pi
    q[:na] = 0
    q[na:na + 7] = [0.2 + 0.1 * u[0], -0.1 + 0.2 * u[1], 0.45, np.cos(yaw / 2), 0, 0, np.sin(yaw / 2)]
    q[na + 7:na + 14] = [-0.3 + 0.1 * u[3], -0.1 + 0.2 * u[4], 0.45, 1, 0, 0, 0]
    sim.set_state(q, np.zeros(sim.nv))
    for _ in range(50):
      sim.control_step(np.zeros(na))
    qs, vs = sim.qpos.copy(), sim.qvel.copy()
    qs[:na] = 0; vs[:na] = 0
    sim.set_state(qs, vs)
  acts = rs.uniform(lo, hi, size=(256, na)) * 0.3
  n, t0 = 0, time.perf_counter()
  while time.perf_counter() - t0 < seconds:
    sim.control_step(acts[n % 256])
    n += 1
  return n, time.perf_counter() - t0


def cpu_baseline(workload, seconds, procs):
  """Times the float64 C oracle (a restatement — `kind: port`; the reference's MuJoCo loop cannot run here: mujoco and
  dm_control are not installed and there is no network)."""
  from oracle import oracle as _o
  _o.build()
  w = WORKLOADS[workload]
  ctx = mp.get_context('fork')
  with ctx.Pool(procs) as pool:
    res = pool.map(_cpu_worker, [(w['model'], w['collide'], seconds, 100 + i) for i in range(procs)])
  total = sum(n / dt for n, dt in res)
  return dict(value=total, unit='env-steps/s', cores=procs, kind='port',
              sample=f'{procs} process(es) x 1 env x {seconds:.0f} s of {w["task"]} control steps on the float64 C oracle '
                     f'({sum(n for n, _ in res)} env-steps)')


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
  def __init__(self, index):
    self.index, self.rows, self._stop = index, [], threading.Event()
    self._t = threading.Thread(target=self._run, daemon=True)

  def _run(self):
    q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
    while not self._stop.is_set():
      try:
        out = subprocess.run(['nvidia-smi', f'--query-gpu={q}', '--format=csv,noheader,nounits', '-i', str(self.index)],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        if out:
          self.rows.append([x.strip() for x in out.split(',')])
      except Exception:
        pass
      self._stop.wait(0.2)

  def __enter__(self):
    self._t.start(); return self

  def __exit__(self, *a):
    self._stop.set(); self._t.join(timeout=6)

  def summary(self):
    if not self.rows:
      return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
    sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
    names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
    reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith('active') for r in self.rows if len(r) > 2 + i)]
    return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=int(self.rows[0][1]) if self.rows[0][1].isdigit() else None,
                reasons=reasons, samples=len(self.rows))


# ------------------------------------------------------------------------------------------------ main
def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=100)
  ap.add_argument('--warmup', type=int, default=10)
  ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
  ap.add_argument('--workload', default=os.environ.get('SO101_BENCH_WORKLOAD', 'banana131072'), choices=list(WORKLOADS))
  ap.add_argument('--envs', type=int, default=0, help='envs per GPU (default: the workload size)')
  ap.add_argument('--precision', default='f32', choices=['f32', 'f64'])
  ap.add_argument('--cpu-seconds', type=float, default=10.0)
  ap.add_argument('--profiler-range', action='store_true', help='bracket the timed steps with cudaProfilerStart/Stop (for `ncu --profile-from-start off`; numbers printed under a profiler are not bench values)')
  ap.add_argument('--ref-seconds', type=float, default=0.0, help='--impl reference: seconds of CPU work per step (default: 120 s spread over the steps, 1..20 s each)')
  ap.add_argument('--no-cpu-baseline', action='store_true')
  ap.add_argument('--no-secondary', action='store_true', help='skip the attached arm4096 measurement')
  ap.add_argument('--no-steady', action='store_true', help='skip the attached steady-state (cycling episodes) measurement')
  ap.add_argument('--steady-steps', type=int, default=200)
  ap.add_argument('--steady-warmup', type=int, default=100)
  ap.add_argument('--dump-outputs', metavar='DIR', help='write the TimeStep of the last timed step of the headline workload (rank 0) '
                                                        'to DIR/<name>.npy, float32; see dump_outputs()')
  a = ap.parse_args()
  global PROFILER_RANGE
  PROFILER_RANGE = bool(a.profiler_range)
  rank, world = int(os.environ.get('RANK', 0)), int(os.environ.get('WORLD_SIZE', 1))
  local_rank = int(os.environ.get('LOCAL_RANK', 0))
  w = WORKLOADS[a.workload]
  envs = a.envs or w['envs']
  config = dict(workload=a.workload, description=w['desc'], envs_per_gpu=envs, substeps_per_step=10, precision=PRECISION_NOTE[a.precision],
                parallelism=f'env-sharded x{world} (no per-step collective)',
                l2='256 MiB memset between timed steps, excluded from the timing by per-step CUDA events')

  if a.impl == 'reference':
    if rank != 0:
      return 0
    procs = os.cpu_count() or 1
    per_step_s = a.ref_seconds if a.ref_seconds > 0 else max(1.0, min(20.0, 120.0 / max(1, a.steps + a.warmup)))
    vals = []
    for i in range(a.warmup + a.steps):
      r = cpu_baseline(a.workload, per_step_s, procs)
      if i >= a.warmup:
        vals.append(r['value'])
    v = float(np.mean(vals)) if vals else r['value']
    r['value'] = v
    print(json.dumps(dict(metric=METRIC, value=v, unit='env-steps/s', impl='reference', n_gpus=a.gpus, steps=a.steps, warmup=a.warmup,
                          ms_per_step=per_step_s * 1e3, higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f64',
                          data='synthetic', config=config, cpu_baseline=r,
                          e2e=dict(value=v, unit='env-steps/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                          note='reference MuJoCo/dm_control loop cannot run here (packages absent, offline); this is the float64 C '
                               'restatement (oracle/) on all host cores'
                          )))
    return 0

  import torch
  import torch.distributed as dist
  if not torch.cuda.is_available():
    raise SystemExit('bench.py: no CUDA device (this framework has no CPU fallback; use --impl reference for the CPU arm)')
  torch.cuda.set_device(local_rank)
  dev = torch.device('cuda', local_rank)
  if world > 1:
    dist.init_process_group('nccl', device_id=dev)
  res = run_workload(a.workload, envs, a.steps, a.warmup, a.precision, dev, rank, world, local_rank, dump_dir=a.dump_outputs)
  if rank == 0:
    out = dict(metric=METRIC, value=res['value'], unit='env-steps/s', n_gpus=world, steps=a.steps, warmup=a.warmup,
               ms_per_step=res['ms_per_step'], higher_is_better=True, scaling='weak', vs_baseline=None,
               dtype=a.precision, data='synthetic', config=config, e2e=res['e2e'], gpu_launches=res['gpu_launches'],
               graph_launches=res['graph_launches'], launches_per_step=res['launches_per_step'], clocks=res['clocks'], roofline=res['roofline'], kernels=res['kernels'], wall_s=res['wall_s'],
               mean_return=res['mean_return'], diverged=res['diverged'], contacts_dropped=res['contacts_dropped'],
               dropped_by_buffer_since_load=res['dropped_by_buffer_since_load'])
    if world == 1 and not a.no_secondary and a.workload != 'arm4096':
      # the other BASELINE configs measured beside the headline workload (short runs, kernel-only and e2e):
      # config 2 (arm-only, 4096 envs), config 3 (pick-place, 16384 envs), config 4 (two-arm hand-over, 8192 envs, synthetic scene)
      r2 = run_workload('arm4096', WORKLOADS['arm4096']['envs'], 50, 5, a.precision, dev, rank, world, local_rank)
      out['other_workloads'] = {'arm4096': {k: r2[k] for k in ('value', 'ms_per_step', 'e2e', 'gpu_launches', 'roofline')}}
      if a.workload != 'banana16384':
        r3 = run_workload('banana16384', WORKLOADS['banana16384']['envs'], 100, 10, a.precision, dev, rank, world, local_rank)
        out['other_workloads']['banana16384'] = dict({k: r3[k] for k in ('value', 'ms_per_step', 'e2e', 'gpu_launches', 'roofline', 'diverged', 'contacts_dropped')},
                                                     description=WORKLOADS['banana16384']['desc'])
      # BASELINE config 4 on the labelled synthetic two-arm scene: a short run as well
      r4 = run_workload('handover8192', WORKLOADS['handover8192']['envs'], 30, 10, a.precision, dev, rank, world, local_rank)
      out['other_workloads']['handover8192'] = dict({k: r4[k] for k in ('value', 'ms_per_step', 'e2e', 'gpu_launches', 'roofline', 'diverged', 'contacts_dropped', 'dropped_by_buffer_since_load')},
                                                    description=WORKLOADS['handover8192']['desc'])
    if world == 1 and not a.no_steady and WORKLOADS[a.workload]['collide']:
      out['steady_state'] = run_steady_state(a.workload, envs, a.steady_steps, a.steady_warmup, a.precision, dev, rank)
    if not a.no_cpu_baseline and world == 1:
      out['cpu_baseline'] = cpu_baseline(a.workload, a.cpu_seconds, os.cpu_count() or 1)
    print(json.dumps(out))
  if world > 1:
    dist.destroy_process_group()
  return 0


def ncu_traffic(workload, envs, kernel):
  """DRAM bytes per launch of `kernel` from the committed `ncu --set full` capture (profiles/traffic.json), or None."""
  p = os.path.join(ROOT, 'profiles', 'traffic.json')
  if not os.path.exists(p):
    return None, None
  t = json.load(open(p)).get(f'{workload}:{envs}', {}).get(kernel)
  return (t['dram_bytes_per_launch'], t['source']) if t else (None, None)


def _actions(env, n, envs, dev, seed):
  import torch
  g = torch.Generator(device=dev); g.manual_seed(seed)
  spec = env.action_spec()
  lo, hi = torch.tensor(spec.minimum, device=dev), torch.tensor(spec.maximum, device=dev)
  return (lo + torch.rand(n, envs, len(spec.minimum), generator=g, device=dev) * (hi - lo)) * 0.3


PROFILER_RANGE = False   # set by --profiler-range
DUMP_MAX_BYTES = 64 * 10**6   # --dump-outputs: .npy headers included


def dump_outputs(out_dir, ts, max_bytes=DUMP_MAX_BYTES):
  """Writes what a caller of env.step() receives - step_type, reward, discount and every non-empty observation - as
  out_dir/<name>.npy in float32, one row per env.  If that exceeds `max_bytes`, a fixed sample of envs (seed 0, sorted, the
  same rows in every file) is written instead, with its env indices in env_index.npy (float64).  Returns the file names.
  With the same arguments the rows repeat bit for bit from run to run, except those of envs that lost contacts to a full per-env
  buffer (BatchedEnvironment.contacts_dropped_per_env): which contacts such an env keeps depends on the order they arrive in."""
  arrays = dict(step_type=ts.step_type, reward=ts.reward, discount=ts.discount, **{k: v for k, v in ts.observation.items() if v.numel()})
  arrays = {k: v.float().cpu().numpy() for k, v in arrays.items()}
  n = len(arrays['reward'])
  header = 128   # bytes of one .npy header for these shapes
  if sum(a.nbytes + header for a in arrays.values()) > max_bytes:
    per_env = sum(a[0].nbytes for a in arrays.values()) + 8
    k = (max_bytes - header * (len(arrays) + 1)) // per_env
    idx = np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))
    arrays = {name: a[idx] for name, a in arrays.items()}
    arrays['env_index'] = idx.astype(np.float64)
  os.makedirs(out_dir, exist_ok=True)
  for name, a in arrays.items():
    np.save(os.path.join(out_dir, name + '.npy'), a)
  return sorted(name + '.npy' for name in arrays)


def run_workload(name, envs, steps, warmup, precision, dev, rank, world, local_rank, dump_dir=None):
  import torch
  import torch.distributed as dist
  from so101_sim_b200.sharding import EpisodeStats, gather_episode_stats, rank_seed
  from so101_sim_b200.task_suite import create_batched_task_env
  w = WORKLOADS[name]
  # config 3: the props are sampled from so100_hand_over.py:37-55 and settled with the arm frozen ON THE DEVICE at creation
  # (initialize_placements).  No episode ends inside this leg's window (30 s episodes), so it runs without nursery envs; the
  # steady-state leg below has them.
  env = create_batched_task_env(w['task'], num_envs=envs, time_limit=30.0, seed=rank_seed(0, rank), device=dev, precision=precision,
                                placement='device', nursery_envs=0)
  if w['task'] == 'SO100ArmOnly':
    env.sample_arm_initial_states(seed=rank_seed(0, rank))
  env.reset()
  total = warmup + steps
  nact = min(total, 64)
  acts = _actions(env, nact, envs, dev, rank_seed(1, rank))
  flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
  ev0 = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
  ev1 = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
  stats = EpisodeStats(envs, dev)
  ret_sum = torch.zeros(envs, device=dev)

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  def max_over_ranks(x):
    t = torch.tensor([x], dtype=torch.float64, device=dev)
    if world > 1:
      dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())

  # ---- value: inputs resident in HBM, one step = one so101_step call (a CUDA-graph replay of the step's kernels); the
  # per-kernel event timers are OFF here (they need eager launches and ~330 event records per step)
  env.kernel_times(False)
  for i in range(warmup):
    env.step(acts[i % nact])
  c0 = env.counters()
  barrier()
  if PROFILER_RANGE:   # `ncu --profile-from-start off ... bench.py --profiler-range`: capture the timed steps only
    torch.cuda.profiler.start()
  with ClockSampler(local_rank) as clocks:
    t_wall0 = time.perf_counter()
    for i in range(steps):
      flush.fill_(i & 0xFF)
      ev0[i].record()
      ts = env.step(acts[(warmup + i) % nact])
      ev1[i].record()
      stats.update(ts.step_type, ts.reward); ret_sum += ts.reward
    barrier()
    t_wall = time.perf_counter() - t_wall0
  if PROFILER_RANGE:
    torch.cuda.synchronize(); torch.cuda.profiler.stop()
  if dump_dir and rank == 0:   # before the passes below step the env again and overwrite the TimeStep's buffers
    dump_outputs(dump_dir, ts)
  c1 = env.counters()
  drop_names = ('per_pair', 'candidates', 'pairs', 'queue', 'raw_contacts', 'jacobian_blocks', 'hits')
  drops = dict(zip(drop_names, [int(x) for x in env.debug_read('dropcat', 8)[0, :7].tolist()])) if w['collide'] and envs >= 8 else {}
  dev_ms = max_over_ranks(float(sum(ev0[i].elapsed_time(ev1[i]) for i in range(steps))))
  value = envs * world * steps / (dev_ms * 1e-3)

  # ---- per-kernel pass (separate from the timed region above): the rollout simply continues for a few steps with CUDA events
  # around every launch (eager launches, all on one stream while the timers are on: each launch is timed alone, as under ncu)
  ksteps = max(2, min(steps, 10))
  k0 = env.kernel_times(True)
  for i in range(ksteps):
    env.step(acts[(total + i) % nact])
  torch.cuda.synchronize()
  k1 = env.kernel_times(False)

  # ---- e2e: host buffers through the public API (H2D of the action + step + D2H of the WHOLE TimeStep - observation dict,
  # reward, discount, step_type - + sync, per step).  The envs go back to the same initial state and replay the same action
  # sequence (warm-up included), so both legs time the same stretch of the rollout.
  h_act = [torch.empty(envs, acts.shape[2], dtype=torch.float32, pin_memory=True).copy_(acts[i].cpu()) for i in range(nact)]
  h_out = env.make_host_timestep()
  env.reset()
  for i in range(warmup):
    env.step_host(h_act[i % nact], h_out)
  barrier()
  e0 = time.perf_counter()
  for i in range(steps):
    d2h = env.step_host(h_act[(warmup + i) % nact], h_out)
  barrier()
  e2e_value = envs * world * steps / max_over_ranks(time.perf_counter() - e0)
  h2d = envs * acts.shape[2] * 4

  # ---- episode statistics: the ONLY collective on this path (NCCL all_gather of return / length / success)
  gathered = gather_episode_stats(torch.cat([stats.local(), ret_sum[:, None]], dim=1))
  mean_return = float(gathered[:, 4].mean())

  # ---- roofline of the dominant kernel: algorithmic bytes per launch / mean launch duration (CUDA events inside the C-ABI,
  # on the launching stream).  One scene-kernel launch advances the envs of ONE pipeline group by one substep.
  peak, peak_src = measured_peak_gbs()
  kern = {k: dict(ms=k1[k][0] - k0[k][0], launches=k1[k][1] - k0[k][1]) for k in k1 if k1[k][1] - k0[k][1] > 0}
  ktot = sum(v['ms'] for v in kern.values()) or 1.0
  for v in kern.values():
    v['share_of_kernel_time'] = v['ms'] / ktot; v['us_per_launch'] = 1e3 * v['ms'] / v['launches']
  dom = max(kern, key=lambda k: kern[k]['ms'])
  per_launch_steps = envs * ksteps / kern[dom]['launches']
  bytes_per_launch = per_launch_steps * w['bytes_per_env_step']
  achieved = bytes_per_launch / (kern[dom]['us_per_launch'] * 1e-6) / 1e9
  traffic, traffic_src = ncu_traffic(name, envs, dom)
  roofline = dict(bound='hbm', achieved=achieved, peak=peak, unit='GB/s', frac=achieved / peak, traffic=traffic, kernel=dom,
                  us_per_launch=kern[dom]['us_per_launch'], algorithmic_bytes_per_launch=bytes_per_launch,
                  bytes_per_env_step=w['bytes_per_env_step'], env_steps_per_launch=per_launch_steps, peak_source=peak_src,
                  traffic_source=traffic_src, whole_step_frac=value / world * w['bytes_per_env_step'] / 1e9 / peak,
                  timed_over=f'{ksteps} control steps continuing the rollout right after the timed region (eager launches on ONE stream, so that every launch is timed alone; the timed region itself replays a CUDA graph with two pipeline groups in flight)',
                  note='state-only algorithmic bytes (SURVEY.md 8d) over the CUDA-event launch time; the path is latency / '
                       'instruction-issue bound, not HBM bound: see profiles/ for issue-slot and stall evidence')
  nsteps = c1['control_steps'] - c0['control_steps']
  res = dict(value=value, ms_per_step=dev_ms / steps, e2e=dict(value=e2e_value, unit='env-steps/s', h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h),
             gpu_launches=c1['kernel_launches'] - c0['kernel_launches'], graph_launches=c1['graph_launches'] - c0['graph_launches'],
             launches_per_step=(c1['kernel_launches'] - c0['kernel_launches']) / max(1, nsteps), clocks=clocks.summary(), roofline=roofline,
             kernels=kern, wall_s=t_wall, mean_return=mean_return, diverged=c1['diverged'], contacts_dropped=c1['contacts_dropped'],
             dropped_by_buffer_since_load=drops)
  env.close()
  return res


def run_steady_state(name, envs, steps, warmup, precision, dev, rank, episode_s=30.0):
  """Steady-state regime (BASELINE.md section 3: >= 200 steps after >= 50 warm-up) with episodes CYCLING through auto-reset and
  the on-device episode initialisation running: the headline workload (30 s episodes = 1501 control steps) with envs / 16 nursery
  envs sampling, collision-checking and settling fresh placements in the background.  After the warm-up the envs' episode step
  counters are spread uniformly over the episode length (so101_set_episode_steps), so that during the timed steps
  ~1/1501 of the envs finish and restart per step, each from a fresh placement.  The nursery envs' physics is inside the timed
  steps; only the user envs' steps are counted."""
  import torch
  from so101_sim_b200.task_suite import create_batched_task_env
  w = WORKLOADS[name]
  nursery = max(1, envs // 16)
  env = create_batched_task_env(w['task'], num_envs=envs, time_limit=episode_s, seed=1000 * rank, device=dev, precision=precision,
                                placement='device', nursery_envs=nursery)
  ep_steps = env.last_step
  nact = 64
  acts = _actions(env, nact, envs, dev, 1 + 1000 * rank)
  for i in range(warmup):
    env.step(acts[i % nact])
  env.set_episode_steps((torch.arange(envs, device=dev) * ep_steps // envs).to(torch.int32))   # phases uniform over the episode
  flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
  ev0 = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
  ev1 = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
  c0, p0 = env.counters(), env.placement_stats()
  nlast = torch.zeros((), dtype=torch.int64, device=dev); nfirst = torch.zeros((), dtype=torch.int64, device=dev)
  torch.cuda.synchronize()
  for i in range(steps):
    flush.fill_(i & 0xFF)
    ev0[i].record()
    ts = env.step(acts[(warmup + i) % nact])
    ev1[i].record()
    nlast += (ts.step_type == 2).sum(); nfirst += (ts.step_type == 0).sum()
  torch.cuda.synchronize()
  c1, p1 = env.counters(), env.placement_stats()
  ms = float(sum(ev0[i].elapsed_time(ev1[i]) for i in range(steps)))
  out = dict(value=envs * steps / (ms * 1e-3), unit='env-steps/s', ms_per_step=ms / steps, steps=steps, warmup=warmup, episode_steps=ep_steps,
             envs=envs, nursery_envs=nursery, last_steps=int(nlast), first_steps=int(nfirst), diverged=c1['diverged'] - c0['diverged'],
             contacts_dropped=c1['contacts_dropped'] - c0['contacts_dropped'],
             placements={k: p1[k] - p0[k] for k in p1},
             note=f'time_limit {episode_s} s episodes ({ep_steps} control steps), episode phases spread uniformly after the warm-up, random actions, '
                  'fresh on-device placement per episode (nursery physics inside the timed steps, not counted as env-steps); a step() that '
                  'lands on an env whose previous step was LAST resets it (FIRST) instead of stepping, as dm_control does')
  env.close()
  return out


if __name__ == '__main__':
  sys.exit(main())
