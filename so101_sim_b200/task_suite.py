"""Batched drop-in for the reference's env factory (so101_sim/task_suite.py:103-155) on the SO100 path.

`create_batched_task_env(...)` mirrors `create_task_env(task_name, time_limit, random_state, control_timestep, cameras,
**kwargs)` and adds `num_envs` / `device`.  The returned `BatchedEnvironment` keeps dm_control's `reset()` / `step()` ->
TimeStep contract with a leading batch dimension; all tensors are torch tensors on the CUDA device and cross a C-ABI
(include/so101_b200.h) into hand-written sm_100a kernels.  There is no CPU fallback.

Reference semantics restated here (host side):
  * task registry + kwargs filtering           task_suite.py:43-100,126-144
  * action_spec bounds                         so100_task.py:232-251
  * observation keys and delays                so100_task.py:189-210,331-368
  * time limit (`physics.time() >= time_limit` with float64 `time += 0.002`)   [upstream dm_control]
  * auto-reset on the step after LAST          [upstream dm_control composer.Environment.step]
"""
from __future__ import annotations

import collections
import ctypes
import dataclasses
import inspect
from typing import Any, NamedTuple

import numpy as np
import torch

from . import _lib
from .calibration import SO101Calibration
from .model import blob_path, body_set, read_blob, tcp_offset

DEFAULT_CONTROL_TIMESTEP = 0.02  # task_suite.py:41
PHYSICS_TIMESTEP = 0.002         # MuJoCo default; scene_pbr.xml sets none

# so100_task.py:45-60
SO100_HOME_CTRL = np.array([0.0, -1.57079, 1.57079, 1.57079, -1.57079, 0.0])
SO100_GRIPPER_CTRL_OPEN, SO100_GRIPPER_CTRL_CLOSE = 0.08, 0.0
_DEFAULT_PHYSICS_DELAY_SECS = 0.3            # so100_task.py:79
_DEFAULT_JOINT_OBSERVATION_DELAY_SECS = 0.1  # so100_task.py:80

STEP_FIRST, STEP_MID, STEP_LAST = 0, 1, 2

# Defaults of the batched inverse kinematics (BatchedEnvironment.solve_ik, so101_ee_ik).  From FK targets of random
# configurations inside 0.8 x the joint ranges, seeded 0.3 rad away, they reach < 1e-4 m and < 1e-3 rad in >= 99 % of the cases
# in 16 iterations (DESIGN.md).  damping in metres, w_rot in metres per radian, max_step in radians.
IK_DEFAULTS = dict(iterations=16, damping=0.01, w_rot=0.2, max_step=0.3, tolerance=0.0)


def ee_params(ee_offset, iterations=None, damping=None, w_rot=None, max_step=None, tolerance=None) -> _lib.EEParams:
  """so101_ee_params from the TCP offset and the IK parameters (None = IK_DEFAULTS); raises ValueError on a bad value."""
  d = dict(IK_DEFAULTS)
  d.update({k: v for k, v in dict(iterations=iterations, damping=damping, w_rot=w_rot, max_step=max_step, tolerance=tolerance).items()
            if v is not None})
  off = np.asarray(ee_offset, dtype=np.float64)
  if off.shape != (3,) or not np.all(np.isfinite(off)):
    raise ValueError(f'ee_offset must be 3 finite numbers, got {ee_offset!r}')
  if int(d['iterations']) != d['iterations'] or d['iterations'] < 0:
    raise ValueError('iterations must be an integer >= 0')
  for k, ok in (('damping', lambda v: v > 0), ('w_rot', lambda v: v >= 0), ('max_step', lambda v: v > 0)):
    if not (np.isfinite(d[k]) and ok(d[k])):
      raise ValueError(f'{k} must be finite and {"> 0" if k != "w_rot" else ">= 0"}, got {d[k]!r}')
  if not d['tolerance'] >= 0:
    raise ValueError(f'tolerance must be >= 0, got {d["tolerance"]!r}')
  p = _lib.EEParams()
  for c in range(3):
    p.tcp_offset[c] = float(off[c])
  p.iterations, p.damping, p.w_rot, p.max_step, p.tolerance = int(d['iterations']), float(d['damping']), float(d['w_rot']), float(d['max_step']), float(d['tolerance'])
  return p


def quat_from_rotvec(r: torch.Tensor) -> torch.Tensor:
  """Unit quaternions (wxyz) of rotation vectors [..., 3] (float64 arithmetic)."""
  r = r.double()
  a = r.norm(dim=-1, keepdim=True)
  k = torch.where(a > 1e-12, torch.sin(0.5 * a) / a.clamp_min(1e-12), torch.full_like(a, 0.5))
  return torch.cat([torch.cos(0.5 * a), k * r], dim=-1)


def quat_mul(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
  """Hamilton product of wxyz quaternions [..., 4]."""
  w1, x1, y1, z1 = a.unbind(-1)
  w2, x2, y2, z2 = b.unbind(-1)
  return torch.stack([w1 * w2 - x1 * x2 - y1 * y2 - z1 * z2, w1 * x2 + x1 * w2 + y1 * z2 - z1 * y2,
                      w1 * y2 - x1 * z2 + y1 * w2 + z1 * x2, w1 * z2 + x1 * y2 - y1 * x2 + z1 * w2], dim=-1)

OBSERVATION_KEYS = ('commanded_joints_pos', 'joints_pos', 'joints_vel', 'physics_state', 'undelayed_joints_pos',
                    'undelayed_joints_vel', 'delayed_physics_state')  # examples/so101_rl_breakdown.ipynb:65


class BatchedTimeStep(NamedTuple):
  """dm_env.TimeStep with a leading env dimension.  FIRST steps carry reward 0 / discount 1 (dm_env uses None)."""
  step_type: torch.Tensor   # uint8 [N]
  reward: torch.Tensor      # float32 [N]
  discount: torch.Tensor    # float32 [N]
  observation: 'collections.OrderedDict[str, torch.Tensor]'

  def first(self): return self.step_type == STEP_FIRST
  def mid(self): return self.step_type == STEP_MID
  def last(self): return self.step_type == STEP_LAST


@dataclasses.dataclass(frozen=True)
class BoundedArraySpec:
  shape: tuple
  dtype: Any
  minimum: np.ndarray
  maximum: np.ndarray


class SO100Task:
  """Host-side description of the base SO100 task (so100_task.py:101-320): reward 0, never succeeds."""
  model_name = 'so100_arm'
  collide = False
  instruction = ''

  def __init__(self, control_timestep, cameras=(), joints_observation_delay_secs=_DEFAULT_JOINT_OBSERVATION_DELAY_SECS,
               image_observation_enabled=True, image_observation_delay_secs=_DEFAULT_PHYSICS_DELAY_SECS, update_interval=1,
               table_height_offset=0.0, rotation_joint_limit=np.pi, terminate_episode=True):
    if cameras:
      raise NotImplementedError('camera rendering is out of scope of the B200 path: pass cameras=()')
    if table_height_offset:
      raise NotImplementedError('table_height_offset needs a recompiled model blob')
    self.control_timestep = control_timestep
    self.rotation_joint_limit = rotation_joint_limit
    self.terminate_episode = terminate_episode
    self.joints_delay_secs = joints_observation_delay_secs
    self.physics_delay_secs = image_observation_delay_secs

  def get_instruction(self):
    return self.instruction


class SO100HandOver(SO100Task):
  """so100_hand_over.py:121-326 (overlap reward): banana -> bowl (:81-96) and pen -> utensil holder (:97-117).  The object /
  container models, the container mesh scale and the overlap boxes are compiled into the model blob (tools/compile_model.py)."""
  collide = True
  # so100_hand_over.py:34-55: placement distributions of the object and the container (position boxes at TABLE_HEIGHT +
  # RESET_HEIGHT = 0.45, object yaw uniform in +-0.1 pi, container rotation identity) and :208-229 the PropPlacers (the object
  # ignores collisions, the container is re-sampled while it collides; both then settle together with the arm frozen)
  PLACE_LO = ((0.2, -0.1, 0.45), (-0.3, -0.1, 0.45))
  PLACE_HI = ((0.3, 0.1, 0.45), (-0.2, 0.1, 0.45))
  PLACE_YAW = ((-0.1 * np.pi, 0.1 * np.pi), (0.0, 0.0))
  PLACE_CHECK_COLLISIONS = (0, 1)
  # object -> (model blob, instruction, (object z, container z) just above rest on the table top or None = spawn height)
  CONFIGS = {
      'banana': ('so100_handover_banana', 'pick up the banana and put it in the bowl using the SO100 arm', (0.4217, 0.4226)),
      'pen': ('so100_handover_pen', 'pick up the pen and put it in the container using the SO100 arm', None),
  }

  def __init__(self, object_name, reward_based_on_overlap=True, **kwargs):
    super().__init__(**kwargs)
    if object_name not in self.CONFIGS:
      raise ValueError(f'Invalid object name: {object_name}, must be one of {self.CONFIGS.keys()}')  # so100_hand_over.py:146-150
    if not reward_based_on_overlap:
      # The reference's fallback (so100_hand_over.py:277-318) looks up the body 'so100/hand_link' (:284-288), which does not
      # exist in the scene it loads (scene_pbr.xml: Base ... Moving_Jaw): mjcf `find` returns None and the first get_reward()
      # raises AttributeError inside env.step().  There is no working behaviour to reproduce, so this fails at construction.
      raise NotImplementedError("reward_based_on_overlap=False is not usable in the reference either: its get_reward() raises "
                                "AttributeError on the missing body 'so100/hand_link' (so100_hand_over.py:284-288)")
    self.object_name = object_name
    self.model_name, self.instruction, self.rest_heights = self.CONFIGS[object_name]


class SO100TwoArmHandOver(SO100HandOver):
  """BASELINE config 4 ("hand-over task, two arms"): a LABELLED SYNTHETIC scene.  The reference has no two-SO100 scene (its only
  two-arm hand-over is the ALOHA task so101_sim/tasks/hand_over.py:122, another robot), so this is scene_pbr.xml with its arm
  at (+0.12, 0.3) and a second identical arm at (-0.12, 0.3) (tools/compile_model.py two_arm_scene_xml), the reference's table,
  obstacles, free props, placement distributions and overlap reward.  Actions / joint observations are 12-vectors (arm A then
  arm B); the kernels are the same sources built for two arms (libso101_b200_2arm.so)."""
  CONFIGS = {'banana': ('so100_twoarm_banana', 'hand the banana over and put it in the bowl using two SO100 arms', (0.4217, 0.4226))}


class SO100ArmOnly(SO100Task):
  """BASELINE config 2: scene_pbr.xml without the free props, collisions off, base-task semantics (reward 0)."""
  model_name = 'so100_arm'
  collide = False


# task_suite.py:98-99 (+ the arm-only benchmark scene, which has no reference registry entry)
TASK_FACTORIES = {
    'SO100HandOverBanana': (SO100HandOver, {'object_name': 'banana'}),
    'SO100HandOverPen': (SO100HandOver, {'object_name': 'pen'}),
    'SO100ArmOnly': (SO100ArmOnly, {}),
    'SO100TwoArmHandOverBanana': (SO100TwoArmHandOver, {'object_name': 'banana'}),   # synthetic (BASELINE config 4), see the class
}


def time_limit_to_last_step(time_limit: float, control_timestep: float, physics_timestep: float = PHYSICS_TIMESTEP) -> int:
  """Control-step index whose TimeStep is LAST: dm_control tests `physics.time() >= time_limit` after each control step and
  MuJoCo accumulates `time += timestep` in float64 (30 s -> step 1501, not 1500; SURVEY.md §6).  The float64 running sum is
  reproduced exactly (np.add.accumulate adds sequentially) in chunks, so large limits cost milliseconds, not a Python loop."""
  if not np.isfinite(time_limit):
    return 0
  nsub = int(round(control_timestep / physics_timestep))
  if time_limit <= 0:
    return 1
  if time_limit / physics_timestep > 2e9:
    raise ValueError('time_limit too large')
  chunk = nsub * 100_000
  t, done = 0.0, 0
  while True:
    acc = np.add.accumulate(np.concatenate(([t], np.full(chunk, physics_timestep))))[1:]
    ends = acc[nsub - 1::nsub]            # time after each control step of this chunk
    hit = np.nonzero(ends >= time_limit)[0]
    if len(hit):
      return done + int(hit[0]) + 1
    t, done = float(acc[-1]), done + len(ends)


class BatchedEnvironment:
  """N lockstep copies of one reference environment (composer.Environment, task_suite.py:148-155)."""

  def __init__(self, task: SO100Task, num_envs: int, time_limit: float, seed: int | None, device, calibration_offsets, precision,
               solver_iterations, solver_tolerance, nursery_envs: int = 0, ring_capacity: int | None = None, integrator: str = 'euler'):
    self.task = task
    self.num_envs = int(num_envs)
    self.device = torch.device(device)
    if self.device.type != 'cuda':
      raise RuntimeError('so101_sim_b200 runs on CUDA devices only (no CPU fallback)')
    if not torch.cuda.is_available():
      raise RuntimeError('CUDA is not available: so101_sim_b200 has no CPU fallback')
    self.seed = 0 if seed is None else int(seed)
    self.control_timestep = task.control_timestep
    self.n_substeps = int(round(task.control_timestep / PHYSICS_TIMESTEP))
    self.model = read_blob(task.model_name)
    self.narm = int(self.model['nu'][0]) // 6
    self._lib = _lib.load(self.narm)
    with open(blob_path(task.model_name), 'rb') as f:
      blob = f.read()
    offs = np.zeros(6) if calibration_offsets is None else np.asarray(calibration_offsets, dtype=np.float64)
    if offs.shape != (6,):
      raise ValueError(f'Expected 6 calibration offsets, got shape {offs.shape}')
    self.calibration_offsets = offs
    cfg = _lib.Config()
    cfg.num_envs = self.num_envs
    cfg.device = self.device.index if self.device.index is not None else torch.cuda.current_device()
    cfg.n_substeps = self.n_substeps
    cfg.last_step = time_limit_to_last_step(time_limit, task.control_timestep)
    cfg.joints_delay_steps = int(round(task.joints_delay_secs / task.control_timestep)) if task.joints_delay_secs else 0
    cfg.physics_delay_steps = int(round(task.physics_delay_secs / task.control_timestep)) if task.physics_delay_secs else 0
    cfg.terminate_on_success = int(task.terminate_episode)
    cfg.solver_iterations = int(solver_iterations)
    cfg.solver_tolerance = float(solver_tolerance)
    cfg.precision = {'f32': 32, 'f64': 64}[precision]
    cfg.collide = int(task.collide)
    if integrator not in ('euler', 'implicitfast'):
      raise ValueError("integrator must be 'euler' (MuJoCo's default, what the reference runs) or 'implicitfast'")
    cfg.integrator = int(integrator == 'implicitfast')
    self.integrator = integrator
    for i in range(6):
      cfg.calibration_offsets[i] = float(offs[i]); cfg.home_ctrl[i] = float(SO100_HOME_CTRL[i])
    # on-device episode initialisation (so100_hand_over.py:208-229,320-323): placement distributions + nursery envs
    self.nursery_envs = int(nursery_envs) if task.collide else 0
    cfg.nursery_envs = self.nursery_envs
    cfg.ring_capacity = int(ring_capacity) if ring_capacity is not None else max(2 * self.nursery_envs, 1)
    cfg.seed = self.seed & 0xFFFFFFFFFFFFFFFF
    if task.collide and hasattr(task, 'PLACE_LO'):
      for p in range(2):
        for k in range(3):
          cfg.place_lo[p][k] = task.PLACE_LO[p][k]; cfg.place_hi[p][k] = task.PLACE_HI[p][k]
        cfg.place_yaw[p][0], cfg.place_yaw[p][1] = task.PLACE_YAW[p]
        cfg.place_check_collisions[p] = task.PLACE_CHECK_COLLISIONS[p]
    cfg.place_max_attempts = 20          # [upstream] PropPlacer max_attempts_per_prop
    cfg.settle_max_substeps = int(round(2.0 / PHYSICS_TIMESTEP))   # [upstream] max_settle_physics_time = 2 s
    cfg.settle_qvel_tol, cfg.settle_qacc_tol = 1e-3, 1e-2          # [upstream] _SETTLE_QVEL_TOL, _SETTLE_QACC_TOL
    self.precision = precision
    self.last_step = cfg.last_step
    h = ctypes.c_void_p()
    rc = self._lib.so101_create(blob, len(blob), ctypes.byref(cfg), ctypes.byref(h))
    if rc != 0:
      raise RuntimeError(f'so101_create failed ({rc}): {self._lib.so101_last_error(None).decode()}')
    self._h = h
    dims = [ctypes.c_int() for _ in range(4)]
    self._check(self._lib.so101_dims(self._h, *[ctypes.byref(d) for d in dims]))
    self.nq, self.nv, self.nu, self.nbody = (d.value for d in dims)
    N, sd, nu = self.num_envs, self.nq + self.nv, self.nu
    f32 = dict(dtype=torch.float32, device=self.device)
    self._buf = dict(commanded_joints_pos=torch.zeros(N, nu, **f32), joints_pos=torch.zeros(N, nu, **f32),
                     undelayed_joints_pos=torch.zeros(N, nu, **f32), physics_state=torch.zeros(N, sd, **f32),
                     delayed_physics_state=torch.zeros(N, sd, **f32), reward=torch.zeros(N, **f32), discount=torch.ones(N, **f32),
                     step_type=torch.zeros(N, dtype=torch.uint8, device=self.device))
    self._empty = torch.zeros(N, 0, **f32)  # joints_vel is an EMPTY array in the reference (so100_task.py:357-364)
    self._out = _lib.StepOut(**{k: v.data_ptr() for k, v in self._buf.items()})
    self._closed = False

  # ------------------------------------------------------------------ plumbing
  def _check(self, rc):
    if rc != 0:
      raise RuntimeError(f'so101_b200 call failed ({rc}): {self._lib.so101_last_error(self._h).decode()}')

  def _stream(self):
    return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

  def _timestep(self) -> BatchedTimeStep:
    b = self._buf
    obs = collections.OrderedDict()
    for k in OBSERVATION_KEYS:
      obs[k] = self._empty if k.endswith('joints_vel') else b[k]
    return BatchedTimeStep(b['step_type'], b['reward'], b['discount'], obs)

  # ------------------------------------------------------------------ reference API
  def action_spec(self) -> BoundedArraySpec:
    """so100_task.py:232-251 — not enforced on step (neither dm_control nor the task clips actions)."""
    lo = self.model['act_ctrlrange'].reshape(-1, 2)[:, 0].astype(np.float32)
    hi = self.model['act_ctrlrange'].reshape(-1, 2)[:, 1].astype(np.float32)
    for k in range(self.narm):   # per arm: rotation joint limit on the first actuator, gripper range on the last
      lo[6 * k], hi[6 * k] = -self.task.rotation_joint_limit, self.task.rotation_joint_limit
      lo[6 * k + 5], hi[6 * k + 5] = SO100_GRIPPER_CTRL_CLOSE, SO100_GRIPPER_CTRL_OPEN
    return BoundedArraySpec(shape=(self.nu,), dtype=np.float32, minimum=lo, maximum=hi)

  def observation_spec(self):
    sd = self.nq + self.nv
    nu = self.nu
    shapes = dict(commanded_joints_pos=(nu,), joints_pos=(nu,), joints_vel=(0,), physics_state=(sd,), undelayed_joints_pos=(nu,),
                  undelayed_joints_vel=(0,), delayed_physics_state=(sd,))
    return collections.OrderedDict((k, shapes[k]) for k in OBSERVATION_KEYS)

  def reset(self, mask: torch.Tensor | None = None) -> BatchedTimeStep:
    """composer.Environment.reset() for all envs (or those with mask != 0)."""
    mp = None
    if mask is not None:
      mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
      if mask.shape != (self.num_envs,):
        raise ValueError('mask must have shape [num_envs]')
      mp = ctypes.c_void_p(mask.data_ptr())
    self._check(self._lib.so101_reset(self._h, mp, ctypes.byref(self._out), self._stream()))
    return self._timestep()

  def step(self, action: torch.Tensor) -> BatchedTimeStep:
    """composer.Environment.step(action) for all envs; action float32 [N,6] on the env's device."""
    if not isinstance(action, torch.Tensor):
      action = torch.as_tensor(np.asarray(action), dtype=torch.float32)
    if action.shape != (self.num_envs, self.nu):
      raise ValueError(f'action must have shape [{self.num_envs}, {self.nu}], got {tuple(action.shape)}')
    action = action.to(device=self.device, dtype=torch.float32).contiguous()
    self._check(self._lib.so101_step(self._h, ctypes.c_void_p(action.data_ptr()), ctypes.byref(self._out), self._stream()))
    return self._timestep()

  def make_host_timestep(self) -> dict:
    """Pinned host tensors for every block of the TimeStep (the observation dict, reward, discount, step_type): the
    destination of step_host()."""
    N, sd = self.num_envs, self.nq + self.nv
    pin = dict(pin_memory=True)
    nu = self.nu
    return dict(commanded_joints_pos=torch.zeros(N, nu, **pin), joints_pos=torch.zeros(N, nu, **pin), undelayed_joints_pos=torch.zeros(N, nu, **pin),
                physics_state=torch.zeros(N, sd, **pin), delayed_physics_state=torch.zeros(N, sd, **pin), reward=torch.zeros(N, **pin),
                discount=torch.zeros(N, **pin), step_type=torch.zeros(N, dtype=torch.uint8, **pin))

  def step_host(self, action_host: torch.Tensor, host_out: dict) -> int:
    """End-to-end step with (pinned) HOST tensors: H2D of the action, the step, D2H of every TimeStep block present in
    `host_out` (see make_host_timestep) and a stream sync, all inside the call (so101_step_host).  Returns the bytes copied
    back."""
    out = _lib.StepOut(**{k: v.data_ptr() for k, v in host_out.items()})
    self._check(self._lib.so101_step_host(self._h, ctypes.c_void_p(action_host.data_ptr()), ctypes.byref(out), self._stream()))
    return sum(v.numel() * v.element_size() for v in host_out.values())

  def close(self):
    if not self._closed and getattr(self, '_h', None):
      self._lib.so101_destroy(self._h)
      self._closed = True

  def __del__(self):
    try:
      self.close()
    except Exception:
      pass

  # ------------------------------------------------------------------ state access (physics.get_state / set_state)
  def _put_state(self, qpos, qvel, initial: bool):
    """float64 tensors go in unrounded (the integration state is float64 in both precisions); anything else as float32."""
    f64 = qpos.dtype == torch.float64 or qvel.dtype == torch.float64
    dt = torch.float64 if f64 else torch.float32
    q = qpos.to(device=self.device, dtype=dt).contiguous(); v = qvel.to(device=self.device, dtype=dt).contiguous()
    assert q.shape == (self.num_envs, self.nq) and v.shape == (self.num_envs, self.nv)
    qp, vp = ctypes.c_void_p(q.data_ptr()), ctypes.c_void_p(v.data_ptr())
    if f64:
      self._check(self._lib.so101_set_state_f64(self._h, qp, vp, int(initial), self._stream()))
    elif initial:
      self._check(self._lib.so101_set_initial_state(self._h, qp, vp, self._stream()))
    else:
      self._check(self._lib.so101_set_state(self._h, qp, vp, self._stream()))

  def set_initial_state(self, qpos: torch.Tensor, qvel: torch.Tensor):
    self._put_state(qpos, qvel, True)

  def set_state(self, qpos: torch.Tensor, qvel: torch.Tensor):
    self._put_state(qpos, qvel, False)

  def get_state(self, dtype=torch.float32):
    q = torch.empty(self.num_envs, self.nq, dtype=dtype, device=self.device); v = torch.empty(self.num_envs, self.nv, dtype=dtype, device=self.device)
    fn = self._lib.so101_get_state if dtype == torch.float32 else self._lib.so101_get_state_f64
    self._check(fn(self._h, ctypes.c_void_p(q.data_ptr()), ctypes.c_void_p(v.data_ptr()), self._stream()))
    return q, v

  def get_episode_steps(self) -> torch.Tensor:
    """int32 [N]: control steps each env has taken in its current episode (decides when the time limit fires)."""
    out = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
    self._check(self._lib.so101_get_episode_steps(self._h, ctypes.c_void_p(out.data_ptr()), self._stream()))
    return out

  def set_episode_steps(self, steps: torch.Tensor):
    """Checkpoint-resume companion of set_state(): restore the per-env episode step counters (also used to start a batch at
    staggered episode phases)."""
    s = steps.to(device=self.device, dtype=torch.int32).contiguous()
    if s.shape != (self.num_envs,):
      raise ValueError('steps must have shape [num_envs]')
    self._check(self._lib.so101_set_episode_steps(self._h, ctypes.c_void_p(s.data_ptr()), self._stream()))

  def save_checkpoint(self) -> torch.Tensor:
    """Everything the env needs to continue this rollout bit for bit, as one uint8 device tensor: physics state, warm starts,
    ctrl, observation delay buffers, episode counters and auto-reset flags, reset states, and the placement machinery (nursery
    envs, Philox draw counters, the ring of settled placements).  get_state() alone is physics.get_state() (so100_task.py:366-368)."""
    n = ctypes.c_size_t(0)
    self._check(self._lib.so101_checkpoint_size(self._h, ctypes.byref(n)))
    buf = torch.empty(n.value, dtype=torch.uint8, device=self.device)
    self._check(self._lib.so101_checkpoint_save(self._h, ctypes.c_void_p(buf.data_ptr()), n.value, self._stream()))
    return buf

  def load_checkpoint(self, buf: torch.Tensor):
    """Restore a save_checkpoint() tensor into this env (same task, precision, num_envs, nursery_envs and ring capacity)."""
    b = buf.to(device=self.device, dtype=torch.uint8).contiguous()
    self._check(self._lib.so101_checkpoint_load(self._h, ctypes.c_void_p(b.data_ptr()), b.numel(), self._stream()))

  def debug_read(self, field: str, width: int = 1) -> torch.Tensor:
    out = torch.empty(self.num_envs, width, dtype=torch.float32, device=self.device)
    self._check(self._lib.so101_debug_read(self._h, field.encode(), ctypes.c_void_p(out.data_ptr()), out.numel(), self._stream()))
    return out

  def debug_contacts(self):
    """Parity probe: contacts of the last substep, per env a list of (geom1, geom2, dist, pos[3], normal[3]).  The first call
    enables the probe and returns empty lists.  Raises if an env had more contacts than the probe holds."""
    width = int(self.debug_read('contacts_width')[0, 0])
    raw = self.debug_read('contacts', 1 + 9 * width).cpu().numpy()
    out = []
    for e in range(self.num_envs):
      n = int(raw[e, 0])
      if n > width:
        raise RuntimeError(f'env {e} had {n} contacts, the contact probe holds {width}')
      rows = raw[e, 1:1 + 9 * n].reshape(n, 9)
      out.append([(int(r[0]), int(r[1]), float(r[2]), r[3:6].copy(), r[6:9].copy()) for r in rows])
    return out

  def counters(self) -> dict:
    c = (ctypes.c_uint64 * 6)()
    self._check(self._lib.so101_counters(self._h, ctypes.byref(c)))
    return dict(kernel_launches=int(c[0]), control_steps=int(c[1]), diverged=int(c[2]), contacts_dropped=int(c[3]), graph_launches=int(c[4]))

  def contacts_dropped_per_env(self) -> torch.Tensor:
    """int64 [N]: contacts / candidate pairs each env has lost to a full per-env buffer since the env was created (candidate pairs
    beyond 64 or raw contacts beyond 128 per substep, Jacobian blocks beyond the largest solver tier's pool).  MuJoCo has no such
    caps; counters()['contacts_dropped'] is the sum."""
    return self.debug_read('dropped').flatten().to(torch.int64)

  # ------------------------------------------------------------------ contact force sensors
  def _body_side(self, side) -> set:
    if isinstance(side, str):
      return set(body_set(self.model, side))
    ids = [side] if isinstance(side, (int, np.integer)) else list(side)
    out = set()
    for b in ids:
      if isinstance(b, bool) or not isinstance(b, (int, np.integer)):
        raise ValueError(f'a body set holds body ids, a name or a list of ids, got {b!r}')
      if not 0 <= int(b) < self.nbody:
        raise ValueError(f'body id {int(b)} out of range (the model has {self.nbody} bodies)')
      out.add(int(b))
    return out

  def set_contact_sensors(self, pairs):
    """Configure up to 16 contact force sensors, one per (A, B) pair of disjoint body sets; [] turns them off (the default).  Each
    side is a body id, an iterable of ids or a name of model.body_set for arm 0 (model.BODY_SET_NAMES); 'others' stands for every body
    not on the other side.  After every step, contact_sensors() gives per env and sensor the net force on A from B (world
    frame, N), the sum of the normal forces and the number of contacts, over the contacts of the step's last substep.  The
    readout follows the new configuration from the next step on."""
    if not self.task.collide:
      raise ValueError('contact sensors need a task with a contact scene')
    pairs = list(pairs)
    if len(pairs) > _lib.MAX_CONTACT_SENSORS:
      raise ValueError(f'at most {_lib.MAX_CONTACT_SENSORS} contact sensors, got {len(pairs)}')
    masks = ((ctypes.c_uint32 * 2) * max(1, len(pairs)))()
    for k, pair in enumerate(pairs):
      if len(pair) != 2:
        raise ValueError(f'sensor {k}: expected a pair (A, B), got {pair!r}')
      a, b = pair
      if isinstance(a, str) and a == 'others' and isinstance(b, str) and b == 'others':
        raise ValueError(f"sensor {k}: only one side may be 'others'")
      sa = None if isinstance(a, str) and a == 'others' else self._body_side(a)
      sb = None if isinstance(b, str) and b == 'others' else self._body_side(b)
      every = set(range(self.nbody))
      sa = every - sb if sa is None else sa
      sb = every - sa if sb is None else sb
      if not sa or not sb:
        raise ValueError(f'sensor {k}: empty body set')
      if sa & sb:
        raise ValueError(f'sensor {k}: bodies {sorted(sa & sb)} are on both sides')
      masks[k][0] = sum(1 << x for x in sa); masks[k][1] = sum(1 << x for x in sb)
    self._check(self._lib.so101_contact_sensors(self._h, len(pairs), ctypes.cast(masks, ctypes.c_void_p)))
    self._nsensor = len(pairs)

  def contact_sensors(self) -> torch.Tensor:
    """float32 [N, K, 5] readout of the K configured sensors after the last step: net force on A from B (x, y, z; world frame,
    newtons), sum of the normal forces, number of contacts.  Zero for envs that returned FIRST, were reset or diverged."""
    out = torch.zeros(self.num_envs, getattr(self, '_nsensor', 0), 5, dtype=torch.float32, device=self.device)
    if out.numel() == 0:
      return out
    self._check(self._lib.so101_contact_sensors_read(self._h, ctypes.c_void_p(out.data_ptr()), out.numel(), self._stream()))
    return out

  KERNEL_NAMES = ("scene_begin_kernel", "scene_narrow_kernel", "scene_solve_kernel", "scene_solve_tier1_kernel", "arm_step_kernel", "scene_gjk_kernel",
                  "scene_kindyn_kernel", "scene_broad_kernel", "scene_epa_kernel", "scene_manifold_kernel", "scene_solve_tier2_kernel")

  def kernel_times(self, enable: bool = True) -> dict:
    """Accumulated per-kernel device time (CUDA events around each launch, recorded while enabled) -> {name: (ms, launches)};
    then switches the recording on/off for the following steps."""
    ms = (ctypes.c_double * 11)(); n = (ctypes.c_uint64 * 11)()
    self._check(self._lib.so101_kernel_times(self._h, int(enable), ctypes.byref(ms), ctypes.byref(n)))
    return {k: (float(ms[i]), int(n[i])) for i, k in enumerate(self.KERNEL_NAMES)}

  # ------------------------------------------------------------------ end-effector queries and Cartesian control
  # The tool centre point (TCP) is a point fixed in each arm's Fixed_Jaw body (model.tcp_offset: between the jaw pads); its
  # orientation is the Fixed_Jaw frame.  Shapes always keep the arm dimension, also with one arm: positions [N, narm, 3],
  # quaternions [N, narm, 4] (wxyz, w >= 0), gripper [N, narm], errors [N, narm, 2].  None of these calls changes the env's state.
  @property
  def tcp_offset(self) -> np.ndarray:
    """Default TCP offset (metres, Fixed_Jaw frame) of this model's arms."""
    if not hasattr(self, '_tcp_offset'):
      offs = [tcp_offset(self.model, k) for k in range(self.narm)]
      if any(not np.array_equal(o, offs[0]) for o in offs):
        raise RuntimeError('the arms of this model have different jaws: pass ee_offset explicitly')
      self._tcp_offset = offs[0]
    return self._tcp_offset

  def _ee_in(self, x, tail: tuple, name: str) -> torch.Tensor:
    t = x.to(device=self.device, dtype=torch.float32) if isinstance(x, torch.Tensor) else torch.as_tensor(np.asarray(x), dtype=torch.float32, device=self.device)
    shape = (self.num_envs, self.narm) + tail
    if tuple(t.shape) != shape:
      raise ValueError(f'{name} must have shape {list(shape)}, got {list(t.shape)}')
    return t.contiguous()

  def ee_pose(self, source: str = 'state', ee_offset=None):
    """TCP pose of every env and arm -> (pos [N, narm, 3], quat [N, narm, 4]) float32, from the current joint state
    (source='state') or the current commanded joint targets (source='command': the last action plus the calibration offsets)."""
    if source not in ('state', 'command'):
      raise ValueError("source must be 'state' or 'command'")
    off = (ctypes.c_float * 3)(*ee_params(self.tcp_offset if ee_offset is None else ee_offset).tcp_offset)
    pos = torch.empty(self.num_envs, self.narm, 3, dtype=torch.float32, device=self.device)
    quat = torch.empty(self.num_envs, self.narm, 4, dtype=torch.float32, device=self.device)
    self._check(self._lib.so101_ee_pose(self._h, int(source == 'command'), ctypes.byref(off), ctypes.c_void_p(pos.data_ptr()),
                                        ctypes.c_void_p(quat.data_ptr()), self._stream()))
    return pos, quat

  def solve_ik(self, target_pos, target_quat=None, gripper=None, seed=None, ee_offset=None, **params):
    """Batched damped-least-squares IK of the TCP on the device (so101_ee_ik) -> (action [N, nu], err [N, narm, 2]).

    target_pos [N, narm, 3] metres; target_quat [N, narm, 4] wxyz or None (position only); gripper [N, narm] jaw actions or None
    (keep the commanded jaw target); seed [N, nu] joint positions to start from or None (the current state).  `action` is what
    step() takes (joint targets minus the calibration offsets); `err` holds the final position error (m) and orientation error
    (rad, 0 without target_quat).  Targets are never rejected: an unreachable one gives joint targets inside the joint ranges
    and a large error.  params: iterations, damping, w_rot, max_step, tolerance (defaults IK_DEFAULTS)."""
    p = ee_params(self.tcp_offset if ee_offset is None else ee_offset, **params)
    tp = self._ee_in(target_pos, (3,), 'target_pos')
    tq = None if target_quat is None else self._ee_in(target_quat, (4,), 'target_quat')
    g = None if gripper is None else self._ee_in(gripper, (), 'gripper')
    sq = None
    if seed is not None:
      sq = seed.to(device=self.device, dtype=torch.float32).contiguous() if isinstance(seed, torch.Tensor) else torch.as_tensor(np.asarray(seed), dtype=torch.float32, device=self.device)
      if tuple(sq.shape) != (self.num_envs, self.nu):
        raise ValueError(f'seed must have shape [{self.num_envs}, {self.nu}], got {list(sq.shape)}')
    ptr = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())
    action = torch.empty(self.num_envs, self.nu, dtype=torch.float32, device=self.device)
    err = torch.empty(self.num_envs, self.narm, 2, dtype=torch.float32, device=self.device)
    self._check(self._lib.so101_ee_ik(self._h, ptr(tp), ptr(tq), ptr(g), ptr(sq), ctypes.byref(p), ptr(action), ptr(err), self._stream()))
    return action, err

  def step_ee(self, delta_pos, gripper, delta_rot=None, base: str = 'state', workspace=None, ee_offset=None, **params) -> BatchedTimeStep:
    """Cartesian end-effector control: target = TCP(base) + delta_pos ([N, narm, 3] metres), clipped to the workspace box
    ((lo[3], hi[3]) in world coordinates, or None), solved by solve_ik with the jaw action `gripper` [N, narm], then step(action).
    delta_rot [N, narm, 3] (rotation vector, world frame) also sets a target orientation exp(delta_rot) * R_tcp(base); without it
    the IK is position only.  base='state' starts from the current TCP, 'command' from the TCP of the commanded targets.  The
    IK errors of the step stay in `last_ee_error` [N, narm, 2]."""
    pos, quat = self.ee_pose(base, ee_offset)
    target = pos + self._ee_in(delta_pos, (3,), 'delta_pos')
    if workspace is not None:
      lo, hi = (torch.as_tensor(np.asarray(w, dtype=np.float32), device=self.device) for w in workspace)
      if lo.shape != (3,) or hi.shape != (3,) or bool((lo > hi).any()):
        raise ValueError('workspace must be (lo[3], hi[3]) with lo <= hi')
      target = torch.minimum(torch.maximum(target, lo), hi)
    tq = None
    if delta_rot is not None:
      tq = quat_mul(quat_from_rotvec(self._ee_in(delta_rot, (3,), 'delta_rot')), quat.double()).float()
    action, self.last_ee_error = self.solve_ik(target, tq, gripper, ee_offset=ee_offset, **params)
    return self.step(action)

  # ------------------------------------------------------------------ synthetic initial states (BASELINE.md §3)
  def sample_arm_initial_states(self, seed: int = 0, fraction: float = 0.25):
    """BASELINE config 2: arm qpos ~ U(fraction * joint range), qvel = 0 (Philox stream `seed`)."""
    g = torch.Generator(device='cpu'); g.manual_seed(int(seed))  # CPU Philox stream: identical states on any device
    rng = torch.tensor(self.model['jnt_range'].reshape(-1, 2)[:6], dtype=torch.float32, device=self.device)
    u = torch.rand(self.num_envs, 6, generator=g).to(self.device)
    q = torch.tensor(self.model['qpos0'], dtype=torch.float32, device=self.device).repeat(self.num_envs, 1)
    q[:, :6] = fraction * (rng[:, 0] + u * (rng[:, 1] - rng[:, 0]))
    v = torch.zeros(self.num_envs, self.nv, dtype=torch.float32, device=self.device)
    self.set_initial_state(q, v)
    return q, v


  # so100_hand_over.py:34-55 placement distributions; rest heights from the reference's own reset state (KAT-1,
  # so101_rl.ipynb:221-223: banana z = 0.4217, bowl z = 0.4226)
  def _bowl_obstacles(self, z_bowl: float):
    """Static upright cylinders the bowl would penetrate when placed at height z_bowl with identity rotation: list of
    (cx, cy, reject_radius).  [upstream] PropPlacer(ignore_collisions=False) rejects such samples (so100_hand_over.py:216-221);
    here the test is geometric: the bowl's hull vertices below the cylinder's top face, as a disc around the bowl axis."""
    m = self.model
    bowl_body = int(m['prop_body'][1])
    verts = m['hull_vert'].reshape(-1, 3)
    bv = np.concatenate([verts[a:a + n] for g, (a, n) in enumerate(zip(m['geom_vertadr'], m['geom_vertnum']))
                         if m['geom_body'][g] == bowl_body and m['geom_type'][g] == 5])
    out = []
    for g in range(int(np.asarray(m['ngeom']).reshape(-1)[0])):
      b = int(m['geom_body'][g])
      if m['geom_type'][g] != 3 or m['body_weld'][b] != 0 or m['body_parent'][b] != 0:
        continue
      c = m['body_pos'].reshape(-1, 3)[b] + m['geom_pos'].reshape(-1, 3)[g]
      r, h = m['geom_size'].reshape(-1, 3)[g][:2]
      low = bv[(z_bowl + bv[:, 2] < c[2] + h) & (z_bowl + bv[:, 2] > c[2] - h)]
      if len(low):  # the YCB bowl's axis is offset from its body origin: measure the disc about the bounding-box centre
        ax = 0.5 * (bv.min(0) + bv.max(0))
        out.append((float(c[0] - ax[0]), float(c[1] - ax[1]), float(r + np.hypot(low[:, 0] - ax[0], low[:, 1] - ax[1]).max())))
    return out

  def sample_prop_initial_states(self, seed: int = 0, clearance: float = 0.003, settle_steps: int = 25, max_attempts: int = 20,
                                 spawn_z: float | None = None):
    """BASELINE config 3 initial states: banana ~ U([0.2,-0.1],[0.3,0.1]) with yaw U(+-0.1 pi) (collisions ignored), bowl ~
    U([-0.3,-0.1],[-0.2,0.1]) re-sampled up to `max_attempts` times while it would penetrate the static bowl obstacle
    (scene_pbr.xml:144-146; so100_hand_over.py:208-229), arm qpos = 0 (home is never applied, so100_task.py:308-313).  Props
    start `clearance` above their rest height and are settled on the device for `settle_steps` control steps with the arm
    command held at 0; the arm state is then restored ([upstream] PropPlacer settle_physics freezes non-prop joints).
    `spawn_z` (the reference uses 0.45 for both props, so100_hand_over.py:37-55) overrides the rest-height start: the props
    then drop ~3 cm and need ~50 settle steps.  Installs the result as the per-env reset state."""
    if self.nq != 20:
      raise RuntimeError('sample_prop_initial_states needs a SO100HandOver model')
    N, dev = self.num_envs, self.device
    g = torch.Generator(device='cpu'); g.manual_seed(int(seed))
    u = torch.rand(N, 5, generator=g)
    rest = getattr(self.task, 'rest_heights', None)
    if spawn_z is None and rest is None:  # no known rest pose (pen / holder): drop from the reference's spawn height
      spawn_z, settle_steps = 0.45, max(settle_steps, 60) if settle_steps > 0 else 0
    zo, zb = (rest[0] + clearance, rest[1] + clearance) if spawn_z is None else (float(spawn_z), float(spawn_z))
    obstacles = self._bowl_obstacles(zb)
    for _ in range(max_attempts - 1):
      bx, by = -0.3 + 0.1 * u[:, 3], -0.1 + 0.2 * u[:, 4]
      bad = torch.zeros(N, dtype=torch.bool)
      for cx, cy, rr in obstacles:
        bad |= torch.hypot(bx - cx, by - cy) < rr
      if not bool(bad.any()):
        break
      u[bad, 3:5] = torch.rand(int(bad.sum()), 2, generator=g)
    u = u.to(dev)
    q = torch.tensor(self.model['qpos0'], dtype=torch.float32, device=dev).repeat(N, 1)
    q[:, :6] = 0
    q[:, 6] = 0.2 + 0.1 * u[:, 0]; q[:, 7] = -0.1 + 0.2 * u[:, 1]; q[:, 8] = zo
    yaw = (2 * u[:, 2] - 1) * 0.1 * np.pi
    q[:, 9] = torch.cos(yaw / 2); q[:, 10] = 0; q[:, 11] = 0; q[:, 12] = torch.sin(yaw / 2)
    q[:, 13] = -0.3 + 0.1 * u[:, 3]; q[:, 14] = -0.1 + 0.2 * u[:, 4]; q[:, 15] = zb
    q[:, 16] = 1; q[:, 17:20] = 0
    v = torch.zeros(N, self.nv, dtype=torch.float32, device=dev)
    self.set_initial_state(q, v)
    if settle_steps > 0:
      self.reset()
      zero = torch.zeros(N, 6, dtype=torch.float32, device=dev)
      for _ in range(settle_steps):
        self.step(zero - torch.tensor(self.calibration_offsets, dtype=torch.float32, device=dev))
      q, v = self.get_state()
      q[:, :6] = 0; v[:, :6] = 0
      self.set_initial_state(q, v)
    self.reset()
    return q, v

  def initialize_placements(self, seed: int | None = None) -> dict:
    """initialize_episode for all envs on the device (so100_hand_over.py:320-323 with the PropPlacers :208-229): every env draws
    an object and a container pose from the task's distributions (Philox keyed on (seed, env, draw)), re-samples the container
    while it penetrates anything at its spawn pose, settles both with the arm frozen until the props' |qvel| < 1e-3 and |qacc| <
    1e-2 or 2 s have passed ([upstream] PropPlacer settle_physics), and is reset to the settled state.  One library call: the
    loop over control steps runs inside so101_sample_and_settle.  With nursery envs the following resets then draw fresh
    placements from the nursery's ring.  Returns the settle statistics."""
    if not self.task.collide:
      raise RuntimeError('initialize_placements needs a SO100HandOver model')
    seed = self.seed if seed is None else int(seed)
    st = (ctypes.c_uint64 * 4)()
    self._check(self._lib.so101_sample_and_settle(self._h, ctypes.c_uint64(seed & 0xFFFFFFFFFFFFFFFF), ctypes.byref(self._out), ctypes.byref(st), self._stream()))
    out = dict(control_steps=int(st[0]), unsettled=int(st[1]), rejected_samples=int(st[2]), attempts_exhausted=int(st[3]))
    if out['attempts_exhausted']:
      # [upstream] PropPlacer raises after max_attempts_per_prop colliding samples
      raise RuntimeError(f"Failed to place the container without collisions in {out['attempts_exhausted']} env(s) after 20 attempts")
    return out

  def placement_stats(self) -> dict:
    c = (ctypes.c_uint64 * 6)()
    self._check(self._lib.so101_placement_stats(self._h, ctypes.byref(c)))
    return dict(published=int(c[0]), consumed=int(c[1]), ring_empty_resets=int(c[2]), unsettled=int(c[3]), attempts_exhausted=int(c[4]),
                rejected_samples=int(c[5]))

  def set_reset_pool(self, qpos: torch.Tensor, qvel: torch.Tensor):
    """Install `rounds` initial states per env (qpos [rounds, N, nq], qvel [rounds, N, nv]): episode e of an env starts from
    entry e % rounds (so101_set_reset_pool).  The episode counters restart at 0."""
    q = qpos.to(device=self.device, dtype=torch.float32).contiguous(); v = qvel.to(device=self.device, dtype=torch.float32).contiguous()
    if q.dim() != 3 or q.shape[1:] != (self.num_envs, self.nq) or v.shape != (q.shape[0], self.num_envs, self.nv):
      raise ValueError(f'expected qpos [R, {self.num_envs}, {self.nq}] and qvel [R, {self.num_envs}, {self.nv}]')
    self._check(self._lib.so101_set_reset_pool(self._h, ctypes.c_void_p(q.data_ptr()), ctypes.c_void_p(v.data_ptr()), int(q.shape[0]),
                                               self._stream()))
    self.reset_rounds = int(q.shape[0])

  def randomize_resets(self, rounds: int = 4, seed: int | None = None, **sample_kwargs):
    """Batched initialize_episode (so100_hand_over.py:320-323): the reference re-samples both prop placements in EVERY reset
    (PropPlacer with the distributions at so100_hand_over.py:37-55, then a physics settle).  Here `rounds` placements per env
    are sampled, rejected against the static obstacles and settled on the device up front (sample_prop_initial_states with
    seeds seed, seed + 1, ...), and every auto-reset / reset() of an env moves on to its next placement: no host work and no
    settle inside step().  Returns the pool (qpos [rounds, N, nq], qvel [rounds, N, nv])."""
    seed = self.seed if seed is None else int(seed)
    qs, vs = [], []
    for r in range(int(rounds)):
      q, v = self.sample_prop_initial_states(seed=seed + r, **sample_kwargs)
      qs.append(q.clone()); vs.append(v.clone())
    Q, V = torch.stack(qs), torch.stack(vs)
    self.set_reset_pool(Q, V)
    self.reset()
    return Q, V


def create_batched_task_env(task_name: str, num_envs: int, time_limit: float, seed: int | None = None,
                            control_timestep: float = DEFAULT_CONTROL_TIMESTEP, cameras: tuple = (), device='cuda:0',
                            calibration_offsets=None, calibration_file: str | None = None, precision: str = 'f32',
                            solver_iterations: int = 100, solver_tolerance: float | None = None, reset_rounds: int = 1,
                            placement: str = 'device', nursery_envs: int | None = None, integrator: str = 'euler',
                            **kwargs) -> BatchedEnvironment:
  """Batched twin of task_suite.create_task_env (task_suite.py:103-155).

  For the SO100HandOver tasks the env comes back with sampled and settled prop placements, as the reference places and settles
  the props in every initialize_episode (so100_hand_over.py:208-229,320-323): a plain create -> reset -> step loop never starts
  from the blob's qpos0, where both free props sit coincident at the world origin.
    placement='device' (default): Philox sampling, collision rejection with the real narrow phase and the frozen-arm settle all
      run on the device (BatchedEnvironment.initialize_placements); `nursery_envs` extra hidden envs (default num_envs / 16)
      keep producing settled placements in the background, so every later episode starts from a fresh one.
    placement='pool': the round-1 path, `reset_rounds` placements per env sampled on the host and settled up front
      (randomize_resets); episodes cycle through them.
    placement='none' or reset_rounds=0: nothing is installed (the caller sets its own states with set_initial_state /
      set_reset_pool / sample_prop_initial_states before the first reset).
  integrator: 'euler' (default: MuJoCo's default semi-implicit Euler, which the reference runs since scene_pbr.xml sets none) or
    'implicitfast' (named by north_star; differs here through the actuators' +1 * qvel bias term, scene_pbr.xml:11)."""
  if task_name not in TASK_FACTORIES:
    raise ValueError(f'Unknown task_name: {task_name}. Available tasks: {list(TASK_FACTORIES.keys())}')  # task_suite.py:126-130
  task_class, task_kwargs = TASK_FACTORIES[task_name]
  # kwargs not in the task class's OWN constructor signature are dropped silently (task_suite.py:134-138)
  allowed = set(inspect.signature(task_class.__init__).parameters.keys()) - {'self'}
  kwargs = {k: v for k, v in kwargs.items() if k in allowed}
  kwargs.update({'control_timestep': control_timestep, 'cameras': cameras, **task_kwargs})
  task = task_class(**kwargs)
  if calibration_offsets is None and calibration_file is not None:
    calibration_offsets = SO101Calibration(calibration_file).homing_offsets
  if solver_tolerance is None:
    solver_tolerance = 1e-8 if precision == 'f64' else 1e-6
  if placement not in ('device', 'pool', 'none'):
    raise ValueError("placement must be 'device', 'pool' or 'none'")
  if not task.collide or reset_rounds <= 0:
    placement = 'none'
  nursery = 0
  if placement == 'device':
    nursery = max(1, int(num_envs) // 16) if nursery_envs is None else int(nursery_envs)
  env = BatchedEnvironment(task, num_envs, time_limit, seed, device, calibration_offsets, precision, solver_iterations, solver_tolerance,
                           nursery_envs=nursery, integrator=integrator)
  if placement == 'device':
    env.initialize_placements()
  elif placement == 'pool':
    env.randomize_resets(rounds=int(reset_rounds))
  return env


@dataclasses.dataclass
class BatchedEnvConfig:
  """The arguments of create_batched_task_env as one typed, serialisable record (run configs, sweeps, checkpoints' metadata).
  The reference passes the same things as loose keyword arguments (task_suite.create_task_env, task_suite.py:103-155)."""
  task_name: str = 'SO100HandOverBanana'
  num_envs: int = 1
  time_limit: float = 30.0
  seed: int | None = None
  control_timestep: float = DEFAULT_CONTROL_TIMESTEP
  cameras: tuple = ()
  device: str = 'cuda:0'
  calibration_offsets: tuple | None = None
  calibration_file: str | None = None
  precision: str = 'f32'
  solver_iterations: int = 100
  solver_tolerance: float | None = None
  reset_rounds: int = 1
  placement: str = 'device'
  nursery_envs: int | None = None
  integrator: str = 'euler'
  task_kwargs: dict = dataclasses.field(default_factory=dict)   # extra task constructor arguments (filtered like the reference does)

  def __post_init__(self):
    if self.task_name not in TASK_FACTORIES:
      raise ValueError(f'Unknown task_name: {self.task_name}. Available tasks: {list(TASK_FACTORIES.keys())}')
    if self.num_envs < 1:
      raise ValueError('num_envs must be >= 1')
    if self.precision not in ('f32', 'f64'):
      raise ValueError("precision must be 'f32' or 'f64'")
    if self.placement not in ('device', 'pool', 'none'):
      raise ValueError("placement must be 'device', 'pool' or 'none'")
    if self.integrator not in ('euler', 'implicitfast'):
      raise ValueError("integrator must be 'euler' or 'implicitfast'")
    self.cameras = tuple(self.cameras)
    if self.calibration_offsets is not None:
      self.calibration_offsets = tuple(float(x) for x in self.calibration_offsets)

  def to_dict(self) -> dict:
    return dataclasses.asdict(self)

  @classmethod
  def from_dict(cls, d: dict) -> 'BatchedEnvConfig':
    known = {f.name for f in dataclasses.fields(cls)}
    unknown = set(d) - known
    if unknown:
      raise ValueError(f'unknown config keys: {sorted(unknown)}')
    return cls(**d)

  def create(self) -> BatchedEnvironment:
    kw = self.to_dict()
    extra = kw.pop('task_kwargs')
    return create_batched_task_env(**kw, **extra)
