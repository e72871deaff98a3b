"""Batched twins of the reference's LeRobot adapter and scripted dataset generator (SURVEY.md §8 a19 and §8f row 2).

  * `BatchedSO101LeRobotWrapper`   scripts/so101_lerobot_wrapper.py:15-188 — TimeStep -> LeRobot-style dict of torch tensors
    with a leading env dimension (`observation.state` = delayed `joints_pos`, action echo, frame / episode indices and the
    reference's `timestamp = frame_index * 0.1`).  State-only: camera rendering is out of scope of the B200 path, so
    `cameras` must be `()` and no `observation.images.*` keys are produced.
  * `BatchedTrajectoryPlanner`, `BatchedDatasetGenerator`   examples/automated_lerobot_dataset_generator.py:52-483 — the
    randomised scripted pick-and-place waypoints (approach / descend / grasp / lift / move / lower / release / retreat with
    the reference's geometric "IK", smooth-step interpolation and waypoint noise), its distance-based grasp-failure test and
    its episode records, for N environments in lockstep.  As in the reference the sampled spawn positions only steer the
    script; they are never written into the simulation (automated_lerobot_dataset_generator.py:367-371).

Everything here is host-side scripting over torch tensors; the physics is `BatchedEnvironment.step` (C-ABI -> CUDA kernels).
"""
from __future__ import annotations

import dataclasses
import math
from typing import Any, Dict, List, Optional

import numpy as np
import torch

from . import task_suite

TABLE_Z = 0.42  # automated_lerobot_dataset_generator.py:68,76,197


def convert_to_lerobot_format(joints_pos: torch.Tensor, action: Optional[torch.Tensor], frame_index: int, episode_index: int,
                              device=None, action_dim: int = 6) -> Dict[str, Any]:
  """so101_lerobot_wrapper.py:77-122 for a batch: `joints_pos` [N,6] (the delayed observation), `action` [N,action_dim] or None
  (the reset observation echoes a zero action)."""
  n = joints_pos.shape[0]
  dev = joints_pos.device if device is None else torch.device(device)
  out: Dict[str, Any] = {}
  # copies: the env re-uses its observation buffers from step to step, a recorded frame must not alias them
  out['observation.state'] = joints_pos.to(device=dev, dtype=torch.float32, copy=True)
  out['action'] = torch.zeros(n, action_dim, device=dev) if action is None else action.to(device=dev, dtype=torch.float32, copy=True)
  out['timestamp'] = torch.full((n,), frame_index * 0.1, dtype=torch.float32, device=dev)  # (sic: 0.1, not the 0.02 s control step)
  out['frame_index'] = torch.full((n,), frame_index, dtype=torch.long, device=dev)
  out['episode_index'] = torch.full((n,), episode_index, dtype=torch.long, device=dev)
  out['index'] = torch.full((n,), frame_index, dtype=torch.long, device=dev)
  out['task_index'] = torch.zeros(n, dtype=torch.long, device=dev)
  out['task'] = 'SO100 manipulation task'
  return out


class BatchedSO101LeRobotWrapper:
  """N lockstep copies of SO101LeRobotWrapper (scripts/so101_lerobot_wrapper.py:15-188).

  action_space='joint' (default): actions are joint targets [N,6], as in the reference.  action_space='ee_delta': actions are
  end-effector deltas [N,4] per arm, (dx, dy, dz) of the tool centre point in metres and the jaw action, run through
  BatchedEnvironment.step_ee from the current TCP (`ee_base`), clipped to the `ee_workspace` box ((lo[3], hi[3]) or None), with
  the IK parameters `ee_params`; the recorded 'action' is the [N,4] delta action."""

  ACTION_SPACES = ('joint', 'ee_delta')
  action_space = 'joint'

  def __init__(self, task_name: str = 'SO100HandOverBanana', num_envs: int = 1, cameras: tuple = (), camera_resolution: tuple = (480, 640),
               time_limit: float = 30.0, device: str = 'cuda:0', seed: int | None = None, reset_rounds: int = 1, action_space: str = 'joint',
               ee_workspace=None, ee_base: str = 'state', ee_params: Optional[dict] = None, **env_kwargs):
    if cameras:
      raise NotImplementedError('camera rendering is out of scope of the B200 path: pass cameras=()')
    if action_space not in self.ACTION_SPACES:
      raise ValueError(f'action_space must be one of {self.ACTION_SPACES}, got {action_space!r}')
    if ee_base not in ('state', 'command'):
      raise ValueError("ee_base must be 'state' or 'command'")
    self.action_space = action_space
    self.ee_workspace, self.ee_base, self.ee_params = ee_workspace, ee_base, dict(ee_params or {})
    self.device = device
    self.cameras = tuple(cameras)
    self.camera_resolution = camera_resolution
    self.use_actual_camera_names = True
    # camera_resolution / image_observation_enabled are dropped by the factory's kwargs filter exactly as in the reference
    # (so101_lerobot_wrapper.py:43-49, task_suite.py:134-138)
    self.env = task_suite.create_batched_task_env(task_name=task_name, num_envs=num_envs, time_limit=time_limit, seed=seed, cameras=cameras,
                                                  camera_resolution=camera_resolution, image_observation_enabled=True, device=device,
                                                  reset_rounds=reset_rounds, **env_kwargs)
    self.num_envs = self.env.num_envs
    self.episode_index = 0
    self.frame_index = 0
    self.start_time = 0.0

  def reset(self) -> Dict[str, Any]:
    ts = self.env.reset()
    self.frame_index = 0
    self.start_time = 0.0
    return convert_to_lerobot_format(ts.observation['joints_pos'], None, self.frame_index, self.episode_index, self.device,
                                     4 * self.env.narm if self.action_space == 'ee_delta' else 6)

  def step(self, action) -> Dict[str, Any]:
    if self.action_space == 'ee_delta':
      return self._step_ee(action)
    action = torch.as_tensor(np.asarray(action) if not isinstance(action, torch.Tensor) else action, dtype=torch.float32)
    if action.dim() == 1:
      action = action.expand(self.num_envs, 6)
    ts = self.env.step(action.to(self.device))
    self.last_timestep = ts
    self.frame_index += 1
    return convert_to_lerobot_format(ts.observation['joints_pos'], action, self.frame_index, self.episode_index, self.device)

  def _step_ee(self, action) -> Dict[str, Any]:
    na = self.env.narm
    action = (action if isinstance(action, torch.Tensor) else torch.as_tensor(np.asarray(action))).to(device=self.device, dtype=torch.float32)
    if action.dim() == 1:
      action = action.expand(self.num_envs, 4 * na)
    if tuple(action.shape) != (self.num_envs, 4 * na):
      raise ValueError(f'ee_delta actions must have shape [{self.num_envs}, {4 * na}] or [{4 * na}], got {list(action.shape)}')
    a = action.reshape(self.num_envs, na, 4)
    ts = self.env.step_ee(a[..., :3], a[..., 3], base=self.ee_base, workspace=self.ee_workspace, **self.ee_params)
    self.last_timestep = ts
    self.frame_index += 1
    return convert_to_lerobot_format(ts.observation['joints_pos'], action, self.frame_index, self.episode_index, self.device, 4 * na)

  def collect_episode(self, actions, save_path: Optional[str] = None) -> List[Dict[str, Any]]:
    """so101_lerobot_wrapper.py:124-158; `actions` is a sequence of [N,6] (or [6]) actions."""
    episode = [self.reset()]
    for a in actions:
      episode.append(self.step(a))
    if save_path:
      torch.save(episode, save_path)
    self.episode_index += 1
    return episode

  def get_action_spec(self) -> Dict[str, Any]:  # so101_lerobot_wrapper.py:160-168
    if self.action_space == 'ee_delta':
      lo, hi = (None, None) if self.ee_workspace is None else (np.asarray(self.ee_workspace[0]), np.asarray(self.ee_workspace[1]))
      return {'shape': (4 * self.env.narm,), 'dtype': np.float32, 'workspace_low': lo, 'workspace_high': hi,
              'names': [f'{n}{"" if self.env.narm == 1 else f"_{k}"}' for k in range(self.env.narm) for n in ('delta_x', 'delta_y', 'delta_z', 'gripper')]}
    return {'shape': (6,), 'dtype': np.float32, 'low': -1.0, 'high': 1.0,
            'names': ['rotation', 'pitch', 'elbow', 'wrist_pitch', 'wrist_roll', 'jaw']}

  def get_observation_spec(self) -> Dict[str, Any]:  # so101_lerobot_wrapper.py:170-188
    return {'images': {}, 'state': {'shape': (6,), 'dtype': np.float32, 'names': [f'joint_{i}' for i in range(6)]}}


# ------------------------------------------------------------------------------------------------ scripted dataset generator
@dataclasses.dataclass
class DatasetConfig:
  """automated_lerobot_dataset_generator.py:23-50 (fields the state-only twin uses)."""
  num_episodes: int = 10
  max_episode_length: int = 50
  banana_spawn_radius: float = 0.25
  bowl_spawn_radius: float = 0.30
  robot_pose_variation: float = 0.2
  approach_height: float = 0.1
  lift_height: float = 0.15
  grasp_success_threshold: float = 0.05
  bowl_success_threshold: float = 0.08
  settling_time: int = 10


class BatchedTrajectoryPlanner:
  """automated_lerobot_dataset_generator.py:52-230 for N environments at once (torch, any device)."""

  JOINT_LIMITS = ((-3.14, 3.14), (-2.5, 0.5), (0.5, 2.5), (0.5, 2.5), (-3.14, 3.14), (0.0, 0.08))  # :93-100
  BASE_POSE = (0.0, -1.57, 1.57, 1.57, -1.57, 0.0)                                                    # :82

  def __init__(self, config: DatasetConfig, homing_offsets=None, generator: torch.Generator | None = None, device='cpu'):
    self.config = config
    self.device = torch.device(device)
    self.gen = generator
    off = np.zeros(6) if homing_offsets is None else np.asarray(homing_offsets, dtype=np.float64)
    self.offsets = torch.tensor(off, dtype=torch.float32, device=self.device)

  def _uniform(self, n, lo, hi):
    return lo + (hi - lo) * torch.rand(n, generator=self.gen, device=self.device)

  def randomize_spawn_positions(self, n: int):
    """:57-78 — banana in a 60 degree front arc, bowl at a second random angle; z = table height."""
    c = self.config
    ba = self._uniform(n, -math.pi / 3, math.pi / 3)
    bd = self._uniform(n, 0.15, c.banana_spawn_radius)
    banana = torch.stack([bd * torch.sin(ba), bd * torch.cos(ba), torch.full_like(bd, TABLE_Z)], dim=1)
    wa = ba + self._uniform(n, -math.pi / 2, math.pi / 2)
    wd = self._uniform(n, 0.12, c.bowl_spawn_radius)
    bowl = torch.stack([wd * torch.sin(wa), wd * torch.cos(wa), torch.full_like(wd, TABLE_Z)], dim=1)
    return banana, bowl

  def randomize_robot_start_pose(self, n: int):
    """:80-106 — home pose + U(+-variation) per joint, clamped to the script's joint limits."""
    v = self.config.robot_pose_variation
    pose = torch.tensor(self.BASE_POSE, device=self.device).expand(n, 6) + (2 * torch.rand(n, 6, generator=self.gen, device=self.device) - 1) * v
    lo = torch.tensor([l for l, _ in self.JOINT_LIMITS], device=self.device); hi = torch.tensor([h for _, h in self.JOINT_LIMITS], device=self.device)
    return torch.minimum(torch.maximum(pose, lo), hi)

  def inverse_kinematics_approximate(self, target: torch.Tensor) -> torch.Tensor:
    """:188-212 — the reference's geometric stand-in for IK, then the calibration offsets (so101_calibration.py:62-77)."""
    x, y, z = target[:, 0], target[:, 1], target[:, 2]
    base = torch.atan2(x, y)
    horiz = torch.sqrt(x * x + y * y)
    vert = z - TABLE_Z
    shoulder = -torch.atan2(vert, horiz) - 0.5
    elbow = math.pi / 2 + torch.atan2(vert, horiz)
    wrist = math.pi / 2 - shoulder - elbow
    zeros = torch.zeros_like(x)
    return torch.stack([base, shoulder, elbow, wrist, zeros, zeros], dim=1) + self.offsets

  def interpolate(self, start: torch.Tensor, end: torch.Tensor, steps: int) -> List[torch.Tensor]:
    """:214-226 — smooth-step easing plus N(0, 0.02) joint noise (none on the gripper) that fades towards the target."""
    out = []
    for i in range(steps):
      t = (i + 1) / steps
      st = t * t * (3 - 2 * t)
      noise = 0.02 * torch.randn(start.shape[0], 6, generator=self.gen, device=self.device)
      noise[:, 5] = 0
      out.append(start + st * (end - start) + noise * (1 - st))
    return out

  def plan_pickup_trajectory(self, start: torch.Tensor, banana: torch.Tensor) -> List[torch.Tensor]:
    """:114-144 — 8 approach + 5 descent + 3 grasp + 5 lift waypoints."""
    c = self.config
    up = lambda dz: banana + torch.tensor([0.0, 0.0, dz], device=self.device)
    wp = self.interpolate(start, self.inverse_kinematics_approximate(up(c.approach_height)), 8)
    grasp = self.inverse_kinematics_approximate(up(0.02))
    wp += self.interpolate(wp[-1], grasp, 5)
    closed = grasp.clone(); closed[:, 5] = 0.05
    wp += self.interpolate(wp[-1], closed, 3)
    lift = self.inverse_kinematics_approximate(up(c.lift_height)); lift[:, 5] = 0.05
    wp += self.interpolate(wp[-1], lift, 5)
    return wp

  def plan_placement_trajectory(self, start: torch.Tensor, bowl: torch.Tensor) -> List[torch.Tensor]:
    """:146-186 — 8 move + 4 lower + 3 release + 5 retreat waypoints."""
    c = self.config
    up = lambda dz: bowl + torch.tensor([0.0, 0.0, dz], device=self.device)
    above = self.inverse_kinematics_approximate(up(c.lift_height)); above[:, 5] = 0.05
    wp = self.interpolate(start, above, 8)
    drop = self.inverse_kinematics_approximate(up(0.05)); drop[:, 5] = 0.05
    wp += self.interpolate(wp[-1], drop, 4)
    release = drop.clone(); release[:, 5] = 0.0
    wp += self.interpolate(wp[-1], release, 3)
    retreat = self.inverse_kinematics_approximate(up(c.lift_height)); retreat[:, 5] = 0.0
    wp += self.interpolate(wp[-1], retreat, 5)
    return wp

  def detect_grasp_failure(self, robot_pos: torch.Tensor, banana: torch.Tensor, gripper: torch.Tensor) -> torch.Tensor:
    """:238-241 — the reference compares the first three JOINT values with the banana position (sic)."""
    return ((robot_pos - banana).norm(dim=1) > self.config.grasp_success_threshold) | (gripper < 0.02)


class BatchedDatasetGenerator:
  """AutomatedLeRobotDatasetGenerator._generate_single_episode (:350-483) for N environments in lockstep.  One call to
  `generate_episodes()` produces N episode records (state-only observations); envs whose scripted grasp check fails end after
  the pick-up phase exactly as in the reference (`failure_reason = 'grasp_failed'`), the others run placement + settling and are
  marked successful with a final reward of 1 (the reference assumes success when no failure was detected, :446-452)."""

  def __init__(self, config: DatasetConfig, wrapper: BatchedSO101LeRobotWrapper, seed: int = 0, homing_offsets=None):
    self.config = config
    self.wrapper = wrapper
    dev = torch.device(wrapper.device)
    self.gen = torch.Generator(device=dev); self.gen.manual_seed(int(seed))
    self.planner = BatchedTrajectoryPlanner(config, homing_offsets, self.gen, dev)
    self.episode_counter = 0

  def generate_episodes(self) -> Dict[str, Any]:
    c, w, n = self.config, self.wrapper, self.wrapper.num_envs
    banana, bowl = self.planner.randomize_spawn_positions(n)
    start = self.planner.randomize_robot_start_pose(n)
    w.reset()
    obs = w.step(start)
    states, actions = [obs['observation.state']], []

    def run(waypoints):
      for wp in waypoints:
        if len(actions) >= c.max_episode_length:
          break
        o = w.step(wp)
        states.append(o['observation.state']); actions.append(wp)

    run(self.planner.plan_pickup_trajectory(start, banana))
    n_pick = len(actions)
    cur = states[-1]
    failed = self.planner.detect_grasp_failure(cur[:, :3], banana, cur[:, 5])
    place = self.planner.plan_placement_trajectory(cur, bowl)
    run(place)
    run([place[-1]] * c.settling_time)  # hold the last waypoint while the physics settles (:433-445)
    T = len(actions)
    length = torch.where(failed, torch.full((n,), n_pick, device=failed.device), torch.full((n,), T, device=failed.device))
    S, A = torch.stack(states), torch.stack(actions)  # [T+1, N, 6], [T, N, 6]
    t_idx = torch.arange(T, device=A.device)[:, None]
    valid = t_idx < length[None, :]
    rewards = ((t_idx == (length - 1)[None, :]) & ~failed[None, :]).float()  # final reward 1 on the last step of a success
    dones = torch.zeros(T + 1, n, dtype=torch.bool, device=A.device)
    dones[length, torch.arange(n, device=A.device)] = True                   # the last recorded observation is marked done
    first = self.episode_counter + 1
    self.episode_counter += n
    w.episode_index += 1
    return {'observations': {'state': S}, 'actions': A, 'rewards': rewards, 'dones': dones, 'valid': valid, 'length': length,
            'episode_metadata': {'episode_ids': [f'episode_{first + i}' for i in range(n)], 'task_name': 'BananaPickAndPlace',
                                 'success': ~failed, 'failure_reason': ['grasp_failed' if f else None for f in failed.tolist()],
                                 'initial_banana_pos': banana, 'initial_bowl_pos': bowl, 'start_robot_pose': start}}

  def generate_dataset(self, save_path: Optional[str] = None) -> List[Dict[str, Any]]:
    """Batches of N episodes until `num_episodes` successful ones exist (or the reference's attempt cap is hit, :332-335)."""
    out, ok = [], 0
    while ok < self.config.num_episodes and self.episode_counter <= self.config.num_episodes * 6 + self.wrapper.num_envs:
      ep = self.generate_episodes()
      out.append(ep)
      ok += int(ep['episode_metadata']['success'].sum())
    if save_path:
      torch.save(out, save_path)
    return out
