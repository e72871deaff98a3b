"""Float64 NumPy restatement of the end-effector pose and the damped-least-squares IK of ee_kernel.cu, on the CPU oracle's
forward kinematics (xpos / xmat) and its point Jacobian so_jac.  Test infrastructure only (test_ee_host.py, test_ee_gpu.py)."""
from __future__ import annotations

import ctypes

import numpy as np

from oracle.oracle import OracleSim, lib

ARM_JOINTS = 5   # the IK moves the five arm hinges of an arm; the jaw (sixth hinge) is left to the caller's command


def _so_jac():
  f = lib().so_jac
  f.restype = None
  f.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
  return f


def jac(sim: OracleSim, body: int, point) -> tuple[np.ndarray, np.ndarray]:
  """so_jac: translational and rotational Jacobian [3, nv] of `point` (world) fixed in `body`, at the last forward()."""
  p = np.ascontiguousarray(point, dtype=np.float64)
  jp, jr = np.zeros(3 * sim.nv), np.zeros(3 * sim.nv)
  _so_jac()(sim._m, sim._d, int(body), p.ctypes.data, jp.ctypes.data, jr.ctypes.data)
  return jp.reshape(3, sim.nv), jr.reshape(3, sim.nv)


def mat2quat(R) -> np.ndarray:
  """Unit quaternion (w, x, y, z) of a rotation matrix, w >= 0."""
  R = np.asarray(R, dtype=np.float64).reshape(3, 3)
  t = np.trace(R)
  if t > 0:
    s = 2 * np.sqrt(1 + t)
    q = np.array([0.25 * s, (R[2, 1] - R[1, 2]) / s, (R[0, 2] - R[2, 0]) / s, (R[1, 0] - R[0, 1]) / s])
  elif R[0, 0] > R[1, 1] and R[0, 0] > R[2, 2]:
    s = 2 * np.sqrt(1 + R[0, 0] - R[1, 1] - R[2, 2])
    q = np.array([(R[2, 1] - R[1, 2]) / s, 0.25 * s, (R[0, 1] + R[1, 0]) / s, (R[0, 2] + R[2, 0]) / s])
  elif R[1, 1] > R[2, 2]:
    s = 2 * np.sqrt(1 + R[1, 1] - R[0, 0] - R[2, 2])
    q = np.array([(R[0, 2] - R[2, 0]) / s, (R[0, 1] + R[1, 0]) / s, 0.25 * s, (R[1, 2] + R[2, 1]) / s])
  else:
    s = 2 * np.sqrt(1 + R[2, 2] - R[0, 0] - R[1, 1])
    q = np.array([(R[1, 0] - R[0, 1]) / s, (R[0, 2] + R[2, 0]) / s, (R[1, 2] + R[2, 1]) / s, 0.25 * s])
  q /= np.linalg.norm(q)
  return -q if q[0] < 0 else q


def quat_mul(a, b) -> np.ndarray:
  w1, x1, y1, z1 = a
  w2, x2, y2, z2 = b
  return np.array([w1 * w2 - x1 * x2 - y1 * y2 - z1 * z2, w1 * x2 + x1 * w2 + y1 * z2 - z1 * y2,
                   w1 * y2 - x1 * z2 + y1 * w2 + z1 * x2, w1 * z2 + x1 * y2 - y1 * x2 + z1 * w2])


def rot_error(q_target, q_tcp) -> np.ndarray:
  """Rotation vector of R_target R_tcp^T (world frame), angle in [0, pi]."""
  qt = np.asarray(q_target, dtype=np.float64)
  qt = qt / np.linalg.norm(qt)
  d = quat_mul(qt, q_tcp * np.array([1, -1, -1, -1]))
  if d[0] < 0:
    d = -d
  s = np.linalg.norm(d[1:])
  return d[1:] * (2 * np.arctan2(s, d[0]) / s) if s > 0 else 2 * d[1:]


class ArmFK:
  """TCP pose and Jacobian of one arm of a model, from the oracle's kinematics."""

  def __init__(self, model: str, arm: int = 0):
    self.sim = OracleSim(model, collide=False)
    m = self.sim.meta
    self.arm = arm
    self.body = int(m['jnt_body'][6 * arm + 4])   # Fixed_Jaw: the body of the fifth hinge (Wrist_Roll)
    rng = m['jnt_range'].reshape(-1, 2)
    self.range = rng[6 * arm:6 * arm + 6].copy()
    self.limited = m['jnt_limited'][6 * arm:6 * arm + 6].copy()
    self.qpos0 = m['qpos0'].copy()

  def pose(self, q_arm, offset):
    """(p_tcp [3], R_tcp [3,3]) for the arm's six joint angles; every other dof at qpos0."""
    s = self.sim
    q = self.qpos0.copy()
    q[6 * self.arm:6 * self.arm + 6] = q_arm
    s.qpos[:] = q
    s.forward()
    R = s.field('xmat').reshape(-1, 9)[self.body].reshape(3, 3).copy()
    p = s.field('xpos').reshape(-1, 3)[self.body] + R @ np.asarray(offset, dtype=np.float64)
    return p, R

  def jacobian(self, p_tcp):
    jp, jr = jac(self.sim, self.body, p_tcp)
    cols = slice(6 * self.arm, 6 * self.arm + ARM_JOINTS)
    return jp[:, cols], jr[:, cols]


def ik(fk: ArmFK, q_arm, target_pos, target_quat, offset, iterations=16, damping=1e-3, w_rot=0.0, max_step=0.2, tolerance=0.0):
  """ee_ik_kernel in float64: returns (q_arm [6], position error m, orientation error rad, iterations taken)."""
  q = np.array(q_arm, dtype=np.float64)
  w = w_rot if target_quat is not None else 0.0
  tp = np.asarray(target_pos, dtype=np.float64)
  it = 0
  while True:
    p, R = fk.pose(q, offset)
    e = np.zeros(6)
    e[:3] = tp - p
    rot = rot_error(target_quat, mat2quat(R)) if target_quat is not None else np.zeros(3)
    e[3:] = w * rot
    if it == iterations or np.sqrt(e @ e) < tolerance:
      break
    jp, jr = fk.jacobian(p)
    J = np.vstack([jp, w * jr])                       # [6, 5]
    A = J @ J.T + damping * damping * np.eye(6)
    L = np.linalg.cholesky(A)
    y = np.linalg.solve(L.T, np.linalg.solve(L, e))
    dq = np.clip(J.T @ y, -max_step, max_step)
    q[:ARM_JOINTS] += dq
    lim = fk.limited[:ARM_JOINTS] != 0
    q[:ARM_JOINTS][lim] = np.clip(q[:ARM_JOINTS][lim], fk.range[:ARM_JOINTS, 0][lim], fk.range[:ARM_JOINTS, 1][lim])
    it += 1
  return q, float(np.linalg.norm(e[:3])), float(np.linalg.norm(rot)) if target_quat is not None else 0.0, it
