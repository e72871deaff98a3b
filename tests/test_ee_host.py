"""End-effector layer, host side: the default tool centre point of every scene, the float64 restatement of the device IK against
the oracle's kinematics, and argument validation.  No GPU needed."""
import numpy as np
import pytest

from ee_reference import ArmFK, ik, jac, mat2quat
from so101_sim_b200 import _lib
from so101_sim_b200.model import read_blob, tcp_offset
from so101_sim_b200.task_suite import IK_DEFAULTS, ee_params

BLOBS = ('so100_arm', 'so100_handover_banana', 'so100_handover_pen', 'so100_twoarm_banana')
TCP_REFERENCE = (1.37714883e-04, -8.22999677e-02, 2.14882785e-07)   # DESIGN.md: TCP of the SO100 jaws in the Fixed_Jaw frame


def _f32(d):
  return {k: float(np.float32(v)) if k != 'iterations' else v for k, v in d.items()}


@pytest.mark.parametrize('blob', BLOBS)
def test_tcp_offset_lies_between_the_jaw_pads(blob):
  m = read_blob(blob)
  narm = int(m['nu'][0]) // 6
  rng = np.random.default_rng(3)
  for arm in range(narm):
    off = tcp_offset(m, arm)
    np.testing.assert_allclose(off, TCP_REFERENCE, atol=1e-10)
    # independent check on the oracle's world kinematics: with the jaw at 0 and the arm anywhere, the TCP is the midpoint of the
    # two pad centroids in world coordinates
    fk = ArmFK(blob, arm)
    q = fk.range[:, 0] + rng.random(6) * (fk.range[:, 1] - fk.range[:, 0])
    q[5] = 0.0
    p, _ = fk.pose(q, off)
    xpos, xmat = fk.sim.field('xpos').reshape(-1, 3), fk.sim.field('xmat').reshape(-1, 3, 3)
    gb, gt, gp = m['geom_body'], m['geom_type'], m['geom_pos'].reshape(-1, 3)
    cents = []
    for b in (fk.body, int(m['jnt_body'][6 * arm + 5])):
      pads = gp[(gb == b) & (gt == 4)]
      cents.append(xpos[b] + xmat[b] @ pads.mean(axis=0))
    np.testing.assert_allclose(p, 0.5 * (cents[0] + cents[1]), atol=1e-12)


def test_tcp_offset_rejects_a_missing_arm():
  with pytest.raises(ValueError):
    tcp_offset(read_blob('so100_arm'), arm=1)


def test_oracle_jacobian_matches_finite_differences():
  fk = ArmFK('so100_arm')
  off = tcp_offset(fk.sim.meta)
  q = np.array([0.3, -1.2, 1.4, 0.4, -0.7, 0.0])
  p, _ = fk.pose(q, off)
  jp, _ = fk.jacobian(p)
  for i in range(5):
    h = 1e-6
    qp, qm = q.copy(), q.copy()
    qp[i] += h; qm[i] -= h
    np.testing.assert_allclose((fk.pose(qp, off)[0] - fk.pose(qm, off)[0]) / (2 * h), jp[:, i], atol=1e-8)
  jp_all, jr_all = jac(fk.sim, fk.body, p)
  assert jp_all.shape == (3, 6) and np.all(jr_all[:, 5] == 0)   # the jaw does not move the Fixed_Jaw


def _fk_targets(fk, off, n, seed):
  """(seed q, target p, target quat) from FK of random configurations inside 0.8 x the joint ranges, seeded 0.3 rad away."""
  rng = np.random.default_rng(seed)
  lo, hi = fk.range[:, 0], fk.range[:, 1]
  out = []
  for _ in range(n):
    qt = 0.5 * (lo + hi) + 0.4 * (hi - lo) * (2 * rng.random(6) - 1)
    p, R = fk.pose(qt, off)
    d = rng.normal(size=5)
    q0 = qt.copy()
    q0[:5] += 0.3 * d / np.linalg.norm(d)
    out.append((q0, p, mat2quat(R)))
  return out


def test_reference_ik_converges_on_reachable_targets():
  fk = ArmFK('so100_arm')
  off = tcp_offset(fk.sim.meta)
  prm = _f32(IK_DEFAULTS)
  cases = _fk_targets(fk, off, 100, seed=11)
  ok_pose = sum(ik(fk, q0, p, qq, off, **prm)[1] < 1e-4 and ik(fk, q0, p, qq, off, **prm)[2] < 1e-3 for q0, p, qq in cases)
  ok_pos = sum(ik(fk, q0, p, None, off, **prm)[1] < 1e-4 for q0, p, _ in cases)
  assert ok_pose >= 98 and ok_pos == 100, (ok_pose, ok_pos)


def test_reference_ik_stays_in_range_for_unreachable_targets():
  fk = ArmFK('so100_arm')
  off = tcp_offset(fk.sim.meta)
  q0 = np.array([0.1, -1.0, 1.0, 0.5, 0.0, 0.0])
  p, _ = fk.pose(q0, off)
  q, pe, _, it = ik(fk, q0, p + np.array([2.0, 0.0, 0.0]), None, off, **_f32(IK_DEFAULTS))
  assert it == IK_DEFAULTS['iterations'] and pe > 1.0
  assert np.all(np.isfinite(q)) and np.all(q >= fk.range[:, 0]) and np.all(q <= fk.range[:, 1])


def test_ik_tolerance_stops_early():
  fk = ArmFK('so100_arm')
  off = tcp_offset(fk.sim.meta)
  q0, p, qq = _fk_targets(fk, off, 1, seed=5)[0]
  _, pe, _, it = ik(fk, q0, p, None, off, **{**_f32(IK_DEFAULTS), 'tolerance': 1e-3})
  assert it < IK_DEFAULTS['iterations'] and pe < 1e-3


@pytest.mark.parametrize('bad', [dict(damping=0.0), dict(damping=-1.0), dict(damping=float('nan')), dict(w_rot=-0.1), dict(max_step=0.0),
                                 dict(max_step=float('inf')), dict(iterations=-1), dict(iterations=2.5), dict(tolerance=-1.0),
                                 dict(tolerance=float('nan'))])
def test_ee_params_rejects_bad_values(bad):
  with pytest.raises(ValueError):
    ee_params(TCP_REFERENCE, **bad)


@pytest.mark.parametrize('off', [(0.0, 0.0), (0.0, float('nan'), 0.0), np.zeros((2, 3))])
def test_ee_params_rejects_bad_offsets(off):
  with pytest.raises(ValueError):
    ee_params(off)


def test_ee_params_defaults():
  p = ee_params(TCP_REFERENCE)
  assert p.iterations == IK_DEFAULTS['iterations'] and p.tolerance == 0.0
  assert (p.damping, p.w_rot, p.max_step) == tuple(float(np.float32(IK_DEFAULTS[k])) for k in ('damping', 'w_rot', 'max_step'))
  assert list(p.tcp_offset) == [float(np.float32(x)) for x in TCP_REFERENCE]


def test_lerobot_wrapper_rejects_unknown_action_space():
  from so101_sim_b200.lerobot import BatchedSO101LeRobotWrapper
  with pytest.raises(ValueError):
    BatchedSO101LeRobotWrapper('SO100ArmOnly', action_space='cartesian')
  with pytest.raises(ValueError):
    BatchedSO101LeRobotWrapper('SO100ArmOnly', action_space='ee_delta', ee_base='target')


def test_ee_entry_points_are_exported(built):
  assert {'so101_ee_pose', 'so101_ee_ik'} <= set(_lib.EXPORTS)
  for narm in (1, 2):
    L = _lib.load(narm)
    # a null handle is an error, not a crash
    assert L.so101_ee_pose(None, 0, None, None, None, None) == -1
    assert L.so101_ee_ik(None, None, None, None, None, None, None, None, None) == -1
