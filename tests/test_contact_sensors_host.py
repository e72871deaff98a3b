"""Contact sensors without a GPU: the named body sets of every model blob, and the float64 restatement of the readout
(tests/contact_sensor_reference.py) over the oracle's own contacts and efc_force against the closed forms of
tests/kat_analytic.py, to the 1e-6 bar of tests/test_oracle_analytic.py."""
import numpy as np
import pytest

import contact_sensor_reference as csr
import kat_analytic as ka
from oracle.oracle import OracleSim
from so101_sim_b200.model import body_set, read_blob


@pytest.mark.parametrize('blob', ['so100_handover_banana', 'so100_handover_pen'])
def test_body_sets_of_the_one_arm_scenes(blob):
  m = read_blob(blob)
  assert body_set(m, 'fixed_jaw') == [6] and body_set(m, 'moving_jaw') == [7] and body_set(m, 'gripper') == [6, 7]
  assert body_set(m, 'arm') == [2, 3, 4, 5, 6, 7]
  assert body_set(m, 'object') == [11] and body_set(m, 'container') == [12]
  assert body_set(m, 'static') == [0, 1, 8, 9, 10]
  with pytest.raises(ValueError):
    body_set(m, 'gripper', arm=1)


def test_body_sets_of_the_two_arm_scene():
  m = read_blob('so100_twoarm_banana')
  assert body_set(m, 'fixed_jaw', 0) == [6] and body_set(m, 'moving_jaw', 0) == [7]
  assert body_set(m, 'fixed_jaw', 1) == [13] and body_set(m, 'moving_jaw', 1) == [14] and body_set(m, 'gripper', 1) == [13, 14]
  assert body_set(m, 'arm', 1) == [9, 10, 11, 12, 13, 14]
  assert body_set(m, 'object') == [18] and body_set(m, 'container') == [19]
  assert body_set(m, 'static') == [0, 1, 8, 15, 16, 17]
  with pytest.raises(ValueError):
    body_set(m, 'arm', arm=2)


def test_body_sets_of_the_arm_only_model():
  m = read_blob('so100_arm')
  assert body_set(m, 'gripper') == [6, 7]
  for name in ('object', 'container'):
    with pytest.raises(ValueError):
      body_set(m, name)
  with pytest.raises(ValueError):
    body_set(m, 'jaws')


def _settle(o, q, steps):
  o.set_state(q, np.zeros(18))
  for _ in range(steps):
    o.control_step(np.zeros(6))


def test_reference_readout_of_a_resting_box_carries_its_weight():
  """Box flat on the table: (box, others) = (0, 0, m_box g), normal sum m_box g, 4 contacts."""
  o = OracleSim(ka.BLOB, collide=True)
  _settle(o, ka.scene_state(o.meta['qpos0'], (0.25, 0.0, ka.TABLE_TOP + ka.BOX_HALF[2])), 100)
  box = body_set(o.meta, 'object')
  r = csr.readout(o.meta, o.contacts(), o.field('efc_force'), [(box, csr.others(o.meta, box))])[0]
  w = ka.BOX_MASS * ka.G
  print('reference readout of the resting box / m g:', r[:4] / w, r[4])
  assert r[4] == 4
  assert abs(r[2] / w - 1) < 1e-6 and abs(r[3] / w - 1) < 1e-6 and np.abs(r[:2]).max() < 1e-6 * w


def test_reference_readout_of_the_stack_passes_the_load_down():
  """Capsule on box on table: (capsule, box) carries m_cap g, (box, static) (m_box + m_cap) g, (box, capsule) is the negation of
  (capsule, box)."""
  o = OracleSim(ka.BLOB, collide=True)
  _settle(o, ka.stack_state(o.meta['qpos0']), 150)
  box, cap, static = body_set(o.meta, 'object'), body_set(o.meta, 'container'), body_set(o.meta, 'static')
  r = csr.readout(o.meta, o.contacts(), o.field('efc_force'), [(cap, box), (box, static), (box, cap)])
  wc, wb = ka.CAP_MASS * ka.G, (ka.BOX_MASS + ka.CAP_MASS) * ka.G
  assert r[0, 4] == 2 and r[1, 4] == 4
  assert abs(r[0, 2] / wc - 1) < 1e-6 and abs(r[0, 3] / wc - 1) < 1e-6
  assert abs(r[1, 2] / wb - 1) < 1e-6 and abs(r[1, 3] / wb - 1) < 1e-6
  assert np.array_equal(r[2, :3], -r[0, :3]) and np.array_equal(r[2, 3:], r[0, 3:])
