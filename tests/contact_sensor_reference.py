"""float64 NumPy restatement of the contact sensor readout (so101_contact_sensors) over the oracle's contact list and efc_force.

A sensor is a pair of disjoint body sets (A, B).  For a contact between geom1 (body b1) and geom2 (body b2) with cone force f in
the contact frame (rows: normal from geom1 to geom2, tangent 1, tangent 2), the force on b2 from b1 is F = f0 n + f1 t1 + f2 t2;
the contact adds +F when b2 is in A and b1 in B, -F when b1 is in A and b2 in B, and in both cases f0 to the normal sum and 1 to
the count.  Torsional and rolling components (condim 4 / 6) are torques and are left out."""
import numpy as np


def readout(meta, contacts, efc_force, pairs):
  """contacts: OracleSim.contacts() of the substep whose efc_force is given; pairs: [(A, B)] of body id collections ->
  float64 [K, 5]: net force on A from B (3), normal force sum, contact count."""
  gb = meta['geom_body']
  sets = [(set(int(x) for x in a), set(int(x) for x in b)) for a, b in pairs]
  out = np.zeros((len(sets), 5))
  for c in contacts:
    b1, b2 = int(gb[c['geom1']]), int(gb[c['geom2']])
    adr, dim = c['efc_address'], c['dim']
    f = np.zeros(3)
    f[:min(dim, 3)] = efc_force[adr:adr + min(dim, 3)]
    F = c['frame'][0] * f[0] + c['frame'][1] * f[1] + c['frame'][2] * f[2]
    for k, (A, B) in enumerate(sets):
      if b2 in A and b1 in B:
        out[k, :3] += F
      elif b1 in A and b2 in B:
        out[k, :3] -= F
      else:
        continue
      out[k, 3] += f[0]
      out[k, 4] += 1
  return out


def others(meta, side):
  """Every body of the model that is not in `side`."""
  return sorted(set(range(int(meta['nbody'][0]))) - set(int(x) for x in side))


def jaw_object_state(model='so100_handover_banana', bowl_xy=(-0.3, 0.0)):
  """A pre-substep state (dict q, v, a, curved like test_solver_tiers_gpu.harvest's records) in which a jaw presses on the
  object: the harvest's random-action rollouts never touch the banana with a jaw away from the curved static obstacles.  The
  arms stand at q = 0 and the bowl rests on the table at bowl_xy, clear of the static obstacles.  The banana, at rest, is
  raised under arm 0's Fixed_Jaw body origin in 1 mm steps from 15 cm below it until the oracle's collision pass finds the
  first contact between a jaw and the banana, then 2 mm further, where the jaw contacts carry force (at first touch they sit
  inside the margin with zero force).  The banana touches nothing else; the other contacts are the bowl's on the table."""
  from oracle.oracle import OracleSim
  from so101_sim_b200.model import body_set
  from test_solver_tiers_gpu import curved_static_geoms
  o = OracleSim(model, collide=True)
  m = o.meta
  na, gb = int(m['nu'][0]), m['geom_body']
  jaws, obj = set(body_set(m, 'gripper')), set(body_set(m, 'object'))
  q = np.array(m['qpos0'], dtype=np.float64)
  q[:na] = 0
  q[na:na + 3] = (0.3, 0.15, 0.6)
  q[na + 7:na + 14] = [bowl_xy[0], bowl_xy[1], 0.4226, 1, 0, 0, 0]
  o.set_state(q, np.zeros(o.nv)); o.forward()
  xp = o.field('xpos').reshape(-1, 3)[body_set(m, 'fixed_jaw')[0]].copy()
  curved = curved_static_geoms(m)
  for z in xp[2] - 0.15 + 0.001 * np.arange(200):
    q[na:na + 3] = (xp[0], xp[1], z)
    o.set_state(q, np.zeros(o.nv)); o.forward()
    cons = o.contacts()
    if any({gb[c['geom1']], gb[c['geom2']]} & jaws and {gb[c['geom1']], gb[c['geom2']]} & obj for c in cons):
      q[na + 2] += 0.002
      o.set_state(q, np.zeros(o.nv)); o.forward()
      cons = o.contacts()
      return dict(q=q.copy(), v=np.zeros(o.nv), a=np.zeros(na), curved=any(c['geom1'] in curved or c['geom2'] in curved for c in cons))
  raise RuntimeError('no jaw / object contact found')
