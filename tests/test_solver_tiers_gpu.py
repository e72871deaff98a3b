"""Newton solver tiers 1 and 2 against the float64 oracle, and the same envs solved in every tier.

scene_classify_kernel sends each env to a solver tier by its raw contact count n and Jacobian-block count nblk: tier 0 for
n <= 32 and nblk <= 36, tier 1 for n <= 64 and nblk <= 80, tier 2 up to CONBUF = 128 contacts and 160 blocks.  Only envs with
more than 32 contacts run the multi-register rank sort of gather_contacts, build_rows' block allocation across 32-contact
chunks, multi-word body masks in assemble and in the decoupled test, and the persistent queue walk of the tier kernels.

The states come from a deterministic harvest of oracle rollouts (CPU only): random actions at 0.6 x ctrlrange, props placed in
the arm's reach, the banana often dropped into the bowl.  Each pre-substep state is classified with the classifier's own rule,
and a batch is kept with a few states of every class: each tier, the tier edges (exactly 32, 33, 64, 65 contacts), tier 1 by
blocks only, and coupled / decoupled Hessians.  The GPU tests solve that batch for one substep against a fresh oracle per state,
roll tier-2 states forward, and check that forcing envs into a larger tier (SO101_SOLVE_TIER_MIN) changes no bit."""
import functools

import numpy as np
import pytest
import torch

from oracle.oracle import OracleSim

DEV = 'cuda:0'
CONBUF, NB_L = 128, 160   # raw contacts per env (scene_collide.cuh) and Jacobian blocks of solver tier 2 (scene_kernel.inl)
TASKS = {'so100_handover_banana': 'SO100HandOverBanana', 'so100_twoarm_banana': 'SO100TwoArmHandOverBanana'}
MODELS = tuple(TASKS)


# ------------------------------------------------------------------------------------------------ harvester (CPU)
def geom_blocks(meta):
  """Jacobian block of each geom's body, as scene_classify_kernel counts them: None for static bodies, one block per arm
  (body_slot / 6 for the arm links), one per prop.  body_slot of a body is the index of its joint (scene_model.cuh)."""
  na = int(meta['nu'][0])
  slot = {int(b): j for j, b in enumerate(meta['jnt_body'])}
  blk = []
  for b in meta['geom_body']:
    s = slot.get(int(b), -1)
    blk.append(None if s < 0 else (s // 6 if s < na else s))
  return blk


def classify(contacts, gblk):
  """(n, nblk, tier, coupled) of a contact list: scene_classify_kernel's rule; coupled = a contact between two dynamic blocks."""
  n, nblk, coupled = len(contacts), 0, False
  for c in contacts:
    a1, a2 = gblk[c['geom1']], gblk[c['geom2']]
    nblk += (a1 is not None) + (a2 is not None and a2 != a1)
    coupled |= a1 is not None and a2 is not None and a1 != a2
  tier = 0 if (n <= 32 and nblk <= 36) else (1 if (n <= 64 and nblk <= 80) else 2)
  return n, nblk, tier, coupled


def curved_static_geoms(meta):
  """Static capsules / cylinders (scene_pbr.xml:141-146): EPA on a curved surface terminates by tolerance, so its contact
  normal is sensitive to FMA-level round-off (see test_scene_gpu.test_f64_scene_matches_oracle)."""
  gbody, gtype = meta['geom_body'], meta['geom_type']
  return {g for g in range(len(gtype)) if gtype[g] in (2, 3) and meta['body_weld'][gbody[g]] == 0}


# (the two-arm rollouts are 2x as expensive per substep and reach the larger tiers more often)
ROLLOUTS = {'so100_handover_banana': (40, 30), 'so100_twoarm_banana': (20, 30)}   # episodes, control steps of 10 substeps


@functools.lru_cache(maxsize=None)
def harvest(model):
  """Every pre-substep state of deterministic oracle rollouts as dicts (q, v, a, n, nblk, tier, coupled, curved).  States that
  would overflow CONBUF or tier 2's block pool (out of scope here: contacts beyond them are dropped) are left out.
  The contacts of a substep's own forward pass are those of its starting state, so they are read after so_substep."""
  o = OracleSim(model, collide=True)
  m = o.meta
  gblk, curved = geom_blocks(m), curved_static_geoms(m)
  na = o.nu
  lo, hi = m['act_ctrlrange'].reshape(-1, 2)[:na, 0], m['act_ctrlrange'].reshape(-1, 2)[:na, 1]
  rng = np.random.RandomState(1234)
  episodes, steps = ROLLOUTS[model]
  out = []
  for _ in range(episodes):
    q = np.array(m['qpos0'], dtype=np.float64)
    q[:na] = 0
    bx, by = rng.uniform(-0.25, -0.12), rng.uniform(-0.15, 0.15)
    q[na + 7:na + 14] = [bx, by, 0.4226 + 0.001, 1, 0, 0, 0]                       # bowl just above its rest height
    if rng.rand() < 0.8:                                                             # banana dropped into the bowl
      q[na:na + 7] = [bx - 0.0255, by - 0.0675, 0.4226 + rng.uniform(0.03, 0.06), np.cos(0.4), 0, 0, np.sin(0.4)]
    else:                                                                            # banana on the table
      yaw = rng.uniform(-0.3, 0.3)
      q[na:na + 7] = [rng.uniform(0.12, 0.3), rng.uniform(-0.15, 0.15), 0.4217 + 0.001, np.cos(yaw / 2), 0, 0, np.sin(yaw / 2)]
    o.set_state(q, np.zeros(o.nv))
    for _ in range(steps):
      a = ((lo + rng.rand(na) * (hi - lo)) * 0.6).astype(np.float32).astype(np.float64)   # the GPU gets float32 actions
      o.ctrl[:] = a
      for _ in range(10):
        q0, v0 = o.qpos.copy(), o.qvel.copy()
        o.substep()
        cons = o.contacts()
        n, nblk, tier, coupled = classify(cons, gblk)
        if n <= CONBUF and nblk <= NB_L:
          on_curved = any(c['geom1'] in curved or c['geom2'] in curved for c in cons)
          out.append(dict(q=q0, v=v0, a=a, n=n, nblk=nblk, tier=tier, coupled=coupled, curved=on_curved))
  return out


CLASSES = {
    'tier0': lambda r: r['tier'] == 0,
    'tier1_count': lambda r: r['tier'] == 1 and r['n'] > 32,
    'tier1_blocks': lambda r: r['tier'] == 1 and r['n'] <= 32,   # nblk > 36 with few contacts: the arm and both props coupled
    'tier2': lambda r: r['tier'] == 2,
    'n32': lambda r: r['n'] == 32,
    'n33': lambda r: r['n'] == 33,
    'n64': lambda r: r['n'] == 64,
    'n65': lambda r: r['n'] == 65,
    'coupled': lambda r: r['coupled'],
    'decoupled': lambda r: not r['coupled'] and r['n'] > 0,
}
PER_CLASS = 6

# Harvest indices left out of the batch after selection, measured on a B200: states where the float64 CUDA path and the oracle
# legitimately part ways for reasons that have nothing to do with the solver tier (both give the same answer in every tier).
EXCLUDED = {
    'so100_handover_banana': {
        417: 'gripper jaw box 7 mm deep in a bowl hull: ill-conditioned EPA, the GPU picks a face 2 mm off the oracle\'s',
        2959: 'more candidate geom pairs than the broad phase holds (PAIRCAP): the GPU drops one pair, 61 instead of 66 contacts',
    },
    'so100_twoarm_banana': {
        5999: 'ends at the Newton tolerance boundary: 14 instead of 12 iterations, qpos / qvel within 1e-12 of the oracle',
    },
}


@functools.lru_cache(maxsize=None)
def batch(model):
  """Harvested states to solve: for each class in turn, states spread evenly over the harvest until the batch holds PER_CLASS
  of that class (or all of them); then the EXCLUDED ones are dropped."""
  recs = harvest(model)
  chosen = []
  for pred in CLASSES.values():
    members = [i for i, r in enumerate(recs) if pred(r)]
    have = sum(1 for i in chosen if pred(recs[i]))
    for i in (members[int(k)] for k in np.linspace(0, len(members) - 1, min(PER_CLASS, len(members)))) if members else ():
      if have >= PER_CLASS:
        break
      if i not in chosen:
        chosen.append(i); have += 1
  return tuple(recs[i] for i in sorted(chosen) if i not in EXCLUDED[model])


@pytest.mark.parametrize('model', MODELS)
def test_harvest_covers_every_solver_tier_and_edge(model):
  """CPU: the harvest reaches every class the GPU tests need, and the batch keeps a few states of each, so that a change of a
  model blob or of the oracle cannot silently take a solver tier out of the GPU tests."""
  recs = harvest(model)
  counts = {k: sum(1 for r in recs if p(r)) for k, p in CLASSES.items()}
  kept = {k: sum(1 for r in batch(model) if p(r)) for k, p in CLASSES.items()}
  print(model, len(recs), 'states; per class (harvest / batch):', {k: (counts[k], kept[k]) for k in CLASSES}, 'batch', len(batch(model)))
  for k in CLASSES:
    assert kept[k] >= 3, (k, counts[k], kept[k])
  assert 40 <= len(batch(model)) <= 64
  assert max(r['n'] for r in recs) > 64 and all(r['n'] <= CONBUF and r['nblk'] <= NB_L for r in recs)


# ------------------------------------------------------------------------------------------------ GPU side
def _env(model, precision, n, **kw):
  from so101_sim_b200.task_suite import create_batched_task_env
  return create_batched_task_env(TASKS[model], num_envs=n, time_limit=30.0, seed=0, device=DEV, reset_rounds=0, precision=precision, **kw)


def _solve_batch(model, precision, recs, probe=False):
  """One substep of every harvested state, one env each, from a zero warm start (set_initial_state + reset)."""
  env = _env(model, precision, len(recs), control_timestep=0.002)
  env.set_initial_state(torch.tensor(np.stack([r['q'] for r in recs])), torch.tensor(np.stack([r['v'] for r in recs])))
  env.reset()
  if probe:
    env.debug_contacts()   # (enables the probe for the next step)
  env.step(torch.tensor(np.stack([r['a'] for r in recs]), dtype=torch.float32, device=DEV))
  q, v = env.get_state(torch.float64)
  out = dict(q=q.cpu().numpy(), v=v.cpu().numpy(), tier=env.debug_read('tier').flatten().cpu().numpy(),
             iters=env.debug_read('solver_iter').flatten().cpu().numpy(), ncon=env.debug_read('ncon').flatten().cpu().numpy(),
             warm=env.debug_read('warm', env.nv).cpu().numpy(), counters=env.counters())
  if probe:
    out['contacts'] = env.debug_contacts()
  env.close()
  return out


def _oracle_substep(model, r):
  o = OracleSim(model, collide=True)
  o.set_state(r['q'], r['v'])
  o.forward()
  cons = o.contacts()
  o.control_step(r['a'], nsub=1)
  return o, cons


def _rel(got, want):
  return float(np.abs(got - want).max() / max(1.0, np.abs(want).max()))


@pytest.mark.gpu
@pytest.mark.parametrize('model', MODELS)
def test_f64_one_substep_in_every_tier_matches_oracle(built, model):
  """float64, one substep of each harvested state against a fresh oracle (both from a zero warm start): the tier the classifier
  picked, the contact list (bars of test_scene_gpu.test_contacts_match_oracle; the probe is float32), the Newton iteration
  count, qpos and qvel.  Same algorithm in float64: measured on a B200, the worst relative qpos / qvel error is 2e-16 / 3e-14
  in every tier; the bar is 1e-10.
  States with a contact on a curved static obstacle are handled as in test_scene_gpu.test_f64_scene_matches_oracle: EPA stops
  there by tolerance, so those contacts' distance / position may differ by more than round-off (measured up to 0.7 mm for an
  arm link 5 cm deep in the static capsule), the Newton iteration count by one or two, qpos by up to 6.4e-6 and qvel by
  1.9e-4 relative; their geom pairs must still match, qpos within 1e-4 and qvel within 1e-3."""
  recs = batch(model)
  got = _solve_batch(model, 'f64', recs, probe=True)
  assert got['counters']['contacts_dropped'] == 0 and got['counters']['diverged'] == 0
  curved = curved_static_geoms(OracleSim(model).meta)
  worst = {t: [0, 0.0, 0.0] for t in range(3)}   # states, worst relative qpos / qvel error (curved-contact states excluded)
  worst_curved = [0, 0.0, 0.0]
  bad = []   # every mismatch of the batch, not only the first
  for e, r in enumerate(recs):
    o, ref = _oracle_substep(model, r)
    if int(got['tier'][e]) != r['tier']:
      bad.append(('tier', e, r['n'], r['nblk'], r['tier'], int(got['tier'][e])))
    if not int(got['ncon'][e]) == r['n'] == len(ref) == len(got['contacts'][e]):
      bad.append(('ncon', e, r['n'], len(ref), int(got['ncon'][e]), len(got['contacts'][e])))
    else:
      for i, (g, c) in enumerate(zip(got['contacts'][e], ref)):
        if (g[0], g[1]) != (c['geom1'], c['geom2']):
          bad.append(('contact pair', e, i, g[:2], (c['geom1'], c['geom2'])))
        elif g[0] not in curved and g[1] not in curved and not (abs(g[2] - c['dist']) < 5e-6 and np.abs(g[3] - c['pos']).max() < 1e-5
                                                                 and np.abs(g[4] - c['frame'][0]).max() < 1e-5):
          bad.append(('contact', e, i, g[:3], c['dist']))
    if not r['curved'] and int(got['iters'][e]) != o.info('solver_iter'):
      bad.append(('solver_iter', e, r['tier'], int(got['iters'][e]), o.info('solver_iter')))
    eq, ev = _rel(got['q'][e], o.qpos), _rel(got['v'][e], o.qvel)
    w = worst_curved if r['curved'] else worst[r['tier']]
    w[0] += 1; w[1] = max(w[1], eq); w[2] = max(w[2], ev)
  print(f'{model} f64 one substep vs oracle, per tier (states, worst rel qpos, worst rel qvel):', worst, 'states on curved obstacles', worst_curved)
  assert not bad, bad
  assert all(worst[t][0] >= 3 for t in range(3))
  for t in range(3):
    assert worst[t][1] < 1e-10 and worst[t][2] < 1e-10, (t, worst[t])
  assert worst_curved[1] < 1e-4 and worst_curved[2] < 1e-3, worst_curved


@pytest.mark.gpu
@pytest.mark.parametrize('model', MODELS)
def test_f32_one_substep_error_is_the_same_in_every_tier(built, model):
  """float32 product arithmetic, the same batch: qacc of the substep (the warm start it leaves) against the float64 oracle,
  relative to max(1, |qacc|), grouped by the tier the env was solved in.  Measured on a B200 (median / worst): one arm
  tier 0 2.3e-5 / 0.52, tier 1 1.3e-5 / 0.21, tier 2 5.3e-6 / 0.32; two arms 7.3e-6 / 0.24, 2.5e-5 / 0.15, 4.3e-5 / 1.6.  The
  worst states are arms driven centimetres into the table or the props, where float32 contact rows are stiff.  Tiers 1 and 2
  must stay within 10x of tier 0's median and worst error."""
  recs = batch(model)
  got = _solve_batch(model, 'f32', recs)
  assert got['counters']['contacts_dropped'] == 0 and got['counters']['diverged'] == 0
  errs = {t: [] for t in range(3)}
  for e, r in enumerate(recs):
    o, _ = _oracle_substep(model, r)
    errs[int(got['tier'][e])].append(   # (the float32 narrow phase may find a contact more or less at a tier edge)
        _rel(got['warm'][e].astype(np.float64), o.field('qacc', o.nv)))
  stats = {t: (len(x), float(np.median(x)), float(np.max(x))) for t, x in errs.items()}
  print(f'{model} f32 one substep, rel qacc error per tier (states, median, worst):', stats)
  assert all(stats[t][0] >= 3 for t in range(3))
  for t in (1, 2):
    assert stats[t][1] < 10 * stats[0][1] and stats[t][2] < 10 * stats[0][2], stats


def _contacts_part(got, ref):
  """Why a GPU contact list (debug_contacts, float32) differs from the oracle's for the same state beyond the bars of
  test_scene_gpu.test_contacts_match_oracle, or None."""
  if len(got) != len(ref):
    return f'{len(got)} contacts instead of {len(ref)}'
  for i, (g, c) in enumerate(zip(got, ref)):
    if (g[0], g[1]) != (c['geom1'], c['geom2']):
      return f'contact {i}: geoms {g[:2]} instead of {(c["geom1"], c["geom2"])}'
    if not (abs(g[2] - c['dist']) < 5e-6 and np.abs(g[3] - c['pos']).max() < 1e-5 and np.abs(g[4] - c['frame'][0]).max() < 1e-5):
      return f'contact {i} (geoms {g[:2]}): dist {g[2]:.6g} instead of {c["dist"]:.6g}'
  return None


@pytest.mark.gpu
def test_f64_rollouts_from_tier2_states_match_oracle(built):
  """float64, 100 substeps from the one-arm batch's tier-2 states with the harvested action held, state and contact list
  compared with the oracle after every substep: warm starts carried through the larger tiers.  Bars of test_scene_gpu's
  float64 scene tests: 1e-7, and 1e-4 once a curved static obstacle is touched.
  These actions drive the arm's 525-vertex link hull up to 5 cm into the table.  Measured on a B200: from states equal to
  1e-15, the narrow phase of such a deep hull-box penetration can return contact depths 0.1 mm apart from the oracle's (same
  normal, different support-feature clipping), and the next substeps part by decimetres - the ill-conditioned EPA case of
  test_twoarm_gpu.test_f64_two_arm_scene_matches_oracle.  That is the narrow phase, not the solver, so each env is compared up
  to the first substep whose contact list departs from the oracle's; the solver has to hold the bars until then, and enough
  substeps solved in tiers 1 and 2 must be compared."""
  model = 'so100_handover_banana'
  recs = [r for r in batch(model) if r['tier'] == 2]
  n = len(recs)
  env = _env(model, 'f64', n, control_timestep=0.002)
  env.set_initial_state(torch.tensor(np.stack([r['q'] for r in recs])), torch.tensor(np.stack([r['v'] for r in recs])))
  env.reset()
  env.debug_contacts()   # (enables the probe for the next step)
  act = torch.tensor(np.stack([r['a'] for r in recs]), dtype=torch.float32, device=DEV)
  sims = []
  for r in recs:
    o = OracleSim(model, collide=True)
    o.set_state(r['q'], r['v'])
    o.forward()
    sims.append(o)
  curved = curved_static_geoms(sims[0].meta)
  touched = [False] * n
  err = np.zeros(n)
  compared = [0] * n                    # substeps compared per env
  parted = [None] * n                   # (substep, reason) where the env's contact list departed from the oracle's
  tier_steps = np.zeros(3, dtype=int)   # compared substeps per solver tier
  for k in range(100):
    ref = [o.contacts() for o in sims]   # contacts of the state this substep starts from
    env.step(act)
    q, _ = env.get_state(torch.float64)
    got, tier = env.debug_contacts(), env.debug_read('tier').flatten().cpu().numpy()
    for e, o in enumerate(sims):
      o.control_step(recs[e]['a'], nsub=1)
      if parted[e] is not None:
        continue
      why = _contacts_part(got[e], ref[e])
      if why is not None:
        parted[e] = (k, why)
        continue
      touched[e] |= any(c['geom1'] in curved or c['geom2'] in curved for c in ref[e])
      err[e] = max(err[e], float(np.abs(q[e].cpu().numpy() - o.qpos).max()))
      compared[e] += 1
      tier_steps[int(tier[e])] += 1
      assert err[e] < (1e-4 if touched[e] else 1e-7), (e, k, err[e], touched[e])
  print(f'{model} f64 from {n} tier-2 states: max |dqpos| per env {err}, substeps compared {compared} (per tier {tier_steps.tolist()}),'
        f' curved {touched}, contact lists parted {parted}')
  assert n >= 3 and tier_steps[2] >= n and tier_steps[1] + tier_steps[2] >= 50 and sum(c >= 20 for c in compared) >= 3
  assert env.counters()['diverged'] == 0 and env.counters()['contacts_dropped'] == 0
  env.close()


def _two_arm_states(model, n, seed):
  rs = np.random.RandomState(seed)
  q = np.tile(np.asarray(OracleSim(model).meta['qpos0'], dtype=np.float64), (n, 1))
  q[:, :12] = 0
  for e in range(n):
    yaw = rs.uniform(-0.3, 0.3)
    q[e, 12:19] = [rs.uniform(0.2, 0.3), rs.uniform(-0.1, 0.1), 0.4217 + 0.002, np.cos(yaw / 2), 0, 0, np.sin(yaw / 2)]
    q[e, 19:26] = [rs.uniform(-0.3, -0.22), rs.uniform(-0.1, -0.02), 0.4226 + 0.002, 1, 0, 0, 0]
  return torch.tensor(q), torch.zeros(n, 24, dtype=torch.float64)


def _forced_rollout(model, precision, tier_min, monkeypatch):
  monkeypatch.setenv('SO101_SOLVE_TIER_MIN', str(tier_min))
  env = _env(model, precision, 64)
  if model == 'so100_handover_banana':
    env.sample_prop_initial_states(seed=11, settle_steps=0)
  else:
    env.set_initial_state(*_two_arm_states(model, 64, seed=11)); env.reset()
  g = torch.Generator(device=DEV); g.manual_seed(5)
  spec = env.action_spec()
  lo, hi = torch.tensor(spec.minimum, device=DEV), torch.tensor(spec.maximum, device=DEV)
  acts = (lo + torch.rand(25, 64, env.nu, generator=g, device=DEV) * (hi - lo)) * 0.6
  for t in range(25):
    env.step(acts[t])
  q, v = env.get_state(torch.float64)
  res = dict(q=q, v=v, ncon=env.debug_read('ncon').flatten(), iters=env.debug_read('solver_iter').flatten(), warm=env.debug_read('warm', env.nv),
             tier=env.debug_read('tier').flatten(), dropped=env.contacts_dropped_per_env())
  env.close()
  return res


@pytest.mark.gpu
@pytest.mark.parametrize('model', MODELS)
@pytest.mark.parametrize('precision', ['f32', 'f64'])
def test_forced_solver_tier_is_bit_identical(built, monkeypatch, model, precision):
  """SO101_SOLVE_TIER_MIN = 0, 1, 2 sends every env to at least that tier.  The per-contact arithmetic does not depend on the
  tier's capacity (loops run to ncon, unused body-mask words are zero), so a 64-env, 25-step random-action rollout must end in
  the same state, contact counts, iteration counts and warm starts bit for bit, and so must the harvested batch solved
  naturally and forced into tier 2.  Envs that lost contacts to a full buffer in any of the runs are left out: which contacts
  survive then depends on arrival order.
  float32 exception, measured: tier 2's kernel (scene_solve_tier_kernel<float, 128, 160>) differs from tiers 0 and 1 in the
  last bits, because nvcc contracts a different set of float32 multiply-adds into FMAs in that instantiation.  The same sources
  built with --fmad=false give bit-identical float32 results in all three tiers (the float64 kernels are always built so).  In
  float32 the rollouts therefore compare tier 1 with tier 0 bit for bit, and the one-substep batch compares tier 2 with the
  natural tiers to 1e-4 relative in qacc (measured up to 9.7e-6)."""
  runs = [_forced_rollout(model, precision, t, monkeypatch) for t in (0, 1, 2)]
  keep = (torch.stack([r['dropped'] for r in runs]) == 0).all(0)
  print(f'{model} {precision} forced tiers: {int(keep.sum())} of 64 envs keep all contacts, max contacts {int(runs[0]["ncon"].max())},'
        f' natural tiers at the end {torch.bincount(runs[0]["tier"].long(), minlength=3).tolist()}')
  assert int(keep.sum()) >= 32 and int(runs[0]['ncon'][keep].max()) > 32
  for t, r in enumerate(runs):
    assert int(r['tier'].min()) >= t
    if precision == 'f32' and t == 2:
      continue
    for k in ('q', 'v', 'ncon', 'iters', 'warm'):
      assert torch.equal(r[k][keep], runs[0][k][keep]), (t, k)
  recs = batch(model)
  monkeypatch.setenv('SO101_SOLVE_TIER_MIN', '0')
  natural = _solve_batch(model, precision, recs)
  monkeypatch.setenv('SO101_SOLVE_TIER_MIN', '2')
  forced = _solve_batch(model, precision, recs)
  assert sorted(set(natural['tier'].tolist())) == [0, 1, 2] and set(forced['tier'].tolist()) == {2}
  if precision == 'f64':
    for k in ('q', 'v', 'ncon', 'iters', 'warm'):
      assert np.array_equal(natural[k], forced[k]), k
  else:
    d = max(_rel(forced['warm'][e], natural['warm'][e]) for e in range(len(recs)))
    print(f'{model} f32 batch forced into tier 2: worst rel qacc difference {d:.3g}')
    assert np.array_equal(natural['ncon'], forced['ncon']) and d < 1e-4
