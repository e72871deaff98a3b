"""Host-side reader for the compiled model blob (format written by tools/compile_model.py).

The blob is the flat, versioned model description of the SO100 scene
(reference: so101_sim/assets/so100/scene_pbr.xml + the two YCB props, so100_hand_over.py:159-206).
"""
from __future__ import annotations

import os
import struct

import numpy as np

DATA_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'data')
BLOB_MAGIC = b'SO1B'
BLOB_VERSION = 2


def blob_path(name: str) -> str:
  return name if os.path.exists(name) else os.path.join(DATA_DIR, name + '.blob')


def read_blob(path: str) -> dict[str, np.ndarray]:
  with open(blob_path(path), 'rb') as f:
    raw = f.read()
  magic, version, n, _ = struct.unpack_from('<4sIII', raw, 0)
  if magic != BLOB_MAGIC or version != BLOB_VERSION:
    raise ValueError(f'{path}: not a so101 model blob (magic={magic!r}, version={version})')
  out = {}
  for i in range(n):
    name, dt, cnt, off = struct.unpack_from('<24sIIQ', raw, 16 + 40 * i)
    out[name.rstrip(b'\0').decode()] = np.frombuffer(raw, dtype=np.float64 if dt == 0 else np.int32, count=cnt, offset=off).copy()
  return out


def tcp_offset(model: dict[str, np.ndarray], arm: int = 0) -> np.ndarray:
  """Default tool centre point of arm `arm`, in the frame of its Fixed_Jaw body (the body of the arm's fifth hinge, Wrist_Roll):
  the midpoint of the centroid of the Fixed_Jaw's box pads and the centroid of the Moving_Jaw's box pads at jaw angle 0 (carried
  into the Fixed_Jaw frame through the Moving_Jaw's body_pos / body_quat and the jaw hinge at qpos0 -> 0).  Metres, float64 [3]."""
  box = 4   # geom type code of a box in the blob (tools/compile_model.py GEOM_BOX)
  jb = model['jnt_body']
  if len(jb) < 6 * arm + 6:
    raise ValueError(f'model has no arm {arm}')
  fixed, moving, jaw = int(jb[6 * arm + 4]), int(jb[6 * arm + 5]), 6 * arm + 5
  gb, gt, gp = model['geom_body'], model['geom_type'], model['geom_pos'].reshape(-1, 3)
  pads_f, pads_m = gp[(gb == fixed) & (gt == box)], gp[(gb == moving) & (gt == box)]
  if not len(pads_f) or not len(pads_m):
    raise ValueError(f'arm {arm}: the jaws have no box pads to define the tool centre point')
  if int(model['body_parent'][moving]) != fixed:
    raise ValueError(f'arm {arm}: the Moving_Jaw is not a child of the Fixed_Jaw')
  w, x, y, z = model['body_quat'].reshape(-1, 4)[moving] / np.linalg.norm(model['body_quat'].reshape(-1, 4)[moving])
  R = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])
  # jaw angle 0: rotate the Moving_Jaw frame about its hinge (anchored at the body origin) by 0 - qpos0
  ax = model['jnt_axis'].reshape(-1, 3)[jaw]
  th = -float(model['qpos0'][jaw])
  K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
  Rj = np.eye(3) + np.sin(th) * K + (1 - np.cos(th)) * K @ K
  moving_in_fixed = model['body_pos'].reshape(-1, 3)[moving] + R @ Rj @ pads_m.mean(axis=0)
  return 0.5 * (pads_f.mean(axis=0) + moving_in_fixed)


BODY_SET_NAMES = ('fixed_jaw', 'moving_jaw', 'gripper', 'arm', 'object', 'container', 'static')


def body_set(model: dict[str, np.ndarray], name: str, arm: int = 0) -> list[int]:
  """Body ids of a named part of the model, read from the blob's own tables: 'fixed_jaw' / 'moving_jaw' (the bodies of arm
  `arm`'s fifth and sixth hinges), 'gripper' (both jaws), 'arm' (the bodies of the arm's six hinges), 'object' / 'container'
  (the two props), 'static' (every body without a joint: the world, the arm bases, the table and the fixed furniture)."""
  jb, nbody = model['jnt_body'], int(model['nbody'][0])
  if name in ('fixed_jaw', 'moving_jaw', 'gripper', 'arm'):
    narm = int(model['nu'][0]) // 6
    if not 0 <= arm < narm:
      raise ValueError(f'model has no arm {arm} (it has {narm})')
    j0 = 6 * arm
    ids = {'fixed_jaw': [j0 + 4], 'moving_jaw': [j0 + 5], 'gripper': [j0 + 4, j0 + 5], 'arm': list(range(j0, j0 + 6))}[name]
    return [int(jb[j]) for j in ids]
  if name in ('object', 'container'):
    pb = model['prop_body']
    p = 0 if name == 'object' else 1
    if len(pb) <= p:
      raise ValueError(f'model has no {name} prop')
    return [int(pb[p])]
  if name == 'static':
    return [b for b in range(nbody) if int(model['body_jntnum'][b]) == 0]
  raise ValueError(f'unknown body set {name!r} (known: {", ".join(BODY_SET_NAMES)})')
