"""ctypes loader for the sm_100a shared library (C-ABI declared in include/so101_b200.h).

There is NO CPU fallback: if the library is missing, cannot be loaded, or no CUDA device is present, this module raises.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('SO101_B200_LIB') or os.path.join(_HERE, 'libso101_b200.so')  # override: developer A/B builds only
# the same sources compiled with -DSO101_NARM=2: the labelled synthetic two-arm hand-over scene (BASELINE config 4)
LIB_PATH_2ARM = os.path.join(_HERE, 'libso101_b200_2arm.so')


class StepOut(ctypes.Structure):
  _fields_ = [(n, ctypes.c_void_p) for n in ('commanded_joints_pos', 'joints_pos', 'undelayed_joints_pos', 'physics_state',
                                             'delayed_physics_state', 'reward', 'discount', 'step_type')]


class Config(ctypes.Structure):
  _fields_ = [('num_envs', ctypes.c_int), ('device', ctypes.c_int), ('n_substeps', ctypes.c_int), ('last_step', ctypes.c_int),
              ('joints_delay_steps', ctypes.c_int), ('physics_delay_steps', ctypes.c_int), ('terminate_on_success', ctypes.c_int),
              ('solver_iterations', ctypes.c_int), ('solver_tolerance', ctypes.c_float), ('precision', ctypes.c_int),
              ('collide', ctypes.c_int), ('calibration_offsets', ctypes.c_float * 6), ('home_ctrl', ctypes.c_float * 6),
              ('nursery_envs', ctypes.c_int), ('ring_capacity', ctypes.c_int), ('seed', ctypes.c_uint64),
              ('place_lo', (ctypes.c_float * 3) * 2), ('place_hi', (ctypes.c_float * 3) * 2), ('place_yaw', (ctypes.c_float * 2) * 2),
              ('place_check_collisions', ctypes.c_int * 2), ('place_max_attempts', ctypes.c_int), ('settle_max_substeps', ctypes.c_int),
              ('settle_qvel_tol', ctypes.c_float), ('settle_qacc_tol', ctypes.c_float), ('integrator', ctypes.c_int)]


class EEParams(ctypes.Structure):
  """so101_ee_params: parameters of so101_ee_ik."""
  _fields_ = [('tcp_offset', ctypes.c_float * 3), ('iterations', ctypes.c_int), ('damping', ctypes.c_float), ('w_rot', ctypes.c_float),
              ('max_step', ctypes.c_float), ('tolerance', ctypes.c_float)]


EXPORTS = ('so101_abi_version', 'so101_create', 'so101_destroy', 'so101_last_error', 'so101_dims', 'so101_set_initial_state',
           'so101_reset', 'so101_step', 'so101_get_state', 'so101_set_state', 'so101_get_state_f64', 'so101_step_host',
           'so101_counters', 'so101_debug_read', 'so101_kernel_times', 'so101_set_reset_pool', 'so101_set_state_f64', 'so101_debug_overlap', 'so101_sample_and_settle', 'so101_placement_stats', 'so101_get_episode_steps', 'so101_set_episode_steps',
           'so101_checkpoint_size', 'so101_checkpoint_save', 'so101_checkpoint_load', 'so101_ee_pose', 'so101_ee_ik',
           'so101_contact_sensors', 'so101_contact_sensors_read')
MAX_CONTACT_SENSORS = 16   # SO101_MAX_CONTACT_SENSORS

_libs = {}


def load(narm: int = 1) -> ctypes.CDLL:
  """The library built for `narm` arms (1: the reference's scenes; 2: the synthetic two-arm scene)."""
  if narm in _libs:
    return _libs[narm]
  if narm not in (1, 2):
    raise RuntimeError(f'no build of the kernels for {narm} arms')
  path = LIB_PATH if narm == 1 else LIB_PATH_2ARM
  if not os.path.exists(path):
    raise RuntimeError(f'{path} is missing: build it with `python -c "import __graft_entry__ as g; g.build()"` '
                       '(so101_sim_b200 has no CPU fallback)')
  L = ctypes.CDLL(path)
  vp, ci = ctypes.c_void_p, ctypes.c_int
  L.so101_abi_version.restype = ci
  L.so101_create.restype = ci; L.so101_create.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.POINTER(Config), ctypes.POINTER(vp)]
  L.so101_destroy.restype = ci; L.so101_destroy.argtypes = [vp]
  L.so101_last_error.restype = ctypes.c_char_p; L.so101_last_error.argtypes = [vp]
  L.so101_dims.restype = ci; L.so101_dims.argtypes = [vp] + [ctypes.POINTER(ci)] * 4
  for f in ('so101_set_initial_state', 'so101_set_state', 'so101_get_state', 'so101_get_state_f64'):
    getattr(L, f).restype = ci; getattr(L, f).argtypes = [vp, vp, vp, vp]
  L.so101_set_state_f64.restype = ci; L.so101_set_state_f64.argtypes = [vp, vp, vp, ci, vp]
  L.so101_debug_overlap.restype = ci; L.so101_debug_overlap.argtypes = [ci, ci, vp, ci, vp, vp]
  L.so101_sample_and_settle.restype = ci; L.so101_sample_and_settle.argtypes = [vp, ctypes.c_uint64, ctypes.POINTER(StepOut), ctypes.POINTER(ctypes.c_uint64 * 4), vp]
  L.so101_get_episode_steps.restype = ci; L.so101_get_episode_steps.argtypes = [vp, vp, vp]
  L.so101_set_episode_steps.restype = ci; L.so101_set_episode_steps.argtypes = [vp, vp, vp]
  L.so101_checkpoint_size.restype = ci; L.so101_checkpoint_size.argtypes = [vp, ctypes.POINTER(ctypes.c_size_t)]
  L.so101_checkpoint_save.restype = ci; L.so101_checkpoint_save.argtypes = [vp, vp, ctypes.c_size_t, vp]
  L.so101_checkpoint_load.restype = ci; L.so101_checkpoint_load.argtypes = [vp, vp, ctypes.c_size_t, vp]
  L.so101_placement_stats.restype = ci; L.so101_placement_stats.argtypes = [vp, ctypes.POINTER(ctypes.c_uint64 * 6)]
  L.so101_set_reset_pool.restype = ci; L.so101_set_reset_pool.argtypes = [vp, vp, vp, ci, vp]
  L.so101_reset.restype = ci; L.so101_reset.argtypes = [vp, vp, ctypes.POINTER(StepOut), vp]
  L.so101_step.restype = ci; L.so101_step.argtypes = [vp, vp, ctypes.POINTER(StepOut), vp]
  L.so101_step_host.restype = ci; L.so101_step_host.argtypes = [vp, vp, ctypes.POINTER(StepOut), vp]
  L.so101_counters.restype = ci; L.so101_counters.argtypes = [vp, ctypes.POINTER(ctypes.c_uint64 * 6)]
  L.so101_kernel_times.restype = ci; L.so101_kernel_times.argtypes = [vp, ci, ctypes.POINTER(ctypes.c_double * 11), ctypes.POINTER(ctypes.c_uint64 * 11)]
  L.so101_debug_read.restype = ci; L.so101_debug_read.argtypes = [vp, ctypes.c_char_p, vp, ctypes.c_size_t, vp]
  L.so101_ee_pose.restype = ci; L.so101_ee_pose.argtypes = [vp, ci, ctypes.POINTER(ctypes.c_float * 3), vp, vp, vp]
  L.so101_ee_ik.restype = ci; L.so101_ee_ik.argtypes = [vp, vp, vp, vp, vp, ctypes.POINTER(EEParams), vp, vp, vp]
  L.so101_contact_sensors.restype = ci; L.so101_contact_sensors.argtypes = [vp, ci, vp]
  L.so101_contact_sensors_read.restype = ci; L.so101_contact_sensors_read.argtypes = [vp, vp, ctypes.c_size_t, vp]
  if L.so101_abi_version() != 5:
    raise RuntimeError(f'{path}: ABI version mismatch')
  _libs[narm] = L
  return L
