// Device-resident state of N lockstep environments, structure-of-arrays: field[k][env] so that a warp touching the
// same component of 32 consecutive envs issues one coalesced 128 B (f32) / 256 B (f64) request.
#pragma once
#include <cstdint>
#include "../../include/so101_b200.h"

namespace so101 {

// The integration state (qpos, qvel and the reset pool) is float64 in BOTH precisions.  The float32 product path runs
// collision, the contact rows and the Newton solver in float32 (> 95 % of the arithmetic), but the arm's smooth dynamics
// (FK, CRB, RNE, actuators, M^-1), and the semi-implicit Euler update in float64: the reference's actuators are anti-damped
// (bias +1 * qvel, scene_pbr.xml:11) and amplify a perturbation ~300x over 100 control steps, so that neither a float32 state
// (1.8e-3 relative error after 100 steps) nor float32 smooth dynamics on a float64 state (1.6e-4) meet north_star's 1e-4;
// float64 smooth dynamics + float32 solver give 9e-6 (profiles/r2c_arm_precision.jsonl; DESIGN.md section 2).
using TS = double;

// On-device episode initialisation of the hand-over tasks (so100_hand_over.py:208-229,320-323; [upstream] dm_control
// PropPlacer): an env in SETTLE mode draws a prop placement from the task's distributions with a counter-based Philox stream,
// rejects it while the collision-checked prop penetrates anything at its spawn pose, then steps physics with the arm frozen
// until the props' |qvel| < 1e-3 and |qacc| < 1e-2 or 2 s have passed.  User envs go through it once (so101_sample_and_settle);
// a few extra NURSERY envs (indices >= NU, invisible to the caller) do it continuously and publish settled placements into a
// ring that auto-resets consume, so that every episode starts from a fresh placement without stalling the batch.
struct PlacementCfg {
  float lo[2][3], hi[2][3];   // position box of prop 0 (object) / prop 1 (container)          so100_hand_over.py:37-41,51-55
  float yaw[2][2];            // rotation about z, uniform in [yaw[p][0], yaw[p][1]]            so100_hand_over.py:42-49
  int check_collisions[2];    // PropPlacer(ignore_collisions=False) for this prop              so100_hand_over.py:216-221
  int max_attempts;           // [upstream] PropPlacer max_attempts_per_prop = 20
  int max_settle_substeps;    // [upstream] max_settle_physics_time 2 s / 0.002 s
  float qvel_tol, qacc_tol;   // [upstream] _SETTLE_QVEL_TOL 1e-3, _SETTLE_QACC_TOL 1e-2
  unsigned long long seed;
};
enum { SETTLE_SAMPLE = 0, SETTLE_RUN = 1, SETTLE_DONE = 2 };
// ring counters
enum { RC_CLAIM = 0 /* placements published */, RC_TAIL = 1 /* placements consumed */, RC_REUSED = 2 /* resets that found the ring empty */,
       RC_UNSETTLED = 3 /* settles that ran into the time limit */, RC_EXHAUSTED = 4 /* placements accepted after max_attempts rejections */,
       RC_REJECTED = 5 /* rejected samples */, RC_PENDING = 6 /* user envs still settling (so101_sample_and_settle) */, RC_N = 8 };

template <typename T>
struct EnvState {
  int N, nq, nv;                    // N = all envs of the handle (user envs first, then the nursery): array strides
  int NU;                           // envs the caller sees (outputs, actions, state access)
  uint8_t *mode;                    // [N] 0 = normal stepping, 1 = SETTLE mode
  uint8_t *sstate;                  // [N] SETTLE_* state of an env in settle mode
  int *settle_sub, *attempt;        // [N] substeps into the current settle / rejected samples of the current placement
  unsigned *draws;                  // [N] Philox draws made by this env (counter)
  TS *ring_q, *ring_v;              // [ring_cap][nq], [ring_cap][nv] settled placements published by the nursery
  int ring_cap;
  int use_ring;                     // resets take placements from the ring / the nursery produces them (off while the caller's own
                                    //   initial states or reset pool are installed)
  int *ring_ctr;                    // [RC_N]
  PlacementCfg place;
  TS *qpos, *qvel;                  // [nq][N], [nv][N]
  T *warm;                          // [nv][N]  (qacc_warmstart)
  TS *init_qpos, *init_qvel;        // reset pool [npool][...same layout as qpos / qvel...]: episode e of an env starts from entry e % npool
  int npool;                        // entries in the reset pool (>= 1)
  int *episode;                     // [N] resets this env has gone through (selects the pool entry)
  T *ctrl;                          // [6][N]
  int *step;                        // [N] control steps since reset
  uint8_t *needs_reset;             // [N] previous step was LAST (dm_control auto-reset on next step)
  float *ring_joints;               // [Dj+1][6][N]
  float *ring_phys;                 // [Dp+1][nq+nv][N]
  int *diverged_count;              // [1]
  int *solver_iter;                 // [N] Newton iterations of the last substep (parity/diagnostics)
  int *ncon;                        // [N] contacts of the last substep
  int *dropped_env;                 // [N] contacts / candidate pairs this env lost to a full buffer since create (see so101_counters)
  float *dbg_contacts;              // optional [N][1 + 9*NCON] parity probe (null unless requested)
};

struct StepCfg {
  int nsub, last_step, dj, dp, terminate_on_success, max_iter;
  int integrator;  // 0 = semi-implicit Euler (the reference's default, scene_pbr.xml sets none), 1 = implicitfast (north_star)
  float tol;
  float offsets[6], home[6];
};

}  // namespace so101
