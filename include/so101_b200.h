/* so101_b200 — C-ABI of the B200-native batched SO100/SO101 environment step.
 *
 * This is the drop-in boundary for the ONE hot path of tuul-ai/so101_sim: the lockstep env step
 * (reference call stack: scripts/so101_lerobot_wrapper.py:70-75 -> dm_control composer.Environment.step ->
 *  SO100Task.before_step so101_sim/tasks/base/so100_task.py:266-287 -> 10x mj_step -> observables
 *  so100_task.py:331-368 -> SO100HandOver.get_reward so101_sim/tasks/so100_hand_over.py:238-275 ->
 *  get_discount / should_terminate_episode so100_task.py:292-302).
 *
 * The reference has no FFI of its own for this path (it is Python over MuJoCo's C API through dm_control); each
 * entry point below names the reference interface it replaces.  Plain pointers and sizes only; no torch types.
 * All device pointers are borrowed for the duration of the call; the caller (PyTorch) owns every tensor.
 * All work is enqueued on the caller's stream; no entry point synchronises the host unless it says so.
 * Return value: 0 = ok, negative = error (see so101_last_error).  Nothing throws across this boundary.
 * One handle per device; calls on one handle must be serialised by the caller.
 */
#ifndef SO101_B200_H
#define SO101_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SO101_ABI_VERSION 5

/* dm_env.StepType values (reference TimeStep.step_type) */
#define SO101_STEP_FIRST 0
#define SO101_STEP_MID 1
#define SO101_STEP_LAST 2

/* contact force sensors a handle holds at most (so101_contact_sensors) */
#define SO101_MAX_CONTACT_SENSORS 16

typedef struct so101_env *so101_handle;

/* Per-step outputs: device pointers into caller-owned row-major tensors, N = num_envs.  Any pointer may be NULL
 * (that block is then not written).  Mirrors the reference TimeStep + observation dict
 * (so100_task.py:331-368; key order examples/so101_rl_breakdown.ipynb:65); joints_vel / undelayed_joints_vel are
 * empty arrays in the reference (so100_task.py:357-364) and therefore have no pointer here. */
typedef struct so101_step_out {
  float *commanded_joints_pos;  /* [N,6]      ctrl after calibration, unclamped  (so100_task.py:344-355) */
  float *joints_pos;            /* [N,6]      qpos[0:6] delayed 5 control steps  (so100_task.py:331-342,196-198) */
  float *undelayed_joints_pos;  /* [N,6]      qpos[0:6] now                      (so100_task.py:189-192) */
  float *physics_state;         /* [N,nq+nv]  qpos || qvel                       (so100_task.py:366-368) */
  float *delayed_physics_state; /* [N,nq+nv]  delayed 15 control steps           (so100_task.py:203-210) */
  float *reward;                /* [N]        SO100HandOver.get_reward           (so100_hand_over.py:238-275) */
  float *discount;              /* [N]        SO100Task.get_discount             (so100_task.py:292-295) */
  uint8_t *step_type;           /* [N]        FIRST / MID / LAST */
} so101_step_out;

typedef struct so101_config {
  int num_envs;
  int device;               /* CUDA device ordinal */
  int n_substeps;           /* control_timestep / physics_timestep = 10 (task_suite.py:41) */
  int last_step;            /* control-step index on which the time limit fires (1501 for 30 s; computed by the host
                               with the reference's float64 `time += dt` accumulation); <=0 = no limit */
  int joints_delay_steps;   /* 5  (0.1 s / 0.02 s, so100_task.py:80,196-198) */
  int physics_delay_steps;  /* 15 (0.3 s / 0.02 s, so100_task.py:79,203-210) */
  int terminate_on_success; /* SO100Task(terminate_episode=True), so100_task.py:119 */
  int solver_iterations;    /* Newton iteration cap per substep (MuJoCo default 100) */
  float solver_tolerance;   /* scaled-gradient / improvement tolerance (MuJoCo default 1e-8, reachable in f64 only) */
  int precision;            /* 32 = float32 arithmetic (north_star dtype), 64 = float64 arithmetic (tight-parity mode) */
  int collide;              /* 0 = collisions off (BASELINE config 2, arm-only), 1 = full contact pipeline */
  float calibration_offsets[6]; /* SO101Calibration.homing_offsets, scripts/so101_calibration.py:62-77 */
  float home_ctrl[6];       /* SO100_HOME_CTRL, so100_task.py:45-47 (ctrl written by initialize_episode :316-317) */
  /* On-device episode initialisation of the hand-over tasks (initialize_episode so100_hand_over.py:320-323, the three
   * PropPlacers :208-229 with the distributions :37-55).  nursery_envs extra envs (hidden from the caller) keep sampling,
   * collision-checking and settling placements with the arm frozen and publish them into a ring of ring_capacity entries;
   * every auto-reset / so101_reset takes a fresh one (falls back to the env's own initial state when the ring is empty). */
  int nursery_envs;         /* 0 = no background placements (resets re-use the installed initial states / reset pool) */
  int ring_capacity;        /* placements the ring can hold */
  uint64_t seed;            /* Philox key of the placement stream */
  float place_lo[2][3], place_hi[2][3]; /* position boxes of prop 0 (object) and prop 1 (container) */
  float place_yaw[2][2];    /* yaw range about z per prop */
  int place_check_collisions[2]; /* 1 = re-sample while the prop penetrates anything at its spawn pose (ignore_collisions=False) */
  int place_max_attempts;   /* [upstream] PropPlacer max_attempts_per_prop (20) */
  int settle_max_substeps;  /* [upstream] max_settle_physics_time / timestep (2 s / 0.002 s = 1000) */
  float settle_qvel_tol, settle_qacc_tol; /* [upstream] 1e-3, 1e-2 */
  int integrator;           /* 0 = semi-implicit Euler: MuJoCo's default, which the reference uses (scene_pbr.xml:4 sets none);
                               1 = implicitfast ([upstream] mj_implicit without the Coriolis derivatives) */
} so101_config;

int so101_abi_version(void);

/* replaces task_suite.create_task_env (so101_sim/task_suite.py:103-155) for the physics + task state of N envs */
int so101_create(const void *model_blob, size_t blob_len, const so101_config *cfg, so101_handle *out);
/* replaces composer.Environment.close() */
int so101_destroy(so101_handle h);
/* last error message of this handle (or of the failed create when h == NULL) */
const char *so101_last_error(so101_handle h);

/* model dimensions: nq, nv, nu, state_dim (= nq + nv) */
int so101_dims(so101_handle h, int *nq, int *nv, int *nu, int *nbody);

/* Install per-env initial states (row-major [N,nq], [N,nv] device pointers).  These are the states an env returns to on
 * reset; replaces the pose sampling of initialize_episode (so100_task.py:304-320, so100_hand_over.py:320-323). */
int so101_set_initial_state(so101_handle h, const float *qpos_dev, const float *qvel_dev, void *stream);
/* Install a POOL of `rounds` initial states per env (row-major [rounds,N,nq], [rounds,N,nv] device pointers): episode e of an
 * env (counted from this call) starts from pool entry e % rounds, so consecutive episodes see different sampled-and-settled
 * prop placements, as the reference re-samples them in every initialize_episode (so100_hand_over.py:208-229,320-323 with
 * the distributions :37-55).  Replaces the single state of so101_set_initial_state. */
int so101_set_reset_pool(so101_handle h, const float *qpos_dev, const float *qvel_dev, int rounds, void *stream);
/* replaces composer.Environment.reset(): envs with mask[i] != 0 (all when mask_dev == NULL) go back to their initial
 * state, ctrl = home + offsets, delay buffers refilled with the initial value, step counter 0.  Writes the FIRST
 * TimeStep blocks of `out` for the reset envs. */
int so101_reset(so101_handle h, const uint8_t *mask_dev, const so101_step_out *out, void *stream);
/* replaces composer.Environment.step(action) for all N envs; action_dev is row-major [N,6] float32.
 * Envs whose previous step was LAST are reset instead and return FIRST (dm_control auto-reset). */
int so101_step(so101_handle h, const float *action_dev, const so101_step_out *out, void *stream);
/* replaces the placement part of initialize_episode for ALL envs at once: every env draws a placement from the configured
 * distributions (Philox keyed on (seed, env, draw)), re-samples while the collision-checked prop penetrates anything at its
 * spawn pose, and settles with the arm frozen ([upstream] PropPlacer settle_physics: props' |qvel| < qvel_tol and |qacc| <
 * qacc_tol, or settle_max_substeps).  The loop over control steps runs inside the library; the settled states become the envs'
 * initial states and the envs are reset.  stats_out (nullable): [0] control steps run, [1] settles that hit the time limit,
 * [2] rejected samples, [3] placements kept after max_attempts rejections.  Synchronises the stream. */
int so101_sample_and_settle(so101_handle h, uint64_t seed, const so101_step_out *out, uint64_t stats_out[4], void *stream);
/* placement ring statistics: [0] published, [1] consumed, [2] resets that found the ring empty (re-used their initial state),
 * [3] settles that hit the time limit, [4] placements kept after max_attempts rejections, [5] rejected samples */
int so101_placement_stats(so101_handle h, uint64_t out[6]);

/* physics.get_state() / set_state() equivalents (so100_task.py:366-368): row-major [N,nq], [N,nv] device pointers */
int so101_get_state(so101_handle h, float *qpos_dev, float *qvel_dev, void *stream);
int so101_set_state(so101_handle h, const float *qpos_dev, const float *qvel_dev, void *stream);
/* The integration state is float64 in both precisions (the float32 path evaluates dynamics and contacts in float32 but
 * accumulates the Euler update in float64): these two move it without rounding to float32.  initial != 0 also installs the
 * state as the reset state (like so101_set_initial_state). */
int so101_get_state_f64(so101_handle h, double *qpos_dev, double *qvel_dev, void *stream);
int so101_set_state_f64(so101_handle h, const double *qpos_dev, const double *qvel_dev, int initial, void *stream);

/* Control steps each env has taken in its current episode ([N] int32 device pointer): the part of the env state that decides when
 * the time limit fires (composer.Environment's `physics.time() >= time_limit`).  Read / written with the physics state for
 * checkpoint-resume and to start a batch at staggered episode phases. */
int so101_get_episode_steps(so101_handle h, int32_t *steps_dev, void *stream);
int so101_set_episode_steps(so101_handle h, const int32_t *steps_dev, void *stream);

/* Checkpoint / resume of a whole handle.  get_state / set_state move the physics state only, as physics.get_state() does
 * (so100_task.py:366-368); a rollout also depends on what composer.Environment and the observables keep between steps: warm
 * starts, ctrl, the observation delay buffers (so100_task.py:196-210), episode counters and auto-reset flags, the reset states,
 * and here the placement machinery (nursery envs in SETTLE mode, Philox draw counters, the ring of settled placements).
 * so101_checkpoint_save copies all of it into ONE caller-owned device buffer of so101_checkpoint_size bytes (a header, then the
 * arrays); so101_checkpoint_load restores it into a handle created with the same model blob, precision, num_envs, nursery_envs,
 * ring_capacity and delay settings, after which stepping continues bit for bit as it would have.  Both synchronise the stream. */
int so101_checkpoint_size(so101_handle h, size_t *bytes);
int so101_checkpoint_save(so101_handle h, void *buf_dev, size_t bytes, void *stream);
int so101_checkpoint_load(so101_handle h, const void *buf_dev, size_t bytes, void *stream);

/* End-to-end variant with HOST buffers (pinned or pageable): copies action_host [N,6] to the device, steps, copies every
 * block of the TimeStep whose pointer in *out_host is non-NULL (HOST pointers, same shapes as so101_step_out) back, and
 * synchronises the stream before returning.  This is composer.Environment.step(action) -> TimeStep as a host caller sees it. */
int so101_step_host(so101_handle h, const float *action_host, const so101_step_out *out_host, void *stream);

/* counters since create: [0] kernels launched by this library (kernels replayed from a captured step graph included),
 * [1] control steps taken, [2] envs that diverged, [3] contacts dropped by a full per-env contact buffer, [4] step-graph
 * launches (one cudaGraphLaunch replays all kernels of a control step of the contact scene), [5] reserved */
int so101_counters(so101_handle h, uint64_t out[6]);

/* Per-kernel device time, measured with CUDA events around every launch while enabled.  While enabled the step is launched
 * eagerly (no graph replay) and all pipeline groups and solver tiers go to the caller's stream, so that every launch is timed
 * alone.  Returns the totals accumulated so far (ms and launch counts; index 0 scene begin, 1 scene EPA + manifold (fused
 * kernel of small batches), 2 scene solve tier 0, 3 scene solve tier 1, 4 arm-only step,
 * 5 scene boolean GJK, 6 scene kinematics + smooth dynamics, 7 scene broad phase / task layer, 8 EPA and 9 manifold kernel
 * of the two-launch narrow phase, 10 scene solve tier 2), then switches recording on/off for the following calls.  Synchronises the host on the
 * recorded events.  No reference counterpart: measurement support for bench.py's roofline leg. */
int so101_kernel_times(so101_handle h, int enable, double ms_out[11], uint64_t launches_out[11]);

/* Debug/parity probe: copy one internal per-env field ("warm", "ncon", "solver_iter", ...) of all envs, row-major, to a
 * caller-owned device buffer of `count` floats.  Used by the parity tests only. */
int so101_debug_read(so101_handle h, const char *field, float *dst_dev, size_t count, void *stream);

/* Contact force sensors (MuJoCo's mj_contactForce summed over a body pair, with its `touch` / `contact` sensor values).  A sensor
 * is an ordered pair of disjoint, non-empty body sets (A, B), given as two 32-bit masks of body ids (bit b = body b of the
 * model), A first.  After every so101_step each sensor gives each user env one float32 row of 5 values, read from the contacts
 * of the LAST substep of the step - exactly those the Newton solve used (contacts dropped by a full buffer, or whose Jacobian
 * blocks did not fit the solver's pool, are not included; friction-loss and limit rows are not contacts):
 *   [0..2] net force on A from B, world frame, newtons;  [3] sum of the normal forces (>= 0);  [4] number of contacts.
 * Sign: for a contact between geom1 (body b1) and geom2 (body b2) with cone force f in the contact frame (normal from geom1 to
 * geom2, tangent 1, tangent 2), the force on b2 from b1 is F = f0 n + f1 t1 + f2 t2; the contact adds +F if b2 is in A and b1 in
 * B, -F if b1 is in A and b2 in B.  Torsional and rolling components are torques and are not reported.  f is the cone force at
 * the solver's final iterate.  Rows read all zeros for envs that return FIRST from the step (auto-reset), envs reset by
 * so101_reset or so101_sample_and_settle, envs whose step ended by divergence, and every env after so101_checkpoint_load until
 * the next step (the sensor configuration is not part of a checkpoint).  Arithmetic runs in the handle's precision, in a fixed
 * order: the same inputs give the same bits.
 * so101_contact_sensors sets n <= SO101_MAX_CONTACT_SENSORS sensors, masks_host[k] = {mask A, mask B}; n = 0 turns them off
 * (the default: the step then does no sensor work).  Returns negative for a handle without a contact scene, n out of range, an
 * empty mask, overlapping masks or a body >= nbody.  It drops the handle's captured step graphs.  The first call with n > 0
 * allocates the readout buffer (cudaMalloc, zero-filled, like the other lazily allocated buffers of a handle); later calls do no
 * device work and never synchronise.  The readout has the new layout from the next step on: read before it, it holds the
 * previous configuration's rows (zeros before any step).  With sensors on, a step adds one memset of the readout to its graph
 * (no kernel launch).
 * so101_contact_sensors_read copies the [N][n][5] float32 readout of the last step to dst_dev (count floats, at least N * n * 5)
 * with cudaMemcpyAsync on the caller's stream. */
int so101_contact_sensors(so101_handle h, int n, const uint32_t masks_host[][2]);
int so101_contact_sensors_read(so101_handle h, float *dst_dev, size_t count, void *stream);

/* End-effector queries.  The tool centre point (TCP) is a point fixed in each arm's Fixed_Jaw body (the body of its fifth hinge,
 * Wrist_Roll) at tcp_offset (metres, Fixed_Jaw frame); its orientation is the Fixed_Jaw frame.  Both functions run FK of the
 * arms in float64 in both precisions, one thread per (env, arm), only for the user envs.  They are enqueued on the caller's
 * stream, never synchronise the host, write only the caller's buffers and leave the handle's state and its captured step
 * graphs untouched.  narm = 1, or 2 for the two-arm build. */
typedef struct so101_ee_params {
  float tcp_offset[3];  /* TCP in the Fixed_Jaw frame (the library's Python layer derives the default from the jaw pads) */
  int iterations;       /* Levenberg-Marquardt iterations (>= 0; default 16) */
  float damping;        /* lambda (metres, > 0): the step solves (J J^T + lambda^2 I) y = e */
  float w_rot;          /* metres per radian of orientation error (>= 0; ignored without a target orientation) */
  float max_step;       /* per-joint clamp of one iteration's step (rad, > 0) */
  float tolerance;      /* stop early once |e| (metres, orientation part weighted by w_rot) < tolerance; 0 = never */
} so101_ee_params;
/* TCP pose of every user env and arm: the current joint state (from_ctrl = 0) or the current commanded joint targets
 * (from_ctrl != 0: ctrl, i.e. the last action plus the calibration offsets).  pos_dev [N,narm,3] float32 world position,
 * quat_dev [N,narm,4] float32 world orientation, wxyz (MuJoCo convention) with w >= 0 (nullable).  The reference has no
 * counterpart: reading the gripper pose there means restating the arm's kinematics on physics.named.data.xpos / xmat. */
int so101_ee_pose(so101_handle h, int from_ctrl, const float tcp_offset[3], float *pos_dev, float *quat_dev, void *stream);
/* Batched inverse kinematics to joint-target actions.  Replaces the reference planner's geometric stand-in
 * inverse_kinematics_approximate (examples/automated_lerobot_dataset_generator.py:188-212), which does not place the jaws at
 * the target.  Damped least squares on the five arm hinges of each arm (the jaw is excluded), started from the env's current
 * joint state or from seed_q_dev ([N,nu] float32 joint positions, nullable):
 *   e = (p_target - p_tcp, w_rot * rotation vector of R_target R_tcp^T), Jacobian columns (a_i x (p_tcp - p_i), w_rot * a_i),
 *   dq = J^T y with (J J^T + damping^2 I) y = e, each component clamped to +-max_step, then q clamped to the joint range,
 * for p->iterations iterations (fewer once |e| < tolerance).  target_pos_dev [N,narm,3]; target_quat_dev [N,narm,4] wxyz,
 * nullable = position only (w_rot is then 0).  action_out_dev [N,nu] float32 receives ACTIONS, q - calibration_offsets, since
 * the step adds the offsets back; its jaw entries are gripper_dev [N,narm] unchanged (nullable: the current commanded jaw
 * target minus its offset).  err_out_dev [N,narm,2] (nullable): final position error (m) and orientation error (rad, 0 without
 * a target orientation).  Targets are not validated: an unreachable target gives finite joint targets inside the joint range
 * and shows only in err_out_dev.  The parameters are validated (negative return on a bad one).  Deterministic: the same
 * inputs give the same bits. */
int so101_ee_ik(so101_handle h, const float *target_pos_dev, const float *target_quat_dev, const float *gripper_dev, const float *seed_q_dev,
                const so101_ee_params *p, float *action_out_dev, float *err_out_dev, void *stream);

/* Parity probe without a handle: the device's 6-axis box overlap test (the reward geometry, so101_sim/utils/oobb_utils.py:202-273)
 * on n box pairs, rows of 20 doubles (pos 3, quat 4 wxyz, half 3 of box A, then of box B), evaluated in float32 or float64
 * (precision = 32 / 64) -> out[i] in {0, 1}.  Used by the golden-vector test of the reward geometry only. */
int so101_debug_overlap(int precision, int device, const double *cases_dev, int n, uint8_t *out_dev, void *stream);

#ifdef __cplusplus
}
#endif
#endif
