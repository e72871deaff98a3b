// Fused control-step kernel for the ARM-ONLY scene (BASELINE config 2: nq = nv = nu = 6, collisions off).
//
// One env per thread; the whole control step — action -> ctrl (so100_task.py:266-287), 10 x {FK, CRB, RNE, actuation,
// M^-1, friction-loss/limit Newton solve, semi-implicit Euler} ([upstream] mj_step; Euler is MuJoCo's default
// integrator, scene_pbr.xml:4), observation delay rings (so100_task.py:189-210), reward (= 0 for the base task,
// so100_task.py:289-290), time limit and dm_control's auto-reset — is ONE launch.  State is read once and written once
// per control step (its row of every state array); nothing else touches HBM.
#include "arm_kernel.cuh"

namespace so101 {

// What write_obs reads: the env's state and commanded targets, held in registers by the kernels below.
template <typename T>
struct ArmObs { const TS *q, *qd; const T *ctrl; };

template <typename T>
__device__ __forceinline__ void reset_env_arm(const StepCfg &cfg, const EnvState<T> &S, const so101_step_out &out, int env) {
  TS q[NJ], qd[NJ];
  T ctrl[NJ];
  const int ep = S.episode[env];
  const size_t pool = ((size_t)(ep % S.npool) * S.N + env) * NJ;  // reset pool entry of this episode
  const int row = env * NJ;
  S.episode[env] = ep + 1;
#pragma unroll
  for (int i = 0; i < NJ; i++) {
    q[i] = S.init_qpos[pool + i]; qd[i] = S.init_qvel[pool + i];
    ctrl[i] = (T)cfg.home[i] + (T)cfg.offsets[i];  // so100_task.py:316-317
    S.qpos[row + i] = q[i]; S.qvel[row + i] = qd[i]; S.warm[row + i] = T(0); S.ctrl[row + i] = ctrl[i];
  }
  S.step[env] = 0;
  S.needs_reset[env] = 0;
  // FIRST TimeStep: reward / discount are None in dm_env; the batched tensors carry 0 / 1.
  write_obs<NJ, NJ, NJ, 1>(cfg, S, out, ArmObs<T>{q, qd, ctrl}, env, 0, 0.f, 1.f, SO101_STEP_FIRST, 0);
}

// T = arithmetic of the friction-loss / limit Newton solve.  The smooth dynamics (FK, CRB, RNE), the actuators, the M^-1 solve
// for qacc_smooth and the Euler update run in float64 on the float64 state in both precisions (env_state.cuh): measured
// against the float64 oracle over 100 control steps, 32 envs, float32 throughout drifts to 1.8e-3 relative, float64 smooth
// dynamics with float32 actuators or M^-1 solve to 1.5e-4 .. 2.3e-4, this split to 9.4e-6, at 481 vs 460 us per 4096-env
// control step (profiles/r2c_arm_precision.jsonl).  amd: the float64 arm model.
template <typename T>
__global__ void __launch_bounds__(128) arm_step_kernel(const __grid_constant__ ArmModelT<T> am, const __grid_constant__ ArmModelT<double> amd,
                                                      const __grid_constant__ StepCfg cfg, const EnvState<T> S, const float *__restrict__ action,
                                                      const so101_step_out out) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= S.N) return;
  if (S.needs_reset[env]) {  // dm_control: the step() after a LAST step resets and returns FIRST
    reset_env_arm(cfg, S, out, env);
    return;
  }
  const int row = env * NJ;   // (32-bit: at 255 registers a 64-bit index costs the float32 kernel stack and spills)
  TS q[NJ], qd[NJ];
  T warm[NJ], ctrl[NJ];
#pragma unroll
  for (int i = 0; i < NJ; i++) {
    q[i] = S.qpos[row + i]; qd[i] = S.qvel[row + i]; warm[i] = S.warm[row + i];
    ctrl[i] = (T)action[env * 6 + i] + (T)cfg.offsets[i];  // before_step: action + homing offsets, unclamped
  }
  int iters = 0;
  bool bad = false;
  for (int sub = 0; sub < cfg.nsub; sub++) {
    ArmKin<double> k;
    arm_fk<double>(amd, q, k, nullptr);
    double Md[21], biasd[NJ];
    arm_crb_rne(amd, k, qd, Md, biasd);
    T M[21], qacc_s[NJ];
#pragma unroll
    for (int i = 0; i < 21; i++) M[i] = (T)Md[i];
    double frc[NJ];
    arm_actuation_d(am, q, qd, ctrl, frc);
    double L[21], rhs[NJ];
#pragma unroll
    for (int i = 0; i < 21; i++) L[i] = Md[i];
    chol6(L);
#pragma unroll
    for (int i = 0; i < NJ; i++) rhs[i] = frc[i] - biasd[i];
    chol6_solve(L, rhs);
    TS qacc_sd[NJ];
#pragma unroll
    for (int i = 0; i < NJ; i++) { qacc_sd[i] = (TS)rhs[i]; qacc_s[i] = (T)rhs[i]; }
    T qt[NJ], qdt[NJ];
#pragma unroll
    for (int i = 0; i < NJ; i++) { qt[i] = (T)q[i]; qdt[i] = (T)qd[i]; }
    ArmRows<T> rows;
    arm_make_rows(am, qt, qdt, qacc_s, rows);
    T delta[NJ];
#pragma unroll
    for (int i = 0; i < NJ; i++) delta[i] = warm[i] - qacc_s[i];
    iters = arm_solve(am, M, rows, delta, cfg.max_iter, (T)cfg.tol);
    TS corr[NJ] = {TS(0), TS(0), TS(0), TS(0), TS(0), TS(0)};
    if (cfg.integrator == 1) {  // implicitfast: velocity update with (M - h D)^-1 M qacc instead of qacc
      const unsigned vm = arm_actuation_vel_mask(am, frc);
      double qa[NJ], dv[NJ], cr[NJ];
#pragma unroll
      for (int i = 0; i < NJ; i++) { qa[i] = qacc_sd[i] + (TS)delta[i]; dv[i] = ((vm >> i) & 1u) ? am.bias_d[i][2] : 0.0; }
      implicitfast_correction<double>(Md, dv, am.dt_d, qa, cr);
#pragma unroll
      for (int i = 0; i < NJ; i++) corr[i] = (TS)cr[i];
    }
#pragma unroll
    for (int i = 0; i < NJ; i++) {
      const TS qacc = qacc_sd[i] + (TS)delta[i];
      warm[i] = (T)qacc;
      bad |= !(t_abs(qacc) < TS(1e10));  // [upstream] mj_checkAcc (also catches NaN)
      qd[i] += am.dt_d * (qacc + corr[i]);  // [upstream] mj_Euler: velocity first, then position with the new velocity
      q[i] += am.dt_d * qd[i];
    }
  }
  const int t = S.step[env] + 1;
  S.step[env] = t;
  S.solver_iter[env] = iters;
  float reward = 0.f, discount = 1.f;  // SO100Task.get_reward / get_discount (so100_task.py:289-295)
  uint8_t st = (cfg.last_step > 0 && t >= cfg.last_step) ? SO101_STEP_LAST : SO101_STEP_MID;
  if (bad) {  // PhysicsError path (task_suite.py:153): reward 0, discount 0, episode ends
    discount = 0.f; st = SO101_STEP_LAST;
    atomicAdd(S.diverged_count, 1);
  }
  S.needs_reset[env] = st == SO101_STEP_LAST;
#pragma unroll
  for (int i = 0; i < NJ; i++) {
    S.qpos[row + i] = q[i]; S.qvel[row + i] = qd[i]; S.warm[row + i] = warm[i]; S.ctrl[row + i] = ctrl[i];
  }
  write_obs<NJ, NJ, NJ, 1>(cfg, S, out, ArmObs<T>{q, qd, ctrl}, env, t, reward, discount, st, 0);
}

template <typename T>
__global__ void arm_reset_kernel(const __grid_constant__ StepCfg cfg, const EnvState<T> S, const uint8_t *__restrict__ mask, const so101_step_out out) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= S.N) return;
  if (mask && !mask[env]) return;
  reset_env_arm(cfg, S, out, env);
}

template <typename T>
void launch_arm_step(const ArmModelT<T> &am, const ArmModelT<double> &am64, const StepCfg &cfg, const EnvState<T> &S, const float *action,
                     const so101_step_out &out, cudaStream_t stream) {
  // one env per thread; small batches use 32-thread CTAs so that every one of the 148 SMs gets work
  const int threads = S.N <= 148 * 32 * 4 ? 32 : (S.N <= 148 * 64 * 4 ? 64 : 128);
  const int grid = (S.N + threads - 1) / threads;
  arm_step_kernel<T><<<grid, threads, 0, stream>>>(am, am64, cfg, S, action, out);
}
template <typename T>
void launch_arm_reset(const StepCfg &cfg, const EnvState<T> &S, const uint8_t *mask, const so101_step_out &out, cudaStream_t stream) {
  const int threads = 128;
  arm_reset_kernel<T><<<(S.N + threads - 1) / threads, threads, 0, stream>>>(cfg, S, mask, out);
}

template void launch_arm_step<float>(const ArmModelT<float> &, const ArmModelT<double> &, const StepCfg &, const EnvState<float> &, const float *, const so101_step_out &, cudaStream_t);
template void launch_arm_step<double>(const ArmModelT<double> &, const ArmModelT<double> &, const StepCfg &, const EnvState<double> &, const float *, const so101_step_out &, cudaStream_t);
template void launch_arm_reset<float>(const StepCfg &, const EnvState<float> &, const uint8_t *, const so101_step_out &, cudaStream_t);
template void launch_arm_reset<double>(const StepCfg &, const EnvState<double> &, const uint8_t *, const so101_step_out &, cudaStream_t);

}  // namespace so101
