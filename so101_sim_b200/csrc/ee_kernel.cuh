#pragma once
#include <cuda_runtime.h>
#include "arm_dynamics.cuh"

namespace so101 {

// Where the arm joint angles of the user envs live: the float64 state S.qpos [N][nq] and the commanded targets S.ctrl [N][NA]
// (float32 or float64 as the handle's precision).
struct EeSrc {
  const double *qpos;
  const void *ctrl;
  int ctrl_f64;   // S.ctrl holds doubles (precision 64) rather than floats
  int NU, nq;     // NU = user envs
  float offsets[NJ];  // calibration offsets: ctrl = action + offsets
};

struct EeIkArgs {
  const float *target_pos;   // [NU][NARM][3]
  const float *target_quat;  // [NU][NARM][4] wxyz, or null: position only
  const float *gripper;      // [NU][NARM] jaw actions, or null: keep the commanded jaw target
  const float *seed_q;       // [NU][NA] joint positions to start from, or null: the current state
  float tcp[3];
  int iterations;
  double damping, w_rot, max_step, tolerance;
  float *action;             // [NU][NA]
  float *err;                // [NU][NARM][2] or null
};

void launch_ee_pose(const ArmSetT<double> &am, const EeSrc &src, int from_ctrl, const float tcp[3], float *pos, float *quat,
                    cudaStream_t stream);
void launch_ee_ik(const ArmSetT<double> &am, const EeSrc &src, const EeIkArgs &a, cudaStream_t stream);

}  // namespace so101
