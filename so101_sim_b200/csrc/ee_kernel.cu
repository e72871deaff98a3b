// End-effector queries on the device: the pose of the tool centre point (TCP) and a batched damped-least-squares inverse
// kinematics towards TCP targets, one thread per (env, arm), float64 arithmetic in both precisions on the float64 arm model.
//
// The TCP is a point fixed in the Fixed_Jaw body (the body of each arm's fifth hinge, Wrist_Roll; FK slot NJ - 2) at a
// caller-given offset; its orientation is the Fixed_Jaw frame.  Neither kernel writes handle state: they read the state or the
// commanded targets and write caller-owned buffers only, outside the captured step graph.
#include "ee_kernel.cuh"

namespace so101 {

namespace {

constexpr int TCP_BODY = NJ - 2;   // Fixed_Jaw
constexpr int IK_JOINTS = NJ - 1;  // the five arm hinges; the jaw is left to the caller's command

__device__ __forceinline__ double load_joint(const EeSrc &s, int env, int j, bool from_ctrl) {
  if (from_ctrl) {
    const size_t i = (size_t)env * NA + j;
    return s.ctrl_f64 ? static_cast<const double *>(s.ctrl)[i] : (double)static_cast<const float *>(s.ctrl)[i];
  }
  return s.qpos[(size_t)env * s.nq + j];
}

// Unit quaternion (w, x, y, z), w >= 0, of a row-major rotation matrix (Shepperd's method: divide by the largest of the four
// candidates, so that no branch loses precision near a 180 degree rotation).
__device__ __forceinline__ void mat2quat(const double (&R)[9], double (&q)[4]) {
  const double tr = R[0] + R[4] + R[8];
  if (tr > 0.0) {
    const double s = 2.0 * sqrt(1.0 + tr);
    q[0] = 0.25 * s; q[1] = (R[7] - R[5]) / s; q[2] = (R[2] - R[6]) / s; q[3] = (R[3] - R[1]) / s;
  } else if (R[0] > R[4] && R[0] > R[8]) {
    const double s = 2.0 * sqrt(1.0 + R[0] - R[4] - R[8]);
    q[0] = (R[7] - R[5]) / s; q[1] = 0.25 * s; q[2] = (R[1] + R[3]) / s; q[3] = (R[2] + R[6]) / s;
  } else if (R[4] > R[8]) {
    const double s = 2.0 * sqrt(1.0 + R[4] - R[0] - R[8]);
    q[0] = (R[2] - R[6]) / s; q[1] = (R[1] + R[3]) / s; q[2] = 0.25 * s; q[3] = (R[5] + R[7]) / s;
  } else {
    const double s = 2.0 * sqrt(1.0 + R[8] - R[0] - R[4]);
    q[0] = (R[3] - R[1]) / s; q[1] = (R[2] + R[6]) / s; q[2] = (R[5] + R[7]) / s; q[3] = 0.25 * s;
  }
  const double n = 1.0 / sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  const double sg = q[0] < 0.0 ? -n : n;
#pragma unroll
  for (int c = 0; c < 4; c++) q[c] *= sg;
}

// Rotation vector (world frame, angle in [0, pi]) of R_target R_tcp^T, from the unit target quaternion qt.
__device__ __forceinline__ V3<double> rot_error(const double (&qt)[4], const double (&R)[9]) {
  double qc[4];
  mat2quat(R, qc);
  // d = qt * conj(qc)
  double w = qt[0] * qc[0] + qt[1] * qc[1] + qt[2] * qc[2] + qt[3] * qc[3];
  V3<double> v = {-qt[0] * qc[1] + qt[1] * qc[0] - qt[2] * qc[3] + qt[3] * qc[2],
                  -qt[0] * qc[2] + qt[1] * qc[3] + qt[2] * qc[0] - qt[3] * qc[1],
                  -qt[0] * qc[3] - qt[1] * qc[2] + qt[2] * qc[1] + qt[3] * qc[0]};
  if (w < 0.0) { w = -w; v = -1.0 * v; }
  const double s = sqrt(dot(v, v));
  return s > 0.0 ? (2.0 * atan2(s, w) / s) * v : 2.0 * v;
}

// TCP position and Fixed_Jaw rotation of one arm; k receives every link's origin and world axis.
__device__ __forceinline__ V3<double> tcp_fk(const ArmModelT<double> &am, const double (&q)[NJ], V3<double> off, ArmKin<double> &k,
                                             double (&R)[9]) {
  double Rb[NJ][9];
  arm_fk<double>(am, q, k, Rb);
#pragma unroll
  for (int e = 0; e < 9; e++) R[e] = Rb[TCP_BODY][e];
  return k.p[TCP_BODY] + mv(R, off);
}

}  // namespace

__global__ void __launch_bounds__(128) ee_pose_kernel(const __grid_constant__ ArmSetT<double> am, const __grid_constant__ EeSrc src,
                                                      int from_ctrl, float tx, float ty, float tz, float *__restrict__ pos,
                                                      float *__restrict__ quat) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= src.NU * NARM) return;
  const int env = t / NARM, arm = t - env * NARM;
  double q[NJ];
#pragma unroll
  for (int i = 0; i < NJ; i++) q[i] = load_joint(src, env, NJ * arm + i, from_ctrl != 0);
  ArmKin<double> k;
  double R[9];
  const V3<double> p = tcp_fk(am[arm], q, V3<double>{(double)tx, (double)ty, (double)tz}, k, R);
  pos[3 * t] = (float)p.x; pos[3 * t + 1] = (float)p.y; pos[3 * t + 2] = (float)p.z;
  if (quat) {
    double qq[4];
    mat2quat(R, qq);
#pragma unroll
    for (int c = 0; c < 4; c++) quat[4 * t + c] = (float)qq[c];
  }
}

// Levenberg-Marquardt on the five arm hinges.  Error e = (p_target - p_tcp, w_rot * rotvec(R_target R_tcp^T)); Jacobian
// columns (a_i x (p_tcp - p_i), w_rot * a_i); step dq = J^T y with (J J^T + damping^2 I) y = e (6x6 Cholesky), every component
// clamped to +-max_step, then q clamped to the range of limited joints.  `iterations` steps, or fewer once |e| < tolerance.
__global__ void __launch_bounds__(128) ee_ik_kernel(const __grid_constant__ ArmSetT<double> am, const __grid_constant__ EeSrc src,
                                                    const __grid_constant__ EeIkArgs a) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= src.NU * NARM) return;
  const int env = t / NARM, arm = t - env * NARM, o = NJ * arm;
  const ArmModelT<double> &m = am[arm];
  double q[NJ];
#pragma unroll
  for (int i = 0; i < NJ; i++) q[i] = a.seed_q ? (double)a.seed_q[(size_t)env * NA + o + i] : load_joint(src, env, o + i, false);
  const V3<double> tp = {(double)a.target_pos[3 * t], (double)a.target_pos[3 * t + 1], (double)a.target_pos[3 * t + 2]};
  const V3<double> off = {(double)a.tcp[0], (double)a.tcp[1], (double)a.tcp[2]};
  const bool orient = a.target_quat != nullptr;
  double qt[4] = {1.0, 0.0, 0.0, 0.0};
  double w = 0.0;
  if (orient) {
    double n = 0.0;
#pragma unroll
    for (int c = 0; c < 4; c++) { qt[c] = (double)a.target_quat[4 * t + c]; n += qt[c] * qt[c]; }
    n = n > 0.0 ? 1.0 / sqrt(n) : 0.0;
#pragma unroll
    for (int c = 0; c < 4; c++) qt[c] *= n;
    w = a.w_rot;
  }
  const double lam2 = a.damping * a.damping;
  double perr = 0.0, rerr = 0.0;
#pragma unroll 1
  for (int it = 0;; it++) {
    ArmKin<double> k;
    double R[9];
    const V3<double> p = tcp_fk(m, q, off, k, R);
    const V3<double> ep = tp - p;
    const V3<double> rv = orient ? rot_error(qt, R) : V3<double>{0.0, 0.0, 0.0};
    perr = sqrt(dot(ep, ep)); rerr = sqrt(dot(rv, rv));
    const double e[NJ] = {ep.x, ep.y, ep.z, w * rv.x, w * rv.y, w * rv.z};
    if (it >= a.iterations || sqrt(perr * perr + w * w * rerr * rerr) < a.tolerance) break;
    double J[NJ][IK_JOINTS];
#pragma unroll
    for (int i = 0; i < IK_JOINTS; i++) {
      const V3<double> jp = cross(k.a[i], p - k.p[i]);
      J[0][i] = jp.x; J[1][i] = jp.y; J[2][i] = jp.z;
      J[3][i] = w * k.a[i].x; J[4][i] = w * k.a[i].y; J[5][i] = w * k.a[i].z;
    }
    double A[21], y[NJ];
#pragma unroll
    for (int r = 0; r < NJ; r++) {
      y[r] = e[r];
#pragma unroll
      for (int c = 0; c <= r; c++) {
        double s = r == c ? lam2 : 0.0;
#pragma unroll
        for (int i = 0; i < IK_JOINTS; i++) s += J[r][i] * J[c][i];
        A[r * (r + 1) / 2 + c] = s;
      }
    }
    chol6(A);
    chol6_solve(A, y);
#pragma unroll
    for (int i = 0; i < IK_JOINTS; i++) {
      double dq = 0.0;
#pragma unroll
      for (int r = 0; r < NJ; r++) dq += J[r][i] * y[r];
      q[i] += t_clamp(dq, -a.max_step, a.max_step);
      if (m.limited[i]) q[i] = t_clamp(q[i], m.range[i][0], m.range[i][1]);
    }
  }
  // the step adds the calibration offsets back (ctrl = action + offsets)
  float *act = a.action + (size_t)env * NA + o;
#pragma unroll
  for (int i = 0; i < IK_JOINTS; i++) act[i] = (float)(q[i] - (double)src.offsets[i]);
  act[NJ - 1] = a.gripper ? a.gripper[t] : (float)(load_joint(src, env, o + NJ - 1, true) - (double)src.offsets[NJ - 1]);
  if (a.err) { a.err[2 * t] = (float)perr; a.err[2 * t + 1] = (float)rerr; }
}

void launch_ee_pose(const ArmSetT<double> &am, const EeSrc &src, int from_ctrl, const float tcp[3], float *pos, float *quat,
                    cudaStream_t stream) {
  const int n = src.NU * NARM, threads = 128;
  ee_pose_kernel<<<(n + threads - 1) / threads, threads, 0, stream>>>(am, src, from_ctrl, tcp[0], tcp[1], tcp[2], pos, quat);
}

void launch_ee_ik(const ArmSetT<double> &am, const EeSrc &src, const EeIkArgs &a, cudaStream_t stream) {
  const int n = src.NU * NARM, threads = 128;
  ee_ik_kernel<<<(n + threads - 1) / threads, threads, 0, stream>>>(am, src, a);
}

}  // namespace so101
