// Per-thread (one env per thread, everything in registers) dynamics of the 6-hinge SO100 arm chain.
//
// Replaces, for the arm bodies of scene_pbr.xml:74-126, what the reference obtains from MuJoCo inside mj_step:
//   mj_kinematics + mj_comPos  -> arm_fk()
//   mj_crb (+ armature)        -> arm_crb_rne()   (world-frame composite-rigid-body sweep, tip -> base)
//   mj_rne (bias forces)       -> arm_crb_rne()   (same sweep; velocity-product accelerations, gravity as base accel)
//   mj_fwdActuation            -> arm_actuation_d() (scene_pbr.xml:11: gain 50, bias "0 -50 1", ctrl/force clamps)
// Templated on the scalar so the same code runs in float32 (north_star dtype) and float64 (tight-parity mode).
#pragma once
#include <cuda_runtime.h>

namespace so101 {

#ifndef SO101_NARM
#define SO101_NARM 1
#endif
// Arms in the scene: 1 = the reference's SO100 scenes (libso101_b200.so); 2 = the labelled synthetic two-arm hand-over scene of
// BASELINE config 4 (libso101_b200_2arm.so, the same sources compiled with -DSO101_NARM=2).  State layout: arm 0's six hinge
// dofs, arm 1's, then the free props.
constexpr int NARM = SO101_NARM;
constexpr int NJ = 6;          // hinge joints = dofs = actuators of ONE arm
constexpr int NA = NJ * NARM;  // arm dofs (= actuators) of the scene; the props' dofs follow

template <typename T>
struct ArmModelT {
  T base_pos[3], base_R[9];  // pose of the (static) parent of joint 0 in the world frame
  T pos[NJ][3];              // body_pos in the parent frame
  T R0[NJ][9];               // body_quat as a rotation matrix (parent <- child at q = qpos0)
  T axis[NJ][3];             // hinge axis, child frame (unit)
  T ipos[NJ][3];             // COM in the child frame
  T Iloc[NJ][6];             // inertia about the COM in the child frame: xx yy zz xy xz yz
  T mass[NJ];
  T qpos0[NJ];
  T armature[NJ], frictionloss[NJ];
  // friction-loss rows (J = e_i, pos = 0): constant R, D and velocity gain B   [upstream mj_makeImpedance]
  T fr_R[NJ], fr_D[NJ], fr_B[NJ];
  // joint limit rows
  T range[NJ][2];
  int limited[NJ];
  T lim_solimp[NJ][5], lim_K[NJ], lim_B[NJ], invweight0[NJ];
  T gravity[3], dt, solver_scale;  // solver_scale = 1 / (meaninertia * max(1, nv))
  // actuators and the Euler update step: float64 in both precisions (env_state.cuh)
  double gain_d[NJ], bias_d[NJ][3], ctrlrange_d[NJ][2], forcerange_d[NJ][2], dt_d;
};

// the scene's arms (kernel parameter); scalars shared by all arms (dt, gravity, solver_scale) are read from arm 0
template <typename T>
struct ArmSetT {
  ArmModelT<T> arm[NARM];
  __host__ __device__ const ArmModelT<T> &operator[](int k) const { return arm[k]; }
};

template <typename T> __device__ __forceinline__ T t_sqrt(T x);
template <> __device__ __forceinline__ float t_sqrt<float>(float x) { return sqrtf(x); }
template <> __device__ __forceinline__ double t_sqrt<double>(double x) { return sqrt(x); }
template <typename T> __device__ __forceinline__ void t_sincos(T x, T *s, T *c);
template <> __device__ __forceinline__ void t_sincos<float>(float x, float *s, float *c) { sincosf(x, s, c); }
template <> __device__ __forceinline__ void t_sincos<double>(double x, double *s, double *c) { sincos(x, s, c); }
template <typename T> __device__ __forceinline__ T t_abs(T x) { return x < T(0) ? -x : x; }
template <typename T> __device__ __forceinline__ T t_pow(T x, T y);
template <> __device__ __forceinline__ float t_pow<float>(float x, float y) { return powf(x, y); }
template <> __device__ __forceinline__ double t_pow<double>(double x, double y) { return pow(x, y); }
template <typename T> __device__ __forceinline__ T t_clamp(T x, T lo, T hi) { return x < lo ? lo : (x > hi ? hi : x); }

template <typename T>
struct V3 {
  T x, y, z;
};
template <typename T> __device__ __forceinline__ V3<T> operator+(V3<T> a, V3<T> b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
template <typename T> __device__ __forceinline__ V3<T> operator-(V3<T> a, V3<T> b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
template <typename T> __device__ __forceinline__ V3<T> operator*(T s, V3<T> a) { return {s * a.x, s * a.y, s * a.z}; }
template <typename T> __device__ __forceinline__ T dot(V3<T> a, V3<T> b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
template <typename T> __device__ __forceinline__ V3<T> cross(V3<T> a, V3<T> b) {
  return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x};
}
template <typename T> __device__ __forceinline__ V3<T> ld3(const T *p) { return {p[0], p[1], p[2]}; }
// r = M v (row-major 3x3)
template <typename T> __device__ __forceinline__ V3<T> mv(const T *m, V3<T> v) {
  return {m[0] * v.x + m[1] * v.y + m[2] * v.z, m[3] * v.x + m[4] * v.y + m[5] * v.z, m[6] * v.x + m[7] * v.y + m[8] * v.z};
}
template <typename T> __device__ __forceinline__ void mm(T *r, const T *a, const T *b) {
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int j = 0; j < 3; j++) r[3 * i + j] = a[3 * i] * b[j] + a[3 * i + 1] * b[3 + j] + a[3 * i + 2] * b[6 + j];
}
// symmetric 3x3 (xx yy zz xy xz yz) times vector
template <typename T> __device__ __forceinline__ V3<T> symv(const T *s, V3<T> v) {
  return {s[0] * v.x + s[3] * v.y + s[4] * v.z, s[3] * v.x + s[1] * v.y + s[5] * v.z, s[4] * v.x + s[5] * v.y + s[2] * v.z};
}

// Per-link world-frame kinematic state kept in registers between the forward and the backward sweep.
template <typename T>
struct ArmKin {
  V3<T> p[NJ];   // joint anchor = body origin
  V3<T> a[NJ];   // hinge axis (world)
  V3<T> c[NJ];   // link COM (world)
  T Iw[NJ][6];   // link inertia about its COM, world axes (xx yy zz xy xz yz)
};

// Forward kinematics.  If R_out != nullptr the 6 body rotation matrices are also returned (collision needs them).
template <typename T>
__device__ __forceinline__ void arm_fk(const ArmModelT<T> &am, const T (&q)[NJ], ArmKin<T> &k, T (*R_out)[9]) {
  T R[9];
  V3<T> p = ld3(am.base_pos);
#pragma unroll
  for (int i = 0; i < 9; i++) R[i] = am.base_R[i];
#pragma unroll
  for (int i = 0; i < NJ; i++) {
    p = p + mv(R, ld3(am.pos[i]));
    T Rb[9];
    mm(Rb, R, am.R0[i]);
    // Rodrigues rotation about the child-frame axis by q - qpos0
    T s, c;
    t_sincos(q[i] - am.qpos0[i], &s, &c);
    const T ax = am.axis[i][0], ay = am.axis[i][1], az = am.axis[i][2], v = T(1) - c;
    const T Rj[9] = {c + ax * ax * v,      ax * ay * v - az * s, ax * az * v + ay * s,
                     ay * ax * v + az * s, c + ay * ay * v,      ay * az * v - ax * s,
                     az * ax * v - ay * s, az * ay * v + ax * s, c + az * az * v};
    mm(R, Rb, Rj);
    k.p[i] = p;
    k.a[i] = mv(R, ld3(am.axis[i]));
    k.c[i] = p + mv(R, ld3(am.ipos[i]));
    // Iw = R Iloc R^T
    const T *L = am.Iloc[i];
    T t[9];  // t = R * Iloc
#pragma unroll
    for (int r = 0; r < 3; r++) {
      t[3 * r + 0] = R[3 * r] * L[0] + R[3 * r + 1] * L[3] + R[3 * r + 2] * L[4];
      t[3 * r + 1] = R[3 * r] * L[3] + R[3 * r + 1] * L[1] + R[3 * r + 2] * L[5];
      t[3 * r + 2] = R[3 * r] * L[4] + R[3 * r + 1] * L[5] + R[3 * r + 2] * L[2];
    }
    k.Iw[i][0] = t[0] * R[0] + t[1] * R[1] + t[2] * R[2];
    k.Iw[i][1] = t[3] * R[3] + t[4] * R[4] + t[5] * R[5];
    k.Iw[i][2] = t[6] * R[6] + t[7] * R[7] + t[8] * R[8];
    k.Iw[i][3] = t[0] * R[3] + t[1] * R[4] + t[2] * R[5];
    k.Iw[i][4] = t[0] * R[6] + t[1] * R[7] + t[2] * R[8];
    k.Iw[i][5] = t[3] * R[6] + t[4] * R[7] + t[5] * R[8];
    if (R_out) {
#pragma unroll
      for (int e = 0; e < 9; e++) R_out[i][e] = R[e];
    }
  }
}

// Mass matrix (packed lower triangle M[i*(i+1)/2 + j], j <= i, armature included) and bias forces in one
// forward (velocities / velocity-product accelerations) + backward (composite inertia, force suffix sums) sweep.
template <typename T>
__device__ __forceinline__ void arm_crb_rne(const ArmModelT<T> &am, const ArmKin<T> &k, const T (&qd)[NJ], T (&M)[21], T (&bias)[NJ]) {
  V3<T> f[NJ], n[NJ];  // inertial force on link i and its moment about the world origin
  {
    V3<T> w = {T(0), T(0), T(0)}, al = {T(0), T(0), T(0)};
    V3<T> ao = {-am.gravity[0], -am.gravity[1], -am.gravity[2]};  // gravity as base acceleration
    V3<T> pp = ld3(am.base_pos);
#pragma unroll
    for (int i = 0; i < NJ; i++) {
      V3<T> r = k.p[i] - pp;
      ao = ao + cross(al, r) + cross(w, cross(w, r));
      al = al + qd[i] * cross(w, k.a[i]);
      w = w + qd[i] * k.a[i];
      pp = k.p[i];
      V3<T> rc = k.c[i] - k.p[i];
      V3<T> ac = ao + cross(al, rc) + cross(w, cross(w, rc));
      f[i] = am.mass[i] * ac;
      V3<T> tau = symv(k.Iw[i], al) + cross(w, symv(k.Iw[i], w));
      n[i] = tau + cross(k.c[i], f[i]);
    }
  }
  // backward: composite spatial inertia about the world origin (mass, h = m c, Io) and force suffix sums
  T cm = T(0);
  V3<T> ch = {T(0), T(0), T(0)}, F = {T(0), T(0), T(0)}, N = {T(0), T(0), T(0)};
  T Io[6] = {T(0), T(0), T(0), T(0), T(0), T(0)};
#pragma unroll
  for (int i = NJ - 1; i >= 0; i--) {
    const T m = am.mass[i];
    const V3<T> c = k.c[i];
    cm += m;
    ch = ch + m * c;
    const T cc = dot(c, c);
    Io[0] += k.Iw[i][0] + m * (cc - c.x * c.x);
    Io[1] += k.Iw[i][1] + m * (cc - c.y * c.y);
    Io[2] += k.Iw[i][2] + m * (cc - c.z * c.z);
    Io[3] += k.Iw[i][3] - m * c.x * c.y;
    Io[4] += k.Iw[i][4] - m * c.x * c.z;
    Io[5] += k.Iw[i][5] - m * c.y * c.z;
    F = F + f[i];
    N = N + n[i];
    const V3<T> a = k.a[i], v = cross(k.p[i], a);  // motion axis: angular a, linear velocity of the origin p x a
    bias[i] = dot(a, N) + dot(v, F);
    const V3<T> l = cm * v + cross(a, ch);          // momentum of the composite body under unit joint velocity
    const V3<T> h = symv(Io, a) + cross(ch, v);
#pragma unroll
    for (int j = 0; j <= i; j++) {
      const V3<T> aj = k.a[j], vj = cross(k.p[j], aj);
      M[i * (i + 1) / 2 + j] = dot(aj, h) + dot(vj, l);
    }
    M[i * (i + 1) / 2 + i] += am.armature[i];
  }
}

// Actuator forces, evaluated in float64 on the float64 integration state in both precisions (the -50 q position feedback would
// otherwise see the state rounded to float32: 50 * 3e-8 / armature 0.1 = 1.5e-5 rad/s^2 of noise per substep).
template <typename T>
__device__ __forceinline__ void arm_actuation_d(const ArmModelT<T> &am, const double (&q)[NJ], const double (&qd)[NJ], const T (&ctrl)[NJ],
                                                double (&frc)[NJ]) {
#pragma unroll
  for (int i = 0; i < NJ; i++) {
    const double c = t_clamp((double)ctrl[i], am.ctrlrange_d[i][0], am.ctrlrange_d[i][1]);
    const double f = am.gain_d[i] * c + am.bias_d[i][0] + am.bias_d[i][1] * q[i] + am.bias_d[i][2] * qd[i];
    frc[i] = t_clamp(f, am.forcerange_d[i][0], am.forcerange_d[i][1]);
  }
}

// [upstream] mjd_actuator_vel for this actuator model: d force / d velocity = biasprm[2] (gear 1) unless the force is clamped by
// forcerange.  Bit i of the result is set when actuator i contributes.
template <typename T>
__device__ __forceinline__ unsigned arm_actuation_vel_mask(const ArmModelT<T> &am, const double (&frc)[NJ]) {
  unsigned m = 0;
#pragma unroll
  for (int i = 0; i < NJ; i++)
    if (frc[i] > am.forcerange_d[i][0] && frc[i] < am.forcerange_d[i][1]) m |= 1u << i;
  return m;
}

// In-place Cholesky of a packed lower-triangular SPD matrix, n = 6.
template <typename T>
__device__ __forceinline__ void chol6(T (&A)[21]) {
#pragma unroll
  for (int j = 0; j < NJ; j++) {
    T s = A[j * (j + 1) / 2 + j];
#pragma unroll
    for (int k = 0; k < j; k++) s -= A[j * (j + 1) / 2 + k] * A[j * (j + 1) / 2 + k];
    s = t_sqrt(s > T(1e-30) ? s : T(1e-30));
    A[j * (j + 1) / 2 + j] = s;
    const T inv = T(1) / s;
#pragma unroll
    for (int i = j + 1; i < NJ; i++) {
      T t = A[i * (i + 1) / 2 + j];
#pragma unroll
      for (int k = 0; k < j; k++) t -= A[i * (i + 1) / 2 + k] * A[j * (j + 1) / 2 + k];
      A[i * (i + 1) / 2 + j] = t * inv;
    }
  }
}
template <typename T>
__device__ __forceinline__ void chol6_solve(const T (&L)[21], T (&x)[NJ]) {
#pragma unroll
  for (int i = 0; i < NJ; i++) {
    T s = x[i];
#pragma unroll
    for (int k = 0; k < i; k++) s -= L[i * (i + 1) / 2 + k] * x[k];
    x[i] = s / L[i * (i + 1) / 2 + i];
  }
#pragma unroll
  for (int i = NJ - 1; i >= 0; i--) {
    T s = x[i];
#pragma unroll
    for (int k = i + 1; k < NJ; k++) s -= L[k * (k + 1) / 2 + i] * x[k];
    x[i] = s / L[i * (i + 1) / 2 + i];
  }
}
template <typename T>
__device__ __forceinline__ void symmv6(const T (&M)[21], const T (&x)[NJ], T (&y)[NJ]) {
#pragma unroll
  for (int i = 0; i < NJ; i++) {
    T s = T(0);
#pragma unroll
    for (int j = 0; j < NJ; j++) s += (j <= i ? M[i * (i + 1) / 2 + j] : M[j * (j + 1) / 2 + i]) * x[j];
    y[i] = s;
  }
}

// [upstream] mj_implicit, integrator = implicitfast, arm block: the velocity update uses x with (M - h D) x = M qacc, D =
// diag(biasprm[2]) over the unclamped actuators (no joint damping, no other velocity-dependent smooth force in this model).
// Returns x - qacc = (M - h D)^-1 (h D qacc): a small correction (h D / M ~ 2 %), so float32 suffices for it.
template <typename T>
__device__ __forceinline__ void implicitfast_correction(const T (&M)[21], const T (&dvel)[NJ], T h, const T (&qacc)[NJ], T (&corr)[NJ]) {
  T A[21];
#pragma unroll
  for (int i = 0; i < 21; i++) A[i] = M[i];
#pragma unroll
  for (int i = 0; i < NJ; i++) { A[i * (i + 1) / 2 + i] -= h * dvel[i]; corr[i] = h * dvel[i] * qacc[i]; }
  chol6(A);
  chol6_solve(A, corr);
}

// [upstream] getimpedance — power-law sigmoid between solimp[0] and solimp[1] over width solimp[2]
template <typename T>
__device__ __forceinline__ T impedance(const T *solimp, T pos, T margin) {
  const T d0 = t_clamp(solimp[0], T(1e-4), T(0.9999)), dmax = t_clamp(solimp[1], T(1e-4), T(0.9999));
  const T width = solimp[2] > T(1e-15) ? solimp[2] : T(1e-15), mid = t_clamp(solimp[3], T(1e-4), T(0.9999));
  const T power = solimp[4] > T(1) ? solimp[4] : T(1);
  const T x = t_abs(pos - margin) / width;
  if (x >= T(1)) return dmax;
  if (x <= T(0)) return d0;
  T y;
  if (power == T(1)) y = x;
  else if (x <= mid) y = t_pow(T(1) / mid, power - T(1)) * t_pow(x, power);
  else y = T(1) - t_pow(T(1) / (T(1) - mid), power - T(1)) * t_pow(T(1) - x, power);
  return d0 + y * (dmax - d0);
}

}  // namespace so101
