// C-ABI implementation (include/so101_b200.h): handle life cycle, model upload, kernel launches.
// PyTorch owns every tensor that crosses this boundary; the handle owns only its SoA state and scratch.
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "../../include/so101_b200.h"
#include "arm_kernel.cuh"
#include "blob.hpp"
#include "layout_kernels.cuh"
#include "scene_kernel.cuh"

namespace so101 {

static thread_local std::string g_create_error;

#define CUDA_OK(expr)                                                                                      \
  do {                                                                                                     \
    cudaError_t e_ = (expr);                                                                               \
    if (e_ != cudaSuccess) throw std::runtime_error(std::string(#expr) + ": " + cudaGetErrorString(e_)); \
  } while (0)

// Every entry point runs with the handle's device current and restores the caller's device on exit (two handles on
// different GPUs in one process, or a caller that changed torch's current device, must not launch on the wrong device).
struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != dev) cudaSetDevice(dev);
    else prev = -1;
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
  DeviceGuard(const DeviceGuard &) = delete;
  DeviceGuard &operator=(const DeviceGuard &) = delete;
};

struct HandleBase {
  std::string err;
  so101_config cfg{};
  int nq = 0, nv = 0, nu = 0, nbody = 0;
  uint64_t launches = 0, steps = 0, dropped = 0, graph_launches = 0;
  virtual ~HandleBase() { for (auto &t : tiers) t.destroy(); }
  virtual void set_state(const float *q, const float *v, bool initial, cudaStream_t s) = 0;
  virtual void set_state_f64(const double *q, const double *v, bool initial, cudaStream_t s) = 0;
  virtual void set_reset_pool(const float *q, const float *v, int rounds, cudaStream_t s) = 0;
  virtual void get_state(float *q, float *v, cudaStream_t s) = 0;
  virtual void get_state_f64(double *q, double *v, cudaStream_t s) = 0;
  virtual void reset(const uint8_t *mask, const so101_step_out &out, cudaStream_t s) = 0;
  virtual void step(const float *action, const so101_step_out &out, cudaStream_t s) = 0;
  virtual void debug_read(const char *field, float *dst, size_t count, cudaStream_t s) = 0;
  virtual void sample_and_settle(uint64_t seed, const so101_step_out &out, uint64_t stats[4], cudaStream_t s) = 0;
  virtual void placement_stats(uint64_t out[6]) = 0;
  virtual void episode_steps(int32_t *steps_dev, bool set, cudaStream_t s) = 0;
  virtual void step_host(const float *action, const so101_step_out &host_out, cudaStream_t s) = 0;
  virtual uint64_t diverged() = 0;
  virtual size_t checkpoint_bytes() = 0;
  virtual void checkpoint(void *buf_dev, size_t bytes, bool load, cudaStream_t s) = 0;
  KernelTimer timer;
  std::vector<TierExec> tiers;  // one per pipeline group
};

static void quat2mat(const double *q, double *m) {
  double n = std::sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  double w = q[0] / n, x = q[1] / n, y = q[2] / n, z = q[3] / n;
  m[0] = 1 - 2 * (y * y + z * z); m[1] = 2 * (x * y - w * z); m[2] = 2 * (x * z + w * y);
  m[3] = 2 * (x * y + w * z); m[4] = 1 - 2 * (x * x + z * z); m[5] = 2 * (y * z - w * x);
  m[6] = 2 * (x * z - w * y); m[7] = 2 * (y * z + w * x); m[8] = 1 - 2 * (x * x + y * y);
}
static void mm3(const double *a, const double *b, double *r) {
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) r[3 * i + j] = a[3 * i] * b[j] + a[3 * i + 1] * b[3 + j] + a[3 * i + 2] * b[6 + j];
}

// Build the description of arm `arm` from the generic blob: joints 6 * arm .. 6 * arm + 5 must be hinges that form a serial chain
// whose root's parent is static (scene_pbr.xml:74-126), with their dofs / actuators at the same indices.
template <typename T>
static void build_arm(const Blob &b, ArmModelT<T> &am, int arm = 0) {
  const auto &jt = b.I("jnt_type"), &jb = b.I("jnt_body"), &bp = b.I("body_parent"), &bw = b.I("body_weld");
  const int j0 = NJ * arm;
  if ((int)jt.size() < j0 + NJ) throw std::runtime_error("model has fewer hinge joints than this build's arms need");
  const auto &opt = b.F("opt");
  const double dt = opt[0];
  std::memset(&am, 0, sizeof(am));
  // static base pose: compose the chain of static ancestors of the first arm body
  {
    int b0 = jb[j0];
    std::vector<int> chain;
    for (int p = bp[b0]; p != 0; p = bp[p]) {
      if (bw[p] != 0) throw std::runtime_error("arm base must be static");
      chain.push_back(p);
    }
    double R[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, p[3] = {0, 0, 0};
    for (auto it = chain.rbegin(); it != chain.rend(); ++it) {
      const double *bpos = &b.F("body_pos")[3 * *it];
      double Rb[9], Rn[9];
      quat2mat(&b.F("body_quat")[4 * *it], Rb);
      for (int c = 0; c < 3; c++) p[c] += R[3 * c] * bpos[0] + R[3 * c + 1] * bpos[1] + R[3 * c + 2] * bpos[2];
      mm3(R, Rb, Rn);
      std::memcpy(R, Rn, sizeof R);
    }
    for (int c = 0; c < 3; c++) am.base_pos[c] = (T)p[c];
    for (int c = 0; c < 9; c++) am.base_R[c] = (T)R[c];
  }
  for (int j = 0; j < NJ; j++) {
    const int gj = j0 + j;   // joint / dof / qpos index in the model
    if (jt[gj] != 1) throw std::runtime_error("arm joints must be hinges");
    const int body = jb[gj];
    if (j > 0 && bp[body] != jb[gj - 1]) throw std::runtime_error("arm joints must form a serial chain");
    if (b.I("jnt_dofadr")[gj] != gj || b.I("jnt_qposadr")[gj] != gj) throw std::runtime_error("arm dofs must come first, arm by arm");
    const double *jp = &b.F("jnt_pos")[3 * gj];
    if (jp[0] != 0 || jp[1] != 0 || jp[2] != 0) throw std::runtime_error("hinge anchors must sit at the body origin");
    double R0[9], Ri[9];
    quat2mat(&b.F("body_quat")[4 * body], R0);
    quat2mat(&b.F("body_iquat")[4 * body], Ri);
    const double *in = &b.F("body_inertia")[3 * body];
    double Il[9];
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 3; c++) Il[3 * r + c] = Ri[3 * r] * in[0] * Ri[3 * c] + Ri[3 * r + 1] * in[1] * Ri[3 * c + 1] + Ri[3 * r + 2] * in[2] * Ri[3 * c + 2];
    for (int c = 0; c < 3; c++) {
      am.pos[j][c] = (T)b.F("body_pos")[3 * body + c];
      am.axis[j][c] = (T)b.F("jnt_axis")[3 * gj + c];
      am.ipos[j][c] = (T)b.F("body_ipos")[3 * body + c];
    }
    for (int c = 0; c < 9; c++) am.R0[j][c] = (T)R0[c];
    am.Iloc[j][0] = (T)Il[0]; am.Iloc[j][1] = (T)Il[4]; am.Iloc[j][2] = (T)Il[8];
    am.Iloc[j][3] = (T)Il[1]; am.Iloc[j][4] = (T)Il[2]; am.Iloc[j][5] = (T)Il[5];
    am.mass[j] = (T)b.F("body_mass")[body];
    am.qpos0[j] = (T)b.F("qpos0")[gj];
    am.armature[j] = (T)b.F("dof_armature")[gj];
    am.frictionloss[j] = (T)b.F("dof_frictionloss")[gj];
    const double invw = b.F("dof_invweight0")[gj];
    am.invweight0[j] = (T)invw;
    auto clampimp = [](double x) { return x < 1e-4 ? 1e-4 : (x > 0.9999 ? 0.9999 : x); };
    {  // friction-loss row constants: pos = 0 -> impedance = d0; K = 0; B = 2 / (dmax * max(tc, 2 dt))
      const double *sr = &b.F("jnt_solreffriction")[2 * gj], *si = &b.F("jnt_solimpfriction")[5 * gj];
      const double imp = clampimp(si[0]), dmax = clampimp(si[1]);
      double R = (1 - imp) / imp * invw;
      if (R < 1e-15) R = 1e-15;
      am.fr_R[j] = (T)R; am.fr_D[j] = (T)(1 / R);
      am.fr_B[j] = (T)(sr[0] > 0 ? 2 / (dmax * std::max(sr[0], 2 * dt)) : -sr[1] / dmax);
    }
    {
      const double *sr = &b.F("jnt_solreflimit")[2 * gj], *si = &b.F("jnt_solimplimit")[5 * gj];
      const double dmax = clampimp(si[1]);
      for (int c = 0; c < 5; c++) am.lim_solimp[j][c] = (T)si[c];
      if (sr[0] > 0) {
        const double tc = std::max(sr[0], 2 * dt);
        am.lim_K[j] = (T)(1 / (dmax * dmax * tc * tc * sr[1] * sr[1])); am.lim_B[j] = (T)(2 / (dmax * tc));
      } else { am.lim_K[j] = (T)(-sr[0] / (dmax * dmax)); am.lim_B[j] = (T)(-sr[1] / dmax); }
      am.limited[j] = b.I("jnt_limited")[gj];
      am.range[j][0] = (T)b.F("jnt_range")[2 * gj]; am.range[j][1] = (T)b.F("jnt_range")[2 * gj + 1];
    }
  }
  if (b.scalar("nu") != NA) throw std::runtime_error("expected 6 actuators per arm");
  for (int a = 0; a < NJ; a++) {
    const int ga = j0 + a;
    if (b.I("act_jnt")[ga] != ga) throw std::runtime_error("actuator a must drive joint a");
    if (b.F("act_gear")[ga] != 1.0) throw std::runtime_error("actuator gear must be 1");
    am.gain_d[a] = b.F("act_gain")[ga];
    for (int c = 0; c < 3; c++) am.bias_d[a][c] = b.F("act_bias")[3 * ga + c];
    for (int c = 0; c < 2; c++) { am.ctrlrange_d[a][c] = b.F("act_ctrlrange")[2 * ga + c]; am.forcerange_d[a][c] = b.F("act_forcerange")[2 * ga + c]; }
  }
  am.dt_d = dt;
  for (int c = 0; c < 3; c++) am.gravity[c] = (T)opt[1 + c];
  am.dt = (T)dt;
  const int nv = b.scalar("nv");
  am.solver_scale = (T)(1.0 / (opt[8] * std::max(1, nv)));
}

template <typename T>
struct Handle : HandleBase {
  ArmSetT<T> am;
  ArmSetT<double> am64;  // float64 arm models for the float64 parts of the float32 path
  std::unique_ptr<SceneModelHost<T>> scene;  // non-null: full contact scene (warp per env, row-major state)
  EnvState<T> S{};
  PipeBuf<T> pipe{};                 // per-env scratch shared by all groups
  std::vector<PipeBuf<T>> groups;    // per-group queues / counters (views of `pipe` with their own work lists)
  StepCfg sc{};
  std::vector<void *> allocs;
  size_t pool_cap = 1;
  float *d_action = nullptr;   // staging copy of the caller's action: the captured step graph reads it from a fixed address
  so101_step_out d_out{};      // device staging of the whole TimeStep for the host-buffer entry point (so101_step_host)
  // One control step of the contact scene is 166 launches (186 with the two-launch narrow phase of large groups) + event
  // fork/joins on 6 streams.  It is captured once per distinct
  // set of output pointers into a CUDA graph and replayed with a single cudaGraphLaunch (SO101_GRAPH=0 disables; the
  // per-kernel event timers need eager launches and bypass it).
  struct StepGraph { so101_step_out key; cudaGraphExec_t exec; int kernels; };
  std::vector<StepGraph> graphs;
  cudaStream_t cap_stream = nullptr;
  bool use_graph = true;
  unsigned settle_epoch = 0;   // so101_sample_and_settle calls so far (high bits of the envs' Philox draw counters)

  template <typename U>
  U *dalloc(size_t n) {
    void *p = nullptr;
    CUDA_OK(cudaMalloc(&p, n * sizeof(U)));
    CUDA_OK(cudaMemset(p, 0, n * sizeof(U)));
    allocs.push_back(p);
    return static_cast<U *>(p);
  }

  Handle(const Blob &b, const so101_config &c) {
    cfg = c;
    nq = b.scalar("nq"); nv = b.scalar("nv"); nu = b.scalar("nu"); nbody = b.scalar("nbody");
    if (nq == NJ && NARM != 1) throw std::runtime_error("the arm-only model needs the one-arm build of the library (libso101_b200.so)");
    for (int k = 0; k < NARM; k++) { build_arm<T>(b, am.arm[k], k); build_arm<double>(b, am64.arm[k], k); }
    if (nq != NJ || c.collide) {
      if (!c.collide) throw std::runtime_error("models with free props need collide=1");
      scene.reset(new SceneModelHost<T>());
      scene->build(b);
      if (scene_smem_bytes<T>() > 227 * 1024) throw std::runtime_error("scene kernel scratch exceeds the 227 KB shared-memory limit");
    }
    // user envs first, then the nursery envs that keep producing settled placements (contact scene only)
    const int nursery = scene ? std::max(0, c.nursery_envs) : 0;
    const size_t N = (size_t)c.num_envs + nursery;
    S.N = (int)N; S.NU = c.num_envs; S.nq = nq; S.nv = nv;
    S.mode = dalloc<uint8_t>(N); S.sstate = dalloc<uint8_t>(N); S.settle_sub = dalloc<int>(N); S.attempt = dalloc<int>(N); S.draws = dalloc<unsigned>(N);
    S.ring_ctr = dalloc<int>(RC_N);
    S.ring_cap = nursery > 0 ? std::max(1, c.ring_capacity) : 0;
    if (S.ring_cap > 0) { S.ring_q = dalloc<TS>((size_t)S.ring_cap * nq); S.ring_v = dalloc<TS>((size_t)S.ring_cap * nv); }
    if (nursery > 0) CUDA_OK(cudaMemset(S.mode + c.num_envs, 1, nursery));   // (sstate 0 = SETTLE_SAMPLE: they start drawing at the first step)
    for (int p = 0; p < 2; p++) {
      for (int k = 0; k < 3; k++) { S.place.lo[p][k] = c.place_lo[p][k]; S.place.hi[p][k] = c.place_hi[p][k]; }
      S.place.yaw[p][0] = c.place_yaw[p][0]; S.place.yaw[p][1] = c.place_yaw[p][1];
      S.place.check_collisions[p] = c.place_check_collisions[p];
    }
    S.place.max_attempts = c.place_max_attempts > 0 ? c.place_max_attempts : 20;
    S.place.max_settle_substeps = c.settle_max_substeps > 0 ? c.settle_max_substeps : 1000;
    S.place.qvel_tol = c.settle_qvel_tol > 0 ? c.settle_qvel_tol : 1e-3f; S.place.qacc_tol = c.settle_qacc_tol > 0 ? c.settle_qacc_tol : 1e-2f;
    S.place.seed = c.seed;
    S.qpos = dalloc<TS>(nq * N); S.qvel = dalloc<TS>(nv * N); S.warm = dalloc<T>(nv * N);
    S.init_qpos = dalloc<TS>(nq * N); S.init_qvel = dalloc<TS>(nv * N); S.ctrl = dalloc<T>(NA * N);
    S.step = dalloc<int>(N); S.needs_reset = dalloc<uint8_t>(N); S.episode = dalloc<int>(N); S.npool = 1;
    S.ring_joints = dalloc<float>((size_t)(c.joints_delay_steps + 1) * NA * N);
    S.ring_phys = dalloc<float>((size_t)(c.physics_delay_steps + 1) * (nq + nv) * N);
    S.diverged_count = dalloc<int>(2); S.solver_iter = dalloc<int>(N); S.ncon = dalloc<int>(N); S.dropped_env = dalloc<int>(N);
    sc.nsub = c.n_substeps; sc.last_step = c.last_step; sc.dj = c.joints_delay_steps; sc.dp = c.physics_delay_steps;
    sc.integrator = c.integrator == 1 ? 1 : 0;
    sc.terminate_on_success = c.terminate_on_success; sc.max_iter = c.solver_iterations; sc.tol = c.solver_tolerance;
    for (int i = 0; i < 6; i++) { sc.offsets[i] = c.calibration_offsets[i]; sc.home[i] = c.home_ctrl[i]; }
    // default initial state: qpos0, zero velocity
    std::vector<TS> q0(nq * N);
    for (int k = 0; k < nq; k++) for (size_t e = 0; e < N; e++) q0[scene ? e * nq + k : k * N + e] = (TS)b.F("qpos0")[k];
    CUDA_OK(cudaMemcpy(S.init_qpos, q0.data(), q0.size() * sizeof(TS), cudaMemcpyHostToDevice));
    d_action = dalloc<float>(NA * N);
    use_graph = !(getenv("SO101_GRAPH") && atoi(getenv("SO101_GRAPH")) == 0);
    if (scene) {  // inter-kernel scratch of the scene pipeline
      if (b.scalar("ngeom") > GMAX_GEOMS) throw std::runtime_error("model has more geoms than the broad phase can hold");
      if (b.scalar("nbody") > BMAX_BODIES) throw std::runtime_error("model has more bodies than the broad phase can hold");
      if (b.scalar("ngeom") > WQ) throw std::runtime_error("model has more geoms than narrow-phase work queues");
      pipe.xpos = dalloc<T>(N * NSLOT * 3); pipe.xmat = dalloc<T>(N * NSLOT * 9); pipe.dyn = dalloc<T>(N * DYNW);
      pipe.con = dalloc<T>(N * CONBUF * 8); pipe.con_key = dalloc<int>(N * CONBUF); pipe.ncon_raw = dalloc<int>(N);
      pipe.active = dalloc<uint8_t>(N); pipe.flags = dalloc<uint8_t>(N); pipe.tier = dalloc<uint8_t>(N);
      // pipeline groups: independent env ranges whose kernel sequences run on their own streams, so that one group's short
      // kernels (kinematics, broad phase, classify) and kernel tails overlap the other's long ones.  Measured on B200 at 16384
      // envs (bench.py, random actions): 1 group 41.7 ms/step, 2 groups 40.7, 3: ~same, 4: 15 % slower (every kernel is bound
      // by the latency of its slowest warps, which shorter launches do not shorten).  With the round-1 kernels 2 groups were
      // slower (profiles/r01_groups.txt).  SO101_GROUPS overrides.
      int ng = getenv("SO101_GROUPS") ? atoi(getenv("SO101_GROUPS")) : 2;
      const int by_size = (int)((N + 2047) / 2048);
      ng = std::max(1, std::min(std::min(ng, 8), by_size));
      tiers.resize(ng);
      for (int g = 0; g < ng; g++) {
        PipeBuf<T> p = pipe;
        p.env0 = (int)(N * g / ng); p.nenv = (int)(N * (g + 1) / ng) - p.env0;   // (groups partition ALL envs, nursery included)
        // A queue holds the candidate pairs of ALL envs that share its key geom.  The static table is the partner of every arm
        // geom that comes down on it (17 of them), so the per-queue capacity must cover many pairs per env (only the used
        // entries are ever touched): 4 per env overflowed in long random-action rollouts and silently lost arm-table contacts.
        p.work_cap = 16 * p.nenv + 64; p.work = dalloc<uint2>((size_t)WQ * p.work_cap);
        p.nwork = dalloc<int>(WSTRIDE * (c.n_substeps + 1)); p.big = dalloc<int>(2 * (size_t)p.nenv);
        // a hit's slot is its queue's item offset + the queue's hit count: any offset below the group's total item count can
        // occur, and an env contributes at most PAIRCAP items
        p.hit_cap = p.nenv * PAIRCAP; p.hits = dalloc<HitRec<T>>((size_t)p.hit_cap);
        groups.push_back(p);
        tiers[g].init();
      }
    }
  }
  // captured graphs hold EnvState / StepCfg BY VALUE in their kernel parameters: anything that changes them (reset pool size or
  // storage, debug probes) must drop the graphs
  void invalidate_graphs() {
    for (auto &g : graphs) cudaGraphExecDestroy(g.exec);
    graphs.clear();
  }
  ~Handle() override {
    for (auto &g : graphs) cudaGraphExecDestroy(g.exec);
    if (cap_stream) cudaStreamDestroy(cap_stream);
    for (void *p : allocs) cudaFree(p);
  }
  template <typename A>
  void set_state_any(const A *q, const A *v, bool initial, cudaStream_t s) {
    auto put = [&](const A *rows, TS *dst, int k) {
      if (scene) launch_cast_copy<A, TS>(rows, dst, (size_t)S.NU * k, s); else launch_rows_to_soa<A, TS>(rows, dst, S.N, k, s);
      launches += 1;
    };
    put(q, S.qpos, nq); put(v, S.qvel, nv);
    if (initial) {  // the caller's own initial states replace the device-side placements
      if (S.npool != 1 || S.use_ring) invalidate_graphs();
      S.npool = 1; S.use_ring = 0;
      put(q, S.init_qpos, nq); put(v, S.init_qvel, nv);
    }
    CUDA_OK(cudaMemsetAsync(S.warm, 0, sizeof(T) * nv * S.N, s));
  }
  void set_state(const float *q, const float *v, bool initial, cudaStream_t s) override { set_state_any(q, v, initial, s); }
  void set_state_f64(const double *q, const double *v, bool initial, cudaStream_t s) override { set_state_any(q, v, initial, s); }
  // Reset pool: `rounds` initial states per env ([rounds][N][nq] / [rounds][N][nv] rows); episode e of an env starts from
  // entry e % rounds.  The pool storage grows on demand and replaces the single initial state.
  void set_reset_pool(const float *q, const float *v, int rounds, cudaStream_t s) override {
    if (rounds < 1) throw std::runtime_error("reset pool needs at least one round");
    invalidate_graphs();
    S.use_ring = 0;
    const size_t N = S.N, NU = S.NU;   // pool rows are strided by all envs of the handle; the caller supplies the user envs
    if ((size_t)rounds > pool_cap) {
      CUDA_OK(cudaStreamSynchronize(s));
      S.init_qpos = dalloc<TS>((size_t)rounds * nq * N); S.init_qvel = dalloc<TS>((size_t)rounds * nv * N);  // (old pool is freed with the handle)
      pool_cap = rounds;
    }
    for (int r = 0; r < rounds; r++) {
      const float *qr = q + (size_t)r * NU * nq, *vr = v + (size_t)r * NU * nv;
      TS *dq = S.init_qpos + (size_t)r * N * nq, *dv = S.init_qvel + (size_t)r * N * nv;
      if (scene) { launch_cast_copy<float, TS>(qr, dq, NU * nq, s); launch_cast_copy<float, TS>(vr, dv, NU * nv, s); }
      else { launch_rows_to_soa<float, TS>(qr, dq, S.N, nq, s); launch_rows_to_soa<float, TS>(vr, dv, S.N, nv, s); }
      launches += 2;
    }
    S.npool = rounds;
    CUDA_OK(cudaMemsetAsync(S.episode, 0, sizeof(int) * N, s));
  }
  void get_state(float *q, float *v, cudaStream_t s) override {
    if (scene) { launch_cast_copy<TS, float>(S.qpos, q, (size_t)S.NU * nq, s); launch_cast_copy<TS, float>(S.qvel, v, (size_t)S.NU * nv, s); }
    else { launch_soa_to_rows<TS, float>(S.qpos, q, S.N, nq, s); launch_soa_to_rows<TS, float>(S.qvel, v, S.N, nv, s); }
    launches += 2;
  }
  void get_state_f64(double *q, double *v, cudaStream_t s) override {
    if (scene) { launch_cast_copy<TS, double>(S.qpos, q, (size_t)S.NU * nq, s); launch_cast_copy<TS, double>(S.qvel, v, (size_t)S.NU * nv, s); }
    else { launch_soa_to_rows<TS, double>(S.qpos, q, S.N, nq, s); launch_soa_to_rows<TS, double>(S.qvel, v, S.N, nv, s); }
    launches += 2;
  }
  void reset(const uint8_t *mask, const so101_step_out &out, cudaStream_t s) override {
    if (scene) launch_scene_reset<T>(sc, S, mask, out, s); else launch_arm_reset<T>(sc, S, mask, out, s);
    launches += 1;
  }
  void step(const float *action, const so101_step_out &out, cudaStream_t s) override {
    if (!scene) { timer.begin(4, s); launch_arm_step<T>(am.arm[0], am64.arm[0], sc, S, action, out, s); timer.end(4, s); launches += 1; steps += 1; return; }
    if (!use_graph || timer.on) {
      launches += launch_scene_step<T>(am, am64, scene->dev, sc, S, groups.data(), tiers.data(), (int)groups.size(), action, out, s, &timer);
      steps += 1;
      return;
    }
    // graph replay: the action goes through a fixed staging buffer so that the graph does not depend on the caller's pointer
    if (action != d_action) CUDA_OK(cudaMemcpyAsync(d_action, action, sizeof(float) * NA * S.NU, cudaMemcpyDeviceToDevice, s));
    cudaGraphExec_t exec = nullptr;
    int nk = 0;
    for (auto &g : graphs) if (std::memcmp(&g.key, &out, sizeof out) == 0) { exec = g.exec; nk = g.kernels; }
    if (!exec) {
      if (graphs.size() >= 8) { cudaGraphExecDestroy(graphs.front().exec); graphs.erase(graphs.begin()); }
      if (!cap_stream) CUDA_OK(cudaStreamCreateWithFlags(&cap_stream, cudaStreamNonBlocking));
      cudaGraph_t graph = nullptr;
      CUDA_OK(cudaStreamBeginCapture(cap_stream, cudaStreamCaptureModeThreadLocal));
      nk = launch_scene_step<T>(am, am64, scene->dev, sc, S, groups.data(), tiers.data(), (int)groups.size(), d_action, out, cap_stream, nullptr);
      const cudaError_t le = cudaGetLastError();   // first launch error inside the capture, if any
      cudaError_t e = cudaStreamEndCapture(cap_stream, &graph);
      if (e != cudaSuccess || !graph) {
        cudaGetLastError();
        throw std::runtime_error(std::string("step graph capture failed: ") + cudaGetErrorString(e) + " (first launch error: " + cudaGetErrorString(le) + ")");
      }
      e = cudaGraphInstantiate(&exec, graph, 0);
      cudaGraphDestroy(graph);
      if (e != cudaSuccess) throw std::runtime_error(std::string("cudaGraphInstantiate: ") + cudaGetErrorString(e));
      graphs.push_back({out, exec, nk});
    }
    CUDA_OK(cudaGraphLaunch(exec, s));
    launches += nk; graph_launches += 1; steps += 1;
  }
  void debug_read(const char *field, float *dst, size_t count, cudaStream_t s) override {
    const std::string f(field);
    if (f == "solver_iter" || f == "ncon" || f == "step" || f == "dropped") {
      const int *src = f == "solver_iter" ? S.solver_iter : (f == "ncon" ? S.ncon : (f == "dropped" ? S.dropped_env : S.step));
      if (count < (size_t)S.NU) throw std::runtime_error("debug_read: buffer too small");
      launch_int_to_float(src, dst, S.NU, s);
      launches += 1;
    } else if (f == "warm") {
      if (count < (size_t)S.NU * nv) throw std::runtime_error("debug_read: buffer too small");
      if (scene) launch_cast_copy<T, float>(S.warm, dst, (size_t)S.NU * nv, s); else launch_soa_to_rows<T, float>(S.warm, dst, S.N, nv, s);
      launches += 1;
    } else if (f == "tier") {
      // solver tier (0, 1, 2) each env was solved in during the last substep (scene_classify_kernel)
      if (!scene) throw std::runtime_error("debug_read: tier needs a contact scene");
      if (count < (size_t)S.NU) throw std::runtime_error("debug_read: buffer too small");
      launch_cast_copy<uint8_t, float>(pipe.tier, dst, S.NU, s);
      launches += 1;
    } else if (f == "contacts_width") {
      // contacts per env the "contacts" probe holds (its rows are 1 + 9 * width floats)
      if (count < 1) throw std::runtime_error("debug_read: buffer too small");
      const float w = (float)NCON;
      CUDA_OK(cudaMemcpyAsync(dst, &w, sizeof w, cudaMemcpyHostToDevice, s));
      CUDA_OK(cudaStreamSynchronize(s));
    } else if (f == "dropcat") {
      // 8 drop counters by buffer (see scene_solve.cuh: g_dropcat), since the library was loaded
      if (count < 8) throw std::runtime_error("debug_read: buffer too small");
      int h[8]; float hf[8];
      CUDA_OK(cudaStreamSynchronize(s));
      scene_dropcat<T>(h);
      for (int i = 0; i < 8; i++) hf[i] = (float)h[i];
      CUDA_OK(cudaMemcpy(dst, hf, sizeof hf, cudaMemcpyHostToDevice));
    } else if (f == "contacts") {
      // [N][1 + 9*NCON]: ncon (may exceed NCON), then (geom1, geom2, dist, pos3, normal3) per contact of the last substep.  The first call only
      // enables the probe (the buffer is filled by subsequent steps).
      const size_t need = (size_t)S.NU * (1 + 9 * NCON);
      if (count < need) throw std::runtime_error("debug_read: buffer too small");
      if (!S.dbg_contacts) { S.dbg_contacts = dalloc<float>((size_t)S.N * (1 + 9 * NCON)); invalidate_graphs(); }
      CUDA_OK(cudaMemcpyAsync(dst, S.dbg_contacts, need * sizeof(float), cudaMemcpyDeviceToDevice, s));
    } else throw std::runtime_error("debug_read: unknown field " + f);
  }
  // e2e path: host buffers in, the WHOLE TimeStep (every block of so101_step_out that is non-null in host_out) out to host
  // buffers; host<->device copies on the caller's stream, one sync at the end
  void step_host(const float *action, const so101_step_out &host_out, cudaStream_t s) override {
    const size_t N = S.NU, sd = (size_t)nq + nv;
    if (!d_out.reward) {
      d_out.commanded_joints_pos = dalloc<float>(NA * N); d_out.joints_pos = dalloc<float>(NA * N); d_out.undelayed_joints_pos = dalloc<float>(NA * N);
      d_out.physics_state = dalloc<float>(sd * N); d_out.delayed_physics_state = dalloc<float>(sd * N);
      d_out.reward = dalloc<float>(N); d_out.discount = dalloc<float>(N); d_out.step_type = dalloc<uint8_t>(N);
    }
    CUDA_OK(cudaMemcpyAsync(d_action, action, NA * N * sizeof(float), cudaMemcpyHostToDevice, s));
    step(d_action, d_out, s);
    auto back = [&](void *dst, const void *src, size_t bytes) { if (dst) CUDA_OK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, s)); };
    back(host_out.commanded_joints_pos, d_out.commanded_joints_pos, NA * N * sizeof(float));
    back(host_out.joints_pos, d_out.joints_pos, NA * N * sizeof(float));
    back(host_out.undelayed_joints_pos, d_out.undelayed_joints_pos, NA * N * sizeof(float));
    back(host_out.physics_state, d_out.physics_state, sd * N * sizeof(float));
    back(host_out.delayed_physics_state, d_out.delayed_physics_state, sd * N * sizeof(float));
    back(host_out.reward, d_out.reward, N * sizeof(float));
    back(host_out.discount, d_out.discount, N * sizeof(float));
    back(host_out.step_type, d_out.step_type, N);
    CUDA_OK(cudaStreamSynchronize(s));
  }
  // All user envs draw a placement and settle it with the arm frozen; the loop over control steps runs here (one graph launch
  // per step), polling the number of envs still settling every few steps.
  void sample_and_settle(uint64_t seed, const so101_step_out &out, uint64_t stats[4], cudaStream_t s) override {
    if (!scene) throw std::runtime_error("sample_and_settle needs a model with free props");
    int before[RC_N], after[RC_N];
    CUDA_OK(cudaStreamSynchronize(s));
    CUDA_OK(cudaMemcpy(before, S.ring_ctr, sizeof before, cudaMemcpyDeviceToHost));
    if (seed != S.place.seed) { S.place.seed = seed; invalidate_graphs(); }
    if (S.npool != 1) { S.npool = 1; invalidate_graphs(); }
    if (S.use_ring != (S.ring_cap > 0)) { S.use_ring = S.ring_cap > 0; invalidate_graphs(); }
    settle_epoch += 1;
    launch_settle_enter<T>(S, settle_epoch << 20, s);
    launches += 1;
    so101_step_out none{};
    const int max_steps = (S.place.max_settle_substeps + sc.nsub - 1) / sc.nsub + S.place.max_attempts + 2;
    int steps_run = 0, pending = 1;
    while (pending > 0 && steps_run < max_steps) {
      for (int k = 0; k < 4 && steps_run < max_steps; k++, steps_run++) {
        CUDA_OK(cudaMemsetAsync(S.ring_ctr + RC_PENDING, 0, sizeof(int), s));
        step(d_action, none, s);   // (settle-mode envs ignore the action)
        steps -= 1;
      }
      CUDA_OK(cudaMemcpyAsync(&pending, S.ring_ctr + RC_PENDING, sizeof(int), cudaMemcpyDeviceToHost, s));
      CUDA_OK(cudaStreamSynchronize(s));
    }
    launch_settle_leave<T>(S, s);
    launches += 1;
    reset(nullptr, out, s);
    CUDA_OK(cudaStreamSynchronize(s));
    CUDA_OK(cudaMemcpy(after, S.ring_ctr, sizeof after, cudaMemcpyDeviceToHost));
    if (stats) {
      stats[0] = (uint64_t)steps_run; stats[1] = (uint64_t)(after[RC_UNSETTLED] - before[RC_UNSETTLED]);
      stats[2] = (uint64_t)(after[RC_REJECTED] - before[RC_REJECTED]); stats[3] = (uint64_t)(after[RC_EXHAUSTED] - before[RC_EXHAUSTED]);
    }
  }
  void placement_stats(uint64_t out[6]) override {
    int c[RC_N] = {};
    CUDA_OK(cudaMemcpy(c, S.ring_ctr, sizeof c, cudaMemcpyDeviceToHost));
    out[0] = c[RC_CLAIM]; out[1] = c[RC_TAIL]; out[2] = c[RC_REUSED]; out[3] = c[RC_UNSETTLED]; out[4] = c[RC_EXHAUSTED]; out[5] = c[RC_REJECTED];
  }
  void episode_steps(int32_t *steps_dev, bool set, cudaStream_t s) override {
    static_assert(sizeof(int32_t) == sizeof(int), "step counters are 32-bit");
    if (set) CUDA_OK(cudaMemcpyAsync(S.step, steps_dev, sizeof(int) * S.NU, cudaMemcpyDeviceToDevice, s));
    else CUDA_OK(cudaMemcpyAsync(steps_dev, S.step, sizeof(int) * S.NU, cudaMemcpyDeviceToDevice, s));
  }
  // ---- checkpoint: everything a handle needs to continue a rollout bit for bit (device buffer: header, then the segments)
  struct CkptHeader {
    uint32_t magic, abi, sizeof_real, narm;
    int32_t N, NU, nq, nv, npool, ring_cap, use_ring, dj, dp, nseg;
    uint32_t settle_epoch, pad;
    uint64_t steps, bytes;
  };
  struct Seg { void *p; size_t bytes; };
  std::vector<Seg> segments() const {
    const size_t N = S.N;
    std::vector<Seg> v = {
      {S.qpos, sizeof(TS) * nq * N}, {S.qvel, sizeof(TS) * nv * N}, {S.warm, sizeof(T) * nv * N}, {S.ctrl, sizeof(T) * NA * N},
      {S.init_qpos, sizeof(TS) * (size_t)S.npool * nq * N}, {S.init_qvel, sizeof(TS) * (size_t)S.npool * nv * N},
      {S.step, sizeof(int) * N}, {S.needs_reset, N}, {S.episode, sizeof(int) * N},
      {S.ring_joints, sizeof(float) * (size_t)(sc.dj + 1) * NA * N}, {S.ring_phys, sizeof(float) * (size_t)(sc.dp + 1) * (nq + nv) * N},
      {S.mode, N}, {S.sstate, N}, {S.settle_sub, sizeof(int) * N}, {S.attempt, sizeof(int) * N}, {S.draws, sizeof(unsigned) * N},
      {S.ring_ctr, sizeof(int) * RC_N}, {S.diverged_count, sizeof(int) * 2}, {S.solver_iter, sizeof(int) * N}, {S.ncon, sizeof(int) * N},
      {S.dropped_env, sizeof(int) * N}};
    if (S.ring_cap > 0) { v.push_back({S.ring_q, sizeof(TS) * (size_t)S.ring_cap * nq}); v.push_back({S.ring_v, sizeof(TS) * (size_t)S.ring_cap * nv}); }
    return v;
  }
  static size_t pad16(size_t b) { return (b + 15) / 16 * 16; }
  size_t checkpoint_bytes() override {
    size_t b = pad16(sizeof(CkptHeader));
    for (const Seg &g : segments()) b += pad16(g.bytes);
    return b;
  }
  void checkpoint(void *buf_dev, size_t bytes, bool load, cudaStream_t s) override {
    unsigned char *buf = static_cast<unsigned char *>(buf_dev);
    CkptHeader hd{};
    if (!load) {
      const size_t need = checkpoint_bytes();
      if (bytes < need) throw std::runtime_error("checkpoint buffer too small (ask so101_checkpoint_size)");
      const auto segs = segments();
      hd = CkptHeader{0x43314f53u /* 'SO1C' */, SO101_ABI_VERSION, (uint32_t)sizeof(T), (uint32_t)NARM, S.N, S.NU, nq, nv, S.npool, S.ring_cap,
                      S.use_ring, sc.dj, sc.dp, (int32_t)segs.size(), settle_epoch, 0u, steps, need};
      CUDA_OK(cudaMemcpyAsync(buf, &hd, sizeof hd, cudaMemcpyHostToDevice, s));
      size_t off = pad16(sizeof hd);
      for (const Seg &g : segs) { CUDA_OK(cudaMemcpyAsync(buf + off, g.p, g.bytes, cudaMemcpyDeviceToDevice, s)); off += pad16(g.bytes); }
      CUDA_OK(cudaStreamSynchronize(s));   // (the header was copied from this stack frame)
      return;
    }
    if (bytes < sizeof hd) throw std::runtime_error("not a checkpoint: buffer shorter than the header");
    CUDA_OK(cudaStreamSynchronize(s));
    CUDA_OK(cudaMemcpy(&hd, buf, sizeof hd, cudaMemcpyDeviceToHost));
    if (hd.magic != 0x43314f53u || hd.abi != SO101_ABI_VERSION) throw std::runtime_error("not a checkpoint of this library version");
    if (hd.sizeof_real != sizeof(T) || hd.narm != (uint32_t)NARM || hd.N != S.N || hd.NU != S.NU || hd.nq != nq || hd.nv != nv || hd.ring_cap != S.ring_cap ||
        hd.dj != sc.dj || hd.dp != sc.dp)
      throw std::runtime_error("checkpoint was taken from a handle with a different model, precision, env count, nursery or observation delays");
    if (hd.npool < 1 || (size_t)hd.npool > pool_cap) throw std::runtime_error("checkpoint holds a larger reset pool than this handle has allocated (install a pool of that many rounds first)");
    if (hd.bytes > bytes) throw std::runtime_error("checkpoint buffer is truncated");
    if (hd.npool != S.npool || hd.use_ring != S.use_ring) { invalidate_graphs(); S.npool = hd.npool; S.use_ring = hd.use_ring; }
    const auto segs = segments();
    if ((int32_t)segs.size() != hd.nseg) throw std::runtime_error("checkpoint layout mismatch");
    size_t off = pad16(sizeof hd);
    for (const Seg &g : segs) { CUDA_OK(cudaMemcpyAsync(g.p, buf + off, g.bytes, cudaMemcpyDeviceToDevice, s)); off += pad16(g.bytes); }
    settle_epoch = hd.settle_epoch; steps = hd.steps;
  }
  uint64_t diverged() override {
    int v[2] = {0, 0};
    cudaMemcpy(v, S.diverged_count, 2 * sizeof(int), cudaMemcpyDeviceToHost);
    dropped = (uint64_t)v[1];
    return (uint64_t)v[0];
  }
};

}  // namespace so101

using namespace so101;

// NVTX range around an entry point (header-only NVTX 3: a no-op unless a profiler injects its library; `ncu --nvtx
// --nvtx-include "so101_step/"` restricts a capture to the kernels of the steps)
struct NvtxRange {
  explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};
#define API_BEGIN(h)                                   \
  if (!(h)) return -1;                                 \
  HandleBase *H = reinterpret_cast<HandleBase *>(h);   \
  DeviceGuard guard_(H->cfg.device);                   \
  try {
#define API_END()                                                                        \
    cudaError_t e_ = cudaPeekAtLastError();                                              \
    if (e_ != cudaSuccess) { H->err = cudaGetErrorString(e_); cudaGetLastError(); return -3; } \
    return 0;                                                                            \
  } catch (const std::exception &ex) { H->err = ex.what(); return -2; }

extern "C" {

int so101_abi_version(void) { return SO101_ABI_VERSION; }

int so101_create(const void *model_blob, size_t blob_len, const so101_config *cfg, so101_handle *out) {
  if (!model_blob || !cfg || !out) { g_create_error = "null argument"; return -1; }
  try {
    if (cfg->num_envs <= 0) throw std::runtime_error("num_envs must be positive");
    if (cfg->n_substeps <= 0) throw std::runtime_error("n_substeps must be positive");
    if (cfg->joints_delay_steps < 0 || cfg->physics_delay_steps < 0) throw std::runtime_error("delays must be >= 0");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) throw std::runtime_error("no CUDA device: this library has no CPU fallback");
    if (cfg->device < 0 || cfg->device >= ndev) throw std::runtime_error("invalid device ordinal");
    Blob b(model_blob, blob_len);
    DeviceGuard guard(cfg->device);
    HandleBase *H = nullptr;
    if (cfg->integrator != 0 && cfg->integrator != 1) throw std::runtime_error("integrator must be 0 (Euler) or 1 (implicitfast)");
    if (cfg->precision == 64) H = new Handle<double>(b, *cfg);
    else if (cfg->precision == 32) H = new Handle<float>(b, *cfg);
    else throw std::runtime_error("precision must be 32 or 64");
    *out = reinterpret_cast<so101_handle>(H);
    return 0;
  } catch (const std::exception &ex) {
    g_create_error = ex.what();
    cudaGetLastError();
    return -2;
  }
}

int so101_destroy(so101_handle h) {
  if (!h) return -1;
  HandleBase *H = reinterpret_cast<HandleBase *>(h);
  DeviceGuard guard(H->cfg.device);
  delete H;
  return 0;
}

const char *so101_last_error(so101_handle h) {
  if (!h) return g_create_error.c_str();
  return reinterpret_cast<HandleBase *>(h)->err.c_str();
}

int so101_dims(so101_handle h, int *nq, int *nv, int *nu, int *nbody) {
  API_BEGIN(h)
  if (nq) *nq = H->nq;
  if (nv) *nv = H->nv;
  if (nu) *nu = H->nu;
  if (nbody) *nbody = H->nbody;
  API_END()
}

int so101_set_initial_state(so101_handle h, const float *qpos_dev, const float *qvel_dev, void *stream) {
  API_BEGIN(h)
  if (!qpos_dev || !qvel_dev) throw std::runtime_error("null state pointer");
  H->set_state(qpos_dev, qvel_dev, true, (cudaStream_t)stream);
  API_END()
}
int so101_set_reset_pool(so101_handle h, const float *qpos_dev, const float *qvel_dev, int rounds, void *stream) {
  API_BEGIN(h)
  if (!qpos_dev || !qvel_dev) throw std::runtime_error("null state pointer");
  H->set_reset_pool(qpos_dev, qvel_dev, rounds, (cudaStream_t)stream);
  API_END()
}
int so101_set_state(so101_handle h, const float *qpos_dev, const float *qvel_dev, void *stream) {
  API_BEGIN(h)
  if (!qpos_dev || !qvel_dev) throw std::runtime_error("null state pointer");
  H->set_state(qpos_dev, qvel_dev, false, (cudaStream_t)stream);
  API_END()
}
int so101_set_state_f64(so101_handle h, const double *qpos_dev, const double *qvel_dev, int initial, void *stream) {
  API_BEGIN(h)
  if (!qpos_dev || !qvel_dev) throw std::runtime_error("null state pointer");
  H->set_state_f64(qpos_dev, qvel_dev, initial != 0, (cudaStream_t)stream);
  API_END()
}
int so101_sample_and_settle(so101_handle h, uint64_t seed, const so101_step_out *out, uint64_t stats_out[4], void *stream) {
  API_BEGIN(h)
  NvtxRange range_("so101_sample_and_settle");
  so101_step_out o{};
  if (out) o = *out;
  H->sample_and_settle(seed, o, stats_out, (cudaStream_t)stream);
  API_END()
}
int so101_get_episode_steps(so101_handle h, int32_t *steps_dev, void *stream) {
  API_BEGIN(h)
  if (!steps_dev) throw std::runtime_error("null pointer");
  H->episode_steps(steps_dev, false, (cudaStream_t)stream);
  API_END()
}
int so101_set_episode_steps(so101_handle h, const int32_t *steps_dev, void *stream) {
  API_BEGIN(h)
  if (!steps_dev) throw std::runtime_error("null pointer");
  H->episode_steps(const_cast<int32_t *>(steps_dev), true, (cudaStream_t)stream);
  API_END()
}
int so101_checkpoint_size(so101_handle h, size_t *bytes) {
  API_BEGIN(h)
  if (!bytes) throw std::runtime_error("null pointer");
  *bytes = H->checkpoint_bytes();
  API_END()
}
int so101_checkpoint_save(so101_handle h, void *buf_dev, size_t bytes, void *stream) {
  API_BEGIN(h)
  NvtxRange range_("so101_checkpoint_save");
  if (!buf_dev) throw std::runtime_error("null pointer");
  H->checkpoint(buf_dev, bytes, false, (cudaStream_t)stream);
  API_END()
}
int so101_checkpoint_load(so101_handle h, const void *buf_dev, size_t bytes, void *stream) {
  API_BEGIN(h)
  NvtxRange range_("so101_checkpoint_load");
  if (!buf_dev) throw std::runtime_error("null pointer");
  H->checkpoint(const_cast<void *>(buf_dev), bytes, true, (cudaStream_t)stream);
  API_END()
}
int so101_placement_stats(so101_handle h, uint64_t out[6]) {
  API_BEGIN(h)
  if (!out) throw std::runtime_error("null output");
  H->placement_stats(out);
  API_END()
}
int so101_get_state(so101_handle h, float *qpos_dev, float *qvel_dev, void *stream) {
  API_BEGIN(h)
  if (!qpos_dev || !qvel_dev) throw std::runtime_error("null state pointer");
  H->get_state(qpos_dev, qvel_dev, (cudaStream_t)stream);
  API_END()
}
int so101_get_state_f64(so101_handle h, double *qpos_dev, double *qvel_dev, void *stream) {
  API_BEGIN(h)
  if (!qpos_dev || !qvel_dev) throw std::runtime_error("null state pointer");
  H->get_state_f64(qpos_dev, qvel_dev, (cudaStream_t)stream);
  API_END()
}
int so101_reset(so101_handle h, const uint8_t *mask_dev, const so101_step_out *out, void *stream) {
  API_BEGIN(h)
  NvtxRange range_("so101_reset");
  so101_step_out o{};
  if (out) o = *out;
  H->reset(mask_dev, o, (cudaStream_t)stream);
  API_END()
}
int so101_step(so101_handle h, const float *action_dev, const so101_step_out *out, void *stream) {
  API_BEGIN(h)
  NvtxRange range_("so101_step");
  if (!action_dev) throw std::runtime_error("null action pointer");
  so101_step_out o{};
  if (out) o = *out;
  H->step(action_dev, o, (cudaStream_t)stream);
  API_END()
}
int so101_step_host(so101_handle h, const float *action_host, const so101_step_out *out_host, void *stream) {
  API_BEGIN(h)
  NvtxRange range_("so101_step_host");
  if (!action_host) throw std::runtime_error("null action pointer");
  so101_step_out o{};
  if (out_host) o = *out_host;
  H->step_host(action_host, o, (cudaStream_t)stream);
  API_END()
}
int so101_counters(so101_handle h, uint64_t out[6]) {
  API_BEGIN(h)
  out[2] = H->diverged(); out[0] = H->launches; out[1] = H->steps; out[3] = H->dropped; out[4] = H->graph_launches; out[5] = 0;
  API_END()
}
int so101_kernel_times(so101_handle h, int enable, double ms_out[11], uint64_t launches_out[11]) {
  API_BEGIN(h)
  H->timer.collect();
  for (int i = 0; i < KernelTimer::NK; i++) {
    if (ms_out) ms_out[i] = H->timer.ms[i];
    if (launches_out) launches_out[i] = H->timer.count[i];
  }
  H->timer.on = enable != 0;
  API_END()
}
int so101_debug_overlap(int precision, int device, const double *cases_dev, int n, uint8_t *out_dev, void *stream) {
  if (!cases_dev || !out_dev || n < 0 || (precision != 32 && precision != 64)) return -1;
  DeviceGuard guard(device);
  if (precision == 32) launch_debug_overlap<float>(cases_dev, n, out_dev, (cudaStream_t)stream);
  else launch_debug_overlap<double>(cases_dev, n, out_dev, (cudaStream_t)stream);
  return cudaPeekAtLastError() == cudaSuccess ? 0 : -3;
}
int so101_debug_read(so101_handle h, const char *field, float *dst_dev, size_t count, void *stream) {
  API_BEGIN(h)
  H->debug_read(field, dst_dev, count, (cudaStream_t)stream);
  API_END()
}

}  // extern "C"
