#pragma once
#include <cuda_runtime.h>

#include <array>
#include <vector>
#include "arm_dynamics.cuh"
#include "arm_solver.cuh"
#include "env_state.cuh"
#include "scene_collide.cuh"
#include "scene_model.cuh"

namespace so101 {
// Scene-kernel state layout is array-of-rows ([N][nq] etc.): one warp owns one env and reads its row with one
// coalesced request (the arm-only kernel, one THREAD per env, uses [k][N] instead).

// Per-env record written by the thread-per-env kinematics + smooth-dynamics kernel and read by the solve kernels:
// joint anchors 18, joint axes 18, arm mass matrix 21, prop mass blocks 2 x 21, qacc_smooth 18, arm rows 24
// (one arm: 0, 18, 36, 57, 99, 117, 141 -> 144 values; two arms: 232)
constexpr int DYN_P = 0, DYN_A = 3 * NA, DYN_MARM = 6 * NA, DYN_MPROP = DYN_MARM + 21 * NARM, DYN_QACC = DYN_MPROP + 21 * NPROP,
              DYN_ROWS = DYN_QACC + NV, DYN_VELMASK = DYN_ROWS + 4 * NA /* per arm: actuators whose force is not clamped (bit mask,
              implicitfast) */, DYNW = (DYN_VELMASK + NARM + 3) / 4 * 4;
constexpr int GMAX_GEOMS = NARM == 1 ? 96 : 128;  // geoms per model the broad phase holds in shared memory
constexpr int BMAX_BODIES = NARM == 1 ? 16 : 24;  // bodies per model the broad phase holds in shared memory
constexpr int WQ = 128;             // work queues (>= ngeom)
constexpr int WSTRIDE = 2 * WQ + 8; // counters per substep
enum { W_CURSOR = WQ, W_NTIER = WQ + 1 /* [2]: envs queued for solver tier 1, 2 */, W_TIERCURSOR = WQ + 3 /* [2] */,
       W_NHIT = WQ + 5 /* intersecting pairs found by the GJK kernel */, W_HITCURSOR = WQ + 6,
       W_QHIT = WQ + 8 /* [WQ]: intersecting pairs per work queue */ };

// An intersecting pair handed from the boolean-GJK kernel (thread per pair) to the EPA / manifold kernel (warp per pair).
template <typename T>
struct HitRec {
  unsigned env, packed;  // packed = g1 | g2 << 8 | pair index << 16
  int n, hintA, hintB, pad;  // simplex size (0: plane pair, no simplex); hill-climbing warm starts of the two shapes after GJK
  T S[4][9];             // GJK simplex: w, a, b of each vertex (MPoint layout)
};

// Device scratch that crosses the kernels of one substep (written by one kernel, read by the next; L2-resident).
template <typename T>
struct PipeBuf {
  T *xpos, *xmat;           // [N][NSLOT*3], [N][NSLOT*9]  world poses of the 8 dynamic bodies
  T *dyn;                   // [N][DYNW]  joint anchors / axes, mass matrices, qacc_smooth and the arm's friction / limit rows at the
                            //   current state (scene_kindyn_kernel -> solve kernels)
  uint2 *work;              // [WQ][work_cap]  narrow-phase work queues, one per second geom g2 (so that consecutive items
                            //   collide the same hull): (env, g1 | g2 << 8 | pair index << 16)
  int work_cap;             // entries per queue
  HitRec<T> *hits;          // [hit_cap]  intersecting pairs of the current substep: the hits of work queue q occupy the first slots of
                            //   the queue's own item range, so that the narrow phase sees them grouped by second geom whatever
                            //   order the GJK warps finished in
  int hit_cap;
  int *nwork;               // [nsub+1][WSTRIDE]  per substep: items per queue [0..WQ), then pair cursor, large-tier envs
                            //   queued, large-tier cursor
  int *big;                 // [2][nenv]  envs of solver tier 1 / tier 2 in this substep
  T *con;                   // [N][CONBUF][8]  raw contacts: normal3, pos3, dist
  int *con_key;             // [N][CONBUF]     pair index << 20 | manifold index << 16 | g1 << 8 | g2  (sort key)
  int *ncon_raw;            // [N]
  uint8_t *active, *flags;  // [N]  env steps this call (not being reset) / env diverged during this control step
  uint8_t *tier;            // [N]  solver tier of the env in this substep (by contact / Jacobian-block count)
  int env0, nenv;           // env range of this pipeline group (work queues, hit list, counters and tier queues are per group)
};

// Streams of one pipeline group.  The envs of a handle are split into a few groups whose kernel sequences run concurrently
// (every kernel here is bound by the latency of its slowest warps, so independent groups fill each other's idle issue
// slots); inside a group the two larger solver tiers run on side streams beside tier 0 and join before the next kernel.
struct TierExec {
  cudaStream_t main = nullptr, sm = nullptr, sl = nullptr;
  cudaEvent_t start = nullptr, fork = nullptr, joinm = nullptr, joinl = nullptr, done = nullptr;
  void init() {
    cudaStreamCreateWithFlags(&main, cudaStreamNonBlocking);
    cudaStreamCreateWithFlags(&sm, cudaStreamNonBlocking); cudaStreamCreateWithFlags(&sl, cudaStreamNonBlocking);
    cudaEventCreateWithFlags(&fork, cudaEventDisableTiming); cudaEventCreateWithFlags(&joinm, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&joinl, cudaEventDisableTiming); cudaEventCreateWithFlags(&done, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&start, cudaEventDisableTiming);
  }
  void destroy() {
    if (main) {
      cudaStreamDestroy(main); cudaStreamDestroy(sm); cudaStreamDestroy(sl);
      cudaEventDestroy(fork); cudaEventDestroy(joinm); cudaEventDestroy(joinl); cudaEventDestroy(done); cudaEventDestroy(start);
      main = nullptr;
    }
  }
};

// Optional per-kernel timing with CUDA events on the launching stream (so101_kernel_times; bench.py's roofline leg).
// Kernel ids: 0 begin, 1 EPA + manifold (fused), 8 EPA / 9 manifold (two-launch narrow phase), 2 solve (tier 0), 3 solve (tier 1), 10 solve (tier 2), 4 arm-only step, 5 boolean GJK,
// 6 kinematics + smooth dynamics (thread per env), 7 broad phase / task layer.
struct KernelTimer {
  static constexpr int NK = 11;
  bool on = false;
  std::vector<std::array<cudaEvent_t, 2>> ev[NK];
  size_t used[NK] = {};
  double ms[NK] = {};
  uint64_t count[NK] = {};
  void begin(int id, cudaStream_t s) {
    if (!on) return;
    if (used[id] == ev[id].size()) {
      std::array<cudaEvent_t, 2> e;
      cudaEventCreate(&e[0]); cudaEventCreate(&e[1]);
      ev[id].push_back(e);
    }
    cudaEventRecord(ev[id][used[id]][0], s);
  }
  void end(int id, cudaStream_t s) {
    if (!on) return;
    cudaEventRecord(ev[id][used[id]][1], s);
    used[id]++;
  }
  void collect() {  // host-synchronises on the recorded events
    for (int id = 0; id < NK; id++) {
      for (size_t i = 0; i < used[id]; i++) {
        float t = 0.f;
        cudaEventSynchronize(ev[id][i][1]);
        if (cudaEventElapsedTime(&t, ev[id][i][0], ev[id][i][1]) == cudaSuccess) { ms[id] += t; count[id]++; }
      }
      used[id] = 0;
    }
  }
  ~KernelTimer() {
    for (auto &v : ev) for (auto &e : v) { cudaEventDestroy(e[0]); cudaEventDestroy(e[1]); }
  }
};

// pb / tx: one entry per pipeline group (ngroups of them)
template <typename T>
int launch_scene_step(const ArmSetT<T> &am, const ArmSetT<double> &am64, const SceneModel<T> &sm, const StepCfg &cfg, const EnvState<T> &S, const PipeBuf<T> *pb,
                      TierExec *tx, int ngroups, const float *action, const so101_step_out &out, cudaStream_t stream, KernelTimer *kt);
template <typename T>
void launch_scene_reset(const StepCfg &cfg, const EnvState<T> &S, const uint8_t *mask, const so101_step_out &out, cudaStream_t stream);
template <typename T>
void launch_settle_enter(const EnvState<T> &S, unsigned draw0, cudaStream_t stream);
template <typename T>
void launch_settle_leave(const EnvState<T> &S, cudaStream_t stream);
template <typename T>
size_t scene_smem_bytes();
template <typename T>
void launch_debug_overlap(const double *cases, int n, uint8_t *out, cudaStream_t stream);
template <typename T>
void scene_dropcat(int out[8]);
}  // namespace so101
