// Constraint rows and the primal Newton solver of the full contact scene, one warp per environment.
//
// Replaces [upstream] mj_makeConstraint + mj_fwdConstraint(solver = Newton, cone = elliptic) for the SO100 scene:
// unknown = delta = qacc - qacc_smooth (nv = 18), cost = 1/2 delta^T M delta + sum_rows s(J qacc - aref), rows =
// 6 friction-loss + <= 6 limit rows of the arm (diagonal Jacobians) and one elliptic cone of dimension condim per contact.
//
// Work mapping (32 lanes): per-contact arithmetic (cone zones, forces, J^T v) is lane-per-contact; the Hessian is assembled
// per 6x6 body block (arm / banana / bowl) with lanes over the block's entries and a warp-uniform loop over the contacts
// that touch the body (bit masks built with the rows); the 18x18 Cholesky is lanes-over-rows.  Everything a contact needs
// between Newton iterations lives in shared memory, so the code is loop-structured (not unrolled over contact slots) and
// small enough to stay in the instruction cache.  The line search re-uses J delta and J search: one evaluation costs a
// cone evaluation per contact and three warp reductions.
#pragma once
#include "arm_solver.cuh"
#include "scene_collide.cuh"

namespace so101 {

// where contacts / candidate pairs were dropped by a full buffer since the library was loaded (diagnostics):
// 0 NOUT per pair, 1 CANDCAP, 2 PAIRCAP, 3 work-queue capacity, 4 CONBUF raw contacts, 5 Jacobian block pool
__device__ int g_dropcat[8];
#define DROPCAT(i, n) atomicAdd(&g_dropcat[i], (int)(n))

constexpr int NH = NV * (NV + 1) / 2;  // 171 packed lower-triangular entries

__device__ __forceinline__ int tri(int i, int j) { return i * (i + 1) / 2 + j; }  // i >= j
// row of packed entry en (the inverse of tri): closed form instead of a search loop
__device__ __forceinline__ int tri_row(int en) {
  int i = (int)((sqrtf(8.f * (float)en + 1.f) - 1.f) * 0.5f);
  if ((i + 1) * (i + 2) / 2 <= en) i++;   // guard the float rounding at the row boundaries
  if (i * (i + 1) / 2 > en) i--;
  return i;
}

template <typename T, int NC, int NB>
struct SolveScratch {
  // Jacobian storage is a pool of 6x6 blocks (rows x dofs of ONE dynamic body); a contact owns one block per dynamic body
  // it touches (prop-vs-table: 1, grasp / prop-vs-prop: 2), block index fastest so that per-lane access is conflict-free.
  T J[36][NB];
  T w1[6][NB], w2[6][NB];  // J^T v1, J^T v2 per block: J^T Hc J = w1 w1^T - w2 w2^T + J^T diag(e) J
  T jar[6][NC];            // J (qacc_smooth + delta) - aref, updated in place by the line search
  T e[6][NC];
  T D0[NC], mu[NC], fri[3][NC];
  int info[NC];            // dim | baseA << 8 | baseB << 16   (dof base 0 / 6 / 12, 31 = no block)
  int blk[2][NC];          // pool index of block A / block B (-1 = none)
  unsigned bmask[NBLK][(NC + 31) / 32];  // contacts touching each 6-dof block (arm(s), object, container)
  union V {
    struct Con { T pos[3][NC], frame[9][NC], dist[NC]; int g1[NC], g2[NC]; } con;  // gathered contacts (until the rows are built)
    struct Ls { T jv[6][NC], frc[6][NC]; } ls;                                     // J search, cone forces (Newton iterations)
  } v;
};

// ------------------------------------------------------------------------------------------------ constraint rows (lane per contact)
// S must provide: sol (SolveScratch), ncon, xpos, xmat, arm_p, arm_a, qd.
template <typename T, typename S>
__device__ __forceinline__ void build_rows(const SceneModel<T> &sm, S &s, int &dropped, int lane) {
  auto &R = s.sol;
  constexpr int NC = sizeof(R.D0) / sizeof(T), NB = sizeof(R.w1[0]) / sizeof(T);
  const int ncon = s.ncon;
  int blk_base = 0;
#pragma unroll 1
  for (int c0 = 0; c0 < NC; c0 += 32) {
    const int c = c0 + lane;
    const bool valid = c < ncon;
    // allocate Jacobian blocks: one per distinct dynamic body (dof base) of the contact, in contact order
    int nb = 0, g1 = 0, g2 = 0, s1 = -1, s2 = -1;
    if (valid) {
      g1 = R.v.con.g1[c]; g2 = R.v.con.g2[c];
      s1 = sm.body_slot[sm.geom_body[g1]]; s2 = sm.body_slot[sm.geom_body[g2]];
      const int a1 = s1 < 0 ? 31 : (s1 < NA ? NJ * (s1 / NJ) : NA + 6 * (s1 - NA)), a2 = s2 < 0 ? 31 : (s2 < NA ? NJ * (s2 / NJ) : NA + 6 * (s2 - NA));
      nb = (a1 != 31) + (a2 != 31 && a2 != a1);
    }
    int incl = nb;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += v; }
    const int my_blk = blk_base + incl - nb;
    blk_base += wshfl(incl, 31);
    const bool fits = my_blk + nb <= NB;
    {
      const int nd = __popc(__ballot_sync(FULL, valid && !fits));
      dropped += nd;
      if (nd && lane == 0) DROPCAT(5, nd);
    }
    int baseA = 31, baseB = 31, bA = -1, bB = -1;
    if (valid) {
      const int b1 = sm.geom_body[g1], b2 = sm.geom_body[g2];
      // [upstream] mj_contactParam
      const int dim = max(sm.geom_condim[g1], sm.geom_condim[g2]);
      const int p1 = sm.geom_priority[g1], p2 = sm.geom_priority[g2];
      T f[3], mix;
      if (p1 == p2) {
        for (int k = 0; k < 3; k++) f[k] = max(sm.geom_friction[3 * g1 + k], sm.geom_friction[3 * g2 + k]);
        const T m1 = sm.geom_solmix[g1], m2 = sm.geom_solmix[g2];
        if (m1 >= T(1e-15) && m2 >= T(1e-15)) mix = m1 / (m1 + m2);
        else if (m1 < T(1e-15) && m2 < T(1e-15)) mix = T(0.5);
        else mix = m1 < T(1e-15) ? T(0) : T(1);
      } else {
        const int g = p1 > p2 ? g1 : g2;
        for (int k = 0; k < 3; k++) f[k] = sm.geom_friction[3 * g + k];
        mix = p1 > p2 ? T(1) : T(0);
      }
      T solref[2], solimp[5];
      const T *r1 = sm.geom_solref + 2 * g1, *r2 = sm.geom_solref + 2 * g2;
      if (r1[0] > T(0) && r2[0] > T(0)) for (int k = 0; k < 2; k++) solref[k] = mix * r1[k] + (T(1) - mix) * r2[k];
      else for (int k = 0; k < 2; k++) solref[k] = min(r1[k], r2[k]);
      for (int k = 0; k < 5; k++) solimp[k] = mix * sm.geom_solimp[5 * g1 + k] + (T(1) - mix) * sm.geom_solimp[5 * g2 + k];
      const T margin = max(sm.geom_margin[g1], sm.geom_margin[g2]) - max(sm.geom_gap[g1], sm.geom_gap[g2]);
      const T dist = R.v.con.dist[c];
      // impedance, reference acceleration gains, regulariser
      const T imp = impedance(solimp, dist, margin);
      const T dmax = t_clamp(solimp[1], T(1e-4), T(0.9999));
      T K, B;
      if (solref[0] > T(0)) {
        const T tc = solref[0] > T(2) * sm.timestep ? solref[0] : T(2) * sm.timestep;
        K = T(1) / (dmax * dmax * tc * tc * solref[1] * solref[1]); B = T(2) / (dmax * tc);
      } else { K = -solref[0] / (dmax * dmax); B = -solref[1] / dmax; }
      const T tran = sm.body_invweight0[2 * b1] + sm.body_invweight0[2 * b2];
      T R0 = (T(1) - imp) / imp * tran;
      R0 = R0 > T(1e-15) ? R0 : T(1e-15);
      R.D0[c] = T(1) / R0;
      R.fri[0][c] = f[0]; R.fri[1][c] = f[1]; R.fri[2][c] = f[2];
      R.mu[c] = dim > 1 ? f[0] * t_sqrt(T(1) / (sm.impratio > T(1e-15) ? sm.impratio : T(1e-15))) : T(0);
      // Jacobian blocks
      const T pos[3] = {R.v.con.pos[0][c], R.v.con.pos[1][c], R.v.con.pos[2][c]};
      T fr[9];
#pragma unroll
      for (int e = 0; e < 9; e++) fr[e] = R.v.con.frame[e][c];
      if (fits) {
        for (int k = 0; k < nb; k++)
          for (int e = 0; e < 36; e++) R.J[e][my_blk + k] = T(0);
#pragma unroll 1
        for (int side = 0; side < 2; side++) {
          const int sl = side ? s2 : s1;
          if (sl < 0) continue;
          const T sgn = side ? T(1) : T(-1);
          const int base = sl < NA ? NJ * (sl / NJ) : NA + 6 * (sl - NA);   // first dof of the body's block
          const int link = sl < NA ? sl - base : 0;                           // arm link index within its chain
          int bi;
          if (baseA == 31 || baseA == base) { baseA = base; bA = my_blk; bi = bA; }
          else { baseB = base; bB = my_blk + 1; bi = bB; }
#pragma unroll 1
          for (int col = 0; col < 6; col++) {
            T tr[3] = {T(0), T(0), T(0)}, ro[3] = {T(0), T(0), T(0)};
            if (sl < NA) {
              if (col > link) continue;
              const T a[3] = {s.arm_a[base + col][0], s.arm_a[base + col][1], s.arm_a[base + col][2]};
              const T r[3] = {pos[0] - s.arm_p[base + col][0], pos[1] - s.arm_p[base + col][1], pos[2] - s.arm_p[base + col][2]};
              cross3(tr, a, r);
              ro[0] = a[0]; ro[1] = a[1]; ro[2] = a[2];
            } else if (col < 3) {
              tr[col] = T(1);
            } else {
              const T *Rm = s.xmat[sl];
              const T a[3] = {Rm[col - 3], Rm[3 + col - 3], Rm[6 + col - 3]};
              const T r[3] = {pos[0] - s.xpos[sl][0], pos[1] - s.xpos[sl][1], pos[2] - s.xpos[sl][2]};
              cross3(tr, a, r);
              ro[0] = a[0]; ro[1] = a[1]; ro[2] = a[2];
            }
#pragma unroll
            for (int r = 0; r < 6; r++) {
              if (r < dim) {
                const T *ax = fr + 3 * (r % 3);
                const T v = sgn * (r < 3 ? dot3(ax, tr) : dot3(ax, ro));
                R.J[r * 6 + col][bi] += v;
              }
            }
          }
        }
      }
      const int edim = fits ? dim : 0;  // a contact whose blocks do not fit the pool is dropped (counted by the caller)
      R.info[c] = edim | (baseA << 8) | (baseB << 16);
      R.blk[0][c] = bA; R.blk[1][c] = bB;
      // jar at delta = 0: J qacc_smooth - aref, aref = -B vel - K imp (dist - margin) on the normal row; friction rows: -B vel
#pragma unroll 1
      for (int r = 0; r < 6; r++) {
        T vel = T(0), acc = T(0);
        if (r < edim) {
          for (int col = 0; col < 6; col++) {
            if (bA >= 0) { const T j = R.J[r * 6 + col][bA]; vel += j * s.qd[baseA + col]; acc += j * s.qacc_s[baseA + col]; }
            if (bB >= 0) { const T j = R.J[r * 6 + col][bB]; vel += j * s.qd[baseB + col]; acc += j * s.qacc_s[baseB + col]; }
          }
        }
        const T aref = r < edim ? (-B * vel - (r == 0 ? K * imp * (dist - margin) : T(0))) : T(0);
        R.jar[r][c] = acc - aref;
        R.e[r][c] = T(0);
      }
    }
    // contacts per body
#pragma unroll
    for (int b = 0; b < NBLK; b++) {
      const bool t = valid && ((bA >= 0 && baseA == 6 * b) || (bB >= 0 && baseB == 6 * b));
      const unsigned m = __ballot_sync(FULL, t);
      if (lane == 0) R.bmask[b][c0 >> 5] = m;
    }
  }
  __syncwarp();
}

// ------------------------------------------------------------------------------------------------ elliptic cone (per lane)
template <typename T>
struct Cone {
  int dim;
  T mu, S[6], D[6];
};
template <typename T, typename RS>
__device__ __forceinline__ void cone_setup(const RS &R, int c, T impratio, Cone<T> &k) {
  k.dim = R.info[c] & 0xff;
  k.mu = R.mu[c];
  const T f0 = R.fri[0][c], ft = R.fri[1][c], fr = R.fri[2][c], D0 = R.D0[c];
  const T D1 = D0 * (impratio > T(1e-15) ? impratio : T(1e-15));
  k.S[0] = k.mu; k.S[1] = f0; k.S[2] = f0; k.S[3] = ft; k.S[4] = fr; k.S[5] = fr;
  k.D[0] = D0; k.D[1] = D1; k.D[2] = D1; k.D[3] = D1 * ft * ft / (f0 * f0); k.D[4] = D1 * fr * fr / (f0 * f0); k.D[5] = k.D[4];
}
// zone 0: satisfied; 1: quadratic (bottom); 2: cone surface.  force = -d cost / d jar.  Hessian = v1 v1^T - v2 v2^T + diag(e).
template <typename T>
__device__ __forceinline__ int cone_eval(const Cone<T> &k, const T *x, T &cost, T *force, T *v1, T *v2, T *e) {
  const int dim = k.dim;
  cost = T(0);
#pragma unroll
  for (int j = 0; j < 6; j++) { force[j] = T(0); v1[j] = T(0); v2[j] = T(0); e[j] = T(0); }
  if (dim == 0) return 0;
  if (dim == 1) {
    if (x[0] >= T(0)) return 0;
    cost = T(0.5) * k.D[0] * x[0] * x[0]; force[0] = -k.D[0] * x[0]; e[0] = k.D[0];
    return 1;
  }
  T U[6], T2 = T(0);
  U[0] = x[0] * k.mu;
#pragma unroll
  for (int j = 1; j < 6; j++) { U[j] = j < dim ? x[j] * k.S[j] : T(0); T2 += U[j] * U[j]; }
  const T N = U[0], Tt = t_sqrt(T2), mu = k.mu;
  if (N >= mu * Tt || (Tt <= T(0) && N >= T(0))) return 0;
  if (mu * N + Tt <= T(0) || (Tt <= T(0) && N < T(0))) {
#pragma unroll
    for (int j = 0; j < 6; j++)
      if (j < dim) { cost += T(0.5) * k.D[j] * x[j] * x[j]; force[j] = -k.D[j] * x[j]; e[j] = k.D[j]; }
    return 1;
  }
  const T Dm = k.D[0] / (mu * mu * (T(1) + mu * mu)), NmT = N - mu * Tt;
  cost = T(0.5) * Dm * NmT * NmT;
  force[0] = -Dm * NmT * mu;
  // c2 > 0 in the middle zone.  Everything is written with the bounded ratios c2 / T and U / T: in float32 the textbook
  // form sqrt(c2 / T^3) overflows when the tangential slip T is tiny (T^3 underflows), which launched props into orbit.
  const T sDm = t_sqrt(Dm), c2 = -Dm * NmT * mu;
  const T ct = c2 / Tt, sct = t_sqrt(ct);
  v1[0] = sDm * mu;  // S0 * g0, g0 = 1
#pragma unroll
  for (int j = 1; j < 6; j++)
    if (j < dim) {
      const T un = U[j] / Tt;
      force[j] = -force[0] * un * k.S[j];
      v1[j] = sDm * k.S[j] * (-mu * un);
      v2[j] = sct * k.S[j] * un;
      e[j] = ct * k.S[j] * k.S[j];
    }
  return 2;
}

// ------------------------------------------------------------------------------------------------ Newton solver (warp)
template <typename T, typename S>
__device__ __forceinline__ T blockdiag_mv(const S &s, const T *x, int i) {  // (M x)_i for i < NV
  T acc = T(0);
  if (i < NA) {
    const int k = i / NJ, li = i % NJ;
#pragma unroll
    for (int j = 0; j < NJ; j++) acc += (j <= li ? s.Marm[k][tri(li, j)] : s.Marm[k][tri(j, li)]) * x[NJ * k + j];
  } else {
    const int p = (i - NA) / 6, li = (i - NA) % 6;
#pragma unroll
    for (int j = 0; j < 6; j++) acc += (j <= li ? s.Mprop[p][tri(li, j)] : s.Mprop[p][tri(j, li)]) * x[NA + 6 * p + j];
  }
  return acc;
}

// v[r][c] = sum_col J[r][col] x[base + col] over the contact's (<= 2) blocks, for the lane's contacts
template <typename T, typename S>
__device__ __forceinline__ void contacts_Jx(S &s, const T *x, int lane) {  // -> R.v.ls.jv
  auto &R = s.sol;
#pragma unroll 1
  for (int c = lane; c < s.ncon; c += 32) {
    const int inf = R.info[c], dim = inf & 0xff, baseA = (inf >> 8) & 0xff, baseB = (inf >> 16) & 0xff, bA = R.blk[0][c], bB = R.blk[1][c];
#pragma unroll 1
    for (int r = 0; r < 6; r++) {
      T acc = T(0);
      if (r < dim) {
#pragma unroll
        for (int col = 0; col < 6; col++) {
          if (bA >= 0) acc += R.J[r * 6 + col][bA] * x[baseA + col];
          if (bB >= 0) acc += R.J[r * 6 + col][bB] * x[baseB + col];
        }
      }
      R.v.ls.jv[r][c] = acc;
    }
  }
  __syncwarp();
}

// per-lane view of the arms' friction-loss / limit rows (lane i < NA owns arm dof i)
template <typename T>
struct ArmLane {
  T jar0_f, eta, rf, frD, jar0_l, D_l, js;
};

// cost, slope and curvature of all constraint rows along delta + alpha * search (warp-uniform result).
// Contacts: jar + alpha * jv through the cone; arm rows on lanes < NJ.
template <typename T, typename S>
__device__ __noinline__ void rows_line(S &s, const ArmLane<T> &al, T impratio, T alpha, T &c, T &g, T &h, int lane) {
  auto &R = s.sol;
  T lc = T(0), lg = T(0), lh = T(0);
#pragma unroll 1
  for (int ci = lane; ci < s.ncon; ci += 32) {
    Cone<T> cone;
    cone_setup(R, ci, impratio, cone);
    if (cone.dim == 0) continue;
    T jv[6], xx[6], force[6], v1[6], v2[6], e[6], cc;
#pragma unroll
    for (int r = 0; r < 6; r++) { jv[r] = R.v.ls.jv[r][ci]; xx[r] = R.jar[r][ci] + alpha * jv[r]; }
    cone_eval(cone, xx, cc, force, v1, v2, e);
    T a1 = T(0), a2 = T(0);
    lc += cc;
#pragma unroll
    for (int r = 0; r < 6; r++) { lg -= force[r] * jv[r]; a1 += v1[r] * jv[r]; a2 += v2[r] * jv[r]; lh += e[r] * jv[r] * jv[r]; }
    lh += a1 * a1 - a2 * a2;
  }
  if (lane < NA) {
    const T sv = s.search[lane];
    const T x = al.jar0_f + s.delta[lane] + alpha * sv;
    if (x <= -al.rf) { lc += al.eta * (T(-0.5) * al.rf - x); lg -= al.eta * sv; }
    else if (x >= al.rf) { lc += al.eta * (T(-0.5) * al.rf + x); lg += al.eta * sv; }
    else { lc += T(0.5) * al.frD * x * x; lg += al.frD * x * sv; lh += al.frD * sv * sv; }
    if (al.D_l > T(0)) {
      const T jvl = al.js * sv, xl = al.jar0_l + al.js * s.delta[lane] + alpha * jvl;
      if (xl < T(0)) { lc += T(0.5) * al.D_l * xl * xl; lg += al.D_l * xl * jvl; lh += al.D_l * jvl * jvl; }
    }
  }
  c += warp_sum(lc); g += warp_sum(lg); h += warp_sum(lh);
}

template <typename T>
__device__ __forceinline__ void cholesky_packed(T *H, int lane) {  // in-place lower Cholesky of the packed NV x NV matrix, lanes = rows
#pragma unroll 1
  for (int j = 0; j < NV; j++) {
    T sacc = T(0);
    if (lane >= j && lane < NV) {
      sacc = H[tri(lane, j)];
      for (int k = 0; k < j; k++) sacc -= H[tri(lane, k)] * H[tri(j, k)];
    }
    T dg = wshfl(sacc, j);
    dg = t_sqrt(dg > T(1e-15) ? dg : T(1e-15));
    if (lane >= j && lane < NV) H[tri(lane, j)] = lane == j ? dg : sacc / dg;
    __syncwarp();
  }
}
template <typename T>
__device__ __forceinline__ T chol_solve_packed(const T *L, T b, int lane) {  // lane i holds b_i; returns x_i
#pragma unroll 1
  for (int k = 0; k < NV; k++) {
    const T yk = wshfl(b, k) / L[tri(k, k)];
    if (lane == k) b = yk;
    else if (lane > k && lane < NV) b -= L[tri(lane, k)] * yk;
  }
#pragma unroll 1
  for (int k = NV - 1; k >= 0; k--) {
    const T xk = wshfl(b, k) / L[tri(k, k)];
    if (lane == k) b = xk;
    else if (lane < k) b -= L[tri(k, lane)] * xk;
  }
  return b;
}

// Block-diagonal case (no contact couples two bodies: the usual resting scene): the three 6x6 blocks factor independently, 6
// columns instead of 18.  Bitwise identical to the full routines on such a matrix (the skipped products are all 0 * x).
template <typename T>
__device__ __forceinline__ void cholesky_blocks(T *H, int lane) {
  const int b = lane / 6, r = lane - 6 * b, base = 6 * b;
  const bool act = lane < NV;
#pragma unroll 1
  for (int j = 0; j < 6; j++) {
    T sacc = T(0);
    if (act && r >= j) {
      sacc = H[tri(base + r, base + j)];
      for (int k = 0; k < j; k++) sacc -= H[tri(base + r, base + k)] * H[tri(base + j, base + k)];
    }
    T dg = __shfl_sync(FULL, sacc, act ? base + j : 0);
    dg = t_sqrt(dg > T(1e-15) ? dg : T(1e-15));
    if (act && r >= j) H[tri(base + r, base + j)] = r == j ? dg : sacc / dg;
    __syncwarp();
  }
}
template <typename T>
__device__ __forceinline__ T chol_solve_blocks(const T *L, T bv, int lane) {
  const int b = lane / 6, r = lane - 6 * b, base = 6 * b;
  const bool act = lane < NV;
#pragma unroll 1
  for (int k = 0; k < 6; k++) {
    const T yk = __shfl_sync(FULL, bv, act ? base + k : 0) / (act ? L[tri(base + k, base + k)] : T(1));
    if (act) { if (r == k) bv = yk; else if (r > k) bv -= L[tri(base + r, base + k)] * yk; }
  }
#pragma unroll 1
  for (int k = 5; k >= 0; k--) {
    const T xk = __shfl_sync(FULL, bv, act ? base + k : 0) / (act ? L[tri(base + k, base + k)] : T(1));
    if (act) { if (r == k) bv = xk; else if (r < k) bv -= L[tri(base + k, base + r)] * xk; }
  }
  return bv;
}

// One Newton pass over the contacts: cone forces, factored cone Hessians (e, w1 = J^T v1, w2 = J^T v2).  Lane per contact.
template <typename T, typename S>
__device__ __forceinline__ void contacts_eval(S &s, T impratio, int lane) {
  auto &R = s.sol;
#pragma unroll 1
  for (int ci = lane; ci < s.ncon; ci += 32) {
    Cone<T> cone;
    cone_setup(R, ci, impratio, cone);
    T xx[6], frc[6], v1[6], v2[6], e[6], cc;
#pragma unroll
    for (int r = 0; r < 6; r++) xx[r] = R.jar[r][ci];
    cone_eval(cone, xx, cc, frc, v1, v2, e);
#pragma unroll
    for (int r = 0; r < 6; r++) { R.e[r][ci] = e[r]; R.v.ls.frc[r][ci] = frc[r]; }
#pragma unroll 1
    for (int side = 0; side < 2; side++) {
      const int bi = R.blk[side][ci];
      if (bi < 0) continue;
#pragma unroll 1
      for (int col = 0; col < 6; col++) {
        T a1 = T(0), a2 = T(0);
#pragma unroll
        for (int r = 0; r < 6; r++) { const T j = R.J[r * 6 + col][bi]; a1 += j * v1[r]; a2 += j * v2[r]; }
        R.w1[col][bi] = a1; R.w2[col][bi] = a2;
      }
    }
  }
  __syncwarp();
}

// Hessian H = M + J^T Hc J (+ arm row curvature) and gradient Md - J^T f - f_arm, assembled per body block.
template <typename T, typename S>
__device__ __forceinline__ void assemble(S &s, T f_arm, T hdiag_arm, int lane) {
  auto &R = s.sol;
  constexpr int NCH = sizeof(R.bmask[0]) / sizeof(unsigned);
  // unpack the lane's entry of a packed 6x6 lower triangle
  const int ti = tri_row(lane), tj = lane - ti * (ti + 1) / 2;
  const int gk = lane - 21;  // gradient entry owned by lanes 21..26
#pragma unroll 1
  for (int b = 0; b < NBLK; b++) {
    const int base = 6 * b;
    T acc = T(0);
    if (lane < 21) acc = b < NARM ? s.Marm[b][lane] : s.Mprop[b - NARM][lane];
    T gacc = T(0);
#pragma unroll 1
    for (int ch = 0; ch < NCH; ch++) {
      unsigned m = R.bmask[b][ch];
      while (m) {
        const int c = 32 * ch + __ffs(m) - 1;
        m &= m - 1;
        const int inf = R.info[c];
        const int bi = ((inf >> 8) & 0xff) == base ? R.blk[0][c] : R.blk[1][c];
        if (lane < 21) {
          T a = R.w1[ti][bi] * R.w1[tj][bi] - R.w2[ti][bi] * R.w2[tj][bi];
#pragma unroll
          for (int r = 0; r < 6; r++) a += R.e[r][c] * R.J[r * 6 + ti][bi] * R.J[r * 6 + tj][bi];
          acc += a;
        } else if (lane < 27) {
#pragma unroll
          for (int r = 0; r < 6; r++) gacc += R.J[r * 6 + gk][bi] * R.v.ls.frc[r][c];
        }
      }
    }
    const T hd = __shfl_sync(FULL, hdiag_arm, (base + ti) & 31);  // arm row curvature of dof base + ti lives on that lane
    if (lane < 21) s.H[tri(base + ti, base + tj)] = acc + ((b < NARM && ti == tj) ? hd : T(0));
    else if (lane < 27) s.grad[base + gk] = s.Md[base + gk] - gacc;
  }
  // off-diagonal blocks (hi, lo): only contacts that touch both bodies (grasp, banana in bowl)
#pragma unroll 1
  for (int pr = 0; pr < NBLK * (NBLK - 1) / 2; pr++) {
    // block pairs (hi, lo), hi > lo, in the order (1,0) (2,0) (2,1) (3,0) ...
    int hi = 1, lo = pr;
    while (lo >= hi) { lo -= hi; hi++; }
#pragma unroll 1
    for (int en = lane; en < 36; en += 32) {
      const int i = en / 6, j = en % 6;
      T acc = T(0);
#pragma unroll 1
      for (int ch = 0; ch < NCH; ch++) {
        unsigned m = R.bmask[hi][ch] & R.bmask[lo][ch];
        while (m) {
          const int c = 32 * ch + __ffs(m) - 1;
          m &= m - 1;
          const int inf = R.info[c];
          const bool a_hi = ((inf >> 8) & 0xff) == 6 * hi;
          const int bh = a_hi ? R.blk[0][c] : R.blk[1][c], bl = a_hi ? R.blk[1][c] : R.blk[0][c];
          T a = R.w1[i][bh] * R.w1[j][bl] - R.w2[i][bh] * R.w2[j][bl];
#pragma unroll
          for (int r = 0; r < 6; r++) a += R.e[r][c] * R.J[r * 6 + i][bh] * R.J[r * 6 + j][bl];
          acc += a;
        }
      }
      s.H[tri(6 * hi + i, 6 * lo + j)] = acc;
    }
  }
  __syncwarp();
  if (lane < NA) s.grad[lane] -= f_arm;
  __syncwarp();
}

// Returns the Newton iteration count.  In: s.delta = warm start (qacc_warmstart - qacc_smooth); out: s.delta = solution.
template <typename T, typename S>
__device__ __noinline__ int scene_solve(const ArmSetT<T> &ams, T impratio, S &s, int max_iter, T tol, int lane) {
  const ArmModelT<T> &am = ams[0];   // (solver_scale is a property of the scene, stored with every arm)
  auto &R = s.sol;
  const int ncon = s.ncon;
  const T xeps = sizeof(T) == 8 ? T(1e-14) : T(2e-6);
  ArmLane<T> al{};
  if (lane < NA) {
    const int k = lane / NJ, j = lane % NJ;
    al.jar0_f = s.arows[k].jar0_f[j]; al.eta = ams[k].frictionloss[j]; al.rf = ams[k].fr_R[j] * al.eta; al.frD = ams[k].fr_D[j];
    al.jar0_l = s.arows[k].jar0_l[j]; al.D_l = s.arows[k].D_l[j]; al.js = s.arows[k].js[j];
  }
  // warm start: keep it only if it beats delta = 0.  Evaluate both along the line 0 + alpha * warm.
  {
    T w = T(0);
    if (lane < NV) { w = s.delta[lane]; s.search[lane] = w; s.delta[lane] = T(0); }
    __syncwarp();
    contacts_Jx<T>(s, s.search, lane);
    T c0 = T(0), cw = T(0), g = T(0), h = T(0);
    rows_line(s, al, impratio, T(0), c0, g, h, lane);
    const T mw = lane < NV ? blockdiag_mv(s, s.search, lane) : T(0);
    cw = T(0.5) * warp_sum(mw * w);
    rows_line(s, al, impratio, T(1), cw, g, h, lane);
    const bool keep = cw < c0;
    if (lane < NV) { s.delta[lane] = keep ? w : T(0); s.Md[lane] = keep ? mw : T(0); }
    if (keep)
      for (int c = lane; c < ncon; c += 32)
#pragma unroll
        for (int r = 0; r < 6; r++) R.jar[r][c] += R.v.ls.jv[r][c];
    __syncwarp();
  }
  // does any contact couple two bodies (grasp, banana in the bowl)?  If not, the Hessian is block diagonal.
  bool decoupled = true;
  for (int ch = 0; ch < (int)(sizeof(R.bmask[0]) / sizeof(unsigned)); ch++) {
    unsigned seen = 0;
    for (int b = 0; b < NBLK; b++) { if (seen & R.bmask[b][ch]) decoupled = false; seen |= R.bmask[b][ch]; }
  }
  int iter = 0;
#pragma unroll 1
  for (; iter < max_iter; iter++) {
    contacts_eval(s, impratio, lane);
    // arm rows: force and diagonal curvature (lane i < NJ)
    T f_arm = T(0), hdiag = T(0);
    if (lane < NA) {
      const T x = al.jar0_f + s.delta[lane];
      if (x <= -al.rf) f_arm = al.eta;
      else if (x >= al.rf) f_arm = -al.eta;
      else { f_arm = -al.frD * x; hdiag = al.frD; }
      if (al.D_l > T(0)) {
        const T xl = al.jar0_l + al.js * s.delta[lane];
        if (xl < T(0)) { f_arm += al.js * (-al.D_l * xl); hdiag += al.D_l; }
      }
    }
    assemble(s, f_arm, hdiag, lane);
    const T gl = lane < NV ? s.grad[lane] : T(0);
    const T mdl = lane < NV ? s.Md[lane] : T(0);
    const T gn = t_sqrt(warp_sum(gl * gl));
    if (am.solver_scale * gn < tol) break;
    // float32 only: symmetric diagonal (Jacobi) scaling H' = S H S, S = diag(H_ii^-1/2).  The Hessian mixes translational
    // and rotational dofs of bodies from 0.04 kg props to the armature-dominated arm with contact stiffness up to 1e5 and
    // rolling-friction rows 1e-4 of that: its condition number exceeds what a float32 Cholesky resolves unless the scales
    // are taken out first.  (float64 keeps the unscaled factorisation: bit-compatible with the oracle.)
    T hs = T(1);
    if (sizeof(T) == 4) {
      if (lane < NV) { const T dgn = s.H[tri(lane, lane)]; hs = dgn > T(1e-30) ? T(1) / t_sqrt(dgn) : T(1); s.hscale[lane] = hs; }
      __syncwarp();
#pragma unroll 1
      for (int en = lane; en < NH; en += 32) {
        const int i = tri_row(en), j = en - i * (i + 1) / 2;
        s.H[en] *= s.hscale[i] * s.hscale[j];
      }
      __syncwarp();
    }
    T sr;
    if (decoupled) { cholesky_blocks(s.H, lane); sr = chol_solve_blocks(s.H, -gl * hs, lane); }
    else { cholesky_packed(s.H, lane); sr = chol_solve_packed(s.H, -gl * hs, lane); }
    sr *= hs;
    if (lane < NV) s.search[lane] = sr;
    __syncwarp();
    contacts_Jx<T>(s, s.search, lane);
    const T msl = lane < NV ? blockdiag_mv(s, s.search, lane) : T(0);
    const T q0 = T(0.5) * warp_sum(lane < NV ? s.delta[lane] * mdl : T(0));
    const T q1 = warp_sum(lane < NV ? sr * mdl : T(0));
    const T q2 = warp_sum(lane < NV ? sr * msl : T(0));
    T f0 = q0, df0 = q1, ddf0 = q2;
    rows_line(s, al, impratio, T(0), f0, df0, ddf0, lane);
    if (df0 >= T(0) || ddf0 <= T(0)) break;
    T alpha = -df0 / ddf0, lo = T(0), hi = T(-1), f = f0;
#pragma unroll 1
    for (int ls = 0; ls < 30; ls++) {
      T df = q1 + alpha * q2, ddf = q2;
      f = q0 + alpha * q1 + T(0.5) * alpha * alpha * q2;
      rows_line(s, al, impratio, alpha, f, df, ddf, lane);
      if (t_abs(df) <= T(0.01) * t_abs(df0)) break;  // [upstream] mjOption.ls_tolerance = 0.01 (same constant in the oracle)
      if (df < T(0)) lo = alpha; else hi = alpha;
      T next = alpha - df / ddf;
      if (hi > T(0) && (next <= lo || next >= hi)) next = T(0.5) * (lo + hi);
      else if (hi < T(0) && next <= lo) next = T(2) * alpha;
      if (next == alpha || t_abs(next - alpha) <= xeps * t_abs(alpha) || (hi > T(0) && hi - lo <= xeps * hi)) { alpha = next; break; }
      alpha = next;
    }
    T st = T(0), am_ = T(1);
    if (lane < NV) {
      st = alpha * sr;
      s.delta[lane] += st;
      s.Md[lane] = mdl + alpha * msl;
      am_ = t_abs(s.qacc_s[lane]) + t_abs(s.delta[lane]);
      st = t_abs(st);
    }
    for (int c = lane; c < ncon; c += 32)
#pragma unroll
      for (int r = 0; r < 6; r++) R.jar[r][c] += alpha * R.v.ls.jv[r][c];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { st = max(st, __shfl_xor_sync(FULL, st, o)); am_ = max(am_, __shfl_xor_sync(FULL, am_, o)); }
    __syncwarp();
    if (am.solver_scale * (f0 - f) < tol || st <= xeps * max(am_, T(1))) { iter++; break; }
  }
  return iter;
}

}  // namespace so101
