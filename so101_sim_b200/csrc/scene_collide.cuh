// Convex narrow phase, shared pieces: shapes, hull support mapping, boolean GJK, polytope / polygon scratch.
//
// Replaces [upstream] mj_collision's narrow phase for the SO100 scene: boolean GJK -> EPA -> support-feature clipping (the
// multiccd manifold, so100_task.py:151), ONE THREAD per geom pair (scene_collide_seq.cuh holds EPA and the manifold).
// The algorithm, its tolerances and its tie-breaking mirror oracle/so101_collide.c so that float64 runs agree to round-off.
#pragma once
#include "scene_model.cuh"

namespace so101 {

constexpr int NCON = 128;        // contacts per env the parity probe (debug_contacts) can report: all CONBUF of them
constexpr int PAIRCAP = 64;      // candidate geom pairs per env per substep (after the OBB mid phase)
constexpr int CONBUF = 128;      // raw contacts per env the narrow phase may write between two kernels
constexpr int EPA_MAXV = 96, EPA_MAXF = 256;
constexpr int EPA_MAXIT = 50;  // [upstream] mjOption.ccd_iterations default (same constant in the oracle)
constexpr int MAXCAND = 32, MAXFEAT = 16, MAXMANI = 4;
// Hull slabs with more than FEAT_EXACT vertices are represented by their extreme points along 16 tangent-plane directions
// (scene_collide_seq.cuh feature_seq; oracle/so101_collide.c feature()); smaller ones keep the exact 2-D hull.
constexpr int FEAT_EXACT = 16;
template <typename T> __device__ __forceinline__ constexpr T feat_cos(int k) {
  return k == 0 ? T(1.0) : k == 1 ? T(0.92387953251128674) : k == 2 ? T(0.70710678118654752) : k == 3 ? T(0.38268343236508977) : k == 4 ? T(0.0)
       : k == 5 ? T(-0.38268343236508977) : k == 6 ? T(-0.70710678118654752) : T(-0.92387953251128674);
}
template <typename T> __device__ __forceinline__ constexpr T feat_sin(int k) {
  return k == 0 ? T(0.0) : k == 1 ? T(0.38268343236508977) : k == 2 ? T(0.70710678118654752) : k == 3 ? T(0.92387953251128674) : k == 4 ? T(1.0)
       : k == 5 ? T(0.92387953251128674) : k == 6 ? T(0.70710678118654752) : T(0.38268343236508977);
}
constexpr unsigned FULL = 0xffffffffu;

template <typename T>
struct Shape {
  int type, geom, vadr, vnum;
  int nbase;  // first adjacency entry of this hull (hull_nbradr[vadr])
  int hint;  // hill-climbing warm start: last support vertex of this shape while its pair is processed
  T pos[3], mat[9], size[3], center[3], rbound;
};

template <typename T>
struct FPt {
  T x, y, h;
};

// Height interpolant of a support feature over its (t1, t2) plane: constant (vertex), line (edge) or plane (face).
template <typename T>
struct HPlane {
  int mode;
  T x0, y0, h0, ex, ey, eh, el, fx, fy, fh, det;
};

// Per-thread scratch of one narrow-phase pair (local memory).  The EPA polytope is dead once epa_seq() has returned
// (normal, depth and witness points are in registers), so the manifold stage re-uses its storage.
template <typename T>
struct CollideScratch {
  union {
    struct {  // EPA polytope
      T Vw[3][EPA_MAXV], Va[3][EPA_MAXV], Vb[3][EPA_MAXV];
      unsigned char Fv[3][EPA_MAXF];  // vertex ids < EPA_MAXV
      T Fn[3][EPA_MAXF], Fd[EPA_MAXF];
      unsigned char Falive[EPA_MAXF];
      unsigned short horizon[EPA_MAXF];  // directed edges a | b << 8 (vertex ids < EPA_MAXV <= 255)
    };
    struct {  // manifold
      T cand[3][MAXCAND];
      FPt<T> P[MAXCAND], Hh[2 * MAXCAND + 2], FA[MAXFEAT], FB[MAXFEAT], R[2 * MAXFEAT + 8], bufA[2 * MAXFEAT + 8], bufB[2 * MAXFEAT + 8];
      T mdist[2 * MAXFEAT + 8], mdist2[2 * MAXFEAT + 8];
      HPlane<T> hp[2];  // height interpolants of the two features
      int candi[FEAT_EXACT];  // hull vertex ids of the first FEAT_EXACT slab vertices (feature_seq)
    };
  };
};

template <typename T> __device__ __forceinline__ T wshfl(T v, int src) { return __shfl_sync(FULL, v, src); }
template <typename T> __device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
  return v;
}

template <typename T> __device__ __forceinline__ T dot3(const T *a, const T *b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
template <typename T> __device__ __forceinline__ void cross3(T *r, const T *a, const T *b) {
  const T x = a[1] * b[2] - a[2] * b[1], y = a[2] * b[0] - a[0] * b[2], z = a[0] * b[1] - a[1] * b[0];
  r[0] = x; r[1] = y; r[2] = z;
}
template <typename T> __device__ __forceinline__ void sub3(T *r, const T *a, const T *b) { r[0] = a[0] - b[0]; r[1] = a[1] - b[1]; r[2] = a[2] - b[2]; }
template <typename T> __device__ __forceinline__ void mulmv(T *r, const T *m, const T *v) {
  const T x = m[0] * v[0] + m[1] * v[1] + m[2] * v[2], y = m[3] * v[0] + m[4] * v[1] + m[5] * v[2], z = m[6] * v[0] + m[7] * v[1] + m[8] * v[2];
  r[0] = x; r[1] = y; r[2] = z;
}
template <typename T> __device__ __forceinline__ void mulmtv(T *r, const T *m, const T *v) {
  const T x = m[0] * v[0] + m[3] * v[1] + m[6] * v[2], y = m[1] * v[0] + m[4] * v[1] + m[7] * v[2], z = m[2] * v[0] + m[5] * v[1] + m[8] * v[2];
  r[0] = x; r[1] = y; r[2] = z;
}
template <typename T> __device__ __forceinline__ void local2world(const Shape<T> &s, const T *l, T *w) {
  mulmv(w, s.mat, l);
  w[0] += s.pos[0]; w[1] += s.pos[1]; w[2] += s.pos[2];
}

// world pose of geom g.  xpos/xmat: the env's dynamic body poses (shared memory).
template <typename T>
__device__ __forceinline__ void make_shape(const SceneModel<T> &sm, const T (*xpos)[3], const T (*xmat)[9], int g, Shape<T> &s) {
  s.type = sm.geom_type[g]; s.geom = g; s.vadr = sm.geom_vertadr[g]; s.vnum = sm.geom_vertnum[g];
  s.nbase = s.type == G_HULL ? sm.hull_nbradr[s.vadr] : 0;
  s.hint = 0;
  s.rbound = sm.geom_rbound[g];
  const int slot = sm.geom_slot[g];
#pragma unroll
  for (int c = 0; c < 3; c++) s.size[c] = sm.geom_size[3 * g + c];
  if (slot < 0) {
#pragma unroll
    for (int c = 0; c < 3; c++) { s.pos[c] = sm.geom_pos[3 * g + c]; s.center[c] = sm.geom_bcenter[3 * g + c]; }
#pragma unroll
    for (int c = 0; c < 9; c++) s.mat[c] = sm.geom_mat[9 * g + c];
  } else {
    const T *X = xpos[slot], *R = xmat[slot];
    T gp[3] = {sm.geom_pos[3 * g], sm.geom_pos[3 * g + 1], sm.geom_pos[3 * g + 2]}, t[3];
    mulmv(t, R, gp);
#pragma unroll
    for (int c = 0; c < 3; c++) s.pos[c] = X[c] + t[c];
    T gc[3] = {sm.geom_bcenter[3 * g], sm.geom_bcenter[3 * g + 1], sm.geom_bcenter[3 * g + 2]};
    mulmv(t, R, gc);
#pragma unroll
    for (int c = 0; c < 3; c++) s.center[c] = X[c] + t[c];
#pragma unroll
    for (int i = 0; i < 3; i++)
#pragma unroll
      for (int j = 0; j < 3; j++) {
        T v = T(0);
#pragma unroll
        for (int k = 0; k < 3; k++) v += R[3 * i + k] * sm.geom_mat[9 * g + 3 * k + j];
        s.mat[3 * i + j] = v;
      }
  }
}

template <typename T>
struct MPoint {
  T w[3], a[3], b[3];
};
// ---- one THREAD per pair (boolean-GJK kernel): the thread scans all hull vertices itself.  Lanes of a warp work on the same
// hull for different envs (queue order), so every vertex load is a warp-wide broadcast.  Same first-maximum tie-break as the
// warp-cooperative support() above.
constexpr int HILLCLIMB_MIN = 40;  // hulls with fewer vertices are scanned exhaustively (same constant in the oracle)

// Hull support: exhaustive scan for small hulls, otherwise steepest-ascent hill climbing on the hull's vertex graph,
// warm-started from the previous support vertex of this shape ([upstream] MuJoCo's mesh support does the same for meshes
// with a vertex graph; on a convex hull a graph-local maximum is the global one).  Mirrors support() of the oracle.
template <typename T>
__device__ __forceinline__ void support_seq(const SceneModel<T> &sm, Shape<T> &s, const T *dir, T *out) {
  T dl[3], p[3];
  mulmtv(dl, s.mat, dir);
  if (s.type == G_HULL) {
    const Vec4<T> *vt = sm.hull_vert + s.vadr;
    int bi;
    if (s.vnum < HILLCLIMB_MIN) {
      T bv = -INFINITY;
      bi = 0;
#pragma unroll 4
      for (int i = 0; i < s.vnum; i++) {
        const Vec4<T> v = vt[i];
        const T val = v.x * dl[0] + v.y * dl[1] + v.z * dl[2];
        if (val > bv) { bv = val; bi = i; }
      }
    } else {
      const int *adr = sm.hull_nbradr + s.vadr;
      int cur = s.hint;
      Vec4<T> v = vt[cur];
      T bv = v.x * dl[0] + v.y * dl[1] + v.z * dl[2];
      int k0 = adr[cur], k1 = adr[cur + 1];
#pragma unroll 1
      for (int guard = 0; guard < s.vnum; guard++) {  // (a non-finite direction cannot climb: the loop ends at once)
        unsigned best = 0xffffffffu;
#pragma unroll 4
        for (int k = k0; k < k1; k++) {
          // neighbour coordinates stored with the adjacency entry, together with where ITS neighbours are: one load per
          // neighbour and no index chase between steps
          const Vec4<T> nb = sm.hull_nbrv[k];
          const T val = nb.x * dl[0] + nb.y * dl[1] + nb.z * dl[2];
          if (val > bv) { bv = val; best = nbr_bits(nb.w); }
        }
        if (best == 0xffffffffu) break;
        cur = (int)(best & ((1u << NBR_ID_BITS) - 1));
        k0 = s.nbase + (int)(best >> (NBR_ID_BITS + NBR_DEG_BITS));
        k1 = k0 + (int)((best >> NBR_ID_BITS) & ((1u << NBR_DEG_BITS) - 1));
      }
      bi = cur;
      s.hint = cur;
    }
    const Vec4<T> vb = vt[bi];
    p[0] = vb.x; p[1] = vb.y; p[2] = vb.z;
  } else if (s.type == G_BOX) {
#pragma unroll
    for (int c = 0; c < 3; c++) p[c] = dl[c] >= T(0) ? s.size[c] : -s.size[c];
  } else if (s.type == G_CYLINDER) {
    const T n = t_sqrt(dl[0] * dl[0] + dl[1] * dl[1]);
    p[0] = n > T(1e-15) ? s.size[0] * dl[0] / n : T(0); p[1] = n > T(1e-15) ? s.size[0] * dl[1] / n : T(0);
    p[2] = dl[2] >= T(0) ? s.size[1] : -s.size[1];
  } else if (s.type == G_CAPSULE || s.type == G_SPHERE) {
    const T n = t_sqrt(dot3(dl, dl));
#pragma unroll
    for (int c = 0; c < 3; c++) p[c] = n > T(1e-15) ? s.size[0] * dl[c] / n : T(0);
    if (s.type == G_CAPSULE) p[2] += dl[2] >= T(0) ? s.size[1] : -s.size[1];
  } else { p[0] = p[1] = p[2] = T(0); }
  local2world(s, p, out);
}
template <typename T>
__device__ __forceinline__ void msupport_seq(const SceneModel<T> &sm, Shape<T> &A, Shape<T> &B, const T *d, MPoint<T> &p) {
  const T nd[3] = {-d[0], -d[1], -d[2]};
  support_seq(sm, A, d, p.a); support_seq(sm, B, nd, p.b);
  sub3(p.w, p.a, p.b);
}

// boolean GJK; mirrors gjk_intersect() of the oracle.  Uniform control flow across the warp.
template <typename T>
__device__ __forceinline__ int gjk_intersect(const SceneModel<T> &sm, Shape<T> &A, Shape<T> &B, MPoint<T> *S, int &np) {
  T d[3];
  sub3(d, B.center, A.center);
  if (dot3(d, d) < T(1e-20)) { d[0] = T(1); d[1] = T(0); d[2] = T(0); }
  int n = 0;
  #pragma unroll 1
  for (int it = 0; it < 64; it++) {
    MPoint<T> p;
    msupport_seq(sm, A, B, d, p);
    if (dot3(p.w, d) < T(0)) { np = n; return 0; }
    S[n++] = p;
    if (n == 1) { d[0] = -S[0].w[0]; d[1] = -S[0].w[1]; d[2] = -S[0].w[2]; }
    else if (n == 2) {
      T ab[3], ao[3] = {-S[1].w[0], -S[1].w[1], -S[1].w[2]}, t[3];
      sub3(ab, S[0].w, S[1].w);
      if (dot3(ab, ao) > T(0)) { cross3(t, ab, ao); cross3(d, t, ab); }
      else { S[0] = S[1]; n = 1; d[0] = ao[0]; d[1] = ao[1]; d[2] = ao[2]; }
    } else if (n == 3) {
      T *a = S[2].w, *b = S[1].w, *c = S[0].w, ab[3], ac[3], ao[3] = {-a[0], -a[1], -a[2]}, abc[3], t[3], u[3];
      sub3(ab, b, a); sub3(ac, c, a); cross3(abc, ab, ac);
      cross3(t, abc, ac);
      bool star = false;
      if (dot3(t, ao) > T(0)) {
        if (dot3(ac, ao) > T(0)) { S[1] = S[2]; n = 2; cross3(u, ac, ao); cross3(d, u, ac); }
        else star = true;
      } else {
        cross3(t, ab, abc);
        if (dot3(t, ao) > T(0)) star = true;
        else if (dot3(abc, ao) > T(0)) { d[0] = abc[0]; d[1] = abc[1]; d[2] = abc[2]; }
        else { MPoint<T> tmp = S[0]; S[0] = S[1]; S[1] = tmp; d[0] = -abc[0]; d[1] = -abc[1]; d[2] = -abc[2]; }
      }
      if (star) {
        if (dot3(ab, ao) > T(0)) { S[0] = S[1]; S[1] = S[2]; n = 2; cross3(u, ab, ao); cross3(d, u, ab); }
        else { S[0] = S[2]; n = 1; d[0] = ao[0]; d[1] = ao[1]; d[2] = ao[2]; }
      }
    } else {
      T *a = S[3].w, *b = S[2].w, *c = S[1].w, *e = S[0].w, ab[3], ac[3], ad[3], ao[3] = {-a[0], -a[1], -a[2]}, abc[3], acd[3], adb[3];
      sub3(ab, b, a); sub3(ac, c, a); sub3(ad, e, a);
      cross3(abc, ab, ac); cross3(acd, ac, ad); cross3(adb, ad, ab);
      if (dot3(abc, ad) > T(0)) { abc[0] = -abc[0]; abc[1] = -abc[1]; abc[2] = -abc[2]; }
      if (dot3(acd, ab) > T(0)) { acd[0] = -acd[0]; acd[1] = -acd[1]; acd[2] = -acd[2]; }
      if (dot3(adb, ac) > T(0)) { adb[0] = -adb[0]; adb[1] = -adb[1]; adb[2] = -adb[2]; }
      const T da = dot3(abc, ao), db = dot3(acd, ao), dc = dot3(adb, ao);
      if (da > T(0) && da >= db && da >= dc) { S[0] = S[1]; S[1] = S[2]; S[2] = S[3]; n = 3; d[0] = abc[0]; d[1] = abc[1]; d[2] = abc[2]; }
      else if (db > T(0) && db >= dc) { S[2] = S[3]; n = 3; d[0] = acd[0]; d[1] = acd[1]; d[2] = acd[2]; }
      else if (dc > T(0)) { S[1] = S[2]; S[2] = S[3]; n = 3; d[0] = adb[0]; d[1] = adb[1]; d[2] = adb[2]; }
      else { np = 4; return 1; }
    }
    if (dot3(d, d) < T(1e-30)) { np = n; return 1; }
  }
  np = n;
  return n == 4;
}

// --------------------------------------------------------------------------------------------- EPA polytope access
template <typename T>
__device__ __forceinline__ void epa_getv(const CollideScratch<T> &cs, int i, T *w) { w[0] = cs.Vw[0][i]; w[1] = cs.Vw[1][i]; w[2] = cs.Vw[2][i]; }
// --------------------------------------------------------------------------------------------- support features
template <typename T>
__device__ __forceinline__ void frame_from_normal(const T *n, T *frame) {  // [upstream] mju_makeFrame
  T *x = frame, *y = frame + 3, *z = frame + 6;
  T l = t_sqrt(dot3(n, n));
  for (int c = 0; c < 3; c++) x[c] = n[c] / l;
  y[0] = y[1] = y[2] = T(0);
  if (x[1] < T(0.5) && x[1] > T(-0.5)) y[1] = T(1); else y[2] = T(1);
  const T dd = dot3(x, y);
  for (int c = 0; c < 3; c++) y[c] -= dd * x[c];
  l = t_sqrt(dot3(y, y));
  for (int c = 0; c < 3; c++) y[c] /= l;
  cross3(z, x, y);
}

// ---- manifold helpers mirroring the oracle (same expressions, evaluated once per feature / in parallel over points)
// Height of feature P at (x, y): the oracle's feature_height() split into a per-feature setup (lane 0) ...
template <typename T>
__device__ __noinline__ void feature_plane(const FPt<T> *P, int n, HPlane<T> &hp) {
  hp.mode = 0; hp.x0 = P[0].x; hp.y0 = P[0].y; hp.h0 = P[0].h;
  if (n == 1) return;
  int i1 = 1;
  T best = T(-1);
#pragma unroll 1
  for (int i = 1; i < n; i++) { const T dx = P[i].x - P[0].x, dy = P[i].y - P[0].y, l = dx * dx + dy * dy; if (l > best) { best = l; i1 = i; } }
  const T ex = P[i1].x - P[0].x, ey = P[i1].y - P[0].y, eh = P[i1].h - P[0].h, el = ex * ex + ey * ey;
  hp.ex = ex; hp.ey = ey; hp.eh = eh; hp.el = el;
  if (el < T(1e-20)) return;
  hp.mode = 1;
  if (n == 2) return;
  int i2 = -1;
  best = T(0);
#pragma unroll 1
  for (int i = 1; i < n; i++) { const T a = t_abs(ex * (P[i].y - P[0].y) - ey * (P[i].x - P[0].x)); if (a > best) { best = a; i2 = i; } }
  if (i2 < 0 || best < T(1e-12) * el) return;
  hp.mode = 2;
  hp.fx = P[i2].x - P[0].x; hp.fy = P[i2].y - P[0].y; hp.fh = P[i2].h - P[0].h; hp.det = ex * hp.fy - ey * hp.fx;
}
// ... and a per-point evaluation (any lane)
template <typename T>
__device__ __forceinline__ T plane_height(const HPlane<T> &hp, T x, T y) {
  if (hp.mode == 0) return hp.h0;
  const T px = x - hp.x0, py = y - hp.y0;
  if (hp.mode == 1) { const T t = (px * hp.ex + py * hp.ey) / hp.el; return hp.h0 + t * hp.eh; }
  const T u = (px * hp.fy - py * hp.fx) / hp.det, v = (hp.ex * py - hp.ey * px) / hp.det;
  return hp.h0 + u * hp.eh + v * hp.fh;
}

template <typename T>
__device__ __noinline__ int reduce_manifold(FPt<T> *P, T *dist, int n) {
  if (n <= MAXMANI) return n;
  int sel[4] = {0, -1, -1, -1};
  // tolerant comparisons: the first candidate in polygon order wins a tie in any arithmetic (see the oracle)
  #pragma unroll 1
  for (int i = 1; i < n; i++) if (dist[i] < dist[sel[0]] - T(1e-7)) sel[0] = i;
  T best = T(-1);
  #pragma unroll 1
  for (int i = 0; i < n; i++) { const T dx = P[i].x - P[sel[0]].x, dy = P[i].y - P[sel[0]].y, l = dx * dx + dy * dy; if (l > best * T(1.0001) + T(1e-12)) { best = l; sel[1] = i; } }
  const T ex = P[sel[1]].x - P[sel[0]].x, ey = P[sel[1]].y - P[sel[0]].y;
  T bp = T(0), bn = T(0);
  #pragma unroll 1
  for (int i = 0; i < n; i++) {
    if (i == sel[0] || i == sel[1]) continue;  // their cross product is 0 up to round-off (FMA contraction makes it +-eps)
    const T s = ex * (P[i].y - P[sel[0]].y) - ey * (P[i].x - P[sel[0]].x);
    if (s > bp * T(1.0001) + T(1e-12)) { bp = s; sel[2] = i; }
    if (s < bn * T(1.0001) - T(1e-12)) { bn = s; sel[3] = i; }
  }
  FPt<T> Q[4];
  T qd[4];
  int k = 0;
  for (int i = 0; i < 4; i++) if (sel[i] >= 0) { Q[k] = P[sel[i]]; qd[k] = dist[sel[i]]; k++; }
  #pragma unroll 1
  for (int i = 0; i < k; i++) { P[i] = Q[i]; dist[i] = qd[i]; }
  return k;
}

}  // namespace so101
