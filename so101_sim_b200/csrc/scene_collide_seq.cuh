// Convex narrow phase with ONE THREAD per intersecting pair: EPA -> support-feature clipping manifold.
//
// Same algorithm, tolerances and tie-breaks as the warp-cooperative routines in scene_collide.cuh (and as
// oracle/so101_collide.c); only the mapping differs.  The 32 lanes of a warp work on 32 different pairs that share the
// second geom (the work queues are per geom), so hull vertex loads are warp-wide broadcasts, and the branchy polytope /
// polygon bookkeeping that used to occupy a whole warp per pair now costs one lane.  Per-thread scratch (polytope or
// manifold buffers, ~9 KB in float) lives in local memory, which the hardware interleaves by lane: lanes that touch the
// same array index share cache lines.
#pragma once
#include "scene_collide.cuh"

namespace so101 {

// contacts a pair can emit (manifold <= MAXMANI)
template <typename T>
struct PairContacts {
  int n;
  T pos[MAXMANI][3], normal[3], dist[MAXMANI];
};

template <typename T>
__device__ __forceinline__ void epa_putv_seq(CollideScratch<T> &cs, int i, const MPoint<T> &p) {
#pragma unroll
  for (int c = 0; c < 3; c++) { cs.Vw[c][i] = p.w[c]; cs.Va[c][i] = p.a[c]; cs.Vb[c][i] = p.b[c]; }
}
template <typename T>
__device__ __forceinline__ int epa_add_face_seq(CollideScratch<T> &cs, int &nf, int a, int b, int c, const T *inside) {
  if (nf >= EPA_MAXF) return -1;
  T va[3], vb[3], vc[3], ab[3], ac[3], n[3], t[3];
  epa_getv(cs, a, va); epa_getv(cs, b, vb); epa_getv(cs, c, vc);
  sub3(ab, vb, va); sub3(ac, vc, va);
  cross3(n, ab, ac);
  const T l = t_sqrt(dot3(n, n));
  if (l < T(1e-30)) return -1;
  n[0] /= l; n[1] /= l; n[2] /= l;
  sub3(t, va, inside);
  int v1 = b, v2 = c;
  if (dot3(n, t) < T(0)) { n[0] = -n[0]; n[1] = -n[1]; n[2] = -n[2]; v1 = c; v2 = b; }
  cs.Fv[0][nf] = a; cs.Fv[1][nf] = v1; cs.Fv[2][nf] = v2;
  cs.Fn[0][nf] = n[0]; cs.Fn[1][nf] = n[1]; cs.Fn[2][nf] = n[2];
  cs.Fd[nf] = dot3(n, va);
  cs.Falive[nf] = 1;
  return nf++;
}
// closest face to the origin (first minimum).  Dead faces carry Fd = +inf, so the scan needs one load per face; four faces
// per trip keep four independent loads in flight (the polytope lives in local memory: a serial chain of ~100-cycle loads
// otherwise).
template <typename T>
__device__ __forceinline__ int epa_best_seq(const CollideScratch<T> &cs, int nf) {
  T bd = INFINITY;
  int bi = -1;
#pragma unroll 1
  for (int f0 = 0; f0 < nf; f0 += 4) {
    const T d0 = cs.Fd[f0], d1 = f0 + 1 < nf ? cs.Fd[f0 + 1] : T(INFINITY), d2 = f0 + 2 < nf ? cs.Fd[f0 + 2] : T(INFINITY),
            d3 = f0 + 3 < nf ? cs.Fd[f0 + 3] : T(INFINITY);
    if (d0 < bd) { bd = d0; bi = f0; }
    if (d1 < bd) { bd = d1; bi = f0 + 1; }
    if (d2 < bd) { bd = d2; bi = f0 + 2; }
    if (d3 < bd) { bd = d3; bi = f0 + 3; }
  }
  return bi;
}

// EPA in three parts, so that a caller can interleave the iterations of different pairs (scene_epa_kernel): the state between
// calls is the polytope in cs plus EpaState.  epa_seq() below runs them back to back.
template <typename T>
struct EpaState {
  int nv, nf, it, best;
  T inside[3];
};

// polytope from the GJK simplex (completed to a tetrahedron).  Returns 0 when there is nothing to expand (EPA reports no contact).
template <typename T>
__device__ __forceinline__ int epa_begin(const SceneModel<T> &sm, CollideScratch<T> &cs, Shape<T> &A, Shape<T> &B, const MPoint<T> *S, int n, EpaState<T> &st) {
  int nv = 0;
  st.nf = 0; st.it = 0; st.best = -1;
  if (n == 1) return 0;
#pragma unroll 1
  for (int i = 0; i < n; i++) epa_putv_seq(cs, nv++, S[i]);
  if (nv == 2) {
    T v0[3], v1[3], ab[3], ax[3] = {T(0), T(0), T(0)}, d[3];
    epa_getv(cs, 0, v0); epa_getv(cs, 1, v1);
    sub3(ab, v1, v0);
    const int k = t_abs(ab[0]) < t_abs(ab[1]) ? (t_abs(ab[0]) < t_abs(ab[2]) ? 0 : 2) : (t_abs(ab[1]) < t_abs(ab[2]) ? 1 : 2);
    ax[k] = T(1); cross3(d, ab, ax);
    MPoint<T> p;
    msupport_seq(sm, A, B, d, p);
    T t[3], cr[3];
    sub3(t, p.w, v0); cross3(cr, ab, t);
    if (dot3(cr, cr) < T(1e-24)) { d[0] = -d[0]; d[1] = -d[1]; d[2] = -d[2]; msupport_seq(sm, A, B, d, p); }
    epa_putv_seq(cs, nv++, p);
  }
  if (nv == 3) {
    T v0[3], v1[3], v2[3], ab[3], ac[3], nn[3], t[3];
    epa_getv(cs, 0, v0); epa_getv(cs, 1, v1); epa_getv(cs, 2, v2);
    sub3(ab, v1, v0); sub3(ac, v2, v0); cross3(nn, ab, ac);
    if (dot3(nn, nn) < T(1e-30)) return 0;
    MPoint<T> p;
    msupport_seq(sm, A, B, nn, p);
    sub3(t, p.w, v0);
    if (t_abs(dot3(t, nn)) < T(1e-12) * t_sqrt(dot3(nn, nn))) {
      const T m[3] = {-nn[0], -nn[1], -nn[2]};
      msupport_seq(sm, A, B, m, p);
      sub3(t, p.w, v0);
      if (t_abs(dot3(t, nn)) < T(1e-12) * t_sqrt(dot3(nn, nn))) return 0;
    }
    epa_putv_seq(cs, nv++, p);
  }
  st.nv = nv;
  st.inside[0] = st.inside[1] = st.inside[2] = T(0);
  for (int i = 0; i < 4; i++) { T v[3]; epa_getv(cs, i, v); for (int k = 0; k < 3; k++) st.inside[k] += T(0.25) * v[k]; }
  if (epa_add_face_seq(cs, st.nf, 0, 1, 2, st.inside) < 0 || epa_add_face_seq(cs, st.nf, 0, 1, 3, st.inside) < 0 ||
      epa_add_face_seq(cs, st.nf, 0, 2, 3, st.inside) < 0 || epa_add_face_seq(cs, st.nf, 1, 2, 3, st.inside) < 0) return 0;
  return 1;
}

// one expansion.  Returns 0 = call again, 1 = finished (epa_end reads the result), -1 = no face left (EPA reports no contact).
template <typename T>
__device__ __forceinline__ int epa_step(const SceneModel<T> &sm, CollideScratch<T> &cs, Shape<T> &A, Shape<T> &B, EpaState<T> &st) {
  if (st.it >= EPA_MAXIT) return 1;
  const int nf0 = st.nf;
  const int best = epa_best_seq(cs, nf0);
  st.best = best;
  if (best < 0) return -1;
  if (st.nv >= EPA_MAXV) return 1;
  st.it++;
  const T bn[3] = {cs.Fn[0][best], cs.Fn[1][best], cs.Fn[2][best]}, bd = cs.Fd[best];
  MPoint<T> p;
  msupport_seq(sm, A, B, bn, p);
  const T adv = dot3(p.w, bn) - bd;
  if (adv < T(sizeof(T) == 8 ? 1e-9 : 1e-6)) return 1;
  const int nv = st.nv;
  epa_putv_seq(cs, nv, p);
  // visibility (p above the face plane: n . p - d > eps; dead faces have d = +inf), four faces per trip, then the horizon
  // edits of the visible ones in face order (same order as the oracle)
  int nh = 0;
  const T veps = T(sizeof(T) == 8 ? 1e-12 : 1e-9);
#pragma unroll 1
  for (int f0 = 0; f0 < nf0; f0 += 4) {
    unsigned vis = 0;
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const int f = f0 + u < nf0 ? f0 + u : f0;
      const T sdist = (cs.Fn[0][f] * p.w[0] + cs.Fn[1][f] * p.w[1] + cs.Fn[2][f] * p.w[2]) - cs.Fd[f];
      if (f0 + u < nf0 && sdist > veps) vis |= 1u << u;
    }
#pragma unroll 1
    while (vis) {
      const int f = f0 + __ffs(vis) - 1;
      vis &= vis - 1;
      cs.Falive[f] = 0; cs.Fd[f] = INFINITY;
      const int fv[3] = {cs.Fv[0][f], cs.Fv[1][f], cs.Fv[2][f]};
      for (int e = 0; e < 3; e++) {
        const int a = fv[e], b = fv[(e + 1) % 3];
        // an edge whose reverse is already listed cancels it (the last entry takes its slot), otherwise it is appended.  A directed
        // edge is listed at most once, so the search can look at four entries per trip (independent local-memory loads).
        const unsigned rev = (unsigned)b | ((unsigned)a << 8);
        int at = -1;
#pragma unroll 1
        for (int h0 = 0; h0 < nh && at < 0; h0 += 4) {
          const unsigned e0 = cs.horizon[h0], e1 = h0 + 1 < nh ? cs.horizon[h0 + 1] : 0xffffu, e2 = h0 + 2 < nh ? cs.horizon[h0 + 2] : 0xffffu,
                         e3 = h0 + 3 < nh ? cs.horizon[h0 + 3] : 0xffffu;
          at = e0 == rev ? h0 : (e1 == rev ? h0 + 1 : (e2 == rev ? h0 + 2 : (e3 == rev ? h0 + 3 : -1)));
        }
        if (at >= 0) { cs.horizon[at] = cs.horizon[nh - 1]; nh--; }
        else if (nh < EPA_MAXF) { cs.horizon[nh] = (unsigned short)((unsigned)a | ((unsigned)b << 8)); nh++; }
      }
    }
  }
  if (nh == 0) return 1;
  int failed = 0;
#pragma unroll 1
  for (int h = 0; h < nh; h++)
    if (epa_add_face_seq(cs, st.nf, (int)(cs.horizon[h] & 0xff), (int)(cs.horizon[h] >> 8), nv, st.inside) < 0) failed = 1;
  st.nv = nv + 1;
  return failed;
}

// penetration normal / depth and witness points from the face closest to the origin.  Returns 0 when no face is left.
template <typename T>
__device__ __forceinline__ int epa_end(CollideScratch<T> &cs, const EpaState<T> &st, T *normal, T &depth, T *pa, T *pb) {
  int best = st.best;
  if (best < 0 || !cs.Falive[best]) {
    best = epa_best_seq(cs, st.nf);
    if (best < 0) return 0;
  }
  const T fn[3] = {cs.Fn[0][best], cs.Fn[1][best], cs.Fn[2][best]}, fd = cs.Fd[best];
  normal[0] = fn[0]; normal[1] = fn[1]; normal[2] = fn[2];
  depth = fd > T(0) ? fd : T(0);
  const T p[3] = {fn[0] * fd, fn[1] * fd, fn[2] * fd};
  const int i0 = cs.Fv[0][best], i1 = cs.Fv[1][best], i2 = cs.Fv[2][best];
  T a[3], b[3], c[3], v0[3], v1[3], v2[3];
  epa_getv(cs, i0, a); epa_getv(cs, i1, b); epa_getv(cs, i2, c);
  sub3(v0, b, a); sub3(v1, c, a); sub3(v2, p, a);
  const T d00 = dot3(v0, v0), d01 = dot3(v0, v1), d11 = dot3(v1, v1), d20 = dot3(v2, v0), d21 = dot3(v2, v1), den = d00 * d11 - d01 * d01;
  T bv = T(1.0 / 3), bw = T(1.0 / 3);
  if (t_abs(den) > T(1e-30)) { bv = (d11 * d20 - d01 * d21) / den; bw = (d00 * d21 - d01 * d20) / den; }
  const T bu = T(1) - bv - bw;
  for (int k = 0; k < 3; k++) {
    pa[k] = bu * cs.Va[k][i0] + bv * cs.Va[k][i1] + bw * cs.Va[k][i2];
    pb[k] = bu * cs.Vb[k][i0] + bv * cs.Vb[k][i1] + bw * cs.Vb[k][i2];
  }
  return 1;
}

template <typename T>
__device__ __noinline__ int epa_seq(const SceneModel<T> &sm, CollideScratch<T> &cs, Shape<T> &A, Shape<T> &B, const MPoint<T> *S, int n, T *normal,
                                    T &depth, T *pa, T *pb) {
  EpaState<T> st;
  if (!epa_begin(sm, cs, A, B, S, n, st)) return 0;
  int r;
#pragma unroll 1
  do { r = epa_step(sm, cs, A, B, st); } while (r == 0);
  if (r < 0) return 0;
  return epa_end(cs, st, normal, depth, pa, pb);
}

// vertices of s within delta of the support plane along dir -> CCW 2-D convex polygon in (t1,t2) with heights
constexpr int SCANW = 8;  // hull vertices examined per trip of the slab scan
template <typename T>
__device__ __noinline__ int feature_seq(const SceneModel<T> &sm, CollideScratch<T> &cs, Shape<T> &s, const T *dir, const T *t1, const T *t2, T delta,
                                        FPt<T> *out) {
  T sp[3];
  support_seq(sm, s, dir, sp);
  const T hmax = dot3(sp, dir);
  int nc = 0;
  T w[3];
  bool projected = false;
  FPt<T> *sorted = cs.bufA;  // nc <= MAXCAND <= size of bufA
  if (s.type == G_HULL) {
    // tangent-plane coordinates are evaluated in the hull frame: x = v . (R^T t1) + pos . t1  (as the oracle does)
    T dl[3], t1l[3], t2l[3];
    mulmtv(dl, s.mat, dir); mulmtv(t1l, s.mat, t1); mulmtv(t2l, s.mat, t2);
    const T off = dot3(s.pos, dir), ox = dot3(s.pos, t1), oy = dot3(s.pos, t2);
    const Vec4<T> *vt = sm.hull_vert + s.vadr;
    // pass 1: count the slab and track its extreme vertices along 16 tangent-plane directions (8 axes, min and max), all in
    // registers.  A slab with more than FEAT_EXACT vertices (rims, finely tessellated patches) is represented by those
    // extremes - an inscribed convex polygon, counter-clockwise from -x - with no candidate storage, sort or hull pass.
    T emax[8], emin[8];
    int imax[8], imin[8], nband = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) { emax[k] = -INFINITY; emin[k] = INFINITY; imax[k] = imin[k] = 0; }
    const T thr = hmax - delta;
    // one in-slab vertex: count it and keep the first FEAT_EXACT (a small slab - the usual case - then needs no second pass and
    // no extremes at all).  The extremes start with vertex FEAT_EXACT + 1: the stored ones are folded in first, in the same
    // (index) order, so the result is what updating them for every vertex would give.
    auto extremes = [&](int i, T x, T y) {
#pragma unroll
      for (int k = 0; k < 8; k++) {
        const T val = feat_cos<T>(k) * x + feat_sin<T>(k) * y;
        if (val > emax[k]) { emax[k] = val; imax[k] = i; }
        if (val < emin[k]) { emin[k] = val; imin[k] = i; }
      }
    };
    auto take = [&](int i, const Vec4<T> &v) {
      const T x = (v.x * t1l[0] + v.y * t1l[1] + v.z * t1l[2]) + ox, y = (v.x * t2l[0] + v.y * t2l[1] + v.z * t2l[2]) + oy;
      if (nband < FEAT_EXACT) {
        cs.cand[0][nband] = x; cs.cand[1][nband] = y; cs.cand[2][nband] = (v.x * dl[0] + v.y * dl[1] + v.z * dl[2]) + off;
        cs.candi[nband] = i;
      } else {
        if (nband == FEAT_EXACT) {
#pragma unroll 1
          for (int j = 0; j < FEAT_EXACT; j++) extremes(cs.candi[j], cs.cand[0][j], cs.cand[1][j]);
        }
        extremes(i, x, y);
      }
      nband++;
    };
    // Full scan, SCANW heights per trip (independent loads: the vertex loads come from L2 while the L1 is busy with the per-thread
    // scratch, so the number of round trips is what counts); the few in-slab vertices are then handled one by one in index order.
    // (A flood fill of the slab over the vertex graph from the support vertex touches far fewer vertices of the banana's 1000-
    // vertex hulls but measured 1.6x SLOWER for the kernel: its visited-bit updates and frontier are a serial chain of local-
    // memory round trips, while this scan streams with all lanes busy.)
#pragma unroll 1
    for (int i0 = 0; i0 < s.vnum; i0 += SCANW) {
      const int rem = s.vnum - i0;
      T hgt[SCANW];
#pragma unroll
      for (int u = 0; u < SCANW; u++) {  // (out-of-range slots re-read the chunk's first vertex and are masked below)
        const Vec4<T> v = vt[i0 + (u < rem ? u : 0)];
        hgt[u] = (v.x * dl[0] + v.y * dl[1] + v.z * dl[2]) + off;
      }
      unsigned hit = 0;
#pragma unroll
      for (int u = 0; u < SCANW; u++) hit |= (u < rem && hgt[u] >= thr) ? (1u << u) : 0u;
#pragma unroll 1
      while (hit) {
        const int i = i0 + __ffs(hit) - 1;
        hit &= hit - 1;
        take(i, vt[i]);
      }
    }
    if (nband > FEAT_EXACT) {
      int kept[16], nk = 0;
#pragma unroll
      for (int j = 0; j < 16; j++) {
        const int idx = j < 8 ? imin[j] : imax[j - 8];
        bool dup = false;
#pragma unroll
        for (int q = 0; q < j; q++) dup = dup || (q < nk && kept[q] == idx);
        if (!dup) {
          // kept[] is indexed statically so that it stays in registers: slot nk is found by unrolled selection
#pragma unroll
          for (int q = 0; q < 16; q++) if (q == nk) kept[q] = idx;
          const Vec4<T> v = vt[idx];
          out[nk].x = (v.x * t1l[0] + v.y * t1l[1] + v.z * t1l[2]) + ox;
          out[nk].y = (v.x * t2l[0] + v.y * t2l[1] + v.z * t2l[2]) + oy;
          out[nk].h = (v.x * dl[0] + v.y * dl[1] + v.z * dl[2]) + off;
          nk++;
        }
      }
      return nk;
    }
    nc = nband;  // small slab: the candidates themselves (stored by the scan, in vertex order)
    projected = nc > 0;
  } else if (s.type == G_BOX) {
#pragma unroll 1
    for (int i = 0; i < 8; i++) {
      const T l[3] = {(i & 1 ? T(1) : T(-1)) * s.size[0], (i & 2 ? T(1) : T(-1)) * s.size[1], (i & 4 ? T(1) : T(-1)) * s.size[2]};
      local2world(s, l, w);
      if (dot3(w, dir) >= hmax - delta) { cs.cand[0][nc] = w[0]; cs.cand[1][nc] = w[1]; cs.cand[2][nc] = w[2]; nc++; }
    }
  } else if (s.type == G_CYLINDER) {
#pragma unroll 1
    for (int cap = -1; cap <= 1; cap += 2)
#pragma unroll 1
      for (int i = 0; i < 16; i++) {
        T sn, cn;
        t_sincos(T(2 * 3.14159265358979323846 / 16) * T(i), &sn, &cn);
        const T l[3] = {s.size[0] * cn, s.size[0] * sn, T(cap) * s.size[1]};
        local2world(s, l, w);
        if (dot3(w, dir) >= hmax - delta) { cs.cand[0][nc] = w[0]; cs.cand[1][nc] = w[1]; cs.cand[2][nc] = w[2]; nc++; }
      }
  } else if (s.type == G_CAPSULE) {
#pragma unroll 1
    for (int e = -1; e <= 1; e += 2) {
      const T l[3] = {T(0), T(0), T(e) * s.size[1]};
      local2world(s, l, w);
      for (int c = 0; c < 3; c++) w[c] += s.size[0] * dir[c];
      if (dot3(w, dir) >= hmax - delta) { cs.cand[0][nc] = w[0]; cs.cand[1][nc] = w[1]; cs.cand[2][nc] = w[2]; nc++; }
    }
  }
  if (nc == 0) { cs.cand[0][0] = sp[0]; cs.cand[1][0] = sp[1]; cs.cand[2][0] = sp[2]; nc = 1; }
  // project, then stable insertion sort by (x, y) [ties keep candidate order] into bufA
#pragma unroll 1
  for (int i = 0; i < nc; i++) {
    const T cw[3] = {cs.cand[0][i], cs.cand[1][i], cs.cand[2][i]};
    const FPt<T> p = projected ? FPt<T>{cw[0], cw[1], cw[2]} : FPt<T>{dot3(cw, t1), dot3(cw, t2), dot3(cw, dir)};
    int j = i;
    while (j > 0 && (p.x < sorted[j - 1].x || (p.x == sorted[j - 1].x && p.y < sorted[j - 1].y))) { sorted[j] = sorted[j - 1]; j--; }
    sorted[j] = p;
  }
  if (nc <= 2) { for (int i = 0; i < nc; i++) out[i] = sorted[i]; return nc; }
  FPt<T> *H = cs.Hh;
  int k = 0;
#pragma unroll 1
  for (int i = 0; i < nc; i++) {
    while (k >= 2 && (H[k - 1].x - H[k - 2].x) * (sorted[i].y - H[k - 2].y) - (H[k - 1].y - H[k - 2].y) * (sorted[i].x - H[k - 2].x) <= T(1e-14)) k--;
    H[k++] = sorted[i];
  }
#pragma unroll 1
  for (int i = nc - 2, t = k + 1; i >= 0; i--) {
    while (k >= t && (H[k - 1].x - H[k - 2].x) * (sorted[i].y - H[k - 2].y) - (H[k - 1].y - H[k - 2].y) * (sorted[i].x - H[k - 2].x) <= T(1e-14)) k--;
    H[k++] = sorted[i];
  }
  k--;
  if (k > MAXFEAT) k = MAXFEAT;
#pragma unroll 1
  for (int i = 0; i < k; i++) out[i] = H[i];
  return k;
}

template <typename T>
__device__ __forceinline__ int clip_poly_seq(CollideScratch<T> &cs, const FPt<T> *subj, int n, const FPt<T> *clip, int m, FPt<T> *out) {
  constexpr int CAP = 2 * MAXFEAT + 8;
  int na = n;
  FPt<T> *in = cs.bufA, *res = cs.bufB;
#pragma unroll 1
  for (int i = 0; i < n; i++) in[i] = subj[i];
#pragma unroll 1
  for (int e = 0; e < m && na > 0; e++) {
    const T ax = clip[e].x, ay = clip[e].y, bx = clip[(e + 1) % m].x, by = clip[(e + 1) % m].y;
    const T ex = bx - ax, ey = by - ay, tol = T(1e-12);
    int nr = 0;
    if (na == 2) {
      const FPt<T> P = in[0], Q = in[1];
      const T sp = ex * (P.y - ay) - ey * (P.x - ax), sq = ex * (Q.y - ay) - ey * (Q.x - ax);
      const bool pin = sp >= -tol, qin = sq >= -tol;
      if (pin && qin) { res[nr++] = P; res[nr++] = Q; }
      else if (pin || qin) {
        const T t = sp / (sp - sq);
        const FPt<T> I = {P.x + t * (Q.x - P.x), P.y + t * (Q.y - P.y), P.h + t * (Q.h - P.h)};
        if (pin) { res[nr++] = P; res[nr++] = I; } else { res[nr++] = I; res[nr++] = Q; }
      }
    } else {
#pragma unroll 1
      for (int i = 0; i < na; i++) {
        const FPt<T> P = in[i], Q = in[(i + 1) % na];
        const T sp = ex * (P.y - ay) - ey * (P.x - ax), sq = ex * (Q.y - ay) - ey * (Q.x - ax);
        const bool pin = sp >= -tol, qin = sq >= -tol;
        if (pin && nr < CAP) res[nr++] = P;
        if (na > 1 && pin != qin && nr < CAP) {
          const T t = sp / (sp - sq);
          res[nr++] = FPt<T>{P.x + t * (Q.x - P.x), P.y + t * (Q.y - P.y), P.h + t * (Q.h - P.h)};
        }
        if (na == 1) break;
      }
    }
    FPt<T> *tmp = in; in = res; res = tmp;
    na = nr;
    if (na > 2 * MAXFEAT) na = 2 * MAXFEAT;
  }
#pragma unroll 1
  for (int i = 0; i < na; i++) out[i] = in[i];
  return na;
}

template <typename T>
__device__ __forceinline__ void emit_seq(PairContacts<T> &pc, const T *pos, T dist) {
  if (pc.n >= MAXMANI) return;  // reduce_manifold keeps <= MAXMANI points
  const int c = pc.n++;
  pc.dist[c] = dist;
  pc.pos[c][0] = pos[0]; pc.pos[c][1] = pos[1]; pc.pos[c][2] = pos[2];
}

// manifold from the two supporting features along normal n (A -> B).  Returns the number of contacts emitted.
template <typename T>
__device__ __noinline__ int manifold_seq(const SceneModel<T> &sm, CollideScratch<T> &cs, Shape<T> &A, Shape<T> &B, const T *n, T depth,
                                         PairContacts<T> &pc) {
  T frame[9];
  frame_from_normal(n, frame);
  const T *t1 = frame + 3, *t2 = frame + 6;
  const T nn[3] = {-frame[0], -frame[1], -frame[2]};
  const T delta = depth + T(1e-7);
  const int na = feature_seq(sm, cs, A, frame, t1, t2, delta, cs.FA);
  const int nb = feature_seq(sm, cs, B, nn, t1, t2, delta, cs.FB);
  for (int i = 0; i < nb; i++) cs.FB[i].h = -cs.FB[i].h;  // heights of B's feature were measured along -n
  int nr = 0;
  {  // subject = the smaller feature when the other one is a polygon
    const bool a_subj = (na >= 3 && nb >= 3) || (nb >= 3 && na <= 2), b_subj = na >= 3 && (nb == 2 || nb == 1);
    if (a_subj) nr = clip_poly_seq(cs, cs.FA, na, cs.FB, nb, cs.R);
    else if (b_subj) nr = clip_poly_seq(cs, cs.FB, nb, cs.FA, na, cs.R);
  }
  feature_plane(cs.FA, na, cs.hp[0]); feature_plane(cs.FB, nb, cs.hp[1]);
  int k = 0;
#pragma unroll 1
  for (int i = 0; i < nr; i++) {
    const T ha = plane_height(cs.hp[0], cs.R[i].x, cs.R[i].y), hb = plane_height(cs.hp[1], cs.R[i].x, cs.R[i].y);
    const T di = hb - ha;
    if (di < T(0)) { cs.R[k] = cs.R[i]; cs.R[k].h = T(0.5) * (ha + hb); cs.mdist[k] = di; k++; }
  }
  int u = 0;
#pragma unroll 1
  for (int i = 0; i < k; i++) {
    int dup = 0;
    for (int j = 0; j < u; j++)
      if (t_abs(cs.R[i].x - cs.R[j].x) + t_abs(cs.R[i].y - cs.R[j].y) < T(1e-7)) {
        dup = 1;
        if (cs.mdist[i] < cs.mdist[j]) { cs.R[j] = cs.R[i]; cs.mdist[j] = cs.mdist[i]; }
        break;
      }
    if (!dup) { cs.R[u] = cs.R[i]; cs.mdist[u] = cs.mdist[i]; u++; }
  }
  u = reduce_manifold(cs.R, cs.mdist, u);
  pc.normal[0] = frame[0]; pc.normal[1] = frame[1]; pc.normal[2] = frame[2];
  for (int i = 0; i < u; i++) {
    T pos[3];
    for (int c = 0; c < 3; c++) pos[c] = cs.R[i].x * t1[c] + cs.R[i].y * t2[c] + cs.R[i].h * frame[c];
    emit_seq(pc, pos, cs.mdist[i]);
  }
  return u;
}

// contacts of a pair whose EPA has finished: the multi-point manifold, or the single EPA point when the features give none
template <typename T>
__device__ __forceinline__ void finish_convex_pair(const SceneModel<T> &sm, CollideScratch<T> &cs, Shape<T> &A, Shape<T> &B, int ok, const T *normal,
                                                   T depth, const T *pa, const T *pb, PairContacts<T> &pc) {
  if (!ok) return;
  if (!(depth > T(0))) return;
  if (manifold_seq(sm, cs, A, B, normal, depth, pc) > 0) return;
  T frame[9], pos[3];
  frame_from_normal(normal, frame);
  for (int c = 0; c < 3; c++) pos[c] = T(0.5) * (pa[c] + pb[c]);
  pc.normal[0] = frame[0]; pc.normal[1] = frame[1]; pc.normal[2] = frame[2];
  emit_seq(pc, pos, -depth);
}

template <typename T>
__device__ __noinline__ void collide_convex_seq(const SceneModel<T> &sm, CollideScratch<T> &cs, Shape<T> &A, Shape<T> &B, const MPoint<T> *S, int n,
                                                PairContacts<T> &pc) {
  T normal[3], depth, pa[3], pb[3];
  const int ok = epa_seq(sm, cs, A, B, S, n, normal, depth, pa, pb);
  finish_convex_pair(sm, cs, A, B, ok, normal, depth, pa, pb, pc);
}

template <typename T>
__device__ __noinline__ void collide_plane_seq(const SceneModel<T> &sm, CollideScratch<T> &cs, const Shape<T> &P, Shape<T> &B, PairContacts<T> &pc) {
  const T n[3] = {P.mat[2], P.mat[5], P.mat[8]}, nn[3] = {-n[0], -n[1], -n[2]};
  T sp[3];
  support_seq(sm, B, nn, sp);
  const T off = dot3(n, P.pos), depth = off - dot3(sp, n);
  if (!(depth > T(0))) return;
  T frame[9];
  frame_from_normal(n, frame);
  const T *t1 = frame + 3, *t2 = frame + 6;
  int nb = feature_seq(sm, cs, B, nn, t1, t2, depth + T(1e-7), cs.FB);
  for (int i = 0; i < nb; i++) { cs.FB[i].h = -cs.FB[i].h; cs.mdist[i] = cs.FB[i].h - off; }
  nb = reduce_manifold(cs.FB, cs.mdist, nb);
  pc.normal[0] = frame[0]; pc.normal[1] = frame[1]; pc.normal[2] = frame[2];
  for (int i = 0; i < nb; i++) {
    if (cs.mdist[i] >= T(0)) continue;
    T pos[3];
    for (int c = 0; c < 3; c++) pos[c] = cs.FB[i].x * t1[c] + cs.FB[i].y * t2[c] + (cs.FB[i].h - T(0.5) * cs.mdist[i]) * frame[c];
    emit_seq(pc, pos, cs.mdist[i]);
  }
}

}  // namespace so101
