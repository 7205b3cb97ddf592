// ag_device.cuh — per-lane bodies of the sm_100a kernels (one env per lane, lock-step).
//
// Every function here is `__host__ __device__`: the CUDA build wraps them in __global__ kernels
// (agphys.cu); tests/kernel_harness compiles the same bodies for the host to check kernel logic
// against the CPU oracle on a box without a GPU.  The harness is a test aid — the package only
// ever loads the CUDA library.
//
// Reference call sites this path replaces: p.stepSimulation (envs/env.py:226, feeding.py:179) and the
// read-back calls in envs/agents/agent.py:40,52,72,108,124.  The algorithms restate what Bullet does
// for that call (SURVEY.md Appendix A): collision detection at the current pose, Featherstone ABA
// for the unconstrained velocity update, velocity-level PGS over joint limits, joint motors, fixed
// constraints and frictional contacts, symplectic Euler.
#pragma once
#include <string.h>
#include "ag_math.cuh"
#include "ag_types.h"

// ------------------------------------------------------------------ SoA accessors
AG_HD float ld1(const float* p, int item, int N, int e) { return p[(size_t)item * N + e]; }
AG_HD void st1(float* p, int item, int N, int e, float v) { p[(size_t)item * N + e] = v; }
AG_HD f3 ld3(const float* p, int item, int N, int e) {
  size_t b = (size_t)item * 3 * N + e;
  return f3(p[b], p[b + N], p[b + 2 * (size_t)N]);
}
AG_HD void st3(float* p, int item, int N, int e, f3 v) {
  size_t b = (size_t)item * 3 * N + e;
  p[b] = v.x; p[b + N] = v.y; p[b + 2 * (size_t)N] = v.z;
}
AG_HD q4 ld4(const float* p, int item, int N, int e) {
  size_t b = (size_t)item * 4 * N + e;
  return q4(p[b], p[b + N], p[b + 2 * (size_t)N], p[b + 3 * (size_t)N]);
}
AG_HD void st4(float* p, int item, int N, int e, q4 v) {
  size_t b = (size_t)item * 4 * N + e;
  p[b] = v.x; p[b + N] = v.y; p[b + 2 * (size_t)N] = v.z; p[b + 3 * (size_t)N] = v.w;
}
AG_HD f3 tv3(const float* p, int i) { return f3(AG_LDG(p + 3 * i), AG_LDG(p + 3 * i + 1), AG_LDG(p + 3 * i + 2)); }
AG_HD q4 tv4(const float* p, int i) { return q4(AG_LDG(p + 4 * i), AG_LDG(p + 4 * i + 1), AG_LDG(p + 4 * i + 2), AG_LDG(p + 4 * i + 3)); }
AG_HD float cf_ld(const float* d, int slot, int f, int N, int e) { return d[((size_t)slot * AG_CF + f) * N + e]; }
AG_HD void cf_st(float* d, int slot, int f, int N, int e, float v) { d[((size_t)slot * AG_CF + f) * N + e] = v; }

// ------------------------------------------------------------------ the fused env steps' shared action handling
// AssistiveEnv.take_step (env.py:187-217): counts the env step, keeps the raw action ([7][N], for the action penalty) and drives
// the robot's 7 arm joints to PD targets: the clipped, scaled action accumulated frame_skip times onto the joint angle, with
// the limit clamp of every accumulation.  `actions` is the step's [N][7] env-major input.
AG_HD void take_step(int e, const SimDev& S, const float* actions, int* iteration, float* action, const int* arm_links,
                     const float* arm_lower, const float* arm_upper, float action_multiplier, int frame_skip) {
  const int N = S.N;
  const float* act = actions + (size_t)e * 7;
  iteration[e] += 1;
  for (int j = 0; j < 7; j++) {
    float raw = act[j];
    action[(size_t)j * N + e] = raw;
    float a = clampf(raw, -1.f, 1.f) * action_multiplier;
    int k = arm_links[j];
    float q = ld1(S.jq, k, N, e);
    float lo = arm_lower[j], hi = arm_upper[j];
    for (int s = 0; s < frame_skip; s++) {
      if (q + a < lo) { a = 0.f; q = lo; }
      if (q + a > hi) { a = 0.f; q = hi; }
      q += a;
    }
    st1(S.motor_target, k, N, e, q);
  }
}
// tremor (env.py:212-215): the person's `nj` joints are driven to rest +- amplitude ([nj][N]), the sign flips every env step
AG_HD void tremor_step(int e, const SimDev& S, int nj, const int* joints, int iteration, const float* rest, const float* amp) {
  const int N = S.N;
  float sgn = (iteration % 2 == 0) ? 1.f : -1.f;
  for (int j = 0; j < nj; j++) st1(S.motor_target, joints[j], N, e, rest[(size_t)j * N + e] + sgn * amp[(size_t)j * N + e]);
}

// plane k of collider (local) -> (n, d)
AG_HD void ld_plane(const float* planes, int k, f3& n, float& d) {
  n = f3(AG_LDG(planes + 4 * k), AG_LDG(planes + 4 * k + 1), AG_LDG(planes + 4 * k + 2)); d = AG_LDG(planes + 4 * k + 3);
}

// ------------------------------------------------------------------ K1: forward kinematics
// thread = (body, env), env fastest.  p.i0 != 0: all bodies (reset / after teleports); else only movable bodies.
AG_HDN inline void fk_body(int tid, const SimDev& S, const KP& p) {
  const int N = S.N;
  const int e = tid % N, b = tid / N;
  if (!p.i0 && (AG_LDG(S.body_kind + b) == BK_STATIC || S.body_mode[(size_t)b * N + e] != 1)) return;   // off / frozen bodies keep their poses
  int l0 = AG_LDG(S.body_link0 + b), nlk = AG_LDG(S.body_nlinks + b);
  f3 bp = ld3(S.base_pos, b, N, e);
  q4 bq = ld4(S.base_quat, b, N, e);
  st3(S.lpos, l0, N, e, bp); st4(S.lquat, l0, N, e, bq);
  for (int k = l0 + 1; k < l0 + nlk; k++) {
    int par = AG_LDG(S.link_parent + k);
    f3 pp = ld3(S.lpos, par, N, e);
    q4 pq = ld4(S.lquat, par, N, e);
    f3 jp = pp + qrot(pq, tv3(S.link_jpos, k));
    q4 jq = qmul(pq, tv4(S.link_jquat, k));
    int jt = AG_LDG(S.link_jtype + k);
    if (jt == 1) jq = qmul(jq, qaxis(tv3(S.link_axis, k), ld1(S.jq, k, N, e)));
    else if (jt == 2) jp = jp + qrot(jq, tv3(S.link_axis, k) * ld1(S.jq, k, N, e));
    st3(S.lpos, k, N, e, jp); st4(S.lquat, k, N, e, qnormalize(jq));
  }
}

// ------------------------------------------------------------------ K2a: collider AABBs
// thread = (collider list index i, env e), env fastest.  p.p0 = list, p.i0 = list length.
AG_HDN inline void aabb_body(int tid, const SimDev& S, const KP& p) {
  const int N = S.N;
  int e = tid % N, i = tid / N;
  int c = AG_LDG((const int*)p.p0 + i);
  int k = AG_LDG(S.col_link + c);
  if (AG_LDG(S.col_type + c) == 3) {   // half-space: unbounded, except along an axis-aligned normal
    f3 n; float d; ld_plane(S.planes, AG_LDG(S.col_p0 + c), n, d);
    q4 q = ld4(S.lquat, k, N, e);
    f3 nw = qrot(q, n);
    float dw = d + dot(nw, ld3(S.lpos, k, N, e));
    f3 mn(-1e30f, -1e30f, -1e30f), mx(1e30f, 1e30f, 1e30f);
    if (nw.x > 0.999999f) mx.x = dw; else if (nw.x < -0.999999f) mn.x = -dw;
    if (nw.y > 0.999999f) mx.y = dw; else if (nw.y < -0.999999f) mn.y = -dw;
    if (nw.z > 0.999999f) mx.z = dw; else if (nw.z < -0.999999f) mn.z = -dw;
    st3(S.cmin, c, N, e, mn); st3(S.cmax, c, N, e, mx);
    return;
  }
  f3 lp = ld3(S.lpos, k, N, e);
  m3 R = qmat(ld4(S.lquat, k, N, e));
  f3 ctr = lp + mul(R, tv3(S.col_center, c));
  f3 h = tv3(S.col_half, c);
  float r = AG_LDG(S.col_radius + c);
  f3 hw(fabsf(R.m[0]) * h.x + fabsf(R.m[1]) * h.y + fabsf(R.m[2]) * h.z + r,
        fabsf(R.m[3]) * h.x + fabsf(R.m[4]) * h.y + fabsf(R.m[5]) * h.z + r,
        fabsf(R.m[6]) * h.x + fabsf(R.m[7]) * h.y + fabsf(R.m[8]) * h.z + r);
  st3(S.cmin, c, N, e, ctr - hw); st3(S.cmax, c, N, e, ctr + hw);
}
// K2b: link AABBs = union over the link's colliders.  thread = (link list index, env).
AG_HDN inline void linkaabb_body(int tid, const SimDev& S, const KP& p) {
  const int N = S.N;
  int e = tid % N, i = tid / N;
  int k = AG_LDG((const int*)p.p0 + i);
  int c0 = AG_LDG(S.link_col0 + k), ncl = AG_LDG(S.link_ncol + k);
  f3 mn(1e30f, 1e30f, 1e30f), mx(-1e30f, -1e30f, -1e30f);
  for (int c = c0; c < c0 + ncl; c++) { mn = fmin3(mn, ld3(S.cmin, c, N, e)); mx = fmax3(mx, ld3(S.cmax, c, N, e)); }
  st3(S.lmin, k, N, e, mn); st3(S.lmax, k, N, e, mx);
}

// ------------------------------------------------------------------ K3: narrowphase
AG_HD bool aabb_ov(f3 amin, f3 amax, f3 bmin, f3 bmax, float m) {
  return !(amin.x > bmax.x + m || bmin.x > amax.x + m || amin.y > bmax.y + m || bmin.y > amax.y + m ||
           amin.z > bmax.z + m || bmin.z > amax.z + m);
}

// closest point on segment / triangle to the origin (barycentric), Ericson RTCD 5.1 — in fp64:
// the simplex vertices are differences of support points that can be ~1 m apart while the origin is
// ~1 mm from the simplex; in fp32 the Voronoi-region determinants lose all significance on such thin
// simplices (measured on B200: 9 % of link-vs-table-edge queries off by up to 2 mm).
AG_HD void seg_origin(d3 a, d3 b, double& u, double& v) {
  d3 ab = b - a;
  double t = -dot(a, ab), den = dot(ab, ab);
  if (t <= 0.0 || den <= 0.0) { u = 1.0; v = 0.0; return; }
  if (t >= den) { u = 0.0; v = 1.0; return; }
  v = t / den; u = 1.0 - v;
}
AG_HD void tri_origin(d3 a, d3 b, d3 c, double& u, double& v, double& w) {
  d3 ab = b - a, ac = c - a;
  double d1 = -dot(ab, a), d2 = -dot(ac, a);
  if (d1 <= 0.0 && d2 <= 0.0) { u = 1.0; v = 0.0; w = 0.0; return; }
  double d3_ = -dot(ab, b), d4 = -dot(ac, b);
  if (d3_ >= 0.0 && d4 <= d3_) { u = 0.0; v = 1.0; w = 0.0; return; }
  double vc = d1 * d4 - d3_ * d2;
  if (vc <= 0.0 && d1 >= 0.0 && d3_ <= 0.0) { double t = d1 / (d1 - d3_); u = 1.0 - t; v = t; w = 0.0; return; }
  double d5 = -dot(ab, c), d6 = -dot(ac, c);
  if (d6 >= 0.0 && d5 <= d6) { u = 0.0; v = 0.0; w = 1.0; return; }
  double vb = d5 * d2 - d1 * d6;
  if (vb <= 0.0 && d2 >= 0.0 && d6 <= 0.0) { double t = d2 / (d2 - d6); u = 1.0 - t; v = 0.0; w = t; return; }
  double va = d3_ * d6 - d5 * d4;
  if (va <= 0.0 && (d4 - d3_) >= 0.0 && (d5 - d6) >= 0.0) { double t = (d4 - d3_) / ((d4 - d3_) + (d5 - d6)); u = 0.0; v = 1.0 - t; w = t; return; }
  double den = 1.0 / (va + vb + vc);
  v = vb * den; w = vc * den; u = 1.0 - v - w;
}

struct NpOut { f3 pa, pb, n; float d; };   // B-local frame: points on the surfaces, normal B->A, surface distance

// GJK closest points between core A (A-local vertices mapped by R,t into B's frame) and core B.
// Vertices, transforms and the support search are fp32; the simplex solve is fp64.
// Returns true if the cores overlap.
// Support search over a collider's core vertices stored 4 at a time as [x0..x3][y0..y3][z0..z3] (`vq`, 16 B
// aligned, padded with copies of vertex 0): 3 vector loads per 4 vertices, 4 independent dot products in
// flight, first index wins ties exactly like a scalar scan.
struct alignas(16) vq4 { float x, y, z, w; };
AG_HD vq4 ldq4(const float* p) {
#if defined(__CUDA_ARCH__)
  float4 v = __ldg((const float4*)p); vq4 r; r.x = v.x; r.y = v.y; r.z = v.z; r.w = v.w; return r;
#else
  return *(const vq4*)p;
#endif
}
AG_HD int support4(const float* vq, int g0, int n, f3 d) {
  int bi = 0; float best = -3.0e38f;
  const int ng = (n + 3) >> 2;
  const float* p = vq + (size_t)g0 * 12;
  for (int g = 0; g < ng; g++, p += 12) {
    vq4 X = ldq4(p), Y = ldq4(p + 4), Z = ldq4(p + 8);
    float d0 = d.x * X.x + d.y * Y.x + d.z * Z.x, d1 = d.x * X.y + d.y * Y.y + d.z * Z.y;
    float d2 = d.x * X.z + d.y * Y.z + d.z * Z.z, d3v = d.x * X.w + d.y * Y.w + d.z * Z.w;
    if (d0 > best) { best = d0; bi = 4 * g; }
    if (d1 > best) { best = d1; bi = 4 * g + 1; }
    if (d2 > best) { best = d2; bi = 4 * g + 2; }
    if (d3v > best) { best = d3v; bi = 4 * g + 3; }
  }
  return bi < n ? bi : 0;      // a pad entry can only tie with vertex 0, never beat it; guard anyway
}

// `vq` / ga0, gb0: the packed copies of the two cores (group offsets); verts / va0, vb0: the plain copies
AG_HDN inline bool gjk_cores(const float* verts, const float* vq, int va0, int ga0, int nA, int vb0, int gb0, int nB, const m3& R, f3 t,
                             f3& pa, f3& pb, f3& nrm, float& dist) {
  d3 W[4]; f3 PA[4], PB[4];
  int IA[4], IB[4];
  double lam[4] = {1.0, 0.0, 0.0, 0.0};
  int n = 0;
  d3 v = to_d3(mul(R, tv3(verts, va0)) + t) - to_d3(tv3(verts, vb0));
  if (dot(v, v) < 1e-20) v = d3(1.0, 0.0, 0.0);
  bool overlap = false;
  double lower_bound = 0.0;
  for (int it = 0; it < 32; it++) {
    // support of A in direction -v (A-local: R^T(-v)), support of B in +v
    f3 vf = to_f3(v);
    f3 da = mulT(R, -vf);
    int ia = support4(vq, ga0, nA, da), ib = support4(vq, gb0, nB, vf);
    f3 sa = mul(R, tv3(verts, va0 + ia)) + t;
    f3 sb = tv3(verts, vb0 + ib);
    d3 w = to_d3(sa) - to_d3(sb);
    double vv = dot(v, v);
    double vw = dot(v, w);
    if (n > 0 && vw > 0.0) lower_bound = fmax(lower_bound, vw / sqrt(vv));
    if (n > 0 && vv - vw <= 1e-10 * vv) break;
    bool dup = false;
    for (int i = 0; i < n; i++) if (IA[i] == ia && IB[i] == ib) dup = true;
    if (dup) break;
    W[n] = w; PA[n] = sa; PB[n] = sb; IA[n] = ia; IB[n] = ib; n++;
    if (n == 1) { lam[0] = 1.0; }
    else if (n == 2) {
      double u, s; seg_origin(W[0], W[1], u, s);
      if (s <= 0.0) { n = 1; lam[0] = 1.0; }
      else if (u <= 0.0) { W[0] = W[1]; PA[0] = PA[1]; PB[0] = PB[1]; IA[0] = IA[1]; IB[0] = IB[1]; n = 1; lam[0] = 1.0; }
      else { lam[0] = u; lam[1] = s; }
    } else if (n == 3) {
      double l3[3]; tri_origin(W[0], W[1], W[2], l3[0], l3[1], l3[2]);
      int m = 0;
      for (int i = 0; i < 3; i++) if (l3[i] > 0.0) { W[m] = W[i]; PA[m] = PA[i]; PB[m] = PB[i]; IA[m] = IA[i]; IB[m] = IB[i]; lam[m] = l3[i]; m++; }
      n = m;
    } else {
      double bestd = 1e300; int bf = -1; double bl[3] = {0.0, 0.0, 0.0};
      double bestd_all = 1e300; int bf_all = 0; double bla[3] = {1.0, 0.0, 0.0};
      bool any_out = false;
      for (int f = 0; f < 4; f++) {
        int i0 = (f == 3) ? 1 : 0, i1 = (f == 0) ? 1 : ((f == 1) ? 2 : 3), i2 = (f == 0) ? 2 : ((f == 1) ? 3 : ((f == 2) ? 1 : 2)), i3 = (f == 0) ? 3 : ((f == 1) ? 1 : ((f == 2) ? 2 : 0));
        d3 a = W[i0], b = W[i1], c = W[i2], d = W[i3];
        d3 nn = cross(b - a, c - a);
        double sp = -dot(a, nn), sd = dot(d - a, nn);
        // inside only if CLEARLY on the opposite vertex's side; flat tetrahedra count as outside
        double nl = sqrt(dot(nn, nn));
        double tol_d = 1e-9 * nl * sqrt(dot(d - a, d - a)), tol_p = 1e-9 * nl * sqrt(dot(a, a));
        bool inside = (sp * sd > 0.0) && (fabs(sd) > tol_d) && (fabs(sp) > tol_p);
        double u, s, r; tri_origin(a, b, c, u, s, r);
        d3 pt = a * u + b * s + c * r;
        double dd = dot(pt, pt);
        if (dd < bestd_all) { bestd_all = dd; bf_all = f; bla[0] = u; bla[1] = s; bla[2] = r; }
        if (inside) continue;
        any_out = true;
        if (dd < bestd) { bestd = dd; bf = f; bl[0] = u; bl[1] = s; bl[2] = r; }
      }
      if (!any_out) {
        // a positive lower bound on the distance (v.w/|v| of an earlier iteration) proves separation
        if (lower_bound <= 1e-7) { overlap = true; break; }
        bf = bf_all; bl[0] = bla[0]; bl[1] = bla[1]; bl[2] = bla[2];
      }
      int f = bf;
      int id[3];
      id[0] = (f == 3) ? 1 : 0; id[1] = (f == 0) ? 1 : ((f == 1) ? 2 : 3); id[2] = (f == 0) ? 2 : ((f == 1) ? 3 : ((f == 2) ? 1 : 2));
      d3 tw[3]; f3 ta[3], tb[3]; int tia[3], tib[3];
      for (int i = 0; i < 3; i++) { tw[i] = W[id[i]]; ta[i] = PA[id[i]]; tb[i] = PB[id[i]]; tia[i] = IA[id[i]]; tib[i] = IB[id[i]]; }
      int m = 0;
      for (int i = 0; i < 3; i++) if (bl[i] > 0.0) { W[m] = tw[i]; PA[m] = ta[i]; PB[m] = tb[i]; IA[m] = tia[i]; IB[m] = tib[i]; lam[m] = bl[i]; m++; }
      n = m;
    }
    d3 nv(0.0, 0.0, 0.0);
    for (int i = 0; i < n; i++) nv = nv + W[i] * lam[i];
    v = nv;
    if (dot(v, v) <= 1e-16) { overlap = true; break; }
  }
  if (overlap) return true;
  d3 qa(0.0, 0.0, 0.0), qb(0.0, 0.0, 0.0);
  for (int i = 0; i < n; i++) { qa = qa + to_d3(PA[i]) * lam[i]; qb = qb + to_d3(PB[i]) * lam[i]; }
  d3 d = qa - qb;
  double dn = sqrt(dot(d, d));
  pa = to_f3(qa); pb = to_f3(qb);
  dist = (float)dn;
  nrm = dn > 0.0 ? to_f3(d * (1.0 / dn)) : f3(0.f, 0.f, 1.f);
  return false;
}

// axis of least penetration over the face normals of both cores (B-local frame)
AG_HDN inline void pen_faces(const SimDev& S, int va0, int nA, int pa0, int npA, int vb0, int nB, int pb0, int npB,
                             const m3& R, f3 t, f3& pa, f3& pb, f3& nrm, float& dist) {
  float best = -1e30f; bool found = false;
  for (int k = 0; k < npA; k++) {
    f3 nl; float dl; ld_plane(S.planes, pa0 + k, nl, dl);
    f3 n = mul(R, nl); float d = dl + dot(n, t);
    int jb = 0; float mn = dot(n, tv3(S.verts, vb0));
    for (int j = 1; j < nB; j++) { float x = dot(n, tv3(S.verts, vb0 + j)); if (x < mn) { mn = x; jb = j; } }
    float sep = mn - d;
    if (sep > best) { best = sep; found = true; nrm = -n; pb = tv3(S.verts, vb0 + jb); pa = pb - n * sep; }
  }
  for (int k = 0; k < npB; k++) {
    f3 n; float d; ld_plane(S.planes, pb0 + k, n, d);
    f3 nl = mulT(R, n);
    int ja = 0; float mn = dot(nl, tv3(S.verts, va0));
    for (int j = 1; j < nA; j++) { float x = dot(nl, tv3(S.verts, va0 + j)); if (x < mn) { mn = x; ja = j; } }
    float sep = mn + dot(n, t) - d;
    if (sep > best) { best = sep; found = true; nrm = n; pa = mul(R, tv3(S.verts, va0 + ja)) + t; pb = pa - n * sep; }
  }
  if (!found) { nrm = f3(0.f, 0.f, 1.f); pa = mul(R, tv3(S.verts, va0)) + t; pb = tv3(S.verts, vb0); best = 0.f; }
  dist = fminf(best, 0.f);
}

struct CandSet { NpOut c[4]; int n; };
// keep the primary + up to 3 more, greedily the farthest from the chosen set
struct CandSel {
  NpOut prim; NpOut pool[12]; int np;
};

// vertices of core V that lie over the supporting face of the plane owner (see oracle for the rule).
// Everything in B-local coordinates; `planes are given by (p0, np, xf)` where xf says whether plane
// normals need mapping by R,t (owner is A) or not (owner is B).
AG_HDN inline void face_cands(const SimDev& S, int vv0, int nV, float rV, bool v_is_a, int p0, int np, float rP,
                              const m3& R, f3 t, f3 n_to_v, float d_primary, float tol, float max_dist, CandSel& cs) {
  // supporting face
  int kf = -1; float best = 0.98f; f3 nf; float df = 0.f;
  for (int k = 0; k < np; k++) {
    f3 n; float d; ld_plane(S.planes, p0 + k, n, d);
    if (!v_is_a) { f3 nw = mul(R, n); d = d + dot(nw, t); n = nw; }   // plane owner is A: map to B-local
    float al = dot(n, n_to_v);
    if (al > best) { best = al; kf = k; nf = n; df = d; }
  }
  if (kf < 0) return;
  for (int i = 0; i < nV; i++) {
    f3 v = tv3(S.verts, vv0 + i);
    if (v_is_a) v = mul(R, v) + t;
    float h = dot(nf, v) - df;
    float d = h - rV - rP;
    if (d > d_primary + tol || d > max_dist) continue;
    f3 proj = v - nf * h;
    bool inside = true;
    for (int k = 0; k < np; k++) {
      if (k == kf) continue;
      f3 n; float dd; ld_plane(S.planes, p0 + k, n, dd);
      if (!v_is_a) { f3 nw = mul(R, n); dd = dd + dot(nw, t); n = nw; }
      if (dot(n, proj) - dd > 1e-6f) { inside = false; break; }
    }
    if (!inside) continue;
    if (cs.np >= 12) {
      // pool full: replace the shallowest entry if this one is deeper
      int wi = 0; for (int q = 1; q < 12; q++) if (cs.pool[q].d > cs.pool[wi].d) wi = q;
      if (d >= cs.pool[wi].d) continue;
      cs.np = 12;
      NpOut& o = cs.pool[wi];
      f3 on_v = v - nf * rV, on_f = proj + nf * rP;
      if (v_is_a) { o.pa = on_v; o.pb = on_f; o.n = nf; } else { o.pa = on_f; o.pb = on_v; o.n = -nf; }
      o.d = d;
      continue;
    }
    NpOut& o = cs.pool[cs.np++];
    f3 on_v = v - nf * rV, on_f = proj + nf * rP;
    if (v_is_a) { o.pa = on_v; o.pb = on_f; o.n = nf; } else { o.pa = on_f; o.pb = on_v; o.n = -nf; }
    o.d = d;
  }
}

// Manifold selection.  The GJK primary point is arbitrary within a flat contact patch (any point of
// two parallel faces is "closest"), so whenever feature candidates exist the manifold is built from
// them only: deepest candidate first, then greedily the candidate farthest from the chosen set.
AG_HDN inline int select_cands(const CandSel& cs, NpOut* out) {
  if (cs.np == 0) { out[0] = cs.prim; return 1; }
  bool used[12];
  int first = 0;
  for (int i = 0; i < 12; i++) used[i] = i >= cs.np;
  for (int i = 1; i < cs.np; i++) if (cs.pool[i].d < cs.pool[first].d) first = i;
  int nc = 0; out[nc++] = cs.pool[first]; used[first] = true;
  while (nc < 4) {
    int bi = -1; float bd = 1e-8f;
    for (int i = 0; i < cs.np; i++) {
      if (used[i]) continue;
      float md = 1e30f;
      for (int k = 0; k < nc; k++) { f3 d = cs.pool[i].pa - out[k].pa; md = fminf(md, dot(d, d)); }
      if (md > bd) { bd = md; bi = i; }
    }
    if (bi < 0) break;
    used[bi] = true; out[nc++] = cs.pool[bi];
  }
  return nc;
}

// contacts between colliders ca (A) and cb (B) of env e; results in WORLD coordinates.
AG_HDN inline int narrow_pair(const SimDev& S, int e, int ca, int cb, float max_dist, bool manifold, NpOut* out) {
  const int N = S.N;
  int ta = AG_LDG(S.col_type + ca), tb = AG_LDG(S.col_type + cb);
  float ra = AG_LDG(S.col_radius + ca), rb = AG_LDG(S.col_radius + cb);
  int ka = AG_LDG(S.col_link + ca), kb = AG_LDG(S.col_link + cb);
  int va0 = AG_LDG(S.col_v0 + ca), nA = AG_LDG(S.col_nv + ca), vb0 = AG_LDG(S.col_v0 + cb), nB = AG_LDG(S.col_nv + cb);
  int pa0 = AG_LDG(S.col_p0 + ca), npA = AG_LDG(S.col_np + ca), pb0 = AG_LDG(S.col_p0 + cb), npB = AG_LDG(S.col_np + cb);
  f3 posA = ld3(S.lpos, ka, N, e), posB = ld3(S.lpos, kb, N, e);
  q4 qA = ld4(S.lquat, ka, N, e), qB = ld4(S.lquat, kb, N, e);
  CandSel cs; cs.np = 0;
  int nout;
  if (ta == 3 || tb == 3) {
    if (ta == tb) return 0;
    bool flip = (ta == 3);                 // half-space is A; compute in the half-space owner's frame
    // work in the plane owner's local frame: treat owner as "B" of the local computation
    q4 qP = flip ? qA : qB, qV = flip ? qB : qA;
    f3 pP = flip ? posA : posB, pV = flip ? posB : posA;
    m3 R = mul(transpose(qmat(qP)), qmat(qV));
    f3 t = qrot_inv(qP, pV - pP);
    int vv0 = flip ? vb0 : va0, nV = flip ? nB : nA; float rv = flip ? rb : ra;
    f3 pn; float pd; ld_plane(S.planes, flip ? pa0 : pb0, pn, pd);
    int j = 0; float mn = 1e30f;
    for (int i = 0; i < nV; i++) { float x = dot(pn, mul(R, tv3(S.verts, vv0 + i)) + t); if (x < mn) { mn = x; j = i; } }
    float d = mn - pd - rv;
    if (d > max_dist) return 0;
    f3 vj = mul(R, tv3(S.verts, vv0 + j)) + t;
    // local result with V playing "A" (normal from plane towards V)
    cs.prim.pa = vj - pn * rv; cs.prim.pb = vj - pn * (mn - pd); cs.prim.n = pn; cs.prim.d = d;
    if (manifold && nV > 1) face_cands(S, vv0, nV, rv, true, flip ? pa0 : pb0, 1, 0.f, R, t, pn, d, max_dist * 0.5f, max_dist, cs);
    nout = select_cands(cs, out);
    m3 RP = qmat(qP);
    for (int i = 0; i < nout; i++) {
      f3 a = mul(RP, out[i].pa) + pP, b = mul(RP, out[i].pb) + pP, n = mul(RP, out[i].n);
      if (!flip) { out[i].pa = a; out[i].pb = b; out[i].n = n; }
      else { out[i].pa = b; out[i].pb = a; out[i].n = -n; }
    }
    return nout;
  }
  m3 RB = qmat(qB);
  m3 R = mul(transpose(RB), qmat(qA));
  f3 t = mulT(RB, posA - posB);
  f3 pa, pb, nrm; float dist = 0.f;
  bool ov = gjk_cores(S.verts, S.vertq, va0, AG_LDG(S.col_g0 + ca), nA, vb0, AG_LDG(S.col_g0 + cb), nB, R, t, pa, pb, nrm, dist);
  if (ov) pen_faces(S, va0, nA, pa0, npA, vb0, nB, pb0, npB, R, t, pa, pb, nrm, dist);
  float d = dist - ra - rb;
  if (d > max_dist) return 0;
  cs.prim.n = nrm; cs.prim.pa = pa - nrm * ra; cs.prim.pb = pb + nrm * rb; cs.prim.d = d;
  if (manifold) {
    if (npB > 0 && nA > 1) face_cands(S, va0, nA, ra, true, pb0, npB, rb, R, t, nrm, d, max_dist * 0.5f, max_dist, cs);
    if (npA > 0 && nB > 1) face_cands(S, vb0, nB, rb, false, pa0, npA, ra, R, t, -nrm, d, max_dist * 0.5f, max_dist, cs);
  }
  nout = select_cands(cs, out);
  for (int i = 0; i < nout; i++) {
    out[i].pa = mul(RB, out[i].pa) + posB; out[i].pb = mul(RB, out[i].pb) + posB; out[i].n = mul(RB, out[i].n);
  }
  return nout;
}

AG_HD int ag_atomic_inc(int* p) {
#if defined(__CUDA_ARCH__)
  return atomicAdd(p, 1);
#else
  int v = *p; *p = v + 1; return v;
#endif
}
AG_HD int ag_atomic_add(int* p, int k) {
#if defined(__CUDA_ARCH__)
  return atomicAdd(p, k);
#else
  int v = *p; *p = v + k; return v;
#endif
}

// K3a: thread = (slice of a link pair, env lane), env fastest (SimDev::pair_slice: a pair's colliders of link a, cut so that a
// thread makes at most ~64 collider box tests); p.i0 = padded env count.  Cheap AABB culls only:
// surviving collider pairs are appended to the env's candidate list.  Light kernel (few registers,
// full occupancy); the heavy GJK work runs in K3b with one thread per candidate.
AG_HDN inline void pairs_body(int tid, const SimDev& S, const KP& kp) {
  const int N = S.N;
  int Npad = kp.i0;
  int e = tid % Npad, sl = tid / Npad;
  if (e >= N) return;
  int la = AG_LDG(S.pair_slice + 4 * sl), lb = AG_LDG(S.pair_slice + 4 * sl + 1);
  int ba = AG_LDG(S.link_body + la), bb = AG_LDG(S.link_body + lb);
  if (S.body_mode[(size_t)ba * N + e] == 0 || S.body_mode[(size_t)bb * N + e] == 0) return;
  float fac = S.contact_thr;
  f3 lamin = ld3(S.lmin, la, N, e), lamax = ld3(S.lmax, la, N, e), lbmin = ld3(S.lmin, lb, N, e), lbmax = ld3(S.lmax, lb, N, e);
  float tla = AG_LDG(S.link_thresh + la), tlb = AG_LDG(S.link_thresh + lb);
  if (!aabb_ov(lamin, lamax, lbmin, lbmax, fac * fminf(tla, tlb))) return;
  int ca0 = AG_LDG(S.pair_slice + 4 * sl + 2), nca = AG_LDG(S.pair_slice + 4 * sl + 3), cb0 = AG_LDG(S.link_col0 + lb), ncb = AG_LDG(S.link_ncol + lb);
  for (int ca = ca0; ca < ca0 + nca; ca++) {
    f3 amin = ld3(S.cmin, ca, N, e), amax = ld3(S.cmax, ca, N, e);
    float tha = AG_LDG(S.col_thresh + ca);
    if (!aabb_ov(amin, amax, lbmin, lbmax, fac * fminf(tha, tlb))) continue;
    for (int cb = cb0; cb < cb0 + ncb; cb++) {
      float thr = fac * fminf(tha, AG_LDG(S.col_thresh + cb));   // size-relative breaking threshold
      if (!aabb_ov(amin, amax, ld3(S.cmin, cb, N, e), ld3(S.cmax, cb, N, e), thr)) continue;
      int slot = ag_atomic_inc(S.cand_count + e);
      // word = (255 - cost) << 24 | pair id: ascending order = most expensive GJK first, ties by pair (K3a')
      int cost = AG_LDG(S.col_nv + ca) + AG_LDG(S.col_nv + cb); if (cost > 255) cost = 255;
      if (slot < S.maxcand) S.cand[(size_t)slot * N + e] = ((unsigned)(255 - cost) << 24) | ((unsigned)ca * (unsigned)S.nc + (unsigned)cb);
    }
  }
}

// K3a': thread = (candidate slot, env): order the env's candidates by (cost descending, pair id).  Every env is
// a copy of the same scene, so after this the 32 envs of a warp of K3b work on pairs of similar cost at the same
// slot (the un-ordered atomic arrival order left 9 of 32 lanes active); it also makes the list deterministic.
AG_HDN inline void csort_body(int tid, const SimDev& S, const KP&) {
  const int N = S.N;
  int e = tid % N, cs = tid / N;
  int n = S.cand_count[e]; if (n > S.maxcand) n = S.maxcand;
  if (cs >= n) return;
  unsigned w = S.cand[(size_t)cs * N + e];
  int rank = 0;
  for (int j = 0; j < n; j++) rank += (S.cand[(size_t)j * N + e] < w) ? 1 : 0;
  S.cand_s[(size_t)rank * N + e] = w;
}

// K3b: thread = (candidate slot, env): GJK / face fallback / manifold for one collider pair.
AG_HDN inline void narrow_body(int tid, const SimDev& S, const KP&) {
  const int N = S.N;
  int e = tid % N, cs = tid / N;
  int ncand = S.cand_count[e]; if (ncand > S.maxcand) ncand = S.maxcand;
  if (cs >= ncand) return;
  unsigned pk = S.cand_s[(size_t)cs * N + e] & 0xffffffu;
  int ca = (int)(pk / (unsigned)S.nc), cb = (int)(pk % (unsigned)S.nc);
  float thr = S.contact_thr * fminf(AG_LDG(S.col_thresh + ca), AG_LDG(S.col_thresh + cb));
  NpOut out[4];
  int n = narrow_pair(S, e, ca, cb, thr, true, out);
  for (int i = 0; i < n; i++) {
    // raw contacts land in arrival order in a buffer 4x the contact budget; K4 keeps the `maxc` smallest keys,
    // so which contacts survive an over-budget env does not depend on the arrival order
    int slot = ag_atomic_inc(S.c_count + e);
    if (slot >= S.maxraw) continue;
    S.c_key[(size_t)slot * N + e] = pk * 4u + (unsigned)i;
    float* c = S.c_data + (size_t)slot * AG_CFR * N + e;
    c[(size_t)CF_PAX * N] = out[i].pa.x; c[(size_t)CF_PAY * N] = out[i].pa.y; c[(size_t)CF_PAZ * N] = out[i].pa.z;
    c[(size_t)CF_PBX * N] = out[i].pb.x; c[(size_t)CF_PBY * N] = out[i].pb.y; c[(size_t)CF_PBZ * N] = out[i].pb.z;
    c[(size_t)CF_NX * N] = out[i].n.x; c[(size_t)CF_NY * N] = out[i].n.y; c[(size_t)CF_NZ * N] = out[i].n.z;
    c[(size_t)CF_DIST * N] = out[i].d;
  }
}

AG_HD void contact_refs(const SimDev& S, int e, unsigned key, int& refA, int& refB);   // ag_solver.cuh
// K4: deterministic order: rank each contact by its key.  thread = (slot, env).
AG_HDN inline void sort_body(int tid, const SimDev& S, const KP&) {
  const int N = S.N;
  int e = tid % N, slot = tid / N;
  int cnt = S.c_count[e];
  int n = cnt < S.maxraw ? cnt : S.maxraw;
  // sticky flag (cleared by ag_overflow_count): contacts over budget were dropped (by key order, or by arrival
  // order beyond the raw buffer), or candidate pairs beyond `maxcand` were dropped
  if (slot == 0 && ((cnt > S.maxc) || (S.cand_count[e] > S.maxcand))) S.overflow[e] = 1;
  if (slot >= n) return;
  unsigned key = S.c_key[(size_t)slot * N + e];
  int rank = 0;
  for (int j = 0; j < n; j++) rank += (S.c_key[(size_t)j * N + e] < key) ? 1 : 0;
  if (rank >= S.maxc) return;
  S.s_key[(size_t)rank * N + e] = key;
  { int ra, rb2; contact_refs(S, e, key, ra, rb2); S.s_ref[(size_t)rank * 4 * N + e] = ra; S.s_ref[((size_t)rank * 4 + 1) * N + e] = rb2; }
  for (int f = 0; f <= CF_DIST; f++) cf_st(S.s_data, rank, f, N, e, S.c_data[((size_t)slot * AG_CFR + f) * N + e]);
}

// ------------------------------------------------------------------ K5: unconstrained dynamics
// 6x6 articulated inertia in world-aligned axes about the link origin: [[A, B],[B^T, D]], A and D symmetric
struct AI { s3 A; m3 B; s3 D; };
struct SVf { f3 a, l; };   // spatial vector (angular, linear)

AG_HD SVf ai_mul(const AI& I, SVf v) {
  SVf r;
  r.a = mul(I.A, v.a) + mul(I.B, v.l);
  r.l = mulT(I.B, v.a) + mul(I.D, v.l);
  return r;
}
AG_HD m3 skew_m(f3 v) { m3 r; r.m[0] = 0; r.m[1] = -v.z; r.m[2] = v.y; r.m[3] = v.z; r.m[4] = 0; r.m[5] = -v.x; r.m[6] = -v.y; r.m[7] = v.x; r.m[8] = 0; return r; }
AG_HD m3 s3_to_m3(const s3& s) { m3 r; r.m[0] = s.xx; r.m[1] = s.xy; r.m[2] = s.xz; r.m[3] = s.xy; r.m[4] = s.yy; r.m[5] = s.yz; r.m[6] = s.xz; r.m[7] = s.yz; r.m[8] = s.zz; return r; }
// move the reference point of an inertia from P to O where P = O + r
AG_HD AI ai_shift(const AI& I, f3 r) {
  AI o;
  m3 rx = skew_m(r);
  m3 D = s3_to_m3(I.D);
  m3 rxD = mul(rx, D);                    // r x D
  o.D = I.D;
  for (int i = 0; i < 9; i++) o.B.m[i] = I.B.m[i] + rxD.m[i];
  // A_O = A + rx B^T - B rx - rx D rx
  m3 rxBT = mul(rx, transpose(I.B));
  m3 Brx = mul(I.B, rx);
  m3 rxDrx = mul(rxD, rx);
  m3 A = s3_to_m3(I.A);
  for (int i = 0; i < 9; i++) A.m[i] = A.m[i] + rxBT.m[i] - Brx.m[i] - rxDrx.m[i];
  o.A.xx = A.m[0]; o.A.yy = A.m[4]; o.A.zz = A.m[8];
  o.A.xy = 0.5f * (A.m[1] + A.m[3]); o.A.xz = 0.5f * (A.m[2] + A.m[6]); o.A.yz = 0.5f * (A.m[5] + A.m[7]);
  return o;
}
AG_HD void ai_add(AI& a, const AI& b) {
  a.A.xx += b.A.xx; a.A.yy += b.A.yy; a.A.zz += b.A.zz; a.A.xy += b.A.xy; a.A.xz += b.A.xz; a.A.yz += b.A.yz;
  for (int i = 0; i < 9; i++) a.B.m[i] += b.B.m[i];
  a.D.xx += b.D.xx; a.D.yy += b.D.yy; a.D.zz += b.D.zz; a.D.xy += b.D.xy; a.D.xz += b.D.xz; a.D.yz += b.D.yz;
}
// I - U U^T * s
AG_HD AI ai_sub_outer(const AI& I, SVf U, float s) {
  AI o = I;
  o.A.xx -= U.a.x * U.a.x * s; o.A.yy -= U.a.y * U.a.y * s; o.A.zz -= U.a.z * U.a.z * s;
  o.A.xy -= U.a.x * U.a.y * s; o.A.xz -= U.a.x * U.a.z * s; o.A.yz -= U.a.y * U.a.z * s;
  float ua[3] = {U.a.x, U.a.y, U.a.z}, ul[3] = {U.l.x, U.l.y, U.l.z};
  for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) o.B.m[3 * i + j] -= ua[i] * ul[j] * s;
  o.D.xx -= U.l.x * U.l.x * s; o.D.yy -= U.l.y * U.l.y * s; o.D.zz -= U.l.z * U.l.z * s;
  o.D.xy -= U.l.x * U.l.y * s; o.D.xz -= U.l.x * U.l.z * s; o.D.yz -= U.l.y * U.l.z * s;
  return o;
}
AG_HD SVf sv_add(SVf a, SVf b) { SVf r; r.a = a.a + b.a; r.l = a.l + b.l; return r; }
AG_HD SVf sv_scale(SVf a, float s) { SVf r; r.a = a.a * s; r.l = a.l * s; return r; }
AG_HD float sv_dot(SVf m, SVf f) { return dot(m.a, f.a) + dot(m.l, f.l); }

// One lane per env: free bodies (gravity, damping, gyroscopic) and articulated bodies (ABA + M^-1).
// thread = (work item, env): work items 0..nf-1 are the free bodies, nf..nf+nart-1 the articulated bodies (independent of each other)
AG_HDN inline void dyn_body(int tid, const SimDev& S, const KP&) {
  const int N = S.N;
  const int e = tid % N, work = tid / N;
  const float dt = S.dt, vmax = S.vmax, kl = S.lin_damp, ka = S.ang_damp;
  // ---- free rigid bodies
  if (work < S.nf) {
    const int f = work;
    int b = AG_LDG(S.free_body + f);
    int l0 = AG_LDG(S.body_link0 + b);
    q4 q = ld4(S.lquat, l0, N, e);
    f3 com = ld3(S.lpos, l0, N, e) + qrot(q, tv3(S.link_com, l0));
    st3(S.fcom, f, N, e, com);
    size_t ib = (size_t)f * 6 * N + e;
    if (S.body_mode[(size_t)b * N + e] != 1) {
      for (int i = 0; i < 6; i++) S.fIinv[ib + (size_t)i * N] = 0.f;
      return;
    }
    m3 R = qmat(qmul(q, tv4(S.link_iquat, l0)));
    f3 Id = tv3(S.link_inertia, l0);
    s3 Il; Il.xx = Id.x; Il.yy = Id.y; Il.zz = Id.z; Il.xy = Il.xz = Il.yz = 0.f;
    s3 Iw = rot_sym(R, Il);
    s3 Ii; Ii.xx = 1.0f / Id.x; Ii.yy = 1.0f / Id.y; Ii.zz = 1.0f / Id.z; Ii.xy = Ii.xz = Ii.yz = 0.f;
    s3 Iinv = rot_sym(R, Ii);
    f3 v = ld3(S.base_lin, b, N, e), w = ld3(S.base_ang, b, N, e);
    f3 g = tv3(S.body_gravity, b);
    f3 acc = g - v * (kl + kl * norm(v));
    f3 Iww = mul(Iw, w);
    f3 tau = -(Iww * (ka + ka * norm(w)));
    if (S.gyro) tau = tau - cross(w, Iww);
    v = v + acc * dt; w = w + mul(Iinv, tau) * dt;
    v = f3(clampf(v.x, -vmax, vmax), clampf(v.y, -vmax, vmax), clampf(v.z, -vmax, vmax));
    w = f3(clampf(w.x, -vmax, vmax), clampf(w.y, -vmax, vmax), clampf(w.z, -vmax, vmax));
    st3(S.base_lin, b, N, e, v); st3(S.base_ang, b, N, e, w);
    S.fIinv[ib] = Iinv.xx; S.fIinv[ib + N] = Iinv.yy; S.fIinv[ib + 2 * (size_t)N] = Iinv.zz;
    S.fIinv[ib + 3 * (size_t)N] = Iinv.xy; S.fIinv[ib + 4 * (size_t)N] = Iinv.xz; S.fIinv[ib + 5 * (size_t)N] = Iinv.yz;
    return;
  }
  // ---- articulated bodies
  {
    const int a = work - S.nf;
    int b = AG_LDG(S.art_body + a), d0 = AG_LDG(S.art_dl0 + a), nd = AG_LDG(S.art_nd + a);
    bool active = S.body_mode[(size_t)b * N + e] == 1;
    AI IA[AG_MAXND]; SVf pA[AG_MAXND], U[AG_MAXND], c[AG_MAXND], vel[AG_MAXND];
    f3 ax[AG_MAXND], rr[AG_MAXND];
    float Dinv[AG_MAXND], u[AG_MAXND], qd[AG_MAXND];
    int par[AG_MAXND], typ[AG_MAXND];
    f3 g = tv3(S.body_gravity, b);
    int l0 = AG_LDG(S.body_link0 + b);
    f3 obase = ld3(S.lpos, l0, N, e);
    // pass 1: velocities, bias, rigid inertias (world-aligned axes, referred to each link's origin)
    for (int i = 0; i < nd; i++) {
      int d = d0 + i, k = AG_LDG(S.dl_link + d);
      par[i] = AG_LDG(S.dl_parent + d); if (par[i] >= 0) par[i] -= d0;
      typ[i] = AG_LDG(S.dl_type + d);
      q4 q = ld4(S.lquat, k, N, e);
      f3 o = ld3(S.lpos, k, N, e);
      m3 R = qmat(q);
      ax[i] = mul(R, tv3(S.link_axis, k));
      st3(S.jax, d, N, e, ax[i]); st3(S.jor, d, N, e, o);
      f3 op = par[i] >= 0 ? ld3(S.lpos, AG_LDG(S.dl_link + d0 + par[i]), N, e) : obase;
      rr[i] = o - op;
      qd[i] = active ? ld1(S.jqd, k, N, e) : 0.f;
      SVf vp; if (par[i] >= 0) vp = vel[par[i]];
      SVf v; v.a = vp.a; v.l = vp.l + cross(vp.a, rr[i]);
      SVf vj; if (typ[i] == 1) { vj.a = ax[i] * qd[i]; } else { vj.l = ax[i] * qd[i]; }
      v = sv_add(v, vj);
      vel[i] = v;
      c[i].a = cross(v.a, vj.a); c[i].l = cross(v.a, vj.l) + cross(v.l, vj.a);
      // rigid inertia about the link origin
      float m = AG_LDG(S.dl_mass + d);
      f3 mc = mul(R, tv3(S.dl_mc, d));
      s3 Jl; Jl.xx = AG_LDG(S.dl_J + 6 * d); Jl.yy = AG_LDG(S.dl_J + 6 * d + 1); Jl.zz = AG_LDG(S.dl_J + 6 * d + 2);
      Jl.xy = AG_LDG(S.dl_J + 6 * d + 3); Jl.xz = AG_LDG(S.dl_J + 6 * d + 4); Jl.yz = AG_LDG(S.dl_J + 6 * d + 5);
      IA[i].A = rot_sym(R, Jl);
      IA[i].B = skew_m(mc);
      IA[i].D.xx = IA[i].D.yy = IA[i].D.zz = m; IA[i].D.xy = IA[i].D.xz = IA[i].D.yz = 0.f;
      SVf Iv = ai_mul(IA[i], v);
      pA[i].a = cross(v.a, Iv.a) + cross(v.l, Iv.l);
      pA[i].l = cross(v.a, Iv.l);
      // velocity damping, applied per rigid part at its COM (Bullet applies it per original link)
      int p0 = AG_LDG(S.dl_part0 + d), npt = AG_LDG(S.dl_nparts + d);
      for (int pi = p0; pi < p0 + npt; pi++) {
        float pm = AG_LDG(S.pt_mass + pi);
        f3 pc = mul(R, tv3(S.pt_com, pi));
        f3 vc = v.l + cross(v.a, pc);
        f3 fd = vc * (-pm * (kl + kl * norm(vc)));
        s3 Ip; Ip.xx = AG_LDG(S.pt_I + 6 * pi); Ip.yy = AG_LDG(S.pt_I + 6 * pi + 1); Ip.zz = AG_LDG(S.pt_I + 6 * pi + 2);
        Ip.xy = AG_LDG(S.pt_I + 6 * pi + 3); Ip.xz = AG_LDG(S.pt_I + 6 * pi + 4); Ip.yz = AG_LDG(S.pt_I + 6 * pi + 5);
        f3 nd_ = mul(rot_sym(R, Ip), v.a) * (-(ka + ka * norm(v.a)));
        pA[i].a = pA[i].a - (nd_ + cross(pc, fd));
        pA[i].l = pA[i].l - fd;
      }
    }
    // pass 2: articulated inertias, leaf to root
    for (int i = nd - 1; i >= 0; i--) {
      SVf Sx; if (typ[i] == 1) Sx.a = ax[i]; else Sx.l = ax[i];
      U[i] = ai_mul(IA[i], Sx);
      float D = sv_dot(Sx, U[i]);
      Dinv[i] = 1.0f / D;
      float tau = -AG_LDG(S.dl_damping + d0 + i) * qd[i];
      u[i] = tau - sv_dot(Sx, pA[i]);
      if (par[i] >= 0) {
        AI Ia = ai_sub_outer(IA[i], U[i], Dinv[i]);
        SVf pa = sv_add(sv_add(pA[i], ai_mul(Ia, c[i])), sv_scale(U[i], u[i] * Dinv[i]));
        AI Is = ai_shift(Ia, rr[i]);
        ai_add(IA[par[i]], Is);
        pA[par[i]].a = pA[par[i]].a + pa.a + cross(rr[i], pa.l);
        pA[par[i]].l = pA[par[i]].l + pa.l;
      }
    }
    // pass 3: accelerations, root to leaf
    SVf acc[AG_MAXND];
    for (int i = 0; i < nd; i++) {
      SVf ap; if (par[i] >= 0) ap = acc[par[i]]; else { ap.l = -g; }
      SVf a1; a1.a = ap.a + c[i].a; a1.l = ap.l + cross(ap.a, rr[i]) + c[i].l;
      float qdd = (u[i] - sv_dot(U[i], a1)) * Dinv[i];
      if (typ[i] == 1) a1.a = a1.a + ax[i] * qdd; else a1.l = a1.l + ax[i] * qdd;
      acc[i] = a1;
      float nq = clampf(qd[i] + dt * qdd, -vmax, vmax);
      if (active) st1(S.jqd, AG_LDG(S.dl_link + d0 + i), N, e, nq);
    }
    // M^-1 by unit joint impulses through the cached articulated inertias
    for (int j = 0; j < nd; j++) {
      SVf p[AG_MAXND]; float uu[AG_MAXND];
      for (int i = 0; i < nd; i++) { p[i] = SVf(); }
      for (int i = nd - 1; i >= 0; i--) {
        SVf Sx; if (typ[i] == 1) Sx.a = ax[i]; else Sx.l = ax[i];
        uu[i] = ((i == j) ? 1.f : 0.f) - sv_dot(Sx, p[i]);
        if (par[i] >= 0) {
          SVf pa = sv_add(p[i], sv_scale(U[i], uu[i] * Dinv[i]));
          p[par[i]].a = p[par[i]].a + pa.a + cross(rr[i], pa.l);
          p[par[i]].l = p[par[i]].l + pa.l;
        }
      }
      SVf aa[AG_MAXND];
      for (int i = 0; i < nd; i++) {
        SVf ap; if (par[i] >= 0) ap = aa[par[i]];
        SVf a1; a1.a = ap.a; a1.l = ap.l + cross(ap.a, rr[i]);
        float qdd = (uu[i] - sv_dot(U[i], a1)) * Dinv[i];
        if (typ[i] == 1) a1.a = a1.a + ax[i] * qdd; else a1.l = a1.l + ax[i] * qdd;
        aa[i] = a1;
        S.Minv[((size_t)(d0 + i) * S.ND + (d0 + j)) * N + e] = active ? qdd : 0.f;
      }
    }
  }
}

// K6 (constraint rows) and K7 (PGS) live in ag_solver.cuh


// ------------------------------------------------------------------ K8: apply deltas, integrate
// `dvf(i)`: solver delta of velocity entry i (dofs first, then 6 per free body); items are dealt to `stride` lanes
// starting at `first` (the PGS kernel integrates with the 8 lanes of the env's group straight from shared memory,
// the stand-alone kernel with one lane from S.dv).
template <class DV>
AG_HD void integrate_env(int e, const SimDev& S, DV dvf, int first, int stride) {
  const int N = S.N;
  const float dt = S.dt, vmax = S.vmax;
  for (int f = first; f < S.nf; f += stride) {
    int b = AG_LDG(S.free_body + f);
    if (S.body_mode[(size_t)b * N + e] != 1) continue;
    int l0 = AG_LDG(S.body_link0 + b);
    int o = S.ND + 6 * f;
    f3 v = ld3(S.base_lin, b, N, e), w = ld3(S.base_ang, b, N, e);
    v = f3(clampf(v.x + dvf(o), -vmax, vmax), clampf(v.y + dvf(o + 1), -vmax, vmax), clampf(v.z + dvf(o + 2), -vmax, vmax));
    w = f3(clampf(w.x + dvf(o + 3), -vmax, vmax), clampf(w.y + dvf(o + 4), -vmax, vmax), clampf(w.z + dvf(o + 5), -vmax, vmax));
    st3(S.base_lin, b, N, e, v); st3(S.base_ang, b, N, e, w);
    f3 com = ld3(S.fcom, f, N, e) + v * dt;
    q4 qn = qnormalize(qmul(qexp(w * dt), ld4(S.base_quat, b, N, e)));
    st4(S.base_quat, b, N, e, qn);
    st3(S.base_pos, b, N, e, com - qrot(qn, tv3(S.link_com, l0)));
  }
  for (int d = first; d < S.ND; d += stride) {
    int k = AG_LDG(S.dl_link + d);
    int b = AG_LDG(S.link_body + k);
    if (S.body_mode[(size_t)b * N + e] != 1) continue;
    float qd = clampf(ld1(S.jqd, k, N, e) + dvf(d), -vmax, vmax);
    float qn = ld1(S.jq, k, N, e) + dt * qd;
    if (S.hard_limit[k]) {                      // Human.enforce_joint_limits: teleport back, zero velocity
      float lo = AG_LDG(S.link_lower + k), hi = AG_LDG(S.link_upper + k);
      if (qn < lo) { qn = lo; qd = 0.f; } else if (qn > hi) { qn = hi; qd = 0.f; }
    }
    st1(S.jqd, k, N, e, qd);
    st1(S.jq, k, N, e, qn);
  }
  if (first == 0) S.c_count[e] = S.c_count[e] > S.maxc ? S.maxc : S.c_count[e];
}
struct DvGlobal { const SimDev* S; int e; AG_HD float operator()(int i) const { return S->dv[(size_t)i * S->N + e]; } };
AG_HDN inline void integrate_body(int e, const SimDev& S, const KP&) {
  DvGlobal dv; dv.S = &S; dv.e = e;
  integrate_env(e, S, dv, 0, 1);
  for (int d = 0; d < S.ND; d++) {
    int k = AG_LDG(S.dl_link + d);
    if (S.body_mode[(size_t)AG_LDG(S.link_body + k) * S.N + e] != 1) continue;
    st1(S.motor_applied, k, S.N, e, ld1(S.dr_lam, 2 * S.ND + d, S.N, e) / S.dt);
  }
}
