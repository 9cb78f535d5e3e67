// lunarlander.cu -- fused LunarLander-v3 step + TimeLimit + autoreset kernel (sm_100a): a 2-D rigid-body
// sequential-impulse solve per env, one thread per env.
//
// Replaces, for a batch of n envs in one launch:
//   LunarLander.step    gymnasium/envs/box2d/lunar_lander.py:471-665  (incl. world.Step(1/50, 180, 60) at :619)
//   LunarLander.reset   lunar_lander.py:321-447 (terrain, bodies, joints, initial force, the embedded step(0) at :447)
//   ContactDetector     lunar_lander.py:58-76
//   TimeLimit / SyncVectorEnv autoreset as in cartpole.cu
// and, below the reference, the part of the third-party Box2D 2.3.x engine (pybox2d, pyproject.toml:38-43 -- not
// vendored in the reference tree) that this scene exercises: b2PolygonShape mass/hull, fat-AABB broad phase,
// b2CollideEdgeAndPolygon manifolds with feature ids (warm starting), b2ContactSolver (friction, 2-point block
// solver, Baumgarte position correction), b2RevoluteJoint (motor + limit), island sleep, b2World::SolveTOI.  Written against Box2D's
// published algorithm; numeric parity with the real wheel is UNPINNED (it is not installable here) -- the checker is
// oracle/lunar_lander.c, which this kernel matches bit for bit, and the reference's heuristic-landing test.
// b2World::SolveTOI (continuous collision against the static terrain: b2TimeOfImpact with its b2Distance / GJK core and
// separation-function root finder, the TOI sub-step island) is restated as well.  Not restated: wind
// (enable_wind=False is the registered default), continuous actions.
//
// Arithmetic: float32 for everything Box2D does, one IEEE rounding per operation (the library is built with
// --fmad=false); float64 for the Python-side glue.  sin/cos come from one fixed double-precision sequence shared with
// the oracle.  Layout: struct-of-arrays over envs for every field (coalesced 4-byte streams); contact manifolds in a
// most-recent-first list of up to kMaxContacts slots per env.  Latency-bound (a 180-iteration serial Gauss-Seidel
// chain per env), not HBM-bound: ~1.3 KB moved per env-step.
#include <string.h>

#include <type_traits>

#include "common.cuh"

namespace b2e {
namespace {

constexpr int kMaxContacts = 12;  // existing (fat-AABB-overlapping) fixture pairs tracked per env
constexpr int kSlotWords = 16;
constexpr int kNE = 11;  // moon fixtures: base edge + 10 terrain edges
constexpr int kND = 3;   // lander, legs[0], legs[1]

struct V2 {
  float x, y;
};
struct Rot {
  float s, c;
};
struct Xf {
  V2 p;
  Rot q;
};
struct Aabb {
  V2 lo, hi;
};

#define DI __device__ __forceinline__
DI V2 mk(float x, float y) { return V2{x, y}; }
DI V2 operator+(V2 a, V2 b) { return mk(a.x + b.x, a.y + b.y); }
DI V2 operator-(V2 a, V2 b) { return mk(a.x - b.x, a.y - b.y); }
DI V2 operator-(V2 a) { return mk(-a.x, -a.y); }
DI V2 operator*(float s, V2 a) { return mk(s * a.x, s * a.y); }
DI float dot(V2 a, V2 b) { return a.x * b.x + a.y * b.y; }
DI float cross(V2 a, V2 b) { return a.x * b.y - a.y * b.x; }
DI V2 cross_vs(V2 a, float s) { return mk(s * a.y, -s * a.x); }
DI V2 cross_sv(float s, V2 a) { return mk(-s * a.y, s * a.x); }
DI float len(V2 a) { return sqrtf(a.x * a.x + a.y * a.y); }
DI V2 vmin(V2 a, V2 b) { return mk(a.x < b.x ? a.x : b.x, a.y < b.y ? a.y : b.y); }
DI V2 vmax(V2 a, V2 b) { return mk(a.x > b.x ? a.x : b.x, a.y > b.y ? a.y : b.y); }
DI float clampf(float a, float lo, float hi) { return fmaxf(lo, fminf(a, hi)); }

// sin/cos in double from a fixed IEEE op sequence (same as oracle/lunar_lander.c: det_sincos)
DI void det_sincos(double x, double* sn, double* cs) {
  const double fn = rint(x * 6.36619772367581382433e-01);
  const double r = x - fn * 1.57079632673412561417e+00;
  const double w = fn * 6.07710050650619224932e-11;
  const double y = r - w;
  const double z = y * y;
  const double ps = 8.33333333332248946124e-03 +
                    z * (-1.98412698298579493134e-04 +
                         z * (2.75573137070700676789e-06 + z * (-2.50507602534068634195e-08 + z * 1.58969099521155010221e-10)));
  const double sk = y + (z * y) * (-1.66666666666666324348e-01 + z * ps);
  const double pc = z * (4.16666666666666019037e-02 +
                         z * (-1.38888888888741095749e-03 +
                              z * (2.48015872894767294178e-05 +
                                   z * (-2.75573143513906633035e-07 +
                                        z * (2.08757232129817482790e-09 + z * -1.13596475577881948265e-11)))));
  const double ck = 1.0 - (0.5 * z - z * pc);
  switch ((int)fn & 3) {
    case 0: *sn = sk; *cs = ck; break;
    case 1: *sn = ck; *cs = -sk; break;
    case 2: *sn = -sk; *cs = -ck; break;
    default: *sn = -ck; *cs = sk; break;
  }
}
DI Rot rot_set(float a) {
  double s, c;
  det_sincos((double)a, &s, &c);
  return Rot{(float)s, (float)c};
}
DI V2 rmul(Rot q, V2 v) { return mk(q.c * v.x - q.s * v.y, q.s * v.x + q.c * v.y); }
DI V2 xmul(Xf T, V2 v) { return mk((T.q.c * v.x - T.q.s * v.y) + T.p.x, (T.q.s * v.x + T.q.c * v.y) + T.p.y); }
DI V2 xmulT(Xf T, V2 v) {
  const float px = v.x - T.p.x, py = v.y - T.p.y;
  return mk(T.q.c * px + T.q.s * py, -T.q.s * px + T.q.c * py);
}
DI void normalize(V2& a) {
  const float l = len(a);
  if (l < 1.19209290e-7f) return;
  const float inv = 1.0f / l;
  a.x *= inv;
  a.y *= inv;
}

// b2Settings.h
constexpr float kPi = 3.14159265359f;
constexpr float kLinearSlop = 0.005f;
constexpr float kAngularSlop = 2.0f / 180.0f * kPi;
constexpr float kPolyRadius = 2.0f * kLinearSlop;
constexpr float kAabbExt = 0.1f;
constexpr float kAabbMul = 2.0f;
constexpr float kMaxLinCorr = 0.2f;
constexpr float kMaxAngCorr = 8.0f / 180.0f * kPi;
constexpr float kMaxTranslation = 2.0f;
constexpr float kMaxRotation = 0.5f * kPi;
constexpr float kBaumgarte = 0.2f;
constexpr float kTimeToSleep = 0.5f;
constexpr float kLinSleepTol = 0.01f;
constexpr float kAngSleepTol = 2.0f / 180.0f * kPi;
constexpr float kFltMax = 3.402823466e+38f;

// lunar_lander.py:34-55
constexpr double kScale = 30.0, kFps = 50.0, kMainPower = 13.0, kSidePower = 0.6, kInitialRandom = 1000.0;
constexpr double kViewW = 600.0, kViewH = 400.0, kW = kViewW / kScale, kH = kViewH / kScale;
constexpr int kLegAway = 20, kLegDown = 18, kLegW = 2, kLegH = 8, kSideEngineHeight = 14, kSideEngineAway = 12;
constexpr int kMainEngineY = 4;

// ---- immutable model: polygons, mass data (computed once on the host by the same float32 formulas) -----------------
struct Poly {
  int count;
  V2 v[6], n[6], centroid;
};
struct Model {
  Poly poly[kND];
  float inv_mass[kND], inv_I[kND], mass[kND];
  V2 local_center[kND];
  float edge_x1[kNE], edge_x2[kNE];  // chunk_x (float) of each moon fixture; y comes from the per-env terrain
  float edge_friction[kNE], poly_friction[kND];
  V2 anchor_b[2];
  float ref_angle[2], lower[2], upper[2], motor_speed[2], max_motor_torque;
  V2 init_pos[kND];
  float init_angle[kND];
};
__constant__ Model g_model;

// ---- per-env state --------------------------------------------------------------------------------------------------
struct Body {
  V2 c;
  float a;
  V2 v;
  float w, sleep;
  Xf xf;  // derived
  V2 c0;
  float a0, alpha0;  // b2Sweep: pose at the start of the step / of the current TOI interval, its time fraction
};
struct Joint {
  float ix, iy, iz, motor;
  int limit_state;
  // solver temporaries
  V2 rA, rB;
  float m00, m10, m20, m11, m21, m22, motor_mass;
};
struct MPoint {
  V2 lp;
  float ni, ti;
  uint32_t id;
};
struct Contact {
  int pair, touching, type, count;
  int enabled, toi_flag, toi_count;  // b2Contact e_enabledFlag (kept across steps), e_toiFlag / m_toiCount (per step)
  float toi;                         // m_toi: cached time of impact of this step
  float friction;
  V2 local_normal, local_point;
  MPoint pt[2];
};
struct Lander {
  Body b[kND];
  Joint j[2];
  float terrain[kNE];  // [0] unused (base edge y = 0), [1..10] -> smooth_y of chunk i-1 .. via edge_y()
  float smooth[11];
  Aabb fat[kND];
  Contact ct[kMaxContacts];
  int nct;
  int awake, game_over, leg_contact[2], overflow;
  V2 force;      // lander only (reset's ApplyForceToCenter, the wind)
  float torque;  // lander only (turbulence: ApplyTorque)
  int32_t wind_idx, torque_idx;  // enable_wind: offsets into the wind / turbulence pattern (lunar_lander.py:401-403)
  double prev_shaping;
};

DI V2 edge_v1(const Lander& L, int e) { return e == 0 ? mk(0.0f, 0.0f) : mk(g_model.edge_x1[e], L.smooth[e - 1]); }
DI V2 edge_v2(const Lander& L, int e) { return e == 0 ? mk((float)kW, 0.0f) : mk(g_model.edge_x2[e], L.smooth[e]); }

DI void sync_transform(Body& b, V2 lc) {
  b.xf.q = rot_set(b.a);
  b.xf.p = b.c - rmul(b.xf.q, lc);
}
DI Aabb poly_aabb(const Poly& p, Xf xf) {
  V2 lo = xmul(xf, p.v[0]), hi = lo;
  for (int i = 1; i < p.count; ++i) {
    const V2 v = xmul(xf, p.v[i]);
    lo = vmin(lo, v);
    hi = vmax(hi, v);
  }
  return Aabb{mk(lo.x - kPolyRadius, lo.y - kPolyRadius), mk(hi.x + kPolyRadius, hi.y + kPolyRadius)};
}
DI Aabb fatten(Aabb a) {
  return Aabb{mk(a.lo.x - kAabbExt, a.lo.y - kAabbExt), mk(a.hi.x + kAabbExt, a.hi.y + kAabbExt)};
}
DI Aabb edge_fat(const Lander& L, int e) {
  const V2 a = edge_v1(L, e), b = edge_v2(L, e);
  const V2 lo = vmin(a, b), hi = vmax(a, b);
  return fatten(Aabb{mk(lo.x - kPolyRadius, lo.y - kPolyRadius), mk(hi.x + kPolyRadius, hi.y + kPolyRadius)});
}
DI bool aabb_contains(Aabb a, Aabb b) { return a.lo.x <= b.lo.x && a.lo.y <= b.lo.y && b.hi.x <= a.hi.x && b.hi.y <= a.hi.y; }
DI bool aabb_overlap(Aabb a, Aabb b) {
  const V2 d1 = b.lo - a.hi, d2 = a.lo - b.hi;
  if (d1.x > 0.0f || d1.y > 0.0f) return false;
  if (d2.x > 0.0f || d2.y > 0.0f) return false;
  return true;
}

// ---- b2CollideEdgeAndPolygon (plain edge, no ghost vertices) -------------------------------------------------------------
struct ClipV {
  V2 v;
  uint32_t id;  // indexA | indexB<<8 | typeA<<16 | typeB<<24
};
DI uint32_t mkid(int ia, int ib, int ta, int tb) { return (uint32_t)ia | ((uint32_t)ib << 8) | ((uint32_t)ta << 16) | ((uint32_t)tb << 24); }
DI int clip_segment(ClipV out[2], const ClipV in[2], V2 normal, float offset, int vertexIndexA) {
  int n = 0;
  const float d0 = dot(normal, in[0].v) - offset, d1 = dot(normal, in[1].v) - offset;
  if (d0 <= 0.0f) out[n++] = in[0];
  if (d1 <= 0.0f) out[n++] = in[1];
  if (d0 * d1 < 0.0f) {
    const float interp = d0 / (d0 - d1);
    out[n].v = in[0].v + interp * (in[1].v - in[0].v);
    out[n].id = mkid(vertexIndexA, (in[0].id >> 8) & 0xff, 0, 1);
    ++n;
  }
  return n;
}

__device__ __noinline__ void collide_edge_polygon(Contact& c, V2 ev1, V2 ev2, const Poly& pb, Xf xf) {
  const V2 centroidB = xmul(xf, pb.centroid);
  V2 edge1 = ev2 - ev1;
  normalize(edge1);
  const V2 normal1 = mk(edge1.y, -edge1.x);
  const float offset1 = dot(normal1, centroidB - ev1);
  const bool front = offset1 >= 0.0f;
  V2 normal, lower, upper;
  if (front) {
    normal = normal1;
    lower = -normal1;
    upper = -normal1;
  } else {
    normal = -normal1;
    lower = normal1;
    upper = normal1;
  }
  V2 pv[6], pn[6];
  const int count = pb.count;
  for (int i = 0; i < count; ++i) {
    pv[i] = xmul(xf, pb.v[i]);
    pn[i] = rmul(xf.q, pb.n[i]);
  }
  const float radius = 2.0f * kPolyRadius;
  c.count = 0;
  float edge_sep = kFltMax;
  for (int i = 0; i < count; ++i) {
    const float s = dot(normal, pv[i] - ev1);
    if (s < edge_sep) edge_sep = s;
  }
  if (edge_sep > radius) return;
  int ptype = 0, pindex = -1;
  float psep = -kFltMax;
  const V2 perp = mk(-normal.y, normal.x);
  for (int i = 0; i < count; ++i) {
    const V2 n = -pn[i];
    const float s1 = dot(n, pv[i] - ev1), s2 = dot(n, pv[i] - ev2), s = s1 < s2 ? s1 : s2;
    if (s > radius) {
      ptype = 2;
      pindex = i;
      psep = s;
      break;
    }
    if (dot(n, perp) >= 0.0f) {
      if (dot(n - upper, normal) < -kAngularSlop) continue;
    } else {
      if (dot(n - lower, normal) < -kAngularSlop) continue;
    }
    if (s > psep) {
      ptype = 2;
      pindex = i;
      psep = s;
    }
  }
  if (ptype != 0 && psep > radius) return;
  bool primary_edge;
  if (ptype == 0) primary_edge = true;
  else if (psep > 0.98f * edge_sep + 0.001f) primary_edge = false;
  else primary_edge = true;
  ClipV ie[2];
  int rf_i1, rf_i2;
  V2 rf_v1, rf_v2, rf_normal;
  if (primary_edge) {
    c.type = 1;
    int best = 0;
    float bestv = dot(normal, pn[0]);
    for (int i = 1; i < count; ++i) {
      const float v = dot(normal, pn[i]);
      if (v < bestv) {
        bestv = v;
        best = i;
      }
    }
    const int i1 = best, i2 = i1 + 1 < count ? i1 + 1 : 0;
    ie[0].v = pv[i1];
    ie[0].id = mkid(0, i1, 1, 0);
    ie[1].v = pv[i2];
    ie[1].id = mkid(0, i2, 1, 0);
    if (front) {
      rf_i1 = 0; rf_i2 = 1; rf_v1 = ev1; rf_v2 = ev2; rf_normal = normal1;
    } else {
      rf_i1 = 1; rf_i2 = 0; rf_v1 = ev2; rf_v2 = ev1; rf_normal = -normal1;
    }
  } else {
    c.type = 2;
    ie[0].v = ev1;
    ie[0].id = mkid(0, pindex, 0, 1);
    ie[1].v = ev2;
    ie[1].id = mkid(0, pindex, 0, 1);
    rf_i1 = pindex;
    rf_i2 = rf_i1 + 1 < count ? rf_i1 + 1 : 0;
    rf_v1 = pv[rf_i1];
    rf_v2 = pv[rf_i2];
    rf_normal = pn[rf_i1];
  }
  const V2 side1 = mk(rf_normal.y, -rf_normal.x), side2 = -side1;
  const float off1 = dot(side1, rf_v1), off2 = dot(side2, rf_v2);
  ClipV c1[2], c2[2];
  if (clip_segment(c1, ie, side1, off1, rf_i1) < 2) return;
  if (clip_segment(c2, c1, side2, off2, rf_i2) < 2) return;
  if (primary_edge) {
    c.local_normal = rf_normal;
    c.local_point = rf_v1;
  } else {
    c.local_normal = pb.n[rf_i1];
    c.local_point = pb.v[rf_i1];
  }
  int pc = 0;
  for (int i = 0; i < 2; ++i) {
    const float sep = dot(rf_normal, c2[i].v - rf_v1);
    if (sep <= radius) {
      MPoint& cp = c.pt[pc];
      if (primary_edge) {
        cp.lp = xmulT(xf, c2[i].v);
        cp.id = c2[i].id;
      } else {
        cp.lp = c2[i].v;
        const uint32_t id = c2[i].id;
        cp.id = mkid((id >> 8) & 0xff, id & 0xff, (id >> 24) & 0xff, (id >> 16) & 0xff);
      }
      ++pc;
    }
  }
  c.count = pc;
}

DI void begin_contact(Lander& L, int dyn) {  // lunar_lander.py:63-71
  if (dyn == 0) L.game_over = 1;
  else L.leg_contact[dyn - 1] = 1;
}
DI void end_contact(Lander& L, int dyn) {  // lunar_lander.py:73-76
  if (dyn >= 1) L.leg_contact[dyn - 1] = 0;
}

// b2ContactManager::Collide + b2Contact::Update over the most-recent-first contact list
__device__ __noinline__ void collide(Lander& L) {
  if (!L.awake) return;
  int k = 0;
  while (k < L.nct) {
    Contact& c = L.ct[k];
    const int dyn = c.pair / kNE, e = c.pair % kNE;
    if (!aabb_overlap(edge_fat(L, e), L.fat[dyn])) {
      if (c.touching) end_contact(L, dyn);
      for (int t = k; t + 1 < L.nct; ++t) L.ct[t] = L.ct[t + 1];
      --L.nct;
      continue;
    }
    MPoint old[2] = {c.pt[0], c.pt[1]};
    const int old_count = c.count, was = c.touching;
    c.enabled = 1;  // b2Contact::Update re-enables the contact
    collide_edge_polygon(c, edge_v1(L, e), edge_v2(L, e), g_model.poly[dyn], L.b[dyn].xf);
    const int touching = c.count > 0;
    for (int i = 0; i < c.count; ++i) {
      MPoint& mp = c.pt[i];
      mp.ni = 0.0f;
      mp.ti = 0.0f;
      for (int j = 0; j < old_count; ++j)
        if (old[j].id == mp.id) {
          mp.ni = old[j].ni;
          mp.ti = old[j].ti;
          break;
        }
    }
    c.touching = touching;
    if (!was && touching) begin_contact(L, dyn);
    if (was && !touching) end_contact(L, dyn);
    ++k;
  }
}

// b2BroadPhase::UpdatePairs -> b2ContactManager::AddPair: pairs sorted by (edge proxy, polygon proxy); new contacts go
// to the head of the list
DI void find_new_contacts(Lander& L, const bool moved[kND]) {
  for (int e = 0; e < kNE; ++e) {
    const Aabb ef = edge_fat(L, e);
    for (int d = 0; d < kND; ++d) {
      if (!moved[d]) continue;
      if (!aabb_overlap(ef, L.fat[d])) continue;
      const int pair = d * kNE + e;
      bool exists = false;
      for (int k = 0; k < L.nct; ++k) exists |= (L.ct[k].pair == pair);
      if (exists) continue;
      if (L.nct == kMaxContacts) {
        L.overflow = 1;  // cannot happen for this scene's geometry; flagged, never silently wrong
        continue;
      }
      for (int t = L.nct; t > 0; --t) L.ct[t] = L.ct[t - 1];
      ++L.nct;
      Contact& c = L.ct[0];
      c.pair = pair;
      c.touching = 0;
      c.type = 0;
      c.count = 0;
      c.enabled = 1;
      c.toi_flag = 0;
      c.toi_count = 0;
      c.toi = 1.0f;
      c.friction = sqrtf(g_model.edge_friction[e] * g_model.poly_friction[d]);
      L.awake = 1;
    }
  }
}

// ---- b2RevoluteJoint ---------------------------------------------------------------------------------------------------
struct Pos {
  V2 c;
  float a;
};
struct Vel {
  V2 v;
  float w;
};

DI V2 solve22(const Joint& j, V2 b) {
  const float a11 = j.m00, a12 = j.m10, a21 = j.m10, a22 = j.m11;
  float det = a11 * a22 - a12 * a21;
  if (det != 0.0f) det = 1.0f / det;
  return mk(det * (a22 * b.x - a12 * b.y), det * (a11 * b.y - a21 * b.x));
}
DI void solve33(const Joint& j, float bx, float by, float bz, float& x, float& y, float& z) {
  // columns ex = (m00, m10, m20), ey = (m10, m11, m21), ez = (m20, m21, m22) (symmetric)
  const float exx = j.m00, exy = j.m10, exz = j.m20, eyx = j.m10, eyy = j.m11, eyz = j.m21;
  const float ezx = j.m20, ezy = j.m21, ezz = j.m22;
  const float cx = eyy * ezz - eyz * ezy, cy = eyz * ezx - eyx * ezz, cz = eyx * ezy - eyy * ezx;
  float det = exx * cx + exy * cy + exz * cz;
  if (det != 0.0f) det = 1.0f / det;
  x = det * (bx * cx + by * cy + bz * cz);
  const float dx = by * ezz - bz * ezy, dy = bz * ezx - bx * ezz, dz = bx * ezy - by * ezx;
  y = det * (exx * dx + exy * dy + exz * dz);
  const float fx = eyy * bz - eyz * by, fy = eyz * bx - eyx * bz, fz = eyx * by - eyy * bx;
  z = det * (exx * fx + exy * fy + exz * fz);
}

DI void joint_init_velocity(Joint& j, int k, const Pos& pA, const Pos& pB, Vel& vA_, Vel& vB_, float dt_ratio) {
  const Model& M = g_model;
  const float mA = M.inv_mass[0], mB = M.inv_mass[1 + k], iA = M.inv_I[0], iB = M.inv_I[1 + k];
  V2 vA = vA_.v, vB = vB_.v;
  float wA = vA_.w, wB = vB_.w;
  const Rot qA = rot_set(pA.a), qB = rot_set(pB.a);
  j.rA = rmul(qA, mk(0.0f, 0.0f) - M.local_center[0]);
  j.rB = rmul(qB, M.anchor_b[k] - M.local_center[1 + k]);
  j.m00 = mA + mB + j.rA.y * j.rA.y * iA + j.rB.y * j.rB.y * iB;
  j.m10 = -j.rA.y * j.rA.x * iA - j.rB.y * j.rB.x * iB;
  j.m20 = -j.rA.y * iA - j.rB.y * iB;
  j.m11 = mA + mB + j.rA.x * j.rA.x * iA + j.rB.x * j.rB.x * iB;
  j.m21 = j.rA.x * iA + j.rB.x * iB;
  j.m22 = iA + iB;
  j.motor_mass = iA + iB;
  if (j.motor_mass > 0.0f) j.motor_mass = 1.0f / j.motor_mass;
  const float angle = pB.a - pA.a - M.ref_angle[k];
  if (fabsf(M.upper[k] - M.lower[k]) < 2.0f * kAngularSlop) {
    j.limit_state = 3;
  } else if (angle <= M.lower[k]) {
    if (j.limit_state != 1) j.iz = 0.0f;
    j.limit_state = 1;
  } else if (angle >= M.upper[k]) {
    if (j.limit_state != 2) j.iz = 0.0f;
    j.limit_state = 2;
  } else {
    j.limit_state = 0;
    j.iz = 0.0f;
  }
  j.ix *= dt_ratio;
  j.iy *= dt_ratio;
  j.iz *= dt_ratio;
  j.motor *= dt_ratio;
  const V2 P = mk(j.ix, j.iy);
  vA = vA - mA * P;
  wA -= iA * (cross(j.rA, P) + j.motor + j.iz);
  vB = vB + mB * P;
  wB += iB * (cross(j.rB, P) + j.motor + j.iz);
  vA_.v = vA; vA_.w = wA; vB_.v = vB; vB_.w = wB;
}

DI void joint_solve_velocity(Joint& j, int k, Vel& vA_, Vel& vB_, float dt) {
  const Model& M = g_model;
  const float mA = M.inv_mass[0], mB = M.inv_mass[1 + k], iA = M.inv_I[0], iB = M.inv_I[1 + k];
  V2 vA = vA_.v, vB = vB_.v;
  float wA = vA_.w, wB = vB_.w;
  if (j.limit_state != 3) {
    const float Cdot = wB - wA - M.motor_speed[k];
    float impulse = -j.motor_mass * Cdot;
    const float old = j.motor, maxi = dt * M.max_motor_torque;
    j.motor = clampf(old + impulse, -maxi, maxi);
    impulse = j.motor - old;
    wA -= iA * impulse;
    wB += iB * impulse;
  }
  if (j.limit_state != 0) {
    const V2 Cdot1 = ((vB + cross_sv(wB, j.rB)) - vA) - cross_sv(wA, j.rA);
    const float Cdot2 = wB - wA;
    float ix, iy, iz;
    solve33(j, Cdot1.x, Cdot1.y, Cdot2, ix, iy, iz);
    ix = -ix; iy = -iy; iz = -iz;
    if (j.limit_state == 3) {
      j.ix += ix; j.iy += iy; j.iz += iz;
    } else {
      const float newi = j.iz + iz;
      const bool reduce = j.limit_state == 1 ? (newi < 0.0f) : (newi > 0.0f);
      if (reduce) {
        const V2 rhs = (-Cdot1) + j.iz * mk(j.m20, j.m21);
        const V2 red = solve22(j, rhs);
        ix = red.x; iy = red.y; iz = -j.iz;
        j.ix += red.x; j.iy += red.y; j.iz = 0.0f;
      } else {
        j.ix += ix; j.iy += iy; j.iz += iz;
      }
    }
    const V2 P = mk(ix, iy);
    vA = vA - mA * P;
    wA -= iA * (cross(j.rA, P) + iz);
    vB = vB + mB * P;
    wB += iB * (cross(j.rB, P) + iz);
  } else {
    const V2 Cdot = ((vB + cross_sv(wB, j.rB)) - vA) - cross_sv(wA, j.rA);
    const V2 imp = solve22(j, -Cdot);
    j.ix += imp.x;
    j.iy += imp.y;
    vA = vA - mA * imp;
    wA -= iA * cross(j.rA, imp);
    vB = vB + mB * imp;
    wB += iB * cross(j.rB, imp);
  }
  vA_.v = vA; vA_.w = wA; vB_.v = vB; vB_.w = wB;
}

DI bool joint_solve_position(const Joint& j, int k, Pos& pA, Pos& pB) {
  const Model& M = g_model;
  const float mA = M.inv_mass[0], mB = M.inv_mass[1 + k], iA = M.inv_I[0], iB = M.inv_I[1 + k];
  V2 cA = pA.c, cB = pB.c;
  float aA = pA.a, aB = pB.a, angular_error = 0.0f, position_error;
  if (j.limit_state != 0) {
    const float angle = aB - aA - M.ref_angle[k];
    float limit_impulse;
    if (j.limit_state == 3) {
      const float C = clampf(angle - M.lower[k], -kMaxAngCorr, kMaxAngCorr);
      limit_impulse = -j.motor_mass * C;
      angular_error = fabsf(C);
    } else if (j.limit_state == 1) {
      float C = angle - M.lower[k];
      angular_error = -C;
      C = clampf(C + kAngularSlop, -kMaxAngCorr, 0.0f);
      limit_impulse = -j.motor_mass * C;
    } else {
      float C = angle - M.upper[k];
      angular_error = C;
      C = clampf(C - kAngularSlop, 0.0f, kMaxAngCorr);
      limit_impulse = -j.motor_mass * C;
    }
    aA -= iA * limit_impulse;
    aB += iB * limit_impulse;
  }
  {
    const Rot qA = rot_set(aA), qB = rot_set(aB);
    const V2 rA = rmul(qA, mk(0.0f, 0.0f) - M.local_center[0]), rB = rmul(qB, M.anchor_b[k] - M.local_center[1 + k]);
    const V2 C = ((cB + rB) - cA) - rA;
    position_error = len(C);
    const float k11 = mA + mB + iA * rA.y * rA.y + iB * rB.y * rB.y;
    const float k12 = -iA * rA.x * rA.y - iB * rB.x * rB.y;
    const float k22 = mA + mB + iA * rA.x * rA.x + iB * rB.x * rB.x;
    float det = k11 * k22 - k12 * k12;
    if (det != 0.0f) det = 1.0f / det;
    const V2 imp = mk(-(det * (k22 * C.x - k12 * C.y)), -(det * (k11 * C.y - k12 * C.x)));
    cA = cA - mA * imp;
    aA -= iA * cross(rA, imp);
    cB = cB + mB * imp;
    aB += iB * cross(rB, imp);
  }
  pA.c = cA; pA.a = aA; pB.c = cB; pB.a = aB;
  return position_error <= kLinearSlop && angular_error <= kAngularSlop;
}

// ---- b2ContactSolver ------------------------------------------------------------------------------------------------------
struct VCP {
  V2 rB;
  float ni, ti, normal_mass, tangent_mass;
};
struct VC {
  int slot, ib, count, pos_count, type;
  VCP p[2];
  V2 normal, local_normal, local_point, lpts[2];
  float k00, k01, k11, n00, n10, n01, n11, friction;
};

// Body access by a RUNTIME index without control flow: the solver keeps the three bodies' positions / velocities in
// registers, and a contact's body index differs lane to lane.  Selecting the operands (and writing the result back) with
// predicated moves lets lanes that touch different bodies execute the same instructions together; a switch on the index
// (three inlined copies of every contact routine, the round-1 version) serialised them for all 180 + 60 iterations.
DI float sel3(int i, float a, float b, float c) { return i == 0 ? a : (i == 1 ? b : c); }
DI Pos get_pos(const Pos (&P)[kND], int ib) {
  Pos r;
  r.c.x = sel3(ib, P[0].c.x, P[1].c.x, P[2].c.x);
  r.c.y = sel3(ib, P[0].c.y, P[1].c.y, P[2].c.y);
  r.a = sel3(ib, P[0].a, P[1].a, P[2].a);
  return r;
}
DI void put_pos(Pos (&P)[kND], int ib, V2 c, float a) {
#pragma unroll
  for (int i = 0; i < kND; ++i) {
    P[i].c.x = ib == i ? c.x : P[i].c.x;
    P[i].c.y = ib == i ? c.y : P[i].c.y;
    P[i].a = ib == i ? a : P[i].a;
  }
}
DI Vel get_vel(const Vel (&V)[kND], int ib) {
  Vel r;
  r.v.x = sel3(ib, V[0].v.x, V[1].v.x, V[2].v.x);
  r.v.y = sel3(ib, V[0].v.y, V[1].v.y, V[2].v.y);
  r.w = sel3(ib, V[0].w, V[1].w, V[2].w);
  return r;
}
DI void put_vel(Vel (&V)[kND], int ib, V2 v, float w) {
#pragma unroll
  for (int i = 0; i < kND; ++i) {
    V[i].v.x = ib == i ? v.x : V[i].v.x;
    V[i].v.y = ib == i ? v.y : V[i].v.y;
    V[i].w = ib == i ? w : V[i].w;
  }
}

// b2World::Solve for the one island {legs[1], lander, legs[0]} (+ the static moon); local body indices 0..2 = lander, legs
__device__ __noinline__ void solve_island(Lander& L, float h, float dt_ratio, float gravity) {
  const Model& M = g_model;
  Pos P[kND];
  Vel Vv[kND];
  Joint j0 = L.j[0], j1 = L.j[1];  // register copies for the 180-iteration loop
  const V2 g = mk(0.0f, gravity);
#pragma unroll
  for (int i = 0; i < kND; ++i) {
    Body& b = L.b[i];
    V2 v = b.v;
    float w = b.w;
    b.c0 = b.c;
    b.a0 = b.a;
    const V2 force = i == 0 ? L.force : mk(0.0f, 0.0f);
    v = v + h * ((1.0f * g) + (M.inv_mass[i] * force));
    w += h * M.inv_I[i] * (i == 0 ? L.torque : 0.0f);
    v = (1.0f / (1.0f + h * 0.0f)) * v;
    w *= 1.0f / (1.0f + h * 0.0f);
    P[i].c = b.c; P[i].a = b.a; Vv[i].v = v; Vv[i].w = w;
  }
  // island contact order: contacts of legs[1], lander, legs[0]; each most-recent-first; touching only
  VC vcs[kMaxContacts];
  int nvc = 0;
  const int order[3] = {2, 0, 1};
  for (int t = 0; t < 3; ++t)
    for (int k = 0; k < L.nct; ++k) {
      const Contact& c = L.ct[k];
      if (!c.touching || c.pair / kNE != order[t]) continue;
      VC& vc = vcs[nvc++];
      vc.slot = k;
      vc.ib = order[t];
      vc.friction = c.friction;
      vc.count = vc.pos_count = c.count;
      vc.type = c.type;
      vc.local_normal = c.local_normal;
      vc.local_point = c.local_point;
      for (int j = 0; j < c.count; ++j) {
        vc.p[j].ni = dt_ratio * c.pt[j].ni;
        vc.p[j].ti = dt_ratio * c.pt[j].ti;
        vc.lpts[j] = c.pt[j].lp;
      }
    }
  for (int k = 0; k < nvc; ++k) {  // InitializeVelocityConstraints (bodyA = static moon at the origin)
    VC& vc = vcs[k];
    {
      const int ib = vc.ib;
      const float mB = sel3(ib, M.inv_mass[0], M.inv_mass[1], M.inv_mass[2]);
      const float iB = sel3(ib, M.inv_I[0], M.inv_I[1], M.inv_I[2]);
      const V2 lcB = mk(sel3(ib, M.local_center[0].x, M.local_center[1].x, M.local_center[2].x),
                        sel3(ib, M.local_center[0].y, M.local_center[1].y, M.local_center[2].y));
      const Pos pB = get_pos(P, ib);
      const V2 cB = pB.c;
      Xf xfB;
      xfB.q = rot_set(pB.a);
      xfB.p = cB - rmul(xfB.q, lcB);
      V2 pts[2];
      if (vc.type == 1) {  // b2WorldManifold::Initialize, e_faceA
        vc.normal = vc.local_normal;
        const V2 plane = vc.local_point;
        for (int j = 0; j < vc.count; ++j) {
          const V2 clip = xmul(xfB, vc.lpts[j]);
          const V2 cA = clip + (kPolyRadius - dot(clip - plane, vc.normal)) * vc.normal;
          const V2 cBp = clip - kPolyRadius * vc.normal;
          pts[j] = 0.5f * (cA + cBp);
        }
      } else {  // e_faceB
        V2 nrm = rmul(xfB.q, vc.local_normal);
        const V2 plane = xmul(xfB, vc.local_point);
        for (int j = 0; j < vc.count; ++j) {
          const V2 clip = vc.lpts[j];
          const V2 cBp = clip + (kPolyRadius - dot(clip - plane, nrm)) * nrm;
          const V2 cA = clip - kPolyRadius * nrm;
          pts[j] = 0.5f * (cA + cBp);
        }
        vc.normal = -nrm;
      }
      for (int j = 0; j < vc.count; ++j) {
        VCP& p = vc.p[j];
        p.rB = pts[j] - cB;
        const float rnB = cross(p.rB, vc.normal);
        const float kN = mB + iB * rnB * rnB;
        p.normal_mass = kN > 0.0f ? 1.0f / kN : 0.0f;
        const V2 tangent = cross_vs(vc.normal, 1.0f);
        const float rtB = cross(p.rB, tangent);
        const float kT = mB + iB * rtB * rtB;
        p.tangent_mass = kT > 0.0f ? 1.0f / kT : 0.0f;
      }
      if (vc.count == 2) {
        const float rn1B = cross(vc.p[0].rB, vc.normal), rn2B = cross(vc.p[1].rB, vc.normal);
        const float k11 = mB + iB * rn1B * rn1B, k22 = mB + iB * rn2B * rn2B, k12 = mB + iB * rn1B * rn2B;
        if (k11 * k11 < 1000.0f * (k11 * k22 - k12 * k12)) {
          vc.k00 = k11; vc.k01 = k12; vc.k11 = k22;
          float det = k11 * k22 - k12 * k12;
          if (det != 0.0f) det = 1.0f / det;
          vc.n00 = det * k22; vc.n10 = -det * k12; vc.n01 = -det * k12; vc.n11 = det * k11;
        } else {
          vc.count = 1;
        }
      }
    }
  }
  for (int k = 0; k < nvc; ++k) {  // WarmStart
    VC& vc = vcs[k];
    const int ib = vc.ib;
    const float mB = sel3(ib, M.inv_mass[0], M.inv_mass[1], M.inv_mass[2]);
    const float iB = sel3(ib, M.inv_I[0], M.inv_I[1], M.inv_I[2]);
    const Vel vel = get_vel(Vv, ib);
    V2 vB = vel.v;
    float wB = vel.w;
    const V2 tangent = cross_vs(vc.normal, 1.0f);
    for (int j = 0; j < vc.count; ++j) {
      const V2 Pi = (vc.p[j].ni * vc.normal) + (vc.p[j].ti * tangent);
      wB += iB * cross(vc.p[j].rB, Pi);
      vB = vB + mB * Pi;
    }
    put_vel(Vv, ib, vB, wB);
  }
  joint_init_velocity(j1, 1, P[0], P[2], Vv[0], Vv[2], dt_ratio);
  joint_init_velocity(j0, 0, P[0], P[1], Vv[0], Vv[1], dt_ratio);
  for (int it = 0; it < 180; ++it) {
    joint_solve_velocity(j1, 1, Vv[0], Vv[2], h);
    joint_solve_velocity(j0, 0, Vv[0], Vv[1], h);
    for (int k = 0; k < nvc; ++k) {
      VC& vc = vcs[k];
      {
        const int ib = vc.ib;
        const float mB = sel3(ib, M.inv_mass[0], M.inv_mass[1], M.inv_mass[2]);
        const float iB = sel3(ib, M.inv_I[0], M.inv_I[1], M.inv_I[2]);
        const Vel vel = get_vel(Vv, ib);
        V2 vB = vel.v;
        float wB = vel.w;
        const V2 normal = vc.normal, tangent = cross_vs(normal, 1.0f);
        for (int j = 0; j < vc.count; ++j) {
          VCP& p = vc.p[j];
          const V2 dv = vB + cross_sv(wB, p.rB);
          const float vt = dot(dv, tangent) - 0.0f;
          float lambda = p.tangent_mass * (-vt);
          const float maxf = vc.friction * p.ni;
          const float newi = clampf(p.ti + lambda, -maxf, maxf);
          lambda = newi - p.ti;
          p.ti = newi;
          const V2 Pi = lambda * tangent;
          vB = vB + mB * Pi;
          wB += iB * cross(p.rB, Pi);
        }
        if (vc.count == 1) {
          VCP& p = vc.p[0];
          const V2 dv = vB + cross_sv(wB, p.rB);
          const float vn = dot(dv, normal);
          float lambda = -p.normal_mass * (vn - 0.0f);
          const float newi = fmaxf(p.ni + lambda, 0.0f);
          lambda = newi - p.ni;
          p.ni = newi;
          const V2 Pi = lambda * normal;
          vB = vB + mB * Pi;
          wB += iB * cross(p.rB, Pi);
        } else {
          VCP &c1 = vc.p[0], &c2 = vc.p[1];
          const float ax = c1.ni, ay = c2.ni;
          const V2 dv1 = vB + cross_sv(wB, c1.rB), dv2 = vB + cross_sv(wB, c2.rB);
          float vn1 = dot(dv1, normal), vn2 = dot(dv2, normal);
          float bx = vn1 - 0.0f, by = vn2 - 0.0f;
          bx -= vc.k00 * ax + vc.k01 * ay;
          by -= vc.k01 * ax + vc.k11 * ay;
          float xx, xy;
          bool solved = false;
          xx = -(vc.n00 * bx + vc.n10 * by);
          xy = -(vc.n01 * bx + vc.n11 * by);
          if (xx >= 0.0f && xy >= 0.0f) solved = true;
          if (!solved) {
            xx = -c1.normal_mass * bx;
            xy = 0.0f;
            vn2 = vc.k01 * xx + by;
            if (xx >= 0.0f && vn2 >= 0.0f) solved = true;
          }
          if (!solved) {
            xx = 0.0f;
            xy = -c2.normal_mass * by;
            vn1 = vc.k01 * xy + bx;
            if (xy >= 0.0f && vn1 >= 0.0f) solved = true;
          }
          if (!solved) {
            xx = 0.0f;
            xy = 0.0f;
            if (bx >= 0.0f && by >= 0.0f) solved = true;
          }
          if (solved) {
            const float dx = xx - ax, dy = xy - ay;
            const V2 P1 = dx * normal, P2 = dy * normal;
            vB = vB + mB * (P1 + P2);
            wB += iB * (cross(c1.rB, P1) + cross(c2.rB, P2));
            c1.ni = xx;
            c2.ni = xy;
          }
        }
        put_vel(Vv, ib, vB, wB);
      }
    }
  }
  for (int k = 0; k < nvc; ++k)  // StoreImpulses
    for (int j = 0; j < vcs[k].count; ++j) {
      L.ct[vcs[k].slot].pt[j].ni = vcs[k].p[j].ni;
      L.ct[vcs[k].slot].pt[j].ti = vcs[k].p[j].ti;
    }
#pragma unroll
  for (int i = 0; i < kND; ++i) {  // integrate positions
    V2 c = P[i].c, v = Vv[i].v;
    float a = P[i].a, w = Vv[i].w;
    const V2 tr = h * v;
    if (dot(tr, tr) > kMaxTranslation * kMaxTranslation) {
      const float ratio = kMaxTranslation / len(tr);
      v = ratio * v;
    }
    const float rotn = h * w;
    if (rotn * rotn > kMaxRotation * kMaxRotation) {
      const float ratio = kMaxRotation / fabsf(rotn);
      w *= ratio;
    }
    c = c + h * v;
    a += h * w;
    P[i].c = c; P[i].a = a; Vv[i].v = v; Vv[i].w = w;
  }
  bool position_solved = false;
  for (int it = 0; it < 60; ++it) {
    float min_sep = 0.0f;
    for (int k = 0; k < nvc; ++k) {
      const VC& vc = vcs[k];
      {
        const int ib = vc.ib;
        const float mB = sel3(ib, M.inv_mass[0], M.inv_mass[1], M.inv_mass[2]);
        const float iB = sel3(ib, M.inv_I[0], M.inv_I[1], M.inv_I[2]);
        const V2 lcB = mk(sel3(ib, M.local_center[0].x, M.local_center[1].x, M.local_center[2].x),
                          sel3(ib, M.local_center[0].y, M.local_center[1].y, M.local_center[2].y));
        const Pos pB = get_pos(P, ib);
        V2 cB = pB.c;
        float aB = pB.a;
        for (int j = 0; j < vc.pos_count; ++j) {
          Xf xfB;
          xfB.q = rot_set(aB);
          xfB.p = cB - rmul(xfB.q, lcB);
          V2 normal, point;
          float sep;
          if (vc.type == 1) {
            normal = vc.local_normal;
            const V2 clip = xmul(xfB, vc.lpts[j]);
            sep = dot(clip - vc.local_point, normal) - kPolyRadius - kPolyRadius;
            point = clip;
          } else {
            normal = rmul(xfB.q, vc.local_normal);
            const V2 plane = xmul(xfB, vc.local_point), clip = vc.lpts[j];
            sep = dot(clip - plane, normal) - kPolyRadius - kPolyRadius;
            point = clip;
            normal = -normal;
          }
          const V2 rB = point - cB;
          min_sep = fminf(min_sep, sep);
          const float C = clampf(kBaumgarte * (sep + kLinearSlop), -kMaxLinCorr, 0.0f);
          const float rnB = cross(rB, normal);
          const float K = mB + iB * rnB * rnB;
          const float impulse = K > 0.0f ? -C / K : 0.0f;
          const V2 Pi = impulse * normal;
          cB = cB + mB * Pi;
          aB += iB * cross(rB, Pi);
        }
        put_pos(P, ib, cB, aB);
      }
    }
    const bool contacts_ok = min_sep >= -3.0f * kLinearSlop;
    const bool ok1 = joint_solve_position(j1, 1, P[0], P[2]);
    const bool ok0 = joint_solve_position(j0, 0, P[0], P[1]);
    if (contacts_ok && ok1 && ok0) {
      position_solved = true;
      break;
    }
  }
  L.j[0] = j0;
  L.j[1] = j1;
  float min_sleep = kFltMax;
#pragma unroll
  for (int i = 0; i < kND; ++i) {
    Body& b = L.b[i];
    b.c = P[i].c; b.a = P[i].a; b.v = Vv[i].v; b.w = Vv[i].w;
    sync_transform(b, M.local_center[i]);
    if (b.w * b.w > kAngSleepTol * kAngSleepTol || dot(b.v, b.v) > kLinSleepTol * kLinSleepTol) {
      b.sleep = 0.0f;
      min_sleep = 0.0f;
    } else {
      b.sleep += h;
      min_sleep = fminf(min_sleep, b.sleep);
    }
  }
  if (min_sleep >= kTimeToSleep && position_solved) {
    L.awake = 0;
#pragma unroll
    for (int i = 0; i < kND; ++i) {
      L.b[i].sleep = 0.0f;
      L.b[i].v = mk(0.0f, 0.0f);
      L.b[i].w = 0.0f;
    }
  }
}

// ---- continuous collision: b2Distance (GJK), b2TimeOfImpact, b2World::SolveTOI / b2Island::SolveTOI --------------------
// Proxy A is always a terrain edge (2 vertices; its body, the static moon, has the identity transform, so b2Mul / b2MulT
// by it are exact no-ops and are written as such), proxy B the polygon of a dynamic body; both have radius b2_polygonRadius.
constexpr float kEpsilon = 1.192092896e-07f;
constexpr int kMaxSubSteps = 8;
constexpr float kToiBaumgarte = 0.75f;
constexpr int kMaxPolyVerts = 8;

struct Sweep {
  V2 lc, c0, c;
  float a0, a, alpha0;
};
DI Xf sweep_xf(const Sweep& s, float beta) {  // b2Sweep::GetTransform
  Xf xf;
  xf.p = ((1.0f - beta) * s.c0) + (beta * s.c);
  const float angle = (1.0f - beta) * s.a0 + beta * s.a;
  xf.q = rot_set(angle);
  xf.p = xf.p - rmul(xf.q, s.lc);
  return xf;
}
DI void sweep_advance(Sweep& s, float alpha) {  // b2Sweep::Advance
  const float beta = (alpha - s.alpha0) / (1.0f - s.alpha0);
  s.c0 = s.c0 + beta * (s.c - s.c0);
  s.a0 += beta * (s.a - s.a0);
  s.alpha0 = alpha;
}
DI Sweep body_sweep(const Body& b, V2 lc) { return Sweep{lc, b.c0, b.c, b.a0, b.a, b.alpha0}; }
DI void body_set_sweep(Body& b, const Sweep& s) {
  b.c0 = s.c0; b.c = s.c; b.a0 = s.a0; b.a = s.a; b.alpha0 = s.alpha0;
}
DI V2 rmulT(Rot q, V2 v) { return mk(q.c * v.x + q.s * v.y, -q.s * v.x + q.c * v.y); }

struct Proxy {
  V2 v[6];
  int count;
};
DI int proxy_support(const Proxy& p, V2 d) {  // b2DistanceProxy::GetSupport
  int best = 0;
  float bestv = dot(p.v[0], d);
  for (int i = 1; i < p.count; ++i) {
    const float v = dot(p.v[i], d);
    if (v > bestv) {
      best = i;
      bestv = v;
    }
  }
  return best;
}

struct SV {  // b2SimplexVertex
  V2 wA, wB, w;
  float a;
  int iA, iB;
};
struct SCache {  // b2SimplexCache
  float metric;
  int count, iA[3], iB[3];
};
struct Simplex {
  SV v[3];
  int count;
};
DI float simplex_metric(const Simplex& s) {
  if (s.count == 2) return len(s.v[0].w - s.v[1].w);
  if (s.count == 3) return cross(s.v[1].w - s.v[0].w, s.v[2].w - s.v[0].w);
  return 0.0f;
}
DI void simplex_solve2(Simplex& s) {
  const V2 w1 = s.v[0].w, w2 = s.v[1].w, e12 = w2 - w1;
  const float d12_2 = -dot(w1, e12);
  if (d12_2 <= 0.0f) { s.v[0].a = 1.0f; s.count = 1; return; }
  const float d12_1 = dot(w2, e12);
  if (d12_1 <= 0.0f) { s.v[1].a = 1.0f; s.count = 1; s.v[0] = s.v[1]; return; }
  const float inv = 1.0f / (d12_1 + d12_2);
  s.v[0].a = d12_1 * inv;
  s.v[1].a = d12_2 * inv;
  s.count = 2;
}
DI void simplex_solve3(Simplex& s) {
  const V2 w1 = s.v[0].w, w2 = s.v[1].w, w3 = s.v[2].w;
  const V2 e12 = w2 - w1;
  const float w1e12 = dot(w1, e12), w2e12 = dot(w2, e12), d12_1 = w2e12, d12_2 = -w1e12;
  const V2 e13 = w3 - w1;
  const float w1e13 = dot(w1, e13), w3e13 = dot(w3, e13), d13_1 = w3e13, d13_2 = -w1e13;
  const V2 e23 = w3 - w2;
  const float w2e23 = dot(w2, e23), w3e23 = dot(w3, e23), d23_1 = w3e23, d23_2 = -w2e23;
  const float n123 = cross(e12, e13);
  const float d123_1 = n123 * cross(w2, w3), d123_2 = n123 * cross(w3, w1), d123_3 = n123 * cross(w1, w2);
  if (d12_2 <= 0.0f && d13_2 <= 0.0f) { s.v[0].a = 1.0f; s.count = 1; return; }
  if (d12_1 > 0.0f && d12_2 > 0.0f && d123_3 <= 0.0f) {
    const float inv = 1.0f / (d12_1 + d12_2);
    s.v[0].a = d12_1 * inv; s.v[1].a = d12_2 * inv; s.count = 2; return;
  }
  if (d13_1 > 0.0f && d13_2 > 0.0f && d123_2 <= 0.0f) {
    const float inv = 1.0f / (d13_1 + d13_2);
    s.v[0].a = d13_1 * inv; s.v[2].a = d13_2 * inv; s.count = 2; s.v[1] = s.v[2]; return;
  }
  if (d12_1 <= 0.0f && d23_2 <= 0.0f) { s.v[1].a = 1.0f; s.count = 1; s.v[0] = s.v[1]; return; }
  if (d13_1 <= 0.0f && d23_1 <= 0.0f) { s.v[2].a = 1.0f; s.count = 1; s.v[0] = s.v[2]; return; }
  if (d23_1 > 0.0f && d23_2 > 0.0f && d123_1 <= 0.0f) {
    const float inv = 1.0f / (d23_1 + d23_2);
    s.v[1].a = d23_1 * inv; s.v[2].a = d23_2 * inv; s.count = 2; s.v[0] = s.v[2]; return;
  }
  const float inv = 1.0f / (d123_1 + d123_2 + d123_3);
  s.v[0].a = d123_1 * inv; s.v[1].a = d123_2 * inv; s.v[2].a = d123_3 * inv; s.count = 3;
}

// b2Distance with useRadii = false: returns the distance and updates the simplex cache
__device__ __noinline__ float gjk_distance(SCache& cache, const Proxy& pA, const Proxy& pB, Xf xfB) {
  Simplex s;
  s.count = cache.count;
  for (int i = 0; i < s.count; ++i) {  // b2Simplex::ReadCache
    SV& v = s.v[i];
    v.iA = cache.iA[i];
    v.iB = cache.iB[i];
    v.wA = pA.v[v.iA];
    v.wB = xmul(xfB, pB.v[v.iB]);
    v.w = v.wB - v.wA;
    v.a = 0.0f;
  }
  if (s.count > 1) {
    const float metric1 = cache.metric, metric2 = simplex_metric(s);
    if (metric2 < 0.5f * metric1 || 2.0f * metric1 < metric2 || metric2 < kEpsilon) s.count = 0;
  }
  if (s.count == 0) {
    SV& v = s.v[0];
    v.iA = 0;
    v.iB = 0;
    v.wA = pA.v[0];
    v.wB = xmul(xfB, pB.v[0]);
    v.w = v.wB - v.wA;
    v.a = 1.0f;
    s.count = 1;
  }
  int saveA[3], saveB[3], iter = 0;
  while (iter < 20) {
    const int save_count = s.count;
    for (int i = 0; i < save_count; ++i) {
      saveA[i] = s.v[i].iA;
      saveB[i] = s.v[i].iB;
    }
    if (s.count == 2) simplex_solve2(s);
    else if (s.count == 3) simplex_solve3(s);
    if (s.count == 3) break;
    V2 d;  // b2Simplex::GetSearchDirection
    if (s.count == 1) {
      d = -s.v[0].w;
    } else {
      const V2 e12 = s.v[1].w - s.v[0].w;
      const float sgn = cross(e12, -s.v[0].w);
      d = sgn > 0.0f ? cross_sv(1.0f, e12) : cross_vs(e12, 1.0f);
    }
    if (dot(d, d) < kEpsilon * kEpsilon) break;
    SV& v = s.v[s.count];
    v.iA = proxy_support(pA, -d);
    v.wA = pA.v[v.iA];
    v.iB = proxy_support(pB, rmulT(xfB.q, d));
    v.wB = xmul(xfB, pB.v[v.iB]);
    v.w = v.wB - v.wA;
    ++iter;
    bool duplicate = false;
    for (int i = 0; i < save_count; ++i)
      if (v.iA == saveA[i] && v.iB == saveB[i]) {
        duplicate = true;
        break;
      }
    if (duplicate) break;
    ++s.count;
  }
  V2 a, b;  // GetWitnessPoints
  if (s.count == 1) {
    a = s.v[0].wA;
    b = s.v[0].wB;
  } else if (s.count == 2) {
    a = (s.v[0].a * s.v[0].wA) + (s.v[1].a * s.v[1].wA);
    b = (s.v[0].a * s.v[0].wB) + (s.v[1].a * s.v[1].wB);
  } else {
    a = ((s.v[0].a * s.v[0].wA) + (s.v[1].a * s.v[1].wA)) + (s.v[2].a * s.v[2].wA);
    b = a;
  }
  cache.metric = simplex_metric(s);  // WriteCache
  cache.count = s.count;
  for (int i = 0; i < s.count; ++i) {
    cache.iA[i] = s.v[i].iA;
    cache.iB[i] = s.v[i].iB;
  }
  return len(a - b);
}

// b2SeparationFunction (sweep A is the identity for every t)
struct SepFn {
  Sweep sB;
  int type;  // 0 points, 1 faceA, 2 faceB
  V2 local_point, axis;
};
DI void sep_init(SepFn& f, const SCache& cache, const Proxy& pA, const Proxy& pB, const Sweep& sB, float t1) {
  f.sB = sB;
  const Xf xfB = sweep_xf(sB, t1);
  if (cache.count == 1) {
    f.type = 0;
    const V2 pointA = pA.v[cache.iA[0]], pointB = xmul(xfB, pB.v[cache.iB[0]]);
    f.axis = pointB - pointA;
    normalize(f.axis);
  } else if (cache.iA[0] == cache.iA[1]) {
    f.type = 2;  // two points on B, one on A
    const V2 b1 = pB.v[cache.iB[0]], b2 = pB.v[cache.iB[1]];
    f.axis = cross_vs(b2 - b1, 1.0f);
    normalize(f.axis);
    const V2 normal = rmul(xfB.q, f.axis);
    f.local_point = 0.5f * (b1 + b2);
    const V2 pointB = xmul(xfB, f.local_point), pointA = pA.v[cache.iA[0]];
    const float s = dot(pointA - pointB, normal);
    if (s < 0.0f) f.axis = -f.axis;
  } else {
    f.type = 1;  // two points on A
    const V2 a1 = pA.v[cache.iA[0]], a2 = pA.v[cache.iA[1]];
    f.axis = cross_vs(a2 - a1, 1.0f);
    normalize(f.axis);
    const V2 normal = f.axis;
    f.local_point = 0.5f * (a1 + a2);
    const V2 pointA = f.local_point, pointB = xmul(xfB, pB.v[cache.iB[0]]);
    const float s = dot(pointB - pointA, normal);
    if (s < 0.0f) f.axis = -f.axis;
  }
}
DI float sep_find_min(const SepFn& f, const Proxy& pA, const Proxy& pB, int& iA, int& iB, float t) {
  const Xf xfB = sweep_xf(f.sB, t);
  if (f.type == 0) {
    iA = proxy_support(pA, f.axis);
    iB = proxy_support(pB, rmulT(xfB.q, -f.axis));
    const V2 pointA = pA.v[iA], pointB = xmul(xfB, pB.v[iB]);
    return dot(pointB - pointA, f.axis);
  } else if (f.type == 1) {
    const V2 normal = f.axis, pointA = f.local_point;
    iA = -1;
    iB = proxy_support(pB, rmulT(xfB.q, -normal));
    const V2 pointB = xmul(xfB, pB.v[iB]);
    return dot(pointB - pointA, normal);
  } else {
    const V2 normal = rmul(xfB.q, f.axis), pointB = xmul(xfB, f.local_point);
    iB = -1;
    iA = proxy_support(pA, -normal);
    const V2 pointA = pA.v[iA];
    return dot(pointA - pointB, normal);
  }
}
DI float sep_evaluate(const SepFn& f, const Proxy& pA, const Proxy& pB, int iA, int iB, float t) {
  const Xf xfB = sweep_xf(f.sB, t);
  if (f.type == 0) {
    const V2 pointA = pA.v[iA], pointB = xmul(xfB, pB.v[iB]);
    return dot(pointB - pointA, f.axis);
  } else if (f.type == 1) {
    const V2 normal = f.axis, pointA = f.local_point, pointB = xmul(xfB, pB.v[iB]);
    return dot(pointB - pointA, normal);
  } else {
    const V2 normal = rmul(xfB.q, f.axis), pointB = xmul(xfB, f.local_point), pointA = pA.v[iA];
    return dot(pointA - pointB, normal);
  }
}

// b2TimeOfImpact with tMax = 1: returns the state (1 failed, 2 overlapped, 3 touching, 4 separated) and t
__device__ __noinline__ int time_of_impact(const Proxy& pA, const Proxy& pB, Sweep sB, float& t_out) {
  const float tMax = 1.0f;
  {  // b2Sweep::Normalize
    const float two_pi = 2.0f * kPi;
    const float d = two_pi * floorf(sB.a0 / two_pi);
    sB.a0 -= d;
    sB.a -= d;
  }
  const float total_radius = kPolyRadius + kPolyRadius;
  const float target = fmaxf(kLinearSlop, total_radius - 3.0f * kLinearSlop), tolerance = 0.25f * kLinearSlop;
  float t1 = 0.0f;
  int iter = 0, state = 0;
  t_out = tMax;
  SCache cache;
  cache.count = 0;
  for (;;) {
    const Xf xfB = sweep_xf(sB, t1);
    const float distance = gjk_distance(cache, pA, pB, xfB);
    if (distance <= 0.0f) { state = 2; t_out = 0.0f; break; }
    if (distance < target + tolerance) { state = 3; t_out = t1; break; }
    SepFn fcn;
    sep_init(fcn, cache, pA, pB, sB, t1);
    bool done = false;
    int push_back = 0;
    float t2 = tMax;
    for (;;) {
      int iA, iB;
      float s2 = sep_find_min(fcn, pA, pB, iA, iB, t2);
      if (s2 > target + tolerance) { state = 4; t_out = tMax; done = true; break; }
      if (s2 > target - tolerance) { t1 = t2; break; }
      float s1 = sep_evaluate(fcn, pA, pB, iA, iB, t1);
      if (s1 < target - tolerance) { state = 1; t_out = t1; done = true; break; }
      if (s1 <= target + tolerance) { state = 3; t_out = t1; done = true; break; }
      int root_iters = 0;
      float a1 = t1, a2 = t2;
      for (;;) {
        float t;
        if (root_iters & 1) t = a1 + (target - s1) * (a2 - a1) / (s2 - s1);
        else t = 0.5f * (a1 + a2);
        ++root_iters;
        const float s = sep_evaluate(fcn, pA, pB, iA, iB, t);
        if (fabsf(s - target) < tolerance) { t2 = t; break; }
        if (s > target) { a1 = t; s1 = s; } else { a2 = t; s2 = s; }
        if (root_iters == 50) break;
      }
      ++push_back;
      if (push_back == kMaxPolyVerts) break;
    }
    ++iter;
    if (done) break;
    if (iter == 20) { state = 1; t_out = t1; break; }
  }
  return state;
}

// b2Contact::Update of list slot k: re-enable, evaluate the manifold at the body's current transform, carry the impulses of
// matching feature ids, Begin/EndContact
DI void contact_update(Lander& L, int k) {
  Contact& c = L.ct[k];
  const int dyn = c.pair / kNE, e = c.pair % kNE;
  MPoint old[2] = {c.pt[0], c.pt[1]};
  const int old_count = c.count, was = c.touching;
  c.enabled = 1;
  collide_edge_polygon(c, edge_v1(L, e), edge_v2(L, e), g_model.poly[dyn], L.b[dyn].xf);
  const int touching = c.count > 0;
  for (int i = 0; i < c.count; ++i) {
    MPoint& mp = c.pt[i];
    mp.ni = 0.0f;
    mp.ti = 0.0f;
    for (int j = 0; j < old_count; ++j)
      if (old[j].id == mp.id) {
        mp.ni = old[j].ni;
        mp.ti = old[j].ti;
        break;
      }
  }
  c.touching = touching;
  if (!was && touching) begin_contact(L, dyn);
  if (was && !touching) end_contact(L, dyn);
}

// b2Body::SynchronizeFixtures + b2DynamicTree::MoveProxy of dynamic body d; true if its fat AABB moved
DI bool sync_fixtures(Lander& L, int d) {
  const Body& b = L.b[d];
  Xf xf1;
  xf1.q = rot_set(b.a0);
  xf1.p = b.c0 - rmul(xf1.q, g_model.local_center[d]);
  const Aabb a1 = poly_aabb(g_model.poly[d], xf1), a2 = poly_aabb(g_model.poly[d], b.xf);
  const Aabb comb{vmin(a1.lo, a2.lo), vmax(a1.hi, a2.hi)};
  const V2 disp = b.xf.p - xf1.p;
  if (aabb_contains(L.fat[d], comb)) return false;
  Aabb fb = fatten(comb);
  const V2 dd = kAabbMul * disp;
  if (dd.x < 0.0f) fb.lo.x += dd.x; else fb.hi.x += dd.x;
  if (dd.y < 0.0f) fb.lo.y += dd.y; else fb.hi.y += dd.y;
  L.fat[d] = fb;
  return true;
}

// b2Island::SolveTOI for the island {moon, body dyn} with the contact slots isl[0..n) (isl[0] is the TOI contact): TOI position
// solve (<= 20 iterations, Baumgarte 0.75), leap of faith, 180 velocity iterations without warm starting and without
// joints, position integration over the rest of the step
__device__ __noinline__ void solve_toi_island(Lander& L, int dyn, const int* isl, int n, float h) {
  const Model& M = g_model;
  Body& B = L.b[dyn];
  const float mB = M.inv_mass[dyn], iB = M.inv_I[dyn];
  const V2 lcB = M.local_center[dyn];
  V2 cB = B.c, vB = B.v;
  float aB = B.a, wB = B.w;
  VC vcs[kMaxContacts];
  for (int k = 0; k < n; ++k) {  // b2ContactSolver constructor, warmStarting = false
    VC& vc = vcs[k];
    const Contact& c = L.ct[isl[k]];
    vc.slot = isl[k];
    vc.ib = dyn;
    vc.friction = c.friction;
    vc.count = vc.pos_count = c.count;
    vc.type = c.type;
    vc.local_normal = c.local_normal;
    vc.local_point = c.local_point;
    for (int j = 0; j < 2; ++j) {
      vc.p[j].ni = 0.0f;
      vc.p[j].ti = 0.0f;
      vc.lpts[j] = c.pt[j].lp;
    }
  }
  for (int it = 0; it < 20; ++it) {  // SolveTOIPositionConstraints
    float min_sep = 0.0f;
    for (int k = 0; k < n; ++k) {
      const VC& vc = vcs[k];
      for (int j = 0; j < vc.pos_count; ++j) {
        Xf xfB;
        xfB.q = rot_set(aB);
        xfB.p = cB - rmul(xfB.q, lcB);
        V2 normal, point;
        float sep;
        if (vc.type == 1) {
          normal = vc.local_normal;
          const V2 clip = xmul(xfB, vc.lpts[j]);
          sep = dot(clip - vc.local_point, normal) - kPolyRadius - kPolyRadius;
          point = clip;
        } else {
          normal = rmul(xfB.q, vc.local_normal);
          const V2 plane = xmul(xfB, vc.local_point), clip = vc.lpts[j];
          sep = dot(clip - plane, normal) - kPolyRadius - kPolyRadius;
          point = clip;
          normal = -normal;
        }
        const V2 rB = point - cB;
        min_sep = fminf(min_sep, sep);
        const float C = clampf(kToiBaumgarte * (sep + kLinearSlop), -kMaxLinCorr, 0.0f);
        const float rnB = cross(rB, normal);
        const float K = mB + iB * rnB * rnB;
        const float impulse = K > 0.0f ? -C / K : 0.0f;
        const V2 Pi = impulse * normal;
        cB = cB + mB * Pi;
        aB += iB * cross(rB, Pi);
      }
    }
    if (min_sep >= -1.5f * kLinearSlop) break;
  }
  B.c0 = cB;  // leap of faith to the new safe state (the moon's sweep does not change)
  B.a0 = aB;
  for (int k = 0; k < n; ++k) {  // InitializeVelocityConstraints
    VC& vc = vcs[k];
    Xf xfB;
    xfB.q = rot_set(aB);
    xfB.p = cB - rmul(xfB.q, lcB);
    V2 pts[2];
    if (vc.type == 1) {
      vc.normal = vc.local_normal;
      const V2 plane = vc.local_point;
      for (int j = 0; j < vc.count; ++j) {
        const V2 clip = xmul(xfB, vc.lpts[j]);
        const V2 cA = clip + (kPolyRadius - dot(clip - plane, vc.normal)) * vc.normal;
        const V2 cBp = clip - kPolyRadius * vc.normal;
        pts[j] = 0.5f * (cA + cBp);
      }
    } else {
      const V2 nrm = rmul(xfB.q, vc.local_normal);
      const V2 plane = xmul(xfB, vc.local_point);
      for (int j = 0; j < vc.count; ++j) {
        const V2 clip = vc.lpts[j];
        const V2 cBp = clip + (kPolyRadius - dot(clip - plane, nrm)) * nrm;
        const V2 cA = clip - kPolyRadius * nrm;
        pts[j] = 0.5f * (cA + cBp);
      }
      vc.normal = -nrm;
    }
    for (int j = 0; j < vc.count; ++j) {
      VCP& p = vc.p[j];
      p.rB = pts[j] - cB;
      const float rnB = cross(p.rB, vc.normal);
      const float kN = mB + iB * rnB * rnB;
      p.normal_mass = kN > 0.0f ? 1.0f / kN : 0.0f;
      const V2 tangent = cross_vs(vc.normal, 1.0f);
      const float rtB = cross(p.rB, tangent);
      const float kT = mB + iB * rtB * rtB;
      p.tangent_mass = kT > 0.0f ? 1.0f / kT : 0.0f;
    }
    if (vc.count == 2) {
      const float rn1B = cross(vc.p[0].rB, vc.normal), rn2B = cross(vc.p[1].rB, vc.normal);
      const float k11 = mB + iB * rn1B * rn1B, k22 = mB + iB * rn2B * rn2B, k12 = mB + iB * rn1B * rn2B;
      if (k11 * k11 < 1000.0f * (k11 * k22 - k12 * k12)) {
        vc.k00 = k11; vc.k01 = k12; vc.k11 = k22;
        float det = k11 * k22 - k12 * k12;
        if (det != 0.0f) det = 1.0f / det;
        vc.n00 = det * k22; vc.n10 = -det * k12; vc.n01 = -det * k12; vc.n11 = det * k11;
      } else {
        vc.count = 1;
      }
    }
  }
  for (int it = 0; it < 180; ++it) {  // SolveVelocityConstraints: contacts only
    // Exact early exit: one sweep is a deterministic function of (vB, wB, accumulated impulses).  If a sweep leaves all of
    // them bit-identical, every later sweep would too -- the remaining iterations are no-ops and can be skipped without
    // changing a single bit (checked against the oracle, which always runs all 180).  Most TOI sub-steps (one body, one or
    // two manifolds, no joints, no warm start) reach that fixed point within ~10 sweeps.
    const V2 v_before = vB;
    const float w_before = wB;
    bool impulses_changed = false;
    for (int k = 0; k < n; ++k) {
      VC& vc = vcs[k];
      const V2 normal = vc.normal, tangent = cross_vs(normal, 1.0f);
      for (int j = 0; j < vc.count; ++j) {
        VCP& p = vc.p[j];
        const V2 dv = vB + cross_sv(wB, p.rB);
        const float vt = dot(dv, tangent) - 0.0f;
        float lambda = p.tangent_mass * (-vt);
        const float maxf = vc.friction * p.ni;
        const float newi = clampf(p.ti + lambda, -maxf, maxf);
        lambda = newi - p.ti;
        impulses_changed |= newi != p.ti;
        p.ti = newi;
        const V2 Pi = lambda * tangent;
        vB = vB + mB * Pi;
        wB += iB * cross(p.rB, Pi);
      }
      if (vc.count == 1) {
        VCP& p = vc.p[0];
        const V2 dv = vB + cross_sv(wB, p.rB);
        const float vn = dot(dv, normal);
        float lambda = -p.normal_mass * (vn - 0.0f);
        const float newi = fmaxf(p.ni + lambda, 0.0f);
        lambda = newi - p.ni;
        impulses_changed |= newi != p.ni;
        p.ni = newi;
        const V2 Pi = lambda * normal;
        vB = vB + mB * Pi;
        wB += iB * cross(p.rB, Pi);
      } else {
        VCP &c1 = vc.p[0], &c2 = vc.p[1];
        const float ax = c1.ni, ay = c2.ni;
        const V2 dv1 = vB + cross_sv(wB, c1.rB), dv2 = vB + cross_sv(wB, c2.rB);
        float vn1 = dot(dv1, normal), vn2 = dot(dv2, normal);
        float bx = vn1 - 0.0f, by = vn2 - 0.0f;
        bx -= vc.k00 * ax + vc.k01 * ay;
        by -= vc.k01 * ax + vc.k11 * ay;
        float xx, xy;
        bool solved = false;
        xx = -(vc.n00 * bx + vc.n10 * by);
        xy = -(vc.n01 * bx + vc.n11 * by);
        if (xx >= 0.0f && xy >= 0.0f) solved = true;
        if (!solved) {
          xx = -c1.normal_mass * bx;
          xy = 0.0f;
          vn2 = vc.k01 * xx + by;
          if (xx >= 0.0f && vn2 >= 0.0f) solved = true;
        }
        if (!solved) {
          xx = 0.0f;
          xy = -c2.normal_mass * by;
          vn1 = vc.k01 * xy + bx;
          if (xy >= 0.0f && vn1 >= 0.0f) solved = true;
        }
        if (!solved) {
          xx = 0.0f;
          xy = 0.0f;
          if (bx >= 0.0f && by >= 0.0f) solved = true;
        }
        if (solved) {
          const float dx = xx - ax, dy = xy - ay;
          const V2 P1 = dx * normal, P2 = dy * normal;
          vB = vB + mB * (P1 + P2);
          wB += iB * (cross(c1.rB, P1) + cross(c2.rB, P2));
          impulses_changed |= (xx != c1.ni) | (xy != c2.ni);
          c1.ni = xx;
          c2.ni = xy;
        }
      }
    }
    if (!impulses_changed && vB.x == v_before.x && vB.y == v_before.y && wB == w_before) break;
  }
  // the TOI impulses are not stored for warm starting; integrate positions over the rest of the step
  const V2 tr = h * vB;
  if (dot(tr, tr) > kMaxTranslation * kMaxTranslation) {
    const float ratio = kMaxTranslation / len(tr);
    vB = ratio * vB;
  }
  const float rotn = h * wB;
  if (rotn * rotn > kMaxRotation * kMaxRotation) {
    const float ratio = kMaxRotation / fabsf(rotn);
    wB *= ratio;
  }
  cB = cB + h * vB;
  aB += h * wB;
  B.c = cB; B.a = aB; B.v = vB; B.w = wB;
  sync_transform(B, lcB);
}

// b2World::SolveTOI(step) with m_stepComplete = true on entry (no sub-stepping mode); the island is awake
// Shortcut around b2TimeOfImpact (restated in oracle/lunar_lander.c: toi_clearly_separated, which counts how often it
// applies and checks that b2TimeOfImpact answers alpha = 1 every time): if every vertex of the polygon stays beside the
// edge's line, or beyond one of the segment's ends along it, by more than the margin during the whole sweep, no point of
// the polygon comes within the TOI target distance (0.005 + 0.00125) of the edge, so b2TimeOfImpact cannot return
// e_touching and SolveTOI's alpha is 1 whatever the root finder does.  The sweep is bounded from the end pose (the body's
// transform): a vertex at sweep time t lies within |c - c0| (projected) + r_max |a - a0| of its end position.  Covers
// ~40 % of the evaluations of the random-action steady state.
constexpr float kToiClearMargin = 0.05f, kToiClearRmax = 0.8f;
DI bool toi_clearly_separated(V2 e1, V2 e2, const Poly& p, const Body& b) {
  const V2 d = e2 - e1;
  const float ln = len(d);
  if (!(ln > 1e-3f)) return false;
  const V2 n = mk(d.y / ln, -d.x / ln), u = mk(d.x / ln, d.y / ln);
  const float da = fabsf(b.a - b.a0);
  if (!(da < 0.5f)) return false;
  const V2 dc = b.c - b.c0;
  const float rot = kToiClearRmax * da + kToiClearMargin;
  const float slack = fabsf(dot(n, dc)) + rot, slack_u = fabsf(dot(u, dc)) + rot;
  float lo = 1e30f, hi = -1e30f, ulo = 1e30f, uhi = -1e30f;
  for (int i = 0; i < p.count; ++i) {
    const V2 r = xmul(b.xf, p.v[i]) - e1;
    const float sd = dot(n, r), su = dot(u, r);
    lo = fminf(lo, sd);
    hi = fmaxf(hi, sd);
    ulo = fminf(ulo, su);
    uhi = fmaxf(uhi, su);
  }
  return lo > slack || hi < -slack || ulo > ln + slack_u || uhi < -slack_u;
}

__device__ __noinline__ void solve_toi(Lander& L, float dt) {
  for (int d = 0; d < kND; ++d) L.b[d].alpha0 = 0.0f;
  float moon_alpha0 = 0.0f;
  for (int k = 0; k < L.nct; ++k) {
    L.ct[k].toi_flag = 0;
    L.ct[k].toi_count = 0;
    L.ct[k].toi = 1.0f;
  }
  for (;;) {
    int min_k = -1;
    float min_alpha = 1.0f;
    for (int k = 0; k < L.nct; ++k) {  // world contact list, most recent first
      Contact& c = L.ct[k];
      if (!c.enabled) continue;
      if (c.toi_count > kMaxSubSteps) continue;
      float alpha = 1.0f;
      if (c.toi_flag) {
        alpha = c.toi;
      } else {
        const int dyn = c.pair / kNE, e = c.pair % kNE;
        Body& bB = L.b[dyn];
        float alpha0 = moon_alpha0;  // put the sweeps onto the same time interval
        if (moon_alpha0 < bB.alpha0) {
          alpha0 = bB.alpha0;
          moon_alpha0 = alpha0;  // b2Sweep::Advance of a sweep with c0 == c, a0 == a
        } else if (bB.alpha0 < moon_alpha0) {
          alpha0 = moon_alpha0;
          Sweep s = body_sweep(bB, g_model.local_center[dyn]);
          sweep_advance(s, alpha0);
          body_set_sweep(bB, s);
        }
        if (toi_clearly_separated(edge_v1(L, e), edge_v2(L, e), g_model.poly[dyn], bB)) {
          alpha = 1.0f;
        } else {
          Proxy pA, pB;
          pA.v[0] = edge_v1(L, e);
          pA.v[1] = edge_v2(L, e);
          pA.count = 2;
          pB.count = g_model.poly[dyn].count;
          for (int i = 0; i < pB.count; ++i) pB.v[i] = g_model.poly[dyn].v[i];
          float beta;
          const int state = time_of_impact(pA, pB, body_sweep(bB, g_model.local_center[dyn]), beta);
          alpha = state == 3 ? fminf(alpha0 + (1.0f - alpha0) * beta, 1.0f) : 1.0f;
        }
        c.toi = alpha;
        c.toi_flag = 1;
      }
      if (alpha < min_alpha) {
        min_k = k;
        min_alpha = alpha;
      }
    }
    if (min_k < 0 || 1.0f - 10.0f * kEpsilon < min_alpha) break;  // no more TOI events
    Contact& mc = L.ct[min_k];
    const int dyn = mc.pair / kNE;
    Body& bB = L.b[dyn];
    const V2 lcB = g_model.local_center[dyn];
    const float moon_backup = moon_alpha0;
    const Sweep backup = body_sweep(bB, lcB);
    moon_alpha0 = min_alpha;  // bA->Advance(minAlpha) on the static body
    {                         // b2Body::Advance
      Sweep s = backup;
      sweep_advance(s, min_alpha);
      s.c = s.c0;
      s.a = s.a0;
      body_set_sweep(bB, s);
      sync_transform(bB, lcB);
    }
    contact_update(L, min_k);  // the TOI contact likely has some new contact points
    mc.toi_flag = 0;
    ++mc.toi_count;
    if (!mc.enabled || !mc.touching) {  // not solid: restore the sweeps
      mc.enabled = 0;
      moon_alpha0 = moon_backup;
      body_set_sweep(bB, backup);
      sync_transform(bB, lcB);
      continue;
    }
    // island: the TOI contact, then the other contacts of bB (most recent first) that touch at the advanced pose
    int isl[kMaxContacts], ni = 0;
    isl[ni++] = min_k;
    for (int k = 0; k < L.nct; ++k) {
      if (k == min_k || L.ct[k].pair / kNE != dyn) continue;
      contact_update(L, k);  // other = the moon, already in the island: not advanced
      if (!L.ct[k].enabled || !L.ct[k].touching) continue;
      isl[ni++] = k;
    }
    solve_toi_island(L, dyn, isl, ni, (1.0f - min_alpha) * dt);
    bool moved[kND] = {false, false, false};
    moved[dyn] = sync_fixtures(L, dyn);
    for (int k = 0; k < L.nct; ++k)  // invalidate all contact TOIs on this displaced body
      if (L.ct[k].pair / kNE == dyn) L.ct[k].toi_flag = 0;
    find_new_contacts(L, moved);
  }
}

// b2World::Step(1/50, 180, 60): new-fixture pairs, Collide, Solve (+ SynchronizeFixtures / FindNewContacts), SolveTOI,
// ClearForces
DI void world_step(Lander& L, float dt, float dt_ratio, float gravity, bool first_step) {
  bool moved[kND] = {true, true, true};
  if (first_step) find_new_contacts(L, moved);  // e_newFixture
  collide(L);
  if (L.awake) {
    solve_island(L, dt, dt_ratio, gravity);
    for (int d = kND - 1; d >= 0; --d) moved[d] = sync_fixtures(L, d);
    find_new_contacts(L, moved);
  }
  if (L.awake) solve_toi(L, dt);  // m_continuousPhysics; a sleeping island has no active body
  L.force = mk(0.0f, 0.0f);  // ClearForces
  L.torque = 0.0f;
}

// ---- kernel arguments / global layout -------------------------------------------------------------------------------------
struct LanderArgs {
  int64_t n, env_offset;
  int32_t max_steps, mode, rng_mode;
  uint64_t philox_seed, call_counter;
  float gravity;
  int32_t continuous, enable_wind;
  double wind_power, turbulence_power;
  int32_t* __restrict__ wind;        // [2][n] wind_idx, torque_idx (enable_wind)
  int64_t* __restrict__ u32buf;      // [n] PCG64's one-word 32-bit buffer: bit 32 = valid (enable_wind, numpy RNG)
  float* __restrict__ bodies;        // [21][n]
  float* __restrict__ joints;        // [8][n]
  float* __restrict__ terrain;       // [11][n] smooth_y
  float* __restrict__ fat;           // [12][n]
  uint32_t* __restrict__ contacts;   // [kMaxContacts * kSlotWords][n]
  int32_t* __restrict__ flags;       // [n]
  double* __restrict__ prev_shaping; // [n]
  int32_t* __restrict__ ctrl;
  uint64_t* __restrict__ rng;
  float* __restrict__ obs;           // [n][8]
  double* __restrict__ reward;
  uint8_t* __restrict__ term;
  uint8_t* __restrict__ trunc;
  float* __restrict__ final_obs;
  const void* __restrict__ actions;
  const uint8_t* __restrict__ mask;
};

// flags word: bit0 awake, bit1 game_over, bit2/3 leg contact, bits 4-5 / 6-7 joint limit states, bits 8-11 n contacts,
// bit 12 contact-list overflow (sticky)
DI void load_state(const LanderArgs& a, int64_t i, Lander& L) {
  const int64_t n = a.n;
#pragma unroll
  for (int b = 0; b < kND; ++b) {
    Body& B = L.b[b];
    B.c = mk(a.bodies[(7 * b + 0) * n + i], a.bodies[(7 * b + 1) * n + i]);
    B.a = a.bodies[(7 * b + 2) * n + i];
    B.v = mk(a.bodies[(7 * b + 3) * n + i], a.bodies[(7 * b + 4) * n + i]);
    B.w = a.bodies[(7 * b + 5) * n + i];
    B.sleep = a.bodies[(7 * b + 6) * n + i];
    B.c0 = B.c;
    B.a0 = B.a;
    sync_transform(B, g_model.local_center[b]);
  }
  const int32_t f = a.flags[i];
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    L.j[k].ix = a.joints[(4 * k + 0) * n + i];
    L.j[k].iy = a.joints[(4 * k + 1) * n + i];
    L.j[k].iz = a.joints[(4 * k + 2) * n + i];
    L.j[k].motor = a.joints[(4 * k + 3) * n + i];
    L.j[k].limit_state = (f >> (4 + 2 * k)) & 3;
  }
#pragma unroll
  for (int e = 0; e < 11; ++e) L.smooth[e] = a.terrain[e * n + i];
#pragma unroll
  for (int d = 0; d < kND; ++d)
    L.fat[d] = Aabb{mk(a.fat[(4 * d + 0) * n + i], a.fat[(4 * d + 1) * n + i]),
                    mk(a.fat[(4 * d + 2) * n + i], a.fat[(4 * d + 3) * n + i])};
  L.awake = f & 1;
  L.game_over = (f >> 1) & 1;
  L.leg_contact[0] = (f >> 2) & 1;
  L.leg_contact[1] = (f >> 3) & 1;
  L.nct = (f >> 8) & 15;
  L.overflow = (f >> 12) & 1;
  L.force = mk(0.0f, 0.0f);
  L.torque = 0.0f;
  L.wind_idx = a.enable_wind ? a.wind[i] : 0;
  L.torque_idx = a.enable_wind ? a.wind[n + i] : 0;
  L.prev_shaping = a.prev_shaping[i];
  for (int k = 0; k < L.nct; ++k) {
    const uint32_t* w = a.contacts + (int64_t)k * kSlotWords * n + i;
    Contact& c = L.ct[k];
    const uint32_t hd = w[0];
    c.pair = hd & 0xff;
    c.touching = (hd >> 8) & 1;
    c.type = (hd >> 9) & 3;
    c.count = (hd >> 11) & 3;
    c.enabled = (hd >> 13) & 1;
    c.friction = __uint_as_float(w[1 * n]);
    c.local_normal = mk(__uint_as_float(w[2 * n]), __uint_as_float(w[3 * n]));
    c.local_point = mk(__uint_as_float(w[4 * n]), __uint_as_float(w[5 * n]));
#pragma unroll
    for (int p = 0; p < 2; ++p) {
      c.pt[p].lp = mk(__uint_as_float(w[(6 + 5 * p) * n]), __uint_as_float(w[(7 + 5 * p) * n]));
      c.pt[p].ni = __uint_as_float(w[(8 + 5 * p) * n]);
      c.pt[p].ti = __uint_as_float(w[(9 + 5 * p) * n]);
      c.pt[p].id = w[(10 + 5 * p) * n];
    }
  }
}

DI void store_state(const LanderArgs& a, int64_t i, const Lander& L) {
  const int64_t n = a.n;
#pragma unroll
  for (int b = 0; b < kND; ++b) {
    const Body& B = L.b[b];
    a.bodies[(7 * b + 0) * n + i] = B.c.x;
    a.bodies[(7 * b + 1) * n + i] = B.c.y;
    a.bodies[(7 * b + 2) * n + i] = B.a;
    a.bodies[(7 * b + 3) * n + i] = B.v.x;
    a.bodies[(7 * b + 4) * n + i] = B.v.y;
    a.bodies[(7 * b + 5) * n + i] = B.w;
    a.bodies[(7 * b + 6) * n + i] = B.sleep;
  }
  int32_t f = (L.awake & 1) | ((L.game_over & 1) << 1) | ((L.leg_contact[0] & 1) << 2) | ((L.leg_contact[1] & 1) << 3) |
              ((L.j[0].limit_state & 3) << 4) | ((L.j[1].limit_state & 3) << 6) | ((L.nct & 15) << 8) |
              ((L.overflow & 1) << 12);
  a.flags[i] = f;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    a.joints[(4 * k + 0) * n + i] = L.j[k].ix;
    a.joints[(4 * k + 1) * n + i] = L.j[k].iy;
    a.joints[(4 * k + 2) * n + i] = L.j[k].iz;
    a.joints[(4 * k + 3) * n + i] = L.j[k].motor;
  }
#pragma unroll
  for (int d = 0; d < kND; ++d) {
    a.fat[(4 * d + 0) * n + i] = L.fat[d].lo.x;
    a.fat[(4 * d + 1) * n + i] = L.fat[d].lo.y;
    a.fat[(4 * d + 2) * n + i] = L.fat[d].hi.x;
    a.fat[(4 * d + 3) * n + i] = L.fat[d].hi.y;
  }
  a.prev_shaping[i] = L.prev_shaping;
  if (a.enable_wind) {
    a.wind[i] = L.wind_idx;
    a.wind[n + i] = L.torque_idx;
  }
  for (int k = 0; k < L.nct; ++k) {
    uint32_t* w = a.contacts + (int64_t)k * kSlotWords * n + i;
    const Contact& c = L.ct[k];
    w[0] = (uint32_t)c.pair | ((uint32_t)c.touching << 8) | ((uint32_t)c.type << 9) | ((uint32_t)c.count << 11) |
           ((uint32_t)c.enabled << 13);
    w[1 * n] = __float_as_uint(c.friction);
    w[2 * n] = __float_as_uint(c.local_normal.x);
    w[3 * n] = __float_as_uint(c.local_normal.y);
    w[4 * n] = __float_as_uint(c.local_point.x);
    w[5 * n] = __float_as_uint(c.local_point.y);
#pragma unroll
    for (int p = 0; p < 2; ++p) {
      w[(6 + 5 * p) * n] = __float_as_uint(c.pt[p].lp.x);
      w[(7 + 5 * p) * n] = __float_as_uint(c.pt[p].lp.y);
      w[(8 + 5 * p) * n] = __float_as_uint(c.pt[p].ni);
      w[(9 + 5 * p) * n] = __float_as_uint(c.pt[p].ti);
      w[(10 + 5 * p) * n] = c.pt[p].id;
    }
  }
}

// uniform double draws for one call: numpy stream or Philox block
struct Draws {
  Pcg64 g;
  bool numpy;
  uint64_t seed, env, counter;
  uint32_t k;
  DI double next() {
    if (numpy) return g.next_double();
    const uint4 r = philox_block(seed, env, counter, 16u + (k >> 1));
    const double u = (k & 1u) ? u53_to_double(r.z, r.w) : u53_to_double(r.x, r.y);
    ++k;
    return u;
  }
  DI double uniform(double lo, double hi) { return lo + (hi - lo) * next(); }
  // Generator.integers(low, high) for a range below 2^32: Lemire's multiply-and-reject on PCG64's buffered 32-bit words
  // (numpy: buffered_bounded_lemire_uint32 over pcg64_next32; oracle/np_rng.py bounded_uint32) -- low half of a fresh
  // 64-bit draw first, the high half on the next call
  bool has32;
  uint32_t word;
  DI uint32_t next32() {
    if (has32) {
      has32 = false;
      return word;
    }
    const uint64_t x = g.next_u64();
    has32 = true;
    word = (uint32_t)(x >> 32);
    return (uint32_t)x;
  }
  DI int64_t integers(int64_t low, int64_t high) {
    const uint32_t rng = (uint32_t)(high - low - 1), rng_excl = rng + 1u;
    if (!numpy) return low + (int64_t)(next() * (double)rng_excl);  // Philox mode: not a parity mode
    uint64_t m = (uint64_t)next32() * rng_excl;
    uint32_t leftover = (uint32_t)m;
    if (leftover < rng_excl) {
      const uint32_t threshold = (0xFFFFFFFFu - rng) % rng_excl;
      while (leftover < threshold) {
        m = (uint64_t)next32() * rng_excl;
        leftover = (uint32_t)m;
      }
    }
    return low + (int64_t)(m >> 32);
  }
};

// LunarLander.reset up to (not including) the embedded step(0): lunar_lander.py:321-445
__device__ __noinline__ void env_reset_state(Lander& L, Draws& D, float* terrain_out, int64_t n, int64_t i,
                                             bool enable_wind) {
  const Model& M = g_model;
  double height[12];
  for (int k = 0; k < 12; ++k) height[k] = D.uniform(0.0, kH / 2);
  const double helipad_y = kH / 4;
  for (int k = 3; k <= 7; ++k) height[k] = helipad_y;
  for (int k = 0; k < 11; ++k) {
    const int km = k - 1 < 0 ? 11 : k - 1;  // height[-1] is the last element
    L.smooth[k] = (float)(0.33 * (height[km] + height[k] + height[k + 1]));
    terrain_out[k * n + i] = L.smooth[k];
  }
  const double fx = D.uniform(-kInitialRandom, kInitialRandom);
  const double fy = D.uniform(-kInitialRandom, kInitialRandom);
  L.force = mk((float)fx, (float)fy);
  L.torque = 0.0f;
  L.wind_idx = L.torque_idx = 0;
  if (enable_wind) {  // lunar_lander.py:401-403
    L.wind_idx = (int32_t)D.integers(-9999, 9999);
    L.torque_idx = (int32_t)D.integers(-9999, 9999);
  }
#pragma unroll
  for (int b = 0; b < kND; ++b) {
    Body& B = L.b[b];
    B.a = B.a0 = M.init_angle[b];
    B.xf.p = M.init_pos[b];
    B.xf.q = rot_set(B.a);
    B.c = B.c0 = xmul(B.xf, M.local_center[b]);
    B.v = mk(0.0f, 0.0f);
    B.w = 0.0f;
    B.sleep = 0.0f;
    L.fat[b] = fatten(poly_aabb(M.poly[b], B.xf));
  }
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    L.j[k].ix = L.j[k].iy = L.j[k].iz = L.j[k].motor = 0.0f;
    L.j[k].limit_state = 0;
  }
  L.nct = 0;
  L.awake = 1;
  L.game_over = 0;
  L.leg_contact[0] = L.leg_contact[1] = 0;
}

struct StepOut {
  float obs[8];
  double reward;
  bool terminated;
};

// tanh in double from a fixed sequence of IEEE operations (the same one as oracle/lunar_lander.c: det_tanh)
DI double det_tanh(double x) {
  const double ax = fabs(x);
  double r;
  if (ax < 1e-3) {
    r = ax * (1.0 - (ax * ax) * (1.0 / 3.0));
  } else if (ax > 20.0) {
    r = 1.0;
  } else {
    const double t = 2.0 * ax;
    const double k = rint(t * 1.44269504088896338700e+00);
    const double y = (t - k * 6.93147180369123816490e-01) - k * 1.90821492927058770002e-10;
    double p = 1.0 / 6227020800.0;
    p = p * y + 1.0 / 479001600.0;
    p = p * y + 1.0 / 39916800.0;
    p = p * y + 1.0 / 3628800.0;
    p = p * y + 1.0 / 362880.0;
    p = p * y + 1.0 / 40320.0;
    p = p * y + 1.0 / 5040.0;
    p = p * y + 1.0 / 720.0;
    p = p * y + 1.0 / 120.0;
    p = p * y + 1.0 / 24.0;
    p = p * y + 1.0 / 6.0;
    p = p * y + 0.5;
    p = p * y + 1.0;
    p = p * y + 1.0;
    const double e = p * (double)(1ull << (int)k);  // 0 <= k <= 58
    r = (e - 1.0) / (e + 1.0);
  }
  return x < 0 ? -r : r;
}

struct EnvCfg {
  float gravity;
  bool continuous, enable_wind;
  double wind_power, turbulence_power;
};

// LunarLander.step: lunar_lander.py:471-665.  `action` for the discrete env; (c0, c1) = the continuous action already
// clipped to [-1, 1] in its own precision and widened (np.clip(action, -1, +1).astype(np.float64), :510)
__device__ __noinline__ void env_step(Lander& L, Draws& D, int action, double a0, double a1, const EnvCfg& cfg,
                                      bool first_step, bool has_prev, StepOut& out) {
  const Model& M = g_model;
  const float gravity = cfg.gravity;
  Body& lander = L.b[0];
  if (cfg.enable_wind && !(L.leg_contact[0] || L.leg_contact[1])) {  // lunar_lander.py:476-506
    constexpr double kPi = 3.141592653589793;
    double s1, s2, unused;
    det_sincos(0.02 * (double)L.wind_idx, &s1, &unused);
    det_sincos((kPi * 0.01) * (double)L.wind_idx, &s2, &unused);
    const double wind_mag = det_tanh(s1 + s2) * cfg.wind_power;
    L.wind_idx += 1;
    if (!L.awake) L.awake = 1;  // ApplyForceToCenter(..., wake=True)
    L.force = L.force + mk((float)wind_mag, 0.0f);
    det_sincos(0.02 * (double)L.torque_idx, &s1, &unused);
    det_sincos((kPi * 0.01) * (double)L.torque_idx, &s2, &unused);
    const double torque_mag = det_tanh(s1 + s2) * cfg.turbulence_power;
    L.torque_idx += 1;
    L.torque += (float)torque_mag;  // ApplyTorque
  }
  const bool fire_main = cfg.continuous ? (a0 > 0.0) : (action == 2);
  const bool fire_side = cfg.continuous ? (fabs(a1) > 0.5) : (action == 1 || action == 3);
  double tip0, tip1;
  det_sincos((double)lander.a, &tip0, &tip1);
  const double side0 = -tip1, side1 = tip0;
  double disp[2];
  disp[0] = D.uniform(-1.0, +1.0) / kScale;
  disp[1] = D.uniform(-1.0, +1.0) / kScale;
  double m_power = 0.0, s_power = 0.0;
  if (fire_main) {
    m_power = cfg.continuous ? (fmin(fmax(a0, 0.0), 1.0) + 1.0) * 0.5 : 1.0;  // 0.5..1.0
    const double ox = tip0 * (kMainEngineY / kScale + 2 * disp[0]) + side0 * disp[1];
    const double oy = -tip1 * (kMainEngineY / kScale + 2 * disp[0]) - side1 * disp[1];
    const double px = (double)lander.xf.p.x + ox, py = (double)lander.xf.p.y + oy;
    const V2 imp = mk((float)(-ox * kMainPower * m_power), (float)(-oy * kMainPower * m_power));
    const V2 pt = mk((float)px, (float)py);
    if (!L.awake) L.awake = 1;
    lander.v = lander.v + M.inv_mass[0] * imp;
    lander.w += M.inv_I[0] * cross(pt - lander.c, imp);
  }
  if (fire_side) {
    const double direction = cfg.continuous ? (a1 > 0 ? 1.0 : -1.0) : (double)(action - 2);  // np.sign(action[1])
    s_power = cfg.continuous ? fmin(fmax(fabs(a1), 0.5), 1.0) : 1.0;
    const double ox = tip0 * disp[0] + side0 * (3 * disp[1] + direction * kSideEngineAway / kScale);
    const double oy = -tip1 * disp[0] - side1 * (3 * disp[1] + direction * kSideEngineAway / kScale);
    const double px = (double)lander.xf.p.x + ox - tip0 * 17 / kScale;
    const double py = (double)lander.xf.p.y + oy + tip1 * kSideEngineHeight / kScale;
    const V2 imp = mk((float)(-ox * kSidePower * s_power), (float)(-oy * kSidePower * s_power));
    const V2 pt = mk((float)px, (float)py);
    if (!L.awake) L.awake = 1;
    lander.v = lander.v + M.inv_mass[0] * imp;
    lander.w += M.inv_I[0] * cross(pt - lander.c, imp);
  }
  const float dt = (float)(1.0 / kFps);
  world_step(L, dt, first_step ? 0.0f : 50.0f * dt, gravity, first_step);
  const double posx = lander.xf.p.x, posy = lander.xf.p.y, velx = lander.v.x, vely = lander.v.y;
  const double helipad_y = kH / 4;
  double s[8];
  s[0] = (posx - kViewW / kScale / 2) / (kViewW / kScale / 2);
  s[1] = (posy - (helipad_y + kLegDown / kScale)) / (kViewH / kScale / 2);
  s[2] = velx * (kViewW / kScale / 2) / kFps;
  s[3] = vely * (kViewH / kScale / 2) / kFps;
  s[4] = (double)lander.a;
  s[5] = 20.0 * (double)lander.w / kFps;
  s[6] = L.leg_contact[0] ? 1.0 : 0.0;
  s[7] = L.leg_contact[1] ? 1.0 : 0.0;
  double reward = 0;
  const double shaping = -100 * sqrt(s[0] * s[0] + s[1] * s[1]) - 100 * sqrt(s[2] * s[2] + s[3] * s[3]) -
                         100 * fabs(s[4]) + 10 * s[6] + 10 * s[7];
  if (has_prev) reward = shaping - L.prev_shaping;
  L.prev_shaping = shaping;
  reward -= m_power * 0.30;
  reward -= s_power * 0.03;
  bool terminated = false;
  if (L.game_over || fabs(s[0]) >= 1.0) {
    terminated = true;
    reward = -100;
  }
  if (!L.awake) {
    terminated = true;
    reward = +100;
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) out.obs[k] = (float)s[k];
  out.reward = reward;
  out.terminated = terminated;
}

DI Draws make_draws(const LanderArgs& a, int64_t i, uint32_t stream_base) {
  Draws D;
  D.numpy = a.rng_mode == B2E_RNG_NUMPY;
  if (D.numpy) D.g = pcg64_load(a.rng, a.n, i);
  D.seed = a.philox_seed;
  D.env = (uint64_t)(a.env_offset + i);
  D.counter = a.call_counter;
  D.k = stream_base;
  D.has32 = false;
  D.word = 0;
  if (D.numpy && a.enable_wind) {
    const int64_t b = a.u32buf[i];
    D.has32 = (b >> 32) & 1;
    D.word = (uint32_t)b;
  }
  return D;
}
DI void store_draws(const LanderArgs& a, int64_t i, const Draws& D) {
  if (!D.numpy) return;
  pcg64_store_state(a.rng, i, D.g);
  if (a.enable_wind) a.u32buf[i] = (int64_t)D.word | ((int64_t)(D.has32 ? 1 : 0) << 32);
}
DI EnvCfg env_cfg(const LanderArgs& a) {
  EnvCfg c;
  c.gravity = a.gravity;
  c.continuous = a.continuous != 0;
  c.enable_wind = a.enable_wind != 0;
  c.wind_power = a.wind_power;
  c.turbulence_power = a.turbulence_power;
  return c;
}
// the action of env i: an integer in 0..3, or (continuous) two floats clipped to [-1, 1] in their own precision and widened
template <typename ActT>
DI void load_lander_action(const LanderArgs& a, int64_t i, int& action, double& a0, double& a1) {
  action = 0;
  a0 = a1 = 0.0;
  if constexpr (std::is_floating_point<ActT>::value) {
    const ActT* p = reinterpret_cast<const ActT*>(a.actions) + 2 * i;
    const ActT c0 = p[0] < (ActT)-1 ? (ActT)-1 : (p[0] > (ActT)1 ? (ActT)1 : p[0]);
    const ActT c1 = p[1] < (ActT)-1 ? (ActT)-1 : (p[1] > (ActT)1 ? (ActT)1 : p[1]);
    a0 = (double)c0;
    a1 = (double)c1;
  } else {
    action = min(max(load_action<ActT>(a.actions, i), 0), 3);
  }
}

DI void write_obs(float* __restrict__ obs, int64_t i, const StepOut& o) {
  float4* p = reinterpret_cast<float4*>(obs) + 2 * i;
  p[0] = make_float4(o.obs[0], o.obs[1], o.obs[2], o.obs[3]);
  p[1] = make_float4(o.obs[4], o.obs[5], o.obs[6], o.obs[7]);
}

// One thread per env.  Grouping envs by the code paths they will walk (into full or sparse warps) was measured slower or
// no faster on B200 at N=16384 (DESIGN.md section 4, profiles/r2_notes.md).
constexpr int kLanderBlock = 64;  // small CTAs: every SM gets work; the kernel is latency- not occupancy-bound

__global__ void __launch_bounds__(kLanderBlock) lunarlander_reset_kernel(const LanderArgs a) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  if (a.mask != nullptr && a.mask[i] == 0) return;
  Lander L;
  L.overflow = 0;
  L.prev_shaping = 0.0;
  Draws D = make_draws(a, i, 0);
  const EnvCfg cfg = env_cfg(a);
  env_reset_state(L, D, a.terrain, a.n, i, cfg.enable_wind);
  StepOut o;
  env_step(L, D, 0, 0.0, 0.0, cfg, true, false, o);  // return self.step(0 / [0, 0])[0] (lunar_lander.py:447)
  store_draws(a, i, D);
  store_state(a, i, L);
  a.ctrl[i] = 0;
  write_obs(a.obs, i, o);
}

template <typename ActT>
__global__ void __launch_bounds__(kLanderBlock) lunarlander_step_kernel(const LanderArgs a) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  const int32_t c = a.ctrl[i];
  int action;
  double a0, a1;
  load_lander_action<ActT>(a, i, action, a0, a1);
  Lander L;
  Draws D = make_draws(a, i, 0);
  const EnvCfg cfg = env_cfg(a);
  StepOut o;
  const bool is_reset = a.mode == B2E_AUTORESET_NEXT_STEP && ctrl_pending(c);
  if (is_reset) {
    L.overflow = 0;
    L.prev_shaping = 0.0;
    env_reset_state(L, D, a.terrain, a.n, i, cfg.enable_wind);
    action = 0;
    a0 = a1 = 0.0;
  } else {
    load_state(a, i, L);
  }
  env_step(L, D, action, a0, a1, cfg, is_reset, !is_reset, o);
  int32_t cn;
  if (is_reset) {  // sync_vector_env.py:279-284
    a.reward[i] = 0.0;
    a.term[i] = 0;
    a.trunc[i] = 0;
    cn = 0;
  } else {
    const int32_t elapsed = ctrl_elapsed(c) + 1;
    const bool trunc = a.max_steps > 0 && elapsed >= a.max_steps;
    a.reward[i] = o.reward;
    a.term[i] = o.terminated;
    a.trunc[i] = trunc;
    cn = elapsed;
    if (o.terminated || trunc) {
      if (a.mode == B2E_AUTORESET_NEXT_STEP) {
        cn |= kPending;
      } else if (a.mode == B2E_AUTORESET_SAME_STEP) {
        write_obs(a.final_obs, i, o);
        L.overflow = 0;
        L.prev_shaping = 0.0;
        env_reset_state(L, D, a.terrain, a.n, i, cfg.enable_wind);
        env_step(L, D, 0, 0.0, 0.0, cfg, true, false, o);
        cn = 0;
      }
    }
  }
  store_draws(a, i, D);
  store_state(a, i, L);
  a.ctrl[i] = cn;
  write_obs(a.obs, i, o);
}

// ---- host: model constants by the same float32 formulas Box2D uses (b2PolygonShape::Set / ComputeMass) --------------------
struct HV2 {
  float x, y;
};
void host_poly_mass(const Poly& p, float density, float& mass, V2& center_out, float& I_out) {
  float cx = 0, cy = 0, sx = 0, sy = 0, area = 0, I = 0;
  for (int i = 0; i < p.count; ++i) {
    sx += p.v[i].x;
    sy += p.v[i].y;
  }
  const float invc = 1.0f / (float)p.count;
  sx *= invc;
  sy *= invc;
  const float inv3 = 1.0f / 3.0f;
  for (int i = 0; i < p.count; ++i) {
    const V2 b = i + 1 < p.count ? p.v[i + 1] : p.v[0];
    const float e1x = p.v[i].x - sx, e1y = p.v[i].y - sy, e2x = b.x - sx, e2y = b.y - sy;
    const float D = e1x * e2y - e1y * e2x, tri = 0.5f * D;
    area += tri;
    cx += (tri * inv3) * (e1x + e2x);
    cy += (tri * inv3) * (e1y + e2y);
    const float intx2 = e1x * e1x + e2x * e1x + e2x * e2x, inty2 = e1y * e1y + e2y * e1y + e2y * e2y;
    I += (0.25f * inv3 * D) * (intx2 + inty2);
  }
  mass = density * area;
  const float inva = 1.0f / area;
  cx *= inva;
  cy *= inva;
  center_out.x = cx + sx;
  center_out.y = cy + sy;
  I_out = density * I;
  I_out += mass * ((center_out.x * center_out.x + center_out.y * center_out.y) - (cx * cx + cy * cy));
}

void build_model(Model& M) {
  memset(&M, 0, sizeof(M));
  // lander hull (lunar_lander.py:45, :377-379): b2PolygonShape::Set orders the convex hull CCW from the lowest
  // right-most vertex: (17,-10), (17,0), (14,17), (-14,17), (-17,0), (-17,-10), all / SCALE
  static const int hull[6][2] = {{17, -10}, {17, 0}, {14, 17}, {-14, 17}, {-17, 0}, {-17, -10}};
  Poly& P0 = M.poly[0];
  P0.count = 6;
  for (int i = 0; i < 6; ++i) {
    P0.v[i].x = (float)(hull[i][0] / kScale);
    P0.v[i].y = (float)(hull[i][1] / kScale);
  }
  for (int i = 0; i < 6; ++i) {
    const int i2 = i + 1 < 6 ? i + 1 : 0;
    const float ex = P0.v[i2].x - P0.v[i].x, ey = P0.v[i2].y - P0.v[i].y;
    float nx = 1.0f * ey, ny = -1.0f * ex;  // b2Cross(edge, 1.0f)
    const float l = sqrtf(nx * nx + ny * ny), inv = 1.0f / l;
    P0.n[i].x = nx * inv;
    P0.n[i].y = ny * inv;
  }
  {  // ComputeCentroid (reference point = origin)
    float cx = 0, cy = 0, area = 0;
    const float inv3 = 1.0f / 3.0f;
    for (int i = 0; i < 6; ++i) {
      const V2 p2 = P0.v[i], p3 = i + 1 < 6 ? P0.v[i + 1] : P0.v[0];
      const float e1x = p2.x - 0.0f, e1y = p2.y - 0.0f, e2x = p3.x - 0.0f, e2y = p3.y - 0.0f;
      const float D = e1x * e2y - e1y * e2x, tri = 0.5f * D;
      area += tri;
      cx += (tri * inv3) * ((0.0f + p2.x) + p3.x);
      cy += (tri * inv3) * ((0.0f + p2.y) + p3.y);
    }
    const float inva = 1.0f / area;
    P0.centroid.x = inva * cx;
    P0.centroid.y = inva * cy;
  }
  for (int k = 0; k < 2; ++k) {  // legs: SetAsBox(LEG_W/SCALE, LEG_H/SCALE) (:413)
    Poly& P = M.poly[1 + k];
    const float hx = (float)(kLegW / kScale), hy = (float)(kLegH / kScale);
    P.count = 4;
    P.v[0] = V2{-hx, -hy};
    P.v[1] = V2{hx, -hy};
    P.v[2] = V2{hx, hy};
    P.v[3] = V2{-hx, hy};
    P.n[0] = V2{0, -1};
    P.n[1] = V2{1, 0};
    P.n[2] = V2{0, 1};
    P.n[3] = V2{-1, 0};
    P.centroid = V2{0, 0};
  }
  const float density[3] = {5.0f, 1.0f, 1.0f};
  for (int b = 0; b < kND; ++b) {  // b2Body::ResetMassData for a one-fixture body
    float mass, I;
    V2 center;
    host_poly_mass(M.poly[b], density[b], mass, center, I);
    M.mass[b] = mass;
    M.inv_mass[b] = 1.0f / mass;
    V2 lc;
    lc.x = M.inv_mass[b] * (mass * center.x);
    lc.y = M.inv_mass[b] * (mass * center.y);
    I -= mass * (lc.x * lc.x + lc.y * lc.y);
    M.inv_I[b] = 1.0f / I;
    M.local_center[b] = lc;
  }
  M.edge_friction[0] = 0.2f;  // base edge: default fixture friction
  M.edge_x1[0] = 0.0f;
  M.edge_x2[0] = (float)kW;
  for (int i = 0; i < 10; ++i) {  // terrain chunks: chunk_x[i] = W / (CHUNKS - 1) * i (:345)
    M.edge_x1[i + 1] = (float)(kW / 10 * i);
    M.edge_x2[i + 1] = (float)(kW / 10 * (i + 1));
    M.edge_friction[i + 1] = 0.1f;
  }
  M.poly_friction[0] = 0.1f;
  M.poly_friction[1] = M.poly_friction[2] = 0.2f;
  const double initial_y = kViewH / kScale, initial_x = kViewW / kScale / 2;
  M.init_pos[0] = V2{(float)initial_x, (float)initial_y};
  M.init_angle[0] = 0.0f;
  for (int k = 0; k < 2; ++k) {
    const int i = k == 0 ? -1 : +1;
    M.init_pos[1 + k] = V2{(float)(initial_x - i * kLegAway / kScale), (float)initial_y};
    M.init_angle[1 + k] = (float)(i * 0.05);
    M.anchor_b[k] = V2{(float)(i * kLegAway / kScale), (float)(kLegDown / kScale)};
    M.ref_angle[k] = M.init_angle[1 + k] - M.init_angle[0];  // pybox2d default: bodyB.angle - bodyA.angle
    M.motor_speed[k] = (float)(+0.3 * i);
    if (i == -1) {
      M.lower[k] = (float)(+0.9 - 0.5);
      M.upper[k] = (float)+0.9;
    } else {
      M.lower[k] = (float)-0.9;
      M.upper[k] = (float)(-0.9 + 0.5);
    }
  }
  M.max_motor_torque = 40.0f;
}

int upload_model() {
  static bool done[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
  if (done[dev]) return 0;
  Model M;
  build_model(M);
  cudaError_t e = cudaMemcpyToSymbol(g_model, &M, sizeof(M));
  if (e != cudaSuccess) return cuda_status(e, "lunarlander model upload");
  done[dev] = true;
  return 0;
}

int fill(const b2e_batch* b, const b2e_lunarlander_cfg* cfg, const b2e_lunarlander_state* st, LanderArgs& a,
         const char* fn) {
  if (int e = check_batch(b, fn)) return e;
  if (!cfg || !st || !st->bodies || !st->joints || !st->terrain || !st->fat || !st->contacts || !st->flags ||
      !st->prev_shaping || !st->ctrl || (b->rng_mode == B2E_RNG_NUMPY && !st->rng)) {
    set_error("%s: null pointer in cfg/state", fn);
    return B2E_EINVAL;
  }
  if (cfg->enable_wind && (!st->wind || (b->rng_mode == B2E_RNG_NUMPY && !st->u32buf))) {
    set_error("%s: enable_wind needs state.wind (and state.u32buf with the numpy RNG)", fn);
    return B2E_EINVAL;
  }
  a = LanderArgs{};
  a.continuous = cfg->continuous != 0;
  a.enable_wind = cfg->enable_wind != 0;
  a.wind_power = cfg->wind_power;
  a.turbulence_power = cfg->turbulence_power;
  a.wind = st->wind;
  a.u32buf = st->u32buf;
  a.n = b->n;
  a.env_offset = b->env_offset;
  a.max_steps = b->max_episode_steps;
  a.mode = b->autoreset_mode;
  a.rng_mode = b->rng_mode;
  a.philox_seed = b->philox_seed;
  a.call_counter = b->call_counter;
  a.gravity = (float)cfg->gravity;
  a.bodies = st->bodies;
  a.joints = st->joints;
  a.terrain = st->terrain;
  a.fat = st->fat;
  a.contacts = st->contacts;
  a.flags = st->flags;
  a.prev_shaping = st->prev_shaping;
  a.ctrl = st->ctrl;
  a.rng = st->rng;
  return upload_model();
}

}  // namespace
}  // namespace b2e

using namespace b2e;

extern "C" int b2e_lunarlander_state_words(void) { return kMaxContacts * kSlotWords; }

extern "C" int b2e_lunarlander_reset(const b2e_batch* b, const b2e_lunarlander_cfg* cfg,
                                     const b2e_lunarlander_state* st, const uint8_t* mask, float* obs, void* stream) {
  LanderArgs a;
  if (int e = fill(b, cfg, st, a, "b2e_lunarlander_reset")) return e;
  if (!obs) {
    set_error("b2e_lunarlander_reset: obs is NULL");
    return B2E_EINVAL;
  }
  if (b->n == 0) return 0;
  a.mask = mask;
  a.obs = obs;
  lunarlander_reset_kernel<<<grid_for(b->n, kLanderBlock), kLanderBlock, 0, (cudaStream_t)stream>>>(a);
  return cuda_status(cudaGetLastError(), "b2e_lunarlander_reset");
}

extern "C" int b2e_lunarlander_step(const b2e_batch* b, const b2e_lunarlander_cfg* cfg, const b2e_lunarlander_state* st,
                                    const void* actions, float* obs, double* reward, uint8_t* terminated,
                                    uint8_t* truncated, float* final_obs, void* stream) {
  LanderArgs a;
  if (int e = fill(b, cfg, st, a, "b2e_lunarlander_step")) return e;
  if (!actions || !obs || !reward || !terminated || !truncated ||
      (b->autoreset_mode == B2E_AUTORESET_SAME_STEP && !final_obs)) {
    set_error("b2e_lunarlander_step: null pointer");
    return B2E_EINVAL;
  }
  if (b->n == 0) return 0;
  a.actions = actions;
  a.obs = obs;
  a.reward = reward;
  a.term = terminated;
  a.trunc = truncated;
  a.final_obs = final_obs;
  const unsigned grid = grid_for(b->n, kLanderBlock);
  cudaStream_t s = (cudaStream_t)stream;
  if (cfg->continuous) {  // actions [n][2] float32 / float64 in [-1, 1] (clipped in-kernel like the reference, :510)
    switch (b->action_dtype) {
      case B2E_ACT_F32: lunarlander_step_kernel<float><<<grid, kLanderBlock, 0, s>>>(a); break;
      case B2E_ACT_F64: lunarlander_step_kernel<double><<<grid, kLanderBlock, 0, s>>>(a); break;
      default: set_error("b2e_lunarlander_step: continuous=1 needs float32 / float64 actions, got dtype %d", b->action_dtype); return B2E_EINVAL;
    }
    return cuda_status(cudaGetLastError(), "b2e_lunarlander_step");
  }
  switch (b->action_dtype) {
    case B2E_ACT_I64: lunarlander_step_kernel<int64_t><<<grid, kLanderBlock, 0, s>>>(a); break;
    case B2E_ACT_I32: lunarlander_step_kernel<int32_t><<<grid, kLanderBlock, 0, s>>>(a); break;
    case B2E_ACT_U8: lunarlander_step_kernel<uint8_t><<<grid, kLanderBlock, 0, s>>>(a); break;
    default: set_error("b2e_lunarlander_step: action_dtype %d is not a discrete dtype", b->action_dtype); return B2E_EINVAL;
  }
  return cuda_status(cudaGetLastError(), "b2e_lunarlander_step");
}
