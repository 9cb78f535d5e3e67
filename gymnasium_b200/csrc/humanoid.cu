// humanoid.cu -- fused Humanoid-v5 step + TimeLimit + autoreset kernel (sm_100a): articulated-body forward dynamics with
// a PGS contact/limit solve, RK4 x frame_skip.  Two mappings of the same physics core: one thread per env (this file) and
// one warp per env with the working set in shared memory (humanoid_warp.cuh, the default); they agree bit for bit.
//
// Replaces, for a batch of n envs in one launch:
//   HumanoidEnv.step / _get_obs / _get_rew / reset_model   gymnasium/envs/mujoco/humanoid_v5.py:436-532
//   MujocoEnv.reset / set_state / _step_mujoco_simulation   gymnasium/envs/mujoco/mujoco_env.py:132-155, 172-187
//   the model                                               gymnasium/envs/mujoco/assets/humanoid.xml:1-121
//   TimeLimit / SyncVectorEnv autoreset as in cartpole.cu
// and, below the reference, the part of the third-party MuJoCo engine (pyproject.toml:45 -- not vendored in the reference
// tree) that this model exercises: mj_kinematics, mj_comPos, mj_crb, mj_factorM/mj_solveM (tree-sparse L^T D L),
// plane/sphere/capsule collision, joint-limit + pyramidal-contact constraint rows with solref/solimp impedance,
// mj_projectConstraint, mj_comVel, mj_passive, mj_rne, actuation (ctrl clamp, gear), PGS (<= 50 sweeps, warm start),
// RK4, mj_rnePostConstraint (cfrc_ext).  Written against MuJoCo's published pipeline; numeric parity with the real
// wheel is UNPINNED (not installable here) -- the checker is oracle/humanoid.c, which this kernel matches bit for bit,
// plus the reference's structural tests.
//
// Arithmetic: float64 like MuJoCo, one IEEE rounding per operation (--fmad=false), sin/cos from the fixed sequence shared
// with the oracle.  The physics core is __host__ __device__: the host runs it once at qpos0 to derive the compile-time
// constants MuJoCo stores in mjModel (body/dof invweight0, meaninertia).  Per-env working set (mass matrix, constraint
// Jacobian, A = J M^-1 J^T + R): thread-local memory (~36 KB/env) in the thread mapping, 24 KB of shared memory in the warp
// mapping; persistent state is 74 doubles per env in struct-of-arrays layout.  ~0.9 MFLOP fp64 per env-step; both
// mappings are bound by dependent-issue latency, not by FLOP/s or HBM (DESIGN.md section 4).
#include <atomic>
#include <assert.h>
#include <string.h>

#include "common.cuh"

namespace b2e {
namespace {

#define HD __host__ __device__ inline

constexpr int NB = 14, NQ = 24, NV = 23, NU = 17, NJ = 18, NG = 18, MAXCON = 12, MAXEFC = 24, MAXPAIR = 160;
constexpr double MINVAL = 1e-15, PI = 3.14159265358979323846;
constexpr int G_PLANE = 0, G_SPHERE = 2, G_CAPSULE = 3;

struct HModel {
  int parent[NB], body_jntadr[NB], body_jntnum[NB], body_dofadr[NB], body_dofnum[NB], body_lastdof[NB];
  double body_pos[NB][3], body_quat[NB][4], body_mass[NB], body_ipos[NB][3], body_inertia[NB][9];
  double subtree_mass[NB], body_invweight0[NB][2];
  int jnt_type[NJ], jnt_body[NJ], jnt_qposadr[NJ], jnt_dofadr[NJ];
  double jnt_pos[NJ][3], jnt_axis[NJ][3], jnt_range[NJ][2], jnt_stiffness[NJ];
  int dof_body[NV], dof_parent[NV];
  double dof_armature[NV], dof_damping[NV], dof_invweight0[NV];
  int geom_type[NG], geom_body[NG], geom_condim[NG];
  double geom_pos[NG][3], geom_mat[NG][9], geom_size[NG][2], geom_rbound[NG], geom_friction[NG];
  int act_dof[NU];
  double act_gear[NU];
  int ten_q[2][2], ten_v[2][2];
  double timestep, gravity[3], meaninertia, margin, solref[2], solimp[5], tolerance;
  int iterations, npair, pair_g1[MAXPAIR], pair_g2[MAXPAIR];
  double qpos0[NQ];
  // tables for the warp-per-env kernel
  int body_depth[NB];           // world 0, torso 1, ...
  int dof_chain_len[NV];        // number of ancestors of dof i
  int dof_chain[NV][13];        // ancestors of dof i, nearest first
  unsigned body_dofmask[NB];    // bit i set: dof i moves body b (ancestor-or-self of its last dof)
  int lvl_parents[7][3];        // bodies of depth lvl that have children (-1 padded)
  int children[NB][3];          // children of body b in descending index order (-1 padded)
};

struct Contact {
  int g1, g2, dim, efc_adr;
  double dist, pos[3], frame[9], mu;
};

struct HData {
  double qpos[NQ], qvel[NV], qacc_warmstart[NV], ctrl[NU];
  double xpos[NB][3], xquat[NB][4], xmat[NB][9], xipos[NB][3], xanchor[NJ][3], xaxis[NJ][3];
  double geom_xpos[NG][3], geom_xmat[NG][9];
  double subtree_com[NB][3], cinert[NB][10], cdof[NV][6], cdof_dot[NV][6], cvel[NB][6], cfrc_ext[NB][6];
  double qM[NV][NV], qLD[NV][NV], qLDiagInv[NV];
  double qfrc_bias[NV], qfrc_passive[NV], qfrc_actuator[NV], qfrc_smooth[NV], qacc_smooth[NV], qacc[NV], qfrc_constraint[NV];
  double ten_length[2], ten_velocity[2];
  int ncon, nefc, overflow;
  Contact con[MAXCON];
  double efc_J[MAXEFC][NV], efc_pos[MAXEFC], efc_margin[MAXEFC], efc_D[MAXEFC], efc_R[MAXEFC], efc_aref[MAXEFC],
      efc_b[MAXEFC], efc_force[MAXEFC], efc_diagApprox[MAXEFC];
  double efc_AR[MAXEFC][MAXEFC];
};

// ---- small helpers --------------------------------------------------------------------------------------------------------
HD void cp3(double* r, const double* a) { r[0] = a[0]; r[1] = a[1]; r[2] = a[2]; }
HD double dot3(const double* a, const double* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
HD void cross3(double* r, const double* a, const double* b) {
  const double x = a[1] * b[2] - a[2] * b[1], y = a[2] * b[0] - a[0] * b[2], z = a[0] * b[1] - a[1] * b[0];
  r[0] = x; r[1] = y; r[2] = z;
}
HD double norm3(const double* a) { return sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]); }
HD double normalize3(double* a) {
  const double n = norm3(a);
  if (n < MINVAL) { a[0] = 1; a[1] = 0; a[2] = 0; return n; }
  const double inv = 1.0 / n;
  a[0] *= inv; a[1] *= inv; a[2] *= inv;
  return n;
}
HD void mulmatvec3(double* r, const double* m, const double* v) {
  const double x = m[0] * v[0] + m[1] * v[1] + m[2] * v[2], y = m[3] * v[0] + m[4] * v[1] + m[5] * v[2],
               z = m[6] * v[0] + m[7] * v[1] + m[8] * v[2];
  r[0] = x; r[1] = y; r[2] = z;
}
HD void mulmat3(double* r, const double* a, const double* b) {
  double t[9];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) t[3 * i + j] = a[3 * i] * b[j] + a[3 * i + 1] * b[3 + j] + a[3 * i + 2] * b[6 + j];
  for (int k = 0; k < 9; ++k) r[k] = t[k];
}
// sin/cos from one fixed IEEE sequence (shared with oracle/humanoid.c: det_sincos)
HD void det_sincos(double x, double* sn, double* cs) {
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
HD void quat_mul(double* r, const double* a, const double* b) {
  const double t0 = a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3], t1 = a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2],
               t2 = a[0] * b[2] - a[1] * b[3] + a[2] * b[0] + a[3] * b[1], t3 = a[0] * b[3] + a[1] * b[2] - a[2] * b[1] + a[3] * b[0];
  r[0] = t0; r[1] = t1; r[2] = t2; r[3] = t3;
}
HD void quat_normalize(double* q) {
  const double n = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  if (n < MINVAL) { q[0] = 1; q[1] = q[2] = q[3] = 0; return; }
  const double inv = 1.0 / n;
  q[0] *= inv; q[1] *= inv; q[2] *= inv; q[3] *= inv;
}
HD void quat_axisangle(double* q, const double* axis, double angle) {
  double s, c;
  det_sincos(0.5 * angle, &s, &c);
  q[0] = c; q[1] = axis[0] * s; q[2] = axis[1] * s; q[3] = axis[2] * s;
}
HD void quat2mat(double* m, const double* q) {
  const double q00 = q[0] * q[0], q01 = q[0] * q[1], q02 = q[0] * q[2], q03 = q[0] * q[3];
  const double q11 = q[1] * q[1], q12 = q[1] * q[2], q13 = q[1] * q[3], q22 = q[2] * q[2], q23 = q[2] * q[3], q33 = q[3] * q[3];
  m[0] = q00 + q11 - q22 - q33; m[4] = q00 - q11 + q22 - q33; m[8] = q00 - q11 - q22 + q33;
  m[1] = 2 * (q12 - q03); m[2] = 2 * (q13 + q02); m[3] = 2 * (q12 + q03);
  m[5] = 2 * (q23 - q01); m[6] = 2 * (q13 - q02); m[7] = 2 * (q23 + q01);
}
HD void quat_rot(double* r, const double* q, const double* v) {
  double m[9];
  quat2mat(m, q);
  mulmatvec3(r, m, v);
}
HD double dot6(const double* a, const double* b) {
  return a[0] * b[0] + a[1] * b[1] + a[2] * b[2] + a[3] * b[3] + a[4] * b[4] + a[5] * b[5];
}
HD void mul_inert_vec(double* res, const double* i, const double* v) {
  res[0] = i[0] * v[0] + i[3] * v[1] + i[4] * v[2] - i[8] * v[4] + i[7] * v[5];
  res[1] = i[3] * v[0] + i[1] * v[1] + i[5] * v[2] + i[8] * v[3] - i[6] * v[5];
  res[2] = i[4] * v[0] + i[5] * v[1] + i[2] * v[2] - i[7] * v[3] + i[6] * v[4];
  res[3] = i[8] * v[1] - i[7] * v[2] + i[9] * v[3];
  res[4] = i[6] * v[2] - i[8] * v[0] + i[9] * v[4];
  res[5] = i[7] * v[0] - i[6] * v[1] + i[9] * v[5];
}

// ---- position stage: mj_kinematics, mj_comPos, tendons, mj_crb, mj_factorM ----------------------------------------------
HD void kinematics(const HModel& m, HData& d) {
  double* q = d.qpos;
  quat_normalize(q + 3);
  for (int k = 0; k < 3; ++k) { d.xpos[0][k] = 0; d.xipos[0][k] = 0; }
  d.xquat[0][0] = 1; d.xquat[0][1] = d.xquat[0][2] = d.xquat[0][3] = 0;
  for (int k = 0; k < 9; ++k) d.xmat[0][k] = (k % 4 == 0) ? 1.0 : 0.0;
  for (int b = 1; b < NB; ++b) {
    double xpos[3], xquat[4];
    if (m.body_jntnum[b] && m.jnt_type[m.body_jntadr[b]] == 0) {
      cp3(xpos, q);
      for (int k = 0; k < 4; ++k) xquat[k] = q[3 + k];
      const int j = m.body_jntadr[b];
      cp3(d.xanchor[j], xpos);
      d.xaxis[j][0] = 0; d.xaxis[j][1] = 0; d.xaxis[j][2] = 1;
    } else {
      const int p = m.parent[b];
      double t[3];
      mulmatvec3(t, d.xmat[p], m.body_pos[b]);
      for (int k = 0; k < 3; ++k) xpos[k] = d.xpos[p][k] + t[k];
      quat_mul(xquat, d.xquat[p], m.body_quat[b]);
      for (int jj = 0; jj < m.body_jntnum[b]; ++jj) {
        const int j = m.body_jntadr[b] + jj;
        double v[3];
        quat_rot(v, xquat, m.jnt_pos[j]);
        for (int k = 0; k < 3; ++k) d.xanchor[j][k] = xpos[k] + v[k];
        quat_rot(d.xaxis[j], xquat, m.jnt_axis[j]);
        double ql[4];
        quat_axisangle(ql, m.jnt_axis[j], q[m.jnt_qposadr[j]] - m.qpos0[m.jnt_qposadr[j]]);
        quat_mul(xquat, xquat, ql);
        quat_rot(v, xquat, m.jnt_pos[j]);
        for (int k = 0; k < 3; ++k) xpos[k] = d.xanchor[j][k] - v[k];
      }
    }
    quat_normalize(xquat);
    cp3(d.xpos[b], xpos);
    for (int k = 0; k < 4; ++k) d.xquat[b][k] = xquat[k];
    quat2mat(d.xmat[b], xquat);
    double t[3];
    mulmatvec3(t, d.xmat[b], m.body_ipos[b]);
    for (int k = 0; k < 3; ++k) d.xipos[b][k] = xpos[k] + t[k];
  }
  for (int g = 0; g < NG; ++g) {
    const int b = m.geom_body[g];
    double t[3];
    mulmatvec3(t, d.xmat[b], m.geom_pos[g]);
    for (int k = 0; k < 3; ++k) d.geom_xpos[g][k] = d.xpos[b][k] + t[k];
    mulmat3(d.geom_xmat[g], d.xmat[b], m.geom_mat[g]);
  }
}

HD void com_pos(const HModel& m, HData& d) {
  for (int b = 0; b < NB; ++b)
    for (int k = 0; k < 3; ++k) d.subtree_com[b][k] = m.body_mass[b] * d.xipos[b][k];
  for (int b = NB - 1; b >= 1; --b)
    for (int k = 0; k < 3; ++k) d.subtree_com[m.parent[b]][k] += d.subtree_com[b][k];
  for (int b = 0; b < NB; ++b) {
    if (m.subtree_mass[b] < MINVAL) cp3(d.subtree_com[b], d.xipos[b]);
    else for (int k = 0; k < 3; ++k) d.subtree_com[b][k] /= m.subtree_mass[b];
  }
  for (int k = 0; k < 10; ++k) d.cinert[0][k] = 0;
  const double* root = d.subtree_com[1];
  for (int b = 1; b < NB; ++b) {
    const double off[3] = {d.xipos[b][0] - root[0], d.xipos[b][1] - root[1], d.xipos[b][2] - root[2]};
    const double* R = d.xmat[b];
    double RI[9], W[9], Rt[9];
    mulmat3(RI, R, m.body_inertia[b]);
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) Rt[3 * i + j] = R[3 * j + i];
    mulmat3(W, RI, Rt);
    const double mass = m.body_mass[b];
    double* c = d.cinert[b];
    c[0] = W[0] + mass * (off[1] * off[1] + off[2] * off[2]);
    c[1] = W[4] + mass * (off[0] * off[0] + off[2] * off[2]);
    c[2] = W[8] + mass * (off[0] * off[0] + off[1] * off[1]);
    c[3] = W[1] - mass * off[0] * off[1];
    c[4] = W[2] - mass * off[0] * off[2];
    c[5] = W[5] - mass * off[1] * off[2];
    c[6] = mass * off[0]; c[7] = mass * off[1]; c[8] = mass * off[2]; c[9] = mass;
  }
  for (int j = 0; j < NJ; ++j) {
    const double off[3] = {root[0] - d.xanchor[j][0], root[1] - d.xanchor[j][1], root[2] - d.xanchor[j][2]};
    const int da = m.jnt_dofadr[j];
    if (m.jnt_type[j] == 0) {
      for (int i = 0; i < 3; ++i) {
        for (int k = 0; k < 6; ++k) d.cdof[da + i][k] = 0;
        d.cdof[da + i][3 + i] = 1.0;
      }
      const double* R = d.xmat[m.jnt_body[j]];
      for (int i = 0; i < 3; ++i) {
        const double ax[3] = {R[i], R[3 + i], R[6 + i]};
        cp3(d.cdof[da + 3 + i], ax);
        cross3(d.cdof[da + 3 + i] + 3, ax, off);
      }
    } else {
      cp3(d.cdof[da], d.xaxis[j]);
      cross3(d.cdof[da] + 3, d.xaxis[j], off);
    }
  }
  for (int t = 0; t < 2; ++t) d.ten_length[t] = -d.qpos[m.ten_q[t][0]] + d.qpos[m.ten_q[t][1]];
}

HD void crb_and_factor(const HModel& m, HData& d) {
  double crb[NB][10];
  for (int b = 0; b < NB; ++b) for (int k = 0; k < 10; ++k) crb[b][k] = d.cinert[b][k];
  for (int b = NB - 1; b >= 1; --b)
    if (m.parent[b] > 0)
      for (int k = 0; k < 10; ++k) crb[m.parent[b]][k] += crb[b][k];
  for (int i = 0; i < NV; ++i) for (int j = 0; j < NV; ++j) d.qM[i][j] = 0;
  for (int i = 0; i < NV; ++i) {
    double buf[6];
    mul_inert_vec(buf, crb[m.dof_body[i]], d.cdof[i]);
    d.qM[i][i] = m.dof_armature[i] + dot6(d.cdof[i], buf);
    for (int j = m.dof_parent[i]; j >= 0; j = m.dof_parent[j]) { d.qM[i][j] = dot6(d.cdof[j], buf); d.qM[j][i] = d.qM[i][j]; }
  }
  for (int i = 0; i < NV; ++i) for (int j = 0; j < NV; ++j) d.qLD[i][j] = d.qM[i][j];
  for (int k = NV - 1; k >= 0; --k) {
    for (int i = m.dof_parent[k]; i >= 0; i = m.dof_parent[i]) {
      const double tmp = d.qLD[k][i] / d.qLD[k][k];
      for (int j = i; j >= 0; j = m.dof_parent[j]) d.qLD[i][j] -= d.qLD[k][j] * tmp;
      d.qLD[k][i] = tmp;
    }
    d.qLDiagInv[k] = 1.0 / d.qLD[k][k];
  }
}
HD void solve_M(const HModel& m, const HData& d, double* x) {
  for (int i = NV - 1; i >= 0; --i)
    for (int j = m.dof_parent[i]; j >= 0; j = m.dof_parent[j]) x[j] -= d.qLD[i][j] * x[i];
  for (int i = 0; i < NV; ++i) x[i] *= d.qLDiagInv[i];
  for (int i = 0; i < NV; ++i)
    for (int j = m.dof_parent[i]; j >= 0; j = m.dof_parent[j]) x[i] -= d.qLD[i][j] * x[j];
}

// ---- collision ----------------------------------------------------------------------------------------------------------------
HD void make_frame(double* f) {
  double* n = f;
  double* t1 = f + 3;
  double* t2 = f + 6;
  if (norm3(t1) < 0.5) {
    t1[0] = t1[1] = t1[2] = 0;
    if (n[1] < 0.5 && n[1] > -0.5) t1[1] = 1; else t1[2] = 1;
  }
  const double dd = dot3(n, t1);
  for (int k = 0; k < 3; ++k) t1[k] -= dd * n[k];
  normalize3(t1);
  cross3(t2, n, t1);
}
HD void add_contact(const HModel& m, HData& d, int g1, int g2, double dist, const double* pos, const double* normal,
                    const double* hint) {
  if (dist >= m.margin) return;
  if (d.ncon >= MAXCON) { d.overflow = 1; return; }
  Contact& c = d.con[d.ncon++];
  c.g1 = g1; c.g2 = g2; c.dist = dist;
  cp3(c.pos, pos);
  cp3(c.frame, normal);
  if (hint) cp3(c.frame + 3, hint); else c.frame[3] = c.frame[4] = c.frame[5] = 0;
  make_frame(c.frame);
  c.dim = m.geom_condim[g1] > m.geom_condim[g2] ? m.geom_condim[g1] : m.geom_condim[g2];
  c.mu = m.geom_friction[g1] > m.geom_friction[g2] ? m.geom_friction[g1] : m.geom_friction[g2];
  c.efc_adr = -1;
}
HD void sphere_sphere(const HModel& m, HData& d, int g1, int g2, const double* p1, double r1, const double* p2, double r2) {
  double n[3] = {p2[0] - p1[0], p2[1] - p1[1], p2[2] - p1[2]};
  const double len = norm3(n);
  const double dist = len - r1 - r2;
  if (dist >= m.margin) return;
  if (len < MINVAL) { n[0] = 1; n[1] = 0; n[2] = 0; } else { n[0] /= len; n[1] /= len; n[2] /= len; }
  double pos[3];
  for (int k = 0; k < 3; ++k) pos[k] = p1[k] + n[k] * (r1 + 0.5 * dist);
  add_contact(m, d, g1, g2, dist, pos, n, nullptr);
}
HD void plane_sphere(const HModel& m, HData& d, int g1, int g2, const double* c, double r, const double* hint) {
  const double* R = d.geom_xmat[g1];
  const double n[3] = {R[2], R[5], R[8]};
  const double df[3] = {c[0] - d.geom_xpos[g1][0], c[1] - d.geom_xpos[g1][1], c[2] - d.geom_xpos[g1][2]};
  const double dist = dot3(df, n) - r;
  if (dist >= m.margin) return;
  double pos[3];
  for (int k = 0; k < 3; ++k) pos[k] = c[k] - n[k] * (r + 0.5 * dist);
  add_contact(m, d, g1, g2, dist, pos, n, hint);
}
HD void collide_pair(const HModel& m, HData& d, int g1, int g2) {
  const int t1 = m.geom_type[g1], t2 = m.geom_type[g2];
  const double *p1 = d.geom_xpos[g1], *p2 = d.geom_xpos[g2];
  if (t1 != G_PLANE) {
    const double df[3] = {p2[0] - p1[0], p2[1] - p1[1], p2[2] - p1[2]};
    const double bound = m.geom_rbound[g1] + m.geom_rbound[g2] + m.margin;
    if (dot3(df, df) > bound * bound) return;
  }
  if (t1 == G_PLANE && t2 == G_SPHERE) {
    plane_sphere(m, d, g1, g2, p2, m.geom_size[g2][0], nullptr);
  } else if (t1 == G_PLANE && t2 == G_CAPSULE) {
    const double* R = d.geom_xmat[g2];
    const double axis[3] = {R[2], R[5], R[8]}, h = m.geom_size[g2][1];
    double e1[3], e2[3];
    for (int k = 0; k < 3; ++k) { e1[k] = p2[k] + axis[k] * h; e2[k] = p2[k] - axis[k] * h; }
    plane_sphere(m, d, g1, g2, e1, m.geom_size[g2][0], axis);
    plane_sphere(m, d, g1, g2, e2, m.geom_size[g2][0], axis);
  } else if (t1 == G_SPHERE && t2 == G_SPHERE) {
    sphere_sphere(m, d, g1, g2, p1, m.geom_size[g1][0], p2, m.geom_size[g2][0]);
  } else if (t1 == G_SPHERE && t2 == G_CAPSULE) {
    const double* R = d.geom_xmat[g2];
    const double axis[3] = {R[2], R[5], R[8]}, h = m.geom_size[g2][1];
    const double df[3] = {p1[0] - p2[0], p1[1] - p2[1], p1[2] - p2[2]};
    double x = dot3(axis, df);
    x = x > h ? h : (x < -h ? -h : x);
    const double cp[3] = {p2[0] + axis[0] * x, p2[1] + axis[1] * x, p2[2] + axis[2] * x};
    sphere_sphere(m, d, g1, g2, p1, m.geom_size[g1][0], cp, m.geom_size[g2][0]);
  } else if (t1 == G_CAPSULE && t2 == G_CAPSULE) {
    const double *R1 = d.geom_xmat[g1], *R2 = d.geom_xmat[g2];
    const double a1[3] = {R1[2], R1[5], R1[8]}, a2[3] = {R2[2], R2[5], R2[8]}, l1 = m.geom_size[g1][1], l2 = m.geom_size[g2][1];
    const double df[3] = {p1[0] - p2[0], p1[1] - p2[1], p1[2] - p2[2]};
    const double ma = dot3(a1, a1), mb = -dot3(a1, a2), mc = dot3(a2, a2), u = -dot3(a1, df), v = dot3(a2, df);
    const double det = ma * mc - mb * mb;
    if (fabs(det) >= MINVAL) {
      double x1 = (mc * u - mb * v) / det, x2 = (ma * v - mb * u) / det;
      if (x1 > l1) { x1 = l1; x2 = (v - mb * l1) / mc; }
      else if (x1 < -l1) { x1 = -l1; x2 = (v + mb * l1) / mc; }
      if (x2 > l2) { x2 = l2; x1 = (u - mb * l2) / ma; if (x1 > l1) x1 = l1; else if (x1 < -l1) x1 = -l1; }
      else if (x2 < -l2) { x2 = -l2; x1 = (u + mb * l2) / ma; if (x1 > l1) x1 = l1; else if (x1 < -l1) x1 = -l1; }
      double c1[3], c2[3];
      for (int k = 0; k < 3; ++k) { c1[k] = p1[k] + a1[k] * x1; c2[k] = p2[k] + a2[k] * x2; }
      sphere_sphere(m, d, g1, g2, c1, m.geom_size[g1][0], c2, m.geom_size[g2][0]);
    } else {
      for (int s = -1; s <= 1; s += 2) {
        double c1[3], c2[3];
        for (int k = 0; k < 3; ++k) c1[k] = p1[k] + a1[k] * (s * l1);
        const double dd[3] = {c1[0] - p2[0], c1[1] - p2[1], c1[2] - p2[2]};
        double x = dot3(a2, dd);
        x = x > l2 ? l2 : (x < -l2 ? -l2 : x);
        for (int k = 0; k < 3; ++k) c2[k] = p2[k] + a2[k] * x;
        sphere_sphere(m, d, g1, g2, c1, m.geom_size[g1][0], c2, m.geom_size[g2][0]);
      }
    }
  }
}

// ---- constraints ----------------------------------------------------------------------------------------------------------------
HD void jac_point(const HModel& m, const HData& d, int b, const double* point, double J[3][NV]) {
  for (int k = 0; k < 3; ++k) for (int i = 0; i < NV; ++i) J[k][i] = 0;
  const double off[3] = {point[0] - d.subtree_com[1][0], point[1] - d.subtree_com[1][1], point[2] - d.subtree_com[1][2]};
  for (int i = m.body_lastdof[b]; i >= 0; i = m.dof_parent[i]) {
    double t[3];
    cross3(t, d.cdof[i], off);
    for (int k = 0; k < 3; ++k) J[k][i] = d.cdof[i][3 + k] + t[k];
  }
}
HD double impedance(const HModel& m, double pos, double margin) {
  const double dmin = m.solimp[0], dmax = m.solimp[1], width = m.solimp[2], mid = m.solimp[3];
  double x = (pos - margin) / width;
  if (x < 0) x = -x;
  if (x >= 1.0) return dmax;
  if (x <= 0.0) return dmin;
  double y;
  if (x <= mid) { const double a = 1.0 / mid; y = a * x * x; }
  else { const double b = 1.0 / (1.0 - mid); y = 1.0 - b * (1.0 - x) * (1.0 - x); }
  return dmin + y * (dmax - dmin);
}
HD void make_constraint(const HModel& m, HData& d) {
  int n = 0;
  for (int j = 1; j < NJ; ++j) {
    const double value = d.qpos[m.jnt_qposadr[j]];
    for (int side = -1; side <= 1; side += 2) {
      const double dist = side * (m.jnt_range[j][(side + 1) / 2] - value);
      if (dist < 0.0 && n < MAXEFC) {
        for (int k = 0; k < NV; ++k) d.efc_J[n][k] = 0;
        d.efc_J[n][m.jnt_dofadr[j]] = -side;
        d.efc_pos[n] = dist; d.efc_margin[n] = 0.0;
        d.efc_diagApprox[n] = m.dof_invweight0[m.jnt_dofadr[j]];
        ++n;
      }
    }
  }
  for (int c = 0; c < d.ncon; ++c) {
    Contact& con = d.con[c];
    const int b1 = m.geom_body[con.g1], b2 = m.geom_body[con.g2];
    double J1[3][NV], J2[3][NV], Jc[3][NV];
    jac_point(m, d, b1, con.pos, J1);
    jac_point(m, d, b2, con.pos, J2);
    for (int r = 0; r < 3; ++r)
      for (int i = 0; i < NV; ++i) {
        double s = 0;
        for (int k = 0; k < 3; ++k) s += con.frame[3 * r + k] * (J2[k][i] - J1[k][i]);
        Jc[r][i] = s;
      }
    const double tran = m.body_invweight0[b1][0] + m.body_invweight0[b2][0];
    const int rows = con.dim == 1 ? 1 : 4;
    if (n + rows > MAXEFC) { con.efc_adr = -1; d.overflow = 1; continue; }
    con.efc_adr = n;
    if (con.dim == 1) {
      for (int i = 0; i < NV; ++i) d.efc_J[n][i] = Jc[0][i];
      d.efc_pos[n] = con.dist; d.efc_margin[n] = m.margin; d.efc_diagApprox[n] = tran;
      ++n;
    } else {
      for (int k = 1; k <= 2; ++k)
        for (int sgn = 1; sgn >= -1; sgn -= 2) {
          for (int i = 0; i < NV; ++i) d.efc_J[n][i] = Jc[0][i] + sgn * con.mu * Jc[k][i];
          d.efc_pos[n] = con.dist; d.efc_margin[n] = m.margin;
          d.efc_diagApprox[n] = tran + con.mu * con.mu * tran;
          ++n;
        }
    }
  }
  d.nefc = n;
  const double timeconst = m.solref[0] > 2 * m.timestep ? m.solref[0] : 2 * m.timestep, dampratio = m.solref[1];
  const double dmax = m.solimp[1];
  const double K = 1.0 / (dmax * dmax * timeconst * timeconst * dampratio * dampratio), B = 2.0 / (dmax * timeconst);
  for (int i = 0; i < n; ++i) {
    const double imp = impedance(m, d.efc_pos[i], d.efc_margin[i]);
    const double R = (1.0 - imp) / imp * d.efc_diagApprox[i];
    d.efc_R[i] = R < MINVAL ? MINVAL : R;
    double vel = 0;
    for (int k = 0; k < NV; ++k) vel += d.efc_J[i][k] * d.qvel[k];
    d.efc_aref[i] = -B * vel - K * imp * (d.efc_pos[i] - d.efc_margin[i]);
  }
  for (int c = 0; c < d.ncon; ++c) {
    const Contact& con = d.con[c];
    if (con.efc_adr >= 0 && con.dim > 1) {
      const double Rpy = 2.0 * con.mu * con.mu * d.efc_R[con.efc_adr];
      for (int k = 0; k < 4; ++k) d.efc_R[con.efc_adr + k] = Rpy;
    }
  }
  for (int i = 0; i < n; ++i) d.efc_D[i] = 1.0 / d.efc_R[i];
  for (int i = 0; i < n; ++i) {  // mj_projectConstraint: AR = J M^-1 J^T + diag(R), one row of M^-1 J^T at a time
    double x[NV];
    for (int k = 0; k < NV; ++k) x[k] = d.efc_J[i][k];
    solve_M(m, d, x);
    for (int j = 0; j <= i; ++j) {
      double s = 0;
      for (int k = 0; k < NV; ++k) s += d.efc_J[j][k] * x[k];
      d.efc_AR[i][j] = s;
      d.efc_AR[j][i] = s;
    }
  }
  for (int i = 0; i < n; ++i) d.efc_AR[i][i] += d.efc_R[i];
}

HD void forward_position(const HModel& m, HData& d) {
  kinematics(m, d);
  com_pos(m, d);
  crb_and_factor(m, d);
  d.ncon = 0;
  for (int p = 0; p < m.npair; ++p) collide_pair(m, d, m.pair_g1[p], m.pair_g2[p]);
  make_constraint(m, d);
}

// ---- velocity / actuation / acceleration / constraint solve ------------------------------------------------------------------------
HD void cross_motion(double* r, const double* vel, const double* v) {
  double t[6];
  t[0] = -vel[2] * v[1] + vel[1] * v[2]; t[1] = vel[2] * v[0] - vel[0] * v[2]; t[2] = -vel[1] * v[0] + vel[0] * v[1];
  t[3] = -vel[2] * v[4] + vel[1] * v[5]; t[4] = vel[2] * v[3] - vel[0] * v[5]; t[5] = -vel[1] * v[3] + vel[0] * v[4];
  t[3] += -vel[5] * v[1] + vel[4] * v[2]; t[4] += vel[5] * v[0] - vel[3] * v[2]; t[5] += -vel[4] * v[0] + vel[3] * v[1];
  for (int k = 0; k < 6; ++k) r[k] = t[k];
}
HD void cross_force(double* r, const double* vel, const double* f) {
  double t[6];
  t[0] = -vel[2] * f[1] + vel[1] * f[2]; t[1] = vel[2] * f[0] - vel[0] * f[2]; t[2] = -vel[1] * f[0] + vel[0] * f[1];
  t[3] = -vel[2] * f[4] + vel[1] * f[5]; t[4] = vel[2] * f[3] - vel[0] * f[5]; t[5] = -vel[1] * f[3] + vel[0] * f[4];
  t[0] += -vel[5] * f[4] + vel[4] * f[5]; t[1] += vel[5] * f[3] - vel[3] * f[5]; t[2] += -vel[4] * f[3] + vel[3] * f[4];
  for (int k = 0; k < 6; ++k) r[k] = t[k];
}
HD void forward_velocity(const HModel& m, HData& d) {
  for (int k = 0; k < 6; ++k) d.cvel[0][k] = 0;
  for (int b = 1; b < NB; ++b) {  // mj_comVel
    double cvel[6];
    for (int k = 0; k < 6; ++k) cvel[k] = d.cvel[m.parent[b]][k];
    for (int jj = 0; jj < m.body_jntnum[b]; ++jj) {
      const int j = m.body_jntadr[b] + jj, da = m.jnt_dofadr[j];
      if (m.jnt_type[j] == 0) {
        for (int i = 0; i < 3; ++i) {
          for (int k = 0; k < 6; ++k) d.cdof_dot[da + i][k] = 0;
          for (int k = 0; k < 6; ++k) cvel[k] += d.cdof[da + i][k] * d.qvel[da + i];
        }
        for (int i = 3; i < 6; ++i) cross_motion(d.cdof_dot[da + i], cvel, d.cdof[da + i]);
        for (int i = 3; i < 6; ++i)
          for (int k = 0; k < 6; ++k) cvel[k] += d.cdof[da + i][k] * d.qvel[da + i];
      } else {
        cross_motion(d.cdof_dot[da], cvel, d.cdof[da]);
        for (int k = 0; k < 6; ++k) cvel[k] += d.cdof[da][k] * d.qvel[da];
      }
    }
    for (int k = 0; k < 6; ++k) d.cvel[b][k] = cvel[k];
  }
  for (int t = 0; t < 2; ++t) d.ten_velocity[t] = -d.qvel[m.ten_v[t][0]] + d.qvel[m.ten_v[t][1]];
  for (int i = 0; i < NV; ++i) d.qfrc_passive[i] = 0;  // mj_passive
  for (int j = 1; j < NJ; ++j) {
    const int da = m.jnt_dofadr[j], qa = m.jnt_qposadr[j];
    d.qfrc_passive[da] = -m.jnt_stiffness[j] * (d.qpos[qa] - 0.0) - m.dof_damping[da] * d.qvel[da];
  }
  double cacc[NB][6], cfrc[NB][6];  // mj_rne without accelerations -> qfrc_bias
  for (int k = 0; k < 3; ++k) { cacc[0][k] = 0; cacc[0][3 + k] = -m.gravity[k]; }
  for (int b = 1; b < NB; ++b) {
    for (int k = 0; k < 6; ++k) cacc[b][k] = cacc[m.parent[b]][k];
    for (int i = 0; i < m.body_dofnum[b]; ++i) {
      const int da = m.body_dofadr[b] + i;
      for (int k = 0; k < 6; ++k) cacc[b][k] += d.cdof_dot[da][k] * d.qvel[da];
    }
    double t1[6], t2[6], t3[6];
    mul_inert_vec(t1, d.cinert[b], cacc[b]);
    mul_inert_vec(t2, d.cinert[b], d.cvel[b]);
    cross_force(t3, d.cvel[b], t2);
    for (int k = 0; k < 6; ++k) cfrc[b][k] = t1[k] + t3[k];
  }
  for (int k = 0; k < 6; ++k) cfrc[0][k] = 0;
  for (int b = NB - 1; b >= 1; --b)
    for (int k = 0; k < 6; ++k) cfrc[m.parent[b]][k] += cfrc[b][k];
  for (int i = 0; i < NV; ++i) d.qfrc_bias[i] = dot6(d.cdof[i], cfrc[m.dof_body[i]]);
}
HD void forward_actuation_acceleration(const HModel& m, HData& d) {
  for (int i = 0; i < NV; ++i) d.qfrc_actuator[i] = 0;
  for (int u = 0; u < NU; ++u) {
    double c = d.ctrl[u];
    c = c < -0.4 ? -0.4 : (c > 0.4 ? 0.4 : c);  // ctrlrange (humanoid.xml:6)
    d.qfrc_actuator[m.act_dof[u]] += m.act_gear[u] * c;
  }
  for (int i = 0; i < NV; ++i) d.qfrc_smooth[i] = d.qfrc_passive[i] - d.qfrc_bias[i] + d.qfrc_actuator[i];
  for (int i = 0; i < NV; ++i) d.qacc_smooth[i] = d.qfrc_smooth[i];
  solve_M(m, d, d.qacc_smooth);
}
HD void forward_constraint(const HModel& m, HData& d) {
  const int n = d.nefc;
  for (int k = 0; k < NV; ++k) d.qfrc_constraint[k] = 0;
  if (n == 0) {
    for (int k = 0; k < NV; ++k) d.qacc[k] = d.qacc_smooth[k];
    return;
  }
  for (int i = 0; i < n; ++i) {
    double s = 0;
    for (int k = 0; k < NV; ++k) s += d.efc_J[i][k] * d.qacc_smooth[k];
    d.efc_b[i] = s - d.efc_aref[i];
  }
  double cost = 0;
  for (int i = 0; i < n; ++i) {
    double jar = 0;
    for (int k = 0; k < NV; ++k) jar += d.efc_J[i][k] * d.qacc_warmstart[k];
    jar -= d.efc_aref[i];
    d.efc_force[i] = jar < 0 ? -d.efc_D[i] * jar : 0.0;
  }
  double res[MAXEFC], ainv[MAXEFC];  /* running residual AR f + b of every row, 1 / AR[i][i] */
  for (int i = 0; i < n; ++i) {
    double s = 0;
    for (int j = 0; j < n; ++j) s += d.efc_AR[i][j] * d.efc_force[j];
    cost += d.efc_force[i] * (0.5 * s + d.efc_b[i]);
    res[i] = d.efc_b[i] + s;
    ainv[i] = 1.0 / d.efc_AR[i][i];
  }
  if (cost > 0)
    for (int i = 0; i < n; ++i) { d.efc_force[i] = 0; res[i] = d.efc_b[i]; }
  const double scale = 1.0 / (m.meaninertia * (NV > 1 ? NV : 1));
  /* Gauss-Seidel sweeps in residual-update form: after row j moves by delta, every residual moves by AR[:, j] * delta
     (same sweep as recomputing AR[j, :] f + b per row; the update form is what maps onto one lane per row) */
  for (int it = 0; it < m.iterations; ++it) {
    double improvement = 0;
    for (int j = 0; j < n; ++j) {
      const double old = d.efc_force[j], r = res[j];
      double f = old - r * ainv[j];
      if (f < 0) f = 0;
      d.efc_force[j] = f;
      const double delta = f - old;
      improvement -= 0.5 * delta * delta * d.efc_AR[j][j] + delta * r;
      for (int i = 0; i < n; ++i) res[i] += d.efc_AR[i][j] * delta;
    }
    if (improvement * scale < m.tolerance) break;
  }
  for (int i = 0; i < n; ++i)
    for (int k = 0; k < NV; ++k) d.qfrc_constraint[k] += d.efc_J[i][k] * d.efc_force[i];
  double t[NV];
  for (int k = 0; k < NV; ++k) t[k] = d.qfrc_constraint[k];
  solve_M(m, d, t);
  for (int k = 0; k < NV; ++k) d.qacc[k] = d.qacc_smooth[k] + t[k];
}
HD void mj_forward(const HModel& m, HData& d) {
  forward_position(m, d);
  forward_velocity(m, d);
  forward_actuation_acceleration(m, d);
  forward_constraint(m, d);
}

// ---- integration -----------------------------------------------------------------------------------------------------------------
HD void integrate_pos(double* qpos, const double* vel, double h) {
  for (int k = 0; k < 3; ++k) qpos[k] += h * vel[k];
  const double w[3] = {vel[3], vel[4], vel[5]};
  const double ang = norm3(w);
  if (ang >= MINVAL) {
    const double axis[3] = {w[0] / ang, w[1] / ang, w[2] / ang};
    double dq[4];
    quat_axisangle(dq, axis, ang * h);
    quat_mul(qpos + 3, qpos + 3, dq);
  }
  quat_normalize(qpos + 3);
  for (int i = 6; i < NV; ++i) qpos[i + 1] += h * vel[i];
}
HD void mj_step_rk4(const HModel& m, HData& d) {
  mj_forward(m, d);
  const double h = m.timestep;
  const double A[3][3] = {{0.5, 0, 0}, {0, 0.5, 0}, {0, 0, 1.0}}, Bw[4] = {1.0 / 6, 1.0 / 3, 1.0 / 3, 1.0 / 6};
  double X0q[NQ], X0v[NV], Xv[4][NV], F[4][NV];
  for (int k = 0; k < NQ; ++k) X0q[k] = d.qpos[k];
  for (int k = 0; k < NV; ++k) { X0v[k] = d.qvel[k]; Xv[0][k] = d.qvel[k]; F[0][k] = d.qacc[k]; }
  for (int i = 1; i < 4; ++i) {
    double dXv[NV], dXa[NV];
    for (int k = 0; k < NV; ++k) { dXv[k] = 0; dXa[k] = 0; }
    for (int j = 0; j < i; ++j)
      for (int k = 0; k < NV; ++k) { dXv[k] += A[i - 1][j] * Xv[j][k]; dXa[k] += A[i - 1][j] * F[j][k]; }
    for (int k = 0; k < NQ; ++k) d.qpos[k] = X0q[k];
    integrate_pos(d.qpos, dXv, h);
    for (int k = 0; k < NV; ++k) d.qvel[k] = X0v[k] + h * dXa[k];
    for (int k = 0; k < NV; ++k) Xv[i][k] = d.qvel[k];
    mj_forward(m, d);
    for (int k = 0; k < NV; ++k) F[i][k] = d.qacc[k];
  }
  double dXv[NV], dXa[NV];
  for (int k = 0; k < NV; ++k) { dXv[k] = 0; dXa[k] = 0; }
  for (int j = 0; j < 4; ++j)
    for (int k = 0; k < NV; ++k) { dXv[k] += Bw[j] * Xv[j][k]; dXa[k] += Bw[j] * F[j][k]; }
  for (int k = 0; k < NQ; ++k) d.qpos[k] = X0q[k];
  for (int k = 0; k < NV; ++k) d.qvel[k] = X0v[k] + h * dXa[k];
  integrate_pos(d.qpos, dXv, h);
  for (int k = 0; k < NV; ++k) d.qacc_warmstart[k] = d.qacc[k];
}
HD void rne_post_constraint(const HModel& m, HData& d) {
  for (int b = 0; b < NB; ++b) for (int k = 0; k < 6; ++k) d.cfrc_ext[b][k] = 0;
  for (int c = 0; c < d.ncon; ++c) {
    const Contact& con = d.con[c];
    if (con.efc_adr < 0) continue;
    double lf[3] = {0, 0, 0};
    const double* f = d.efc_force + con.efc_adr;
    if (con.dim == 1) lf[0] = f[0];
    else { lf[0] = f[0] + f[1] + f[2] + f[3]; lf[1] = (f[0] - f[1]) * con.mu; lf[2] = (f[2] - f[3]) * con.mu; }
    double wf[3];
    for (int k = 0; k < 3; ++k) wf[k] = con.frame[k] * lf[0] + con.frame[3 + k] * lf[1] + con.frame[6 + k] * lf[2];
    const int b1 = m.geom_body[con.g1], b2 = m.geom_body[con.g2];
    for (int side = 0; side < 2; ++side) {
      const int b = side ? b2 : b1;
      const double sgn = side ? 1.0 : -1.0;
      const double* com = d.subtree_com[b == 0 ? 0 : 1];
      const double r[3] = {con.pos[0] - com[0], con.pos[1] - com[1], con.pos[2] - com[2]};
      double tq[3];
      cross3(tq, r, wf);
      for (int k = 0; k < 3; ++k) { d.cfrc_ext[b][k] += sgn * tq[k]; d.cfrc_ext[b][3 + k] += sgn * wf[k]; }
    }
  }
}

// ---- model (humanoid.xml re-typed as data) + compile -----------------------------------------------------------------------------
struct JDef { int body; double pos[3], axis[3], lo, hi, stiffness, damping, armature; };
struct GDef { int type, body; double a[3], b[3], r; };
struct BDef { int parent; double pos[3], quat[4]; };

void build_model(HModel& m) {
  static const BDef BODY[NB] = {
      {0, {0, 0, 0}, {1, 0, 0, 0}},            {0, {0, 0, 1.4}, {1, 0, 0, 0}},          {1, {-.01, 0, -0.260}, {1.000, 0, -0.002, 0}},
      {2, {0, 0, -0.165}, {1.000, 0, -0.002, 0}}, {3, {0, -0.1, -0.04}, {1, 0, 0, 0}},   {4, {0, 0.01, -0.403}, {1, 0, 0, 0}},
      {5, {0, 0, -0.45}, {1, 0, 0, 0}},        {3, {0, 0.1, -0.04}, {1, 0, 0, 0}},      {7, {0, -0.01, -0.403}, {1, 0, 0, 0}},
      {8, {0, 0, -0.45}, {1, 0, 0, 0}},        {1, {0, -0.17, 0.06}, {1, 0, 0, 0}},     {10, {.18, -.18, -.18}, {1, 0, 0, 0}},
      {1, {0, 0.17, 0.06}, {1, 0, 0, 0}},      {12, {.18, .18, -.18}, {1, 0, 0, 0}}};
  static const JDef HINGE[17] = {
      {2, {0, 0, 0.065}, {0, 0, 1}, -45, 45, 20, 5, 0.02},   {2, {0, 0, 0.065}, {0, 1, 0}, -75, 30, 10, 5, 0.02},
      {3, {0, 0, 0.1}, {1, 0, 0}, -35, 35, 10, 5, 0.02},     {4, {0, 0, 0}, {1, 0, 0}, -25, 5, 10, 5, 0.01},
      {4, {0, 0, 0}, {0, 0, 1}, -60, 35, 10, 5, 0.01},       {4, {0, 0, 0}, {0, 1, 0}, -110, 20, 20, 5, 0.0080},
      {5, {0, 0, .02}, {0, -1, 0}, -160, -2, 0, 1, 0.0060},  {7, {0, 0, 0}, {-1, 0, 0}, -25, 5, 10, 5, 0.01},
      {7, {0, 0, 0}, {0, 0, -1}, -60, 35, 10, 5, 0.01},      {7, {0, 0, 0}, {0, 1, 0}, -110, 20, 20, 5, 0.01},
      {8, {0, 0, .02}, {0, -1, 0}, -160, -2, 1, 1, 0.0060},  {10, {0, 0, 0}, {2, 1, 1}, -85, 60, 1, 1, 0.0068},
      {10, {0, 0, 0}, {0, -1, 1}, -85, 60, 1, 1, 0.0051},    {11, {0, 0, 0}, {0, -1, 1}, -90, 50, 0, 1, 0.0028},
      {12, {0, 0, 0}, {2, -1, 1}, -60, 85, 1, 1, 0.0068},    {12, {0, 0, 0}, {0, 1, 1}, -60, 85, 1, 1, 0.0051},
      {13, {0, 0, 0}, {0, -1, -1}, -90, 50, 0, 1, 0.0028}};
  static const GDef GEOM[NG] = {
      {G_PLANE, 0, {0, 0, 0}, {0, 0, 0}, 0},
      {G_CAPSULE, 1, {0, -.07, 0}, {0, .07, 0}, 0.07},
      {G_SPHERE, 1, {0, 0, .19}, {0, 0, 0}, .09},
      {G_CAPSULE, 1, {-.01, -.06, -.12}, {-.01, .06, -.12}, 0.06},
      {G_CAPSULE, 2, {0, -.06, 0}, {0, .06, 0}, 0.06},
      {G_CAPSULE, 3, {-.02, -.07, 0}, {-.02, .07, 0}, 0.09},
      {G_CAPSULE, 4, {0, 0, 0}, {0, 0.01, -.34}, 0.06},
      {G_CAPSULE, 5, {0, 0, 0}, {0, 0, -.3}, 0.049},
      {G_SPHERE, 6, {0, 0, 0.1}, {0, 0, 0}, 0.075},
      {G_CAPSULE, 7, {0, 0, 0}, {0, -0.01, -.34}, 0.06},
      {G_CAPSULE, 8, {0, 0, 0}, {0, 0, -.3}, 0.049},
      {G_SPHERE, 9, {0, 0, 0.1}, {0, 0, 0}, 0.075},
      {G_CAPSULE, 10, {0, 0, 0}, {.16, -.16, -.16}, 0.04},
      {G_CAPSULE, 11, {0.01, 0.01, 0.01}, {.17, .17, .17}, 0.031},
      {G_SPHERE, 11, {.18, .18, .18}, {0, 0, 0}, 0.04},
      {G_CAPSULE, 12, {0, 0, 0}, {.16, .16, -.16}, 0.04},
      {G_CAPSULE, 13, {0.01, -0.01, 0.01}, {.17, -.17, .17}, 0.031},
      {G_SPHERE, 13, {.18, -.18, .18}, {0, 0, 0}, 0.04}};
  static const int ACT_HINGE[NU] = {1, 0, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16};
  static const double ACT_GEAR[NU] = {100, 100, 100, 100, 100, 300, 200, 100, 100, 300, 200, 25, 25, 25, 25, 25, 25};
  const double DEG = PI / 180.0;
  memset(&m, 0, sizeof(m));
  m.timestep = 0.003; m.gravity[2] = -9.81; m.margin = 0.001; m.tolerance = 1e-8; m.iterations = 50;
  m.solref[0] = 0.02; m.solref[1] = 1.0;
  m.solimp[0] = 0.9; m.solimp[1] = 0.95; m.solimp[2] = 0.001; m.solimp[3] = 0.5; m.solimp[4] = 2.0;
  for (int b = 0; b < NB; ++b) {
    m.parent[b] = BODY[b].parent;
    cp3(m.body_pos[b], BODY[b].pos);
    for (int k = 0; k < 4; ++k) m.body_quat[b][k] = BODY[b].quat[k];
    quat_normalize(m.body_quat[b]);
    m.body_jntadr[b] = -1; m.body_dofadr[b] = -1;
  }
  m.jnt_type[0] = 0; m.jnt_body[0] = 1; m.jnt_qposadr[0] = 0; m.jnt_dofadr[0] = 0;
  for (int k = 0; k < 17; ++k) {
    const int j = k + 1;
    m.jnt_type[j] = 3; m.jnt_body[j] = HINGE[k].body; m.jnt_qposadr[j] = 7 + k; m.jnt_dofadr[j] = 6 + k;
    cp3(m.jnt_pos[j], HINGE[k].pos);
    cp3(m.jnt_axis[j], HINGE[k].axis);
    normalize3(m.jnt_axis[j]);
    m.jnt_range[j][0] = HINGE[k].lo * DEG; m.jnt_range[j][1] = HINGE[k].hi * DEG;
    m.jnt_stiffness[j] = HINGE[k].stiffness;
    m.dof_armature[6 + k] = HINGE[k].armature; m.dof_damping[6 + k] = HINGE[k].damping;
  }
  for (int j = 0; j < NJ; ++j) {
    const int b = m.jnt_body[j];
    if (m.body_jntadr[b] < 0) { m.body_jntadr[b] = j; m.body_dofadr[b] = m.jnt_dofadr[j]; }
    m.body_jntnum[b] += 1;
    m.body_dofnum[b] += m.jnt_type[j] == 0 ? 6 : 1;
  }
  for (int i = 0; i < NV; ++i) m.dof_body[i] = m.jnt_body[i < 6 ? 0 : i - 5];
  m.body_lastdof[0] = -1;
  for (int b = 1; b < NB; ++b)
    m.body_lastdof[b] = m.body_dofnum[b] ? m.body_dofadr[b] + m.body_dofnum[b] - 1 : m.body_lastdof[m.parent[b]];
  for (int i = 0; i < NV; ++i) {
    const int b = m.dof_body[i];
    m.dof_parent[i] = i > m.body_dofadr[b] ? i - 1 : m.body_lastdof[m.parent[b]];
  }
  double bm[NB] = {0}, bcom[NB][3] = {{0}}, gmass[NG], gI[NG][9];
  for (int g = 0; g < NG; ++g) {
    const GDef& G = GEOM[g];
    m.geom_type[g] = G.type; m.geom_body[g] = G.body; m.geom_condim[g] = g == 0 ? 3 : 1;
    m.geom_friction[g] = 1.0;
    double I[3] = {0, 0, 0};
    gmass[g] = 0;
    for (int k = 0; k < 9; ++k) m.geom_mat[g][k] = (k % 4 == 0) ? 1.0 : 0.0;
    if (G.type == G_SPHERE) {
      cp3(m.geom_pos[g], G.a);
      m.geom_size[g][0] = G.r;
      m.geom_rbound[g] = G.r;
      gmass[g] = 1000.0 * (4.0 / 3.0) * PI * G.r * G.r * G.r;
      I[0] = I[1] = I[2] = 0.4 * gmass[g] * G.r * G.r;
    } else if (G.type == G_CAPSULE) {
      double dv[3] = {G.b[0] - G.a[0], G.b[1] - G.a[1], G.b[2] - G.a[2]};
      const double len = norm3(dv), half = 0.5 * len, r = G.r, h = len;
      for (int k = 0; k < 3; ++k) m.geom_pos[g][k] = 0.5 * (G.a[k] + G.b[k]);
      {  // rotation taking z to the capsule axis, from sqrt only (half-angle formulas)
        double vec[3] = {dv[0], dv[1], dv[2]}, q[4] = {1, 0, 0, 0};
        normalize3(vec);
        double axis[3] = {-vec[1], vec[0], 0.0};
        const double a = norm3(axis);
        if (a >= MINVAL) {
          const double c = vec[2], ch = sqrt(0.5 * (1.0 + c)), sh = sqrt(0.5 * (1.0 - c));
          q[0] = ch; q[1] = axis[0] / a * sh; q[2] = axis[1] / a * sh; q[3] = 0.0;
        } else if (vec[2] < 0) {
          q[0] = 0; q[1] = 1; q[2] = 0; q[3] = 0;
        }
        quat2mat(m.geom_mat[g], q);
      }
      m.geom_size[g][0] = r; m.geom_size[g][1] = half;
      m.geom_rbound[g] = r + half;
      const double ms = 1000.0 * (4.0 / 3.0) * PI * r * r * r, mc = 1000.0 * PI * r * r * h;
      gmass[g] = ms + mc;
      I[0] = I[1] = mc * (3 * r * r + h * h) / 12.0 + ms * (0.4 * r * r + 0.25 * h * h + 0.375 * r * h);
      I[2] = 0.5 * mc * r * r + 0.4 * ms * r * r;
    }
    const double* R = m.geom_mat[g];
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j)
        gI[g][3 * i + j] = R[3 * i] * I[0] * R[3 * j] + R[3 * i + 1] * I[1] * R[3 * j + 1] + R[3 * i + 2] * I[2] * R[3 * j + 2];
    bm[G.body] += gmass[g];
    for (int k = 0; k < 3; ++k) bcom[G.body][k] += gmass[g] * m.geom_pos[g][k];
  }
  for (int b = 1; b < NB; ++b) {
    m.body_mass[b] = bm[b];
    for (int k = 0; k < 3; ++k) m.body_ipos[b][k] = bcom[b][k] / bm[b];
  }
  for (int g = 1; g < NG; ++g) {
    const int b = GEOM[g].body;
    const double dv[3] = {m.geom_pos[g][0] - m.body_ipos[b][0], m.geom_pos[g][1] - m.body_ipos[b][1],
                          m.geom_pos[g][2] - m.body_ipos[b][2]};
    const double d2 = dot3(dv, dv);
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j)
        m.body_inertia[b][3 * i + j] += gI[g][3 * i + j] + gmass[g] * ((i == j ? d2 : 0.0) - dv[i] * dv[j]);
  }
  for (int b = NB - 1; b >= 0; --b) m.subtree_mass[b] = m.body_mass[b];
  for (int b = NB - 1; b >= 1; --b) m.subtree_mass[m.parent[b]] += m.subtree_mass[b];
  for (int u = 0; u < NU; ++u) { m.act_dof[u] = 6 + ACT_HINGE[u]; m.act_gear[u] = ACT_GEAR[u]; }
  m.ten_q[0][0] = 7 + 9; m.ten_q[0][1] = 7 + 10; m.ten_v[0][0] = 6 + 9; m.ten_v[0][1] = 6 + 10;
  m.ten_q[1][0] = 7 + 5; m.ten_q[1][1] = 7 + 6; m.ten_v[1][0] = 6 + 5; m.ten_v[1][1] = 6 + 6;
  m.npair = 0;
  for (int b1 = 0; b1 < NB; ++b1)
    for (int b2 = b1 + 1; b2 < NB; ++b2) {
      if (b1 != 0 && (m.parent[b2] == b1 || m.parent[b1] == b2)) continue;
      for (int g1 = 0; g1 < NG; ++g1)
        for (int g2 = 0; g2 < NG; ++g2) {
          if (m.geom_body[g1] != b1 || m.geom_body[g2] != b2) continue;
          int a = g1, c = g2;
          if (m.geom_type[a] > m.geom_type[c]) { const int t = a; a = c; c = t; }
          m.pair_g1[m.npair] = a; m.pair_g2[m.npair] = c; m.npair++;
        }
    }
  m.qpos0[2] = 1.4; m.qpos0[3] = 1.0;
  for (int b = 1; b < NB; ++b) m.body_depth[b] = m.body_depth[m.parent[b]] + 1;
  for (int i = 0; i < NV; ++i) {
    int len = 0;
    for (int j = m.dof_parent[i]; j >= 0; j = m.dof_parent[j]) m.dof_chain[i][len++] = j;
    m.dof_chain_len[i] = len;
  }
  for (int b = 1; b < NB; ++b)
    for (int i = m.body_lastdof[b]; i >= 0; i = m.dof_parent[i]) m.body_dofmask[b] |= 1u << i;
  for (int l = 0; l < 7; ++l) for (int k = 0; k < 3; ++k) m.lvl_parents[l][k] = -1;
  for (int b = 0; b < NB; ++b) {
    int nc = 0;
    for (int k = 0; k < 3; ++k) m.children[b][k] = -1;
    for (int c = NB - 1; c >= 1; --c)
      if (m.parent[c] == b) { assert(nc < 3); m.children[b][nc++] = c; }
    if (nc) {
      int* row = m.lvl_parents[m.body_depth[b]];
      int k = 0;
      while (row[k] >= 0) { ++k; assert(k < 3); }
      row[k] = b;
    }
  }
  // constants MuJoCo derives at qpos0 (mj_setConst): meaninertia, dof/body invweight0 -- with the same physics core
  HData* d = new HData();
  memset(d, 0, sizeof(HData));
  for (int k = 0; k < NQ; ++k) d->qpos[k] = m.qpos0[k];
  forward_position(m, *d);
  static double Minv[NV][NV];
  for (int i = 0; i < NV; ++i) {
    double e[NV] = {0};
    e[i] = 1.0;
    solve_M(m, *d, e);
    for (int j = 0; j < NV; ++j) Minv[j][i] = e[j];
  }
  double mi = 0;
  for (int i = 0; i < NV; ++i) mi += d->qM[i][i];
  m.meaninertia = mi / NV;
  for (int i = 0; i < NV; ++i) m.dof_invweight0[i] = Minv[i][i];
  {
    const double t = (Minv[0][0] + Minv[1][1] + Minv[2][2]) / 3, r = (Minv[3][3] + Minv[4][4] + Minv[5][5]) / 3;
    for (int i = 0; i < 3; ++i) { m.dof_invweight0[i] = t; m.dof_invweight0[3 + i] = r; }
  }
  for (int b = 1; b < NB; ++b) {
    static double Jp[3][NV], Jr[3][NV];
    for (int k = 0; k < 3; ++k) for (int i = 0; i < NV; ++i) { Jp[k][i] = 0; Jr[k][i] = 0; }
    int i = m.body_lastdof[b];
    while (i >= 0) {
      const double off[3] = {d->xipos[b][0] - d->subtree_com[1][0], d->xipos[b][1] - d->subtree_com[1][1],
                             d->xipos[b][2] - d->subtree_com[1][2]};
      double t[3];
      cross3(t, d->cdof[i], off);
      for (int k = 0; k < 3; ++k) { Jp[k][i] = d->cdof[i][3 + k] + t[k]; Jr[k][i] = d->cdof[i][k]; }
      i = m.dof_parent[i];
    }
    double tp = 0, tr = 0;
    for (int k = 0; k < 3; ++k)
      for (int a = 0; a < NV; ++a)
        for (int c = 0; c < NV; ++c) { tp += Jp[k][a] * Minv[a][c] * Jp[k][c]; tr += Jr[k][a] * Minv[a][c] * Jr[k][c]; }
    m.body_invweight0[b][0] = tp / 3; m.body_invweight0[b][1] = tr / 3;
  }
  delete d;
}

__device__ HModel g_hmodel;  // global (not __constant__): the pair list / tables are indexed divergently

#include "humanoid_tree.inc"
// what the warp-per-env kernels read: the model plus the index tables of the packed L / M storage (humanoid_tree.inc);
// the step kernel stages one copy per CTA in shared memory
struct alignas(16) WModel {
  HModel m;
  unsigned short fac_start[NV + 1], fac_pair[B2E_FAC_NPAIR];
  unsigned char rowoff[NV + 1];
};
static_assert(sizeof(WModel) % 16 == 0, "WModel is copied as 16-byte words");
__device__ WModel g_wmodel;

const HModel& host_model() {
  static HModel M;
  static bool built = false;
  if (!built) { build_model(M); built = true; }
  return M;
}
int upload_model() {
  static bool done[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
  if (done[dev]) return 0;
  const HModel& M = host_model();
  cudaError_t e = cudaMemcpyToSymbol(g_hmodel, &M, sizeof(HModel));
  if (e != cudaSuccess) return cuda_status(e, "humanoid model upload");
  static WModel W;  // zero-initialised padding
  W.m = M;
  memcpy(W.fac_start, B2E_FAC_START_H, sizeof(B2E_FAC_START_H));
  memcpy(W.fac_pair, B2E_FAC_PAIR_H, sizeof(B2E_FAC_PAIR_H));
  memcpy(W.rowoff, B2E_LD_ROWOFF_H, sizeof(B2E_LD_ROWOFF_H));
  e = cudaMemcpyToSymbol(g_wmodel, &W, sizeof(WModel));
  if (e != cudaSuccess) return cuda_status(e, "humanoid model upload");
  done[dev] = true;
  return 0;
}

// ---- kernels -------------------------------------------------------------------------------------------------------------------
struct HumanoidArgs {
  int64_t n, env_offset;
  int32_t max_steps, mode, rng_mode, frame_skip, terminate_when_unhealthy;
  uint64_t philox_seed, call_counter;
  double noise, w_forward, w_ctrl, w_contact, contact_max, healthy_reward, z_min, z_max;
  double* __restrict__ qpos;   // [24][n]
  double* __restrict__ qvel;   // [23][n]
  double* __restrict__ warm;   // [23][n]
  double* __restrict__ com_xy; // [2][n]  mass centre (x, y) of the last forward evaluation (stale xipos, humanoid_v5.py:473)
  int32_t* __restrict__ ctrl;
  uint64_t* __restrict__ rng;
  int32_t* __restrict__ overflow;  // [1] sticky
  int32_t* __restrict__ work;      // [n] or null: solver work of the last step
  int32_t* __restrict__ order;     // [n] or null: envs grouped by work (warp mapping only)
  double* __restrict__ obs;        // [n][348]
  double* __restrict__ reward;
  uint8_t* __restrict__ term;
  uint8_t* __restrict__ trunc;
  double* __restrict__ info;       // [13][n]
  double* __restrict__ final_obs;
  const void* __restrict__ actions; // [n][17] float32 or float64
  const uint8_t* __restrict__ mask;
};

__device__ void write_obs(const HData& d, double* __restrict__ obs) {  // humanoid_v5.py:436-470
  int o = 0;
  for (int i = 2; i < NQ; ++i) obs[o++] = d.qpos[i];
  for (int i = 0; i < NV; ++i) obs[o++] = d.qvel[i];
  for (int b = 1; b < NB; ++b) for (int k = 0; k < 10; ++k) obs[o++] = d.cinert[b][k];
  for (int b = 1; b < NB; ++b) for (int k = 0; k < 6; ++k) obs[o++] = d.cvel[b][k];
  for (int i = 6; i < NV; ++i) obs[o++] = d.qfrc_actuator[i];
  for (int b = 1; b < NB; ++b) for (int k = 0; k < 6; ++k) obs[o++] = d.cfrc_ext[b][k];
}
__device__ void mass_center(const HModel& m, const HData& d, double* xy) {  // humanoid_v5.py:17-21
  double nx = 0, ny = 0, den = 0;
  for (int b = 0; b < NB; ++b) { nx += m.body_mass[b] * d.xipos[b][0]; ny += m.body_mass[b] * d.xipos[b][1]; den += m.body_mass[b]; }
  xy[0] = nx / den; xy[1] = ny / den;
}
__device__ void write_info_base(const HumanoidArgs& a, int64_t i, const HData& d) {
  const int64_t n = a.n;
  a.info[0 * n + i] = d.qpos[0];
  a.info[1 * n + i] = d.qpos[1];
  a.info[2 * n + i] = d.ten_length[0];
  a.info[3 * n + i] = d.ten_length[1];
  a.info[4 * n + i] = d.ten_velocity[0];
  a.info[5 * n + i] = d.ten_velocity[1];
  a.info[6 * n + i] = sqrt(d.qpos[0] * d.qpos[0] + d.qpos[1] * d.qpos[1]);
}

// uniform draws for reset noise: numpy stream or Philox
struct HDraws {
  Pcg64 g;
  bool numpy;
  uint64_t seed, env, counter;
  uint32_t k;
  __device__ double next() {
    if (numpy) return g.next_double();
    const uint4 r = philox_block(seed, env, counter, 32u + (k >> 1));
    const double u = (k & 1u) ? u53_to_double(r.z, r.w) : u53_to_double(r.x, r.y);
    ++k;
    return u;
  }
};

// MujocoEnv.reset + HumanoidEnv.reset_model (mujoco_env.py:172-187, humanoid_v5.py:519-532)
__device__ void env_reset(const HumanoidArgs& a, int64_t i, HData& d, HDraws& D, double* __restrict__ obs) {
  const HModel& m = g_hmodel;
  for (int k = 0; k < NV; ++k) d.qacc_warmstart[k] = 0;  // mj_resetData
  for (int u = 0; u < NU; ++u) d.ctrl[u] = 0;
  for (int b = 0; b < NB; ++b) for (int k = 0; k < 6; ++k) d.cfrc_ext[b][k] = 0;
  const double c = a.noise;
  for (int k = 0; k < NQ; ++k) d.qpos[k] = m.qpos0[k] + (-c + (c - -c) * D.next());
  for (int k = 0; k < NV; ++k) d.qvel[k] = 0.0 + (-c + (c - -c) * D.next());
  mj_forward(m, d);
  write_obs(d, obs);
  for (int k = 7; k < 13; ++k) a.info[k * a.n + i] = 0.0;
  write_info_base(a, i, d);
}

__device__ void load_state(const HumanoidArgs& a, int64_t i, HData& d) {
  const int64_t n = a.n;
  for (int k = 0; k < NQ; ++k) d.qpos[k] = a.qpos[k * n + i];
  for (int k = 0; k < NV; ++k) { d.qvel[k] = a.qvel[k * n + i]; d.qacc_warmstart[k] = a.warm[k * n + i]; }
}
__device__ void store_state(const HumanoidArgs& a, int64_t i, const HData& d) {
  const int64_t n = a.n;
  for (int k = 0; k < NQ; ++k) a.qpos[k * n + i] = d.qpos[k];
  for (int k = 0; k < NV; ++k) { a.qvel[k * n + i] = d.qvel[k]; a.warm[k * n + i] = d.qacc_warmstart[k]; }
  double xy[2];
  mass_center(g_hmodel, d, xy);
  a.com_xy[i] = xy[0];
  a.com_xy[n + i] = xy[1];
  if (d.overflow) *a.overflow = 1;
}

constexpr int kHumanoidBlock = 32;
constexpr int kWarpEnvsPerCta = 10;  // warp mapping: envs (warps) per CTA; N=8192: 8 per CTA 8.4 ms, 10 per CTA 7.5 ms
                                     // (10 x 20.2 KB + the 12.9 KB model = 215 KB of the 227 KB an sm_100a CTA can have)

__global__ void __launch_bounds__(kHumanoidBlock) humanoid_reset_kernel(const HumanoidArgs a) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  if (a.mask != nullptr && a.mask[i] == 0) return;
  HData d;
  d.overflow = 0;
  HDraws D;
  D.numpy = a.rng_mode == B2E_RNG_NUMPY;
  if (D.numpy) D.g = pcg64_load(a.rng, a.n, i);
  D.seed = a.philox_seed; D.env = (uint64_t)(a.env_offset + i); D.counter = a.call_counter; D.k = 0;
  env_reset(a, i, d, D, a.obs + 348 * i);
  if (D.numpy) pcg64_store_state(a.rng, i, D.g);
  store_state(a, i, d);
  a.ctrl[i] = 0;
}

template <typename ActT>
__global__ void __launch_bounds__(kHumanoidBlock) humanoid_step_kernel(const HumanoidArgs a) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  const HModel& m = g_hmodel;
  const int32_t c = a.ctrl[i];
  HData d;
  d.overflow = 0;
  HDraws D;
  D.numpy = a.rng_mode == B2E_RNG_NUMPY;
  D.seed = a.philox_seed; D.env = (uint64_t)(a.env_offset + i); D.counter = a.call_counter; D.k = 0;
  double* __restrict__ obs = a.obs + 348 * i;
  if (a.mode == B2E_AUTORESET_NEXT_STEP && ctrl_pending(c)) {  // sync_vector_env.py:279-284
    if (D.numpy) D.g = pcg64_load(a.rng, a.n, i);
    env_reset(a, i, d, D, obs);
    if (D.numpy) pcg64_store_state(a.rng, i, D.g);
    store_state(a, i, d);
    a.ctrl[i] = 0;
    a.reward[i] = 0.0;
    a.term[i] = 0;
    a.trunc[i] = 0;
    return;
  }
  load_state(a, i, d);
  const double before[2] = {a.com_xy[i], a.com_xy[a.n + i]};  // mass_center before do_simulation (humanoid_v5.py:473)
  double ctrl_sq = 0;
  for (int u = 0; u < NU; ++u) {
    d.ctrl[u] = (double)reinterpret_cast<const ActT*>(a.actions)[i * NU + u];
    ctrl_sq += d.ctrl[u] * d.ctrl[u];
  }
  for (int k = 0; k < a.frame_skip; ++k) mj_step_rk4(m, d);  // mj_step(nstep=frame_skip), mujoco_env.py:150
  rne_post_constraint(m, d);                                   // mujoco_env.py:155
  double after[2];
  mass_center(m, d, after);
  const double dt = m.timestep * a.frame_skip;
  const double xv = (after[0] - before[0]) / dt, yv = (after[1] - before[1]) / dt;
  write_obs(d, obs);
  const bool healthy = a.z_min < d.qpos[2] && d.qpos[2] < a.z_max;  // humanoid_v5.py:430-434
  const double forward_reward = a.w_forward * xv, healthy_reward = healthy ? a.healthy_reward : 0.0;
  double cf = 0;
  for (int b = 0; b < NB; ++b) for (int k = 0; k < 6; ++k) cf += d.cfrc_ext[b][k] * d.cfrc_ext[b][k];
  const double ctrl_cost = a.w_ctrl * ctrl_sq;
  double contact_cost = a.w_contact * cf;
  if (contact_cost > a.contact_max) contact_cost = a.contact_max;
  const double reward = (forward_reward + healthy_reward) - (ctrl_cost + contact_cost);
  const bool term = !healthy && a.terminate_when_unhealthy;
  write_info_base(a, i, d);
  const int64_t n = a.n;
  a.info[7 * n + i] = xv;
  a.info[8 * n + i] = yv;
  a.info[9 * n + i] = healthy_reward;
  a.info[10 * n + i] = forward_reward;
  a.info[11 * n + i] = -ctrl_cost;
  a.info[12 * n + i] = -contact_cost;
  const int32_t elapsed = ctrl_elapsed(c) + 1;
  const bool trunc = a.max_steps > 0 && elapsed >= a.max_steps;
  a.reward[i] = reward;
  a.term[i] = term;
  a.trunc[i] = trunc;
  int32_t cn = elapsed;
  if (term || trunc) {
    if (a.mode == B2E_AUTORESET_NEXT_STEP) {
      cn |= kPending;
    } else if (a.mode == B2E_AUTORESET_SAME_STEP) {
      for (int k = 0; k < 348; ++k) a.final_obs[348 * i + k] = obs[k];
      if (D.numpy) D.g = pcg64_load(a.rng, a.n, i);
      env_reset(a, i, d, D, obs);
      if (D.numpy) pcg64_store_state(a.rng, i, D.g);
      cn = 0;
    }
  }
  store_state(a, i, d);
  a.ctrl[i] = cn;
}


#include "humanoid_warp.cuh"  // warp-per-env mapping of the same physics (shares every HD helper above)

static_assert(sizeof(WModel) + kWarpEnvsPerCta * sizeof(WS) <= 227 * 1024,
              "10 envs per CTA must fit the 227 KB of shared memory an sm_100a CTA can opt in to");

template <typename ActT>
int launch_warp_step(const HumanoidArgs& a, cudaStream_t s) {
  constexpr int W = kWarpEnvsPerCta;
  // opt in to > 48 KB of dynamic shared memory once per instantiation AND device (the attribute is per device/context)
  static std::atomic<bool> configured[64];
  const int smem = (int)sizeof(WModel) + W * (int)sizeof(WS);
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 63;  // slot 63 is never latched: always re-applied
  if (dev == 63 || !configured[dev].load(std::memory_order_acquire)) {
    cudaError_t e = cudaFuncSetAttribute(humanoid_step_warp_kernel<ActT, W>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return cuda_status(e, "b2e_humanoid_step (shared memory opt-in)");
    if (dev != 63) configured[dev].store(true, std::memory_order_release);
  }
  if (a.order) humanoid_group_kernel<<<1, 1024, 0, s>>>(a.work, a.order, a.n);
  humanoid_step_warp_kernel<ActT, W><<<(unsigned)((a.n + W - 1) / W), 32 * W, smem, s>>>(a);
  return cuda_status(cudaGetLastError(), "b2e_humanoid_step");
}

int fill(const b2e_batch* b, const b2e_humanoid_cfg* cfg, const b2e_humanoid_state* st, HumanoidArgs& a, const char* fn) {
  if (int e = check_batch(b, fn)) return e;
  if (!cfg || !st || !st->qpos || !st->qvel || !st->qacc_warmstart || !st->com_xy || !st->ctrl || !st->overflow ||
      (b->rng_mode == B2E_RNG_NUMPY && !st->rng)) {
    set_error("%s: null pointer in cfg/state", fn);
    return B2E_EINVAL;
  }
  if (cfg->frame_skip <= 0) {
    set_error("%s: frame_skip must be positive", fn);
    return B2E_EINVAL;
  }
  a = HumanoidArgs{};
  a.n = b->n; a.env_offset = b->env_offset; a.max_steps = b->max_episode_steps; a.mode = b->autoreset_mode;
  a.rng_mode = b->rng_mode; a.philox_seed = b->philox_seed; a.call_counter = b->call_counter;
  a.frame_skip = cfg->frame_skip; a.terminate_when_unhealthy = cfg->terminate_when_unhealthy;
  a.noise = cfg->reset_noise_scale; a.w_forward = cfg->forward_reward_weight; a.w_ctrl = cfg->ctrl_cost_weight;
  a.w_contact = cfg->contact_cost_weight; a.contact_max = cfg->contact_cost_max; a.healthy_reward = cfg->healthy_reward;
  a.z_min = cfg->healthy_z_min; a.z_max = cfg->healthy_z_max;
  a.qpos = st->qpos; a.qvel = st->qvel; a.warm = st->qacc_warmstart; a.com_xy = st->com_xy; a.ctrl = st->ctrl;
  a.rng = st->rng; a.overflow = st->overflow;
  a.work = st->work; a.order = (st->work && st->order) ? st->order : nullptr;
  return upload_model();
}

}  // namespace
}  // namespace b2e

using namespace b2e;

extern "C" int b2e_humanoid_model_info(double* body_mass, double* misc, double* invweight) {
  if (!body_mass || !misc || !invweight) {
    set_error("b2e_humanoid_model_info: null pointer");
    return B2E_EINVAL;
  }
  const HModel& m = host_model();
  for (int b = 0; b < NB; ++b) body_mass[b] = m.body_mass[b];
  misc[0] = m.meaninertia; misc[1] = m.npair; misc[2] = m.subtree_mass[0];
  for (int k = 3; k < 8; ++k) misc[k] = 0;
  for (int b = 0; b < NB; ++b) { invweight[2 * b] = m.body_invweight0[b][0]; invweight[2 * b + 1] = m.body_invweight0[b][1]; }
  for (int i = 0; i < NV; ++i) invweight[2 * NB + i] = m.dof_invweight0[i];
  return 0;
}

extern "C" int b2e_humanoid_reset(const b2e_batch* b, const b2e_humanoid_cfg* cfg, const b2e_humanoid_state* st,
                                  const uint8_t* mask, double* obs, double* info, void* stream) {
  HumanoidArgs a;
  if (int e = fill(b, cfg, st, a, "b2e_humanoid_reset")) return e;
  if (!obs || !info) {
    set_error("b2e_humanoid_reset: null output pointer");
    return B2E_EINVAL;
  }
  if (b->n == 0) return 0;
  a.mask = mask; a.obs = obs; a.info = info;
  if (cfg->impl == 1)
    humanoid_reset_kernel<<<grid_for(b->n, kHumanoidBlock), kHumanoidBlock, 0, (cudaStream_t)stream>>>(a);
  else
    humanoid_reset_warp_kernel<<<(unsigned)b->n, 32, 0, (cudaStream_t)stream>>>(a);
  return cuda_status(cudaGetLastError(), "b2e_humanoid_reset");
}

extern "C" int b2e_humanoid_step(const b2e_batch* b, const b2e_humanoid_cfg* cfg, const b2e_humanoid_state* st,
                                 const void* actions, double* obs, double* reward, uint8_t* terminated,
                                 uint8_t* truncated, double* info, double* final_obs, void* stream) {
  HumanoidArgs a;
  if (int e = fill(b, cfg, st, a, "b2e_humanoid_step")) return e;
  if (!actions || !obs || !reward || !terminated || !truncated || !info ||
      (b->autoreset_mode == B2E_AUTORESET_SAME_STEP && !final_obs)) {
    set_error("b2e_humanoid_step: null pointer");
    return B2E_EINVAL;
  }
  if (b->n == 0) return 0;
  a.actions = actions; a.obs = obs; a.reward = reward; a.term = terminated; a.trunc = truncated; a.info = info;
  a.final_obs = final_obs;
  cudaStream_t s = (cudaStream_t)stream;
  if (cfg->impl != 1) {
    switch (b->action_dtype) {
      case B2E_ACT_F32: return launch_warp_step<float>(a, s);
      case B2E_ACT_F64: return launch_warp_step<double>(a, s);
      default: set_error("b2e_humanoid_step: action_dtype %d is not a float dtype", b->action_dtype); return B2E_EINVAL;
    }
  }
  const unsigned grid = grid_for(b->n, kHumanoidBlock);
  switch (b->action_dtype) {
    case B2E_ACT_F32: humanoid_step_kernel<float><<<grid, kHumanoidBlock, 0, s>>>(a); break;
    case B2E_ACT_F64: humanoid_step_kernel<double><<<grid, kHumanoidBlock, 0, s>>>(a); break;
    default: set_error("b2e_humanoid_step: action_dtype %d is not a float dtype", b->action_dtype); return B2E_EINVAL;
  }
  return cuda_status(cudaGetLastError(), "b2e_humanoid_step");
}
