// mjc_planar.cuh -- fused step + TimeLimit + autoreset kernels (sm_100a) of the planar MuJoCo robots, Hopper-v5 and
// Walker2d-v5: the articulated-body / PGS core of humanoid.cu generalised to slide + hinge joints (no free joint), joint
// `ref`, per-geom friction / condim / contype / conaffinity, capsules given by size + pos + quat, contact solimp and margin
// from the geoms, actuator gear and ctrlrange +-1.  One thread per env (a 6- or 9-dof working set is 6-15 KB).  Included by
// hopper.cu / walker2d.cu, which select the robot with MJC_ROBOT_HOPPER / MJC_ROBOT_WALKER2D.
//
// Replaces, for a batch of n envs in one launch:
//   HopperEnv / Walker2dEnv .step / _get_obs / _get_rew / is_healthy / reset_model
//                                               gymnasium/envs/mujoco/hopper_v5.py:226-343, walker2d_v5.py:257-342
//   MujocoEnv.reset / set_state / _step_mujoco_simulation   gymnasium/envs/mujoco/mujoco_env.py:132-155, 172-187
//   the models                                  gymnasium/envs/mujoco/assets/hopper.xml:1-61, walker2d_v5.xml:1-70
//   TimeLimit / SyncVectorEnv autoreset as in cartpole.cu
// and, below the reference, the MuJoCo subset these models exercise (see humanoid.cu).  Numeric parity with the real wheel is
// UNPINNED (not installable here); the checker is oracle/mjc_planar.h, which these kernels match bit for bit.  Known
// deviation: neither XML names a solver, so MuJoCo runs its default Newton solver (100 iterations, tolerance 1e-8) on the
// pyramidal-cone problem; this file (and the oracle) run PGS on the same convex problem with the same stopping rule -- the
// solutions agree to solver tolerance, the iterates do not.
//
// Arithmetic: float64 like MuJoCo, one IEEE rounding per operation (--fmad=false); control cost in float32 like the
// reference's NumPy expression on float32 actions (hopper_v5.py:226-228, walker2d_v5.py:257-259).
#include <atomic>
#include <assert.h>
#include <string.h>

#include "common.cuh"

#if defined(MJC_ROBOT_HOPPER)
#define MJC_API(name) b2e_hopper_##name
#define MJC_NAME "hopper"
#elif defined(MJC_ROBOT_WALKER2D)
#define MJC_API(name) b2e_walker2d_##name
#define MJC_NAME "walker2d"
#elif defined(MJC_ROBOT_HALFCHEETAH)
#define MJC_API(name) b2e_half_cheetah_##name
#define MJC_NAME "half_cheetah"
#elif defined(MJC_ROBOT_INVPEND)
#define MJC_API(name) b2e_inverted_pendulum_##name
#define MJC_NAME "inverted_pendulum"
#else
#error "define MJC_ROBOT_HOPPER, MJC_ROBOT_WALKER2D, MJC_ROBOT_HALFCHEETAH or MJC_ROBOT_INVPEND before including mjc_planar.cuh"
#endif
#define MJC_STR2(x) #x
#define MJC_STR(x) MJC_STR2(x)

namespace b2e {
namespace {

#define HD __host__ __device__ inline

#if defined(MJC_ROBOT_HOPPER)
constexpr int NB = 5, NQ = 6, NV = 6, NU = 3, NJ = 6, NG = 5, MAXCON = 8, MAXEFC = 16, MAXPAIR = 16;
#elif defined(MJC_ROBOT_HALFCHEETAH)
constexpr int NB = 8, NQ = 9, NV = 9, NU = 6, NJ = 9, NG = 9, MAXCON = 12, MAXEFC = 56, MAXPAIR = 16;
#elif defined(MJC_ROBOT_INVPEND)
constexpr int NB = 3, NQ = 2, NV = 2, NU = 1, NJ = 2, NG = 2, MAXCON = 2, MAXEFC = 4, MAXPAIR = 2;
#else
constexpr int NB = 8, NQ = 9, NV = 9, NU = 6, NJ = 9, NG = 8, MAXCON = 8, MAXEFC = 32, MAXPAIR = 16;
#endif
constexpr double MINVAL = 1e-15, PI = 3.14159265358979323846;
constexpr int G_PLANE = 0, G_SPHERE = 2, G_CAPSULE = 3;

struct HModel {
  int parent[NB], body_jntadr[NB], body_jntnum[NB], body_dofadr[NB], body_dofnum[NB], body_lastdof[NB];
  double body_pos[NB][3], body_quat[NB][4], body_mass[NB], body_ipos[NB][3], body_inertia[NB][9];
  double subtree_mass[NB], body_invweight0[NB][2];
  int jnt_type[NJ] /* 2 slide, 3 hinge */, jnt_body[NJ], jnt_qposadr[NJ], jnt_dofadr[NJ], jnt_limited[NJ];
  double jnt_pos[NJ][3], jnt_axis[NJ][3], jnt_range[NJ][2], jnt_stiffness[NJ];
  int dof_body[NV], dof_parent[NV];
  double dof_armature[NV], dof_damping[NV], dof_invweight0[NV];
  int geom_type[NG], geom_body[NG], geom_condim[NG], geom_contype[NG], geom_conaffinity[NG];
  double geom_pos[NG][3], geom_mat[NG][9], geom_size[NG][2], geom_rbound[NG], geom_friction[NG];
  int act_dof[NU];
  double act_gear[NU], act_ctrlrange[NU][2];
  // solimp: default (joint limits); solimp_contact: the geoms' (hopper.xml:10)
  double timestep, gravity[3], meaninertia, margin, solref[2], solimp[5], solimp_contact[5], tolerance;
  int iterations, npair, pair_g1[MAXPAIR], pair_g2[MAXPAIR];
  double qpos0[NQ];
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
  int ncon, nefc, overflow;
  Contact con[MAXCON];
  double efc_J[MAXEFC][NV], efc_pos[MAXEFC], efc_margin[MAXEFC], efc_D[MAXEFC], efc_R[MAXEFC], efc_aref[MAXEFC],
      efc_b[MAXEFC], efc_force[MAXEFC], efc_diagApprox[MAXEFC];
  int efc_contact[MAXEFC];  // row of a contact (solimp_contact) or of a joint limit (solimp)
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
  const double* q = d.qpos;
  for (int k = 0; k < 3; ++k) { d.xpos[0][k] = 0; d.xipos[0][k] = 0; }
  d.xquat[0][0] = 1; d.xquat[0][1] = d.xquat[0][2] = d.xquat[0][3] = 0;
  for (int k = 0; k < 9; ++k) d.xmat[0][k] = (k % 4 == 0) ? 1.0 : 0.0;
  for (int b = 1; b < NB; ++b) {
    double xpos[3], xquat[4], t[3];
    const int p = m.parent[b];
    mulmatvec3(t, d.xmat[p], m.body_pos[b]);
    for (int k = 0; k < 3; ++k) xpos[k] = d.xpos[p][k] + t[k];
    quat_mul(xquat, d.xquat[p], m.body_quat[b]);
    for (int jj = 0; jj < m.body_jntnum[b]; ++jj) {
      const int j = m.body_jntadr[b] + jj;
      double v[3];
      quat_rot(v, xquat, m.jnt_pos[j]);
      for (int k = 0; k < 3; ++k) d.xanchor[j][k] = xpos[k] + v[k];
      quat_rot(d.xaxis[j], xquat, m.jnt_axis[j]);
      const double disp = q[m.jnt_qposadr[j]] - m.qpos0[m.jnt_qposadr[j]];
      if (m.jnt_type[j] == 2) {  // slide: translate along the axis
        for (int k = 0; k < 3; ++k) xpos[k] += d.xaxis[j][k] * disp;
      } else {  // hinge: rotate about the axis through the anchor
        double ql[4];
        quat_axisangle(ql, m.jnt_axis[j], disp);
        quat_mul(xquat, xquat, ql);
        quat_rot(v, xquat, m.jnt_pos[j]);
        for (int k = 0; k < 3; ++k) xpos[k] = d.xanchor[j][k] - v[k];
      }
    }
    quat_normalize(xquat);
    cp3(d.xpos[b], xpos);
    for (int k = 0; k < 4; ++k) d.xquat[b][k] = xquat[k];
    quat2mat(d.xmat[b], xquat);
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
    if (m.jnt_type[j] == 2) {  // slide: pure translation along the axis
      d.cdof[da][0] = d.cdof[da][1] = d.cdof[da][2] = 0;
      cp3(d.cdof[da] + 3, d.xaxis[j]);
    } else {
      cp3(d.cdof[da], d.xaxis[j]);
      cross3(d.cdof[da] + 3, d.xaxis[j], off);
    }
  }
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
HD double impedance(const double* solimp, double pos, double margin) {
  const double dmin = solimp[0], dmax = solimp[1], width = solimp[2], mid = solimp[3];
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
  for (int j = 0; j < NJ; ++j) {
    if (!m.jnt_limited[j]) continue;
    const double value = d.qpos[m.jnt_qposadr[j]];
    for (int side = -1; side <= 1; side += 2) {
      const double dist = side * (m.jnt_range[j][(side + 1) / 2] - value);
      if (dist < 0.0 && n < MAXEFC) {
        for (int k = 0; k < NV; ++k) d.efc_J[n][k] = 0;
        d.efc_J[n][m.jnt_dofadr[j]] = -side;
        d.efc_pos[n] = dist; d.efc_margin[n] = 0.0;
        d.efc_diagApprox[n] = m.dof_invweight0[m.jnt_dofadr[j]];
        d.efc_contact[n] = 0;
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
      d.efc_contact[n] = 1;
      ++n;
    } else {
      for (int k = 1; k <= 2; ++k)
        for (int sgn = 1; sgn >= -1; sgn -= 2) {
          for (int i = 0; i < NV; ++i) d.efc_J[n][i] = Jc[0][i] + sgn * con.mu * Jc[k][i];
          d.efc_pos[n] = con.dist; d.efc_margin[n] = m.margin;
          d.efc_diagApprox[n] = tran + con.mu * con.mu * tran;
          d.efc_contact[n] = 1;
          ++n;
        }
    }
  }
  d.nefc = n;
  const double timeconst = m.solref[0] > 2 * m.timestep ? m.solref[0] : 2 * m.timestep, dampratio = m.solref[1];
  for (int i = 0; i < n; ++i) {
    const double* solimp = d.efc_contact[i] ? m.solimp_contact : m.solimp;
    const double dmax = solimp[1];
    const double K = 1.0 / (dmax * dmax * timeconst * timeconst * dampratio * dampratio), B = 2.0 / (dmax * timeconst);
    const double imp = impedance(solimp, d.efc_pos[i], d.efc_margin[i]);
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
      cross_motion(d.cdof_dot[da], cvel, d.cdof[da]);  // slide and hinge alike
      for (int k = 0; k < 6; ++k) cvel[k] += d.cdof[da][k] * d.qvel[da];
    }
    for (int k = 0; k < 6; ++k) d.cvel[b][k] = cvel[k];
  }
  for (int i = 0; i < NV; ++i) d.qfrc_passive[i] = 0;  // mj_passive
  for (int j = 0; j < NJ; ++j) {
    const int da = m.jnt_dofadr[j], qa = m.jnt_qposadr[j];
    d.qfrc_passive[da] = -m.jnt_stiffness[j] * (d.qpos[qa] - m.qpos0[qa]) - m.dof_damping[da] * d.qvel[da];
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
    c = c < m.act_ctrlrange[u][0] ? m.act_ctrlrange[u][0] : (c > m.act_ctrlrange[u][1] ? m.act_ctrlrange[u][1] : c);  // hopper.xml:45-47
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
  for (int i = 0; i < NV; ++i) qpos[i] += h * vel[i];  // slide and hinge joints only
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
// mj_Euler (engine_forward.c: mj_EulerSkip + mj_advance): semi-implicit Euler with the joint damping treated implicitly --
// qacc' = (M + h diag(B))^-1 (qfrc_smooth + qfrc_constraint); qvel += h qacc'; qpos += h qvel (the NEW velocity);
// qacc_warmstart = the forward dynamics' qacc
HD void mj_step_euler(const HModel& m, HData& d) {
  const double h = m.timestep;
  mj_forward(m, d);
  double qacc[NV];
  bool damped = false;
  for (int i = 0; i < NV; ++i) damped = damped || m.dof_damping[i] > 0;
  if (!damped) {
    for (int i = 0; i < NV; ++i) qacc[i] = d.qacc[i];
  } else {
    double H[NV][NV], Hinv[NV];
    for (int i = 0; i < NV; ++i) for (int j = 0; j < NV; ++j) H[i][j] = d.qM[i][j];
    for (int i = 0; i < NV; ++i) H[i][i] += h * m.dof_damping[i];
    for (int k = NV - 1; k >= 0; --k) {  // mj_factorI: the same L^T D L as crb_and_factor
      for (int i = m.dof_parent[k]; i >= 0; i = m.dof_parent[i]) {
        const double tmp = H[k][i] / H[k][k];
        for (int j = i; j >= 0; j = m.dof_parent[j]) H[i][j] -= H[k][j] * tmp;
        H[k][i] = tmp;
      }
      Hinv[k] = 1.0 / H[k][k];
    }
    for (int i = 0; i < NV; ++i) qacc[i] = d.qfrc_smooth[i] + d.qfrc_constraint[i];
    for (int i = NV - 1; i >= 0; --i)  // mj_solveLD
      for (int j = m.dof_parent[i]; j >= 0; j = m.dof_parent[j]) qacc[j] -= H[i][j] * qacc[i];
    for (int i = 0; i < NV; ++i) qacc[i] *= Hinv[i];
    for (int i = 0; i < NV; ++i)
      for (int j = m.dof_parent[i]; j >= 0; j = m.dof_parent[j]) qacc[i] -= H[i][j] * qacc[j];
  }
  for (int k = 0; k < NV; ++k) d.qvel[k] += h * qacc[k];
  integrate_pos(d.qpos, d.qvel, h);
  for (int k = 0; k < NV; ++k) d.qacc_warmstart[k] = d.qacc[k];  // mj_advance
}
// ---- models (hopper.xml / walker2d_v5.xml re-typed as data) + compile --------------------------------------------------------
struct BDef { int parent; double pos[3]; };
struct JDef { int type, body; double pos[3], axis[3]; int limited; double lo, hi, armature, damping, ref; };
struct GDef { int type, body; double pos[3], quat[4], r, half, friction; int condim, contype, conaffinity; };
#define MJC_FOOT_QUAT {0.70710678118654757, 0, -0.70710678118654746, 0}
#if defined(MJC_ROBOT_HOPPER)
// hopper.xml: defaults joint armature 1 damping 1 limited (:9), geom condim 1 contype 1 conaffinity 1 margin 0.001 solimp
// .8 .8 .01 (:10); floor condim 3 (:19); RK4, timestep 0.002 (:12); motors gear 200, ctrlrange +-1 (:44-48)
const BDef BODY[NB] = {{0, {0, 0, 0}}, {0, {0, 0, 1.25}}, {1, {0, 0, -0.19999999999999996}}, {2, {0, 0, -0.70000000000000007}},
                       {3, {0.13, 0, -0.35}}};
const JDef JOINT[NJ] = {
    {2, 1, {0, 0, -1.25}, {1, 0, 0}, 0, 0, 0, 0, 0, 0},        // rootx (slide)
    {2, 1, {0, 0, -1.25}, {0, 0, 1}, 0, 0, 0, 0, 0, 1.25},     // rootz (slide, ref 1.25)
    {3, 1, {0, 0, 0}, {0, 1, 0}, 0, 0, 0, 0, 0, 0},            // rooty
    {3, 2, {0, 0, 0}, {0, -1, 0}, 1, -150, 0, 1, 1, 0},        // thigh_joint
    {3, 3, {0, 0, 0.25}, {0, -1, 0}, 1, -150, 0, 1, 1, 0},     // leg_joint
    {3, 4, {-0.13, 0, 0.1}, {0, -1, 0}, 1, -45, 45, 1, 1, 0},  // foot_joint
};
const GDef GEOM[NG] = {
    {G_PLANE, 0, {0, 0, 0}, {1, 0, 0, 0}, 0, 0, 1.0, 3, 1, 1},
    {G_CAPSULE, 1, {0, 0, 0}, {1, 0, 0, 0}, 0.05, 0.19999999999999996, 0.9, 1, 1, 1},
    {G_CAPSULE, 2, {0, 0, -0.22500000000000009}, {1, 0, 0, 0}, 0.05, 0.22500000000000003, 0.9, 1, 1, 1},
    {G_CAPSULE, 3, {0, 0, 0}, {1, 0, 0, 0}, 0.04, 0.25, 0.9, 1, 1, 1},
    {G_CAPSULE, 4, {-0.065, 0, 0.1}, MJC_FOOT_QUAT, 0.06, 0.195, 2.0, 1, 1, 1},
};
const int ACT_JOINT[NU] = {3, 4, 5};
constexpr double kGear = 200.0, kMargin = 0.001;
const double kSolimpContact[5] = {0.8, 0.8, 0.01, 0.5, 2.0};
#elif defined(MJC_ROBOT_HALFCHEETAH)
// half_cheetah.xml: compiler angle="radian" settotalmass="14" (:35); defaults joint armature .1 damping .01 limited solimplimit
// 0 .8 .03 solreflimit .02 1 stiffness 8 (:37; every hinge overrides damping / stiffness), geom conaffinity 0 condim 3 contype 1
// friction .4 solimp 0 .8 .01 solref .02 1 (:38: the robot collides with the floor only); option timestep 0.01, integrator left
// at its default = Euler (:42); root joints: armature 0 damping 0 stiffness 0 (:55-57); motors gear 120 90 60 120 60 30 (:88-93)
const BDef BODY[NB] = {{0, {0, 0, 0}}, {0, {0, 0, 0.7}},
                       {1, {-0.5, 0, 0}}, {2, {0.16, 0, -0.25}}, {3, {-0.28, 0, -0.14}},
                       {1, {0.5, 0, 0}}, {5, {-0.14, 0, -0.24}}, {6, {0.13, 0, -0.18}}};
const JDef JOINT[NJ] = {  // ranges in radians
    {2, 1, {0, 0, 0}, {1, 0, 0}, 0, 0, 0, 0, 0, 0},             // rootx
    {2, 1, {0, 0, 0}, {0, 0, 1}, 0, 0, 0, 0, 0, 0},             // rootz
    {3, 1, {0, 0, 0}, {0, 1, 0}, 0, 0, 0, 0, 0, 0},             // rooty
    {3, 2, {0, 0, 0}, {0, 1, 0}, 1, -0.52, 1.05, 0.1, 6, 0},     // bthigh
    {3, 3, {0, 0, 0}, {0, 1, 0}, 1, -0.785, 0.785, 0.1, 4.5, 0}, // bshin
    {3, 4, {0, 0, 0}, {0, 1, 0}, 1, -0.4, 0.785, 0.1, 3, 0},     // bfoot
    {3, 5, {0, 0, 0}, {0, 1, 0}, 1, -1, 0.7, 0.1, 4.5, 0},       // fthigh
    {3, 6, {0, 0, 0}, {0, 1, 0}, 1, -1.2, 0.87, 0.1, 3, 0},      // fshin
    {3, 7, {0, 0, 0}, {0, 1, 0}, 1, -0.5, 0.5, 0.1, 1.5, 0},     // ffoot
};
const double JOINT_STIFFNESS[NJ] = {0, 0, 0, 240, 180, 120, 180, 120, 60};
const GDef GEOM[NG] = {
    {G_PLANE, 0, {0, 0, 0}, {1, 0, 0, 0}, 0, 0, 0.4, 3, 1, 1},
    {G_CAPSULE, 1, {0, 0, 0}, {1, 0, 0, 0}, 0.046, 0.5, 0.4, 3, 1, 0},           // torso: fromto -.5 0 0 .5 0 0
    {G_CAPSULE, 1, {0.6, 0, 0.1}, {1, 0, 0, 0}, 0.046, 0.15, 0.4, 3, 1, 0},      // head: axisangle 0 1 0 .87
    {G_CAPSULE, 2, {0.1, 0, -0.13}, {1, 0, 0, 0}, 0.046, 0.145, 0.4, 3, 1, 0},   // bthigh: -3.8
    {G_CAPSULE, 3, {-0.14, 0, -0.07}, {1, 0, 0, 0}, 0.046, 0.15, 0.4, 3, 1, 0},  // bshin: -2.03
    {G_CAPSULE, 4, {0.03, 0, -0.097}, {1, 0, 0, 0}, 0.046, 0.094, 0.4, 3, 1, 0}, // bfoot: -.27
    {G_CAPSULE, 5, {-0.07, 0, -0.12}, {1, 0, 0, 0}, 0.046, 0.133, 0.4, 3, 1, 0}, // fthigh: .52
    {G_CAPSULE, 6, {0.065, 0, -0.09}, {1, 0, 0, 0}, 0.046, 0.106, 0.4, 3, 1, 0}, // fshin: -.6
    {G_CAPSULE, 7, {0.045, 0, -0.07}, {1, 0, 0, 0}, 0.046, 0.07, 0.4, 3, 1, 0},  // ffoot: -.6
};
// orientation / placement spec per geom: kind 0 = the quat above, 1 = axisangle about +y with angle a[0], 2 = fromto a[0..5]
struct GSpec { int kind; double a[6]; };
const GSpec GEOM_SPEC[NG] = {
    {0, {0}}, {2, {-0.5, 0, 0, 0.5, 0, 0}}, {1, {0.87}}, {1, {-3.8}}, {1, {-2.03}}, {1, {-0.27}}, {1, {0.52}}, {1, {-0.6}}, {1, {-0.6}}};
const int ACT_JOINT[NU] = {3, 4, 5, 6, 7, 8};
const double ACT_GEAR[NU] = {120.0, 90.0, 60.0, 120.0, 60.0, 30.0};
constexpr double kGear = 0.0, kMargin = 0.0;  // kGear unused: per-actuator gears above
const double kSolimpContact[5] = {0.0, 0.8, 0.01, 0.5, 2.0};
const double kSolimpLimit[5] = {0.0, 0.8, 0.03, 0.5, 2.0};
#define MJC_TIMESTEP 0.01
#define MJC_CTRLRANGE 1.0
#define MJC_ANGLE_RADIAN 1
#define MJC_TOTALMASS 14.0
#define MJC_EULER 1
#elif defined(MJC_ROBOT_INVPEND)
// inverted_pendulum.xml: defaults joint armature 0 damping 1 limited (:4), geom contype 0 (:5: nothing collides), motor
// ctrlrange -3 3 gear 100 (:7, :27); RK4, timestep 0.02 (:9); the rail (a world geom, :13) takes part in nothing and is left
// out.  Slide ranges are lengths, hinge ranges degrees.  The pole's capsule is given by fromto (:19): see build_model.
const BDef BODY[NB] = {{0, {0, 0, 0}}, {0, {0, 0, 0}}, {1, {0, 0, 0}}};
const JDef JOINT[NJ] = {
    {2, 1, {0, 0, 0}, {1, 0, 0}, 1, -1, 1, 0, 1, 0},    // slider
    {3, 2, {0, 0, 0}, {0, 1, 0}, 1, -90, 90, 0, 1, 0},  // hinge
};
const double kPoleFromTo[6] = {0, 0, 0, 0.001, 0, 0.6};
const GDef GEOM[NG] = {
    {G_CAPSULE, 1, {0, 0, 0}, {0.707, 0, 0.707, 0}, 0.1, 0.1, 1.0, 3, 0, 1},  // cart
    {G_CAPSULE, 2, {0, 0, 0}, {1, 0, 0, 0}, 0.049, 0.3, 1.0, 3, 0, 1},         // cpole: pos / quat / half length from fromto
};
const int ACT_JOINT[NU] = {0};
constexpr double kGear = 100.0, kMargin = 0.0;
const double kSolimpContact[5] = {0.9, 0.95, 0.001, 0.5, 2.0};
#define MJC_TIMESTEP 0.02
#define MJC_CTRLRANGE 3.0
#else
// walker2d_v5.xml: defaults joint armature 0.01 damping .1 limited (:10), geom condim 3 contype 1 conaffinity 0 friction .7
// (:11: the robot's geoms collide with the floor only); floor conaffinity 1 (:16); RK4, timestep 0.002 (:13); gear 100 (:57-62)
const BDef BODY[NB] = {{0, {0, 0, 0}}, {0, {0, 0, 1.25}},
                       {1, {0, 0, -0.19999999999999996}}, {2, {0, 0, -0.70000000000000007}},
                       {3, {0.20000000000000001, 0, -0.34999999999999998}},
                       {1, {0, 0, -0.19999999999999996}}, {5, {0, 0, -0.70000000000000007}},
                       {6, {0.20000000000000001, 0, -0.34999999999999998}}};
const JDef JOINT[NJ] = {
    {2, 1, {0, 0, -1.25}, {1, 0, 0}, 0, 0, 0, 0, 0, 0},
    {2, 1, {0, 0, -1.25}, {0, 0, 1}, 0, 0, 0, 0, 0, 1.25},
    {3, 1, {0, 0, 0}, {0, 1, 0}, 0, 0, 0, 0, 0, 0},
    {3, 2, {0, 0, 0}, {0, -1, 0}, 1, -150, 0, 0.01, 0.1, 0},
    {3, 3, {0, 0, 0.25}, {0, -1, 0}, 1, -150, 0, 0.01, 0.1, 0},
    {3, 4, {-0.20000000000000001, 0, 0.10000000000000001}, {0, -1, 0}, 1, -45, 45, 0.01, 0.1, 0},
    {3, 5, {0, 0, 0}, {0, -1, 0}, 1, -150, 0, 0.01, 0.1, 0},
    {3, 6, {0, 0, 0.25}, {0, -1, 0}, 1, -150, 0, 0.01, 0.1, 0},
    {3, 7, {-0.20000000000000001, 0, 0.10000000000000001}, {0, -1, 0}, 1, -45, 45, 0.01, 0.1, 0},
};
const GDef GEOM[NG] = {
    {G_PLANE, 0, {0, 0, 0}, {1, 0, 0, 0}, 0, 0, 0.7, 3, 1, 1},
    {G_CAPSULE, 1, {0, 0, 0}, {1, 0, 0, 0}, 0.050000000000000003, 0.19999999999999996, 0.9, 3, 1, 0},
    {G_CAPSULE, 2, {0, 0, -0.22500000000000009}, {1, 0, 0, 0}, 0.050000000000000003, 0.22500000000000003, 0.9, 3, 1, 0},
    {G_CAPSULE, 3, {0, 0, 0}, {1, 0, 0, 0}, 0.040000000000000001, 0.25, 0.9, 3, 1, 0},
    {G_CAPSULE, 4, {-0.10000000000000001, 0, 0.10000000000000001}, MJC_FOOT_QUAT, 0.059999999999999998, 0.10000000000000001, 1.9, 3, 1, 0},
    {G_CAPSULE, 5, {0, 0, -0.22500000000000009}, {1, 0, 0, 0}, 0.050000000000000003, 0.22500000000000003, 0.9, 3, 1, 0},
    {G_CAPSULE, 6, {0, 0, 0}, {1, 0, 0, 0}, 0.040000000000000001, 0.25, 0.9, 3, 1, 0},
    {G_CAPSULE, 7, {-0.10000000000000001, 0, 0.10000000000000001}, MJC_FOOT_QUAT, 0.059999999999999998, 0.10000000000000001, 1.9, 3, 1, 0},
};
const int ACT_JOINT[NU] = {3, 4, 5, 6, 7, 8};
constexpr double kGear = 100.0, kMargin = 0.0;
const double kSolimpContact[5] = {0.9, 0.95, 0.001, 0.5, 2.0};
#endif

#ifndef MJC_TIMESTEP
#define MJC_TIMESTEP 0.002
#define MJC_CTRLRANGE 1.0
#endif

void build_model(HModel& m) {
  const double DEG = PI / 180.0;
  memset(&m, 0, sizeof(m));
  m.timestep = MJC_TIMESTEP; m.gravity[2] = -9.81; m.margin = kMargin; m.tolerance = 1e-8; m.iterations = 100;
  m.solref[0] = 0.02; m.solref[1] = 1.0;
  m.solimp[0] = 0.9; m.solimp[1] = 0.95; m.solimp[2] = 0.001; m.solimp[3] = 0.5; m.solimp[4] = 2.0;
  for (int k = 0; k < 5; ++k) m.solimp_contact[k] = kSolimpContact[k];
#if defined(MJC_ROBOT_HALFCHEETAH)
  for (int k = 0; k < 5; ++k) m.solimp[k] = kSolimpLimit[k];
#endif
  // getsolparam (engine_core_constraint.c): dmin and dmax are clipped to [mjMINIMP, mjMAXIMP] = [0.0001, 0.9999]
  for (int k = 0; k < 2; ++k) {
    m.solimp[k] = m.solimp[k] < 0.0001 ? 0.0001 : (m.solimp[k] > 0.9999 ? 0.9999 : m.solimp[k]);
    m.solimp_contact[k] = m.solimp_contact[k] < 0.0001 ? 0.0001 : (m.solimp_contact[k] > 0.9999 ? 0.9999 : m.solimp_contact[k]);
  }
  for (int b = 0; b < NB; ++b) {
    m.parent[b] = BODY[b].parent;
    cp3(m.body_pos[b], BODY[b].pos);
    m.body_quat[b][0] = 1;
    m.body_jntadr[b] = -1; m.body_dofadr[b] = -1;
  }
  for (int j = 0; j < NJ; ++j) {  // one dof and one qpos entry per joint
    const JDef& J = JOINT[j];
    m.jnt_type[j] = J.type; m.jnt_body[j] = J.body; m.jnt_qposadr[j] = j; m.jnt_dofadr[j] = j;
    cp3(m.jnt_pos[j], J.pos);
    cp3(m.jnt_axis[j], J.axis);
    normalize3(m.jnt_axis[j]);
    m.jnt_limited[j] = J.limited;
#if defined(MJC_ANGLE_RADIAN)
    const double unit = 1.0;                       // compiler angle="radian"
#else
    const double unit = J.type == 3 ? DEG : 1.0;  // compiler angle="degree" applies to hinges only
#endif
    m.jnt_range[j][0] = J.lo * unit; m.jnt_range[j][1] = J.hi * unit;
#if defined(MJC_ROBOT_HALFCHEETAH)
    m.jnt_stiffness[j] = JOINT_STIFFNESS[j];
#else
    m.jnt_stiffness[j] = 0.0;
#endif
    m.dof_armature[j] = J.armature; m.dof_damping[j] = J.damping;
    m.qpos0[j] = J.ref;
  }
  for (int j = 0; j < NJ; ++j) {
    const int b = m.jnt_body[j];
    if (m.body_jntadr[b] < 0) { m.body_jntadr[b] = j; m.body_dofadr[b] = m.jnt_dofadr[j]; }
    m.body_jntnum[b] += 1;
    m.body_dofnum[b] += 1;
  }
  for (int i = 0; i < NV; ++i) m.dof_body[i] = m.jnt_body[i];
  m.body_lastdof[0] = -1;
  for (int b = 1; b < NB; ++b)
    m.body_lastdof[b] = m.body_dofnum[b] ? m.body_dofadr[b] + m.body_dofnum[b] - 1 : m.body_lastdof[m.parent[b]];
  for (int i = 0; i < NV; ++i) {
    const int b = m.dof_body[i];
    m.dof_parent[i] = i > m.body_dofadr[b] ? i - 1 : m.body_lastdof[m.parent[b]];
  }
  double bm[NB] = {0}, bcom[NB][3] = {{0}}, gmass[NG], gI[NG][9];
  for (int g = 0; g < NG; ++g) {  // geoms + inertia from geoms (density 1000)
    const GDef& G = GEOM[g];
    m.geom_type[g] = G.type; m.geom_body[g] = G.body; m.geom_condim[g] = G.condim;
    m.geom_contype[g] = G.contype; m.geom_conaffinity[g] = G.conaffinity;
    m.geom_friction[g] = G.friction;
    double I[3] = {0, 0, 0}, q[4] = {G.quat[0], G.quat[1], G.quat[2], G.quat[3]}, gpos[3], ghalf = G.half;
    cp3(gpos, G.pos);
#if defined(MJC_ROBOT_INVPEND)
    if (g == 1) {  // capsule from `fromto`: centre = midpoint, half length = |to - from| / 2, frame = the rotation taking z
                   // onto the segment about z x segment (user_objects.cc mjCGeom::Compile / mjuu_z2quat)
      const double* ft = kPoleFromTo;
      double vec[3] = {ft[3] - ft[0], ft[4] - ft[1], ft[5] - ft[2]}, z[3] = {0, 0, 1}, axis[3];
      for (int k = 0; k < 3; ++k) gpos[k] = 0.5 * (ft[k] + ft[3 + k]);
      ghalf = 0.5 * normalize3(vec);
      cross3(axis, z, vec);
      const double sn = norm3(axis);
      if (sn < 1e-10) { axis[0] = 1; axis[1] = 0; axis[2] = 0; } else { axis[0] /= sn; axis[1] /= sn; axis[2] /= sn; }
      const double ang = atan2(sn, vec[2]);
      q[0] = cos(0.5 * ang); q[1] = axis[0] * sin(0.5 * ang); q[2] = axis[1] * sin(0.5 * ang); q[3] = axis[2] * sin(0.5 * ang);
    }
#endif
#if defined(MJC_ROBOT_HALFCHEETAH)
    if (GEOM_SPEC[g].kind == 1) {  // axisangle="0 1 0 a" (radians): quat = (cos a/2, 0, sin a/2, 0)
      const double ang = GEOM_SPEC[g].a[0];
      q[0] = cos(0.5 * ang); q[1] = 0; q[2] = sin(0.5 * ang); q[3] = 0;
    } else if (GEOM_SPEC[g].kind == 2) {  // fromto: as for the inverted pendulum's pole
      const double* ft = GEOM_SPEC[g].a;
      double vec[3] = {ft[3] - ft[0], ft[4] - ft[1], ft[5] - ft[2]}, z[3] = {0, 0, 1}, axis[3];
      for (int k = 0; k < 3; ++k) gpos[k] = 0.5 * (ft[k] + ft[3 + k]);
      ghalf = 0.5 * normalize3(vec);
      cross3(axis, z, vec);
      const double sn = norm3(axis);
      if (sn < 1e-10) { axis[0] = 1; axis[1] = 0; axis[2] = 0; } else { axis[0] /= sn; axis[1] /= sn; axis[2] /= sn; }
      const double ang = atan2(sn, vec[2]);
      q[0] = cos(0.5 * ang); q[1] = axis[0] * sin(0.5 * ang); q[2] = axis[1] * sin(0.5 * ang); q[3] = axis[2] * sin(0.5 * ang);
    }
#endif
    quat_normalize(q);
    quat2mat(m.geom_mat[g], q);
    cp3(m.geom_pos[g], gpos);
    gmass[g] = 0;
    if (G.type == G_PLANE) {
      m.geom_rbound[g] = 0;
    } else {
      const double r = G.r, half = ghalf, h = 2.0 * half;
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
    const int b = G.body;
    bm[b] += gmass[g];
    for (int k = 0; k < 3; ++k) bcom[b][k] += gmass[g] * m.geom_pos[g][k];
  }
  for (int b = 1; b < NB; ++b) {
    m.body_mass[b] = bm[b];
    for (int k = 0; k < 3; ++k) m.body_ipos[b][k] = bcom[b][k] / bm[b];
  }
  for (int g = 0; g < NG; ++g) {  // parallel-axis accumulation about the body com
    const int b = GEOM[g].body;
    if (b == 0) continue;  // world geoms (the floor) carry no inertia
    const double dv[3] = {m.geom_pos[g][0] - m.body_ipos[b][0], m.geom_pos[g][1] - m.body_ipos[b][1],
                          m.geom_pos[g][2] - m.body_ipos[b][2]};
    const double d2 = dot3(dv, dv);
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j)
        m.body_inertia[b][3 * i + j] += gI[g][3 * i + j] + gmass[g] * ((i == j ? d2 : 0.0) - dv[i] * dv[j]);
  }
#if defined(MJC_TOTALMASS)
  {  // compiler settotalmass: every body's mass and inertia scaled so that the masses add up to it (user_model.cc)
    double total = 0;
    for (int b = 1; b < NB; ++b) total += m.body_mass[b];
    const double scale = MJC_TOTALMASS / total;
    for (int b = 1; b < NB; ++b) {
      m.body_mass[b] *= scale;
      for (int k = 0; k < 9; ++k) m.body_inertia[b][k] *= scale;
    }
  }
#endif
  for (int b = NB - 1; b >= 0; --b) m.subtree_mass[b] = m.body_mass[b];
  for (int b = NB - 1; b >= 1; --b) m.subtree_mass[m.parent[b]] += m.subtree_mass[b];
  for (int u = 0; u < NU; ++u) {
#if defined(MJC_ROBOT_HALFCHEETAH)
    m.act_dof[u] = m.jnt_dofadr[ACT_JOINT[u]]; m.act_gear[u] = ACT_GEAR[u];
#else
    m.act_dof[u] = m.jnt_dofadr[ACT_JOINT[u]]; m.act_gear[u] = kGear;
#endif
    m.act_ctrlrange[u][0] = -MJC_CTRLRANGE; m.act_ctrlrange[u][1] = MJC_CTRLRANGE;
  }
  m.npair = 0;
  for (int b1 = 0; b1 < NB; ++b1)
    for (int b2 = b1 + 1; b2 < NB; ++b2) {
      if (b1 != 0 && (m.parent[b2] == b1 || m.parent[b1] == b2)) continue;
      for (int g1 = 0; g1 < NG; ++g1)
        for (int g2 = 0; g2 < NG; ++g2) {
          if (m.geom_body[g1] != b1 || m.geom_body[g2] != b2) continue;
          if (!((m.geom_contype[g1] & m.geom_conaffinity[g2]) || (m.geom_contype[g2] & m.geom_conaffinity[g1]))) continue;
          int a = g1, c = g2;
          if (m.geom_type[a] > m.geom_type[c]) { const int t = a; a = c; c = t; }
          assert(m.npair < MAXPAIR);
          m.pair_g1[m.npair] = a; m.pair_g2[m.npair] = c; m.npair++;
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

__device__ HModel g_pmodel;  // global (not __constant__): the pair list is indexed divergently

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
  cudaError_t e = cudaMemcpyToSymbol(g_pmodel, &M, sizeof(HModel));
  if (e != cudaSuccess) return cuda_status(e, MJC_NAME " model upload");
  done[dev] = true;
  return 0;
}

// ---- kernels -------------------------------------------------------------------------------------------------------------------
#if defined(MJC_ROBOT_INVPEND)
constexpr int kObs = NQ + NV;  // inverted_pendulum_v5.py:185-186: qpos | qvel, nothing skipped or clipped
#elif defined(MJC_ROBOT_HALFCHEETAH)
constexpr int kObs = NQ - 1 + NV;  // half_cheetah_v5.py:251-259: qpos[1:] | qvel, nothing clipped
#else
constexpr int kObs = NQ - 1 + NV;
#endif
constexpr int kInfo = 6;  // info rows: x_position, z_distance_from_origin, x_velocity, reward_forward, reward_ctrl, reward_survive
struct HopperArgs {
  int64_t n, env_offset;
  int32_t max_steps, mode, rng_mode, frame_skip, terminate_when_unhealthy;
  uint64_t philox_seed, call_counter;
  double noise, w_forward, w_ctrl, healthy_reward, z_min, z_max, angle_min, angle_max, state_min, state_max;
  double* __restrict__ qpos;  // [6][n]
  double* __restrict__ qvel;  // [6][n]
  double* __restrict__ warm;  // [6][n] qacc_warmstart
  int32_t* __restrict__ ctrl;
  uint64_t* __restrict__ rng;
  int32_t* __restrict__ overflow;  // [1] sticky
  double* __restrict__ obs;        // [n][11]
  double* __restrict__ reward;
  uint8_t* __restrict__ term;
  uint8_t* __restrict__ trunc;
  double* __restrict__ info;       // [6][n]
  double* __restrict__ final_obs;
  const void* __restrict__ actions; // [n][3] float32 or float64
  const uint8_t* __restrict__ mask;
};

#if defined(MJC_ROBOT_INVPEND)
__device__ void write_obs(const HData& d, double* __restrict__ obs) {  // inverted_pendulum_v5.py:185-186
  for (int i = 0; i < NQ; ++i) obs[i] = d.qpos[i];
  for (int i = 0; i < NV; ++i) obs[NQ + i] = d.qvel[i];
}
#elif defined(MJC_ROBOT_HALFCHEETAH)
__device__ void write_obs(const HData& d, double* __restrict__ obs) {  // half_cheetah_v5.py:251-259
  int o = 0;
  for (int i = 1; i < NQ; ++i) obs[o++] = d.qpos[i];
  for (int i = 0; i < NV; ++i) obs[o++] = d.qvel[i];
}
#else
__device__ void write_obs(const HData& d, double* __restrict__ obs) {  // hopper_v5.py:253-261
  int o = 0;
  for (int i = 1; i < NQ; ++i) obs[o++] = d.qpos[i];
  for (int i = 0; i < NV; ++i) { const double v = d.qvel[i]; obs[o++] = v < -10.0 ? -10.0 : (v > 10.0 ? 10.0 : v); }
}
#endif
__device__ bool is_healthy(const HopperArgs& a, const HData& d) {
  const double z = d.qpos[1], angle = d.qpos[2];
  bool ok = true;
#if defined(MJC_ROBOT_HOPPER)  // hopper_v5.py:231-247: state = qpos[2:] + qvel inside healthy_state_range
  for (int i = 2; i < NQ; ++i) ok = ok && (a.state_min < d.qpos[i] && d.qpos[i] < a.state_max);
  for (int i = 0; i < NV; ++i) ok = ok && (a.state_min < d.qvel[i] && d.qvel[i] < a.state_max);
#endif  // walker2d_v5.py:261-272: height and angle only
  return ok && (a.z_min < z && z < a.z_max) && (a.angle_min < angle && angle < a.angle_max);
}

#if defined(MJC_ROBOT_HALFCHEETAH)
// Generator.standard_normal: numpy/random/src/distributions/distributions.c random_standard_normal (256-strip ziggurat over the
// 64-bit words of the env's PCG64 stream; tables = numpy's own doubles).  The two slow paths use exp / log from fixed IEEE
// sequences shared with oracle/mjc_planar.h (det_exp, det_log).
#define B2E_ZIG_QUAL __device__
#include "ziggurat_tables.inc"
__device__ inline double det_exp(double y) {  // y <= 0 here
  const double k = rint(y * 1.44269504088896338700e+00);
  const double r = (y - k * 6.93147180369123816490e-01) - k * 1.90821492927058770002e-10;
  double p = 1.0 / 6227020800.0;
  p = p * r + 1.0 / 479001600.0;
  p = p * r + 1.0 / 39916800.0;
  p = p * r + 1.0 / 3628800.0;
  p = p * r + 1.0 / 362880.0;
  p = p * r + 1.0 / 40320.0;
  p = p * r + 1.0 / 5040.0;
  p = p * r + 1.0 / 720.0;
  p = p * r + 1.0 / 120.0;
  p = p * r + 1.0 / 24.0;
  p = p * r + 1.0 / 6.0;
  p = p * r + 0.5;
  p = p * r + 1.0;
  p = p * r + 1.0;
  const int ik = (int)k;
  return ik >= 0 ? p * (double)(1ull << ik) : (ik > -63 ? p / (double)(1ull << -ik) : 0.0);
}
__device__ inline double det_log(double y) {  // y in (0, 1]
  uint64_t bits = (uint64_t)__double_as_longlong(y);
  int e = (int)((bits >> 52) & 0x7ff) - 1023;
  bits = (bits & 0x000fffffffffffffull) | 0x3ff0000000000000ull;
  double mant = __longlong_as_double((long long)bits);  // [1, 2)
  if (mant > 1.41421356237309514547) { mant *= 0.5; e += 1; }
  const double s = (mant - 1.0) / (mant + 1.0), z = s * s;
  double p = 1.0 / 23.0;
  p = p * z + 1.0 / 21.0;
  p = p * z + 1.0 / 19.0;
  p = p * z + 1.0 / 17.0;
  p = p * z + 1.0 / 15.0;
  p = p * z + 1.0 / 13.0;
  p = p * z + 1.0 / 11.0;
  p = p * z + 1.0 / 9.0;
  p = p * z + 1.0 / 7.0;
  p = p * z + 1.0 / 5.0;
  p = p * z + 1.0 / 3.0;
  p = p * z + 1.0;
  return (double)e * 6.93147180369123816490e-01 + ((double)e * 1.90821492927058770002e-10 + 2.0 * s * p);
}
#endif

// uniform draws for reset noise: numpy stream or Philox
struct PDraws {
  Pcg64 g;
  bool numpy;
  uint64_t seed, env, counter;
  uint32_t k;
  __device__ double next() {
    if (numpy) return g.next_double();
    const uint4 r = philox_block(seed, env, counter, 48u + (k >> 1));
    const double u = (k & 1u) ? u53_to_double(r.z, r.w) : u53_to_double(r.x, r.y);
    ++k;
    return u;
  }
#if defined(MJC_ROBOT_HALFCHEETAH)
  __device__ double normal() {
    if (!numpy) {  // Philox mode is not a parity mode: Box-Muller on two counter-based uniforms
      const double u1 = 1.0 - next(), u2 = next();
      return sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
    }
    const double nor_r = 3.6541528853610087963519472518, nor_inv_r = 0.27366123732975827203338247596;
    for (;;) {
      uint64_t r = g.next_u64();
      const int idx = (int)(r & 0xff);
      r >>= 8;
      const int sign = (int)(r & 0x1);
      const uint64_t rabs = (r >> 1) & 0x000fffffffffffffull;
      double x = (double)rabs * zig_wi[idx];
      if (sign) x = -x;
      if (rabs < zig_ki[idx]) return x;
      if (idx == 0) {
        for (;;) {
          const double xx = -nor_inv_r * det_log(1.0 - g.next_double());
          const double yy = -det_log(1.0 - g.next_double());
          if (yy + yy > xx * xx) return ((rabs >> 8) & 0x1) ? -(nor_r + xx) : nor_r + xx;
        }
      } else if ((zig_fi[idx - 1] - zig_fi[idx]) * g.next_double() + zig_fi[idx] < det_exp(-0.5 * x * x)) {
        return x;
      }
    }
  }
#endif
};

// MujocoEnv.reset + HopperEnv.reset_model (mujoco_env.py:172-187, hopper_v5.py:322-337)
__device__ void env_reset(const HopperArgs& a, int64_t i, HData& d, PDraws& D, double* __restrict__ obs) {
  const HModel& m = g_pmodel;
  for (int k = 0; k < NV; ++k) d.qacc_warmstart[k] = 0;  // mj_resetData
  for (int u = 0; u < NU; ++u) d.ctrl[u] = 0;
  const double c = a.noise;
  for (int k = 0; k < NQ; ++k) d.qpos[k] = m.qpos0[k] + (-c + (c - -c) * D.next());
#if defined(MJC_ROBOT_HALFCHEETAH)
  for (int k = 0; k < NV; ++k) d.qvel[k] = 0.0 + c * D.normal();  // half_cheetah_v5.py:268-271
#else
  for (int k = 0; k < NV; ++k) d.qvel[k] = 0.0 + (-c + (c - -c) * D.next());
#endif
  mj_forward(m, d);
  write_obs(d, obs);
#if defined(MJC_ROBOT_INVPEND)
  for (int k = 0; k < kInfo; ++k) a.info[k * a.n + i] = 0.0;  // MujocoEnv._get_reset_info: {}
#elif defined(MJC_ROBOT_HALFCHEETAH)
  for (int k = 1; k < kInfo; ++k) a.info[k * a.n + i] = 0.0;
  a.info[0 * a.n + i] = d.qpos[0];                    // _get_reset_info: x_position (half_cheetah_v5.py:278-281)
#else
  for (int k = 2; k < kInfo; ++k) a.info[k * a.n + i] = 0.0;
  a.info[0 * a.n + i] = d.qpos[0];                    // _get_reset_info, hopper_v5.py:339-343
  a.info[1 * a.n + i] = d.qpos[1] - m.qpos0[1];
#endif
}

__device__ void load_state(const HopperArgs& a, int64_t i, HData& d) {
  const int64_t n = a.n;
  for (int k = 0; k < NQ; ++k) d.qpos[k] = a.qpos[k * n + i];
  for (int k = 0; k < NV; ++k) { d.qvel[k] = a.qvel[k * n + i]; d.qacc_warmstart[k] = a.warm[k * n + i]; }
}
__device__ void store_state(const HopperArgs& a, int64_t i, const HData& d) {
  const int64_t n = a.n;
  for (int k = 0; k < NQ; ++k) a.qpos[k * n + i] = d.qpos[k];
  for (int k = 0; k < NV; ++k) { a.qvel[k * n + i] = d.qvel[k]; a.warm[k * n + i] = d.qacc_warmstart[k]; }
  if (d.overflow) *a.overflow = 1;
}

constexpr int kHopperBlock = 64;

__device__ PDraws make_draws(const HopperArgs& a, int64_t i) {
  PDraws D;
  D.numpy = a.rng_mode == B2E_RNG_NUMPY;
  D.seed = a.philox_seed; D.env = (uint64_t)(a.env_offset + i); D.counter = a.call_counter; D.k = 0;
  return D;
}

__global__ void __launch_bounds__(kHopperBlock) hopper_reset_kernel(const HopperArgs a) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  if (a.mask != nullptr && a.mask[i] == 0) return;
  HData d;
  d.overflow = 0;
  PDraws D = make_draws(a, i);
  if (D.numpy) D.g = pcg64_load(a.rng, a.n, i);
  env_reset(a, i, d, D, a.obs + kObs * i);
  if (D.numpy) pcg64_store_state(a.rng, i, D.g);
  store_state(a, i, d);
  a.ctrl[i] = 0;
}

template <typename ActT>
__global__ void __launch_bounds__(kHopperBlock) hopper_step_kernel(const HopperArgs a) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  const HModel& m = g_pmodel;
  const int32_t c = a.ctrl[i];
  HData d;
  d.overflow = 0;
  PDraws D = make_draws(a, i);
  double* __restrict__ obs = a.obs + kObs * i;
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
  const int64_t n = a.n;
  const ActT* act = reinterpret_cast<const ActT*>(a.actions) + i * NU;
  for (int u = 0; u < NU; ++u) d.ctrl[u] = (double)act[u];
#if defined(MJC_ROBOT_INVPEND)
  for (int k = 0; k < a.frame_skip; ++k) mj_step_rk4(m, d);  // do_simulation, inverted_pendulum_v5.py:148
  write_obs(d, obs);
  bool finite = true;
  for (int k = 0; k < kObs; ++k) finite = finite && isfinite(obs[k]);
  const bool term = !finite || fabs(obs[1]) > 0.2;  // inverted_pendulum_v5.py:152-156
  const double reward = term ? 0.0 : 1.0;           // int(not terminated)
  for (int k = 0; k < kInfo - 1; ++k) a.info[k * n + i] = 0.0;
  a.info[5 * n + i] = reward;                       // info["reward_survive"]
#elif defined(MJC_ROBOT_HALFCHEETAH)
  const double x_before = d.qpos[0];  // half_cheetah_v5.py:225
  ActT sq = (ActT)0;  // control_cost on the action as passed (float32: NumPy 2 keeps weight * sum in float32, NEP 50)
  for (int u = 0; u < NU; ++u) sq += act[u] * act[u];
  const double ctrl_cost = (double)((ActT)a.w_ctrl * sq);
  for (int k = 0; k < a.frame_skip; ++k) mj_step_euler(m, d);  // mj_step(nstep=frame_skip), integrator Euler
  const double x_after = d.qpos[0];
  const double dt = m.timestep * a.frame_skip;
  const double xv = (x_after - x_before) / dt;
  write_obs(d, obs);
  const double forward_reward = a.w_forward * xv;
  const double reward = forward_reward - ctrl_cost;  // half_cheetah_v5.py:239-243
  const bool term = false;                           // never terminates
  a.info[0 * n + i] = x_after;
  a.info[1 * n + i] = 0.0;
  a.info[2 * n + i] = xv;
  a.info[3 * n + i] = forward_reward;
  a.info[4 * n + i] = -ctrl_cost;
  a.info[5 * n + i] = 0.0;
#else
  const double x_before = d.qpos[0];  // hopper_v5.py:272
  // control_cost (hopper_v5.py:226-228) squares and sums the ACTION as passed; for float32 actions NumPy 2 keeps the
  // product with the Python float weight in float32 (NEP 50): one rounding per operation, left to right
  ActT sq = (ActT)0;
  for (int u = 0; u < NU; ++u) sq += act[u] * act[u];
  const double ctrl_cost = (double)((ActT)a.w_ctrl * sq);
  for (int k = 0; k < a.frame_skip; ++k) mj_step_rk4(m, d);  // mj_step(nstep=frame_skip), mujoco_env.py:150
  const double x_after = d.qpos[0];
  const double dt = m.timestep * a.frame_skip;
  const double xv = (x_after - x_before) / dt;
  write_obs(d, obs);
  const bool healthy = is_healthy(a, d);
  const double forward_reward = a.w_forward * xv, healthy_reward = healthy ? a.healthy_reward : 0.0;
  const double reward = (forward_reward + healthy_reward) - ctrl_cost;  // hopper_v5.py:305-312
  const bool term = !healthy && a.terminate_when_unhealthy;
  a.info[0 * n + i] = x_after;
  a.info[1 * n + i] = d.qpos[1] - m.qpos0[1];
  a.info[2 * n + i] = xv;
  a.info[3 * n + i] = forward_reward;
  a.info[4 * n + i] = -ctrl_cost;
  a.info[5 * n + i] = healthy_reward;
#endif
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
      for (int k = 0; k < kObs; ++k) a.final_obs[kObs * i + k] = obs[k];
      if (D.numpy) D.g = pcg64_load(a.rng, a.n, i);
      env_reset(a, i, d, D, obs);
      if (D.numpy) pcg64_store_state(a.rng, i, D.g);
      cn = 0;
    }
  }
  store_state(a, i, d);
  a.ctrl[i] = cn;
}

int fill(const b2e_batch* b, const b2e_mjplanar_cfg* cfg, const b2e_mjplanar_state* st, HopperArgs& a, const char* fn) {
  if (int e = check_batch(b, fn)) return e;
  if (!cfg || !st || !st->qpos || !st->qvel || !st->qacc_warmstart || !st->ctrl || !st->overflow ||
      (b->rng_mode == B2E_RNG_NUMPY && !st->rng)) {
    set_error("%s: null pointer in cfg/state", fn);
    return B2E_EINVAL;
  }
  if (cfg->frame_skip <= 0) {
    set_error("%s: frame_skip must be positive", fn);
    return B2E_EINVAL;
  }
  a = HopperArgs{};
  a.n = b->n; a.env_offset = b->env_offset; a.max_steps = b->max_episode_steps; a.mode = b->autoreset_mode;
  a.rng_mode = b->rng_mode; a.philox_seed = b->philox_seed; a.call_counter = b->call_counter;
  a.frame_skip = cfg->frame_skip; a.terminate_when_unhealthy = cfg->terminate_when_unhealthy;
  a.noise = cfg->reset_noise_scale; a.w_forward = cfg->forward_reward_weight; a.w_ctrl = cfg->ctrl_cost_weight;
  a.healthy_reward = cfg->healthy_reward;
  a.z_min = cfg->healthy_z_min; a.z_max = cfg->healthy_z_max;
  a.angle_min = cfg->healthy_angle_min; a.angle_max = cfg->healthy_angle_max;
  a.state_min = cfg->healthy_state_min; a.state_max = cfg->healthy_state_max;
  a.qpos = st->qpos; a.qvel = st->qvel; a.warm = st->qacc_warmstart; a.ctrl = st->ctrl;
  a.rng = st->rng; a.overflow = st->overflow;
  return upload_model();
}

}  // namespace
}  // namespace b2e

using namespace b2e;

extern "C" int MJC_API(model_info)(double* body_mass, double* misc, double* invweight) {
  if (!body_mass || !misc || !invweight) {
    set_error("b2e_" MJC_NAME "_model_info: null pointer");
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

extern "C" int MJC_API(reset)(const b2e_batch* b, const b2e_mjplanar_cfg* cfg, const b2e_mjplanar_state* st,
                                const uint8_t* mask, double* obs, double* info, void* stream) {
  HopperArgs a;
  if (int e = fill(b, cfg, st, a, "b2e_" MJC_NAME "_reset")) return e;
  if (!obs || !info) {
    set_error("b2e_" MJC_NAME "_reset: null output pointer");
    return B2E_EINVAL;
  }
  if (b->n == 0) return 0;
  a.mask = mask; a.obs = obs; a.info = info;
  hopper_reset_kernel<<<grid_for(b->n, kHopperBlock), kHopperBlock, 0, (cudaStream_t)stream>>>(a);
  return cuda_status(cudaGetLastError(), "b2e_" MJC_NAME "_reset");
}

extern "C" int MJC_API(step)(const b2e_batch* b, const b2e_mjplanar_cfg* cfg, const b2e_mjplanar_state* st,
                               const void* actions, double* obs, double* reward, uint8_t* terminated,
                               uint8_t* truncated, double* info, double* final_obs, void* stream) {
  HopperArgs a;
  if (int e = fill(b, cfg, st, a, "b2e_" MJC_NAME "_step")) return e;
  if (!actions || !obs || !reward || !terminated || !truncated || !info ||
      (b->autoreset_mode == B2E_AUTORESET_SAME_STEP && !final_obs)) {
    set_error("b2e_" MJC_NAME "_step: null pointer");
    return B2E_EINVAL;
  }
  if (b->n == 0) return 0;
  a.actions = actions; a.obs = obs; a.reward = reward; a.term = terminated; a.trunc = truncated; a.info = info;
  a.final_obs = final_obs;
  const unsigned grid = grid_for(b->n, kHopperBlock);
  cudaStream_t s = (cudaStream_t)stream;
  switch (b->action_dtype) {
    case B2E_ACT_F32: hopper_step_kernel<float><<<grid, kHopperBlock, 0, s>>>(a); break;
    case B2E_ACT_F64: hopper_step_kernel<double><<<grid, kHopperBlock, 0, s>>>(a); break;
    default: set_error("b2e_" MJC_NAME "_step: action_dtype %d is not a float dtype", b->action_dtype); return B2E_EINVAL;
  }
  return cuda_status(cudaGetLastError(), "b2e_" MJC_NAME "_step");
}
